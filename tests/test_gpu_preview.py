"""GPU parity tests for the channel preview / colour statistics pass (SURVEY.md §8f N3/N4): CalcChannelPreviewFull with
bHistoEn / bStatClipEn (ConvertYCCtoRGB + CapYccRange + CapRgbRange, ImgDecode.cpp:4229-4601), the preview modes
(ChannelExtract, :4832-4876) and the YCC level shift (:4733-4739) — DIB, m_sHisto, m_sStatClip, m_anCcHisto_*, m_anHistoYFull,
the histogram bitmaps, the "YCC Clipped" notes and the whole non-quiet report against what the compiled reference computed
(tests/golden/ref_outputs.json.gz, recorded by record_reference below)."""
import numpy as np
import pytest

import jpeg_cases as JC
import ref_golden as RG

pytestmark = pytest.mark.gpu

HISTO_FLAGS = [(True, False, True), (True, False, False), (False, True, False)]
STEPS = [("mode", m) for m in (2, 3, 4, 5, 6, 7, 8, 1, 0, 9)] + [("shift", (3, 2, 100, -50, 30)), ("mode", 2), ("shift", (0, 0, -2000, 900, 3000)),
                                                               ("mode", 1), ("shift", (0, 0, 0, 0, 0))]


@pytest.fixture(scope="module")
def cases():
    return JC.small_cases()


def _flipped(j, n, seed):
    r = np.random.default_rng(seed)
    a = bytearray(j); lo = j.index(b"\xff\xda") + 14
    for p in r.integers(lo, len(j) - 2, n):
        a[p] ^= 1 << int(r.integers(0, 8))
    return bytes(a)


def _histo_cases(cases):
    return list(cases) + [("flip200", _flipped(cases[2][1], 200, 1)), ("flip40_nodri", _flipped(cases[3][1], 40, 2)), ("flip3_444", _flipped(cases[0][1], 3, 3))]


def _shift_cases(cases):
    return (cases[0], cases[2], ("flip200", _flipped(cases[2][1], 200, 1)))


def _batch_cases(cases):
    return [n for n, _ in cases] + ["flip200"], [j for _, j in cases] + [_flipped(cases[2][1], 200, 1)]


def _same_stats(want, got, what):
    got = RG.colour_stats(got)
    for k in ("clip", "ranges", "cc_histo", "y_histo"):
        assert want[k] == got[k], (what, k, want[k], got[k])
    assert want["count"] == got["count"], (what, want["count"], got["count"])


@pytest.mark.parametrize("flags", HISTO_FLAGS, ids=["histo+dumpY", "histo", "statclip"])
def test_histogram_and_clip_statistics_match_the_reference(built, cases, flags):
    from jpegsnoop_b200 import CimgDecode
    dec = CimgDecode(); dec.config_histo(*flags)
    for name, j in _histo_cases(cases):
        key = f"histo/{flags}/{name}"
        want = RG.get_decoded(key); got = dec.decode(j, quiet=False)
        bad = JC.compare(want, got)
        assert not bad, f"{name}: mismatch in {bad}"
        assert np.array_equal(np.asarray(want.stats), np.asarray(got.stats)), (name, want.stats, got.stats)
        _same_stats(RG.get(key + "/colour"), dec.colour_stats(), name)
        for which in (0, 1):
            assert RG.same(RG.get(f"{key}/histo_dib{which}"), dec.histo_dib(which)), (name, "histogram bitmap", which)
        diff = RG.lines_diff(RG.get(key + "/lines"), dec.log_lines(-1))
        assert not diff, (name, diff)


def test_preview_modes_and_ycc_shift_match_the_reference(built, cases):
    """SetPreviewMode / SetPreviewYccOffset recompute the DIB from the pixel maps (ImgDecode.cpp:631-659); with the histogram
    on, every pass ADDS to the statistics (they are cleared by DecodeScanImg only, :3144-3156) and draws on what is left of the
    ten "YCC Clipped" notes."""
    from jpegsnoop_b200 import CimgDecode
    for histo in (False, True):
        dec = CimgDecode(); dec.config_histo(histo, False, False)
        for name, j in _shift_cases(cases):
            key = f"shift/{histo}/{name}"
            got = dec.decode(j)
            assert not JC.compare(RG.get_decoded(key), got), name
            for k, (kind, arg) in enumerate(STEPS):
                if kind == "mode":
                    dec.SetPreviewMode(arg)
                else:
                    dec.SetPreviewYccOffset(*arg)
                    assert dec.GetPreviewYccOffset() == arg
                want = RG.get(f"{key}/{k}")
                assert RG.same(want["bitmap"], dec.bitmap()), (name, histo, kind, arg)
                gs = np.zeros(12, np.int32); dec.L.jsimg_GetStats(dec.h, gs.ctypes.data)
                assert want["stats"] == gs.tolist(), (name, histo, kind, arg, want["stats"], gs)
                _same_stats(want["colour"], dec.colour_stats(), (name, histo, kind, arg))
            assert not RG.lines_diff(RG.get(key + "/lines"), dec.log_lines(-1)), name
            # both decoders end in the default state for the next image (the settings outlive a decode, as in the reference)
        dec.close()


def test_batch_preview_matches_the_reference(built, cases):
    """The same pass through the batch C-ABI: jsgpu_set_preview makes jsgpu_batch_decode run it, jsgpu_batch_preview runs it
    again with other settings, jsgpu_batch_colour_stats hands out the per-image statistics."""
    from jpegsnoop_b200 import BatchDecoder
    names, jpegs = _batch_cases(cases)
    bd = BatchDecoder()
    bd.set_preview(hist_en=1)
    bd.set_batch(jpegs)
    bd.decode(); bd.sync()
    order = (0, 1, 2, 3, 4, 5, 9, 10, 11, 6, 7, 8)          # PixelCcHisto's member order -> jsgpu_colour_stats channel order
    for i, name in enumerate(names):
        key = f"batch/{name}"
        want = RG.get_decoded(key); got = bd.fetch(i)
        bad = JC.compare(want, got, what=("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo"))
        assert not bad, f"{name}: mismatch in {bad}"
        ws = RG.get(key + "/colour"); s = bd.colour_stats(i)
        assert RG.same(ws["clip"], np.array(s.clip[:], np.uint32)), (name, ws["clip"], s.clip[:])
        assert RG.same(ws["y_histo"], np.array(s.y_histo[:], np.uint32)), name
        assert RG.same(ws["cc_histo"], np.array([list(r) for r in s.cc_histo], np.uint32)), name
        assert ws["count"] == s.count, name
        rng = np.array([[s.vmin[k], s.vmax[k], np.int64(s.vsum[k]).astype(np.int32)] for k in order], np.int32).ravel()
        assert RG.same(ws["ranges"], rng), (name, ws["ranges"], rng)
    # a second pass over the resident batch: luminance-only preview with a level shift, no statistics
    bd.preview(mode=6, shift_y=64, shift_mcu_x=1, shift_mcu_y=1)
    bd.sync()
    for i, name in enumerate(names):
        assert RG.same(RG.get(f"batch/{name}/luma_shift64"), bd.fetch(i).dib), name


def record_reference(orc):
    """What the compiled reference computes for the tests above, in the same order (tests/golden/make_golden.py stores it)."""
    out = {}
    cases = JC.small_cases()

    def fresh():
        o = orc("ref_fixed")
        o.config_histo(False, False, False)                 # the reference's configuration is process-wide
        return o
    for flags in HISTO_FLAGS:
        ref = fresh(); ref.config_histo(*flags)
        for name, j in _histo_cases(cases):
            key = f"histo/{flags}/{name}"
            out[key] = RG.decoded(ref.decode(j, quiet=False))
            out[key + "/colour"] = RG.colour_stats(ref.colour_stats())
            for which in (0, 1):
                out[f"{key}/histo_dib{which}"] = RG.arr(ref.histo_dib(which))
            out[key + "/lines"] = RG.lines(ref.log_lines())
        ref.config_histo(False, False, False); ref.close()
    ref = fresh()
    for histo in (False, True):
        ref.config_histo(histo, False, False)
        for name, j in _shift_cases(cases):
            key = f"shift/{histo}/{name}"
            out[key] = RG.decoded(ref.decode(j))
            for k, (kind, arg) in enumerate(STEPS):
                if kind == "mode":
                    ref.set_preview_mode(arg)
                else:
                    ref.set_ycc_offset(*arg)
                ws = np.zeros(12, np.int32); ref._f("stats")(ref.ctx, ws.ctypes.data)
                out[f"{key}/{k}"] = {"bitmap": RG.arr(ref.bitmap()), "stats": ws.tolist(), "colour": RG.colour_stats(ref.colour_stats())}
            out[key + "/lines"] = RG.lines(ref.log_lines())
    ref.config_histo(False, False, False); ref.close()
    ref = fresh()
    ref.config_histo(True, False, False)
    names, jpegs = _batch_cases(cases)
    for name, j in zip(names, jpegs):
        out[f"batch/{name}"] = RG.decoded(ref.decode(j))
        out[f"batch/{name}/colour"] = RG.colour_stats(ref.colour_stats())
    ref.config_histo(False, False, False)
    for name, j in zip(names, jpegs):
        ref.decode(j); ref.set_ycc_offset(1, 1, 64, 0, 0); ref.set_preview_mode(6)
        out[f"batch/{name}/luma_shift64"] = RG.arr(ref.bitmap())
        ref.set_ycc_offset(0, 0, 0, 0, 0); ref.set_preview_mode(1)
    ref.close()
    return out
