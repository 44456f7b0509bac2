"""GPU parity for the "Detailed Decode" (CimgDecode::SetDetailVlc, ImgDecode.cpp:4880-4904): DecodeScanCompPrint's symbol-by-symbol
ReportVlc lines and coefficient matrices (:1859-2232) and CalcChannelPreviewFull's RGB dump of the chosen MCU (:4683-4799) —
the complete log, line for line, and every output buffer (in DC-only mode the printed MCUs are decoded in full, as there),
against what the compiled reference computed (tests/golden/ref_outputs.json.gz, recorded by record_reference below)."""
import numpy as np
import pytest

import jpeg_cases as JC
import ref_golden as RG

pytestmark = pytest.mark.gpu


def _flipped(j, n, seed):
    r = np.random.default_rng(seed)
    a = bytearray(j); lo = j.index(b"\xff\xda") + 14
    for p in r.integers(lo, len(j) - 2, n):
        a[p] ^= 1 << int(r.integers(0, 8))
    return bytes(a)


def _check(dec, key, name, j, what):
    got = dec.decode(j, quiet=False)
    bad = JC.compare(RG.get_decoded(key), got)
    assert not bad, f"{name} {what}: mismatch in {bad}"
    diff = RG.lines_diff(RG.get(key + "/lines"), dec.log_lines(-1))
    assert not diff, (name, what, diff)


def _detail_runs(cases, decode_ac, geom):
    """(name, jpeg, (x, y, n)) of the detailed decodes; geom(name, jpeg) gives the image's geometry."""
    runs = []
    for name, j in cases[:4]:
        g = geom(name, j)
        mxm, mym = int(g[2]), int(g[3])
        ranges = [(0, 0, 1), (1, 0, 2), (mxm - 1, 0, 2),                  # first MCU; two MCUs; across the end of an MCU row (right edge)
                  (mxm // 2, mym // 2, 3), (mxm - 2, mym - 1, 5),           # middle; past the last MCU of the image
                  (mxm + 3, 0, 1), (0, mym + 2, 1)]                         # column beyond the image / row beyond it: nothing to print
        runs += [(name, j, r) for r in (ranges[:4 if decode_ac else 7] if name != cases[0][0] else ranges)]
    # damaged scans: error lines and dump lines interleave; the error cap is shared
    good = cases[2][1]
    for seed, r in ((1, (0, 0, 40)), (7, (10, 3, 30))):
        runs.append((f"flip200/{seed}", _flipped(good, 200, seed), r))
    return runs


@pytest.mark.parametrize("decode_ac", [True, False], ids=["full_idct", "dc_only"])
def test_detailed_decode_matches_the_reference(built, decode_ac):
    from jpegsnoop_b200 import CimgDecode
    dec = CimgDecode(decode_ac=decode_ac)
    for name, j, (x, y, n) in _detail_runs(JC.small_cases(), decode_ac, lambda name, j: RG.get(f"detail/geom/{name}")):
        dec.SetDetailVlc(True, x, y, n)
        _check(dec, f"detail/{decode_ac}/{name}/{x},{y},{n}", name, j, (x, y, n))


def test_detailed_rgb_dump_with_histogram_notes_and_preview_modes(built):
    """The RGB dump prints the pixel before ChannelExtract, whatever the preview mode; "YCC Clipped" notes of the same pass appear
    between its lines; SetPreviewMode repeats the dump."""
    from jpegsnoop_b200 import CimgDecode
    cases = JC.small_cases()
    dec = CimgDecode(); dec.config_histo(True, False, False)
    j = _flipped(cases[2][1], 200, 1)
    # an MCU in the first MCU row that has clip notes, and one at the right edge
    for (x, y) in ((105, 1), (int(RG.get("rgbdump/geom")[2]) - 1, 1), (3, 0)):
        key = f"rgbdump/{x},{y}"
        dec.SetDetailVlc(True, x, y, 1)
        _check(dec, key, "flip200+histo", j, (x, y))
        for mode in (2, 6, 1):
            dec.SetPreviewMode(mode)
            assert RG.same(RG.get(f"{key}/mode{mode}"), dec.bitmap()), (x, y, mode)
            assert not RG.lines_diff(RG.get(f"{key}/mode{mode}/lines"), dec.log_lines(-1)), (x, y, mode)
        dec.SetPreviewYccOffset(0, 0, 300, -40, 25)
        dec.SetPreviewMode(2)
        assert not RG.lines_diff(RG.get(key + "/shift/lines"), dec.log_lines(-1)), (x, y, "shift")
        dec.SetPreviewYccOffset(0, 0, 0, 0, 0)
        dec.SetPreviewMode(1)
    # the fast conversion (no histogram), a non-RGB mode set BEFORE the decode
    dec.config_histo(False, False, False)
    dec.SetPreviewMode(7)
    dec.SetDetailVlc(True, 4, 2, 2)
    _check(dec, "rgbdump/mode7", "mode7", cases[1][1], (4, 2, 2))
    dec.SetPreviewMode(1)


def record_reference(orc):
    """What the compiled reference computes for the tests above, in the same order (tests/golden/make_golden.py stores it)."""
    out = {}
    cases = JC.small_cases()

    def run(ref, key, j):
        out[key] = RG.decoded(ref.decode(j, quiet=False)); out[key + "/lines"] = RG.lines(ref.log_lines())

    def geom(name, j):
        out[f"detail/geom/{name}"] = ref.decode(j).geom.tolist()
        return out[f"detail/geom/{name}"]
    for decode_ac in (True, False):
        ref = orc("ref_fixed", decode_ac=decode_ac)
        try:
            for name, j, (x, y, n) in _detail_runs(cases, decode_ac, geom):
                ref.set_detail_vlc(True, x, y, n)
                run(ref, f"detail/{decode_ac}/{name}/{x},{y},{n}", j)
        finally:
            ref.set_detail_vlc(False); ref.close()
    ref = orc("ref_fixed")
    try:
        ref.config_histo(True, False, False)
        j = _flipped(cases[2][1], 200, 1)
        out["rgbdump/geom"] = ref.decode(j).geom.tolist()
        for (x, y) in ((105, 1), (out["rgbdump/geom"][2] - 1, 1), (3, 0)):
            key = f"rgbdump/{x},{y}"
            ref.set_detail_vlc(True, x, y, 1)
            run(ref, key, j)
            for mode in (2, 6, 1):
                ref.set_preview_mode(mode)
                out[f"{key}/mode{mode}"] = RG.arr(ref.bitmap()); out[f"{key}/mode{mode}/lines"] = RG.lines(ref.log_lines())
            ref.set_ycc_offset(0, 0, 300, -40, 25)
            ref.set_preview_mode(2)
            out[key + "/shift/lines"] = RG.lines(ref.log_lines())
            ref.set_ycc_offset(0, 0, 0, 0, 0)
            ref.set_preview_mode(1)
        ref.config_histo(False, False, False)
        ref.set_preview_mode(7)
        ref.set_detail_vlc(True, 4, 2, 2)
        run(ref, "rgbdump/mode7", cases[1][1])
        ref.set_preview_mode(1)
    finally:
        ref.set_detail_vlc(False); ref.config_histo(False, False, False); ref.close()
    return out
