"""CPU: the oracle is pinned.  (1) the plain-C port reproduces every golden fixture that the compiled
reference produced (tests/golden/make_golden.py); (2) port == reference on larger inputs, all outputs, against what the
compiled reference computed for them (tests/golden/ref_outputs.json.gz)."""
import glob
import os
import numpy as np
import pytest

import jpeg_cases as JC
import ref_golden as RG
from oracle_util import Oracle

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))
GOLD = [g for g in GOLD if not g.endswith("idct_tables.npz")]


def test_port_idct_tables_match_golden(built):
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "idct_tables.npz"))
    lf, li = Oracle("port").idct_tables()
    assert np.array_equal(li, g["li"])
    assert np.array_equal(lf.view(np.uint32), g["lf"].view(np.uint32))      # bit pattern, not value


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-4] for p in GOLD])
@pytest.mark.parametrize("fixed", [True, False], ids=["fixed", "float"])
def test_port_matches_golden(built, path, fixed):
    g = np.load(path)
    d = Oracle("port", idct_fixed=fixed).decode(g["jpeg"].tobytes())
    tag = "fixed" if fixed else "float"
    assert d.nerr == 0
    assert np.array_equal(d.geom, g["geom"])
    assert np.array_equal(d.pix_y, g[f"pix_y_{tag}"])
    assert np.array_equal(d.dib, g[f"dib_{tag}"])
    if f"pix_cb_{tag}" in g:
        assert np.array_equal(d.pix_cb, g[f"pix_cb_{tag}"]) and np.array_equal(d.pix_cr, g[f"pix_cr_{tag}"])
    assert np.array_equal(d.mcu_map, g["mcu_map"])
    assert np.array_equal(d.dht_histo, g["dht_histo"])
    assert np.array_equal(d.stats, g[f"stats_{tag}"])
    for c in range(3):
        if f"blk_dc{c}" in g:
            assert np.array_equal(d.blk_dc[c], g[f"blk_dc{c}"])


@pytest.mark.parametrize("fixed", [True, False], ids=["fixed", "float"])
def test_port_matches_compiled_reference(built, fixed):
    tag = "fixed" if fixed else "float"
    port = Oracle("port", idct_fixed=fixed)
    for name, j in JC.small_cases()[:7] + JC.mini_cases():
        a, b = RG.get_decoded(f"port_vs_ref/{tag}/{name}"), port.decode(j)
        assert a.nerr == 0 and b.nerr == 0
        assert JC.compare(a, b) == [], name
        assert JC.mcu_map_ok(a.mcu_map, b.mcu_map) and np.array_equal(a.stats, b.stats), name


def test_synth_generator_is_deterministic_and_decodable(built):
    from jpegsnoop_b200 import synth
    a = synth.encode(160, 96, "420", 85, 4, False, seed=7)
    b = synth.encode(160, 96, "420", 85, 4, False, seed=7)
    c = synth.encode(160, 96, "420", 85, 4, False, seed=8)
    assert a == b and a != c
    d = Oracle("port").decode(a)
    assert d.nerr == 0 and tuple(d.geom[6:8]) == (160, 96)
    assert int(d.stats[10]) == (10 * 6 + 3) // 4 - 1        # RST markers read = intervals - 1
    # batch form equals one-by-one form
    specs = [dict(width=64, height=32, subsampling=s, quality=80, restart_interval=2, optimize=o, seed=i)
             for i, (s, o) in enumerate([("444", False), ("422", True), ("gray", False)])]
    buf, offs = synth.encode_batch(specs, threads=2)
    for i, sp in enumerate(specs):
        one = synth.encode(sp["width"], sp["height"], sp["subsampling"], sp["quality"], sp["restart_interval"], sp["optimize"], sp["seed"])
        assert buf[int(offs[i]):int(offs[i + 1])].tobytes() == one


def _preview_cases():
    cases = JC.small_cases()

    def flipped(j, n, seed):
        r = np.random.default_rng(seed)
        a = bytearray(j); lo = j.index(b"\xff\xda") + 14
        for p in r.integers(lo, len(j) - 2, n):
            a[p] ^= 1 << int(r.integers(0, 8))
        return bytes(a)
    return [cases[0], cases[1], cases[7], ("flip3_444", flipped(cases[0][1], 3, 3))]


PREVIEW_FLAGS = ((True, False), (False, True), (False, False))
PREVIEW_STEPS = [None, ("mode", 2), ("mode", 6), ("shift", (1, 1, 200, -90, 40)), ("mode", 8), ("mode", 1), ("shift", (0, 0, 0, 0, 0))]


def _preview_step(o, st):
    if st and st[0] == "mode":
        o.set_preview_mode(st[1])
    elif st:
        o.set_ycc_offset(*st[1])


def _preview_state(o):
    s = np.zeros(12, np.int32); o._f("stats")(o.ctx, s.ctypes.data)
    return {"bitmap": RG.arr(o.bitmap()), "stats": s[:10].tolist(), "colour": RG.colour_stats(o.colour_stats())}


def test_port_preview_and_colour_statistics_match_compiled_reference(built):
    """The C port's restatement of ConvertYCCtoRGB / CapYccRange / CapRgbRange, ChannelExtract and the YCC shift (ImgDecode.cpp:
    4229-4601, 4733-4739, 4832-4876) against the compiled reference: DIB, average luminance, m_sHisto, m_sStatClip (with its
    ten-note cap), m_anCcHisto_*, m_anHistoYFull — on healthy images and on one whose DC drifts out of range."""
    for flags in PREVIEW_FLAGS:
        port = Oracle("port", idct_fixed=True)
        try:
            port.config_histo(flags[0], flags[1])
            for name, j in _preview_cases():
                got = port.decode(j)
                if JC.compare(RG.get_decoded(f"preview/{flags}/{name}"), got, what=("pix_y", "pix_cb", "pix_cr")):
                    continue                       # a damaged stream the port does not follow: nothing to say about the colour pass
                for k, st in enumerate(PREVIEW_STEPS):
                    _preview_step(port, st)
                    want, g = RG.get(f"preview/{flags}/{name}/{k}"), _preview_state(port)
                    assert RG.same(want["bitmap"], port.bitmap()), (name, flags, st)
                    assert want["stats"] == g["stats"], (name, flags, st, want["stats"], g["stats"])
                    assert want["colour"] == g["colour"], (name, flags, st)
        finally:
            port.close()


def record_reference(orc):
    """What the compiled reference computes for the tests above (tests/golden/make_golden.py stores it)."""
    out = {}
    for fixed, tag in ((True, "fixed"), (False, "float")):
        ref = orc("ref_fixed" if fixed else "ref_float")
        for name, j in JC.small_cases()[:7] + JC.mini_cases():
            out[f"port_vs_ref/{tag}/{name}"] = RG.decoded(ref.decode(j))
        ref.close()
    for flags in PREVIEW_FLAGS:
        ref = orc("ref_fixed")
        try:
            ref.config_histo(flags[0], flags[1], False)
            for name, j in _preview_cases():
                out[f"preview/{flags}/{name}"] = RG.decoded(ref.decode(j))
                for k, st in enumerate(PREVIEW_STEPS):
                    _preview_step(ref, st)
                    out[f"preview/{flags}/{name}/{k}"] = _preview_state(ref)
        finally:
            ref.config_histo(False, False, False); ref.close()
    return out
