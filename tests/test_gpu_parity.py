"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C-ABI
(jsimg_* = CimgDecode drop-in, jsgpu_* = batch), against the CPU oracle — bit-exact on every
output buffer: int16 Y/Cb/Cr maps, BGRA DIB, block-DC maps, MCU file map, code-length histogram,
brightest-pixel / average-luma scalars."""
import numpy as np
import pytest

import jpeg_cases as JC
import ref_golden as RG
from oracle_util import Oracle, ref_available

pytestmark = pytest.mark.gpu


def _oracle(fixed):
    if ref_available("fixed" if fixed else "float"):
        return Oracle("ref_fixed" if fixed else "ref_float")      # the compiled reference itself
    return Oracle("port", idct_fixed=fixed)


@pytest.fixture(scope="module")
def cases():
    return JC.small_cases()


@pytest.mark.parametrize("kernels", [(1, 1), (2, 2), (1, 3), (2, 1), (0, 0)], ids=["warp+simple", "lane+tma_tile", "warp+ldg_tile", "lane+simple", "auto"])
@pytest.mark.parametrize("fixed", [True, False], ids=["idct_fixed", "idct_float"])
def test_single_image_dropin_matches_oracle(built, cases, fixed, kernels):
    from jpegsnoop_b200 import CimgDecode
    orc = _oracle(fixed)
    dec = CimgDecode(idct_fixedpt=fixed, huff_kernel=kernels[0], idct_kernel=kernels[1])
    for name, j in cases:
        want = orc.decode(j)
        got = dec.decode(j)
        assert got.nerr == 0 and want.nerr == 0, (name, dec.log_lines(3))
        bad = JC.compare(want, got)
        assert not bad, f"{name}: mismatch in {bad}"
        want_stats = np.asarray(want.stats); got_stats = np.asarray(got.stats)
        assert np.array_equal(want_stats, got_stats), (name, want_stats, got_stats)


@pytest.mark.parametrize("kernels", [(1, 1), (2, 2), (2, 3), (0, 0)], ids=["warp+simple", "lane+tma_tile", "lane+ldg_tile", "auto"])
def test_batch_matches_oracle(built, cases, kernels):
    from jpegsnoop_b200 import BatchDecoder
    orc = _oracle(True)
    bd = BatchDecoder(huff_kernel=kernels[0], idct_kernel=kernels[1])
    jpegs = [j for _, j in cases]
    bd.set_batch(jpegs)
    bd.decode(); bd.sync()
    for i, (name, j) in enumerate(cases):
        want = orc.decode(j); got = bd.fetch(i)
        assert got.status == 0, (name, got.status)
        bad = JC.compare(want, got, what=("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo"))
        assert not bad, f"{name}: mismatch in {bad}"


@pytest.mark.parametrize("huff", [1, 2, 0], ids=["warp", "lane", "auto"])
def test_unusual_tables_and_layouts_match_oracle(built, huff):
    """Hand-made DHTs with many long codes (second-level look-up larger / smaller than the lane kernel's
    shared-memory copy) and 4:1:1 / 4:4:0 layouts, single-image drop-in and batch."""
    from jpegsnoop_b200 import CimgDecode, BatchDecoder
    orc = _oracle(True)
    cases = JC.mini_cases()
    dec = CimgDecode(idct_fixedpt=True, huff_kernel=huff, idct_kernel=0)
    for name, j in cases:
        want = orc.decode(j); got = dec.decode(j)
        assert got.nerr == 0 and want.nerr == 0, (name, dec.log_lines(3))
        assert not JC.compare(want, got), name
    bd = BatchDecoder(huff_kernel=huff, idct_kernel=0)
    bd.set_batch([j for _, j in cases]); bd.decode(); bd.sync()
    for i, (name, j) in enumerate(cases):
        got = bd.fetch(i)
        assert got.status == 0, (name, got.status)
        assert not JC.compare(orc.decode(j), got, what=("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo")), name


@pytest.mark.parametrize("huff", [0, 1, 2], ids=["auto_selfsync", "warp", "lane"])
def test_long_intervals_match_oracle(built, huff):
    """Scans without restart markers (BASELINE config 5: the reference's single serial walk, ImgDecode.cpp:3164-3630) and
    DRIs of whole MCU rows, incl. a full 4K 4:2:0 frame; plus a full 4K frame with DRI = 8 (config 3).  huff_kernel 0 takes
    the self-synchronising passes; 1 and 2 decode the same images as one chain per interval.  Single-image drop-in and one
    mixed batch (long and short intervals side by side), every output buffer."""
    from jpegsnoop_b200 import CimgDecode, BatchDecoder
    orc = _oracle(True)
    cases = JC.long_cases()
    want = [orc.decode(j) for _, j in cases]
    dec = CimgDecode(idct_fixedpt=True, huff_kernel=huff, idct_kernel=0)
    for (name, j), w in zip(cases, want):
        got = dec.decode(j)
        assert got.nerr == 0 and w.nerr == 0, (name, dec.log_lines(3))
        bad = JC.compare(w, got)
        assert not bad, f"{name}: mismatch in {bad}"
    short = JC.small_cases()[:2]
    allc = [cases[0], short[0]] + cases[2:] + [short[1], cases[1]]
    bd = BatchDecoder(huff_kernel=huff, idct_kernel=0)
    bd.set_batch([j for _, j in allc]); bd.decode(); bd.sync()
    if huff == 0:
        nimg, nslots, chg = bd.selfsync_info()
        assert nimg >= len(cases) - 1 and nslots > 0, (nimg, nslots)
    for i, (name, j) in enumerate(allc):
        got = bd.fetch(i)
        assert got.status == 0, (name, got.status)
        bad = JC.compare(orc.decode(j), got, what=("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo"))
        assert not bad, f"{name} (batch): mismatch in {bad}"


@pytest.mark.parametrize("huff", [0, 1, 2], ids=["auto", "warp", "lane"])
def test_dc_only_mode_matches_oracle(built, cases, huff):
    """CSnoopConfig::bDecodeScanImgAc = false: AC symbols are parsed but not stored (ImgDecode.cpp:1759-1766)."""
    from jpegsnoop_b200 import CimgDecode
    orc = Oracle("ref_fixed", decode_ac=False) if ref_available("fixed") else Oracle("port", idct_fixed=True, decode_ac=False)
    dec = CimgDecode(decode_ac=False, idct_fixedpt=True, huff_kernel=huff, idct_kernel=0)
    for name, j in cases[:6] + JC.mini_cases()[:2] + JC.long_cases()[2:4]:
        want = orc.decode(j); got = dec.decode(j)
        assert got.nerr == 0 and want.nerr == 0, (name, dec.log_lines(3))
        assert not JC.compare(want, got), name


def _damaged_cases(cases):
    """name -> (jpeg bytes, overlays): truncation, bit flips, zero fill, stray markers, FFFF runs, restart markers swapped /
    removed / inserted — what JPEGsnoop exists to look at (SURVEY.md §8f N2)."""
    good_name, good = cases[2]                               # 1080p 4:2:0 DRI=4
    nodri = cases[3][1]                                      # no restart markers: one long interval
    g444 = cases[0][1]                                       # 4:4:4, RST every MCU row
    body0 = good.index(b"\xff\xda") + 14

    def flipped(j, n, seed):
        r = np.random.default_rng(seed)
        a = bytearray(j); lo = j.index(b"\xff\xda") + 14
        for p in r.integers(lo, len(j) - 2, n): a[p] ^= 1 << int(r.integers(0, 8))
        return bytes(a)

    def rst_positions(j):
        lo = j.index(b"\xff\xda") + 14
        return [i for i in range(lo, len(j) - 1) if j[i] == 0xFF and 0xD0 <= j[i + 1] <= 0xD7]
    rp = rst_positions(good)
    swapped = bytearray(good); swapped[rp[10] + 1], swapped[rp[11] + 1] = swapped[rp[11] + 1], swapped[rp[10] + 1]
    removed = good[:rp[20]] + good[rp[20] + 2:]
    inserted = good[:rp[30] + 40] + b"\xff\xd3" + good[rp[30] + 40:]
    mid = body0 + 30000
    return {
        "trunc_mid": (good[: body0 + (len(good) - body0) // 2] + b"\xff\xd9", ()),
        "flip200": (flipped(good, 200, 1), ()),
        "flip40_nodri": (flipped(nodri, 40, 2), ()),
        "zerotail": (good[: body0 + 5000] + bytes(len(good) - body0 - 5002) + b"\xff\xd9", ()),
        "cut_noeoi": (nodri[: len(nodri) // 2], ()),
        "flip3_444": (flipped(g444, 3, 3), ()),
        "flip1": (flipped(good, 1, 4), ()),
        "flip2_nodri": (flipped(nodri, 2, 6), ()),
        "stray_marker": (good[:mid] + b"\xff\xe1" + good[mid:], ()),
        "early_eoi": (good[:mid] + b"\xff\xd9" + good[mid:], ()),
        "ffff_run": (good[:mid] + b"\xff\xff\xff" + good[mid:], ()),
        "rst_swapped": (bytes(swapped), ()),
        "rst_removed": (removed, ()),
        "rst_inserted": (inserted, ()),
        "overlay_bytes": (good, ((mid, b"\x12\x34\x56\x78"), (mid + 2, b"\xab"))),      # CwindowBuf overlays (WindowBuf.cpp:516-560), the later one wins
    }


@pytest.mark.parametrize("huff", [0, 1, 2], ids=["auto", "warp", "lane"])
def test_damaged_scans_match_the_reference(built, cases, huff):
    """Damaged scans, single-image drop-in: every output buffer AND every error line equal to the compiled reference's
    (tests/golden/ref_outputs.json.gz) —
    its one-bit resynchronisation (ImgDecode.cpp:1166-1187), stray-marker handling (:1486-1561, 1683-1706), lazy restarts
    (:1644-1680), underflowing blocks (:1737-1760), the one-MCU-per-row tail after an overread (:3621-3625) and the
    nErrMaxDecodeScan cap (:1100-1110)."""
    from jpegsnoop_b200 import CimgDecode
    dec = CimgDecode(idct_fixedpt=True, huff_kernel=huff, idct_kernel=0)
    for name, (j, ovl) in _damaged_cases(cases).items():
        want = RG.get_decoded(f"damaged/{name}"); want_lines = RG.get(f"damaged/{name}/err_lines")
        dec.L.jsimg_overlay_remove_all(dec.h)
        keep = []
        for off, data in ovl:
            ob = np.frombuffer(bytes(data), np.uint8).copy(); keep.append(ob)
            dec.L.jsimg_overlay_install(dec.h, int(off), ob.ctypes.data, ob.size)
        got = dec.decode(j)
        bad = JC.compare(want, got)
        assert not bad, f"{name}: mismatch in {bad}"
        assert np.array_equal(np.asarray(want.stats)[10:12], np.asarray(got.stats)[10:12]), (name, want.stats, got.stats)     # m_nRestartRead, m_bScanBad
        diff = RG.lines_diff(want_lines, dec.log_lines(3))
        assert not diff, (name, diff)


def test_damaged_images_in_a_batch_match_the_reference(built, cases):
    """The same in one batch next to healthy images: the damaged ones carry JSGPU_ST_EXACT, their outputs are the reference's,
    their neighbours are untouched; the error-line count comes back through jsgpu_batch_errors."""
    from jpegsnoop_b200 import BatchDecoder
    names, jpegs = _damaged_batch(cases)
    WHAT = ("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo")
    for dc_only in (False, True):
        bd = BatchDecoder(huff_kernel=0, idct_kernel=0, decode_ac=not dc_only)
        bd.set_batch(jpegs); bd.decode(); bd.sync()
        for i, (name, j) in enumerate(zip(names, jpegs)):
            want = RG.get_decoded(f"damaged_batch/{dc_only}/{name}"); got = bd.fetch(i)
            assert not JC.compare(want, got, what=WHAT), (name, dc_only)
            if name.startswith("ok"):
                assert got.status == 0, (name, hex(got.status))
            elif want.nerr:
                assert got.status & 0x40000000, (name, hex(got.status))
                e = bd.scan_errors(i)
                assert e.nerr_lines == want.nerr and e.scan_bad == int(want.stats[11]), (name, e.nerr_lines, want.nerr)


def _damaged_batch(cases):
    dmg = {k: v for k, v in _damaged_cases(cases).items() if not v[1]}
    return ["ok0"] + list(dmg) + ["ok1"], [cases[2][1]] + [v[0] for v in dmg.values()] + [cases[1][1]]


@pytest.mark.parametrize("nrep", [1, 2], ids=["single_stream_15", "chunked_30"])
def test_decode_batch_host_matches_oracle(built, cases, nrep):
    """jsgpu_decode_batch_host (the end-to-end entry point): host bitstream in, host buffers out; with >= 16 images
    it runs as 4 overlapped image ranges on separate streams (tests/conftest.py drops the size threshold)."""
    from jpegsnoop_b200 import BatchDecoder
    allc = (list(cases) + JC.mini_cases()) * nrep
    jpegs = [j for _, j in allc]
    bd = BatchDecoder(huff_kernel=0, idct_kernel=0)
    tarr, darr, bits = bd.prepare(jpegs)
    bd.set_tables(tarr); bd.plan(darr, bits.size)
    lay = bd.layout
    pix_n = sum((int(l.img_x) * int(l.img_y) + 63) // 64 * 64 for l in lay)
    dib_n = sum((int(l.img_x) * int(l.img_y) * 4 + 255) // 256 * 256 for l in lay)
    blk_n = sum((int(l.blk_xmax) * int(l.blk_ymax) + 63) // 64 * 64 for l in lay)
    mcu_n = sum((int(l.mcu_xmax) * int(l.mcu_ymax) + 31) // 32 * 32 for l in lay)
    outs = {"pix_y": np.zeros(pix_n, np.int16), "pix_cb": np.zeros(pix_n, np.int16), "pix_cr": np.zeros(pix_n, np.int16),
            "dib": np.zeros(dib_n, np.uint8), "blk_y": np.zeros(blk_n, np.int16), "blk_cb": np.zeros(blk_n, np.int16),
            "blk_cr": np.zeros(blk_n, np.int16), "mcu_map": np.zeros(mcu_n, np.uint32),
            "dht_histo": np.zeros(len(jpegs) * 136, np.uint32), "stats": np.zeros(len(jpegs) * 16, np.int32)}
    bd.decode_host(darr, bits, outs)
    orc = _oracle(True)
    for i, (name, j) in enumerate(allc):
        got = bd.fetch_host(i, outs)
        assert got.status == 0, (name, got.status)
        assert not JC.compare(orc.decode(j), got, what=("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo")), (i, name)


def test_random_corpus_matches_oracle(built):
    """A seeded corpus of 48 small images — random size, sampling layout, quality, restart interval, optimised or
    standard Huffman tables (Pillow) plus 4:1:1 / 4:4:0 / long-code tables (tests/mini_jpeg.py) — decoded as ONE batch
    (many table sets, many geometries) and compared with the oracle on every output, MCU file map included."""
    import mini_jpeg as MJ
    from jpegsnoop_b200 import BatchDecoder
    rng = np.random.default_rng(20260923)
    named = []
    for i in range(36):
        W, H = int(rng.integers(8, 420)), int(rng.integers(8, 300))
        ss = int(rng.integers(0, 3)); q = int(rng.integers(25, 99)); kw = {}
        mode = int(rng.integers(0, 4))
        if mode == 1: kw["restart_marker_blocks"] = int(rng.integers(1, 9))
        if mode == 2: kw["restart_marker_rows"] = int(rng.integers(1, 3))
        if mode == 3: kw["restart_marker_blocks"] = 1
        img = JC.synth_rgb(W, H, 1000 + i)
        if rng.integers(0, 6) == 0: img = img[:, :, 0]; ss = None
        args = dict(quality=q, optimize=bool(rng.integers(0, 2)), **kw)
        if ss is not None: args["subsampling"] = ss
        named.append((f"pil_{i}_{W}x{H}_ss{ss}_q{q}_{mode}", JC.enc(img, **args)))
    for i in range(12):
        W, H = int(rng.integers(16, 260)), int(rng.integers(16, 200))
        samp = [((2, 2), (1, 1), (1, 1)), ((4, 1), (1, 1), (1, 1)), ((1, 2), (1, 1), (1, 1)), ((2, 1), (1, 1), (1, 1)), ((1, 1), (1, 1), (1, 1))][int(rng.integers(0, 5))]
        n11 = int(rng.integers(0, 28))
        ac = MJ.long_code_table(MJ.all_ac_symbols(), n11=n11)
        named.append((f"mini_{i}_{W}x{H}_{samp[0]}_n11={n11}", MJ.encode(JC.synth_rgb(W, H, 2000 + i), quality=int(rng.integers(40, 97)), samp=samp,
                                                                       dri=int(rng.integers(0, 7)), ac_tabs=[ac, ac])))
    orc = _oracle(True)
    for huff in (0, 2):
        bd = BatchDecoder(huff_kernel=huff, idct_kernel=0)
        bd.set_batch([j for _, j in named]); bd.decode(); bd.sync()
        for i, (name, j) in enumerate(named):
            want = orc.decode(j); got = bd.fetch(i)
            assert want.nerr == 0 and got.status == 0, (name, want.nerr, got.status)
            bad = JC.compare(want, got, what=("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo"))
            assert not bad, f"{name} (huff_kernel={huff}): mismatch in {bad}"


@pytest.mark.parametrize("tab", [0, 1, 2], ids=["table_in_smem", "table_in_constant_bank", "table_as_immediates"])
def test_idct_table_sources_match_oracle(built, cases, tab, monkeypatch):
    """The three sources of the quadrant IDCT table in the fused kernel (JSGPU_IDCT_TABLE: what runs when the host libm's table
    differs from the build box's, and the default immediates) produce the same pixels."""
    from jpegsnoop_b200 import BatchDecoder
    monkeypatch.setenv("JSGPU_IDCT_TABLE", str(tab))
    orc = _oracle(True)
    bd = BatchDecoder(huff_kernel=0, idct_kernel=3)
    bd.set_batch([j for _, j in cases]); bd.decode(); bd.sync()
    for i, (name, j) in enumerate(cases):
        assert not JC.compare(orc.decode(j), bd.fetch(i), what=("pix_y", "pix_cb", "pix_cr", "dib")), (name, tab)


def test_host_marker_walk_equals_device_marker_scan(built, cases):
    from jpegsnoop_b200 import BatchDecoder
    jpegs = [j for _, j in cases]
    outs = []
    for dm in (True, False):
        bd = BatchDecoder(idct_kernel=1, device_markers=dm)
        bd.set_batch(jpegs); bd.decode(); bd.sync()
        outs.append([bd.fetch(i) for i in range(len(jpegs))])
    for a, b, (name, _) in zip(outs[0], outs[1], cases):
        assert not JC.compare(a, b, what=("pix_y", "dib", "mcu_map", "dht_histo")), name


def test_unsupported_images_in_a_batch_are_skipped(built, cases):
    """Images the reference's DecodeScanImg would refuse (here: 4-component CMYK scans) occupy no pool space, carry
    status 0x80000000 and do not disturb their neighbours — also at the start of an image range of the pipelined
    host call."""
    import io
    from PIL import Image
    from jpegsnoop_b200 import BatchDecoder
    b = io.BytesIO(); Image.fromarray(JC.synth_rgb(64, 48, 77)).convert("CMYK").save(b, "JPEG", quality=80); cmyk = b.getvalue()
    good = [j for _, j in cases[:6]] * 3                       # 18 decodable images
    jpegs = list(good); names = ["ok"] * len(good)
    for at in (0, 5, 11):
        jpegs.insert(at, cmyk); names.insert(at, "cmyk")
    bd = BatchDecoder(huff_kernel=0, idct_kernel=0)
    tarr, darr, bits = bd.prepare(jpegs)
    bd.set_tables(tarr); bd.plan(darr, bits.size)
    lay = bd.layout
    tot = lambda f, a: sum((f(l) + a - 1) // a * a for l, nm in zip(lay, names) if nm == "ok")
    pix_n = tot(lambda l: int(l.img_x) * int(l.img_y), 64); dib_n = tot(lambda l: int(l.img_x) * int(l.img_y) * 4, 256)
    blk_n = tot(lambda l: int(l.blk_xmax) * int(l.blk_ymax), 64); mcu_n = tot(lambda l: int(l.mcu_xmax) * int(l.mcu_ymax), 32)
    outs = {"pix_y": np.zeros(pix_n, np.int16), "pix_cb": np.zeros(pix_n, np.int16), "pix_cr": np.zeros(pix_n, np.int16),
            "dib": np.zeros(dib_n, np.uint8), "blk_y": np.zeros(blk_n, np.int16), "blk_cb": np.zeros(blk_n, np.int16),
            "blk_cr": np.zeros(blk_n, np.int16), "mcu_map": np.zeros(mcu_n, np.uint32),
            "dht_histo": np.zeros(len(jpegs) * 136, np.uint32), "stats": np.zeros(len(jpegs) * 16, np.int32)}
    bd.decode_host(darr, bits, outs)
    orc = _oracle(True)
    st = [int(l.status) for l in bd.refresh_layout()]
    for i, (nm, j) in enumerate(zip(names, jpegs)):
        if nm == "cmyk":
            assert st[i] == 0x80000000, (i, hex(st[i]))
        else:
            assert st[i] == 0, (i, hex(st[i]))
            assert not JC.compare(orc.decode(j), bd.fetch_host(i, outs), what=("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo")), i
    bd.set_batch(jpegs); bd.decode(); bd.sync()                 # and the device-resident path
    for i, (nm, j) in enumerate(zip(names, jpegs)):
        if nm == "ok":
            assert not JC.compare(orc.decode(j), bd.fetch(i), what=("pix_y", "dib", "mcu_map")), i


def record_reference(orc):
    """What the compiled reference computes for the damaged-scan tests above (tests/golden/make_golden.py stores it)."""
    out = {}
    cases = JC.small_cases()
    ref = orc("ref_fixed")
    for name, (j, ovl) in _damaged_cases(cases).items():
        out[f"damaged/{name}"] = RG.decoded(ref.decode(j, overlays=ovl)); out[f"damaged/{name}/err_lines"] = RG.lines(ref.err_lines())
    ref.close()
    names, jpegs = _damaged_batch(cases)
    for dc_only in (False, True):
        o = orc("ref_fixed", decode_ac=not dc_only)
        for name, j in zip(names, jpegs):
            out[f"damaged_batch/{dc_only}/{name}"] = RG.decoded(o.decode(j))
        o.close()
    return out
