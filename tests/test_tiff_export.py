"""Export-to-TIFF consumer (SURVEY.md §8f N4): the file writer against the reference's own FileTiff.cpp (compiled in place
into oracle/_ref), and — on the GPU — the device-packed sample arrays + complete files against
CJPEGsnoopDoc::OnToolsExporttiff's loops (JPEGsnoopDoc.cpp:2098-2170, restated in oracle/ref_harness.cpp).  The reference's
files are stored as their length, first 64 bytes and digest (tests/golden/ref_outputs.json.gz, recorded by
record_reference below)."""
import ctypes as C
import os

import numpy as np
import pytest

import jpeg_cases as JC
import ref_golden as RG

MODES = [(0, 0), (0, 1), (1, 0)]
SIZES = [(8, 8), (640, 480), (1920, 1088), (3840, 2160), (70000, 2)]


def _file(path, tail=None):
    """A TIFF file in stored form; tail: digest of its last `tail` bytes too (the sample array)."""
    b = np.fromfile(path, np.uint8)
    r = {"len": int(b.size), "head": b[:64].tobytes().hex(), "digest": RG.digest(b)}
    if tail is not None:
        r["tail"] = RG.digest(b[b.size - tail:])
    return r


def _data(size, b16):
    w, h = size
    return np.random.default_rng(w * 31 + h).integers(0, 256, w * h * (6 if b16 else 3), dtype=np.uint8)


@pytest.mark.parametrize("mode", MODES, ids=["rgb8", "rgb16", "ycc8"])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_tiff_file_equals_the_references(built, tmp_path, mode, size):
    """Header, IFD (dimensions and strip offset are SHORTs there: 70000 columns wrap like the reference's), out-of-line values
    and sample data, byte for byte."""
    from jpegsnoop_b200 import _lib
    L = _lib.load()
    ycc, b16 = mode; w, h = size
    data = _data(size, b16)
    b = str(tmp_path / "new.tif")
    assert L.jsimg_tiff_write(b.encode(), ycc, b16, data.ctypes.data, w, h) == 1
    want, got = RG.get(f"tiff/{mode}/{size}"), _file(b)
    assert want["len"] > data.size and want == got, (want["len"], got["len"], want["head"], got["head"])


@pytest.mark.gpu
def test_exported_tiffs_match_the_reference(built, tmp_path):
    from jpegsnoop_b200 import CimgDecode, BatchDecoder
    cases = JC.small_cases()
    dec = CimgDecode()
    bd = BatchDecoder(); bd.set_batch([j for _, j in cases]); bd.decode(); bd.sync()
    for i, (name, j) in enumerate(cases):
        got = dec.decode(j)
        assert not JC.compare(RG.get_decoded(f"export/{name}"), got), name
        three = got.pix_cb is not None
        for mode in (0, 1, 2):
            b = str(tmp_path / f"new{mode}.tif")
            if os.path.exists(b):
                os.remove(b)
            want = RG.get(f"export/{name}/{mode}")
            ok_new = dec.ExportTiff(b, mode)
            assert (want is not None) == ok_new == (three or mode != 2), (name, mode, want is not None, ok_new)
            if not ok_new:
                continue
            gb = _file(b)
            assert {k: want[k] for k in gb} == gb, (name, mode, want["len"], gb["len"])
            # the batch entry point hands out the same sample array
            arr = bd.export(i, mode)
            assert RG.digest(arr) == want["tail"], (name, mode)
    # the export follows the preview the DIB shows (the reference reads m_pDibTemp, whatever mode painted it)
    name, j = cases[0]
    dec.decode(j)
    dec.SetPreviewMode(6)
    b = str(tmp_path / "new_y.tif")
    assert dec.ExportTiff(b, 0)
    assert RG.get("export/luma_preview") == _file(b)


def record_reference(orc):
    """What the compiled reference writes for the tests above (tests/golden/make_golden.py stores it)."""
    import tempfile
    out = {}
    ref = orc("ref_fixed")
    ref.lib.ref_tiff_write.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_uint, C.c_uint]
    ref.lib.ref_export_tiff.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    with tempfile.TemporaryDirectory() as tmp:
        a = os.path.join(tmp, "ref.tif")
        for mode in MODES:
            for size in SIZES:
                data = _data(size, mode[1])
                ref.lib.ref_tiff_write(a.encode(), mode[0], mode[1], data.ctypes.data, size[0], size[1])
                out[f"tiff/{mode}/{size}"] = _file(a)
        for name, j in JC.small_cases():
            d = ref.decode(j)
            out[f"export/{name}"] = RG.decoded(d)
            for mode in (0, 1, 2):
                if os.path.exists(a):
                    os.remove(a)
                ok = ref.lib.ref_export_tiff(ref.ctx, a.encode(), mode)
                npix = int(d.geom[6]) * int(d.geom[7])
                out[f"export/{name}/{mode}"] = _file(a, npix * (6 if mode == 1 else 3)) if ok else None
        name, j = JC.small_cases()[0]
        ref.decode(j)
        ref.set_preview_mode(6)
        ref.lib.ref_export_tiff(ref.ctx, a.encode(), 0)
        out["export/luma_preview"] = _file(a)
        ref.set_preview_mode(1)
    ref.close()
    return out
