"""TEST INFRASTRUCTURE: seeded test JPEGs made with Pillow/libjpeg-turbo (an encoder independent of
both the reference and this repo), covering the layouts BASELINE.json's configs name."""
import io
import numpy as np
from PIL import Image

import ref_golden as RG


def synth_rgb(W, H, seed):
    """Smooth sinusoid field + N(0,12) noise per channel (SURVEY.md §8d content)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    img = np.stack([128 + 80 * np.sin(xx / 37.0) * np.cos(yy / 23.0),
                    128 + 60 * np.sin(xx / 11.0 + yy / 50.0),
                    128 + 70 * np.cos(yy / 17.0)], -1) + rng.normal(0, 12, (H, W, 3))
    return np.clip(img, 0, 255).astype(np.uint8)


def enc(img, **kw):
    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", **kw)
    return b.getvalue()


def small_cases():
    """(name, jpeg bytes) — small enough that the CPU oracle finishes each in well under a second."""
    return [
        ("444_rst_row_640x480", enc(synth_rgb(640, 480, 1), quality=85, subsampling=0, restart_marker_rows=1)),   # BASELINE config 1
        ("422_opt_dri5", enc(synth_rgb(640, 480, 2), quality=75, subsampling=1, optimize=True, restart_marker_blocks=5)),
        ("420_dri4_1080p", enc(synth_rgb(1920, 1080, 3), quality=85, subsampling=2, restart_marker_blocks=4)),     # one image of config 2
        ("420_norst_odd", enc(synth_rgb(333, 211, 4), quality=92, subsampling=2)),                                # no DRI, ragged size
        ("gray_dri3", enc(synth_rgb(200, 100, 5)[:, :, 0], quality=80, restart_marker_blocks=3)),
        ("444_q100_tiny", enc(synth_rgb(64, 48, 6), quality=100, subsampling=0)),
        ("420_q30_opt_rst2rows", enc(synth_rgb(800, 600, 7), quality=30, subsampling=2, optimize=True, restart_marker_rows=2)),
        ("444_1x1_8px", enc(synth_rgb(8, 8, 8), quality=90, subsampling=0)),
        ("420_dri1", enc(synth_rgb(160, 96, 9), quality=70, subsampling=2, restart_marker_blocks=1)),
        ("420_dri8_4k_strip", enc(synth_rgb(3840, 64, 10), quality=85, subsampling=2, restart_marker_blocks=8)),  # config 3 geometry, 4 MCU rows
    ]


def mini_cases():
    """(name, jpeg bytes) from tests/mini_jpeg.py: what Pillow cannot produce — unusual Huffman code-length
    distributions (large second-level look-up; the lane Huffman kernel must hand these to the warp kernel when
    the second level does not fit its shared-memory copy) and sampling layouts 4:1:1 / 4:4:0."""
    import mini_jpeg as MJ
    ac_big = MJ.long_code_table(MJ.all_ac_symbols(), n11=24)     # ~15 ten-bit prefixes with longer codes: second level > 512 entries
    ac_fit = MJ.long_code_table(MJ.all_ac_symbols(), n11=8)      # fits the staged second level
    return [
        ("mini_longcodes_big_420_dri4", MJ.encode(synth_rgb(320, 176, 21), quality=90, samp=((2, 2), (1, 1), (1, 1)), dri=4, ac_tabs=[ac_big, ac_big])),
        ("mini_longcodes_fit_420_dri2", MJ.encode(synth_rgb(320, 176, 22), quality=90, samp=((2, 2), (1, 1), (1, 1)), dri=2, ac_tabs=[ac_fit, ac_big])),
        ("mini_411_dri3", MJ.encode(synth_rgb(200, 72, 23), quality=75, samp=((4, 1), (1, 1), (1, 1)), dri=3)),
        ("mini_440_nodri", MJ.encode(synth_rgb(120, 88, 24), quality=80, samp=((1, 2), (1, 1), (1, 1)))),
        ("mini_gray_longcodes_nodri", MJ.encode(synth_rgb(136, 64, 25)[:, :, 1], quality=95, ac_tabs=[ac_big, ac_big])),
    ] + [
        # every sampling factor up to 4 is legal for the reference (ImgDecode.cpp:2819-2828): 32x32-pixel MCUs, factors of 3,
        # components with 1 < H < Hmax (tiles larger than the fused IDCT kernel's shared memory go to the literal kernels)
        ("mini_samp_%s" % "_".join("%dx%d" % hv for hv in samp), MJ.encode(synth_rgb(200, 136, 31 + k), quality=80, samp=samp, dri=dri))
        for k, (samp, dri) in enumerate([(((4, 4), (1, 1), (1, 1)), 2), (((4, 4), (2, 4), (1, 4)), 0), (((1, 3), (1, 1), (1, 1)), 3),
                                          (((3, 1), (1, 1), (1, 1)), 2), (((2, 3), (1, 1), (1, 1)), 0), (((4, 2), (2, 2), (1, 1)), 5),
                                          (((2, 4), (2, 2), (2, 1)), 1)])
    ]


def long_cases():
    """(name, jpeg bytes): long restart intervals — scans without restart markers (BASELINE config 5) or with a DRI of
    whole MCU rows — which take the self-synchronising Huffman passes, plus one full 4K frame with DRI = 8 (config 3)."""
    import mini_jpeg as MJ
    ac_fit = MJ.long_code_table(MJ.all_ac_symbols(), n11=8)
    return [
        ("420_norst_4k", enc(synth_rgb(3840, 2160, 41), quality=85, subsampling=2)),                              # one image of config 5
        ("420_dri8_4k", enc(synth_rgb(3840, 2160, 42), quality=85, subsampling=2, restart_marker_blocks=8)),      # one image of config 3
        ("444_norst_640x480", enc(synth_rgb(640, 480, 43), quality=90, subsampling=0)),
        ("422_opt_norst_800x600", enc(synth_rgb(800, 600, 44), quality=60, subsampling=1, optimize=True)),
        ("gray_norst_1024x768_q30", enc(synth_rgb(1024, 768, 45)[:, :, 0], quality=30)),
        ("420_rst2rows_1080p", enc(synth_rgb(1920, 1080, 46), quality=80, subsampling=2, restart_marker_rows=2)),
        ("420_norst_flat", enc(np.full((480, 640, 3), 128, np.uint8), quality=85, subsampling=2)),                # hundreds of MCUs per slot
        ("mini_longcodes_fit_420_norst", MJ.encode(synth_rgb(320, 176, 47), quality=90, samp=((2, 2), (1, 1), (1, 1)), ac_tabs=[ac_fit, ac_fit])),
        ("mini_411_norst_shared_tables", MJ.encode(synth_rgb(400, 304, 48), quality=75, samp=((4, 1), (1, 1), (1, 1)))),   # block phase not observable: settles through k_ph_fix_cta
        ("444_q100_noise_norst", enc(np.random.default_rng(7).integers(0, 256, (96, 128, 3)).astype(np.uint8), quality=100, subsampling=0)),
    ]


def compare(a, b, what=("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo", "stats")):
    """Bit-exact comparison of two Decoded-like objects; returns list of mismatching field names.  The arrays of `a` may be
    stored reference results (tests/ref_golden.py: values or digests)."""
    bad = []

    def eq(x, y):
        if isinstance(x, str):
            return y is not None and RG.same(x, y)
        if x is None and y is None:
            return True
        if x is None or y is None:
            return False
        return np.array_equal(np.asarray(x), np.asarray(y))
    for f in what:
        if f == "blk_dc":
            if not all(eq(p, q) for p, q in zip(a.blk_dc, b.blk_dc)):
                bad.append(f)
        elif f == "stats":
            if not eq(np.asarray(a.stats)[:11], np.asarray(b.stats)[:11]):
                bad.append(f)
        elif f == "mcu_map":
            if not mcu_map_ok(a.mcu_map, b.mcu_map):
                bad.append(f)
        elif not eq(getattr(a, f), getattr(b, f)):
            bad.append(f)
    return bad


def mcu_map_ok(want, got):
    """MCU file map comparison: exact.  (Round 1 accepted one documented deviation here — the stale byte position the
    reference reports after an interval was consumed to its last bit by a read that stepped over two byte boundaries;
    k_finalize_mcumap_emptied now reproduces it.)"""
    if isinstance(want, str):
        return RG.same(want, got)
    want = np.asarray(want); got = np.asarray(got)
    return want.shape == got.shape and bool(np.array_equal(want, got))
