"""Generates the golden fixtures under tests/golden/ by running the COMPILED REFERENCE
(oracle/_ref/liboracle_ref_{fixed,float}.so = /root/reference/source/ImgDecode.cpp built unmodified)
on small seeded JPEGs.  Run in the build container (needs /root/reference); the .npz files it
writes are committed so the oracle port and the CUDA path can be checked where the reference is
absent.  It also stores, in ref_outputs.json.gz, what the compiled reference computes for the tests that compare with it
(record_reference() of each module in REF_MODULES).
Usage: python tests/golden/make_golden.py [ref_outputs]     (ref_outputs: only ref_outputs.json.gz)
"""
import io
import os
import sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle_util import Oracle, build_oracles      # noqa: E402
import jpeg_cases as JC                            # noqa: E402
import ref_golden as RG                            # noqa: E402

REF_MODULES = ("test_oracle", "test_gpu_parity", "test_gpu_preview", "test_gpu_detail", "test_tiff_export")


def fixtures():
    from jpegsnoop_b200 import synth
    yield "synth_444_64x48_rstrow", synth.encode(64, 48, "444", 85, 8, False, seed=11)
    yield "synth_420_48x32_dri2", synth.encode(48, 32, "420", 75, 2, False, seed=12)
    yield "synth_422_40x24_opt_dri1", synth.encode(40, 24, "422", 60, 1, True, seed=13)
    yield "synth_gray_33x17_dri3", synth.encode(33, 17, "gray", 90, 3, True, seed=14)
    yield "synth_420_96x64_norst", synth.encode(96, 64, "420", 92, 0, False, seed=15)
    yield "pil_420_50x38_q30_opt", JC.enc(JC.synth_rgb(50, 38, 16), quality=30, subsampling=2, optimize=True, restart_marker_blocks=3)
    yield "pil_444_24x16_q100", JC.enc(JC.synth_rgb(24, 16, 17), quality=100, subsampling=0)


def main():
    build_oracles()
    fx = Oracle("ref_fixed"); fl = Oracle("ref_float")
    lf, li = fx.idct_tables()
    np.savez_compressed(os.path.join(HERE, "idct_tables.npz"), lf=lf, li=li)
    for name, j in fixtures():
        a = fx.decode(j); b = fl.decode(j)
        assert a.nerr == 0 and b.nerr == 0, name
        d = dict(jpeg=np.frombuffer(j, np.uint8), geom=a.geom, mcu_map=a.mcu_map, dht_histo=a.dht_histo, stats_fixed=a.stats, stats_float=b.stats)
        for tag, r in (("fixed", a), ("float", b)):
            d[f"pix_y_{tag}"] = r.pix_y; d[f"dib_{tag}"] = r.dib
            if r.pix_cb is not None:
                d[f"pix_cb_{tag}"] = r.pix_cb; d[f"pix_cr_{tag}"] = r.pix_cr
        for c, arr in enumerate(a.blk_dc):
            if arr is not None:
                d[f"blk_dc{c}"] = arr
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **d)
        print(name, len(j), "bytes ->", os.path.getsize(os.path.join(HERE, name + ".npz")), "bytes npz")


def ref_outputs():
    import importlib
    build_oracles()
    out = {}
    for m in REF_MODULES:
        rec = importlib.import_module(m).record_reference(Oracle)
        assert not set(rec) & set(out), m
        out.update(rec)
    RG.save(out)
    print(len(out), "entries ->", os.path.getsize(RG.PATH), "bytes", RG.PATH)


if __name__ == "__main__":
    if sys.argv[1:] != ["ref_outputs"]:
        main()
    ref_outputs()
