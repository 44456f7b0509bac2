#!/usr/bin/env python
"""bench.py — MPixels/s decoded, bit-exact vs the reference, on BASELINE.json's configs.

  python bench.py --gpus N --steps K --warmup W          our arm (one rank per GPU, torchrun for N>1)
  python bench.py --impl reference --steps K --warmup W  the reference's CPU DecodeScanImg on the host cores

Headline (`value`, `roofline`, `e2e`, `cpu_baseline`) = BASELINE configs[1]: batch=1024 1920x1080 4:2:0, RST interval = 4
MCUs, per B200 (weak scaling).  The same JSON line carries a `configs` array with the other BASELINE configs measured the
same way (device-resident MPix/s, stage times, K2 roofline fraction, bit-exact flag): configs[0] (one 640x480 4:4:4
image), configs[2] as its per-GPU shard (512 x 4K 4:2:0, DRI = 8 — at N = 8 that is the whole config), configs[3] (mixed
sampling / per-image DQT+DHT, 512 images per GPU) and configs[4] (512 x 4K, NO restart markers).

A "step" = one pass of the hot path over the whole batch: marker scan -> unstuff -> Huffman -> dequant/IDCT/upsample/
colour -> maps/statistics, i.e. everything CimgDecode::DecodeScanImg does (ImgDecode.cpp:2723-3745), for every image.
  value : SOF pixels (X*Y, not padded) of all ranks / device time, inputs resident in HBM.
  e2e   : same metric through the one-call C-ABI jsgpu_decode_batch_host: pinned host bitstream in, every reference
          output (Y/Cb/Cr int16 maps, BGRA DIB, block-DC maps, MCU map, histo, stats) back in pinned host memory,
          H2D and D2H inside the timed region.
  bit-exactness: EVERY image of EVERY rank — checksums of all output buffers computed on the device
          (jsgpu_batch_checksums) against the same checksums of the compiled reference's CPU decode of the same image
          (oracle/_ref, ref_bench_ck); the mismatch count is all-reduced.  That CPU pass is also the `cpu_baseline`.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True                     # the tree may be read-only
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CONFIGS = {
    # name: (BASELINE configs index, images per GPU, description)
    "cfg1": (0, 1, "single 640x480 4:4:4 baseline JPEG, RST every MCU row"),
    "cfg2": (1, 1024, "batch=1024 1920x1080 4:2:0 baseline, q85, RST interval=4 MCUs"),
    "cfg3shard": (2, 512, "batch=512 per GPU of 3840x2160 4:2:0 baseline, q85, RST interval=8 MCUs (BASELINE configs[2] image-sharded: 4096 images at 8 GPUs)"),
    "cfg4": (3, 512, "batch=512 per GPU (2048 at 4 GPUs), mixed 4:2:0/4:2:2/4:4:4, sizes 1080p/720p/4K, q50..95 and optimised DHT per image, DRI in {MCU row,4,8,16}"),
    "cfg5": (4, 512, "batch=512 3840x2160 4:2:0 baseline, q85, NO restart markers (one serial segment per image)"),
    # the same images as cfg2 decoded with the reference's DEFAULT build arithmetic (float IDCT, ImgDecode.cpp:2372-2392), verified
    # against the float-IDCT build of the compiled reference
    "cfg2float": (1, 1024, "batch=1024 1920x1080 4:2:0 baseline, q85, RST interval=4 MCUs, FLOAT-IDCT arithmetic (the reference's shipping default build)"),
}
METRIC = "MPixels/s decoded (bit-exact vs ref)"
UNIT = "MPix/s"
BPP = {"420": 13.0, "422": 14.0, "444": 16.0, "gray": 8.0}


def specs_for(cfg, rank, nimg=None):
    """Seeded specs of this rank's images (SURVEY.md §8d: seed = 1234 + cfg*1000 + global image index)."""
    idx, batch, _ = CONFIGS[cfg]
    if nimg is not None:
        batch = nimg
    num = idx + 1
    out = []
    for i in range(batch):
        g = rank * batch + i
        seed = 1234 + num * 1000 + g
        if cfg == "cfg1":
            s = dict(width=640, height=480, subsampling="444", quality=85, restart_interval=80, optimize=False)
        elif cfg in ("cfg2", "cfg2float"):
            s = dict(width=1920, height=1080, subsampling="420", quality=85, restart_interval=4, optimize=False)
        elif cfg == "cfg3shard":
            s = dict(width=3840, height=2160, subsampling="420", quality=85, restart_interval=8, optimize=False)
        elif cfg == "cfg5":
            s = dict(width=3840, height=2160, subsampling="420", quality=85, restart_interval=0, optimize=False)
        else:   # cfg4
            ss = ("420", "422", "444")[g % 3]
            w, h = ((1920, 1080), (1280, 720), (3840, 2160))[(g // 3) % 3]
            mcu_w = 8 if ss == "444" else 16
            row = (w + mcu_w - 1) // mcu_w
            ri = (row, 4, 8, 16)[(g // 9) % 4]
            q = 50 + (seed * 2654435761 >> 7) % 46
            s = dict(width=w, height=h, subsampling=ss, quality=int(q), restart_interval=ri, optimize=True)
        s["seed"] = seed
        out.append(s)
    return out


def make_batch(cfg, rank, nimg=None):
    from jpegsnoop_b200 import synth
    specs = specs_for(cfg, rank, nimg)
    buf, offs = synth.encode_batch(specs)
    return [buf[int(offs[i]):int(offs[i + 1])] for i in range(len(specs))], specs


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []; self.p = None; self.index = index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.p:
            self.p.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # median of the upper half = clocks under load (idle samples before/after drag the plain median down)
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": (load[len(load) // 2] if load else None), "sm_max_mhz": (max(mx) if mx else None),
                "reasons": sorted(reasons), "samples": len(sm)}


def load_oracle(fixed=True):
    """The compiled reference (oracle/_ref; integer-IDCT build unless fixed=False) when present, else the C port (spot checks only)."""
    from oracle_util import Oracle, ref_available
    if ref_available("fixed" if fixed else "float"):
        return Oracle("ref_fixed" if fixed else "ref_float"), "reference"
    return Oracle("port", idct_fixed=fixed), "port"


def verify_all(bd, jpegs, orc, kind, threads, max_images=None):
    """Checksums of every output buffer of every image: device vs the reference's CPU decode.
    Returns (images checked, images that differ, cpu wall seconds, cpu error lines)."""
    import numpy as np
    n = len(jpegs)
    if kind != "reference":                # no compiled reference here: full-buffer comparison of a few images against the port
        import jpeg_cases as JC
        WHAT = ("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo")
        pick = sorted(set([0, n // 3, (2 * n) // 3, n - 1])); t0 = time.time(); bad = 0
        for i in pick:
            bad += 1 if JC.compare(orc.decode(bytes(jpegs[i])), bd.fetch(i), what=WHAT) else 0
        return len(pick), bad, time.time() - t0, 0
    sel = list(range(n))
    if max_images is not None and max_images < n:
        stride = n / float(max_images)
        sel = sorted(set(int(k * stride) for k in range(max_images)))
    gck = bd.checksums()
    t, errs, cck = orc.bench_ck([jpegs[i] for i in sel], threads=threads)
    g = gck[sel]
    cols = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 11]
    diff = (g[:, cols] != cck[:, cols]).any(axis=1) | (g[:, 10] != 0) | (cck[:, 10] != 0)
    return len(sel), int(diff.sum()), t, errs


def dump_outputs(bd, out_dir, max_images=16, max_elems=1 << 20):
    """What the last timed step left for the caller, as out_dir/<name>.npy: every output buffer (BatchDecoder.fetch) of a fixed,
    seeded sample of images, concatenated in image order, and of a concatenation longer than max_elems a fixed, seeded sample
    of elements.  float32, or float64 for 32-bit integers.  The inputs are seeded too, so two builds compare output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(20261017)
    imgs = np.arange(bd.n) if bd.n <= max_images else np.sort(rng.choice(bd.n, max_images, replace=False))
    cols = {}
    for i in imgs:
        d = bd.fetch(int(i))
        for name, a in (("geom", d.geom), ("pix_y", d.pix_y), ("pix_cb", d.pix_cb), ("pix_cr", d.pix_cr), ("dib", d.dib), ("mcu_map", d.mcu_map),
                        ("blk_dc_y", d.blk_dc[0]), ("blk_dc_cb", d.blk_dc[1]), ("blk_dc_cr", d.blk_dc[2]), ("dht_histo", d.dht_histo),
                        ("stats", d.stats)):
            if a is not None:
                cols.setdefault(name, []).append(np.asarray(a).ravel())
    np.save(os.path.join(out_dir, "image_index.npy"), imgs.astype(np.float64))
    for name, parts in cols.items():
        a = np.concatenate(parts)
        if a.size > max_elems:
            a = a[np.sort(rng.integers(0, a.size, max_elems))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype.itemsize >= 4 else np.float32))


def algorithmic_bytes_stage_b(specs, bd):
    """SURVEY.md §8d: 2 B x samples + 6 B maps + 4 B BGRA per PADDED pixel, per image by its sampling."""
    tot = 0.0
    for s, l in zip(specs, bd.layout):
        tot += float(int(l.img_x) * int(l.img_y)) * BPP[s["subsampling"]]
    return tot


def run_config(cfg, args, env, orc, kind, threads, steps, warmup, verify_budget_s=None, cpu_rate_hint=None):
    """Generate this rank's shard of `cfg`, decode it device-resident `steps` times, verify every image.
    Returns (record for the JSON line, BatchDecoder, jpegs, specs, context) — caller closes the decoder."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from jpegsnoop_b200 import BatchDecoder
    rank, world, local = env
    t0 = time.time()
    jpegs, specs = make_batch(cfg, rank, nimg=args.batch if cfg == args.config else (args.side_batch if cfg != "cfg1" else None))
    t_gen = time.time() - t0
    if cfg == "cfg2float":
        orc, kind = load_oracle(fixed=False)
    bd = BatchDecoder(device=local, idct_fixedpt=(cfg != "cfg2float"), huff_kernel=args.huff_kernel, idct_kernel=args.idct_kernel,
                      want_histo=not args.no_histo, want_mcu_map=not args.no_mcu_map)
    tarr, darr, bits = BatchDecoder.prepare(jpegs)
    shared_tables = cfg != "cfg4"
    if world > 1 and shared_tables:      # shared Huffman/quant tables: ONE broadcast of rank 0's table blob over NCCL (NVLink)
        from jpegsnoop_b200.shard import broadcast_tables
        tarr = broadcast_tables(tarr, src=0, device=torch.device("cuda", local))
    bd.set_tables(tarr)
    bd.plan(darr, bits.size)
    bd.upload(bits); bd.sync()
    for _ in range(warmup):
        bd.decode()
    bd.sync()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    bd.timer_start()
    for _ in range(steps):
        bd.decode()
    ms_total = bd.timer_stop()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    stage_ms = bd.stage_ms()
    launches = bd.launches()
    status = sorted(set(int(l.status) for l in bd.refresh_layout()))
    try:
        ss_info = bd.selfsync_info()
    except Exception:
        ss_info = None
    if cfg == args.config and args.dump_outputs and rank == 0:
        dump_outputs(bd, args.dump_outputs)
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    npx = torch.tensor([float(bd.nsof_pixels)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(npx, op=dist.ReduceOp.SUM)
    ms_max = float(t.item()); total_px = float(npx.item())
    value = total_px * steps / (ms_max / 1e3) / 1e6
    # ---- verification of every image of this rank (bounded only when a slow host would blow the time budget) ----------
    max_images = None
    if verify_budget_s is not None and cpu_rate_hint:
        est = bd.nsof_pixels / 1e6 / cpu_rate_hint
        if est > verify_budget_s:
            max_images = max(8, int(len(jpegs) * verify_budget_s / est))
    if args.no_cpu:
        max_images = 4
    nchk, nbad, cpu_s, cpu_errs = verify_all(bd, jpegs, orc, kind, threads, max_images)
    v = torch.tensor([float(nchk), float(nbad), float(len(jpegs))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(v, op=dist.ReduceOp.SUM)
    checked_all, bad_all, nimg_all = int(v[0].item()), int(v[1].item()), int(v[2].item())
    cpu_px = bd.nsof_pixels * (nchk / float(len(jpegs)))
    alg_b = algorithmic_bytes_stage_b(specs, bd)
    peak = env_peak()[0]
    idct_ms = float(stage_ms[2])
    rec = {"name": cfg, "baseline_config_index": CONFIGS[cfg][0], "workload": CONFIGS[cfg][2], "images_per_gpu": len(jpegs),
           "value": round(value, 1), "unit": UNIT, "ms_per_step": round(ms_max / steps, 3), "steps": steps,
           "stage_ms": {"marker_scan+unstuff": round(float(stage_ms[0]), 3), "huffman": round(float(stage_ms[1]), 3),
                        "idct+colour": round(idct_ms, 3), "finalize": round(float(stage_ms[3]), 3), "step_total": round(float(stage_ms[4]), 3)},
           "k2_frac_of_hbm_peak": round(alg_b / (idct_ms / 1e3) / 1e9 / peak, 4) if idct_ms > 0 else None,
           "bitstream_bytes_per_padded_px": round(bits.size / float(bd.npadded_pixels), 4),
           "idct": "float (reference default build)" if cfg == "cfg2float" else "integer (-DIDCT_FIXEDPT build)",
           "bit_exact": bad_all == 0 and checked_all > 0, "bit_exact_checked_images": checked_all, "images_all_ranks": nimg_all,
           "mismatching_images": bad_all, "checked_by": "device checksums of all output buffers vs " + ("oracle/_ref (compiled reference) checksums" if kind == "reference" else "C port, spot check"),
           "decoder_status_words": status, "gpu_launches_per_step": launches, "gen_s": round(t_gen, 1),
           "cpu_reference_mpix_s": round(cpu_px / cpu_s / 1e6, 2) if cpu_s > 0 else None, "cpu_threads": threads, "cpu_err_lines": cpu_errs}
    if cfg == args.config:
        # K2 with the device to itself: in the product the MCU-file-map kernels run on a second stream NEXT TO it (the step is
        # shorter, K2's own span a little longer); without the map they are not launched.  Outside the timed region.
        try:
            bd.set_options(want_mcu_map=0)
            for _ in range(3):
                bd.decode()
            bd.sync()
            rec["k2_alone_ms"] = round(float(bd.stage_ms()[2]), 3)
            bd.set_options(want_mcu_map=1); bd.decode(); bd.sync()
        except Exception as e:
            rec["k2_alone_ms"] = None; rec["k2_alone_error"] = str(e)[:200]
    if cfg == "cfg2" and not getattr(args, "no_preview", False):
        # the channel-preview pass (SURVEY §8f N3/N4) over the resident batch, after the verification above: histogram/clip
        # statistics conversion, then a plain luminance preview; 6 B read + 4 B written per padded pixel
        try:
            pv = {}
            for key, kw in (("histogram+clip_stats", dict(hist_en=1)), ("luminance_preview", dict(mode=6))):
                bd.preview(**kw); bd.sync()
                bd.timer_start(); bd.preview(**kw); ms = bd.timer_stop()
                pv[key] = {"ms": round(ms, 3), "gbs": round(10.0 * bd.npadded_pixels / (ms / 1e3) / 1e9, 1)}
                if kw.get("hist_en"):
                    pv[key]["image0_pixels_counted"] = int(bd.colour_stats(0).count)
            bd.preview(); bd.sync()                                   # back to the default RGB DIB
            rec["preview_pass"] = pv
        except Exception as e:                                        # a side figure: never fail the headline over it
            rec["preview_pass"] = {"error": str(e)[:200]}
    if ss_info and ss_info[0]:
        rec["selfsync"] = {"images": ss_info[0], "slots": ss_info[1], "slots_changed_per_fix_round": ss_info[2]}
    ctx = {"bits": bits, "darr": darr, "ms_max": ms_max, "total_px": total_px, "stage_ms": stage_ms, "alg_b": alg_b, "cpu_s": cpu_s, "cpu_px": cpu_px,
           "launches": launches, "nchk": nchk}
    return rec, bd, jpegs, specs, ctx


_PEAK = None


def env_peak():
    global _PEAK
    if _PEAK is None:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        _PEAK = (float(peaks.get("hbm_gbs", 6650.0)), "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)")
    return _PEAK


def ensure_checker_built():
    """The reference arm must not load the product library: build (if missing) with make, never import/dlopen libjsgpu."""
    need = [os.path.join(ROOT, "jpegsnoop_b200", "libjssynth.so")]
    if not all(os.path.exists(p) for p in need):
        subprocess.run(["make", "-C", os.path.join(ROOT, "jpegsnoop_b200", "csrc"), "../libjssynth.so"], capture_output=True)
    if not os.path.exists(os.path.join(ROOT, "oracle", "liboracle_port.so")) or os.path.isdir("/root/reference"):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "port", "ref"], capture_output=True)


def run_reference(args):
    """The reference's own CPU DecodeScanImg (oracle/_ref, unmodified sources, -DIDCT_FIXEDPT) on the host cores this
    process may really use; every step decodes >= 8 images per thread so that no step ends on one straggler."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    ensure_checker_built()
    from oracle_util import effective_cores
    cores, cinfo = effective_cores()
    nimg = max(8 * cores, 64)
    nimg = min(nimg, CONFIGS[args.config][1]) if args.config != "cfg1" else 64
    jpegs, specs = make_batch(args.config, 0, nimg=nimg)
    npix = sum(s["width"] * s["height"] for s in specs)
    orc, kind = load_oracle()
    sample = [bytes(j) for j in jpegs]
    for _ in range(min(args.warmup, 2)):
        orc.bench(sample[:max(cores, 8)], threads=cores, reps=1)
    tot = 0.0
    for _ in range(args.steps):
        t, errs = orc.bench(sample, threads=cores, reps=1); tot += t
    val = args.steps * npix / tot / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 2), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(tot / args.steps * 1e3, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32 IDCT + f32 colour", "data": "synthetic",
            "config": {"workload": f"{CONFIGS[args.config][2]} (BASELINE configs[{CONFIGS[args.config][0]}]); each step = a bounded sample of "
                                   f"{len(sample)} images of that batch ({len(sample) // cores} per thread)", "host_cpu": cinfo,
                       "generator": "libjssynth.so only; libjsgpu.so is not loaded by this arm"},
            "cpu_baseline": {"value": round(val, 2), "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": f"{len(sample)} images per step, {cores} host threads (effective cores: affinity capped by the cgroup quota), "
                                       f"one CimgDecode per thread, integer-IDCT build"},
            "e2e": {"value": round(val, 2), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def numa_pin(local):
    """Run the calling thread on the cores next to GPU `local` (pinned pages are first-touch local). Returns (old affinity, node)."""
    import torch
    try:
        bus = torch.cuda.get_device_properties(local)
        busid = "%04x:%02x:%02x.0" % (getattr(bus, "pci_domain_id", 0), bus.pci_bus_id, bus.pci_device_id)
        cl = open(f"/sys/bus/pci/devices/{busid}/local_cpulist").read().strip()
        numa = int(open(f"/sys/bus/pci/devices/{busid}/numa_node").read())
        cpus = set()
        for part in cl.split(","):
            a, _, b2 = part.partition("-"); cpus.update(range(int(a), int(b2 or a) + 1))
        if cpus and numa >= 0:
            old = os.sched_getaffinity(0); os.sched_setaffinity(0, cpus & old or old)
            return old, numa
        return None, numa
    except Exception:
        return None, None


def e2e_leg(args, env, bd, jpegs, ctx, orc, kind):
    """jsgpu_decode_batch_host with pinned host buffers, all outputs; the raw D2H ceiling of this box measured next to it
    (all ranks copying at once), and a second, labelled figure for the DIB-only output set."""
    import numpy as np
    import ctypes as C
    import torch
    import torch.distributed as dist
    from jpegsnoop_b200 import _lib as B
    rank, world, local = env
    L = B.load()
    old_aff, numa = numa_pin(local)
    bits, darr = ctx["bits"], ctx["darr"]; nimg = len(jpegs)

    def pinned(nbytes, dtype):
        p = L.jsgpu_host_alloc(int(nbytes))
        if not p:
            return None
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(int(nbytes),)).view(dtype)
    lay = bd.layout
    pix_n = sum((int(l.img_x) * int(l.img_y) + 63) // 64 * 64 for l in lay)
    dib_n = sum((int(l.img_x) * int(l.img_y) * 4 + 255) // 256 * 256 for l in lay)
    blk_n = sum((int(l.blk_xmax) * int(l.blk_ymax) + 63) // 64 * 64 for l in lay)
    mcu_n = sum((int(l.mcu_xmax) * int(l.mcu_ymax) + 31) // 32 * 32 for l in lay)
    outs = {"pix_y": pinned(pix_n * 2, np.int16), "pix_cb": pinned(pix_n * 2, np.int16), "pix_cr": pinned(pix_n * 2, np.int16),
            "dib": pinned(dib_n, np.uint8), "blk_y": pinned(blk_n * 2, np.int16), "blk_cb": pinned(blk_n * 2, np.int16),
            "blk_cr": pinned(blk_n * 2, np.int16), "mcu_map": pinned(mcu_n * 4, np.uint32),
            "dht_histo": pinned(nimg * 136 * 4, np.uint32), "stats": pinned(nimg * 16 * 4, np.int32)}
    hbits = pinned(bits.size, np.uint8)
    if hbits is None or any(v is None for v in outs.values()):
        return {"value": None, "unit": UNIT, "error": "pinned host allocation failed"}
    hbits[:] = bits

    def timed(outset, nsteps):
        bd.decode_host(darr, hbits, outset)            # warm-up (allocations are grow-only)
        if world > 1:
            dist.barrier()
        t1 = time.perf_counter()
        for _ in range(nsteps):
            bd.decode_host(darr, hbits, outset)
        dt = time.perf_counter() - t1
        te = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return float(te.item())
    dt = timed(outs, args.e2e_steps)
    d2h = sum(v.nbytes for v in outs.values())
    e2e = {"value": round(ctx["total_px"] * args.e2e_steps / dt / 1e6, 1), "unit": UNIT,
           "h2d_bytes_per_step": int(bits.size), "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps,
           "what": "jsgpu_decode_batch_host: pinned bitstream -> all reference outputs in pinned host memory "
                   "(8 image ranges, D2H of one overlapping upload+decode of the next)",
           "achieved_d2h_gbs_per_gpu": round(d2h * args.e2e_steps / dt / 1e9, 2)}
    if rank == 0:                                   # the host buffers themselves against the oracle
        import jpeg_cases as JC
        WHAT = ("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "blk_dc", "dht_histo")
        ok = True; picks = sorted(set([0, nimg // 3, (2 * nimg) // 3, nimg - 1]))
        for i in picks:
            ok = ok and not JC.compare(orc.decode(bytes(jpegs[i])), bd.fetch_host(i, outs), what=WHAT)
        e2e["host_buffers_bit_exact_vs_oracle"] = bool(ok); e2e["host_buffers_checked_images"] = picks
    # ---- the box's D2H ceiling: every rank copies 1 GiB device -> pinned host at the same time (plain cudaMemcpyAsync) ----
    try:
        if world > 1:
            dist.barrier()
        rate = bd.host_copy_rate(direction=1, nbytes=1 << 30, reps=3)
        tb = torch.tensor([rate], dtype=torch.float64, device="cuda"); tsum = tb.clone()
        if world > 1:
            dist.all_reduce(tb, op=dist.ReduceOp.MIN); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        e2e["d2h_ceiling_gbs_per_gpu_min_over_ranks"] = round(float(tb.item()), 2)
        e2e["d2h_ceiling_gbs_all_gpus"] = round(float(tsum.item()), 2)
        e2e["frac_of_d2h_ceiling"] = round(e2e["achieved_d2h_gbs_per_gpu"] / float(tb.item()), 3)
        e2e["limiter"] = ("PCIe device->host copy of the reference's outputs (10.2 B per padded pixel); the ceiling is this box's measured "
                          "cudaMemcpyAsync D2H rate into pinned memory with all ranks copying at once (jsgpu_host_copy_rate)")
    except Exception as ex:
        e2e["d2h_ceiling_error"] = str(ex)[:200]
    # ---- DIB-only output set (what a viewer needs): labelled, not the headline -------------------------------------------
    try:
        dt2 = timed({"dib": outs["dib"], "stats": outs["stats"]}, args.e2e_steps)
        e2e["dib_only"] = {"value": round(ctx["total_px"] * args.e2e_steps / dt2 / 1e6, 1), "unit": UNIT,
                           "d2h_bytes_per_step": int(outs["dib"].nbytes + outs["stats"].nbytes), "note": "BGRA DIB + scalar stats only; NOT the headline e2e"}
    except Exception as ex:
        e2e["dib_only"] = {"error": str(ex)[:200]}
    numas = [None] * world
    if world > 1:
        dist.all_gather_object(numas, numa)
    else:
        numas = [numa]
    e2e["host_numa_node_per_rank"] = numas
    if old_aff is not None:
        os.sched_setaffinity(0, old_aff)
    for v in list(outs.values()) + [hbits]:
        L.jsgpu_host_free(C.c_void_p(v.ctypes.data))
    return e2e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=list(CONFIGS), help="headline workload (default: BASELINE configs[1])")
    ap.add_argument("--configs", default="auto", help="other BASELINE configs reported in the `configs` array: auto | none | comma list")
    ap.add_argument("--batch", type=int, default=None, help="override images per GPU of the headline config (debug only; invalidates the headline)")
    ap.add_argument("--side-batch", type=int, default=None, help="override images per GPU of the non-headline configs (debug only)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="debug: verify 4 images only instead of the whole batch")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--side-steps", type=int, default=5, help="timed steps of the non-headline configs")
    ap.add_argument("--verify-seconds", type=float, default=45.0, help="CPU budget per non-headline config; a slower host verifies a strided subset and says so")
    ap.add_argument("--no-histo", action="store_true", help="debug: skip m_anDhtHisto (invalidates the headline)")
    ap.add_argument("--no-mcu-map", action="store_true", help="debug: skip m_pMcuFileMap (invalidates the headline)")
    ap.add_argument("--huff-kernel", type=int, default=0)
    ap.add_argument("--idct-kernel", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline config computed to DIR/<name>.npy (a seeded sample, < 64 MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the decode path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        from jpegsnoop_b200 import _lib
        _lib.load()                                # what build() made: this script compiles nothing and writes nothing in the tree
    if world > 1:
        dist.barrier()
    env = (rank, world, local)
    from oracle_util import effective_cores
    cores, cinfo = effective_cores()
    threads = max(1, cores // world)               # the ranks share the host
    orc, kind = load_oracle()

    # ---- headline ----------------------------------------------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start(); time.sleep(0.3)
    head, bd, jpegs, specs, ctx = run_config(args.config, args, env, orc, kind, threads, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    cpu_rate = (ctx["cpu_px"] / ctx["cpu_s"] / 1e6) if ctx["cpu_s"] > 0 else None
    e2e = None
    if not args.no_e2e:
        e2e = e2e_leg(args, env, bd, jpegs, ctx, orc, kind)
    # extras for the cpu_baseline object (rank 0, N=1): one thread, and the float-IDCT build
    cb = None
    if rank == 0:
        cb = {"value": head["cpu_reference_mpix_s"], "unit": UNIT, "cores": threads, "kind": kind,
              "sample": f"{ctx['nchk']} images of rank 0's batch (the same pass that verifies them), {threads} threads, one CimgDecode per thread, "
                        f"integer-IDCT build, {ctx['cpu_s']:.2f} s wall", "err_lines": head["cpu_err_lines"], "host_cpu": cinfo}
        if world == 1 and kind == "reference":
            try:
                from oracle_util import Oracle, ref_available
                k1 = [bytes(j) for j in jpegs[:max(1, min(len(jpegs), 8))]]
                t1, _ = orc.bench(k1, threads=1, reps=1)
                cb["one_thread_value"] = round(sum(s["width"] * s["height"] for s in specs[:len(k1)]) / t1 / 1e6, 2)
                if ref_available("float"):
                    of = Oracle("ref_float"); kf = [bytes(j) for j in jpegs[:max(threads * 2, 16)]]
                    tf, _ = of.bench(kf, threads=threads, reps=1)
                    cb["float_idct_build_value"] = round(sum(s["width"] * s["height"] for s in specs[:len(kf)]) / tf / 1e6, 2)
            except Exception as ex:
                cb["extras_error"] = str(ex)[:200]
    bits_size = int(ctx["bits"].size); npad = bd.npadded_pixels
    bd.close(); del bd, jpegs

    # ---- the other BASELINE configs ------------------------------------------------------------------------------------
    if args.configs == "auto":
        side = {1: ["cfg1", "cfg5", "cfg3shard", "cfg4", "cfg2float"], 2: ["cfg3shard"], 4: ["cfg3shard", "cfg4"], 8: ["cfg3shard"]}.get(world, ["cfg3shard"])
    elif args.configs in ("none", ""):
        side = []
    else:
        side = [c for c in args.configs.split(",") if c in CONFIGS]
    side = [c for c in side if c != args.config]
    side_recs = []
    for c in side:
        try:
            rec, bd2, j2, s2, _ = run_config(c, args, env, orc, kind, threads, args.side_steps, 2, verify_budget_s=args.verify_seconds, cpu_rate_hint=cpu_rate)
            bd2.close(); del bd2, j2
            side_recs.append(rec)
        except Exception as ex:                     # a failing side config must not take the headline down with it
            side_recs.append({"name": c, "error": str(ex)[:300]})

    # ---- roofline of the dominant kernel (rank 0) ------------------------------------------------------------------------
    if rank == 0:
        peak, peak_src = env_peak()
        sm = ctx["stage_ms"]; idct_ms = float(sm[2]); huff_ms = float(sm[1])
        ach = ctx["alg_b"] / (idct_ms / 1e3) / 1e9
        bpp_img = ctx["alg_b"] / float(npad)
        huff_gbs = (bits_size + npad * (bpp_img - 10.0)) / (huff_ms / 1e3) / 1e9      # bitstream read + coefficient rows written
        traffic = None; traffic_rw = None       # DRAM bytes of one K2 launch from the committed ncu capture of this workload (GB), if there is one
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.config)
            if tj and args.batch is None:
                traffic = round(tj["dram_read_gb"] + tj["dram_write_gb"], 3); traffic_rw = (tj["dram_read_gb"], tj["dram_write_gb"])
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": "k_idct_tile (dequant+IDCT+upsample+YCC->BGRA, stage B)", "achieved": round(ach, 1), "peak": peak,
                "unit": "GB/s", "frac": round(ach / peak, 4), "traffic": traffic, "traffic_unit": "GB per launch (algorithmic: %.3f)" % (ctx["alg_b"] / 1e9),
                "traffic_source": "profiles/traffic.json (ncu --set full capture of this workload, see profiles/README.md)", "peak_source": peak_src,
                "algorithmic_bytes_per_padded_px": round(bpp_img, 3), "ms_per_launch": round(idct_ms, 3),
                "stage_ms": head["stage_ms"], "huffman_achieved_gbs": round(huff_gbs, 1),
                "whole_step_frac_of_hbm_peak": round((bits_size + npad * (bpp_img - 10.0) + ctx["alg_b"]) / (float(sm[4]) / 1e3) / 1e9 / peak, 4)}
        if head.get("k2_alone_ms"):
            roof["ms_per_launch_kernel_alone"] = head["k2_alone_ms"]
            roof["frac_kernel_alone"] = round(ctx["alg_b"] / (head["k2_alone_ms"] / 1e3) / 1e9 / peak, 4)
            roof["note"] = ("`frac` is K2's span inside the timed steps, where the MCU-file-map kernels share the device with it on a second stream; "
                            "`frac_kernel_alone` is the same kernel without them (want_mcu_map=0, measured after the timed region)")
        if traffic_rw:        # SURVEY.md §8(d): read-only and write-only rates of the same launch
            roof["dram_read_gbs"] = round(traffic_rw[0] / (idct_ms / 1e3), 1); roof["dram_write_gbs"] = round(traffic_rw[1] / (idct_ms / 1e3), 1)
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int32 IDCT + f32 colour (int16/u8 outputs)", "data": "synthetic",
                "config": {"workload": f"{head['images_per_gpu']} images per GPU: {CONFIGS[args.config][2]} (BASELINE configs[{CONFIGS[args.config][0]}]); "
                                       f"image-sharded, shared DHT/DQT broadcast over NCCL",
                           "l2": "inputs larger than L2: bitstream %.0f MB + coefficient rows %.0f MB per step" % (bits_size / 1e6, npad * (bpp_img - 10.0) / 1e6),
                           "decoder_status_words": head["decoder_status_words"], "bit_exact_vs_oracle": head["bit_exact"],
                           "bit_exact_checked_images": head["bit_exact_checked_images"], "images_all_ranks": head["images_all_ranks"],
                           "mismatching_images": head["mismatching_images"], "checked_by": head["checked_by"], "gen_s": head["gen_s"]},
                "roofline": roof, "cpu_baseline": cb, "e2e": e2e, "gpu_launches": ctx["launches"] * args.steps, "clocks": clocks,
                "configs": [head] + side_recs}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
