"""VBZ ingest on one GPU: the zstd stage of pod5's signal form decoded on the device (zstd_decode_kernel) against
svb16 containers and against host decompression (ctx option "host_zstd").

For RNA004 (CNN) and RNA002 (LLR) at their shipped preload windows, synthetic reads (adapted_b200.synth.make_reads_torch,
the squiggles bench.py times; real signal compresses differently) are written as three ADBSIG02 containers of the same
reads -- svb16 streams, zstd frames over them (level 1, as pod5 writes VBZ) -- and run through the native file
pipeline (adb_detect_files) as

  svb16        svb16 container
  zstd_device  zstd container, frames copied as they are and decoded on the GPU
  zstd_host    zstd container, frames decompressed by the reader's copy threads (libzstd), today's path

Per form: file -> tables reads/s (second of two runs: page cache, pinned ring and contexts warm), the reader's busy
time, wire bytes per sample (container blob / samples).  In memory: detect_reads_vbz against detect_reads_svb with
their pipeline_copy_only ceilings.  In a separate run under torch.profiler: zstd_decode_kernel time per chunk next
to that chunk's host -> device copy.

    python tools/vbz_ingest_bench.py OUT_DIR [--reads 400000] [--rna002-reads 400000]

Prints the card and its power limit, and writes OUT_DIR/vbz_ingest_b200.json.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.stream_session_bench import gpu_name_power  # noqa: E402

MBS, CHUNK = 1000, 16


def make_inputs(chem, n, seed):
    import torch

    from adapted_b200 import svb16
    from adapted_b200.config import get_chemistry_specific_config
    from adapted_b200.synth import make_reads_torch

    spc = get_chemistry_specific_config(chem)
    m = int(spc.sig_preload_size)
    d = make_reads_torch(n, chem, m, seed=seed, device="cuda")
    comp, coff, ns = svb16.encode_reads_torch(d["adc"], d["offsets"], m)
    torch.cuda.synchronize()
    comp, coff, ns = comp.cpu().numpy(), coff.cpu().numpy(), ns.cpu().numpy()
    frames, foff = svb16.zstd_frames(comp, coff, 1)
    host = {k: d[k].cpu().numpy() for k in ("full_lens", "calib_offset", "calib_scale")}
    del d
    torch.cuda.empty_cache()
    return spc, m, comp, coff, ns, frames, foff, host


def run(args):
    import torch

    from adapted_b200 import _lib
    from adapted_b200.detect import detect_reads_svb, detect_reads_vbz
    from adapted_b200.ingest import detect_files_native, write_container_v2
    from tests.golden_io import load_cnn_weights

    card = gpu_name_power()
    print("card, power limit:", card, flush=True)
    ctx = _lib.default_context(0)
    result = {"card_power_limit": card, "minibatch_size": MBS, "chunk_minibatches": CHUNK,
              "note": "synthetic reads (adapted_b200.synth); real signal compresses differently", "chemistries": {}}
    for chem, n in (("rna004", args.reads), ("rna002", args.rna002_reads)):
        spc, m, comp, coff, ns, frames, foff, host = make_inputs(chem, n, 4321)
        w = load_cnn_weights() if chem == "rna004" else None
        samples = int(ns.astype(np.int64).sum())
        r = {"reads": n, "window": m, "samples": samples,
             "wire_bytes_per_sample": {"svb16": float(coff[-1]) / samples, "zstd": float(foff[-1]) / samples}}
        tmp = tempfile.mkdtemp(prefix="adb_vbz_", dir=args.tmp or None)
        try:
            ids = np.char.add(np.char.zfill(np.arange(n).astype("U8"), 8), "-0000-4000-8000-000000000000")
            paths = {}
            for form in ("svb16", "zstd"):
                paths[form] = write_container_v2(os.path.join(tmp, form), None, np.arange(n + 1), host["full_lens"], host["calib_offset"],
                                                 host["calib_scale"], ids, encoded=(comp, coff, ns), zstd=form == "zstd")
            r["container_bytes"] = {k: os.path.getsize(p) for k, p in paths.items()}
            files = {}
            for rep in range(2):  # alternate the forms; the second round is reported
                for form, path, host_z in (("svb16", paths["svb16"], 0), ("zstd_device", paths["zstd"], 0), ("zstd_host", paths["zstd"], 1)):
                    ctx.set_option("host_zstd", host_z)
                    out = os.path.join(tmp, f"out_{form}_{rep}")
                    t0 = time.perf_counter()
                    st = detect_files_native([path], out, spc, model=w, minibatch_size=MBS, chunk_minibatches=CHUNK)
                    dt = time.perf_counter() - t0
                    ctx.set_option("host_zstd", 0)
                    files[form] = {"seconds": dt, "reads_per_s": n / dt, "reader_busy_s": st["reader_busy_s"],
                                   "writer_wait_gpu_s": st["writer_wait_gpu_s"], "h2d_bytes": st["h2d_bytes"],
                                   "host_frames": ctx.query("zstd_host_frames"), "pass": st["pass"], "fail": st["fail"]}
                    shutil.rmtree(out, ignore_errors=True)
                    print(chem, rep, form, json.dumps(files[form]), flush=True)
            r["file_to_tables"] = files
            r["zstd_device_over_svb16"] = files["zstd_device"]["reads_per_s"] / files["svb16"]["reads_per_s"]
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        # in memory, host buffers -> records
        args_ = (host["full_lens"], host["calib_offset"], host["calib_scale"], spc, w)
        mem = {}
        for rep in range(2):
            for name, fn, blob, offs in (("svb16", detect_reads_svb, comp, coff), ("vbz", detect_reads_vbz, frames, foff)):
                for copy_only in (0, 1):
                    ctx.set_option("pipeline_copy_only", copy_only)
                    t0 = time.perf_counter()
                    recs, _ = fn(blob, offs, ns, *args_, minibatch_size=MBS, chunk_minibatches=CHUNK)
                    dt = time.perf_counter() - t0
                    ctx.set_option("pipeline_copy_only", 0)
                    mem[name + ("_copy_only" if copy_only else "")] = {"seconds": dt, "reads_per_s": n / dt}
                    if not copy_only:
                        mem[name + "_records"] = recs
        r["records_identical"] = bool(mem.pop("svb16_records").tobytes() == mem.pop("vbz_records").tobytes())
        r["in_memory"] = mem
        print(chem, "in memory", json.dumps(mem), "records identical:", r["records_identical"], flush=True)
        # kernel time per chunk under the profiler (a run of its own)
        from torch.profiler import ProfilerActivity, profile

        k = min(n, 64000)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            detect_reads_vbz(frames, foff[: k + 1], ns[:k], host["full_lens"][:k], host["calib_offset"][:k], host["calib_scale"][:k],
                             spc, w, minibatch_size=MBS, chunk_minibatches=CHUNK)
            torch.cuda.synchronize()
        zk = [e.device_time for e in prof.events() if e.name.startswith("zstd_decode_kernel")]
        sk = [e.device_time for e in prof.events() if e.name.startswith("svb16_decode_kernel")]
        h2d = [e.device_time for e in prof.events() if "HtoD" in e.name and e.device_time > 50]
        r["profile"] = {"reads": k, "chunks": len(zk), "zstd_decode_kernel_us_per_chunk": zk, "svb16_decode_kernel_us_per_chunk": sk,
                        "frames_h2d_us_per_chunk": h2d,
                        "note": "chunks of 16 000 reads in the middle, 4000 / 8000 at both ends (pipeline_schedule)"}
        print(chem, "profile", json.dumps(r["profile"]), flush=True)
        result["chemistries"][chem] = r
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "vbz_ingest_b200.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("out")
    ap.add_argument("--reads", type=int, default=400000)
    ap.add_argument("--rna002-reads", type=int, default=400000)
    ap.add_argument("--tmp", default=None, help="directory for the containers (default: the system's temporary directory)")
    run(ap.parse_args())
