"""Detection time against the preload window (long poly(A) tails): device-resident int16 reads through adb_detect_dev
for RNA004 / CNN and RNA002 / LLR, at the shipped window and at windows of about 2x, 4x and 7.5x it (capped at
131 072 samples, the longest window the kernels are built for).

Reads: the long-poly(A) stress set of bench.py --stress (poly(A) lengths up to the window, 10 % cut short), generated
in HBM by adapted_b200.synth.make_reads_torch.  For each window: milliseconds per 100 000 reads (CUDA events around
--steps calls after --warmup calls), the per-class kernel timers of adb_ctx_set_timing (bench.py's class names), and
the number of reads validate_fast_kernel / validate_hist_kernel handed to validate_kernel (0 where the window is too
long for validate_fast_kernel's staged layout: every read then goes through validate_kernel, timed as class 2).

    python tools/long_window_bench.py OUT_DIR [--reads 50000] [--warmup 1] [--steps 3]

Prints the card and its power limit, and writes OUT_DIR/long_window_b200.json.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.stream_session_bench import gpu_name_power  # noqa: E402

MAX_WINDOW = 131072
CLS_NAMES = ["global_select_pass", "global_select_small", "validate_hist_kernel | validate_fast_kernel", "llr_primary_kernel",
             "mvs_series_kernel + series_median_kernel", "cnn_conv_kernels", "cnn_pre_post | start_peak | svb16_decode",
             "handover_kernels"]


def window_config(chem: str, m: int):
    from adapted_b200.config import config_as_dict, config_from_dict, get_chemistry_specific_config

    base = get_chemistry_specific_config(chem)
    d = config_as_dict(base)
    d["core"]["max_obs_trace"] = m - (base.sig_preload_size - base.core.max_obs_trace)
    spc = config_from_dict(d)
    assert spc.sig_preload_size == m
    return spc


def run(chem: str, m: int, n: int, warmup: int, steps: int, dev, weights):
    import torch

    from adapted_b200 import _lib
    from adapted_b200.config import flatten_config
    from adapted_b200.synth import make_reads_torch

    spc = window_config(chem, m)
    flat = flatten_config(spc)
    mbs = 1000
    data = make_reads_torch(n, chem, m, seed=4321, device=dev, stress=True, short_frac=0.1,
                            short_min=50 if flat["primary_method"] == 1 else flat["min_obs_adapter"] + 200)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    samples = int(data["offsets"][-1].item())
    cfg = _lib.fill_config(flat)
    w_dev = None
    if flat["primary_method"] == 1:
        from adapted_b200.detect import flatten_cnn_weights

        w_dev = torch.from_numpy(flatten_cnn_weights(weights)).to(dev)
    records = torch.zeros(n * 512, dtype=torch.uint8, device=dev)
    status = torch.zeros((n + mbs - 1) // mbs, dtype=torch.int32, device=dev)
    batch = _lib.AdbBatch(signal=data["adc"].data_ptr(), sig_type=_lib.SIG_I16, n_reads=n, m=m, batch_size=mbs,
                          offsets=data["offsets"].data_ptr(), full_lens=data["full_lens"].data_ptr(),
                          calib_offset=data["calib_offset"].data_ptr(), calib_scale=data["calib_scale"].data_ptr())
    ctx = _lib.default_context(dev.index or 0)
    L = _lib.load()
    # a stream of its own: the events below are recorded on it, and adb_detect_dev would take its context's stream for 0
    ts = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(ts)
    stream = ts.cuda_stream
    assert stream != 0

    def step():
        _lib.check(L.adb_detect_dev(ctx.handle, C.byref(batch), C.byref(cfg), w_dev.data_ptr() if w_dev is not None else None,
                                    records.data_ptr(), status.data_ptr(), C.c_void_p(stream)))

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    L.adb_ctx_set_timing(ctx.handle, 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ts)
    for _ in range(steps):
        step()
    e1.record(ts)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    tim = (C.c_double * 16)()
    L.adb_ctx_get_timing(ctx.handle, tim)
    L.adb_ctx_set_timing(ctx.handle, 0)
    recs = records.cpu().numpy().view(_lib.RECORD_DTYPE)
    pe = recs["polya_end"] if "polya_end" in recs.dtype.names else None
    out = dict(chemistry=chem, primary=spc.primary_method, window=m, reads=n, samples=samples, steps=steps,
               ms_per_call=ms, ms_per_100k_reads=ms * 100000.0 / n,
               kernel_ms_per_100k_reads={CLS_NAMES[k]: tim[2 * k] / steps * 100000.0 / n for k in range(8) if tim[2 * k + 1]},
               validate_handovers=int(ctx.query("validate_handovers")),
               lost_minibatches=int((status != 0).sum().item()),
               n_pass=int(recs["success"].sum()),
               polya_end_beyond_17500=int((pe > 17500).sum()) if pe is not None else None)
    del data, records, status
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("out_dir")
    ap.add_argument("--reads", type=int, default=50000)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--chemistry", nargs="+", default=["rna004", "rna002"])
    args = ap.parse_args()
    import torch

    from adapted_b200.config import get_chemistry_specific_config
    from tests.golden_io import load_cnn_weights

    card = gpu_name_power()
    print(f"card, power limit: {card}", flush=True)
    dev = torch.device("cuda", 0)
    results = []
    for chem in args.chemistry:
        shipped = get_chemistry_specific_config(chem).sig_preload_size
        windows = [shipped] + [min(MAX_WINDOW, int(round(shipped * f / 100.0)) * 100) for f in (2, 4, 7.5)]
        for m in sorted(set(windows)):
            r = run(chem, m, args.reads, args.warmup, args.steps, dev, load_cnn_weights() if chem == "rna004" else None)
            print(json.dumps(r), flush=True)
            results.append(r)
    doc = dict(tool="long_window_bench", gpu=card, timing="CUDA events around adb_detect_dev on device-resident int16 "
               "reads (minibatches of 1000); kernel timers from adb_ctx_set_timing", results=results)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "long_window_b200.json"), "w") as f:
        f.write(json.dumps(doc, indent=1) + "\n")
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
