"""Read-until simulation: per-push cost of StreamSession against the stateless streaming detector on the full caches.

Every channel receives one chunk of 0.4 s of signal per step (1600 samples RNA004, 1200 RNA002, synthetic reads of
adapted_b200.synth.make_reads); an exhausted read is replaced by the next one (reset).  Each step is answered twice:
by StreamSession.push on the chunks, and by the stateless call on every channel's whole cache (what a caller without
a session does).  Both are timed with the host clock around the synchronous calls, and must answer identically at
every step.  The hypothesis under test: a push costs in proportion to the chunk, the stateless call in proportion to
the caches -- the JSON reports both timings for the steps with the smaller and the larger half of the cached samples.

--dtype picks the sessions: int16 (ADC chunks with each read's calibration, against mean_var_shift_polyA_detect_i16
on the ragged caches) and / or float32 (the same reads as calibrate(adc, offset, scale) pA chunks, against
mean_var_shift_polyA_detect_batch on a dense float32 matrix of the caches).  Both run the same schedule.  The
stateless float32 call stages whole caches of 4-byte samples in shared memory, so it takes --max-samples up to about
55 000 (int16: about 110 000).

    python tools/stream_session_bench.py OUT_DIR [--slots 512 3000] [--warmup 20] [--steps 200]
    python tools/stream_session_bench.py OUT_DIR --dtype int16 float32 --max-samples 50000

Prints the card and its power limit, and writes one JSON line to OUT_DIR/stream_session_bench.json.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CHUNK = {"rna004": 1600, "rna002": 1200}  # 0.4 s at 4 kHz / 3 kHz


def gpu_name_power() -> str:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout
    return out.strip().splitlines()[0]


def pctl(a, q):
    return float(np.percentile(np.asarray(a, dtype=np.float64), q))


def simulate(chem, n_slots, reads, max_samples, warmup, steps, seed, dtype="int16"):
    from adapted_b200.config import StreamingConfig
    from adapted_b200.detect import mean_var_shift_polyA_detect_batch, mean_var_shift_polyA_detect_i16
    from adapted_b200.stream import StreamSession

    f32 = dtype == "float32"
    p = StreamingConfig()
    chunk = CHUNK[chem]
    rng = np.random.default_rng(seed)
    n_pool = len(reads)
    cur = rng.integers(0, n_pool, n_slots)  # read index per channel
    pos = np.zeros(n_slots, np.int64)
    nxt = int(rng.integers(0, n_pool))
    slots = np.arange(n_slots, dtype=np.int32)
    t_push, t_stateless, cached, n_settled = [], [], [], []
    # float32: the stateless call's dense [n_slots, max_samples] matrix, kept up to date chunk by chunk (row c holds
    # channel c's cache in its first min(pos[c], max_samples) entries)
    dense = np.zeros((n_slots, max_samples), np.float32) if f32 else None
    with StreamSession(p, n_slots, max_samples, dtype=np.float32 if f32 else np.int16) as s:
        for step in range(warmup + steps):
            reset = np.zeros(n_slots, bool)
            if step == 0:
                reset[:] = True
            chunks = []
            for c in range(n_slots):
                if pos[c] >= reads[cur[c]][0].size:
                    cur[c], pos[c], reset[c] = nxt, 0, True
                    nxt = (nxt + 1) % n_pool
                sig = reads[cur[c]][3 if f32 else 0]
                chunks.append(sig[pos[c]: pos[c] + chunk])
                if f32 and pos[c] < max_samples:
                    k = min(chunks[-1].size, max_samples - int(pos[c]))
                    dense[c, pos[c]: pos[c] + k] = chunks[-1][:k]
                pos[c] += chunks[-1].size
            if f32:
                t0 = time.perf_counter()
                got, settled = s.push(slots, chunks, reset=reset)
                t1 = time.perf_counter()
                lens = np.minimum(pos, max_samples).astype(np.int32)
                t2 = time.perf_counter()
                want = mean_var_shift_polyA_detect_batch(dense, lens, p)
                t3 = time.perf_counter()
                total = int(lens.sum())
            else:
                coff = np.array([reads[r][1] for r in cur], np.float32)
                cscale = np.array([reads[r][2] for r in cur], np.float32)
                t0 = time.perf_counter()
                got, settled = s.push(slots, chunks, reset=reset, calib_offset=coff, calib_scale=cscale)
                t1 = time.perf_counter()
                caches = [reads[cur[c]][0][: min(int(pos[c]), max_samples)] for c in range(n_slots)]
                offsets = np.zeros(n_slots + 1, np.int64)
                offsets[1:] = np.cumsum([a.size for a in caches])
                blob = np.concatenate(caches)
                t2 = time.perf_counter()
                want = mean_var_shift_polyA_detect_i16(blob, offsets, coff, cscale, p, window=max_samples)
                t3 = time.perf_counter()
                total = int(offsets[-1])
            if not np.array_equal(got, want):
                bad = np.flatnonzero(got != want)
                raise AssertionError(f"{chem} {n_slots} {dtype} step {step}: session != stateless at channels {bad[:8]}: "
                                     f"{got[bad[:8]]} vs {want[bad[:8]]}")
            if step >= warmup:
                t_push.append(t1 - t0)
                t_stateless.append(t3 - t2)
                cached.append(total)
                n_settled.append(int(settled.sum()))
    cached = np.asarray(cached)
    lo = cached <= np.median(cached)
    ms = lambda a: round(pctl(a, 50) * 1e3, 3)  # noqa: E731
    return dict(
        chemistry=chem, n_slots=n_slots, dtype=dtype, chunk=chunk, steps=steps, warmup=warmup,
        stateless_call="mean_var_shift_polyA_detect_batch" if f32 else "mean_var_shift_polyA_detect_i16",
        push_ms_median=ms(t_push), push_ms_p99=round(pctl(t_push, 99) * 1e3, 3),
        stateless_ms_median=ms(t_stateless), stateless_ms_p99=round(pctl(t_stateless, 99) * 1e3, 3),
        cached_samples_median=int(np.median(cached)), settled_median=int(np.median(n_settled)),
        # the hypothesis: push time does not follow the cached samples, the stateless call does
        push_ms_median_smaller_caches=ms(np.asarray(t_push)[lo]), push_ms_median_larger_caches=ms(np.asarray(t_push)[~lo]),
        stateless_ms_median_smaller_caches=ms(np.asarray(t_stateless)[lo]),
        stateless_ms_median_larger_caches=ms(np.asarray(t_stateless)[~lo]),
        cached_samples_median_smaller=int(np.median(cached[lo])), cached_samples_median_larger=int(np.median(cached[~lo])),
    )


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("out_dir")
    ap.add_argument("--slots", type=int, nargs="+", default=[512, 3000])
    ap.add_argument("--chemistry", nargs="+", default=["rna004", "rna002"])
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--pool", type=int, default=1200, help="synthetic reads per chemistry, reused round robin")
    ap.add_argument("--max-samples", type=int, default=100000,
                    help="cache per channel; the stateless call stages whole caches in shared memory (<= ~110 000 "
                         "int16, ~55 000 float32)")
    ap.add_argument("--dtype", nargs="+", choices=["int16", "float32"], default=["int16"],
                    help="session sample types to run, each against its stateless call")
    args = ap.parse_args()
    from adapted_b200.synth import calibrate, make_reads

    card = gpu_name_power()
    print(f"card, power limit: {card}", flush=True)
    results = []
    for chem in args.chemistry:
        b = make_reads(args.pool, chem, args.max_samples, seed=1234)
        reads = []
        for i in range(b.n):
            adc, co, cs = b.adc[b.offsets[i]: b.offsets[i + 1]], float(b.calib_offset[i]), float(b.calib_scale[i])
            reads.append((adc, co, cs, calibrate(adc, co, cs) if "float32" in args.dtype else None))
        for n_slots in args.slots:
            for dtype in args.dtype:
                r = simulate(chem, n_slots, reads, args.max_samples, args.warmup, args.steps, seed=n_slots, dtype=dtype)
                print(json.dumps(r), flush=True)
                results.append(r)
    doc = dict(tool="stream_session_bench", gpu=card, max_samples=args.max_samples, timing="host clock around "
               "synchronous calls; stateless excludes building its ragged blob (int16) or dense matrix (float32)",
               results=results)
    os.makedirs(args.out_dir, exist_ok=True)
    line = json.dumps(doc)
    with open(os.path.join(args.out_dir, "stream_session_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
