"""Read-until simulation of device pushes: per-push latency of StreamSession.push against push_device.

The schedule is that of tools/stream_session_bench.py: every channel receives one chunk of 0.4 s of signal per step
(1600 samples RNA004, 1200 RNA002), an exhausted read is replaced by the next one (reset).  Three sessions of the same
sample type run it:
  host           StreamSession.push on host chunks, host clock around the synchronous call;
  dev_sync       push_device on chunks already on the device, then a synchronise of its stream, host clock around
                 both (plus CUDA events around the push: its device time);
  back_to_back   push_device for every step enqueued on one stream while the host synchronises once per step, on the
                 previous step's push, so one push always waits behind the running one, as for a client that overlaps
                 its own work with the pushes; per push the host time between consecutive synchronisations.
All chunks of a run are uploaded to the device before its timed steps.  The answers of the three sessions are asserted
identical at every step.

    python tools/stream_session_dev_bench.py OUT_DIR [--slots 512 3000] [--chemistry rna004 rna002]
                                             [--dtype int16 float32] [--warmup 20] [--steps 200]

Prints the card and its power limit, and writes one JSON line to OUT_DIR/stream_session_dev_bench.json.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.stream_session_bench import CHUNK, gpu_name_power, pctl  # noqa: E402


def schedule(chem, n_slots, reads, warmup, steps, seed, f32):
    """per step: (host chunks, reset, calib_offset, calib_scale) as StreamSession.push takes them"""
    chunk = CHUNK[chem]
    rng = np.random.default_rng(seed)
    n_pool = len(reads)
    cur = rng.integers(0, n_pool, n_slots)
    pos = np.zeros(n_slots, np.int64)
    nxt = int(rng.integers(0, n_pool))
    out = []
    for step in range(warmup + steps):
        reset = np.full(n_slots, step == 0)
        chunks = []
        for c in range(n_slots):
            if pos[c] >= reads[cur[c]][0].size:
                cur[c], pos[c], reset[c] = nxt, 0, True
                nxt = (nxt + 1) % n_pool
            sig = reads[cur[c]][3 if f32 else 0]
            chunks.append(sig[pos[c]: pos[c] + chunk])
            pos[c] += chunks[-1].size
        coff = np.array([reads[r][1] for r in cur], np.float32)
        cscale = np.array([reads[r][2] for r in cur], np.float32)
        out.append((chunks, reset, coff, cscale))
    return out


def simulate(chem, n_slots, reads, max_samples, warmup, steps, seed, dtype):
    import torch

    from adapted_b200.config import StreamingConfig
    from adapted_b200.stream import StreamSession, pack_chunks

    f32 = dtype == "float32"
    npt = np.float32 if f32 else np.int16
    p = StreamingConfig()
    sched = schedule(chem, n_slots, reads, warmup, steps, seed, f32)
    slots = np.arange(n_slots, dtype=np.int32)
    dev = torch.device("cuda", 0)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    d_slots = up(slots)
    staged = []
    for chunks, reset, coff, cscale in sched:
        _, samples, offsets = pack_chunks(slots, chunks, npt)
        kw = dict(reset=up(reset.astype(np.uint8)))
        if not f32:
            kw.update(calib_offset=up(coff), calib_scale=up(cscale))
        staged.append(((d_slots, up(offsets), up(samples)), kw))
    torch.cuda.synchronize()
    st = torch.cuda.Stream(dev)
    mk = lambda dp: StreamSession(p, n_slots, max_samples, dtype=npt, device_push=dp)  # noqa: E731
    t_host, t_sync, t_dev, t_b2b, answers = [], [], [], [], []
    with mk(False) as h, mk(True) as d, mk(True) as d2:
        for step, ((chunks, reset, coff, cscale), (args, kw)) in enumerate(zip(sched, staged)):
            cal = {} if f32 else dict(calib_offset=coff, calib_scale=cscale)
            t0 = time.perf_counter()
            want, wset = h.push(slots, chunks, reset=reset, **cal)
            t1 = time.perf_counter()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t2 = time.perf_counter()
            e0.record(st)
            got, gset, status = d.push_device(*args, stream=st, **kw)
            e1.record(st)
            st.synchronize()
            t3 = time.perf_counter()
            if status.tolist() != [0, 0] or not np.array_equal(got.cpu().numpy(), want) or \
                    not np.array_equal(gset.cpu().numpy(), wset):
                raise AssertionError(f"{chem} {n_slots} {dtype} step {step}: device push != host push")
            answers.append((want, wset))
            if step >= warmup:
                t_host.append(t1 - t0)
                t_sync.append(t3 - t2)
                t_dev.append(e0.elapsed_time(e1) * 1e-3)
        outs, evs = [], []
        torch.cuda.synchronize()
        t_prev = time.perf_counter()
        for step, (args, kw) in enumerate(staged):
            outs.append(d2.push_device(*args, stream=st, **kw))
            evs.append(torch.cuda.Event())
            evs[-1].record(st)
            if step > 0:
                evs[step - 1].synchronize()
                t = time.perf_counter()
                if step - 1 >= warmup:
                    t_b2b.append(t - t_prev)
                t_prev = t
        evs[-1].synchronize()
        t_b2b.append(time.perf_counter() - t_prev)
        for step, ((want, wset), (got, gset, status)) in enumerate(zip(answers, outs)):
            if status.tolist() != [0, 0] or not np.array_equal(got.cpu().numpy(), want) or \
                    not np.array_equal(gset.cpu().numpy(), wset):
                raise AssertionError(f"{chem} {n_slots} {dtype} step {step}: back-to-back device push != host push")
    ms = lambda a, q: round(pctl(a, q) * 1e3, 3)  # noqa: E731
    return dict(
        chemistry=chem, n_slots=n_slots, dtype=dtype, chunk=CHUNK[chem], steps=steps, warmup=warmup,
        host_push_ms_median=ms(t_host, 50), host_push_ms_p99=ms(t_host, 99),
        dev_sync_ms_median=ms(t_sync, 50), dev_sync_ms_p99=ms(t_sync, 99),
        dev_device_ms_median=ms(t_dev, 50), dev_device_ms_p99=ms(t_dev, 99),
        back_to_back_ms_median=ms(t_b2b, 50), back_to_back_ms_p99=ms(t_b2b, 99),
        settled_median=int(np.median([a[1].sum() for a in answers[warmup:]])),
    )


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("out_dir")
    ap.add_argument("--slots", type=int, nargs="+", default=[512, 3000])
    ap.add_argument("--chemistry", nargs="+", default=["rna004", "rna002"])
    ap.add_argument("--dtype", nargs="+", choices=["int16", "float32"], default=["int16", "float32"])
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--pool", type=int, default=1200, help="synthetic reads per chemistry, reused round robin")
    ap.add_argument("--max-samples", type=int, default=100000, help="cache per channel")
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
    doc = dict(tool="stream_session_dev_bench", gpu=card, max_samples=args.max_samples,
               timing="host clock; host: around the synchronous push; dev_sync: around push_device plus a stream "
                      "synchronise (dev_device: CUDA events around the push); back_to_back: between consecutive "
                      "per-step synchronisations with one push queued ahead", results=results)
    os.makedirs(args.out_dir, exist_ok=True)
    line = json.dumps(doc)
    with open(os.path.join(args.out_dir, "stream_session_dev_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
