#!/usr/bin/env python
"""bench.py -- throughput of the boundary-detection hot path on B200 (contract: the task brief / DESIGN.md section 5).

Default workload = BASELINE.json configs[2]: RNA004 (rna004_130bps config, CNN primary path + hail-mary LLR fallback),
1 000 000 synthetic reads per GPU in minibatches of 1000.  A "step" is one pass over all reads of the rank.

  value      reads/s with the int16 ADC reads already resident in HBM (CUDA events on the launching stream)
  e2e        reads/s through the compressed pipelined ingest: pinned host svb16 streams -> H2D -> device decode ->
             kernels -> D2H of the records (adb_detect_pipelined_svb_host); e2e.copy_only = the same chunks with the
             kernels skipped, i.e. this box's host -> device ceiling for the run
  roofline   dominant kernel class: algorithmic bytes / its event-timed duration vs the measured HBM peak; for the CNN
             workload both views (tensor view of the convolution class, HBM view of the dominant non-tensor class)
  file_to_csv  BASELINE configs[4] scaled to the box: ADBSIG02 container on local storage -> native pipeline
             (adb_detect_files) -> CSV tables, reads/s wall clock
  secondary  BASELINE configs[1] in the same run: RNA002 / LLR path, 100 000 reads per GPU (value, e2e, roofline) and
             its start-peak companion configuration (value)
  cpu_baseline / --impl reference : the EXECUTED reference (oracle/_ref/pkg: combined_detect_cnn / combined_detect_llr2
             of KleistLab/ADAPTed v0.2.4 under ProcessPoolExecutor(os.cpu_count()) on 1000-read minibatches, wall clock
             around the pool, file_proc.py:738-784); the oracle port only where that package was not built
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "reads_per_sec"
WORKLOADS = {
    "rna002": "RNA002 rna002_70bps, LLR primary path, synthetic squiggles, minibatches of 1000 reads",
    "rna004": "RNA004 rna004_130bps, CNN primary path (+ hail-mary LLR fallback), synthetic squiggles, minibatches of 1000 reads",
}
DEFAULT_READS = {"rna004": 1000000, "rna002": 100000}


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def workload_config(chem: str, reads: int, minibatch: int, world: int, stress: bool, preload: int) -> dict:
    """the `config` block: identical for both arms (the driver compares them)"""
    w = WORKLOADS.get(chem, chem)
    if stress:
        w += " -- stress set (config 4: long poly(A) / truncated preload, short reads)"
    return {"workload": w, "chemistry": chem, "reads_per_gpu": reads, "minibatch": minibatch, "preload_window": preload,
            "l2": "inputs (>= 3.5 GB per GPU) exceed the 126 MB L2",
            "parallelism": f"minibatches sharded over {world} GPU(s), no collective"}


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the executed reference (oracle/_ref/pkg) under a process pool, 1000-read minibatches
# ---------------------------------------------------------------------------------------------------------
_REF = {}


def _ref_init(chem: str, kind: str):
    import logging
    import warnings

    warnings.simplefilter("ignore")
    logging.disable(logging.CRITICAL)
    if kind == "reference":
        from oracle import build_ref

        sys.path.insert(0, build_ref.PKG)
        from adapted.config.sig_proc import get_chemistry_specific_config
        from adapted.detect import combined
        from adapted.detect.cnn import load_cnn_model

        spc = get_chemistry_specific_config(chem)
        spc.update_primary_method()
        spc.update_sig_preload_size()
        model = load_cnn_model(spc.cnn_boundaries.model_name) if spc.primary_method == "cnn" else None
        _REF.update(kind=kind, spc=spc, model=model, combined=combined)
    else:
        from adapted_b200.config import get_chemistry_specific_config
        from oracle import detect_ref

        spc = get_chemistry_specific_config(chem)
        _REF.update(kind=kind, spc=spc, model=_cnn_weights() if spc.primary_method == "cnn" else None, combined=detect_ref)


def _ref_task(args):
    """one minibatch through the reference's seam function, as a pool worker runs it (file_proc.py:217-266)"""
    x, lens = args
    spc, model, mod = _REF["spc"], _REF["model"], _REF["combined"]
    t0 = time.perf_counter()
    if _REF["kind"] == "reference":
        res = mod.combined_detect_cnn(x, lens, model, spc) if model is not None else mod.combined_detect_llr2(x, lens, spc)
        res = res if isinstance(res, list) else [res]
        ok = sum(bool(r.success) for r in res)
    else:
        res = mod.detect_cnn(x, lens, model, spc) if model is not None else mod.detect_llr2(x, lens, spc)
        res = res if isinstance(res, list) else [res]
        ok = sum(bool(r["success"]) for r in res)
    return len(res), ok, time.perf_counter() - t0


def _cnn_weights():
    """the shipped model's weights (adapted/models/rna004_130bps@v0.2.4.pth) as committed fixture"""
    with np.load(os.path.join(ROOT, "tests", "golden", "cnn_weights_rna004_130bps_v0.2.4.npz")) as z:
        return {k: z[k] for k in z.files}


def cpu_arm(chem: str, steps: int, warmup: int, minibatch: int, cores: int, stress: bool, budget_s: float = 240.0):
    """`steps` passes; a pass = `cores` minibatches of `minibatch` reads submitted to a pool of `cores` worker processes
    (the minibatch matrix is pickled to the worker like the reference's executor.submit does), wall clock around the
    pass.  Inputs are generated before the clock starts."""
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor

    from adapted_b200.config import get_chemistry_specific_config
    from adapted_b200.synth import make_reads
    from oracle import build_ref
    from oracle._clib import build as build_oracle

    build_oracle()
    kind = "reference" if build_ref.package_present() else "port"
    spc = get_chemistry_specific_config(chem)
    m = spc.sig_preload_size
    kw = dict(stress=True, short_frac=0.1) if stress else {}
    batches = []
    for i in range(cores):
        b = make_reads(minibatch, chem, m, seed=2000 + i, **kw)
        batches.append((b.to_dense_pa(), b.full_lens, int(np.minimum(b.full_lens, m).sum())))
    small = [(x[:16].copy(), lens[:16].copy()) for x, lens, _ in batches]
    t_all = time.perf_counter()
    with ProcessPoolExecutor(max_workers=cores, mp_context=mp.get_context("spawn"), initializer=_ref_init, initargs=(chem, kind)) as ex:
        for _ in range(max(warmup, 1)):
            list(ex.map(_ref_task, small))
        reads = ok = done = 0
        dt = 0.0
        for s in range(steps):
            t0 = time.perf_counter()
            res = list(ex.map(_ref_task, [(x, lens) for x, lens, _ in batches]))
            dt += time.perf_counter() - t0
            reads += sum(r[0] for r in res)
            ok += sum(r[1] for r in res)
            done += 1
            if time.perf_counter() - t_all > budget_s:  # bounded sample: the whole arm ends within a few minutes
                break
    samples = sum(b[2] for b in batches) * done
    return {"kind": kind, "reads_per_s": reads / dt, "samples_per_s": samples / dt, "s_per_step": dt / done, "steps": done,
            "reads_per_step": reads // done, "pass_fraction": ok / max(reads, 1)}


def lib_versions():
    import scipy
    import torch

    return {"numpy": np.__version__, "scipy": scipy.__version__, "torch": torch.__version__}


# ---------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.sm, self.smax, self.reasons = [], [], set()

    def run(self):
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [v.strip() for v in out.strip().split(",")]
                self.sm.append(float(f[0]))
                self.smax.append(float(f[1]))
                for nm, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": float(max(self.smax)), "reasons": sorted(self.reasons)}


def bind_to_gpu_local_cpus(local_rank: int):
    """Run this rank (and place its pinned staging memory by first touch) on the CPUs that are PCIe-local to its GPU:
    /sys/bus/pci/devices/<bdf>/local_cpulist (numa_node reads -1 on boxes whose firmware does not describe the nodes).
    Returns a description for the JSON line."""
    info = {"local_cpulist": None, "bound": False, "numa_node": None}
    try:
        import torch

        pr = torch.cuda.get_device_properties(local_rank)
        dev = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{dev}"
        try:
            info["numa_node"] = int(open(f"{base}/numa_node").read().strip())
        except Exception:
            pass
        txt = open(f"{base}/local_cpulist").read().strip()
        info["local_cpulist"] = txt
        cpus = set()
        for part in txt.split(","):
            if part:
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        # binding only helps when the local set is a proper part of what the process may use
        if cpus and len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            info["bound"] = True
    except Exception:  # noqa: BLE001 -- topology files missing (containers): keep the inherited affinity
        pass
    return info


DUMP_READS = 65536  # 65 536 records of 105 values (plus read_index) in float64 stay under 64 MB


def dump_outputs(out_dir: str, recs: np.ndarray, status: np.ndarray):
    """What the last timed step handed its caller: every field of the adb_record array (as records_<field>.npy, one row
    per read) and the per-minibatch status.  Runs with more than DUMP_READS reads keep a fixed, seeded sample of the
    reads (read_index.npy), so two builds given the same arguments write comparable files."""
    os.makedirs(out_dir, exist_ok=True)
    idx = np.arange(len(recs))
    if len(recs) > DUMP_READS:
        idx = np.sort(np.random.default_rng(0).choice(len(recs), DUMP_READS, replace=False))
    arrays = {"read_index": idx, "status": status}
    for name in recs.dtype.names:
        if name != "_reserved":
            arrays["records_" + name] = recs[name][idx]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


CLS_NAMES = ["global_select_pass", "global_select_small", "validate_hist_kernel", "llr_primary_kernel", "mvs_series_kernel + series_median_kernel",
             "cnn_conv_kernels", "cnn_pre_post | start_peak | svb16_decode", "handover_kernels"]


class Runner:
    """one rank's GPU side: context, data of a workload, the timed loops"""

    def __init__(self, local_rank, rank, world, barrier, all_reduce):
        import torch

        from adapted_b200 import _lib

        self.torch, self._lib = torch, _lib
        self.L = _lib.load()
        self.local_rank, self.rank, self.world = local_rank, rank, world
        self.dev = torch.device("cuda", local_rank)
        self.ctx = _lib.Context(local_rank)
        _lib._default_ctx[local_rank] = self.ctx  # the file-level block runs on the same context (one scratch arena per GPU)
        self.barrier, self.all_reduce = barrier, all_reduce
        self.tstream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.tstream)
        self.peaks = {}
        try:
            self.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass

    def run(self, chem, n, args, spc=None, e2e=True, steps=None, label=None):
        torch, _lib, L, dev = self.torch, self._lib, self.L, self.dev
        from adapted_b200 import svb16
        from adapted_b200.config import flatten_config, get_chemistry_specific_config
        from adapted_b200.synth import make_reads_torch

        spc = spc or get_chemistry_specific_config(chem)
        flat = flatten_config(spc)
        m, mbs = flat["sig_preload_size"], args.minibatch
        steps = steps or args.steps
        gen_kw = {}
        if args.stress:
            gen_kw = dict(stress=True, short_frac=0.1, short_min=50 if flat["primary_method"] == 1 else flat["min_obs_adapter"] + 200)
        data = make_reads_torch(n, chem, m, seed=1234 + self.rank, device=dev, **gen_kw)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()  # the generator's temporaries: the library allocates with cudaMalloc, not from torch's cache
        samples = int(data["offsets"][-1].item())
        trace_samples = int(torch.clamp(data["offsets"][1:] - data["offsets"][:-1], max=flat["max_obs_trace"]).sum().item())
        cfg = _lib.fill_config(flat)
        w_host = w_dev = None
        if flat["primary_method"] == 1:
            from adapted_b200.detect import flatten_cnn_weights

            w_host = torch.from_numpy(flatten_cnn_weights(_cnn_weights()))
            w_dev = w_host.to(dev)
        records = torch.zeros(n * 512, dtype=torch.uint8, device=dev)
        n_batches = (n + mbs - 1) // mbs
        status = torch.zeros(n_batches, dtype=torch.int32, device=dev)
        batch = _lib.AdbBatch(signal=data["adc"].data_ptr(), sig_type=_lib.SIG_I16, n_reads=n, m=m, batch_size=mbs,
                              offsets=data["offsets"].data_ptr(), full_lens=data["full_lens"].data_ptr(),
                              calib_offset=data["calib_offset"].data_ptr(), calib_scale=data["calib_scale"].data_ptr())
        stream = self.tstream.cuda_stream
        assert stream != 0
        ctx = self.ctx

        def step():
            _lib.check(L.adb_detect_dev(ctx.handle, C.byref(batch), C.byref(cfg), w_dev.data_ptr() if w_dev is not None else None,
                                        records.data_ptr(), status.data_ptr(), C.c_void_p(stream)))

        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        L.adb_ctx_set_timing(ctx.handle, 1)
        launches0 = ctx.launches
        self.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        self.barrier()
        ms = e0.elapsed_time(e1)
        launches = ctx.launches - launches0
        tim = (C.c_double * 16)()
        L.adb_ctx_get_timing(ctx.handle, tim)
        L.adb_ctx_set_timing(ctx.handle, 0)
        rec_dev_host = records.cpu()
        n_pass = int(torch.frombuffer(rec_dev_host.numpy(), dtype=torch.int32).reshape(n, 128)[:, 0].sum().item())
        lost = int((status != 0).sum().item())
        if args.dump_outputs and label == "main" and self.rank == 0:
            dump_outputs(args.dump_outputs, rec_dev_host.numpy().view(_lib.RECORD_DTYPE), status.cpu().numpy())
        gsel_fallbacks = ctx.query("global_select_fallbacks") if flat["primary_method"] == 0 else 0
        val_handovers = ctx.query("validate_handovers")

        out = {"n": n, "samples": samples, "ms": ms, "steps": steps, "launches": launches, "n_pass": n_pass, "lost": lost,
               "gsel_fallbacks": int(gsel_fallbacks), "val_handovers": int(val_handovers), "tim": list(tim), "flat": flat,
               "trace_samples": trace_samples,
               "e2e": None, "file": None}

        # ---------------- e2e: pinned host (compressed) -> H2D -> decode -> kernels -> D2H ----------------
        if e2e and not args.profile_steps_only:
            comp, coff, ns = svb16.encode_reads_torch(data["adc"], data["offsets"], m)
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            host = {}
            for k, t in (("comp", comp), ("coff", coff), ("ns", ns), ("full_lens", data["full_lens"]),
                         ("calib_offset", data["calib_offset"]), ("calib_scale", data["calib_scale"])):
                h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                h.copy_(t)
                host[k] = h
            comp_bytes = int(coff[-1].item()) + 16
            del comp
            torch.cuda.empty_cache()
            rec_host = torch.zeros(n * 512, dtype=torch.uint8).pin_memory()
            st_host = torch.zeros(n_batches, dtype=torch.int32).pin_memory()
            sb = _lib.AdbSvbBatch(comp=host["comp"].data_ptr(), comp_offsets=host["coff"].data_ptr(), n_samples=host["ns"].data_ptr(),
                                  n_reads=n, m=m, batch_size=mbs, full_lens=host["full_lens"].data_ptr(),
                                  calib_offset=host["calib_offset"].data_ptr(), calib_scale=host["calib_scale"].data_ptr())
            chunk = args.chunk_batches if args.chunk_batches > 0 else (64 if flat["primary_method"] == 1 else 16)  # measured: 16 / 32 / 64 / 128 minibatches -> 1.55 / 1.70 / 1.88 / 1.85 M reads/s end to end (RNA004)

            def e2e_step():
                _lib.check(L.adb_detect_pipelined_svb_host(ctx.handle, C.byref(sb), C.byref(cfg),
                                                           w_host.data_ptr() if w_host is not None else None, rec_host.data_ptr(),
                                                           st_host.data_ptr(), chunk))

            def timed(k):
                self.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(k):
                    e2e_step()
                torch.cuda.synchronize()
                self.barrier()
                return time.perf_counter() - t0

            e2e_steps = max(args.e2e_steps, 10)
            e2e_step()  # warm-up: staging buffers, twin context
            e2e_s = timed(e2e_steps)
            same = bool(torch.equal(rec_host, rec_dev_host))
            # the same chunks with the kernels skipped: what the host -> device path of this box delivers
            ctx.set_option("pipeline_copy_only", 1)
            e2e_step()
            copy_s = timed(3)
            ctx.set_option("pipeline_copy_only", 0)
            h2d = comp_bytes + n * (8 + 4 + 4 + 4 + 4)
            out["e2e"] = {"seconds": e2e_s, "steps": e2e_steps, "copy_seconds": copy_s, "copy_steps": 3, "h2d": h2d,
                          "d2h": n * 512 + n_batches * 4, "same": same, "chunk": chunk, "raw_int16_bytes": 2 * samples,
                          "bytes_per_sample": comp_bytes / max(samples, 1)}

            # ---------------- file level: container on local storage -> native pipeline -> CSV tables ----------------
            if args.file_reads != 0 and label == "main":
                from adapted_b200.ingest import detect_files_native, write_container_v2

                # (several ranks share the box's temporary storage: half the container per rank there)
                nf = n if args.file_reads < 0 else min(n, args.file_reads if self.world == 1 else min(args.file_reads, 200000))
                nf = max(mbs, nf // mbs * mbs)
                tmp = tempfile.mkdtemp(prefix=f"adb_bench_r{self.rank}_", dir=args.file_dir or None)
                try:
                    cend = int(host["coff"][nf].item())
                    ids = np.char.add(np.char.zfill(np.arange(nf).astype("U8"), 8), f"-0000-4000-8000-{self.rank:012d}")
                    path = write_container_v2(os.path.join(tmp, "reads"), None, np.arange(nf + 1), host["full_lens"][:nf].numpy(),
                                              host["calib_offset"][:nf].numpy(), host["calib_scale"][:nf].numpy(), ids,
                                              encoded=(host["comp"][: cend + 16].numpy(), host["coff"][: nf + 1].numpy(), host["ns"][:nf].numpy()))
                    size = os.path.getsize(path)
                    detect_files_native([path], os.path.join(tmp, "warm"), spc, model=_cnn_weights() if w_host is not None else None,
                                        minibatch_size=mbs, chunk_minibatches=chunk, device=self.local_rank)  # warm-up: page cache, pinned ring, contexts
                    self.barrier()
                    t0 = time.perf_counter()
                    st = detect_files_native([path], os.path.join(tmp, "out"), spc, model=_cnn_weights() if w_host is not None else None,
                                             minibatch_size=mbs, chunk_minibatches=chunk, device=self.local_rank)
                    dt = time.perf_counter() - t0
                    self.barrier()
                    st2 = detect_files_native([path], os.path.join(tmp, "nocsv"), spc, model=_cnn_weights() if w_host is not None else None,
                                              minibatch_size=mbs, chunk_minibatches=chunk, write_csv=False, device=self.local_rank)
                    out["file"] = {"reads": nf, "seconds": dt, "container_bytes": size, "tables": st["files"], "pass": st["pass"],
                                   "fail": st["fail"], "lost": st["lost"], "stage_busy_s": {k: st[k] for k in ("reader_busy_s", "writer_wait_gpu_s", "writer_busy_s")},
                                   "seconds_without_tables": st2["seconds"], "storage": os.path.dirname(path)}
                finally:
                    shutil.rmtree(tmp, ignore_errors=True)
            del host, rec_host, st_host
        del data, records
        torch.cuda.empty_cache()
        return out

    # -------------------------------------------------------------------------------------------------
    def reduce(self, out, args):
        """max-over-ranks times, summed counts -> the numbers of the JSON line"""
        tr = self.all_reduce
        n, steps = out["n"], out["steps"]
        ms_max = tr([out["ms"]], "max")[0]
        tot = tr([n, out["samples"], out["launches"], out["n_pass"], out["lost"]], "sum")
        res = {"value": tot[0] * steps / (ms_max / 1e3), "ms_per_step": ms_max / steps, "samples_per_sec": tot[1] * steps / (ms_max / 1e3),
               "gpu_launches": int(tot[2]), "pass_fraction": tot[3] / tot[0], "lost_minibatches": int(tot[4]), "total_reads": tot[0]}
        if out["e2e"]:
            e = out["e2e"]
            s_max, c_max = tr([e["seconds"], e["copy_seconds"]], "max")
            res["e2e"] = {"value": tot[0] * e["steps"] / s_max, "unit": "reads/s", "h2d_bytes_per_step": e["h2d"], "d2h_bytes_per_step": e["d2h"],
                          "steps": e["steps"], "records_identical_to_device_run": e["same"], "chunk_minibatches": e["chunk"],
                          "wire_bytes_per_sample": round(e["bytes_per_sample"], 4), "raw_int16_bytes_per_step": e["raw_int16_bytes"],
                          "h2d_GBps_per_gpu": e["h2d"] * e["steps"] / s_max / 1e9,
                          "copy_only": {"value": tot[0] * e["copy_steps"] / c_max, "unit": "reads/s", "h2d_GBps_per_gpu": e["h2d"] * e["copy_steps"] / c_max / 1e9,
                                        "what": "the same chunks with the kernels skipped: the host -> device ceiling of this box for this run"},
                          "api": "adb_detect_pipelined_svb_host (pinned host svb16 streams -> H2D -> device decode -> kernels -> D2H records)"}
            res["e2e"]["fraction_of_copy_ceiling"] = res["e2e"]["value"] / res["e2e"]["copy_only"]["value"]
        if out["file"]:
            f = out["file"]
            s_max, s2_max = tr([f["seconds"], f["seconds_without_tables"]], "max")
            reads = tr([f["reads"]], "sum")[0]
            res["file_to_csv"] = {"value": reads / s_max, "unit": "reads/s", "reads_per_gpu": f["reads"], "container_bytes_per_gpu": f["container_bytes"],
                                  "tables_rank0": f["tables"], "lost_rank0": f["lost"], "stage_busy_s_rank0": f["stage_busy_s"],
                                  "value_without_tables": reads / s2_max, "storage": f["storage"],
                                  "api": "adb_detect_files (ADBSIG02 svb16 container -> pinned ring -> H2D -> decode -> kernels -> records -> CSV tables)"}
        return res

    def roofline(self, out, args, chem):
        tim, flat, n, samples, steps = out["tim"], out["flat"], out["n"], out["samples"], out["steps"]
        peaks = self.peaks
        peak = float(peaks.get("hbm_gbs", 6650.0))
        per_cls = {CLS_NAMES[i]: {"ms": tim[2 * i], "launches": int(tim[2 * i + 1])} for i in range(8) if tim[2 * i + 1] > 0}
        alg_bytes_per_step = 2.0 * samples + (8 + 4 + 512) * n

        def hbm_view(dom):
            # classes 0 / 3 stream the first max_obs_trace samples of every read once per launch; the others the window
            launches_dom = max(int(tim[2 * dom + 1]), 1)
            if dom in (1, 6, 7):  # classes of several unlike kernels per step: the unit is the class's time per step
                launches_dom = steps
            # one launch covers at most 256 minibatches (adb_detect_dev cuts larger calls): bytes per launch follow
            launches_per_step = max(1, launches_dom // steps)
            # classes 0 / 3 stream the first max_obs_trace samples of every read, the others the whole preload window
            alg_launch = (2.0 * out["trace_samples"] if dom in (0, 3) else alg_bytes_per_step) / launches_per_step
            avg_ms = tim[2 * dom] / launches_dom
            ach = alg_launch / (avg_ms / 1e3) / 1e9 if avg_ms > 0 else 0.0
            return {"kernel": CLS_NAMES[dom], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "algorithmic_bytes_per_launch": alg_launch, "avg_launch_ms": avg_ms, "launches_per_step": launches_per_step}

        dom = max(range(8), key=lambda i: tim[2 * i])
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            traffic = tj.get(f"{CLS_NAMES[dom]} ({chem})", tj.get(CLS_NAMES[dom] if chem == "rna002" else "cnn" if dom == 5 else None))
        except Exception:
            pass
        whole = (alg_bytes_per_step / ((out["ms"] / steps) / 1e3) / 1e9) / peak
        if dom == 5:
            # the tensor-core convolutions (cnn_conv64_tc_kernel<2>, <3>) are a dense contraction: 64 556 800 algorithmic
            # flop per read (SURVEY 8d); every product is executed as three fp16 split products
            tpeak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 2250.0)))
            tf = 64556800.0 * n * steps / (tim[10] / 1e3) / 1e12 if tim[10] > 0 else 0.0
            nontensor = max((i for i in range(8) if i != 5), key=lambda i: tim[2 * i])
            roof = {"bound": "tensor", "kernel": CLS_NAMES[5], "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak,
                    "avg_launch_ms": tim[10] / max(int(tim[11]), 1), "executed_tensor_flops_factor": 3.0,
                    "algorithmic_flops_per_launch": 64556800.0 * n * steps / max(int(tim[11]), 1),
                    "hbm_view_same_class": hbm_view(5), "hbm_view_dominant_non_tensor_class": hbm_view(nontensor)}
        else:
            roof = dict(bound="hbm", **hbm_view(dom))
        roof.update({"traffic": traffic, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback", "kernel_classes": per_cls,
                     "whole_step_frac": whole})
        return roof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU (default: 1 000 000 RNA004, 100 000 RNA002)")
    ap.add_argument("--chemistry", default="rna004")
    ap.add_argument("--minibatch", type=int, default=1000)
    ap.add_argument("--chunk-batches", type=int, default=0,
                    help="minibatches per full-size H2D chunk of the pipelined ingest (default: 16, CNN path 32)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the RNA002 / start-peak blocks")
    ap.add_argument("--file-reads", type=int, default=400000, help="reads per GPU of the file -> CSV block (0: skip, -1: all)")
    ap.add_argument("--file-dir", default="", help="where the container and the tables go (default: the system temp dir)")
    ap.add_argument("--profile-steps-only", action="store_true",
                    help="for ncu launch lists: device-resident steps only")
    ap.add_argument("--stress", action="store_true",
                    help="BASELINE config 4: poly(A) lengths up to the preload limit, 10 %% of the reads ending early")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step of the main workload returned (records, status) to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    chem = args.chemistry.lower()
    reads = args.reads or DEFAULT_READS.get(chem, 100000)

    rank, world = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1)
    local_rank = _env_int("LOCAL_RANK", 0)
    cores = os.cpu_count() or 1

    from adapted_b200.config import flatten_config, get_chemistry_specific_config

    preload = flatten_config(get_chemistry_specific_config(chem))["sig_preload_size"]
    config = workload_config(chem, reads, args.minibatch, max(world, args.gpus), args.stress, preload)

    # ---------------- reference arm: CPU only, rank 0 only ----------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        r = cpu_arm(chem, args.steps, args.warmup, args.minibatch, cores, args.stress)
        sample = (f"{r['reads_per_step']} reads per step = {cores} minibatches of {args.minibatch} reads over a pool of {cores} worker "
                  f"processes (wall clock around the pool, {r['steps']} steps of {r['s_per_step']:.1f} s), "
                  + ("KleistLab/ADAPTed v0.2.4 executed from oracle/_ref/pkg (combined_detect_cnn / combined_detect_llr2, stock torch threads)"
                     if r["kind"] == "reference" else "oracle/detect_ref.py (port)"))
        line = {"impl": "reference", "metric": METRIC, "value": r["reads_per_s"], "unit": "reads/s", "n_gpus": args.gpus,
                "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["s_per_step"] * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 traces / f32 statistics", "data": "synthetic",
                "config": config, "samples_per_sec": r["samples_per_s"], "pass_fraction": r["pass_fraction"],
                "cpu_baseline": {"value": r["reads_per_s"], "unit": "reads/s", "cores": cores, "kind": r["kind"], "sample": sample,
                                 "libraries": lib_versions()},
                "e2e": {"value": r["reads_per_s"], "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ---------------- our arm ----------------
    import torch

    if not torch.cuda.is_available():
        sys.exit("bench.py needs a CUDA device (adapted_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    host_info = bind_to_gpu_local_cpus(local_rank) if world > 1 else {"local_cpulist": None, "bound": False, "numa_node": None}
    dist = None
    if world > 1:
        # the path has no collective (SURVEY 8e): ranks only meet at barriers and when the timings are reduced -- over
        # gloo on the host, no NCCL communicator exists in this program
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo")

    def barrier():
        if dist is not None:
            dist.barrier()

    def all_reduce(vals, op):
        t = torch.tensor(vals, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return [float(v) for v in t]

    R = Runner(local_rank, rank, world, barrier, all_reduce)
    sampler = ClockSampler(local_rank)
    if rank == 0:  # one nvidia-smi process every 100 ms per rank would load the host of an 8-GPU box
        sampler.start()
    out = R.run(chem, reads, args, label="main")
    sampler.stop_flag = True
    main_res = R.reduce(out, args)
    roof = R.roofline(out, args, chem)
    line = None
    if rank == 0:
        sampler.join(timeout=2)
        line = {"metric": METRIC, "value": main_res["value"], "unit": "reads/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64 traces / f32 statistics / fp16-split tensor-core convolutions / i16 input", "data": "synthetic",
                "config": config, "samples_per_sec": main_res["samples_per_sec"], "e2e": main_res.get("e2e"),
                "gpu_launches": main_res["gpu_launches"], "roofline": roof, "clocks": sampler.summary(),
                "pass_fraction": main_res["pass_fraction"], "lost_minibatches": main_res["lost_minibatches"],
                "global_select_handovers_rank0": out["gsel_fallbacks"], "validate_handovers_rank0": out["val_handovers"],
                "host": dict(host_info, cores=cores, barrier="gloo" if world > 1 else None)}
        if "file_to_csv" in main_res:
            line["file_to_csv"] = main_res["file_to_csv"]

    # ---------------- secondary: BASELINE configs[1] (RNA002 / LLR + its start-peak companion) ----------------
    if not args.no_secondary and not args.profile_steps_only and chem == "rna004" and not args.stress:
        from adapted_b200.config import start_peak_config

        n2 = DEFAULT_READS["rna002"]
        o2 = R.run("rna002", n2, args, label="secondary")
        r2 = R.reduce(o2, args)
        roof2 = R.roofline(o2, args, "rna002")
        o3 = R.run("rna002", n2, args, spc=start_peak_config("rna002"), e2e=False, label="start_peak")
        r3 = R.reduce(o3, args)
        if rank == 0:
            pre2 = flatten_config(get_chemistry_specific_config("rna002"))["sig_preload_size"]
            line["secondary"] = {"config": workload_config("rna002", n2, args.minibatch, world, False, pre2), "value": r2["value"], "unit": "reads/s",
                                 "ms_per_step": r2["ms_per_step"], "samples_per_sec": r2["samples_per_sec"], "e2e": r2.get("e2e"),
                                 "gpu_launches": r2["gpu_launches"], "roofline": roof2, "pass_fraction": r2["pass_fraction"],
                                 "global_select_handovers_rank0": o2["gsel_fallbacks"], "validate_handovers_rank0": o2["val_handovers"]}
            per_cls3 = {CLS_NAMES[i]: {"ms": o3["tim"][2 * i], "launches": int(o3["tim"][2 * i + 1])} for i in range(8) if o3["tim"][2 * i + 1] > 0}
            line["secondary_start_peak"] = {"config": dict(workload_config("rna002", n2, args.minibatch, world, False, pre2),
                                                           workload="RNA002 start-peak companion configuration (combined_detect_start_peak: "
                                                                    "start-peak primary, MVS check off, median-shift check on), minibatches of 1000 reads"),
                                            "value": r3["value"], "unit": "reads/s", "ms_per_step": r3["ms_per_step"],
                                            "gpu_launches": r3["gpu_launches"], "pass_fraction": r3["pass_fraction"], "kernel_classes": per_cls3}

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline and not args.profile_steps_only:
            # the CPU arm runs in a fresh interpreter (no CUDA context, no torch thread pools inherited by the workers)
            def cpu(chem_):
                try:
                    o = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--chemistry", chem_,
                                        "--steps", "1", "--warmup", "1"] + (["--stress"] if args.stress else []),
                                       capture_output=True, text=True, timeout=600).stdout
                    ref = json.loads(o.strip().splitlines()[-1])
                    cb = ref["cpu_baseline"]
                    cb["samples_per_sec"] = ref["samples_per_sec"]
                    return cb
                except Exception as e:  # noqa: BLE001 -- the GPU line must still be printed
                    return {"value": None, "unit": "reads/s", "cores": cores, "kind": "reference", "sample": f"failed: {type(e).__name__}: {e}"}

            line["cpu_baseline"] = cpu(chem)
            if "secondary" in line:
                line["secondary"]["cpu_baseline"] = cpu("rna002")
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main() or 0)
