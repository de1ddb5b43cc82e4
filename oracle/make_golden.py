"""Generate tests/golden/* by EXECUTING THE REFERENCE (TEST INFRASTRUCTURE; needs the reference's source).

    python -m oracle.make_golden
    python -m oracle.make_golden --checks [--from-oracle]   (the oracle-vs-reference tests' data, see write_checks)

Inputs are seeded synthetic minibatches from adapted_b200.synth.make_reads; each golden file records the
generator arguments and a sha256 of the generated ADC blob (so a drifting generator is detected instead
of silently comparing different inputs) together with what the reference returned for every
DetectResults field.  The reference is run from the patched scratch copy built by oracle/build_ref.py
with this container's numpy/scipy/torch/pandas (versions recorded in the file) and the
oracle's bottleneck stand-in (third-party, absent from the image: PARITY UNPINNED for that dependency).
"""
from __future__ import annotations

import gzip
import hashlib
import json
import logging
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from adapted_b200.config import config_as_dict  # noqa: E402
from adapted_b200.synth import make_reads  # noqa: E402
from oracle import build_ref  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

CASES = [
    # name, seam, chemistry/config, n, seed, generator kwargs
    ("llr_rna002_basic", "llr2", "rna002", 48, 11, {}),
    ("llr_rna002_stress", "llr2", "rna002", 32, 12, {"stress": True}),
    ("llr_rna002_lost_minibatch", "llr2", "rna002", 8, 13, {"short_frac": 1.0}),
    ("cnn_rna004_basic", "cnn", "rna004", 48, 21, {}),
    ("cnn_rna004_short", "cnn", "rna004", 64, 22, {"short_frac": 0.3}),
    ("cnn_rna004_stress", "cnn", "rna004", 32, 23, {"stress": True}),
    ("start_peak_rna004_basic", "start_peak", "rna004", 48, 31, {}),
    ("start_peak_rna004_poisoned", "start_peak", "rna004", 8, 32, {"short_frac": 0.5}),
    # mvs_detect_overwrite = true (SURVEY f3): mean_var_shift_polyA_detect_at_loc moves adapter_end
    ("llr_rna002_overwrite", "llr2", "rna002", 48, 41, {}, "overwrite"),
    ("llr_rna002_overwrite_stress", "llr2", "rna002", 32, 42, {"stress": True}, "overwrite"),
    ("cnn_rna004_overwrite", "cnn", "rna004", 48, 43, {}, "overwrite"),
    ("cnn_rna004_overwrite_short", "cnn", "rna004", 32, 44, {"short_frac": 0.3}, "overwrite"),
]


JOB = dict(n=150, seed=61, minibatch=50, batch_size_output=64)  # file-level job (ingest.detect_file)
STREAM_WINDOW = 20000  # samples of the read-until cache looked at per read
STREAM_CASES = [
    # name, chemistry of the synthetic reads, n, seed, generator kwargs, StreamingConfig overrides
    ("defaults_rna002", "rna002", 48, 51, {}, {}),
    ("defaults_rna004", "rna004", 48, 52, {}, {}),
    ("stress_short", "rna002", 48, 53, {"stress": True, "short_frac": 0.3}, {}),
    # a tight median window and local range reject the first matches: the offset loop advances by the step
    ("retry_loop", "rna004", 48, 54, {}, {"min_obs_adapter": 500, "pA_mean_range": [60.0, 130.0], "pA_var_range": [None, 70.0],
                                          "polyA_med_range": [100.3, 115.7], "polyA_local_range": [0.0, 8.3],
                                          "search_increment_step": 37, "median_shift_range": [12.5, None]}),
    ("odd_windows", "rna002", 32, 55, {}, {"pA_mean_window": 33, "pA_var_window": 64, "median_shift_window": 700,
                                           "polyA_window": 150, "min_obs_post_loc": 1200, "polyA_local_range": [None, None]}),
]


def read_ids_for(name: str, n: int):
    """deterministic uuid-shaped read ids (what pod5 gives the reference, file_proc.py:175)"""
    import uuid

    h = int.from_bytes(hashlib.sha256(name.encode()).digest()[:8], "little")
    return [str(uuid.UUID(int=(h << 64) | i)) for i in range(n)]


def reference_csvs(res, read_ids):
    """What worker_detect_on_preloaded_signals + the saver threads write for one minibatch (file_proc.py:246-266,
    418-457; output.py:26-51): the pass table and the fail table as text."""
    import tempfile

    from adapted.container_types import ReadResult
    from adapted.output import save_detected_boundaries

    rr = [ReadResult(read_id=i, success=r.success, fail_reason=r.fail_reason, detect_results=r)
          for r, i in zip(res, read_ids)]
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for key, sel, with_reason in (("csv_pass", [r for r in rr if r.success], False),
                                      ("csv_fail", [r for r in rr if not r.success], True)):
            fn = os.path.join(d, key + ".csv")
            save_detected_boundaries(sel, fn, save_fail_reasons=with_reason)
            with open(fn, newline="") as f:
                out[key] = f.read()
    return out


def _jsonable(v):
    if v is None or isinstance(v, (str, bool)):
        return v
    if isinstance(v, np.ndarray):
        return {"array": v.tolist(), "dtype": str(v.dtype)}
    if isinstance(v, (np.bool_,)):
        return bool(v)
    if isinstance(v, (int, np.integer)):
        return int(v)
    if isinstance(v, (float, np.floating)):
        return float(v)  # float32 -> float64 is exact; repr round-trips
    raise TypeError(type(v))


def reference_configs():
    from adapted.config.base import nested_config_from_dict
    from adapted.config.sig_proc import SigProcConfig, config_name_to_dict, get_chemistry_specific_config

    out = {}
    for chem in ("rna002", "rna004"):
        spc = get_chemistry_specific_config(chem)
        spc.update_primary_method()
        spc.update_sig_preload_size()
        out[("plain", chem)] = spc
        d = config_name_to_dict({"rna002": "rna002_70bps@v0.2.4", "rna004": "rna004_130bps@v0.2.4"}[chem])
        d["rna_start_peak"]["detect_rna_start_peak"] = True
        d["llr_boundaries"]["llr_detect"] = False
        d["cnn_boundaries"]["cnn_detect"] = False
        d["mvs_polya"]["mvs_detect_check"] = False
        d["med_shift"]["detect_med_shift"] = True
        sp = nested_config_from_dict(d, SigProcConfig)
        sp.update_primary_method()
        sp.update_sig_preload_size()
        out[("start_peak", chem)] = sp
        d = config_name_to_dict({"rna002": "rna002_70bps@v0.2.4", "rna004": "rna004_130bps@v0.2.4"}[chem])
        d["mvs_polya"]["mvs_detect_overwrite"] = True
        ow = nested_config_from_dict(d, SigProcConfig)
        ow.update_primary_method()
        ow.update_sig_preload_size()
        out[("overwrite", chem)] = ow
    return out


CHECK_CASES = [
    # the fresh seeds of tests/test_oracle_vs_reference.py: name, seam, chemistry, n, seed, generator kwargs
    ("check_llr_rna002_101", "llr2", "rna002", 40, 101, {}),
    ("check_llr_rna002_102", "llr2", "rna002", 40, 102, {"stress": True}),
    ("check_cnn_rna004_201", "cnn", "rna004", 60, 201, {}),
    ("check_cnn_rna004_202", "cnn", "rna004", 60, 202, {"short_frac": 0.3}),
    ("check_cnn_rna004_203", "cnn", "rna004", 60, 203, {"stress": True}),
    ("check_start_peak_rna004_301", "start_peak", "rna004", 40, 301, {}),
    ("check_start_peak_rna004_302", "start_peak", "rna004", 40, 302, {"short_frac": 0.3}),
]


def write_checks(from_oracle: bool = False):
    """tests/golden/check_*.json.gz and c_llr_calls.json.gz: what the reference returns for the inputs of
    tests/test_oracle_vs_reference.py and tests/test_oracle_llr.py, which compare the oracle with them where no copy of
    the reference is present.  Needs such a copy (its source, or a prebuilt oracle/_ref).  Only with from_oracle
    (--from-oracle) are the oracle's own results recorded instead, and every file then says so in its "source"."""
    from oracle import detect_ref
    from tests import test_oracle_llr as t
    from tests.golden_io import C_LLR_CALLS, KernelCalls, ORACLE_SOURCE, load_cnn_weights

    logging.disable(logging.CRITICAL)
    warnings.simplefilter("ignore")
    live = (build_ref.reference_present() or build_ref.package_present()) and build_ref.kernel_available()
    if not live and not from_oracle:
        sys.exit("--checks runs the reference: build oracle/_ref from its source first (python -m oracle.build_ref); "
                 "--from-oracle records the oracle's own results instead")
    if live:
        build_ref.import_reference()
        from adapted.detect import combined
        from adapted.detect.cnn import load_cnn_model

        cfgs = reference_configs()
        model = load_cnn_model(cfgs[("plain", "rna004")].cnn_boundaries.model_name)
        kernel, source = build_ref.load_c_llr(), "KleistLab/ADAPTed v0.2.4 (executed)"
    else:
        from types import SimpleNamespace

        from adapted_b200.config import get_chemistry_specific_config, start_peak_config

        cfgs = {(v, c): (start_peak_config(c) if v == "start_peak" else get_chemistry_specific_config(c))
                for v in ("plain", "start_peak") for c in ("rna002", "rna004")}
        # the oracle's restatement under the names of the reference's _c_llr module
        kernel = SimpleNamespace(c_llr_trace=detect_ref.llr_trace, c_llr_detect_adapter=detect_ref.llr_detect_adapter,
                                 c_llr_detect_adapter_polya=detect_ref.llr_detect_adapter_polya,
                                 c_llr_detect_adapter_polya_trace=detect_ref.llr_boundary_traces,
                                 c_llr_boundary_traces=detect_ref.llr_boundary_traces)
        source = ORACLE_SOURCE
    for name, seam, chem, n, seed, kw in CHECK_CASES:
        spc = cfgs[("start_peak" if seam == "start_peak" else "plain", chem)]
        batch = make_reads(n, chem, spc.sig_preload_size, seed=seed, **kw)
        x = batch.to_dense_pa()
        if seam == "llr2":
            res = (combined.combined_detect_llr2 if live else detect_ref.detect_llr2)(x, batch.full_lens, spc)
        elif seam == "cnn":
            res = combined.combined_detect_cnn(x.copy(), batch.full_lens, model, spc) if live else \
                detect_ref.detect_cnn(x, batch.full_lens, load_cnn_weights(), spc)
        else:
            res = (combined.combined_detect_start_peak if live else detect_ref.detect_start_peak)(x, batch.full_lens, spc)
        res = [r if isinstance(r, dict) else r.to_dict() for r in (res if isinstance(res, list) else [res])]
        rec = dict(name=name, seam=seam, chemistry=chem, n=n, seed=seed, gen_kwargs=kw, m=int(spc.sig_preload_size),
                   adc_sha256=hashlib.sha256(batch.adc.tobytes()).hexdigest(), config=config_as_dict(spc), source=source,
                   results=[{k: _jsonable(v) for k, v in r.items()} for r in res])
        with gzip.GzipFile(os.path.join(GOLDEN, name + ".json.gz"), "wb", mtime=0) as f:
            f.write(json.dumps(rec).encode())
    # the test functions themselves make the kernel calls, so the recorded arguments are exactly theirs
    rec = KernelCalls(kernel)
    for fn, params in ((t.test_full_trace_bit_identical, [(s,) for s in range(6)]),
                       (t.test_early_stop_variants_bit_identical, [(s, k) for s in range(6) for k in (1, 2, 5)]),
                       (t.test_degenerate_variances, [()]),
                       (t.test_legacy_three_split_detectors_match_reference_kernel, [(s,) for s in range(4)])):
        for p in params:
            fn(rec, *p)
    with gzip.GzipFile(C_LLR_CALLS, "wb", mtime=0) as f:
        f.write(json.dumps(dict(source=source, calls=rec.calls)).encode())
    print(f"{len(CHECK_CASES)} seam checks and {len(rec.calls)} kernel calls from {source}")


def main():
    if "--checks" in sys.argv:
        return write_checks(from_oracle="--from-oracle" in sys.argv)
    if not build_ref.reference_present():
        sys.exit("needs /root/reference")
    build_ref.import_reference()
    logging.disable(logging.CRITICAL)
    warnings.simplefilter("ignore")
    import pandas
    import scipy
    import torch
    from adapted.detect.cnn import load_cnn_model
    from adapted.detect.combined import combined_detect_cnn, combined_detect_llr2, combined_detect_start_peak

    os.makedirs(GOLDEN, exist_ok=True)
    cfgs = reference_configs()
    model = load_cnn_model(cfgs[("plain", "rna004")].cnn_boundaries.model_name)
    np.savez_compressed(
        os.path.join(GOLDEN, "cnn_weights_rna004_130bps_v0.2.4.npz"),
        **{k: v.detach().numpy() for k, v in model.state_dict().items()},
    )
    versions = dict(numpy=np.__version__, scipy=scipy.__version__, torch=torch.__version__,
                    pandas=pandas.__version__, reference="KleistLab/ADAPTed v0.2.4",
                    bottleneck="oracle.bn_restate stand-in (unpinned)")
    for name, seam, chem, n, seed, kw, *variant in CASES:
        spc = cfgs[(variant[0] if variant else "start_peak" if seam == "start_peak" else "plain", chem)]
        batch = make_reads(n, chem, spc.sig_preload_size, seed=seed, **kw)
        x = batch.to_dense_pa()
        rec = dict(name=name, seam=seam, chemistry=chem, n=n, seed=seed, gen_kwargs=kw,
                   m=int(spc.sig_preload_size), adc_sha256=hashlib.sha256(batch.adc.tobytes()).hexdigest(),
                   config=config_as_dict(spc), versions=versions)
        try:
            if seam == "llr2":
                res = combined_detect_llr2(x, batch.full_lens, spc)
            elif seam == "cnn":
                res = combined_detect_cnn(x, batch.full_lens, model, spc)
            else:
                res = combined_detect_start_peak(x, batch.full_lens, spc)
            if not isinstance(res, list):
                res = [res]
            rec["results"] = [{k: _jsonable(v) for k, v in r.to_dict().items()} for r in res]
            rec["read_ids"] = read_ids_for(name, n)
            rec.update(reference_csvs(res, rec["read_ids"]))
            n_pass = sum(bool(r.success) for r in res)
        except Exception as e:  # whole-minibatch failure (SURVEY A.11)
            rec["raises"] = dict(type=type(e).__name__, message=str(e))
            n_pass = -1
        path = os.path.join(GOLDEN, name + ".json.gz")
        with gzip.GzipFile(path, "wb", mtime=0) as f:
            f.write(json.dumps(rec).encode())
        print(f"{name}: n={n} pass={n_pass} -> {os.path.relpath(path, ROOT)} ({os.path.getsize(path)} B)")

    # a whole job: three minibatches through the seam + the saver threads' batching (file_proc.py:246-266,312-351)
    from adapted.container_types import ReadResult
    from adapted.output import save_detected_boundaries

    spc = cfgs[("plain", "rna002")]
    jb = make_reads(JOB["n"], "rna002", spc.sig_preload_size, seed=JOB["seed"], stress=True)
    jx = jb.to_dense_pa()
    jids = read_ids_for("job", JOB["n"])
    queues = {"pass": [], "fail": []}
    for s in range(0, JOB["n"], JOB["minibatch"]):
        res = combined_detect_llr2(jx[s: s + JOB["minibatch"]], jb.full_lens[s: s + JOB["minibatch"]], spc)
        rr = [ReadResult(read_id=i, success=r.success, fail_reason=r.fail_reason, detect_results=r)
              for r, i in zip(res, jids[s: s + JOB["minibatch"]])]
        queues["fail"] += [r for r in rr if not r.success]
        queues["pass"] += [r for r in rr if r.success]
    files = {}
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        for key, stem in (("pass", "boundaries/detected_boundaries"), ("fail", "failed_reads/failed_reads")):
            for bi, s in enumerate(range(0, len(queues[key]), JOB["batch_size_output"])):
                fn = os.path.join(d, "t.csv")
                save_detected_boundaries(queues[key][s: s + JOB["batch_size_output"]], fn, save_fail_reasons=key == "fail")
                with open(fn, newline="") as f:
                    files[f"{stem}_{bi}.csv"] = f.read()
    with gzip.GzipFile(os.path.join(GOLDEN, "job_llr_rna002.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(dict(versions=versions, job=JOB, m=int(spc.sig_preload_size), config=config_as_dict(spc),
                                adc_sha256=hashlib.sha256(jb.adc.tobytes()).hexdigest(), read_ids=jids, files=files)).encode())
    print("job_llr_rna002:", {k: len(v) for k, v in queues.items()}, sorted(files))

    # streaming poly(A) detector (mean_var_shift_polyA_detect, mvs.py:341-426): expected start per read
    from adapted.config.sig_proc import StreamingConfig
    from adapted.detect.mvs import mean_var_shift_polyA_detect

    stream = []
    for name, chem, n, seed, kw, overrides in STREAM_CASES:
        p = StreamingConfig()
        for k, v in overrides.items():
            setattr(p, k, tuple(v) if isinstance(v, list) else v)
        batch = make_reads(n, chem, STREAM_WINDOW, seed=seed, **kw)
        x = batch.to_dense_pa()
        lens = np.minimum(batch.full_lens, STREAM_WINDOW)
        want = [int(mean_var_shift_polyA_detect(x[i, : lens[i]], p)) for i in range(n)]
        stream.append(dict(name=name, chemistry=chem, n=n, seed=seed, gen_kwargs=kw, overrides=overrides,
                           m=STREAM_WINDOW, adc_sha256=hashlib.sha256(batch.adc.tobytes()).hexdigest(),
                           polya_start=want))
        print(f"mvs_stream {name}: found {sum(w > 0 for w in want)}/{n}")
    with gzip.GzipFile(os.path.join(GOLDEN, "mvs_stream.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(dict(versions=versions, cases=stream)).encode())

    # kernel-level golden vectors for c_llr_trace incl. the early-stop dispatch branches
    from adapted.detect._c_llr import c_llr_trace

    rng = np.random.default_rng(99)
    arrays = {}
    for i in range(6):
        nn = int(rng.integers(300, 1650))
        k1, k2 = sorted(rng.integers(20, nn - 20, size=2))
        sig = np.concatenate([rng.normal(-1, 1, k1), rng.normal(1.5, .3, k2 - k1), rng.normal(.5, 1.4, nn - k2)])
        sig = sig.astype(np.float32).astype(np.float64)
        arrays[f"x{i}"] = sig
        for tag, args in (("full", (0, nn - 1, 5, 5, 1, 0, 0, 0, 0, 0, 0)),
                          ("aes", (0, nn - 1, 5, 5, 1, 1, 100, 20, 0, 0, 0)),
                          ("pes", (0, nn - 1, 5, 5, 1, 1, 100, 20, 1, 30, 10)),
                          ("tail", (int(k1), nn - 1, 1, 1, 1, 0, 0, 0, 0, 0, 0))):
            arrays[f"g{i}_{tag}"] = c_llr_trace(sig, *args, 0)
            arrays[f"a{i}_{tag}"] = np.asarray(args, dtype=np.int64)
    np.savez_compressed(os.path.join(GOLDEN, "c_llr_trace.npz"), **arrays)
    print("c_llr_trace.npz written")


if __name__ == "__main__":
    main()
