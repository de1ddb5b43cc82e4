"""Load tests/golden/*.json.gz (written by oracle/make_golden.py, each file naming where its expected values came from
where that is not the executed reference)."""
from __future__ import annotations

import gzip
import hashlib
import json
import os
from typing import Any, Dict

import numpy as np

from adapted_b200.config import config_from_dict
from adapted_b200.synth import make_reads

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

SEAM_CASES = {
    "llr2": ["llr_rna002_basic", "llr_rna002_stress", "llr_rna002_lost_minibatch", "llr_rna002_overwrite",
             "llr_rna002_overwrite_stress"],
    "cnn": ["cnn_rna004_basic", "cnn_rna004_short", "cnn_rna004_stress", "cnn_rna004_overwrite",
            "cnn_rna004_overwrite_short"],
    "start_peak": ["start_peak_rna004_basic", "start_peak_rna004_poisoned"],
}


def _decode(v):
    if isinstance(v, dict) and "array" in v:
        return np.asarray(v["array"], dtype=v["dtype"])
    return v


def load_case(name: str) -> Dict[str, Any]:
    with gzip.open(os.path.join(GOLDEN, name + ".json.gz"), "rb") as f:
        rec = json.loads(f.read().decode())
    if "results" in rec:
        rec["results"] = [{k: _decode(v) for k, v in r.items()} for r in rec["results"]]
    cfg = rec["config"]
    for sec in cfg.values():
        for k, v in sec.items():
            if isinstance(v, list):
                sec[k] = tuple(v)
    rec["spc"] = config_from_dict(cfg)
    batch = make_reads(rec["n"], rec["chemistry"], rec["m"], seed=rec["seed"], **rec["gen_kwargs"])
    sha = hashlib.sha256(batch.adc.tobytes()).hexdigest()
    assert sha == rec["adc_sha256"], "synthetic generator drifted: golden inputs cannot be regenerated"
    rec["batch"] = batch
    return rec


def load_cnn_weights() -> Dict[str, np.ndarray]:
    with np.load(os.path.join(GOLDEN, "cnn_weights_rna004_130bps_v0.2.4.npz")) as z:
        return {k: z[k] for k in z.files}


def array_digest(a) -> str:
    """Digest of a float64 array in which every NaN counts as the same NaN and -0.0 as 0.0: two arrays have the same
    digest exactly when np.array_equal(a, b, equal_nan=True) holds (up to hash collisions)."""
    a = np.asarray(a, dtype=np.float64) + 0.0
    a[np.isnan(a)] = np.nan
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()[:32]


C_LLR_CALLS = os.path.join(GOLDEN, "c_llr_calls.json.gz")
# the "source" of golden files written by oracle/make_golden.py --checks --from-oracle
ORACLE_SOURCE = "oracle/detect_ref.py (the oracle's own output, not the reference's)"


def warn_if_oracle_source(source: str, what: str) -> None:
    """A test that compares the oracle with recorded values checks it against the reference only where the reference
    wrote them; where the oracle did, say so in the test report."""
    if source == ORACLE_SOURCE:
        import warnings

        warnings.warn(f"{what}: the expected values are the oracle's own recorded output (no copy of the reference was "
                      "present when they were written), so this pins the oracle against change and does not check it "
                      "against the reference")


class KernelCalls:
    """Calls of the reference's compiled ``_c_llr`` module and what they returned (arrays as array_digest).  Given a
    module, every call is forwarded to it and recorded (oracle/make_golden.py --checks writes them to
    tests/golden/c_llr_calls.json.gz); without one, a call returns what was recorded for the same function and
    arguments, and ``source`` says where the recorded values came from."""

    def __init__(self, module=None):
        self.module, self.calls, self.source = module, {}, None
        if module is None:
            with gzip.open(C_LLR_CALLS, "rb") as f:
                doc = json.loads(f.read().decode())
            self.calls, self.source = doc["calls"], doc["source"]

    def __getattr__(self, fn):
        def call(x, *args):
            key = f"{fn}{args}:{array_digest(x)}"
            if self.module is None:
                return self.calls[key]
            out = getattr(self.module, fn)(x, *args)
            rec = [array_digest(v) for v in out] if isinstance(out, tuple) and isinstance(out[0], np.ndarray) else \
                array_digest(out) if isinstance(out, np.ndarray) else [int(v) for v in out]
            self.calls[key] = rec
            return rec
        return call


def load_stream_cases():
    """tests/golden/mvs_stream.json.gz: expected poly(A) starts of mean_var_shift_polyA_detect (executed reference)."""
    from adapted_b200.config import StreamingConfig

    with gzip.open(os.path.join(GOLDEN, "mvs_stream.json.gz"), "rb") as f:
        doc = json.loads(f.read().decode())
    out = []
    for c in doc["cases"]:
        p = StreamingConfig()
        for k, v in c["overrides"].items():
            setattr(p, k, tuple(v) if isinstance(v, list) else v)
        batch = make_reads(c["n"], c["chemistry"], c["m"], seed=c["seed"], **c["gen_kwargs"])
        assert hashlib.sha256(batch.adc.tobytes()).hexdigest() == c["adc_sha256"], "synthetic generator drifted"
        out.append(dict(name=c["name"], params=p, batch=batch, m=c["m"], want=np.asarray(c["polya_start"], dtype=np.int64)))
    return out
