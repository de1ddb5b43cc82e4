"""Differential test of the oracle against the reference on fresh seeds, every DetectResults field compared exactly.
Where a copy of the reference is present (its source, or a prebuilt oracle/_ref) it is run here.  Elsewhere the
presets come from the configs the executed reference wrote into its goldens, and the results from
tests/golden/check_*.json.gz (oracle/make_golden.py --checks).  Those files name their source: where it is the oracle's
own earlier output rather than the reference's, these tests pin the oracle against change instead of checking it
against the reference, and they warn."""
import copy
import logging
import warnings

import pytest

from adapted_b200.config import config_as_dict, config_from_dict, flatten_config, get_chemistry_specific_config, start_peak_config
from oracle import build_ref, detect_ref
from tests.golden_io import load_case, load_cnn_weights, warn_if_oracle_source
from tests.helpers import diff_results

# the reference's presets as the executed reference wrote them into its goldens (oracle/make_golden.py CASES)
PRESET_GOLDEN = {"rna002": ("llr_rna002_basic", "llr2"), "rna004": ("cnn_rna004_basic", "cnn")}
START_PEAK_GOLDEN = {"rna004": "start_peak_rna004_basic"}


@pytest.fixture(scope="module")
def ref():
    """the running reference (configs, seam functions, CNN model), or None where no copy of it is present"""
    if not (build_ref.reference_present() or build_ref.package_present()):
        return None
    build_ref.import_reference()
    logging.disable(logging.CRITICAL)
    warnings.simplefilter("ignore")
    from adapted.detect import combined
    from adapted.detect.cnn import load_cnn_model
    from oracle.make_golden import reference_configs

    cfgs = reference_configs()
    return dict(cfgs=cfgs, combined=combined, model=load_cnn_model(cfgs[("plain", "rna004")].cnn_boundaries.model_name))


def _reference_start_peak(plain):
    """the start-peak companion built from the reference's preset like oracle.make_golden.reference_configs does (no
    golden of the executed reference holds the rna002 one)"""
    d = copy.deepcopy(config_as_dict(plain))
    d["rna_start_peak"]["detect_rna_start_peak"] = True
    d["llr_boundaries"]["llr_detect"] = False
    d["cnn_boundaries"]["cnn_detect"] = False
    d["mvs_polya"]["mvs_detect_check"] = False
    d["med_shift"]["detect_med_shift"] = True
    return config_from_dict(d)


@pytest.mark.parametrize("chem", ["rna002", "rna004"])
def test_presets_match_reference_toml(ref, chem):
    if ref is not None:
        want, want_sp = flatten_config(ref["cfgs"][("plain", chem)]), flatten_config(ref["cfgs"][("start_peak", chem)])
    else:
        name, seam = PRESET_GOLDEN[chem]
        rec = load_case(name)
        want = flatten_config(rec["spc"])
        assert (want["sig_preload_size"], want["primary_method"]) == (rec["m"], {"llr2": 0, "cnn": 1}[seam])
        if chem in START_PEAK_GOLDEN:
            sp = load_case(START_PEAK_GOLDEN[chem])
            want_sp = flatten_config(sp["spc"])
            assert (want_sp["sig_preload_size"], want_sp["primary_method"]) == (sp["m"], 2)
        else:
            want_sp = flatten_config(_reference_start_peak(rec["spc"]))
    assert flatten_config(get_chemistry_specific_config(chem)) == want
    assert flatten_config(start_peak_config(chem)) == want_sp


def _case(ref, name, seam, variant, n, seed, kw):
    """the inputs of a case and what the reference returns for them (run here, or as recorded)"""
    rec = load_case(name)
    assert (rec["n"], rec["seed"], rec["gen_kwargs"]) == (n, seed, kw)
    x, lens = rec["batch"].to_dense_pa(), rec["batch"].full_lens
    if ref is None:
        warn_if_oracle_source(rec.get("source"), f"tests/golden/{name}.json.gz")
        return x, lens, rec["results"]
    spc, comb = ref["cfgs"][(variant, rec["chemistry"])], ref["combined"]
    if seam == "llr2":
        return x, lens, comb.combined_detect_llr2(x, lens, spc)
    if seam == "cnn":
        return x, lens, comb.combined_detect_cnn(x.copy(), lens, ref["model"], spc)
    return x, lens, comb.combined_detect_start_peak(x, lens, spc)


@pytest.mark.parametrize("seed,kw", [(101, {}), (102, {"stress": True})])
def test_llr2_matches_reference(ref, seed, kw):
    x, lens, want = _case(ref, f"check_llr_rna002_{seed}", "llr2", "plain", 40, seed, kw)
    got = detect_ref.detect_llr2(x, lens, get_chemistry_specific_config("rna002"))
    assert diff_results(got, want, exact_floats=True) == []


@pytest.mark.parametrize("seed,kw", [(201, {}), (202, {"short_frac": 0.3}), (203, {"stress": True})])
def test_cnn_matches_reference(ref, seed, kw):
    x, lens, want = _case(ref, f"check_cnn_rna004_{seed}", "cnn", "plain", 60, seed, kw)
    got = detect_ref.detect_cnn(x.copy(), lens, load_cnn_weights(), get_chemistry_specific_config("rna004"))
    assert diff_results(got, want, exact_floats=True) == []


@pytest.mark.parametrize("seed,kw", [(301, {}), (302, {"short_frac": 0.3})])
def test_start_peak_matches_reference(ref, seed, kw):
    x, lens, want = _case(ref, f"check_start_peak_rna004_{seed}", "start_peak", "start_peak", 40, seed, kw)
    got = detect_ref.detect_start_peak(x, lens, start_peak_config("rna004"))
    assert diff_results(got, want, exact_floats=True) == []
