"""Drop-in test with the UNMODIFIED reference orchestrator (polyfuzz.PolyFuzz, copied into oracle/_ref by build()
when a reference checkout is readable): the B200 matchers are handed to PolyFuzz.match / fit /
transform / group exactly as the reference's own tests do (tests/test_polyfuzz.py:40-146)."""
import os
import sys

import numpy as np
import pandas as pd
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
REF = os.path.join(ROOT, "oracle", "_ref")
FROM = ["apple", "apples", "appl", "recal", "house", "similarity"]
TO = ["apple", "apples", "mouse"]


@pytest.fixture(scope="module")
def PolyFuzz():
    if not os.path.isdir(os.path.join(REF, "polyfuzz")):
        pytest.skip("oracle/_ref (the reference's polyfuzz package, copied by build()) not present")
    os.environ["PFZ_REFERENCE_ROOT"] = REF
    from oracle import ref_shim
    ref_shim.REFERENCE_ROOT = REF
    ref_shim.install()                      # stubs for the absent rapidfuzz / matplotlib / seaborn
    from polyfuzz import PolyFuzz as PF
    return PF


def _matchers():
    from polyfuzz_b200 import TFIDF, RapidFuzz, EditDistance
    return TFIDF, RapidFuzz, EditDistance


@pytest.mark.parametrize("which", ["tfidf", "rapidfuzz", "editdistance"])
def test_match_fit_transform(PolyFuzz, which):
    TFIDF, RapidFuzz, EditDistance = _matchers()
    import polyfuzz.models
    mk = {"tfidf": lambda: TFIDF(min_similarity=0, model_id="B200"), "rapidfuzz": lambda: RapidFuzz(model_id="B200"),
          "editdistance": lambda: EditDistance(model_id="B200", normalize=False)}[which]   # min-max of identical scores is 0/0 in the reference too
    m = mk()
    assert isinstance(m, polyfuzz.models.BaseMatcher)
    model = PolyFuzz(m).match(FROM, TO)
    matches = model.get_matches()
    assert isinstance(matches, pd.DataFrame) and len(matches) == 6 and list(matches.columns) == ["From", "To", "Similarity"]
    assert matches.Similarity.mean() > 0.3
    model = PolyFuzz(mk()).fit(FROM, TO)
    results = model.transform(TO)
    key = list(results.keys())[0]
    assert isinstance(results[key], pd.DataFrame) and results[key].Similarity.sum() > 0


def test_grouper_matches_reference_expectations(PolyFuzz):
    TFIDF, _, _ = _matchers()
    model = PolyFuzz(TFIDF(min_similarity=0)).match(FROM, TO)
    model.group(model=TFIDF(n_gram_range=(3, 3), min_similarity=0.75), link_min_similarity=0.75)
    matches = model.get_matches()
    assert list(matches.columns) == ["From", "To", "Similarity", "Group"]
    assert model.get_clusters() == {1: ["apples", "apple"]}                  # tests/test_polyfuzz.py:85-86
    assert model.get_cluster_mappings() == {"apples": 1, "apple": 1}
    model = PolyFuzz(TFIDF(min_similarity=0)).match(FROM, FROM)
    model.group(model=TFIDF(n_gram_range=(3, 3), min_similarity=0.75), link_min_similarity=0.75, group_all_strings=True)
    assert model.get_clusters() == {1: ["apples", "apple", "appl"]}          # tests/test_polyfuzz.py:99-100


def test_multiple_models_and_save_load(PolyFuzz, tmp_path):
    TFIDF, RapidFuzz, EditDistance = _matchers()
    matchers = [TFIDF(n_gram_range=(3, 3), min_similarity=0, model_id="TF-IDF"), TFIDF(n_gram_range=(3, 6), min_similarity=0, model_id="TF-IDF-36"),
                EditDistance(n_jobs=1, model_id="ED"), RapidFuzz(n_jobs=1, model_id="RF")]
    model = PolyFuzz(matchers).match(FROM, TO)
    for model_id in model.get_ids():
        assert isinstance(model.get_matches(model_id), pd.DataFrame)
    assert len(model.get_matches()) == len(matchers)
    with pytest.raises(ValueError):
        model.get_clusters()
    model = PolyFuzz(TFIDF(min_similarity=0, model_id="B200")).fit(FROM, TO)
    model.save(str(tmp_path / "pf.joblib"))                                   # polyfuzz/polyfuzz.py:429-441
    loaded = PolyFuzz.load(str(tmp_path / "pf.joblib"))
    a = model.transform(["appl", "mouses"]); b = loaded.transform(["appl", "mouses"])
    k = list(a.keys())[0]
    assert a[k].equals(b[k])
