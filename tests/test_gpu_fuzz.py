"""GPU parity tests of K3b (rapidfuzz token / partial / weighted scorers + extractOne arg-best) against oracle/fuzz.py,
which restates rapidfuzz 3.x and is pinned on rapidfuzz's published known answers (tests/golden/rapidfuzz_published.json).
Scores are the same IEEE double expressions: compared with ==; the arg-best index is the first maximum."""
import json
import os

import numpy as np
import pytest

from oracle import fuzz as ofuzz

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(scope="module")
def fz():
    from polyfuzz_b200 import fuzzy
    return fuzzy


def _oracle_best(frm, to, scorer, cutoff=0.0, exclude_self=False):
    fn = ofuzz.SCORERS[scorer]
    bi = np.full(len(frm), -1, np.int32); bs = np.zeros(len(frm))
    for i, q in enumerate(frm):
        r = ofuzz.extract_one(q, to, fn, cutoff, exclude_index=i if exclude_self else None)
        if r is not None:
            bi[i], bs[i] = r[2], r[1]
    return bi, bs


def test_published_vectors_through_the_gpu(fz, golden_dir):
    g = json.load(open(os.path.join(golden_dir, "rapidfuzz_published.json")))
    for v in g["scorers"]:
        bi, bs = fz.fuzz_argbest([v["a"]], [v["b"]], v["fn"])
        assert int(bi[0]) == 0 and float(bs[0]) == v["expect"], (v, float(bs[0]))
    for v in g["extract_one"]:
        bi, bs = fz.fuzz_argbest([v["query"]], v["choices"], v["scorer"])
        assert [v["choices"][int(bi[0])], float(bs[0]), int(bi[0])] == v["expect"]


def _titles(rng, n, words, lo=1, hi=6):
    out = []
    for _ in range(n):
        k = rng.integers(lo, hi + 1)
        ws = list(rng.choice(words, k))
        if rng.random() < 0.15:
            ws.append(ws[0])                                   # duplicate token: U(s) != S(s)
        s = " ".join(ws)
        if rng.random() < 0.1:
            s = s.replace(" ", "  ", 1) + " "                  # whitespace runs / trailing space
        out.append(s)
    return out


WORDS = ["The", "of", "and", "a", "Night", "Day", "Love", "Man", "Last", "Story", "Dead", "II", "Return", "King", "night", "é", "Noël",
         "x", "Zorro", "Christmas", "Carol", "day", "man", "House", "Home"]


@pytest.mark.parametrize("scorer", ["WRatio", "QRatio", "partial_ratio", "token_sort_ratio", "token_set_ratio", "token_ratio",
                                    "partial_token_sort_ratio", "partial_token_set_ratio", "partial_token_ratio", "ratio"])
def test_every_scorer_vs_oracle_on_title_like_strings(fz, scorer):
    rng = np.random.default_rng(len(scorer) * 7 + 1)
    frm = _titles(rng, 60, WORDS) + ["", " ", "The", "a a", "Night of the Living Dead", "x" * 70 + " tail", "long " * 30]
    to = _titles(rng, 260, WORDS, 1, 9) + ["", "  ", "The", "a", "Dead Night", "x" * 64, "long " * 40, frm[3]]
    bi, bs = fz.fuzz_argbest(frm, to, scorer, n_splits=3)
    oi, os_ = _oracle_best(frm, to, scorer)
    np.testing.assert_array_equal(bs.cpu().numpy(), os_)
    np.testing.assert_array_equal(bi.cpu().numpy(), oi)


@pytest.mark.parametrize("scorer,cutoff", [("WRatio", 86.0), ("token_set_ratio", 60.0), ("partial_ratio", 75.0)])
def test_score_cutoff_and_self_match(fz, scorer, cutoff):
    rng = np.random.default_rng(11)
    names = _titles(rng, 150, WORDS, 1, 5)
    bi, bs = fz.fuzz_argbest(names, names, scorer, cutoff, exclude_self=True)
    oi, os_ = _oracle_best(names, names, scorer, cutoff, exclude_self=True)
    np.testing.assert_array_equal(bs.cpu().numpy(), os_)
    np.testing.assert_array_equal(bi.cpu().numpy(), oi)
    assert (bi.cpu().numpy() != np.arange(len(names))).all()


def test_matchers_default_to_wratio_like_the_reference():
    """RapidFuzz() scores with fuzz.WRatio (polyfuzz/models/_rapidfuzz.py:48); the README's extractOne example, /100."""
    from polyfuzz_b200 import RapidFuzz, EditDistance
    choices = ["Atlanta Falcons", "New York Jets", "New York Giants", "Dallas Cowboys"]
    m = RapidFuzz().match(["cowboys", "new york jets"], choices)
    assert m.To.tolist() == ["Dallas Cowboys", "New York Jets"]
    assert m.Similarity.tolist() == [83.07692307692308 / 100, 76.92307692307692 / 100]
    m = RapidFuzz(scorer="ratio").match(["cowboys"], choices)
    assert m.Similarity.tolist() == [ofuzz.ratio("cowboys", "Dallas Cowboys") / 100]
    e = EditDistance(scorer="token_set_ratio", normalize=False).match(["fuzzy was a bear but not a dog"], ["x", "fuzzy was a bear but not a cat"])
    assert e.To.tolist() == ["fuzzy was a bear but not a cat"] and e.Similarity.tolist() == [92.3076923076923]
    with pytest.raises(NotImplementedError):
        RapidFuzz(scorer=lambda a, b: 1.0)


def test_string_shortcut_through_the_unmodified_orchestrator():
    """polyfuzz_b200.install() + PolyFuzz("EditDistance") (polyfuzz/polyfuzz.py:128-130: RapidFuzz() -> WRatio) reproduces
    rapidfuzz's published extractOne answer through the reference's own orchestrator."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref, "polyfuzz")):
        pytest.skip("oracle/_ref (the reference's polyfuzz package, copied by build()) not present")
    os.environ["PFZ_REFERENCE_ROOT"] = ref
    from oracle import ref_shim
    ref_shim.REFERENCE_ROOT = ref
    ref_shim.install()
    import polyfuzz_b200
    from polyfuzz import PolyFuzz
    polyfuzz_b200.install()
    choices = ["Atlanta Falcons", "New York Jets", "New York Giants", "Dallas Cowboys"]
    model = PolyFuzz("EditDistance").match(["cowboys", "new york jets"], choices)
    m = model.get_matches()
    assert m.To.tolist() == ["Dallas Cowboys", "New York Jets"]
    assert m.Similarity.tolist() == [0.8307692307692308, 0.7692307692307692]
    model = PolyFuzz("TF-IDF").match(["apple", "apples", "appl", "recal", "house", "similarity"], ["apple", "apples", "mouse"])
    assert model.get_matches().Similarity.tolist() == [1.0, 1.0, 0.784, 0.0, 0.588, 0.0]          # README.md:88-96, 3 decimals
