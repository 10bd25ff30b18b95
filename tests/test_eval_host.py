"""CPU: the evaluation helpers (SURVEY §8f-1; reference dalm/eval/utils.py) against the committed outputs of the reference's
own functions (tests/golden/eval_helpers.json, oracle/make_golden.py) and the exact-search oracle's conventions."""
import json
import os

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def gold():
    with open(os.path.join(GOLD, "eval_helpers.json")) as f:
        return json.load(f)


def test_precision_recall_and_aggregation(gold):
    from dalm_b200.eval.utils import calc_eval_results, calculate_precision_recall
    for c in gold["precision_recall"]:
        assert list(calculate_precision_recall(c["retrieved"], c["correct"])) == c["out"]
    with pytest.raises(ZeroDivisionError):                      # empty retrieved set: same failure as the reference
        calculate_precision_recall([], ["a"])
    r = calc_eval_results(*gold["calc_eval_results"]["args"])
    assert r.model_dump() == gold["calc_eval_results"]["out"]


def test_unique_passage_filter_keeps_first_occurrence(gold):
    import datasets
    from dalm_b200.eval.utils import filter_unique_passages
    ds = datasets.Dataset.from_dict(gold["filter_unique"]["rows"])
    assert list(filter_unique_passages(ds, "Abstract")["Question"]) == gold["filter_unique"]["kept_questions"]


def test_tokenisation_is_bit_exact(gold):
    from transformers import AutoTokenizer
    from dalm_b200.eval.utils import preprocess_function
    tok = AutoTokenizer.from_pretrained(os.path.join(GOLD, "tok_bert"))
    g = gold["preprocess_function"]
    out = preprocess_function(g["examples"], tok, query_column_name="Question", passage_column_name="Abstract",
                              max_length=g["max_length"])
    assert {k: v for k, v in out.items()} == g["out"]


def test_neighbour_formatting_and_threshold(gold):
    from dalm_b200.eval.utils import get_nearest_neighbours

    class FixedIndex:
        def set_ef(self, ef): self.ef = ef
        def knn_query(self, q, k):
            return (np.array([[2, 0, 1], [1, 2, 0]])[:, :k],
                    np.array([[0.05, 0.4, 1.2], [0.3, 0.31, 0.95]], dtype=np.float32)[:, :k])
    ids = {0: "zero", 1: "one", 2: "two"}
    for thr, want in gold["nearest_neighbours"].items():
        idx = FixedIndex()
        got = get_nearest_neighbours(3, idx, np.zeros((2, 4)), ids, threshold=float(thr))
        assert [[[p, float(s)] for p, s in row] for row in got] == want
        assert idx.ef == 100


def test_mixed_collate(gold):
    from dalm_b200.eval.utils import mixed_collate_fn
    out = mixed_collate_fn(gold["mixed_collate"]["batch"])
    assert {k: (v.tolist() if torch.is_tensor(v) else v) for k, v in out.items()} == gold["mixed_collate"]["out"]


def test_exact_search_oracle_conventions():
    """oracle/topk.py: hnswlib 'ip' space — distance = 1 - <q,p>, nearest first, ties towards the lower id"""
    from oracle import topk
    data = np.array([[1.0, 0.0], [0.0, 1.0], [0.6, 0.8], [1.0, 0.0]])
    labels, dist = topk.knn_query(data, np.array([[1.0, 0.0]]), 3)
    assert labels.tolist() == [[0, 3, 2]]
    assert np.allclose(dist, [[0.0, 0.0, 0.4]])


def test_live_reference_helpers_if_present(gold):
    """spot checks against the reference's stored answers (tests/golden/reference_spot_checks.json)"""
    from dalm_b200.eval import utils as ours
    with open(os.path.join(GOLD, "reference_spot_checks.json")) as f:
        spot = json.load(f)
    assert len(spot["precision_recall"]) == 3
    for c in spot["precision_recall"]:
        assert list(ours.calculate_precision_recall(c["retrieved"], c["correct"])) == c["out"]
    a = spot["calc_eval_results"]
    assert ours.calc_eval_results(*a["args"]).model_dump() == a["out"]


def test_nf4_oracle_properties():
    """oracle/nf4.py: levels are fixed points, codes are monotone in the value, zero blocks decode to zero"""
    from oracle import nf4
    lv = nf4.NF4.astype(np.float32)
    blk = np.zeros(64, np.float32); blk[:16] = lv
    deq, codes, absmax = nf4.roundtrip(blk)
    assert absmax.tolist() == [1.0] and codes[:16].tolist() == list(range(16))
    assert np.array_equal(deq[:16], lv.astype(np.float16).astype(np.float32))
    x = np.linspace(-1, 1, 64).astype(np.float32)
    _, c, _ = nf4.roundtrip(x)
    assert (np.diff(c.astype(int)) >= 0).all() and c[0] == 0 and c[-1] == 15
    z, cz, az = nf4.roundtrip(np.zeros(70, np.float32))
    assert (z == 0).all() and (cz == 7).all() and (az == 0).all()


def test_exact_match_rule():
    """reference eval_rag.py:268-277: text after the FIRST `#answer#`, stripped, equals the gold answer; no marker -> skipped"""
    from dalm_b200.eval.eval_rag import exact_match_hits
    gen = ["#query# q #passage# p #answer# blue whale", "#query# q #passage# p #answer#  blue whale \n", "no marker here",
           "#query# q #answer# a #answer# a", "#query# q #passage# p #answer# blue"]
    gold = ["blue whale", "blue whale", "blue whale", "a", "blue whale"]
    assert exact_match_hits(gen, gold) == 3
    with pytest.raises(ValueError):
        exact_match_hits(gen, gold[:-1])                                          # zip(strict=True) like the reference
