"""Generate tests/golden/* by RUNNING THE UNMODIFIED REFERENCE (/root/reference, peft/accelerate stubbed).

    python -m oracle.make_golden

TEST INFRASTRUCTURE ONLY. The reference tree exists only in the build container; the generated fixtures are committed
so that the CPU test-suite (and the GPU box) can pin oracle/ and dalm_b200's host code without it.
  losses.npz      reference train_utils.{get_cosine_sim,get_nt_xent_loss,compute_marginalized_loss_from_logits} outputs
                  and autograd gradients for seeded cases incl. left/right padding and qlen in {1, L-1, L, >L}
  pooling.npz     reference AutoModelForRagE2E.mean_pooling + F.normalize, dalm.utils.eos_mask
  preprocess.json reference batch builders (e2e + retriever-only) on synthetic rows with the fixture tokenizers
  eval_helpers.json reference dalm/eval/utils.py helpers (precision/recall, result aggregation, unique-passage filter,
                  tokenisation, neighbour formatting over a fixed (labels, distances) answer) — hnswlib itself is stubbed
  reference_spot_checks.json  reference compute_marginalized_loss_from_logits on a fresh seed, and eval-helper spot checks
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")


def loss_cases():
    # (B, D, L, V, pad, seed)
    return [(2, 16, 6, 11, "right", 0), (4, 32, 9, 23, "left", 1), (5, 64, 12, 50, "right", 2), (18, 128, 16, 97, "left", 3),
            (3, 8, 5, 7, "none", 4)]


def make_case(B, D, L, V, pad, seed):
    g = torch.Generator().manual_seed(seed)
    q = torch.nn.functional.normalize(torch.randn(B, D, generator=g), dim=1)
    p = torch.nn.functional.normalize(torch.randn(B, D, generator=g) + 0.3 * q, dim=1)
    logits = torch.randn(B, L, V, generator=g) * 2
    ids = torch.randint(0, V, (B, L), generator=g)
    mask = torch.ones(B, L, dtype=torch.int64)
    for b in range(B):
        n = int(torch.randint(0, L // 2, (1,), generator=g))
        if n and pad == "right": mask[b, L - n:] = 0
        if n and pad == "left": mask[b, :n] = 0
    qlen = torch.randint(1, L + 3, (B,), generator=g)
    edge = [1, L - 1, L, L + 2]
    for i in range(min(B, 4)):
        qlen[i] = edge[i]
    return q, p, logits, ids, mask, qlen


def gen_losses(ref):
    tu = ref.train_utils
    out = {}
    for ci, (B, D, L, V, pad, seed) in enumerate(loss_cases()):
        q, p, logits, ids, mask, qlen = make_case(B, D, L, V, pad, seed)
        qd, pd, ld = (t.clone().double().requires_grad_(True) for t in (q, p, logits))
        S = tu.get_cosine_sim(qd, pd, 100)
        lq, lp = tu.get_nt_xent_loss(S), tu.get_nt_xent_loss(S.t())
        lm = tu.compute_marginalized_loss_from_logits(ld, ids, mask, S, qlen)
        total = (lq + lp) / 2.0 + lm
        total.backward()
        pre = f"c{ci}_"
        for k, v in dict(q=q, p=p, logits=logits, ids=ids, mask=mask, qlen=qlen, S=S.detach(), loss_query=lq.detach(),
                         loss_passage=lp.detach(), loss_marginal=lm.detach(), loss_total=total.detach(), dQ=qd.grad,
                         dP=pd.grad, dlogits=ld.grad).items():
            out[pre + k] = v.numpy()
    out["n_cases"] = np.array(len(loss_cases()))
    np.savez_compressed(os.path.join(GOLD, "losses.npz"), **out)


def gen_pooling(ref):
    g = torch.Generator().manual_seed(10)
    tok = torch.randn(4, 9, 24, generator=g)
    mask = torch.ones(4, 9, dtype=torch.int64)
    mask[0, 5:] = 0; mask[1, :3] = 0; mask[3, 1:] = 0
    pooled = ref.AutoModelForRagE2E.mean_pooling(None, tok, mask)
    pooled2 = ref.AutoModelForSentenceEmbedding.mean_pooling(None, tok, mask)
    assert torch.equal(pooled, pooled2)
    emb = torch.nn.functional.normalize(pooled, p=2, dim=1)
    np.savez_compressed(os.path.join(GOLD, "pooling.npz"), tok=tok.numpy(), mask=mask.numpy(), pooled=pooled.numpy(),
                        emb=emb.numpy(), eos_left=ref.eos_mask(mask).numpy(), eos_right=ref.eos_mask(mask, "right").numpy())


def gen_preprocess(ref):
    from transformers import AutoTokenizer

    from dalm_b200 import synthetic

    tb, tl = os.path.join(GOLD, "tok_bert"), os.path.join(GOLD, "tok_llama")
    if not os.path.exists(os.path.join(tb, "tokenizer_config.json")):
        synthetic.build_bert_tokenizer(tb, vocab_size=1200)
    if not os.path.exists(os.path.join(tl, "tokenizer_config.json")):
        synthetic.build_llama_tokenizer(tl, vocab_size=900)
    rt, gt = AutoTokenizer.from_pretrained(tb), AutoTokenizer.from_pretrained(tl)
    gt.pad_token = gt.eos_token          # reference train_rage2e.py:301
    gt.add_eos_token = True              # reference train_rage2e.py:304
    rows = list(synthetic.synthetic_rows(5, seed=77)) + list(synthetic.synthetic_rows(2, seed=78, full=True))
    rows.append({"Abstract": "Kato miren. Sol-va!", "Question": "", "Answer": "x"})          # empty query, punctuation, case
    ex = {k: [r[k] for r in rows] for k in ("Abstract", "Question", "Answer")}
    e2e = ref.preprocess_e2e(ex, retriever_tokenizer=rt, generator_tokenizer=gt, query_column_name="Question",
                             passage_column_name="Abstract", answer_column_name="Answer", query_max_len=50,
                             passage_max_len=128, generator_max_len=256)
    ret = ref.preprocess_retriever(ex, rt, query_column_name="Question", passage_column_name="Abstract",
                                   query_max_len=50, passage_max_len=128)
    with open(os.path.join(GOLD, "preprocess.json"), "w") as f:
        json.dump({"rows": rows, "e2e": {k: v for k, v in e2e.items()}, "retriever": {k: v for k, v in ret.items()}}, f)


def gen_eval_helpers(ref):
    import datasets
    from transformers import AutoTokenizer

    eu = ref.eval_utils
    out = {}
    pr_cases = [(["a", "b", "c"], ["a"]), (["x", "y"], ["z"]), (["p", "p", "q"], ["q"]), (["only"], ["only"])]
    out["precision_recall"] = [{"retrieved": r, "correct": c, "out": list(eu.calculate_precision_recall(r, c))} for r, c in pr_cases]
    res = eu.calc_eval_results(7, [0.1, 0.2, 0.0, 0.1, 0.1, 0.5, 1.0], [1, 1, 0, 1, 1, 1, 1], 6)
    out["calc_eval_results"] = {"args": [7, [0.1, 0.2, 0.0, 0.1, 0.1, 0.5, 1.0], [1, 1, 0, 1, 1, 1, 1], 6],
                                "out": res.model_dump() if hasattr(res, "model_dump") else res.dict()}
    rows = {"Abstract": ["p one", "p two", "p one", "p three", "p two", "p four"], "Question": [f"q{i}" for i in range(6)]}
    ds = datasets.Dataset.from_dict(rows)
    out["filter_unique"] = {"rows": rows, "kept_questions": list(eu.filter_unique_passages(ds, "Abstract")["Question"])}
    tok = AutoTokenizer.from_pretrained(os.path.join(GOLD, "tok_bert"))
    ex = {"Question": ["kato miren sol", ""], "Abstract": ["sol va kato miren " * 12, "x"]}
    pre = eu.preprocess_function(ex, tok, query_column_name="Question", passage_column_name="Abstract", max_length=16)
    out["preprocess_function"] = {"examples": ex, "max_length": 16, "out": {k: v for k, v in pre.items()}}

    class FixedIndex:                                           # stands in for hnswlib.Index: a fixed answer
        def set_ef(self, ef): self.ef = ef
        def knn_query(self, q, k):
            labels = np.array([[2, 0, 1], [1, 2, 0]])[:, :k]
            dist = np.array([[0.05, 0.4, 1.2], [0.3, 0.31, 0.95]], dtype=np.float32)[:, :k]
            return labels, dist
    ids = {0: "zero", 1: "one", 2: "two"}
    nn = {}
    for thr in (0.7, 0.0):
        nn[str(thr)] = [[[p, float(s)] for p, s in row] for row in eu.get_nearest_neighbours(3, FixedIndex(), np.zeros((2, 4)), ids, threshold=thr)]
    out["nearest_neighbours"] = nn
    batch = [{"a": [1, 2], "s": "x", "n": None}, {"a": [3, 4], "s": "y", "n": None}]
    mc = eu.mixed_collate_fn(batch)
    out["mixed_collate"] = {"batch": batch, "out": {k: (v.tolist() if torch.is_tensor(v) else v) for k, v in mc.items()}}
    with open(os.path.join(GOLD, "eval_helpers.json"), "w") as f:
        json.dump(out, f)


def spot_check_marginal_inputs():
    """inputs of the fresh-seed marginalized-loss check (tests/test_oracle_golden.py), separate from loss_cases()"""
    g = torch.Generator().manual_seed(123)
    B, L, V, D = 6, 10, 31, 24
    q = torch.nn.functional.normalize(torch.randn(B, D, generator=g), dim=1)
    p = torch.nn.functional.normalize(torch.randn(B, D, generator=g), dim=1)
    lg = torch.randn(B, L, V, generator=g); ids = torch.randint(0, V, (B, L), generator=g)
    mask = torch.ones(B, L, dtype=torch.int64); mask[2, :4] = 0; mask[4, 7:] = 0
    ql = torch.tensor([1, 2, 9, 10, 12, 5])
    return q, p, lg, ids, mask, ql


SPOT_PRECISION_RECALL = [(["a", "b"], ["b"]), (["k"] * 4, ["k"]), (["m", "n", "o"], ["z"])]
SPOT_EVAL_RESULTS = (5, [0.1] * 5, [1, 0, 1, 1, 0], 3)


def gen_spot_checks(ref):
    """the reference's answers for the fresh-seed loss check and the eval-helper spot checks"""
    q, p, lg, ids, mask, ql = spot_check_marginal_inputs()
    S = ref.train_utils.get_cosine_sim(q, p, 100)
    lm = ref.train_utils.compute_marginalized_loss_from_logits(lg, ids, mask, S, ql)
    eu = ref.eval_utils
    res = eu.calc_eval_results(*SPOT_EVAL_RESULTS)
    out = {"marginalized_loss": {"dtype": str(lm.dtype).replace("torch.", ""), "value": lm.item()},
           "precision_recall": [{"retrieved": r, "correct": c, "out": list(eu.calculate_precision_recall(r, c))}
                                for r, c in SPOT_PRECISION_RECALL],
           "calc_eval_results": {"args": list(SPOT_EVAL_RESULTS),
                                 "out": res.model_dump() if hasattr(res, "model_dump") else res.dict()}}
    with open(os.path.join(GOLD, "reference_spot_checks.json"), "w") as f:
        json.dump(out, f, indent=1)


def main():
    from oracle import ref_import

    os.makedirs(GOLD, exist_ok=True)
    ref = ref_import.load()
    gen_losses(ref)
    gen_pooling(ref)
    gen_preprocess(ref)
    gen_eval_helpers(ref)
    gen_spot_checks(ref)
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()
