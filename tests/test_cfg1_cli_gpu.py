"""-m gpu: BASELINE.json configs[0] — `dalm train-retriever-only` on the reference's own toy fixture
(`dalm/datasets/toy_data_train.csv`, committed here as tests/golden/ref_toy_data_train.csv: a 1.7 KB DATA fixture, not
source), retriever = bge-small-en (random init: no checkpoints offline), bs 2 — through the console-script entry point
(reference dalm/cli.py:170-277, pyproject.toml:35-36 `dalm = dalm.cli:cli`; tests/test_cli.py pins that script).
The reference lists this config as CPU plumbing; dalm_b200 has no CPU path by contract, so the plumbing runs on the GPU."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOY = os.path.join(ROOT, "tests", "golden", "ref_toy_data_train.csv")


def test_toy_fixture_is_the_reference_file():
    """the committed fixture is byte-identical to the reference's dalm/datasets/toy_data_train.csv (its SHA-256)"""
    import hashlib
    assert hashlib.sha256(open(TOY, "rb").read()).hexdigest() == "783d2a65fdccc11c5f88bf351469af579547c48296c0c8544f7b9d9a97cba477"
    import csv
    rows = list(csv.DictReader(open(TOY)))
    assert {"Question", "Abstract", "Answer"} <= set(rows[0]) and len(rows) >= 10


def test_dalm_train_retriever_only_cli_on_reference_toy_csv(cuda_dev, tmp_path):
    from dalm_b200 import synthetic
    rdir = synthetic.write_model_dir(str(tmp_path / "bge-small-en"), "bert", "bge-small-en")      # 384 wide, 12 layers, 12 x 32
    out = str(tmp_path / "out")
    cmd = [sys.executable, "-m", "dalm_b200.cli", "train-retriever-only", rdir, TOY, "--output-dir", out,
           "--per-device-train-batch-size", "2", "--num-train-epochs", "2", "--no-use-bnb", "--checkpointing-steps", "epoch",
           "--learning-rate", "1e-3"]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=900,
                       env=dict(os.environ, PYTHONPATH=ROOT, PYTHONIOENCODING="utf-8"))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    # the reference's artefacts (train_retriever_only.py:405-420): <out>/retriever adapter + tokenizer, epoch_N state dirs
    cfg = json.load(open(os.path.join(out, "retriever", "adapter_config.json")))
    assert cfg["r"] == 8 and cfg["lora_alpha"] == 16 and cfg["target_modules"] == ["query", "key", "value"]
    assert cfg["base_model_name_or_path"] == rdir
    sd = torch.load(os.path.join(out, "retriever", "adapter_model.bin"), weights_only=True)
    assert len(sd) == 12 * 3 * 2 and any(v.abs().max() > 0 for k, v in sd.items() if "lora_B" in k)
    assert os.path.isdir(os.path.join(out, "epoch_0")) and os.path.isdir(os.path.join(out, "epoch_1"))
    losses = [json.loads(l) for l in open(os.path.join(out, "metrics.jsonl")) if "train/epoch_loss" in l]
    assert len(losses) == 2 and all(l["train/epoch_loss"] > 0 for l in losses)
    # 18 rows x 2 epochs at bs 2 under dropout: the epoch means differ by a few 1e-3 either way (the LoRA wgrad's fp32 atomics
    # are order-dependent, so two runs are not bit-identical) - assert "stable and learning-sized", not a strict decrease
    l0, l1 = losses[0]["train/epoch_loss"], losses[1]["train/epoch_loss"]
    assert l1 < l0 + 0.02 and max(l0, l1) < 0.80, (l0, l1)                       # chance level for 2 in-batch candidates: ln 2
