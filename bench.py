#!/usr/bin/env python
"""bench.py — RAG-e2e train-step throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" = one pass of the hot path over one bs-18 batch per GPU: 2x encoder forward (bge-large shape), fused in-batch
loss, decoder forward (Llama-2-7B shape), marginalised NLL, full backward (LoRA / PEFT mode: dgrad everywhere, wgrad for
the adapters), gradient all-reduce (N>1), Adam, adapter repack. Synthetic 200k-row set ("full" variant: every sequence
hits truncation, so padded tokens == useful tokens), seeded random-init weights of the public architectures.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "RAG-e2e train-step samples/sec (bge-large + Llama-2-7B, bs=18)"
BS, LQ, LP, LG = 18, 50, 128, 256
STEP_TFLOP_PEFT = 127.6          # SURVEY §8d: algorithmic TFLOP per bs-18 step in PEFT mode (fwd + dgrad + attn-bwd extra)

# BASELINE.json configs this bench can run (default cfg-3 = the config the headline metric is quoted on; the others are
# supplementary lines for `profiles/`). tflop = algorithmic TFLOP per step (SURVEY §8d table / formulae).
CONFIGS = {
    "cfg-3": dict(metric=METRIC, bs=18, lg=256, tflop=127.6, gen="llama", peft="both",
                  workload="cfg-3 train_rage2e {r} + {g} + PEFT(both) LoRA r=8, bs=18/GPU, Lq50/Lp128/Lg256"),
    "cfg-3-full": dict(metric="RAG-e2e train-step samples/sec, full fine-tuning (bge-large + Llama-2-7B, bs=18)", bs=18, lg=256, tflop=190.4,
                       gen="llama", peft=None,
                       workload="cfg-3/4 train_rage2e {r} + {g}, use_peft=None (the reference's CLI default: every parameter trained, fp32 Adam), bs=18/GPU, Lq50/Lp128/Lg256"),
    "cfg-2": dict(metric="retriever-only train-step samples/sec (bge-large, bs=150)", bs=150, lg=0, tflop=33.1, gen=None, peft="retriever",
                  workload="cfg-2 train_retriever_only {r} + PEFT LoRA r=8, per-device bs=150, Lq50/Lp128"),
    "cfg-5": dict(metric="RAG-e2e train-step samples/sec (bge-large + Falcon-7B, seq 2048, bs=18)", bs=18, lg=2048, tflop=1669.0, gen="falcon", peft="retriever",
                  workload="cfg-5 train_rage2e {r} (LoRA) + falcon-7b FULLY fine-tuned (reference semantics of --use-peft retriever: Falcon has no q_proj/v_proj), bs=18/GPU, Lg=2048, per-layer recomputation"),
    "cfg-5-frozen": dict(metric="RAG-e2e train-step samples/sec (bge-large + frozen Falcon-7B, seq 2048, bs=18)", bs=18, lg=2048, tflop=558.2, gen="falcon-frozen", peft="retriever",
                         workload="cfg-5 variant: {r} (LoRA) + falcon-7b FROZEN (forward only), bs=18/GPU, Lg=2048"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=str, default="cfg-3", choices=sorted(CONFIGS),
                    help="BASELINE.json config: cfg-3 (default, the metric's config) | cfg-3-full (use_peft=None) | cfg-2 | cfg-5 | cfg-5-frozen")
    ap.add_argument("--retriever", type=str, default="bge-large-en")
    ap.add_argument("--generator", type=str, default="Llama-2-7b-hf")
    ap.add_argument("--cpu-baseline", type=int, default=1, help="0 to skip the bounded CPU-oracle timing on rank 0")
    ap.add_argument("--gpu-eager-baseline", type=int, default=1, help="0 to skip the same-box HF-eager GPU baseline (rank 0, N=1)")
    ap.add_argument("--ref-rows", type=int, default=2, help="rows per step of the bounded CPU sample (reference arm / cpu_baseline)")
    ap.add_argument("--ref-budget-s", type=float, default=120.0, help="wall-clock budget of the reference arm's step loop (model build, ~1 min, comes on top)")
    ap.add_argument("--through-trainer", type=int, default=1,
                    help="1: also time the same steps through the public trainer API (dalm_b200.training...train_e2e: CSV -> "
                         "datasets.map -> DataLoader -> scheduler -> tracker); cfg-3 only")
    ap.add_argument("--graph", type=int, default=1, help="1: replay the step's launch sequence as one CUDA graph (default); 0: eager launches")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (loss, losses, S, the trained "
                         "parameters after Adam) as DIR/<name>.npy in float32 (rank 0; at most 64 MB, larger outputs sampled)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


DUMP_BYTES = 60 << 20          # array payload of --dump-outputs: with the .npy headers it stays under 64 MB


def collect_outputs(out, loss, model):
    """host float32 copies of what one step hands its caller: the reduced loss, the loss terms, the similarity matrix and
    every trainable parameter after the optimizer step. The first three are small and kept whole; if the parameters do not
    fit in the rest of DUMP_BYTES, each is replaced by a fixed, seeded sample of the same fraction of its elements (1-D, same
    indices on every run with the same shapes)."""
    import numpy as np
    import torch
    small = {"loss": loss, "losses": out["losses"], "S": out["S"]}
    params = {n: p for n, p in model.named_parameters() if p.requires_grad}
    budget = DUMP_BYTES - 4 * sum(t.numel() for t in small.values())
    keep = min(1.0, budget / (4 * sum(p.numel() for p in params.values())))
    g = torch.Generator().manual_seed(0)
    host = {n: np.array(t.detach().float().cpu(), dtype=np.float32) for n, t in small.items()}
    for name, p in params.items():
        t = p.detach()
        k = int(t.numel() * keep)
        if k < t.numel():
            idx = torch.randint(0, t.numel(), (k,), generator=g).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        host[name] = np.array(t.float().cpu(), dtype=np.float32)
    return host


def write_outputs(dirname, host):
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------------------------
# synthetic batches (first rows of the 200k-row "full" set, tokenised with the offline synthetic tokenizers)
# ----------------------------------------------------------------------------------------------------------------
def make_batches(n_batches: int, rank: int, world: int, cache_dir: str):
    import torch
    from dalm_b200 import synthetic
    from dalm_b200.training.utils.rag_e2e_dataloader_utils import preprocess_dataset
    from transformers import AutoTokenizer

    tb, tl = os.path.join(cache_dir, "tok_bert"), os.path.join(cache_dir, "tok_llama")
    if rank == 0:
        if not os.path.exists(os.path.join(tb, "tokenizer_config.json")):
            synthetic.build_bert_tokenizer(tb, 30522)
        if not os.path.exists(os.path.join(tl, "tokenizer_config.json")):
            synthetic.build_llama_tokenizer(tl, 32000)
    if world > 1:
        torch.distributed.barrier()
    rt, gt = AutoTokenizer.from_pretrained(tb), AutoTokenizer.from_pretrained(tl)
    gt.pad_token = gt.eos_token
    gt.add_eos_token = True
    rows = []
    need = n_batches * BS * world
    for i, r in enumerate(synthetic.synthetic_rows(need, seed=1234, full=True)):
        rows.append(r)
    ex = {k: [r[k] for r in rows] for k in ("Abstract", "Question", "Answer")}
    tok = preprocess_dataset(ex, rt, gt, "Question", "Abstract", "Answer", LQ, LP, LG)
    batches = []
    for b in range(n_batches):
        lo = (b * world + rank) * BS                        # rank-strided batches (accelerate semantics)
        batches.append({k: torch.tensor(v[lo:lo + BS], dtype=torch.int64) for k, v in tok.items()})
    return batches


class ClockSampler(threading.Thread):
    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        reasons = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for j, n in enumerate(names):
            if any(len(r) > 3 + j and r[3 + j].lower().startswith("active") for r in self.rows):
                reasons.append(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows and self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


# ----------------------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle (reference loss code + HF modeling code, fp32, eager PyTorch on the host cores)
# at FULL depth (24 + 32 layers) and full widths / sequence lengths; the bound is on ROWS per step, nothing is extrapolated
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_run(batch, rows: int, warmup: int, steps: int, budget_s: float):
    """Runs the reference's loop body (train_rage2e.py:429-474: forwards, losses, backward, Adam step) on the host cores with
    the complete bge-large + Llama-2-7B modules (LoRA r=8 on the reference's targets, train() mode, fp32 = the reference's
    default precision) on the first `rows` samples of a bs-18 batch. `warmup` untimed + up to `steps` timed steps, stopping
    early when `budget_s` of wall clock is spent (at least one timed step). Every reported step was really executed.
    -> dict(value samples/s, cores, steps_run, warmup_run, s_per_step, sample)"""
    import torch
    from dalm_b200 import synthetic
    from oracle import models as om

    # torch's CPU GEMMs stop scaling (and regress badly) long before 128 threads on these hosts: measured 0.013 samples/s
    # with 128 threads vs 0.157 with 8; use up to 32 threads and report that count as `cores`
    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    t_build = time.perf_counter()
    bcfg, lcfg = synthetic.bert_config("bge-large-en"), synthetic.llama_config("Llama-2-7b-hf")
    bert, llama = om.build_for_timing("bert", bcfg), om.build_for_timing("llama", lcfg)
    om.attach_lora(bert, om.timing_lora_factors("bert", bcfg), dropout=0.05)
    om.attach_lora(llama, om.timing_lora_factors("llama", lcfg), dropout=0.05)
    bert.train(); llama.train()
    opt = torch.optim.Adam([p for m in (bert, llama) for p in m.parameters() if p.requires_grad], lr=1e-4)
    batch = {k: v[:rows].clone() for k, v in batch.items()}
    t_build = time.perf_counter() - t_build
    t_start = time.perf_counter()
    warm_run = 0
    for _ in range(max(warmup, 0)):
        if warm_run >= 1 and time.perf_counter() - t_start > 0.3 * budget_s:
            break
        om.loop_body_step(bert, llama, batch, opt)
        warm_run += 1
    times = []
    for _ in range(max(steps, 1)):
        t0 = time.perf_counter()
        om.loop_body_step(bert, llama, batch, opt)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    per = sum(times) / len(times)
    desc = (f"MEASURED, nothing extrapolated: reference loop body (oracle: reference loss code + HF BertModel 24 layers + "
            f"LlamaForCausalLM 32 layers, fp32, LoRA r=8 + dropout, torch.optim.Adam; {cores} threads) on the first {rows} rows "
            f"of a bs-{BS} batch at Lq/Lp/Lg={LQ}/{LP}/{LG}: {warm_run} warm-up + {len(times)} timed steps of {per:.2f} s "
            f"(min {min(times):.2f}, max {max(times):.2f}); model build {t_build:.0f} s outside the timed region; "
            f"samples/s = {rows} / {per:.2f}")
    del bert, llama, opt
    return {"value": rows / per, "cores": cores, "steps_run": len(times), "warmup_run": warm_run, "s_per_step": per,
            "rows": rows, "sample": desc}


# ----------------------------------------------------------------------------------------------------------------
# same-box GPU baseline (SURVEY §8d-ii, BASELINE.md §3 row 2): the reference's loop body over HF modules + LoRA in eager
# PyTorch on THIS B200 - no dalm_b200 kernel on its path
# ----------------------------------------------------------------------------------------------------------------
def gpu_eager_baseline(dev, host_batches, warmup: int = 5, steps: int = 20):
    import torch
    from dalm_b200 import synthetic
    from oracle import models as om

    bcfg, lcfg = synthetic.bert_config("bge-large-en"), synthetic.llama_config("Llama-2-7b-hf")
    bert, llama = om.build_for_timing("bert", bcfg, device=dev), om.build_for_timing("llama", lcfg, device=dev)
    om.attach_lora(bert, om.timing_lora_factors("bert", bcfg, device=dev), dropout=0.05)
    om.attach_lora(llama, om.timing_lora_factors("llama", lcfg, device=dev), dropout=0.05)
    bert.train(); llama.train()
    opt = torch.optim.Adam([p for m in (bert, llama) for p in m.parameters() if p.requires_grad], lr=1e-4)
    batches = [{k: v.to(dev) for k, v in b.items()} for b in host_batches]

    def run(autocast, w, k):
        for i in range(w):
            om.loop_body_step(bert, llama, batches[i % len(batches)], opt, autocast=autocast)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            loss = om.loop_body_step(bert, llama, batches[(w + i) % len(batches)], opt, autocast=autocast)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k, float(loss.item())

    out = {"unit": "samples/s", "what": "reference loop body (train_rage2e.py:429-474) in eager PyTorch on this B200: HF BertModel "
           "(24 layers) + LlamaForCausalLM (32 layers), fp32 master weights, LoRA r=8 restatement (peft absent offline) + dropout, "
           "torch.optim.Adam, SDPA attention as transformers selects it; same synthetic batches; CUDA events; no dalm_b200 kernel"}
    ms, loss = run(torch.bfloat16, warmup, steps)
    out.update({"value": BS / (ms * 1e-3), "ms_per_step": ms, "precision": "bf16 autocast (accelerate --mixed_precision bf16)",
                "warmup": warmup, "steps": steps, "loss_last": loss})
    torch.backends.cuda.matmul.allow_tf32 = False
    ms32, _ = run(None, 1, 3)                              # the reference's literal default: no mixed precision, fp32 matmuls
    out["fp32_default"] = {"value": BS / (ms32 * 1e-3), "ms_per_step": ms32, "warmup": 1, "steps": 3,
                           "precision": "fp32, TF32 off (accelerate default: no mixed precision)"}
    del bert, llama, opt, batches
    torch.cuda.empty_cache()
    return out


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the newest committed `ncu --set full` capture of four consecutive
    generator-forward GEMM launches of one cfg-3 step (tools/profile_step.py under ncu: QKV+LoRA+RoPE, o_proj, gate|up+SwiGLU, down of
    decoder layer 1): mean of dram__bytes_read.sum + dram__bytes_write.sum over the captured launches, next to the algorithmic
    bytes (A + B + every output, + the fp32 residual where the epilogue reads one) of the same launches.
    Returns (bytes_per_launch or None, detail dict)."""
    import csv
    M = 4608
    # capture file -> [(M, N, K, output bytes per element summed over outputs (x N columns), residual bytes per element)] in launch order
    captures = [
        ("r02b_gemm_v5_ncu_full_raw.csv", [(M, 12288, 4112, 2, 0), (M, 4096, 4096, 4, 4), (M, 22016, 4096, 3, 0), (M, 4096, 11008, 4, 4)],
         "automatic raster + L2 hints; down-proj (4th) stays at ~1.6x: neither 50 MB operand band survives next to the other's stream"),
        ("r02_gemm_v4_ncu_full_raw.csv", [(M, 12288, 4112, 2, 0), (M, 4096, 4096, 4, 4), (M, 22016, 4096, 3, 0), (M, 4096, 11008, 4, 4)],
         "round-2a rule (bands for every multi-wave problem): B of QKV / gate|up read once per band"),
        ("r01_gemm_v3_ncu_full_raw.csv", [(M, 22016, 4096, 2, 0), (M, 4096, 11008, 4, 4), (M, 12288, 4112, 2, 0), (M, 4096, 4096, 4, 4)],
         "m-fastest everywhere: down-proj (2nd) re-reads A on each of its 4 tile waves"),
    ]
    for name, shapes, note in captures:
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        algo = [2 * (m * k + n * k) + m * n * (ob + rb) for m, n, k, ob, rb in shapes]      # gate|up: 2 B (gate|up) + 1 B (act = N/2 cols x 2 B)
        try:
            rows = list(csv.reader(open(path)))
            hdr = rows[0]
            rd, wr = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            ur, uw = unit[rows[1][rd]], unit[rows[1][wr]]
            per = [float(r[rd]) * ur + float(r[wr]) * uw for r in rows[2:] if len(r) > max(rd, wr)]
            if not per:
                return None, {"source": "no launches in " + os.path.relpath(path, ROOT)}
            return sum(per) / len(per), {"source": os.path.relpath(path, ROOT), "launches": len(per), "dram_bytes_per_launch": per,
                                         "algorithmic_bytes_per_launch": algo[:len(per)],
                                         "ratio_per_launch": [round(a / b, 3) for a, b in zip(per, algo)], "note": note}
        except Exception as e:
            return None, {"source": f"{name} unreadable ({type(e).__name__})"}
    return None, {"source": "no capture under profiles/"}


def trainer_e2e_run(args, rank: int, world: int, cache_dir: str):
    """The SAME workload through the repo's public entry point - `train_e2e(csv, retriever_dir, generator_dir, ...)`, the function
    `dalm train-rag-e2e` calls (reference train_rage2e.py:229-260) - instead of bench.py's private loop: CSV on disk ->
    load_dataset -> datasets.map tokenisation -> shuffled DataLoader + collate (pinned) -> H2D copy -> fused step (CUDA graph) ->
    gradient sync -> Adam -> LR scheduler -> tracker. Model directories hold config + tokenizer + a random-init marker (no
    checkpoints offline). Timed window: optimizer steps W..W+K between device synchronisations (loop.STEP_PROBE); model
    construction and the one-off tokenisation pass happen before it and are excluded."""
    import shutil
    import torch
    from dalm_b200 import synthetic
    from dalm_b200.models.rag_e2e_base_model import Mode
    from dalm_b200.training.rag_e2e.train_rage2e import train_e2e
    from dalm_b200.training.utils import loop

    W, K = args.warmup, args.steps
    rows = (W + K + 2) * BS * world
    csv = os.path.join(cache_dir, f"trainer_rows_{rows}.csv")
    rdir, gdir = os.path.join(cache_dir, "dir_" + args.retriever), os.path.join(cache_dir, "dir_" + args.generator)
    if rank == 0:
        if not os.path.exists(csv):
            synthetic.write_csv(csv, rows, seed=1234, full=True)
        if not os.path.exists(os.path.join(rdir, "config.json")):
            synthetic.write_model_dir(rdir, "bert", args.retriever, with_weights=False)
        if not os.path.exists(os.path.join(gdir, "config.json")):
            synthetic.write_model_dir(gdir, "llama", args.generator, with_weights=False)
    if world > 1:
        torch.distributed.barrier()
    out = os.path.join(cache_dir, "trainer_out")
    if rank == 0:
        shutil.rmtree(out, ignore_errors=True)
    if world > 1:
        torch.distributed.barrier()
    loop.STEP_PROBE = {"warmup": W, "steps": K}
    try:
        train_e2e(csv, rdir, gdir, per_device_train_batch_size=BS, max_train_steps=(W + K) * world, num_train_epochs=1,
                  use_peft=Mode.BOTH, num_warmup_steps=2, with_tracking=True, output_dir=out, seed=42)   # same dir on every rank
        probe = loop.STEP_PROBE
    finally:
        loop.STEP_PROBE = None
    if "seconds" not in probe:
        return {"value": None, "unit": "samples/s", "what": "probe did not fire"}
    t = torch.tensor([probe["seconds"]], device="cuda")
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    sec = t.item()
    return {"value": BS * world * K / sec, "unit": "samples/s", "ms_per_step": sec / K * 1e3, "steps": K, "warmup": W,
            "what": "public API: dalm_b200.training.rag_e2e.train_rage2e.train_e2e(csv, retriever_dir, generator_dir, bs=18, use_peft=both, "
                    "with_tracking=True) on the first rows of the synthetic 200k-row CSV ('full' variant); DataLoader(shuffle, collate, "
                    "pinned) + H2D + graph step + gradient sync + Adam + linear scheduler + jsonl tracker inside the timed window; "
                    "model construction and the datasets.map tokenisation pass before it (excluded); wall clock between device syncs"}


def workload_name(args) -> str:
    return CONFIGS[getattr(args, "config", "cfg-3")]["workload"].format(r=args.retriever, g=args.generator)


def random_batches(n: int, cfgd, rank: int, seed: int = 0):
    """token-id batches for the supplementary configs: uniform random ids, all-ones masks (every sequence at full length, as in
    the 'full' synthetic set the default config tokenises) - identical compute to tokenised text of that length"""
    import torch
    g = torch.Generator().manual_seed(seed * 1000 + rank)
    B = cfgd["bs"]
    rnd = lambda L, V: torch.randint(5, V, (B, L), generator=g)
    ones = lambda L: torch.ones(B, L, dtype=torch.int64)
    out = []
    for _ in range(n):
        if cfgd["gen"] is None:
            out.append({"query_input_ids": rnd(LQ, 30522), "query_attention_mask": ones(LQ),
                        "passage_input_ids": rnd(LP, 30522), "passage_attention_mask": ones(LP)})
        else:
            V = 32000 if cfgd["gen"] == "llama" else 65024
            out.append({"retriever_query_input_ids": rnd(LQ, 30522), "retriever_query_attention_mask": ones(LQ),
                        "retriever_passage_input_ids": rnd(LP, 30522), "retriever_passage_attention_mask": ones(LP),
                        "generator_input_input_ids": rnd(cfgd["lg"], V), "generator_input_attention_mask": ones(cfgd["lg"]),
                        "query_passage_input_len": torch.full((B,), min(200, cfgd["lg"] // 2))})
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # tokenizers, CSV, model dirs and the datasets cache live outside the tree, which may be read-only; one directory per
    # user, shared by the ranks of a run
    cache_dir = os.path.join(tempfile.gettempdir(), f"dalm_b200_bench_{os.getuid()}")
    os.makedirs(cache_dir, exist_ok=True)

    if args.impl == "reference":
        # the reference's own CPU implementation of the path (oracle port) on the host cores: rank 0 only. Each step is a
        # BOUNDED SAMPLE of the workload (the first REF_ROWS rows of a bs-18 batch through the full-depth models); every step
        # reported was executed and timed; if --steps does not fit the time budget fewer are run and `steps` says how many.
        if rank != 0:
            return
        batch = make_batches(1, 0, 1, cache_dir)[0]
        r = cpu_reference_run(batch, rows=args.ref_rows, warmup=args.warmup, steps=args.steps, budget_s=args.ref_budget_s)
        v = r["value"]
        line = {"metric": METRIC, "value": v, "unit": "samples/s", "n_gpus": args.gpus, "steps": r["steps_run"],
                "warmup": r["warmup_run"], "steps_requested": args.steps, "warmup_requested": args.warmup,
                "ms_per_step": r["s_per_step"] * 1e3, "rows_per_step": r["rows"], "extrapolated": False,
                "higher_is_better": True, "scaling": "weak",
                "vs_baseline": v / 7.94, "dtype": "f32", "data": "synthetic", "impl": "reference",
                "config": {"workload": workload_name(args), "global_batch": BS * max(1, args.gpus),
                           "parallelism": "cpu (rank 0 host cores; the other ranks exit)",
                           "dataset": "first rows of the synthetic 200k-row (Abstract,Question,Answer) 'full' set (all sequences truncated)",
                           "weights": "random (tiled N(0,0.02) block; timing only, no checkpoints offline)"},
                "cpu_baseline": {"value": v, "unit": "samples/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
                "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return

    # the trainer arm loads its CSV through `datasets`: keep that cache next to the others (set before `datasets` is imported)
    os.environ["HF_DATASETS_CACHE"] = os.path.join(cache_dir, "hf_datasets")
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        from dalm_b200.accel import nccl_env_defaults
        nccl_env_defaults()                                   # NCCL_MAX_CTAS before the communicator exists
        dist.init_process_group("nccl", device_id=dev)
    from dalm_b200 import _lib, ops, synthetic
    from dalm_b200.engine import params
    from dalm_b200.engine.bert import BertEncoder
    from dalm_b200.engine.llama import LlamaDecoder
    from dalm_b200.models.rag_e2e_base_model import AutoModelForRagE2E, Mode
    from dalm_b200.optim import FusedAdam
    from dalm_b200.training.utils.train_utils import GraphedStep, fused_rag_step

    _lib.call("dalm_b200_probe_device")
    cfgd = CONFIGS[args.config]
    B_step = cfgd["bs"]
    bf = torch.bfloat16
    bcfg = dict(synthetic.bert_config(args.retriever), _device_rng=True)
    full_r = cfgd["peft"] is None
    # supplementary variant (not the metric's configuration): DALM_B200_BENCH_NF4=1 keeps both base models as packed NF4 codes
    # (`use_bnb` with DALM_B200_NF4_STORAGE semantics, engine/nf4store.py) - reports what 4-bit storage costs per step and saves in HBM
    nf4 = os.environ.get("DALM_B200_BENCH_NF4", "0") == "1" and cfgd["peft"] is not None
    enc = BertEncoder(bcfg, params.random_state_dict("bert", bcfg, seed=0, dtype=bf, device=dev), device=dev, lora=not full_r, full=full_r,
                      nf4_storage=nf4 and not full_r)
    if cfgd["gen"] is None:                                   # cfg-2: retriever-only trainer (train_retriever_only.py:365-379)
        from dalm_b200.models.retriever_only_base_model import AutoModelForSentenceEmbedding
        from dalm_b200.training.utils.train_utils import fused_retriever_step as step_fn
        model = AutoModelForSentenceEmbedding("", use_bnb=False, get_peft=True, _model=enc, _load_tokenizer=False)
        banks = enc.banks()
        repack = enc.repack_lora
    else:
        from dalm_b200.training.utils.train_utils import fused_rag_step as step_fn
        if cfgd["gen"] == "llama":
            lcfg = dict(synthetic.llama_config(args.generator), _device_rng=True)
            dec = LlamaDecoder(lcfg, params.random_state_dict("llama", lcfg, seed=0, dtype=bf, device=dev), device=dev,
                               lora=cfgd["peft"] == "both", full=cfgd["peft"] is None, nf4_storage=nf4 and cfgd["peft"] == "both")
        else:
            from dalm_b200.engine.falcon import FalconDecoder
            fcfg = dict(synthetic.falcon_config("falcon-7b"), _device_rng=True)
            dec = FalconDecoder(fcfg, params.random_state_dict("falcon", fcfg, seed=0, dtype=bf, device=dev), device=dev,
                                full=cfgd["gen"] == "falcon")
        torch.cuda.empty_cache()
        model = AutoModelForRagE2E("", "", get_peft={"both": Mode.BOTH, "retriever": Mode.RETRIEVER, None: None}[cfgd["peft"]],
                                   _retriever=enc, _generator=dec, _load_tokenizers=False)
        banks = model.trainable_banks()
        repack = model.repack
    # PEFT initialises B = 0; after a few optimizer steps it is not. Same seed on every rank (DDP broadcast semantics).
    opt = FusedAdam(model.parameters(), lr=1e-4)
    model.train()                          # reference train_rage2e.py:421: dropout sites are live during the timed steps

    n_batches = args.warmup + args.steps
    if args.config == "cfg-3":
        host_batches = make_batches(n_batches, rank, world, cache_dir)
    else:
        host_batches = random_batches(min(n_batches, 4), cfgd, rank)
        host_batches = [host_batches[i % len(host_batches)] for i in range(n_batches)]
    pinned = [{k: v.pin_memory() for k, v in b.items()} for b in host_batches]
    resident = [{k: v.to(dev) for k, v in b.items()} for b in host_batches]
    h2d_bytes = sum(v.numel() * v.element_size() for v in host_batches[0].values())

    # the data-parallel reducer re-homes the LoRA gradient buffers into one arena: build it before the graph capture
    from dalm_b200.accel import GradientSync
    sync = GradientSync(banks, world, dev, nccl=True)
    graphed = None
    big = args.config == "cfg-5"       # 125 GB of parameters + Adam state: no room for a graph's private pool NEXT TO the eager
    #                                    roofline pass's activations; a 3 s step hides its launch overhead anyway
    from dalm_b200.training.utils import negatives
    xneg = negatives.active()          # optional extension (not the reference's semantics): an all-gather sits inside the step
    if args.graph and not sync.overlaps_backward and not big and not xneg:   # full fine-tuning on N > 1: bucket all-reduces are issued during backward
        try:
            graphed = GraphedStep(step_fn, model, resident[0], 100.0, zero_grads=opt.zero_grad)
        except Exception as e:
            if rank == 0:
                print(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); eager launches", file=sys.stderr, flush=True)

    rank_ev = []                                             # (start, compute done, step done) events of the timed steps
    last = {}                                                # the most recent step's outputs (--dump-outputs)

    def train_step(batch, eager=False, record=False):
        if record:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
        out = graphed(batch) if (graphed is not None and not eager) else step_fn(model, batch, 100.0, backward=True)
        last["out"] = out
        if record:
            ev[1].record()
        loss = sync.reduce(out["loss"])                      # ONE all-reduce: both LoRA banks' gradients (mean) + the loss (rank sum)
        opt.step()
        repack()
        opt.zero_grad()
        if record:
            ev[2].record()
            rank_ev.append(ev)
        return loss

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(batches, use_timer, eager=False, record=False):
        for i in range(args.warmup):
            train_step(batches[i], eager)
        sync_all()
        _lib.reset_launch_count()
        if use_timer is not None:
            use_timer.reset()
            ops.GEMM_TIMER = use_timer
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = None
        for i in range(args.steps):
            loss = train_step(batches[args.warmup + i], eager, record=record)
        e1.record()
        sync_all()
        ops.GEMM_TIMER = None
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), loss, _lib.launch_count()

    # ---- device-resident run (value) -------------------------------------------------------------------------
    timer = ops.GemmTimer(capacity=2000 * args.steps + 64)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    total_ms, loss, launches = timed(resident, None if graphed is not None else timer, record=world > 1)
    if args.dump_outputs and rank == 0:                       # before the passes below run more steps on the same model
        write_outputs(args.dump_outputs, collect_outputs(last["out"], loss, model))
    coll_per_step = sync.collectives / (args.warmup + args.steps) if world > 1 else 0
    if sampler:
        sampler.stop_flag = True
    eager_ms = total_ms
    if graphed is not None:
        # per-launch CUDA events cannot be recorded inside a graph replay: the roofline pass re-runs the SAME steps with
        # eager launches (identical kernels, shapes and data) right after the timed region, events around every GEMM.
        # `launches` = kernels per timed region, counted by the library during this eager pass (a replay launches the same set)
        # (single stream during this pass so the per-kernel event durations are not inflated by cross-stream overlap)
        from dalm_b200.training.utils import train_utils as _tu
        _two = _tu._TWO_STREAMS
        _tu._TWO_STREAMS = False
        eager_ms, _, launches = timed(resident, timer, eager=True)
        _tu._TWO_STREAMS = _two
    gsum = timer.summary()
    if os.environ.get("DALM_B200_GEMM_SHAPES") and rank == 0:   # per-shape breakdown of the GEMM time (stderr; profiles/)
        for tag, n, ms, tf in timer.by_shape():
            print(f"[gemm-shape] {tag} launches={n} total_ms={ms:.3f} tflops={tf:.1f}", file=sys.stderr, flush=True)

    # ---- end-to-end run through the public step with host (pinned) batches: H2D inside, loss read back each step ----
    def e2e_run():
        for i in range(args.warmup):
            train_step(pinned[i]).item()
        sync_all()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        last = None
        for i in range(args.steps):
            last = train_step(pinned[args.warmup + i]).item()      # device->host read of the step's loss
        t1.record()
        sync_all()
        t = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), last
    e2e_ms, e2e_loss = e2e_run()

    # per-rank step anatomy (N > 1): device time of the step's own compute vs. everything after it (collective incl. the wait
    # for the slowest rank, Adam, repack) - names what the weak-scaling loss is made of
    per_rank = None
    if world > 1 and rank_ev:
        comp = sum(e[0].elapsed_time(e[1]) for e in rank_ev) / len(rank_ev)
        rest = sum(e[1].elapsed_time(e[2]) for e in rank_ev) / len(rank_ev)
        t = torch.tensor([comp, rest], device=dev)
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = [{"rank": i, "compute_ms": round(x[0].item(), 3), "reduce_wait_adam_ms": round(x[1].item(), 3)} for i, x in enumerate(allt)]

    # everything the JSON line needs from the live objects, then free them: the trainer run / eager baseline below build their own models
    loss_last = float(loss.item())
    used_graph = graphed is not None
    arena_mb = sync.arena.numel() * 4 / 1e6
    peak_mem_gb = torch.cuda.max_memory_allocated() / 2 ** 30
    nf4_store_gb = sum(m.nf4.nbytes() for m in (enc, dec if cfgd["gen"] is not None else None)
                       if getattr(m, "nf4", None) is not None) / 2 ** 30
    graphed = model = enc = opt = sync = banks = repack = resident = pinned = None
    if cfgd["gen"] is not None:
        dec = None
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    trainer_line = None
    if args.through_trainer and args.config == "cfg-3":       # the same steps through the public trainer API (all ranks take part)
        try:
            trainer_line = trainer_e2e_run(args, rank, world, cache_dir)
        except Exception as e:
            trainer_line = {"value": None, "unit": "samples/s", "what": f"failed: {type(e).__name__}: {e}"}
        gc.collect()
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
    samples = B_step * world * args.steps
    value = samples / (total_ms * 1e-3)
    gemm_tf = gsum["total_flops"] / max(gsum["total_ms"] * 1e-3, 1e-9) / 1e12
    traffic, traffic_detail = ncu_traffic()
    line = {
        "metric": cfgd["metric"], "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": value / 7.94 if args.config == "cfg-3" else None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(args),
                   "global_batch": B_step * world, "parallelism": f"dp{world}", "rows_used": n_batches * B_step * world,
                   "dataset": ("first rows of the synthetic 200k-row (Abstract,Question,Answer) 'full' set (all sequences truncated)"
                               if args.config == "cfg-3" else "uniform random token ids at the config's full sequence lengths, all-ones masks"),
                   "l2": "per-step working set (weights + activations: tens of GB) >> 126 MB L2; no explicit flush",
                   "weights": "seeded random-init (no checkpoints offline)", "dropout": "train() mode as in the reference loop: BERT hidden 0.1 + attention-prob 0.1, LoRA input 0.05 (Philox, masks regenerated in backward)",
                   "launch": "one CUDA graph replay per step (fwd+bwd) + Adam/repack launches" if used_graph else "eager launches",
                   "eager_ms_per_step": eager_ms / args.steps,
                   "loss_last": loss_last,
                   **({"negatives": "DALM_B200_CROSS_RANK_NEGATIVES=1: in-batch negatives all-gathered over the ranks (extension; "
                                    "NOT the reference's rank-local semantics)"} if xneg else {}),
                   **({"variant": "DALM_B200_BENCH_NF4=1: base weights of both models kept as packed NF4 codes (4-bit storage), "
                                  "expanded to bf16 per GEMM; NOT the metric's configuration",
                       "nf4_store_gb": nf4_store_gb}
                      if nf4 else {})},
        "e2e": {"value": samples / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "step_tflops": cfgd["tflop"] * args.steps * world / (total_ms * 1e-3),
        "peak_mem_gb": peak_mem_gb,
        "roofline": {"bound": "tensor", "achieved": gemm_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": gemm_tf / peak_tf,
                     "traffic": traffic, "traffic_detail": traffic_detail,
                     "kernel": "gemm_bf16_tn_kernel (tcgen05)", "launches_timed": gsum["launches"],
                     "share_of_step": gsum["total_ms"] / eager_ms, "peak_source": peak_src,
                     "note": "achieved = sum of 2MNK over all GEMM launches / sum of their CUDA-event durations in the timed region"},
        "clocks": sampler.summary() if sampler else None,
    }
    if per_rank is not None:
        cm = [r["compute_ms"] for r in per_rank]
        line["per_rank"] = per_rank
        line["scaling_note"] = (f"step = max over ranks every step (the all-reduce is a barrier): slowest rank's own compute "
                                f"{max(cm):.2f} ms vs fastest {min(cm):.2f} ms; {coll_per_step:g} collective(s) per step "
                                f"({arena_mb:.1f} MB: the small (LoRA) banks + loss scalar in one all-reduce; dense banks in per-layer buckets)")
    if trainer_line is not None:
        line["trainer_e2e"] = trainer_line
    if world == 1 and args.gpu_eager_baseline and args.config == "cfg-3":   # same-box eager-PyTorch comparator (rank 0, N=1 only)
        try:
            line["gpu_eager_baseline"] = gpu_eager_baseline(dev, host_batches[:8])
        except Exception as e:
            line["gpu_eager_baseline"] = {"value": None, "unit": "samples/s", "what": f"failed: {type(e).__name__}: {e}"}
    if args.cpu_baseline and world == 1 and args.config == "cfg-3":   # reported CPU baseline: rank 0, N=1 only
        try:
            r = cpu_reference_run(host_batches[0], rows=args.ref_rows, warmup=1, steps=2, budget_s=30.0)
            line["cpu_baseline"] = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port",
                                    "sample": r["sample"], "extrapolated": False}
        except Exception as e:                                   # never lose the GPU line to a host-side problem
            line["cpu_baseline"] = {"value": None, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"failed: {type(e).__name__}: {e}"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
