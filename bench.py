#!/usr/bin/env python
"""Headline benchmark: GPT-2 pre-training throughput (tokens/s) on N B200 GPUs of one node.

Model/config = the reference's published GPT-2 benchmark (docs Benchmark.md:20-26, BASELINE.md rows
6-8: 24 layers, hidden 1024, 16 heads, seq 1024, data parallel, micro-batch per GPU fixed → weak
scaling), bf16 compute with fp32 master weights, synthetic tokens, random-init weights.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 20 --warmup 5
    python bench.py --impl reference ...      # the unmodified reference (needs OneFlow)
    python bench.py --steps 20 --warmup 5 --dump-outputs output/bench   # + what the last timed step computed (.npy)

Prints ONE JSON line (rank 0).  ``value`` is device-timed (CUDA events, max over ranks) over exactly
``--steps`` full training steps (fwd + bwd + grad sync + optimizer); ``e2e`` repeats the
measurement through the public trainer API including the per-step pinned-host→device input copy and
the device→host loss read.  Inputs and initial weights are seeded, so two builds run with the same
arguments can be compared output for output through ``--dump-outputs``.  Nothing is written into the
source tree: the trainer's output directory is a temporary one.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

# published LiBai numbers for the GPT-2 data-parallel rows (samples/s × 1024 tokens), BASELINE.md #6-#8
PUBLISHED_TOKENS_PER_S = {1: 17940.0, 4: 64973.0, 8: 128655.0}

# benchmark models: the headline (gpt2 = the reference's benchmark GPT-2) and the other BASELINE.json configs
MODELS = {
    "gpt2": dict(cfg="configs/gpt2_synthetic.py", layers=24, hidden=1024, heads=16, seq=1024, micro=8, unit="tokens/s",
                 name="GPT-2 nl{layers} h{hidden} a{heads} (reference benchmark model, ~355M params)"),
    "gpt2_large": dict(cfg="configs/gpt2_synthetic.py", layers=36, hidden=1280, heads=20, seq=1024, micro=8, unit="tokens/s",
                       name="GPT-2 large nl{layers} h{hidden} a{heads} (~774M params)"),
    "bert_large": dict(cfg="configs/bert_large_synthetic.py", layers=24, hidden=1024, heads=16, seq=512, micro=16,
                       unit="tokens/s", name="BERT-large nl{layers} h{hidden} a{heads} s512 (reference benchmark BERT)"),
    "llama7b": dict(cfg="projects/Llama/configs/llama7b_synthetic.py", layers=32, hidden=4096, heads=32, seq=2048, micro=1,
                    unit="tokens/s", name="Llama-2 7B nl{layers} h{hidden} a{heads} ffn11008 s2048"),
    "vit_l": dict(cfg="configs/vit_large_synthetic.py", layers=24, hidden=1024, heads=16, seq=197, micro=128, unit="images/s",
                  name="ViT-Large/16 224x224 nl{layers} h{hidden} a{heads}"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "ref", "reference"])
    ap.add_argument("--model", default="gpt2", choices=sorted(MODELS),
                    help="gpt2 (default, the headline: reference benchmark GPT-2 nl24 h1024) | gpt2_large | bert_large | "
                         "llama7b | vit_l — the other BASELINE.json configs; metric stays tokens/s (images/s for vit_l)")
    ap.add_argument("--micro-batch", type=int, default=0, help="samples per GPU per step (0 = the model's default)")
    ap.add_argument("--layers", type=int, default=0)
    ap.add_argument("--hidden", type=int, default=0)
    ap.add_argument("--heads", type=int, default=0)
    ap.add_argument("--seq", type=int, default=0)
    ap.add_argument("--dropout", type=float, default=-1.0,
                    help="override every dropout probability of the model (the reference's gpt2_pretrain recipe trains "
                         "with 0.1; the synthetic benchmark config and the published benchmark use 0)")
    ap.add_argument("--tp", type=int, default=1, help="tensor-parallel size of the PRIMARY layout (sequence parallel + "
                    "collectives fused into the GEMM kernels); per-DP-rank micro-batch is scaled so that the global batch "
                    "stays --micro-batch x --gpus")
    ap.add_argument("--pp", type=int, default=1, help="pipeline-parallel size of the primary layout (1F1B, 4 micro-batches per stage)")
    ap.add_argument("--layout", default="", help="shorthand for the primary layout: dp | tp2 | tp4 | pp2 | 3d (= tp2 x pp2 x dp(N/4) + ZeRO-1)")
    ap.add_argument("--extras", type=int, default=1,
                    help="1 (default): after the primary (data-parallel) measurement also measure the tensor-parallel / "
                         "3-D layouts that fit --gpus in the same launch and report them under `layouts`")
    ap.add_argument("--extra-steps", type=int, default=8)
    ap.add_argument("--ref-same-box", type=int, default=1,
                    help="1 (default): also time baseline/pytorch_baseline.py (stock PyTorch: SDPA, fused AdamW, DDP, bf16 "
                         "autocast) in this launch and report it as `ref_same_box`")
    ap.add_argument("--zero", type=int, default=-1, help="ZeRO stage; -1 = auto (stage 1 with the fused NVLink kernels when dp > 1)")
    ap.add_argument("--acc", type=int, default=1)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--graphs", type=int, default=1,
                    help="1 (default = train.cuda_graphs.enabled default): replay the transformer blocks from CUDA graphs "
                         "(data-parallel and fused tensor-parallel layouts; pipeline-parallel runs launch eagerly)")
    ap.add_argument("--fused-bias-grad", type=int, default=-1,
                    help="1/0: bias gradient of the MLP's first linear inside the dgrad epilogue (-1: library default)")
    ap.add_argument("--fp8", type=int, default=0,
                    help="1: forward GEMMs with E4M3 operands (experiment; the headline number is the bf16 default — "
                         "the JSON line then says dtype fp8-fwd/bf16-bwd)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps write what the last one computed (its loss dict and a seeded sample of "
                         "the updated model state, rank 0) as DIR/<name>.npy, float32")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    spec = MODELS[a.model]
    for k in ("layers", "hidden", "heads", "seq"):
        if not getattr(a, k):
            setattr(a, k, spec[k])
    if not a.micro_batch:
        a.micro_batch = spec["micro"]
    return a


# ---------------------------------------------------------------------------------------------------
# reference arm
# ---------------------------------------------------------------------------------------------------
def run_reference(args):
    """Run the UNMODIFIED reference (baseline/_ref) through its own public API.  LiBai is a thin
    layer over OneFlow; without OneFlow (not in the image, no network) it cannot execute."""
    ref_dir = os.path.join(REPO, "baseline", "_ref")
    why = None
    if not os.path.isdir(ref_dir):
        why = "baseline/_ref not installed"
    else:
        sys.path.insert(0, ref_dir)
        try:
            import oneflow  # noqa: F401
        except Exception as e:  # noqa
            why = f"reference needs OneFlow which is not installed/installable offline ({type(e).__name__}: {e})"
    if why is None:
        try:
            import libai  # noqa: F401

            why = "reference import succeeded but no OneFlow CUDA runtime path is wired for sm_100"
        except Exception as e:  # noqa
            why = f"import libai failed: {type(e).__name__}: {e}"
    print(json.dumps({"impl": "reference", "unavailable": why.replace("\n", " ")[:300]}))
    return 0


# ---------------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons),
            "samples": len(sm),
        }


# ---------------------------------------------------------------------------------------------------
# native / ref arms
# ---------------------------------------------------------------------------------------------------
def layout_of(args, world, name=""):
    """(tp, pp, acc, zero) of a named layout; the global batch is always --micro-batch x world samples per step."""
    name = name or args.layout
    tp, pp = args.tp, args.pp
    if name in ("tp2", "tp4", "tp8"):
        tp, pp = int(name[2:]), 1
    elif name == "pp2":
        tp, pp = 1, 2
    elif name == "3d":
        tp, pp = 2, 2
    elif name == "dp":
        tp, pp = 1, 1
    assert world % (tp * pp) == 0, f"layout {name or (tp, pp)} does not fit {world} GPUs"
    dp = world // (tp * pp)
    acc = args.acc if pp == 1 else max(args.acc, 4)          # 1F1B: 4 micro-batches in flight per step
    zero = args.zero if args.zero >= 0 else (1 if dp > 1 else 0)
    # samples per DP rank and step = micro_batch x tp x pp (a model-parallel group of tp*pp GPUs carries their share)
    micro = args.micro_batch * tp * pp // acc
    assert micro >= 1 and micro * acc == args.micro_batch * tp * pp, "micro-batch not divisible by the accumulation count"
    return dict(tp=tp, pp=pp, dp=dp, acc=acc, zero=zero, micro=micro)


def layout_name(lay):
    par = f"dp{lay['dp']}"
    if lay["tp"] > 1:
        par += f"_tp{lay['tp']}_sp_fused-comm-gemm"
    if lay["pp"] > 1:
        par += f"_pp{lay['pp']}_1f1b-x{lay['acc']}"
    if lay["zero"]:
        par += f"_zero{lay['zero']}"
    return par


def build_cfg(args, lay):
    from libai_b200.config import LazyConfig

    spec = MODELS[args.model]
    cfg = LazyConfig.load(os.path.join(REPO, spec["cfg"]))
    m = cfg.model.cfg
    if args.model in ("gpt2", "gpt2_large"):
        m.hidden_layers, m.hidden_size, m.num_attention_heads = args.layers, args.hidden, args.heads
        m.ffn_hidden_size = 4 * args.hidden
        m.max_seq_length = args.seq
        for ds in cfg.dataloader.train.dataset:
            ds.seq_length = args.seq
            ds.vocab_size = m.vocab_size
    elif args.model == "bert_large":
        m.hidden_layers, m.hidden_size, m.num_attention_heads = args.layers, args.hidden, args.heads
        m.intermediate_size = 4 * args.hidden
        if args.dropout < 0:   # like the GPT-2 benchmark config: dropout-free unless asked for
            m.hidden_dropout_prob = m.attention_probs_dropout_prob = 0.0
    elif args.model == "llama7b":
        m.hidden_layers, m.hidden_size, m.num_attention_heads = args.layers, args.hidden, args.heads
        if args.hidden != 4096:
            m.intermediate_size = (int(args.hidden * 8 / 3) + 127) // 128 * 128
        m.max_position_embeddings = args.seq
        for ds in cfg.dataloader.train.dataset:
            ds.seq_length = args.seq
    elif args.model == "vit_l":
        m.depth, m.embed_dim, m.num_heads = args.layers, args.hidden, args.heads
    if args.dropout >= 0:
        for k in list(m.keys()):
            if "dropout" in k or k in ("drop_rate", "attn_drop_rate"):
                m[k] = args.dropout
    cfg.dataloader.train.num_workers = 2
    cfg.train.train_micro_batch_size = lay["micro"]
    cfg.train.num_accumulation_steps = lay["acc"]
    cfg.train.global_batch_size = None
    cfg.train.train_iter = 10 ** 6
    cfg.train.log_period = 1            # the end-to-end loop reads the loss on the host every step
    cfg.train.amp.enabled = True
    cfg.train.evaluation.enabled = False
    cfg.train.checkpointer.period = 10 ** 9
    cfg.train.output_dir = args.output_dir
    cfg.train.cuda_graphs.enabled = bool(args.graphs)
    cfg.train.dist.tensor_parallel_size = lay["tp"]
    cfg.train.dist.pipeline_parallel_size = lay["pp"]
    cfg.train.dist.pipeline_num_layers = args.layers
    cfg.train.dist.data_parallel_size = lay["dp"]
    cfg.train.input_placement_device = "cuda"
    # tensor parallelism = token-sharded activations + AG->GEMM / GEMM->RS kernels ("auto" resolves to this for GPT-2;
    # spelled out so that the bench line can state it)
    cfg.train.dist.sequence_parallel = lay["tp"] > 1
    cfg.train.dist.fused_tp_comm = lay["tp"] > 1
    cfg.train.zero_optimization.enabled = lay["zero"] > 0
    cfg.train.zero_optimization.stage = max(lay["zero"], 1)
    return cfg


DUMP_SAMPLES_PER_TENSOR = 4096     # ~3 MB of float32 for the headline model (its whole state would be ~1.4 GB)


def dump_outputs(out_dir, loss, model):
    """Write what a training step computed as ``out_dir/<name>.npy`` (float32): every entry of the loss dict the step
    returns (``lm_loss.npy``) and ``state_sample.npy``, the same seeded sample of ``DUMP_SAMPLES_PER_TENSOR`` elements
    of every floating-point tensor of the updated state dict (all of a smaller tensor), concatenated in state-dict
    order."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for k, v in (loss or {}).items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v.detach().float().cpu().numpy())
    g = torch.Generator().manual_seed(0)
    parts = []
    for t in model.state_dict().values():
        if not t.is_floating_point():
            continue
        flat = t.detach().reshape(-1)
        n = flat.numel()
        k = DUMP_SAMPLES_PER_TENSOR
        idx = torch.arange(n) if n <= k else torch.randint(0, n, (k,), generator=g)
        parts.append(flat[idx.to(flat.device)].float().cpu())
    np.save(os.path.join(out_dir, "state_sample.npy"), torch.cat(parts).numpy())


def measure_native(args, lay, world, rank, local_rank, steps, warmup, with_e2e, clock_sampler=None, dump_dir=""):
    """Build the trainer for ``lay`` through the public API, time ``steps`` optimizer steps on the device (CUDA events,
    max over ranks) and optionally the end-to-end loop through ``trainer.run_step()``.  With ``dump_dir``, rank 0 then
    writes what the last timed step computed there (:func:`dump_outputs`)."""
    import gc
    import logging

    import torch
    import torch.distributed as dist

    from libai_b200 import ops
    from libai_b200.engine import DefaultTrainer, default_setup
    from libai_b200.utils import distributed as dutil
    from libai_b200.utils.events import EventStorage

    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    h2d_counter = {"bytes": 0}

    class BenchTrainer(DefaultTrainer):
        """``get_batch`` is a documented override point: count the bytes of every host→device input copy."""

        @classmethod
        def get_batch(cls, data, input_placement_device="cuda", mixup_func=None):
            h2d_counter["bytes"] += sum(v.tensor.numel() * v.tensor.element_size() for v in data.get_fields().values()
                                        if not v.tensor.is_cuda)
            return super().get_batch(data, input_placement_device, mixup_func)

    dutil.reset_dist_util()
    cfg = build_cfg(args, lay)
    default_setup(cfg, argparse.Namespace(resume=False, config_file=""))
    logging.getLogger("libai_b200").setLevel(logging.WARNING)
    torch.manual_seed(dutil.model_parallel_seed(cfg.train.seed))
    trainer = BenchTrainer(cfg)  # public API: builds model, optimizer, scheduler, loader, hooks
    step = trainer._trainer      # the StepTrainer behind trainer.run_step()
    topo = dutil.get_dist_util()
    # work units per step: tokens (images for the vision model)
    tokens_per_step = cfg.train.global_batch_size * (1 if args.model == "vit_l" else args.seq)
    assert cfg.train.global_batch_size == args.micro_batch * world, (cfg.train.global_batch_size, args.micro_batch, world)
    if args.fp8:
        ops.set_fp8(True)
    if args.fused_bias_grad >= 0:
        ops.set_fused_bias_grad(bool(args.fused_bias_grad))

    # ---- device-timed: batches staged on the device, CUDA events around exactly K trainer steps ---------------------
    staged = []
    it = iter(trainer.train_loader)
    for _ in range(lay["acc"] * 4):
        staged.append(DefaultTrainer.get_batch(next(it), "cuda"))
    torch.cuda.synchronize()
    acc = lay["acc"]

    def one_step(i):
        return step.train_on_batches([staged[(i * acc + k) % len(staged)] for k in range(acc)])

    for i in range(warmup):
        one_step(i)
    barrier()
    if clock_sampler is not None:
        clock_sampler.start()
    ops.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    t_enq = time.perf_counter()
    # `ncu --nvtx --nvtx-include "bench_step"` → exactly the timed steps.  A start/end range (process-wide), not
    # push/pop (per thread): the backward kernels are launched from the autograd engine's thread.
    nvtx = os.environ.get("LIBAI_B200_NVTX", "0") == "1"
    loss = None
    for i in range(steps):
        rid = torch.cuda.nvtx.range_start("bench_step") if nvtx else None
        loss = one_step(warmup + i)
        if nvtx:
            torch.cuda.synchronize()
            torch.cuda.nvtx.range_end(rid)
    e1.record()
    # host time spent ENQUEUEING the timed steps (no sync inside): close to the device time = the step is launch-bound
    enqueue_ms = max_over_ranks((time.perf_counter() - t_enq) * 1e3) / steps
    barrier()
    launches = ops.launch_count()
    clocks = clock_sampler.stop() if clock_sampler is not None else None
    dev_ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    res = {
        "value": tokens_per_step / (dev_ms * 1e-3),
        "ms_per_step": dev_ms,
        "parallelism": layout_name(lay),
        "global_batch": cfg.train.global_batch_size,
        "micro_batch_per_dp_rank": lay["micro"],
        "accumulation": lay["acc"],
        "cuda_graphs": bool(step.graphs_enabled),
        "gpu_launches": launches,
        "host_enqueue_ms_per_step": enqueue_ms,
        "clocks": clocks,
        "final_loss": None,
    }
    # (under pipeline parallelism only the last stage holds the loss: take it from whoever has it)
    lv = torch.full((1,), -1e30, dtype=torch.float32, device=dev)
    if loss:
        lv[0] = sum(v for k, v in loss.items() if "loss" in k).float()
    if world > 1:
        dist.all_reduce(lv, op=dist.ReduceOp.MAX)
    res["final_loss"] = float(lv) if float(lv) > -1e29 else None
    if dump_dir and rank == 0:        # before the end-to-end loop trains on
        dump_outputs(dump_dir, loss, step.model.module if hasattr(step.model, "module") else step.model)

    # ---- end to end through the trainer API: loader (pinned host) → H2D → step → loss D2H, every step ---------------
    if with_e2e:
        with EventStorage(0) as storage:
            trainer.storage = storage
            for i in range(max(2, min(warmup, 3))):
                trainer.iter = i
                trainer.run_step()
            barrier()
            h2d_counter["bytes"] = 0
            t0 = time.perf_counter()
            for i in range(steps):
                trainer.iter = 10 + i
                storage.iter = 10 + i
                # run_step = next(loader) [pinned host memory] → get_batch (H2D) → fwd/bwd/optimizer → write_metrics
                # (log_period = 1: the loss is reduced to rank 0 and read on the host, which synchronises the step)
                trainer.run_step()
            barrier()
            wall = time.perf_counter() - t0
            last = storage.latest().get("total_loss")
        wall = max_over_ranks(wall)
        res["e2e"] = {
            "value": tokens_per_step * steps / wall,
            "unit": "tokens/s",
            "h2d_bytes_per_step": h2d_counter["bytes"] // steps,
            "d2h_bytes_per_step": 4 * len(loss or {"lm_loss": 0}),
            "last_loss": float(last[0]) if last is not None else None,
            "api": "DefaultTrainer.run_step() with train.log_period=1",
        }
    # ---- tear down so that the next layout starts from a clean process-group / symmetric-memory state --------------
    del trainer, step, staged, it
    from libai_b200.ops import comm_gemm
    from libai_b200.parallel import symm_mem

    comm_gemm.reset_states()
    symm_mem.release_workspaces()    # collective: unmap the peers' buffers before anyone frees them
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    barrier()
    return res


def measure_pytorch_baseline(args, world, rank, local_rank, steps, warmup):
    """Stock-PyTorch comparator (baseline/pytorch_baseline.py), same model/config/global batch, same launch."""
    import importlib.util

    import torch
    import torch.distributed as dist

    spec = importlib.util.spec_from_file_location("pytorch_baseline", os.path.join(REPO, "baseline", "pytorch_baseline.py"))
    pb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(pb)
    dev = torch.device("cuda", local_rank)
    torch.manual_seed(1234)
    model, opt = pb.build(args.layers, args.hidden, args.heads, 50304, args.seq, dev, world, local_rank)
    g = torch.Generator(device="cpu").manual_seed(100 + rank)
    host = [torch.randint(0, 50304, (args.micro_batch, args.seq + 1), generator=g).pin_memory() for _ in range(4)]
    staged = [h.to(dev) for h in host]

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def mx(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for i in range(warmup):
        b = staged[i % 4]
        pb.train_step(model, opt, b[:, :-1], b[:, 1:])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        b = staged[i % 4]
        loss = pb.train_step(model, opt, b[:, :-1], b[:, 1:])
    e1.record()
    barrier()
    dev_ms = mx(e0.elapsed_time(e1)) / steps
    # end to end: pinned host → device copy of the step's tokens + loss read on the host, every step
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        b = host[i % 4].to(dev, non_blocking=True)
        lv = float(pb.train_step(model, opt, b[:, :-1], b[:, 1:]))
    barrier()
    wall = mx(time.perf_counter() - t0)
    tokens = args.micro_batch * world * args.seq
    out = {"impl": "stock PyTorch (SDPA, cuBLAS bf16 autocast, fused AdamW, DDP/NCCL) — baseline/pytorch_baseline.py",
           "value": tokens / (dev_ms * 1e-3), "ms_per_step": dev_ms, "e2e_value": tokens * steps / wall,
           "unit": "tokens/s", "final_loss": lv}
    del model, opt, staged
    import gc

    gc.collect()
    torch.cuda.empty_cache()
    return out


def _extras_flag_path():
    return os.path.join("/tmp", f"libai_b200_bench_fail_{os.environ.get('MASTER_PORT', '0')}_{os.getppid()}")


class _ExtrasWatchdog:
    """Keeps the headline line safe while the extra layouts run.  One node, so a flag file is the signal: the rank
    that fails (or sees a layout exceed ``limit_s``) creates it; a polling thread on every rank notices, rank 0 prints
    the JSON line with what was measured so far, and every rank leaves with exit code 0 (ranks blocked inside a
    collective cannot be unwound any other way)."""

    def __init__(self, world, emit, layouts, limit_s):
        import threading

        self.world, self.emit, self.layouts, self.limit_s = world, emit, layouts, limit_s
        self.flag = _extras_flag_path()     # (a stale file of an earlier launch was removed in main(), before the rendezvous)
        self.current, self.t0, self._stop = None, 0.0, False
        self.thread = None
        if world > 1:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()

    def begin(self, name):
        self.t0 = time.time()      # (before `current`: the poller must never pair a new phase with an old start time)
        self.current = name

    def idle(self):
        """Between two supervised phases: no time limit is running."""
        self.current = None

    def stop(self):
        self._stop = True
        self.current = None

    def _leave(self, why):
        name = self.current or "extra"
        self.layouts.setdefault(name, {"error": why})
        try:
            self.emit()
        finally:
            sys.stdout.flush()
            os._exit(0)

    def _poll(self):
        while not self._stop:
            time.sleep(0.5)
            if os.path.exists(self.flag):
                try:
                    why = open(self.flag).read()[:400] or "a peer rank failed"
                except OSError:
                    why = "a peer rank failed"
                self._leave(why)
            if self.current is not None and time.time() - self.t0 > self.limit_s:
                self.fail(self.current, f"layout exceeded {self.limit_s:.0f} s")

    def fail(self, name, why):
        if self.world == 1:
            return
        try:
            with open(self.flag, "w") as f:
                f.write(f"{name}: {why}")
        except OSError:
            pass
        time.sleep(1.5)          # let the peers' pollers see the flag before this process goes away
        self._leave(f"{name}: {why}")


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "ref":
        os.environ["LIBAI_B200_IMPL"] = "ref"

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    assert torch.cuda.is_available(), "bench.py needs a GPU"
    torch.cuda.set_device(local_rank)
    from libai_b200.utils import distributed as _dutil

    if local_rank == 0 and os.path.exists(_extras_flag_path()):
        os.remove(_extras_flag_path())       # before the rendezvous: no rank can have raised it yet in this launch
    _dutil.init_process_group("cuda")        # torchrun environment → NCCL (+ gloo for host objects)
    # the trainer's output directory (config dump, log): the source tree may be read-only
    args.output_dir = tempfile.mkdtemp(prefix="libai_b200_bench_")

    primary = layout_of(args, world)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    main_res = measure_native(args, primary, world, rank, local_rank, args.steps, args.warmup, not args.no_e2e, sampler,
                              args.dump_outputs)

    layouts = {main_res["parallelism"]: {k: main_res[k] for k in ("value", "ms_per_step", "cuda_graphs", "gpu_launches",
                                                                  "host_enqueue_ms_per_step", "global_batch")}}
    state = {"ref": None}      # filled in below; `emit` prints whatever has been measured when it is called

    def emit():
        if rank != 0:
            return
        ref_same_box = state["ref"]
        base = PUBLISHED_TOKENS_PER_S.get(world) if args.model == "gpt2" else None
        value = main_res["value"]
        spec = MODELS[args.model]
        unit = spec["unit"]
        line = {
            "metric": ("tokens/sec GPT-2 (nl24 h1024 a16 s1024) pre-training, device-timed max-over-ranks" if args.model == "gpt2"
                       else f"{unit.replace('/s', '/sec')} {args.model} pre-training, device-timed max-over-ranks"),
            "value": value,
            "unit": unit,
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": main_res["ms_per_step"],
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": (value / base) if base else None,
            "dtype": "bf16" if not args.fp8 else "fp8(e4m3)-fwd/bf16-bwd",
            "data": ("synthetic images" if args.model == "vit_l" else "synthetic tokens") + ", random-init weights",
            "impl": args.impl,
            "config": {
                "model": spec["name"].format(layers=args.layers, hidden=args.hidden, heads=args.heads),
                "global_batch": main_res["global_batch"],
                "micro_batch_per_gpu": args.micro_batch,
                "seq_len": args.seq,
                "parallelism": main_res["parallelism"],
                "l2_policy": "working set (weights+activations+optimizer state >> 126MB L2) exceeds L2 every step",
                "cuda_graphs": main_res["cuda_graphs"],
            },
            "clocks": main_res["clocks"],
            "e2e": main_res.get("e2e"),
            "gpu_launches": main_res["gpu_launches"],
            "host_enqueue_ms_per_step": main_res["host_enqueue_ms_per_step"],
            "host_cpus": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count(),
            "final_loss": main_res["final_loss"],
            # every layout measured in this launch (same model, same global batch): data parallel (the headline `value`),
            # tensor parallel with the collectives inside the GEMM kernels, and the 3-D layout
            "layouts": layouts,
            # stock-PyTorch comparator measured in this same launch on this same box (NOT the OneFlow reference)
            "ref_same_box": ref_same_box,
            "vs_ref_same_box": (value / ref_same_box["value"]) if ref_same_box else None,
        }
        print(json.dumps(line), flush=True)

    # Everything after the headline measurement runs under a watchdog: a failure or a hang in the comparator or in an
    # extra layout, on any rank, ends every rank cleanly with the line printed — it must never take the headline down.
    watch = _ExtrasWatchdog(world, emit, layouts, limit_s=float(os.environ.get("LIBAI_B200_BENCH_EXTRA_LIMIT_S", "420")))
    if args.ref_same_box and args.impl == "native" and args.model == "gpt2":
        watch.begin("ref_same_box")
        try:
            state["ref"] = measure_pytorch_baseline(args, world, rank, local_rank, min(args.steps, 10), 3)
        except BaseException as e:  # noqa: BLE001
            watch.fail("ref_same_box", f"{type(e).__name__}: {str(e)[:300]}")   # does not return when world > 1
            state["ref"] = None
            layouts["ref_same_box"] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
        watch.idle()

    if args.extras and args.impl == "native" and args.model == "gpt2" and not args.layout and args.tp == 1 and args.pp == 1:
        # the model-parallel layouts that fit this GPU count, same global batch, same launch (BASELINE.json configs:
        # "TP=2 DP=4", "TP=2 PP=2 DP=2 + ZeRO-1").  They run LAST and under a watchdog: the headline measurement above
        # is already complete, and a failure (or a hang) in an extra layout on any rank ends every rank cleanly with
        # the line printed — it must never take the headline down.
        names = {2: ["tp2"], 4: ["tp2", "3d"], 8: ["tp2", "3d"]}.get(world, [])
        for name in names:
            lay = layout_of(args, world, name)
            watch.begin(name)
            try:
                if os.environ.get("LIBAI_B200_BENCH_INJECT_EXTRA_FAIL", "") == str(rank):   # exercises the watchdog path
                    raise RuntimeError("injected failure in an extra layout")
                r = measure_native(args, lay, world, rank, local_rank, args.extra_steps, max(3, min(args.warmup, 4)), False)
                layouts[r["parallelism"]] = {k: r[k] for k in ("value", "ms_per_step", "cuda_graphs", "gpu_launches",
                                                               "host_enqueue_ms_per_step", "global_batch", "final_loss")}
                layouts[r["parallelism"]]["steps"] = args.extra_steps
            except BaseException as e:  # noqa: BLE001 - incl. KeyboardInterrupt/SystemExit raised inside the trainer
                watch.fail(name, f"{type(e).__name__}: {str(e)[:300]}")   # does not return when world > 1
                layouts[name] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
            watch.idle()
    watch.stop()

    emit()
    shutil.rmtree(args.output_dir, ignore_errors=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
