"""GPU tier (run on a B200 with ``pytest -m gpu``): every sm_100a kernel against fp32 PyTorch references, the native
training step against the PyTorch/cuBLAS reference path, the fused NVLink collectives (when ≥ 2 GPUs are visible) and
the bench / smoke contracts.  The native extension must be the code that runs: tests fail if it is not loaded."""
import json
import os
import subprocess
import sys

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _run(cmd, timeout=900, env=None):
    e = dict(os.environ)
    e.update(env or {})
    e["PYTHONPATH"] = REPO + os.pathsep + e.get("PYTHONPATH", "")
    return subprocess.run(cmd, cwd=REPO, capture_output=True, text=True, timeout=timeout, env=e)


def test_native_extension_is_loaded():
    from libai_b200 import ops

    ext = ops.load_ext()
    assert ext is not None and os.path.exists(os.path.join(REPO, "libai_b200", "_C.so"))
    x = torch.randn(256, 256, device="cuda").bfloat16()
    before = ops.launch_count()
    from libai_b200.ops import functional as OF

    y = OF.linear(x, x)
    assert ops.launch_count() > before and torch.isfinite(y.float()).all()


def test_kernels_match_fp32_references(tmp_path):
    out = str(tmp_path / "kc.json")
    r = _run([sys.executable, "tests/gpu_kernel_check.py", "--quick", "--out", out])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    results = json.load(open(out))
    bad = [x["name"] for x in results if not x.get("ok")]
    assert not bad and len(results) > 40, bad


def _tiny_gpt(impl):
    os.environ["LIBAI_B200_IMPL"] = impl
    from libai_b200.config import DictConfig
    from libai_b200.models import GPTForPreTraining
    from libai_b200.optim import AdamW
    from libai_b200.utils import distributed as dutil

    dutil.reset_dist_util()
    torch.manual_seed(0)
    cfg = DictConfig(dict(
        hidden_layers=2, vocab_size=512, hidden_size=256, ffn_hidden_size=1024, num_attention_heads=4, max_seq_length=256,
        embedding_dropout_prob=0.0, attention_dropout_prob=0.0, output_dropout_prob=0.0, layernorm_epsilon=1e-5,
        initializer_range=0.02, use_scaled_init_for_output_weights=True, bias_gelu_fusion=True, bias_dropout_fusion=True,
        scale_mask_softmax_fusion=True, apply_query_key_layer_scaling=False, apply_residual_post_layernorm=False,
        amp_enabled=False))
    model = GPTForPreTraining(cfg).cuda().bfloat16()
    opt = AdamW([{"params": list(model.parameters())}], lr=1e-3)
    opt.setup()
    g = torch.Generator(device="cuda").manual_seed(1)
    ids = torch.randint(0, 512, (4, 256), device="cuda", generator=g)  # one fixed batch: the loss must go down
    losses = []
    for _ in range(6):
        opt.zero_grad()
        loss = model(ids, ids)["lm_loss"]
        loss.backward()
        opt.step()
        losses.append(loss.item())
    return losses


def test_native_training_step_matches_reference_path():
    from libai_b200 import ops

    n0 = ops.launch_count()
    native = _tiny_gpt("native")
    assert ops.launch_count() - n0 > 50, "the native kernels did not run"
    ref = _tiny_gpt("ref")
    os.environ["LIBAI_B200_IMPL"] = "native"
    # two different bf16 implementations: identical maths, different rounding points → close at step 0, same
    # convergence afterwards (trajectories drift slowly apart at lr 1e-3)
    assert abs(native[0] - ref[0]) < 6e-2 and all(abs(a - b) < 0.3 for a, b in zip(native, ref)), (native, ref)
    assert native[-1] < native[0] - 0.05, native


def test_cuda_graph_blocks_match_eager():
    """Blocks replayed from CUDA graphs (engine/cuda_graphs.py) train like the eager blocks: same kernels, same
    addresses (main_grad accumulation happens inside the captured backward)."""
    from libai_b200 import ops
    from libai_b200.config import DictConfig
    from libai_b200.engine.cuda_graphs import enable_for_model
    from libai_b200.layers._param import param_defaults
    from libai_b200.models import GPTForPreTraining
    from libai_b200.optim import AdamW, get_default_optimizer_params
    from libai_b200.utils import distributed as dutil

    os.environ["LIBAI_B200_IMPL"] = "native"
    cfg = DictConfig(dict(
        hidden_layers=3, vocab_size=512, hidden_size=256, ffn_hidden_size=1024, num_attention_heads=4, max_seq_length=256,
        embedding_dropout_prob=0.0, attention_dropout_prob=0.0, output_dropout_prob=0.0, layernorm_epsilon=1e-5,
        initializer_range=0.02, use_scaled_init_for_output_weights=True, bias_gelu_fusion=True, bias_dropout_fusion=True,
        scale_mask_softmax_fusion=True, apply_query_key_layer_scaling=False, apply_residual_post_layernorm=False,
        amp_enabled=True))
    runs = []
    for graphed in (False, True):
        dutil.reset_dist_util()
        dutil.setup_dist_util(DictConfig(dict(data_parallel_size=1, tensor_parallel_size=1, pipeline_parallel_size=1)))
        with param_defaults(dtype=torch.bfloat16, device="cuda", seed=3):
            model = GPTForPreTraining(cfg).train()
        opt = AdamW(get_default_optimizer_params(model, clip_grad_max_norm=1.0, clip_grad_norm_type=2.0), lr=1e-3)
        opt.configure(param_names={id(p): n for n, p in model.named_parameters()})
        opt.setup()
        g = torch.Generator(device="cuda").manual_seed(7)
        batches = [torch.randint(0, 512, (4, 256), device="cuda", generator=g) for _ in range(5)]
        if graphed:
            keys_before = list(model.state_dict().keys())
            assert enable_for_model(model, dict(input_ids=batches[0], labels=batches[0]))
            assert list(model.state_dict().keys()) == keys_before          # checkpoints keep their names
        losses = []
        n0 = ops.launch_count()
        for ids in batches:
            opt.zero_grad()
            loss = model(ids, ids)["lm_loss"]
            loss.backward()
            opt.step()
            losses.append(loss.item())
        runs.append((losses, ops.launch_count() - n0))
    (eager, n_eager), (graph, n_graph) = runs
    assert all(abs(a - b) < 2e-2 for a, b in zip(eager, graph)), (eager, graph)
    assert graph[-1] < graph[0]
    assert abs(n_graph - n_eager) <= 0.1 * n_eager, (n_eager, n_graph)     # replayed kernels are still counted


def test_fp8_forward_gemms_train_like_bf16():
    """``ops.set_fp8(True)``: the linear layers' forward GEMMs take E4M3 operands (quantise + tcgen05 kind::f8f6f4
    kernel); losses track the bf16 run, eagerly (cached weight copies refreshed per optimizer step) and under CUDA
    graphs (quantisation captured)."""
    from libai_b200 import ops
    from libai_b200.config import DictConfig
    from libai_b200.engine.cuda_graphs import enable_for_model
    from libai_b200.layers._param import param_defaults
    from libai_b200.models import GPTForPreTraining
    from libai_b200.optim import AdamW, get_default_optimizer_params
    from libai_b200.utils import distributed as dutil

    os.environ["LIBAI_B200_IMPL"] = "native"
    cfg = DictConfig(dict(
        hidden_layers=2, vocab_size=512, hidden_size=256, ffn_hidden_size=1024, num_attention_heads=4, max_seq_length=256,
        embedding_dropout_prob=0.0, attention_dropout_prob=0.0, output_dropout_prob=0.0, layernorm_epsilon=1e-5,
        initializer_range=0.02, use_scaled_init_for_output_weights=True, bias_gelu_fusion=True, bias_dropout_fusion=True,
        scale_mask_softmax_fusion=True, apply_query_key_layer_scaling=False, apply_residual_post_layernorm=False,
        amp_enabled=True))
    runs = {}
    try:
        for mode in ("bf16", "fp8", "fp8+graphs"):
            ops.set_fp8(mode != "bf16")
            dutil.reset_dist_util()
            dutil.setup_dist_util(DictConfig(dict(data_parallel_size=1, tensor_parallel_size=1, pipeline_parallel_size=1)))
            with param_defaults(dtype=torch.bfloat16, device="cuda", seed=3):
                model = GPTForPreTraining(cfg).train()
            opt = AdamW(get_default_optimizer_params(model, clip_grad_max_norm=1.0, clip_grad_norm_type=2.0), lr=1e-3)
            opt.configure(param_names={id(p): n for n, p in model.named_parameters()})
            opt.setup()
            g = torch.Generator(device="cuda").manual_seed(7)
            batches = [torch.randint(0, 512, (4, 256), device="cuda", generator=g) for _ in range(6)]
            if mode.endswith("graphs"):
                assert enable_for_model(model, dict(input_ids=batches[0], labels=batches[0]))
            losses = []
            for ids in batches:
                opt.zero_grad()
                loss = model(ids, ids)["lm_loss"]
                loss.backward()
                opt.step()
                losses.append(loss.item())
            runs[mode] = losses
    finally:
        ops.set_fp8(False)
    assert all(abs(a - b) < 5e-2 for a, b in zip(runs["bf16"], runs["fp8"])), runs
    assert all(abs(a - b) < 2e-2 for a, b in zip(runs["fp8"], runs["fp8+graphs"])), runs
    assert runs["fp8"][-1] < runs["fp8"][0] and runs["fp8"] != runs["bf16"]


def test_smoke_entry_point():
    sys.path.insert(0, REPO)
    import __graft_entry__

    __graft_entry__.smoke()


def test_bench_contract(tmp_path):
    import numpy as np

    dump = tmp_path / "outputs"
    r = _run([sys.executable, "bench.py", "--steps", "2", "--warmup", "3", "--dump-outputs", str(dump)], timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["value"] > 0 and line["gpu_launches"] > 0 and line["e2e"]["h2d_bytes_per_step"] > 0
    # what the last timed step computed: its loss (the line's final_loss) and a sample of the updated weights
    assert sorted(os.listdir(dump)) == ["lm_loss.npy", "state_sample.npy"]
    assert sum(os.path.getsize(dump / f) for f in os.listdir(dump)) <= 64 << 20
    loss, state = np.load(dump / "lm_loss.npy"), np.load(dump / "state_sample.npy")
    assert loss.dtype == state.dtype == np.float32 and np.isfinite(state).all()
    assert abs(float(loss) - line["final_loss"]) < 1e-6 * abs(line["final_loss"])
    ref = _run([sys.executable, "bench.py", "--impl", "reference"])
    assert ref.returncode == 0 and json.loads(ref.stdout.strip().splitlines()[-1])["impl"] == "reference"


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_fused_nvlink_collectives(tmp_path):
    out = str(tmp_path / "comm.json")
    r = _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
              "--master-port", "29533", "tests/gpu_comm_check.py", "--out", out], timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    results = json.load(open(out))
    assert all(x.get("ok") for x in results), [x for x in results if not x.get("ok")]


def _trajectory(tmp_path, name, nproc, *flags):
    out = str(tmp_path / f"{name}.json")
    cmd = [sys.executable]
    if nproc > 1:
        cmd += ["-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
                "--master-port", "29541"]
    r = _run(cmd + ["tests/gpu_tp_parity.py", "--out", out, *flags], timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.load(open(out))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_fused_tensor_parallel_trains_like_one_gpu(tmp_path):
    """VERDICT r1 #1(d): GPT-2 with TP2 + sequence parallelism + AG→GEMM / GEMM→RS kernels (blocks replayed from CUDA
    graphs) follows the single-GPU native loss trajectory within bf16 tolerance — and so does the NCCL form."""
    one = _trajectory(tmp_path, "one", 1)
    fused = _trajectory(tmp_path, "tp2_fused", 2, "--tp", "2", "--fused", "1")
    nccl = _trajectory(tmp_path, "tp2_nccl", 2, "--tp", "2", "--fused", "0")
    assert fused["graphs"], "fused tensor-parallel blocks must be CUDA-graph captured"
    assert one["losses"][-1] < one["losses"][0] - 0.2, one["losses"]        # it actually learns
    for a, b, c in zip(one["losses"], fused["losses"], nccl["losses"]):
        assert abs(a - b) < 0.05 * max(1.0, abs(a)), (one["losses"], fused["losses"])
        assert abs(a - c) < 0.05 * max(1.0, abs(a)), (one["losses"], nccl["losses"])
