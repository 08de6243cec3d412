"""Small unit tests mirroring the reference's tests/test_basic.py, test_utils.py, test_activations.py, test_wandb.py
and test_layernorm_order.py (CPU)."""
import os
import sys

import pytest
import torch
from torch.nn import functional as F

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), os.pardir))
sys.path.insert(0, ROOT)


def test_import_and_compat_alias():
    import megatron_llm_b200  # noqa: F401
    import megatron
    from megatron.core import tensor_parallel, parallel_state  # noqa: F401
    from megatron.model import GPTModel, LlamaModel  # noqa: F401
    from megatron.core.tensor_parallel import ColumnParallelLinear, RowParallelLinear, vocab_parallel_cross_entropy  # noqa
    assert megatron.get_args is megatron_llm_b200.get_args


def test_divide_and_viewless_helpers():
    from megatron_llm_b200.utils import core_utils as util
    assert util.divide(4, 2) == 2
    with pytest.raises(AssertionError):
        util.divide(4, 5)
    inp = torch.rand(3, 4)
    assert torch.equal(inp, util.make_viewless_tensor(inp, True, True))
    assert torch.equal(inp, util.make_viewless_tensor(inp, True, False))
    view = inp.view(4, 3)
    out = util.make_viewless_tensor(view, False, False)
    assert out._base is None and torch.equal(out, view)
    t = torch.zeros(3, 4)
    new = torch.rand(3, 4)
    util.safely_set_viewless_tensor_data(t, new)
    assert torch.equal(t, new)
    assert torch.equal(util.assert_viewless_tensor(inp), inp)
    assert all(torch.equal(a, inp) for a in util.assert_viewless_tensor([inp, inp]))


@pytest.mark.parametrize("name,act", [("liglu", lambda x: x), ("geglu", F.gelu), ("reglu", F.relu), ("swiglu", F.silu)])
def test_glu_activations(name, act):
    from megatron_llm_b200.models.activations import GLU_ACTIVATIONS
    torch.manual_seed(11)
    x = torch.randn(3, 257, 2 * 38)
    x1, x2 = x.chunk(2, dim=-1)
    out = GLU_ACTIVATIONS[name](x)
    assert list(out.shape) == [3, 257, 38]
    assert torch.allclose(out, x1 * act(x2), atol=1e-6)


def test_wandb_shim_without_wandb(tmp_path, monkeypatch):
    """The TensorBoard-compatible shim must work (mirror to TB, drop 'vs samples' duplicates) with wandb offline or
    absent."""
    from megatron_llm_b200 import wandb_logger
    monkeypatch.setenv("WANDB_MODE", "offline")
    monkeypatch.setenv("WANDB_DIR", str(tmp_path))
    cfg = wandb_logger.WandBConfig.default("test-logger")
    cfg.logdir = str(tmp_path / "tb")
    cfg.with_tensorboard = True
    w = wandb_logger.WandbTBShim(cfg)
    for step in range(3):
        w.add_scalar("lm loss", 1.0 / (step + 1), step)
        w.add_scalar("lm loss vs samples", 1.0, step * 8)
    w.add_text("args", "x=1")
    w.flush_all()
    assert w._pending == {}


def _layer(rank, world, extra):
    from megatron_llm_b200.initialize import initialize_megatron
    from megatron_llm_b200.global_vars import get_args
    initialize_megatron(args_list=["--num_layers", "2", "--hidden_size", "16", "--num_attention_heads", "4",
                                   "--seq_length", "8", "--max_position_embeddings", "8", "--micro_batch_size", "2",
                                   "--tokenizer_type", "NullTokenizer", "--vocab_file", "32", "--train_iters", "1",
                                   "--lr", "1e-3", "--hidden_dropout", "0.0", "--attention_dropout", "0.0",
                                   "--use_bias"] + extra)
    args = get_args()
    from megatron_llm_b200.models.activations import init_method_normal, scaled_init_method_normal
    from megatron_llm_b200.models.enums import LayerType
    from megatron_llm_b200.models.transformer import ParallelTransformerLayer
    torch.manual_seed(0)
    layer = ParallelTransformerLayer(init_method_normal(0.02), scaled_init_method_normal(0.02, 2), 1,
                                     layer_type=LayerType.encoder, args=args, world_size=1)
    x = torch.randn(8, 2, 16)
    mask = torch.zeros(2, 1, 8, 8, dtype=torch.bool)
    out = layer(x, mask)
    return layer, x, out


def _layernorm_order(rank, world):
    """pre-LN: out = x' + mlp(LN2(x')), x' = x + attn(LN1(x));  post-LN: out = LN(x' + mlp(x')), x' = x + attn(x)."""
    layer, x, out = _layer(rank, world, [])
    mask = torch.zeros(2, 1, 8, 8, dtype=torch.bool)
    a, ab = layer.self_attention(layer.input_layernorm(x), mask)
    x1 = x + a + (ab if ab is not None else 0)
    m, mb = layer.mlp(layer.post_attention_layernorm(x1))
    ref = x1 + m + (mb if mb is not None else 0)
    assert torch.allclose(out, ref, atol=1e-5), (out - ref).abs().max()
    assert isinstance(layer.output_layernorm, torch.nn.Identity)


def _post_ln(rank, world):
    layer, x, out = _layer(rank, world, ["--use_post_ln"])
    assert isinstance(layer.input_layernorm, torch.nn.Identity)
    mask = torch.zeros(2, 1, 8, 8, dtype=torch.bool)
    a, ab = layer.self_attention(x, mask)
    x1 = x + a + (ab if ab is not None else 0)
    m, mb = layer.mlp(layer.post_attention_layernorm(x1))
    ref = layer.output_layernorm(x1 + m + (mb if mb is not None else 0))
    assert torch.allclose(out, ref, atol=1e-5), (out - ref).abs().max()


def test_layernorm_order():
    from tests.dist_utils import run_distributed
    run_distributed(_layernorm_order, 1)
    run_distributed(_post_ln, 1)


def test_bench_presets_build_valid_arguments(monkeypatch):
    """bench.py's argument builder for the headline run (TP = #GPUs) and for the other BASELINE.json configurations
    must produce flag lists that the framework's parser and validator accept."""
    import argparse
    import bench
    import finetune
    from megatron_llm_b200.arguments import parse_args, validate_args

    def ns(**kw):
        base = dict(model="llama2-7b", layers=None, seq=4096, micro_batch=1, global_batch=8, graph=-1, tp=None, pp=1,
                    recompute=False, dist_opt=False)
        base.update(kw)
        return argparse.Namespace(**base)

    cases = [
        (ns(), 1, "tp1", (1, 1, 1)),
        (ns(), 8, "tp8+sp", (8, 1, 1)),
        (ns(model="mistral-7b", tp=2, dist_opt=True), 8, "tp2+sp+dp4(zero1)", (2, 1, 4)),
        (ns(model="falcon-40b", tp=4, pp=2, global_batch=16), 8, "tp4+sp+pp2", (4, 2, 1)),
        (ns(model="llama2-70b", recompute=True), 8, "tp8+sp+recompute", (8, 1, 1)),
    ]
    assert [bench.resolve_micro_batch(ns(micro_batch=0), n) for n in (1, 2, 4, 8)] == [1, 2, 4, 8]
    assert bench.resolve_micro_batch(ns(micro_batch=0, model="mistral-7b", tp=2, dist_opt=True), 8) == 2
    assert bench.resolve_micro_batch(ns(micro_batch=0, model="falcon-40b", tp=4, pp=2, global_batch=16), 8) == 1
    assert bench.resolve_micro_batch(ns(micro_batch=3), 8) == 3
    for a, gpus, name, layout in cases:
        assert bench.parallel_layout(a, gpus) == layout
        assert bench.parallelism_string(a, gpus) == name
        argv, vocab = bench.megatron_argv(a, gpus)
        monkeypatch.setenv("WORLD_SIZE", str(gpus))
        monkeypatch.setenv("RANK", "0")
        args = parse_args(finetune.extra_args, False, args_list=argv + ["--tokenizer_type", "NullTokenizer",
                                                                        "--vocab_file", str(vocab), "--data_type",
                                                                        "synthetic"])
        if not hasattr(args, "data_parallel_size"):
            args = validate_args(args, {})
        assert args.tensor_model_parallel_size == layout[0] and args.pipeline_model_parallel_size == layout[1]
        assert args.data_parallel_size == layout[2]
        # the micro-batch graph is requested when one TP group of > 1 GPUs spans the job, no pipeline, no recompute
        assert bool(getattr(args, "cuda_graph_microbatch", False)) == (layout[0] > 1 and layout[0] == gpus
                                                                        and layout[1] == 1 and not a.recompute)


def test_bench_dump_outputs_reads_the_same_positions_every_run(tmp_path):
    """``bench.py --dump-outputs``: float32 loss, grad norm and a parameter sample whose positions depend only on the
    tensor sizes, so the files of two runs with the same arguments line up element for element."""
    import numpy as np
    import bench
    torch.manual_seed(0)
    model = [torch.nn.Sequential(torch.nn.Linear(64, 48), torch.nn.LayerNorm(48)).to(torch.bfloat16)]
    loss = {"lm loss": torch.tensor(10.5)}
    bench.dump_outputs(str(tmp_path / "a"), loss, torch.tensor([2.25]), model)
    bench.dump_outputs(str(tmp_path / "b"), {}, 3.0, model)
    assert sorted(os.listdir(tmp_path / "a")) == ["grad_norm.npy", "lm_loss.npy", "params_sample.npy"]
    assert sorted(os.listdir(tmp_path / "b")) == ["grad_norm.npy", "params_sample.npy"]
    assert np.load(tmp_path / "a" / "lm_loss.npy").tolist() == [10.5]
    assert np.load(tmp_path / "a" / "grad_norm.npy").dtype == np.float32
    a, b = np.load(tmp_path / "a" / "params_sample.npy"), np.load(tmp_path / "b" / "params_sample.npy")
    params = list(model[0].parameters())
    assert a.dtype == np.float32 and a.shape == (len(params), bench.DUMP_SAMPLES_PER_TENSOR)
    assert np.array_equal(a, b)
    for row, p in zip(a, params):       # every sampled value is an element of its tensor; 4096 draws cover 48 elements
        vals = set(p.detach().float().reshape(-1).tolist())
        assert set(row.tolist()) <= vals
        if p.numel() <= 48:
            assert set(row.tolist()) == vals


def test_reference_helper_names_behave():
    """Small public helpers that scripts written against the reference import by name."""
    import os
    from megatron_llm_b200.models import activations as A
    from megatron_llm_b200.models import norms as N
    from megatron_llm_b200.models import transformer as T
    from megatron_llm_b200.optimizer import distrib_optimizer as D
    from megatron_llm_b200.optimizer import optimizer as O
    torch.manual_seed(0)
    x = torch.randn(5, 7, dtype=torch.float64, requires_grad=True)
    b = torch.randn(7, dtype=torch.float64, requires_grad=True)
    y = A.bias_gelu(b, x)
    assert torch.allclose(y, F.gelu(x + b, approximate="tanh"), atol=1e-6)
    g = torch.randn_like(y)
    dx, = torch.autograd.grad(F.gelu(x + b, approximate="tanh"), x, g)
    assert torch.allclose(A.bias_gelu_back(g, b, x), dx, atol=1e-5)
    out = A.GeLUFunction.apply(x, b)
    gx, gb = torch.autograd.grad(out, (x, b), g)
    assert torch.allclose(gx, dx, atol=1e-5) and torch.allclose(gb, dx.sum(0), atol=1e-5)
    # bias-dropout-add family (inference closures are deterministic)
    r = torch.randn(5, 7)
    f = T.get_bias_dropout_add(False)
    assert torch.allclose(f(x.float(), b.float(), r, 0.3), r + x.float() + b.float())
    assert torch.allclose(T.get_dropout_add(False)(x.float(), None, r, 0.3), r + x.float())
    assert torch.allclose(T.bias_dropout_add_fused_inference(x.float(), b.float(), r, 0.5), r + x.float() + b.float())
    kept = T.bias_dropout_add_fused_train(torch.ones(64, 64), None, torch.zeros(64, 64), 0.5)
    assert set(kept.unique().tolist()) <= {0.0, 2.0} and 0.3 < (kept > 0).float().mean() < 0.7
    # functional layer norm
    w, bias = torch.rand(7), torch.rand(7)
    got = N.FusedLayerNormAffineFunction.apply(r, w, bias, (7,), 1e-5)
    assert torch.allclose(got, F.layer_norm(r, (7,), w, bias, 1e-5), atol=1e-5)
    # optimizer class tree + shard range helper
    assert issubclass(O.Float16OptimizerWithFloat16Params, O.MixedPrecisionOptimizer)
    assert issubclass(D.DistributedOptimizer, O.MixedPrecisionOptimizer)
    assert not issubclass(O.FP32Optimizer, O.MixedPrecisionOptimizer)
    rg = D.Range(8, 20)
    assert (rg.size, str(rg.normalize(2))) == (12, "2,14 [12]")
    # checkpoint file name
    from megatron_llm_b200.checkpointing import get_checkpoint_name
    assert get_checkpoint_name("/c", 12, False, True, 1, 3) == os.path.join("/c", "iter_0000012", "mp_rank_01_003",
                                                                            "model_optim_rng.pt")
    assert get_checkpoint_name("/c", 0, True, False, 0, 0) == os.path.join("/c", "release", "mp_rank_00",
                                                                           "model_optim_rng.pt")


def test_conversion_helper_names():
    import weights_conversion.hf_to_megatron as C
    import weights_conversion.megatron_to_hf as R
    import verify_correctness as V
    assert V.Llama2Wrapper is V.MetaLlamaWrapper
    torch.manual_seed(0)
    h, n, nkv, ffn = 64, 8, 2, 96
    wq, wk, wv = torch.randn(h, h), torch.randn(h // 4, h), torch.randn(h // 4, h)
    up, gate = torch.randn(ffn, h), torch.randn(ffn, h)
    meta = {"tok_embeddings.weight": torch.randn(32, h), "norm.weight": torch.ones(h), "output.weight": torch.randn(32, h),
            "layers.0.attention.wo.weight": torch.randn(h, h), "layers.0.ffn_norm.weight": torch.ones(h),
            "layers.0.attention_norm.weight": torch.ones(h), "layers.0.feed_forward.w2.weight": torch.randn(h, ffn),
            "layers.0.feed_forward.w3.weight": up, "layers.0.feed_forward.w1.weight": gate,
            "layers.0.attention.wq.weight": wq, "layers.0.attention.wk.weight": wk, "layers.0.attention.wv.weight": wv}
    mega = C.llama_like_to_megatron(dict(meta), 1, h, n, nkv, "hf")
    q2, k2, v2 = R.convert_wqkv(mega, 0, n, nkv)
    assert torch.equal(q2, wq) and torch.equal(k2, wk) and torch.equal(v2, wv)
    w1, w3 = R.convert_ffn(mega, 0, ffn)
    assert torch.equal(w1, gate) and torch.equal(w3, up)
