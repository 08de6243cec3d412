"""Headline benchmark: Llama-2-7B training step, bf16, seq 4096, TP = #GPUs (sequence parallel), synthetic data,
random-init weights -> tokens/s for the whole job (BASELINE.json metric).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the unmodified reference (baseline/_ref) on the same config
    python bench.py ... --dump-outputs DIR    # also write the last timed step's loss, grad norm, parameters as .npy

Timing: W untimed warm-up steps, then exactly K steps bracketed by barrier + torch.cuda.synchronize(), measured with
CUDA events on the launching stream, MAX over ranks.  Two timed phases through the SAME public API
(``setup_model_and_optimizer`` + ``train_step`` + ``finetune.forward_step``):
  * ``value``: inputs already resident on the device, loss left on the device;
  * ``e2e``:   every micro-batch is copied host->device from pinned memory inside the timed region and the step's
               loss is read back to the host every step.
Every step streams > 100 GB of weights/grads/optimizer state, far larger than the 126 MB L2, so no explicit L2
flush is needed between iterations.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODELS = {
    # name: (layers, hidden, heads, kv_heads, ffn, vocab)
    "llama2-7b": (32, 4096, 32, 32, 11008, 32000),
    "llama2-70b": (80, 8192, 64, 8, 28672, 32000),
    "mistral-7b": (32, 4096, 32, 8, 14336, 32000),
    "llama2-tiny": (4, 1024, 8, 8, 2816, 32000),
    "mistral-tiny": (4, 1024, 8, 2, 3584, 32000),
    "falcon-tiny": (4, 1024, 16, 2, 4096, 65024),     # head_dim 64, GQA, parallel attention + MLP (Falcon-40B shape, small)
    "falcon-40b": (60, 8192, 128, 8, 32768, 65024),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--model", default="llama2-7b", choices=list(MODELS))
    p.add_argument("--seq", type=int, default=4096)
    p.add_argument("--global_batch", type=int, default=8)
    p.add_argument("--micro_batch", type=int, default=0,
                   help="sequences per micro-batch; 0 = auto: the tensor-parallel size when there is no pipeline (every "
                        "GPU then runs kernels of the single-GPU size and the TP collectives move tp x larger messages "
                        "tp x less often), 1 with pipeline parallelism.  Same rule for both --impl arms.")
    p.add_argument("--layers", type=int, default=None, help="DEV ONLY: override layer count (invalidates the number)")
    # the headline config is TP = #GPUs; the other BASELINE.json configs (Mistral TP2xDP4, Falcon-40B TP4xPP2,
    # Llama-2-70B TP8 + recompute) are reachable with these
    p.add_argument("--tp", type=int, default=None, help="tensor-parallel size (default: --gpus)")
    p.add_argument("--pp", type=int, default=1, help="pipeline-parallel size; data-parallel = gpus / (tp * pp)")
    p.add_argument("--recompute", action="store_true", help="full activation recompute (uniform, 1 layer per chunk)")
    p.add_argument("--dist_opt", action="store_true", help="ZeRO-1 distributed optimizer over the DP group")
    p.add_argument("--no_e2e", action="store_true")
    p.add_argument("--graph", type=int, default=-1,
                   help="1/0: replay each micro-batch from a CUDA graph (default: on when one TP group of > 1 GPUs spans "
                        "the job; see host_enqueue_ms_per_step)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step computed to DIR/*.npy (see "
                        "dump_outputs), so that two builds run with the same arguments can be compared output for output")
    a = p.parse_args()
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs is implemented for --impl ours only")
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def parallel_layout(a, n_gpus):
    """(tp, pp, dp) for this run: TP = #GPUs unless --tp / --pp say otherwise."""
    pp = getattr(a, "pp", 1) or 1
    tp = getattr(a, "tp", None) or max(n_gpus // pp, 1)
    assert n_gpus % (tp * pp) == 0, f"--gpus {n_gpus} is not a multiple of tp*pp = {tp * pp}"
    return tp, pp, n_gpus // (tp * pp)


def resolve_micro_batch(a, n_gpus):
    """The micro-batch both arms use (see --micro_batch)."""
    if a.micro_batch and a.micro_batch > 0:
        return a.micro_batch
    tp, pp, dp = parallel_layout(a, n_gpus)
    per_dp = a.global_batch // dp
    mb = tp if pp == 1 else 1
    while mb > 1 and per_dp % mb:
        mb //= 2
    return max(1, min(mb, per_dp))


def bench_config(a, n_gpus):
    """``config`` of the JSON line: identical keys and values from both arms for the same command line."""
    return {"model": a.model if not a.layers else f"{a.model}[layers={a.layers}:DEV-ONLY]",
            "global_batch": a.global_batch, "micro_batch": a.micro_batch, "seq_len": a.seq,
            "parallelism": parallelism_string(a, n_gpus),
            "optimizer": "AdamW fp32 master weights (in the timed region), clip 1.0",
            "l2": "no flush needed: each step streams >100 GB of weights/grads/optimizer state (>> 126 MB L2)"}


METRIC = "tokens/sec (whole job, device-timed, max over ranks), {model} {par} seq{seq} training step"


def parallelism_string(a, n_gpus):
    tp, pp, dp = parallel_layout(a, n_gpus)
    s = f"tp{tp}" + ("+sp" if tp > 1 else "")
    if pp > 1:
        s += f"+pp{pp}"
    if dp > 1:
        s += f"+dp{dp}" + ("(zero1)" if getattr(a, "dist_opt", False) else "")
    if getattr(a, "recompute", False):
        s += "+recompute"
    return s


def megatron_argv(a, n_gpus):
    layers, hidden, heads, kv, ffn, vocab = MODELS[a.model]
    if a.layers:
        layers = a.layers
    tp, pp = parallel_layout(a, n_gpus)[:2]
    family = a.model.split("-")[0].rstrip("2")          # llama / mistral / falcon
    argv = ["--model_name", {"llama": "llama2", "mistral": "mistral", "falcon": "falcon"}[family],
            "--num_layers", str(layers), "--hidden_size", str(hidden), "--num_attention_heads", str(heads),
            "--num_attention_heads_kv", str(kv), "--ffn_hidden_size", str(ffn), "--seq_length", str(a.seq),
            "--max_position_embeddings", str(a.seq), "--micro_batch_size", str(a.micro_batch),
            "--global_batch_size", str(a.global_batch), "--tensor_model_parallel_size", str(tp),
            "--pipeline_model_parallel_size", str(pp), "--train_iters", "1000000", "--lr", "1e-5", "--min_lr", "1e-6",
            "--lr_decay_style", "cosine", "--weight_decay", "0.1", "--clip_grad", "1.0", "--adam_beta1", "0.9",
            "--adam_beta2", "0.95", "--adam_eps", "1e-5", "--bf16", "--use_flash_attn",
            "--position_embedding_type", "rotary",
            "--hidden_dropout", "0.0", "--attention_dropout", "0.0", "--layernorm_epsilon", "1e-5",
            "--no_bias_gelu_fusion", "--no_bias_dropout_fusion", "--log_interval", "1000000", "--eval_iters", "0",
            "--eval_interval", "1000000", "--num_workers", "0", "--seed", "1234"]
    if family == "falcon":      # parallel attention + MLP, two layernorms, GELU MLP, tied embeddings, MQA/GQA
        argv += ["--parallel_attn", "--parallel_layernorm"]
    else:
        argv += ["--use_rms_norm", "--glu_activation", "swiglu", "--no_tie_embed_logits"]
    if tp > 1:
        argv.append("--sequence_parallel")
    if family == "mistral":
        argv += ["--sliding_window_size", "4096"]
    if getattr(a, "recompute", False):
        argv += ["--recompute_granularity", "full", "--recompute_method", "uniform", "--recompute_num_layers", "1"]
    if getattr(a, "dist_opt", False):
        argv.append("--use_distributed_optimizer")
    graph = getattr(a, "graph", -1)
    # one TP group over the whole job.  (N = 1 measured both ways in round 2: 22.9k tok/s eager, 22.5k with the graph --
    # the host keeps up with full-size kernels -- so it stays eager there; `--graph 1` forces it.)
    use_graph = graph == 1 or (graph == -1 and tp > 1 and tp == n_gpus and pp == 1
                                 and not getattr(a, "recompute", False)
                                 and os.environ.get("MLB200_BENCH_GRAPH", "1") == "1")
    if use_graph:
        argv += ["--cuda_graph_microbatch"]
    return argv, vocab


DUMP_SAMPLES_PER_TENSOR = 4096


def dump_outputs(out_dir, loss, grad_norm, model):
    """Writes the results of one training step as ``out_dir/<name>.npy``:

    * ``lm_loss.npy`` (float32 [1]): the step's loss, averaged over its micro-batches (absent on ranks that do not
      compute the loss, i.e. all but the last pipeline stage);
    * ``grad_norm.npy`` (float32 [1]): the gradient norm before clipping;
    * ``params_sample.npy`` (float32 [n_tensors, 4096]): every parameter tensor this rank holds after the optimizer
      update, in ``named_parameters`` order, read at 4096 positions drawn with replacement from a fixed seed: 16 KB per
      tensor, far below 64 MB in all for every model here.

    The positions depend only on the tensor sizes, so two builds run with the same arguments read the same elements."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    if loss and "lm loss" in loss:
        np.save(os.path.join(out_dir, "lm_loss.npy"), loss["lm loss"].detach().float().reshape(1).cpu().numpy())
    np.save(os.path.join(out_dir, "grad_norm.npy"), np.asarray([float(grad_norm)], dtype=np.float32))
    g = torch.Generator().manual_seed(0)
    rows = []
    for m in model:
        for _, p in m.named_parameters():
            idx = torch.randint(0, p.numel(), (DUMP_SAMPLES_PER_TENSOR,), generator=g).to(p.device)
            rows.append(p.detach().reshape(-1)[idx].float().cpu())
    np.save(os.path.join(out_dir, "params_sample.npy"), torch.stack(rows).numpy())


def _fused_tp_active():
    from megatron_llm_b200.parallel import fused_tp
    c = fused_tp.communicator()
    return c is not None and c.enabled


def run_ours(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29577")
    os.environ.setdefault("RANK", "0")
    os.environ.setdefault("WORLD_SIZE", "1")
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {a.gpus}"

    import finetune
    from megatron_llm_b200 import get_args, ops
    from megatron_llm_b200.initialize import initialize_megatron
    from megatron_llm_b200.models import ModelType
    from megatron_llm_b200.training import setup_model_and_optimizer, train_step

    argv, vocab = megatron_argv(a, a.gpus)
    argv += ["--tokenizer_type", "NullTokenizer", "--vocab_file", str(vocab), "--data_type", "synthetic"]
    # a timed-out peer-memory handshake is fatal in training (symm.check_timeouts); here the flags are examined after
    # the warm-up (fall back to the NCCL path and say so) and after the timed region (reported in `details`)
    os.environ.setdefault("MLB200_TIMEOUT_FATAL", "0")
    devnull = open(os.devnull, "w")
    real_stdout = sys.stdout
    sys.stdout = devnull if rank == 0 else sys.stdout      # keep the JSON line the only rank-0 output
    try:
        initialize_megatron(finetune.extra_args, {}, args_list=argv)
        args = get_args()
        model, optimizer, scheduler = setup_model_and_optimizer(finetune.model_provider, ModelType.encoder_or_decoder)
        for m in model:
            m.train()
    finally:
        pass
    dev = torch.device("cuda", torch.cuda.current_device())
    from megatron_llm_b200.parallel import state as ps
    dp_world, dp_rank = ps.get_data_parallel_world_size(), ps.get_data_parallel_rank()
    n_mb = a.global_batch // (a.micro_batch * dp_world)     # micro-batches per step on this data-parallel rank
    g = torch.Generator().manual_seed(1234 + dp_rank)
    # distinct synthetic micro-batches for every step of the run (uniform random tokens: nothing to memorise, the loss
    # stays near ln(vocab)), pinned on the host; both feeds walk the same pool with one shared cursor
    n_pool = min(4096, n_mb * (a.warmup + 2 * a.steps + 3))
    pool = [torch.randint(0, vocab, (a.micro_batch, a.seq + 1), generator=g, dtype=torch.int64).pin_memory()
            for _ in range(n_pool)]
    pool_dev = [t.to(dev) for t in pool]
    cursor = [0]

    def host_iter():
        while True:
            i = cursor[0]
            cursor[0] += 1
            yield {"text": pool[i % n_pool]}

    def dev_iter():
        while True:
            i = cursor[0]
            cursor[0] += 1
            yield {"text": pool_dev[i % n_pool]}

    feeds = ps.get_tensor_model_parallel_rank() == 0
    it_dev = dev_iter() if feeds else None
    it_host = host_iter() if feeds else None

    last_step = {}

    def step(it):
        loss, skipped, gnorm, _ = train_step(finetune.forward_step, it, model, optimizer, scheduler)
        last_step["loss"], last_step["grad_norm"] = loss, gnorm
        return loss

    def timed(it, k, read_loss):
        dist.barrier()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = ops.launches()
        s.record()
        last = None
        t_host = time.perf_counter()
        for _ in range(k):
            loss = step(it)
            if read_loss and loss:
                last = loss["lm loss"].item()          # D2H read of the step's result, every step
        e.record()
        host_ms = (time.perf_counter() - t_host) * 1e3   # time the host needed to enqueue the work (no sync inside)
        torch.cuda.synchronize()
        dist.barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        timed.host_enqueue_ms = host_ms / k
        return ms.item(), ops.launches() - n0, last

    for _ in range(a.warmup):
        step(it_dev)
    # safety net: a timed-out handshake inside the fused GEMM+collective kernels (PAD_ERROR) means those results
    # cannot be trusted -> redo the warm-up on the NCCL path and say so in `config.tp_comm`
    fused_fallback = False
    from megatron_llm_b200.parallel import fused_tp, schedules
    if fused_tp.communicator() is not None:
        torch.cuda.synchronize()
        err = torch.tensor([fused_tp.communicator().error_flag()], device=dev, dtype=torch.int32)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        if err.item() != 0:
            fused_tp.communicator().enabled = False
            schedules._GRAPH_RUNNERS.clear()
            fused_fallback = True
            for _ in range(a.warmup):
                step(it_dev)
    sampler = ClockSampler(index=int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        sampler.start()
    tp_comm = fused_tp.communicator() if _fused_tp_active() else None
    exposed0 = tp_comm.exposed_ms() if tp_comm is not None else None
    # exposed DP-reduction / PP-p2p time (CUDA events on the compute stream; BASELINE configs 3 and 4)
    from megatron_llm_b200.parallel import p2p
    tp_, pp_, dp_ = parallel_layout(a, a.gpus)
    if pp_ > 1:
        p2p.enable_accounting(True)
    if dp_ > 1:
        for m in model:
            m.account_exposed = True
            m.exposed_reduce_ms()
    ms_dev, launches, _ = timed(it_dev, a.steps, read_loss=False)
    exposed_dp = exposed_pp = None
    if dp_ > 1:
        t = torch.tensor([sum(m.exposed_reduce_ms() for m in model) / a.steps], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        exposed_dp = round(t.item(), 3)
        for m in model:
            m.account_exposed = False
    if pp_ > 1:
        t = torch.tensor([p2p.exposed_recv_ms() / a.steps], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        exposed_pp = round(t.item(), 3)
        p2p.enable_accounting(False)
    exposed = None
    if tp_comm is not None:
        # device-side %globaltimer accounting of the fused kernels: time their GEMM tiles could not hide
        e1 = tp_comm.exposed_ms()
        ex = torch.tensor([(e1[0] - exposed0[0]) / a.steps, (e1[1] - exposed0[1]) / a.steps], device=dev)
        dist.all_reduce(ex, op=dist.ReduceOp.MAX)
        exposed = {"all_gather_wait": round(ex[0].item(), 3), "reduce_scatter_tail": round(ex[1].item(), 3),
                   "total": round(ex.sum().item(), 3)}
    host_enqueue_ms = timed.host_enqueue_ms
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        # before the e2e phase, which trains on: these are the results of the last step timed in `value`
        dump_outputs(a.dump_outputs, last_step["loss"], last_step["grad_norm"], model)
    e2e = None
    if not a.no_e2e:
        step(it_host)  # one untimed step on the host-fed path
        ms_e2e, _, last_loss = timed(it_host, a.steps, read_loss=True)
        tokens = a.steps * a.global_batch * a.seq
        e2e = {"value": tokens / (ms_e2e / 1e3), "unit": "tokens/s",
               "h2d_bytes_per_step": a.global_batch * (a.seq + 1) * 8, "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e2e / a.steps, "last_loss": last_loss}
    timed_out = False
    if fused_tp.communicator() is not None and not fused_fallback:
        err = torch.tensor([fused_tp.communicator().error_flag()], device=dev, dtype=torch.int32)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        timed_out = bool(err.item())
    peak = torch.tensor([torch.cuda.max_memory_allocated() / 2 ** 30], device=dev)
    dist.all_reduce(peak, op=dist.ReduceOp.MAX)
    peak_gb = peak.item()
    sys.stdout = real_stdout
    if rank == 0:
        tokens = a.steps * a.global_batch * a.seq
        tp = parallel_layout(a, a.gpus)[0]
        out = {"metric": METRIC.format(model=a.model, par=parallelism_string(a, a.gpus), seq=a.seq),
               "value": tokens / (ms_dev / 1e3), "unit": "tokens/s", "n_gpus": a.gpus, "steps": a.steps,
               "warmup": a.warmup, "ms_per_step": ms_dev / a.steps, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "bf16", "data": "synthetic tokens (fresh uniform-random micro-batches every step), random-init weights",
               "impl": "ours",
               "config": bench_config(a, a.gpus),
               "details": {"cuda_graph_microbatch": bool(getattr(args, "cuda_graph_microbatch", False)),
                           "tp_comm": ("n/a" if tp == 1 else "fused GEMM+collective kernels over peer memory"
                                       if _fused_tp_active() else
                                       "nccl (fused kernels disabled after a handshake timeout)" if fused_fallback
                                       else "nccl"),
                           "peak_mem_gb": round(peak_gb, 2),
                           "handshake_timeout_in_timed_region": timed_out},
               "exposed_tp_collective_ms_per_step": exposed,
               "exposed_dp_reduce_ms_per_step": exposed_dp, "exposed_pp_p2p_ms_per_step": exposed_pp,
               "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
               "host_enqueue_ms_per_step": host_enqueue_ms}
        print(json.dumps(out), flush=True)
    torch.cuda.synchronize()
    dist.barrier()
    # orderly shutdown: the captured micro-batch graphs hold the NCCL communicators' kernels and the symmetric buffers,
    # so they go first; then the model / optimizer, then the process group.  A watchdog ends the process if the
    # teardown still blocks (seen with NCCL 2.28 when a graph outlives its communicator) -- the result is already out.
    import gc
    sys.stdout.flush()
    sys.stderr.flush()
    watchdog = threading.Timer(30.0, lambda: (sys.stderr.write("bench: teardown timed out, leaving\n"), os._exit(0)))
    watchdog.daemon = True
    watchdog.start()
    schedules._GRAPH_RUNNERS.clear()
    del model, optimizer, scheduler
    gc.collect()
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()
    watchdog.cancel()


def run_reference(a):
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "megatron")):
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref/megatron is missing (reference not installed)"}))
        return
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import reference_runner
        reference_runner.main(a, MODELS, ClockSampler, sys.modules[__name__])
    except SystemExit:
        raise
    except Exception as e:
        import traceback
        traceback.print_exc(file=sys.stderr)
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"reference failed to run: {type(e).__name__}: {e}"[:300]}))


if __name__ == "__main__":
    a = parse()
    a.micro_batch = resolve_micro_batch(a, a.gpus)
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
