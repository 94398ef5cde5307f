#!/usr/bin/env python
"""Flagship benchmark: bloom-560m training tokens/s (TP2 x DP, weak scaling) on N B200s.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29511 bench.py --gpus 8 --steps 10 --warmup 3
    python bench.py --impl reference ...      # the unmodified reference (baseline/_ref) on the same config
    python bench.py --gpus 2 --hf             # our arm fed with a transformers BloomForCausalLM (the reference's input)
    python bench.py --device cpu --model bloom-tiny --seq-len 64 --batch-per-gpu 2 --gpus 2    # dry run of this script

Metric/config follow BASELINE.json: bloom-560m, seq 1024, bf16, synthetic token ids, random-init
weights, Adam; N=1 -> TP1xDP1, N>=2 -> TP2 x DP(N/2); per-GPU work is fixed (weak scaling):
global batch = batch_per_gpu * N sequences.  One JSON line is printed by rank 0; both arms spell the
`config` dict identically (`config_of`).  `--model/--tp/--pp/--experts/--seq-len/--batch-per-gpu` select the
other BASELINE.json configs for BOTH arms (bloom-7b1 TP8, Switch-MoE EP8, bloom-3b TP2xPP2xDP2).

Two timed regions of K steps each, both bracketed by barrier + synchronize, timed with CUDA events
on the device, max over ranks:
  value : full train step (fwd, bwd, grad sync, optimizer) with device-resident inputs
  e2e   : the same step through the public API including, every step, the pinned-host -> device
          copy of that step's token ids and a device -> host read of the loss.
At N > 1 our arm first runs a numerics self-check (outside the timed regions): 3 steps of a 2-layer model of the
benchmark's width through the fused NVLink engines and through NCCL + plain kernels; `numerics_ok`, the largest
relative loss difference and the parameter-checksum difference travel in the JSON line.

`--dump-outputs DIR` (our arm) writes, after the timed regions, what the last timed step computed on rank 0 as
DIR/<name>.npy (see `dump_outputs`; with --pp > 1 that is the first stage, whose loss is 0).  Weights and token ids are
seeded, so two builds run with the same arguments get the same inputs and can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _env_defaults():
    os.environ.setdefault("RANK", "0")
    os.environ.setdefault("LOCAL_RANK", "0")
    os.environ.setdefault("WORLD_SIZE", "1")
    os.environ.setdefault("LOCAL_WORLD_SIZE", os.environ["WORLD_SIZE"])
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if "MASTER_PORT" not in os.environ:
        os.environ["MASTER_PORT"] = str(_free_port())


def _peak_mem_gb(torch, args):
    """Peak bytes this rank's caching allocator handed out (GiB; the NVLink workspaces, mapped with the VMM API, are not
    the allocator's and not counted).  Informational: how far the config is from the 180 GB of a B200."""
    try:
        if args.device == "cuda" and torch.cuda.is_available():
            return round(torch.cuda.max_memory_allocated() / 2**30, 3)
    except Exception:
        pass
    return None


def dump_outputs(out_dir, torch, model, loss):
    """What the last timed step hands back: ``loss.npy`` (float64 scalar) and ``weights_sample.npy``, the weights after that
    step's optimizer update (float32, tensors concatenated in ``model.parameters()`` order).  A tensor larger than the
    per-tensor share of 16 M values (64 MB, at most 16384 a tensor) contributes a sorted sample of positions drawn from a
    generator seeded with 0, so the same model always yields the same positions.  GPU runs are not bit-reproducible, so
    compare with a tolerance: two runs of one build (bloom-560m, --gpus 1 --steps 10, B200 at a 1000 W power limit)
    differed by 7e-5 in the loss and by at most 2.2e-3 in a sampled weight."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array(loss, dtype=np.float64))
    params = list(model.parameters())
    per_tensor = max(1, min(16384, (16 << 20) // max(len(params), 1)))
    gen = torch.Generator().manual_seed(0)
    parts = []
    with torch.no_grad():
        for p in params:
            flat = p.detach().reshape(-1)
            if flat.numel() > per_tensor:
                idx = torch.randint(0, flat.numel(), (per_tensor,), generator=gen).sort().values
                flat = flat[idx.to(flat.device)]
            parts.append(flat.float().cpu())
    np.save(os.path.join(out_dir, "weights_sample.npy"), torch.cat(parts).numpy())


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 9:
                self.samples.append(parts)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for p in self.samples:
            try:
                sm.append(float(p[1]))
                mx = max(mx, float(p[2]))
            except ValueError:
                continue
            for n, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def parallel_layout(n_gpus: int):
    if n_gpus == 1:
        return 1, 1
    return 2, n_gpus // 2


def layout_of(args):
    """``(tp, pp, dp)`` of a run — the same for both arms.  Default: BASELINE.json's headline layout (N=1: tp1, N>=2:
    tp2 x dp N/2); ``--tp / --pp`` select the other BASELINE configs."""
    tp, dp = parallel_layout(args.gpus)
    pp = max(args.pp, 1)
    if args.tp > 0 or pp > 1:
        tp = args.tp if args.tp > 0 else 1
        assert args.gpus % (tp * pp) == 0, "--gpus must be a multiple of tp * pp"
        dp = args.gpus // (tp * pp)
    return tp, pp, dp


def config_of(args, tp, pp, dp):
    """The benchmark configuration, spelled identically by both arms (the driver compares these dicts)."""
    return {
        "model": args.model, "global_batch": args.batch_per_gpu * args.gpus, "seq_len": args.seq_len,
        "parallelism": f"tp{tp}" + (f"pp{pp}(1f1b,{args.microbatches}mb)" if pp > 1 else "") + f"dp{dp}"
        + ("+zero1" if dp > 1 else "") + (f"+moe{args.experts}e" if args.experts > 0 else ""),
        "optimizer": "Adam", "batch_per_gpu": args.batch_per_gpu,
        "l2": "no explicit flush: per-step working set (weights + activations, several GB) >> 126 MB L2",
    }


class _HostTimer:
    """CPU dry runs (``--device cpu``: both arms on tiny shapes, to test this script without a GPU)."""

    def __init__(self):
        self.t = None

    def record(self):
        import time

        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return (other.t - self.t) * 1e3


def timed_region(torch, dist, steps, fn):
    """barrier + sync, K steps between two CUDA events, sync + barrier; returns max-over-ranks ms."""
    world = dist.get_world_size() if dist.is_initialized() else 1
    if world > 1:
        dist.barrier()
    cuda = torch.cuda.is_available()
    if cuda:
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    else:
        start, end = _HostTimer(), _HostTimer()
    start.record()
    for i in range(steps):
        fn(i)
    end.record()
    if cuda:
        torch.cuda.synchronize()
    ms = torch.tensor([start.elapsed_time(end)], device="cuda" if cuda else "cpu")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.barrier()
    return float(ms.item())


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
MODEL_SIZES = {"bloom-tiny": (128, 4, 8, 1024), "bloom-560m": (1024, 24, 16, 250880), "bloom-1b7": (2048, 24, 16, 250880),
               "bloom-3b": (2560, 30, 32, 250880), "bloom-7b1": (4096, 30, 32, 250880)}   # hidden, layers, heads, vocab


def _init_on_gpu(args) -> bool:
    """Initialise the weights on the GPU instead of on the host?  ``--init-device auto``: for the multi-billion
    parameter configs only (filling 7B weights on the host takes minutes per rank)."""
    if args.device != "cuda":
        return False
    mode = getattr(args, "init_device", "auto")
    return mode == "cuda" or (mode == "auto" and args.model in ("bloom-1b7", "bloom-3b", "bloom-7b1"))


def _make_model_ours(args, ctx, torch, n_layer, vocab, hf, dtype):
    from pipegoose_b200.models.bloom import BloomConfig, BloomForCausalLM

    if args.model.startswith("gpt2"):  # not a BASELINE.json config: the second model family on the same kernels
        from pipegoose_b200.models.gpt2 import GPT2Config, GPT2LMHeadModel

        cfg = getattr(GPT2Config, args.model.replace("-", "_"))()
        model = GPT2LMHeadModel(cfg).to(dtype)
    elif hf:
        # the reference's canonical input: a transformers BloomForCausalLM; TensorParallel converts it in place
        from transformers import BloomConfig as HFConfig
        from transformers import BloomForCausalLM as HFBloom

        h, L, nh, V = MODEL_SIZES[args.model]
        model = HFBloom(HFConfig(hidden_size=h, n_layer=n_layer or L, n_head=nh, vocab_size=vocab or V)).to(dtype)
        cfg = model.config
    else:
        cfg = getattr(BloomConfig, args.model.replace("-", "_"))()
        if n_layer is not None:
            cfg.n_layer = n_layer
        if vocab is not None:
            cfg.vocab_size = vocab
        model = BloomForCausalLM(cfg).to(dtype)
    if args.experts > 0:
        from pipegoose_b200.nn import ExpertParallel
        from pipegoose_b200.nn.expert_parallel import SwitchNoisePolicy, Top1Router

        router = Top1Router(SwitchNoisePolicy(), args.experts, cfg.hidden_size, expert_capacity=(1.25, 2.0))
        layers = list(range(0, cfg.n_layer, max(args.moe_every, 1)))
        model = ExpertParallel(model, args.experts, mapping=layers, router=router.to(dtype),
                               parallel_context=ctx).parallelize()
    return model, cfg


def _build_ours(args, ctx, torch, n_layer=None, vocab=None, hf=False, fused=True):
    """Model -> ExpertParallel -> TensorParallel -> PipelineParallel -> DataParallel -> ZeRO-1(FusedAdam): the public API a
    user of the reference calls, on this repo's kernels.  ``fused=False``: the same stack with the hand-written
    compute+collective kernels switched off (NCCL collectives around plain kernels) — the numerics self-check's yardstick."""
    from pipegoose_b200.models.bloom import BloomConfig, BloomForCausalLM
    from pipegoose_b200.nn import DataParallel, TensorParallel
    from pipegoose_b200.optim import DistributedOptimizer
    from pipegoose_b200.optim.fused_adam import FusedAdam

    switches = {"PIPEGOOSE_B200_FUSED_TP": "1" if fused else "0", "PIPEGOOSE_B200_FUSED_DP": "1" if fused else "0",
                "PIPEGOOSE_B200_FUSED_MOE": "1" if fused else "0"}
    saved = {k: os.environ.get(k) for k in switches}
    if not fused:
        os.environ.update(switches)
    import contextlib

    # weights are initialised ON the GPU (seeded: identical on every rank): a 7B model takes minutes to fill on the host
    init_on = torch.device("cuda", torch.cuda.current_device()) if _init_on_gpu(args) else contextlib.nullcontext()
    try:
        pp = ctx.pipeline_parallel_size
        dtype = torch.bfloat16 if args.device == "cuda" else torch.float32
        with init_on:
            model, cfg = _make_model_ours(args, ctx, torch, n_layer, vocab, hf, dtype)
        model = TensorParallel(model, ctx, sequence_parallel=True if hf else None).parallelize()
        if pp > 1:
            from pipegoose_b200.nn import PipelineParallel

            model = PipelineParallel(model, num_microbatches=args.microbatches, parallel_context=ctx).parallelize()
        model = DataParallel(model, ctx).parallelize()
        model.to(args.device)
        optim = DistributedOptimizer(FusedAdam(model.parameters(), lr=args.lr), ctx)
        return model, optim, cfg
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _total_loss(model, ids, experts):
    loss = model(ids, labels=ids).loss
    if experts > 0:
        # Switch training objective: task loss + load-balancing and router-z terms the MoE layers pushed
        from pipegoose_b200.nn.expert_parallel import ExpertContext

        store = ExpertContext.get_instance()
        loss = loss + 0.01 * sum(store.pop_all_aux_loss()) + 0.001 * sum(store.pop_all_z_loss())
    return loss


def numerics_self_check(args, ctx, torch, dist):
    """Multi-GPU correctness that travels with every N>1 bench line (outside the timed regions): 3 optimizer steps of a
    2-layer model of the benchmark's width through the fused engines (AG->GEMM / GEMM->RS, in-kernel gradient
    reduce-scatter, ZeRO-1 all-gather, fused MoE) and through the same stack with them switched off (NCCL collectives
    around plain kernels), same init, same data.  Reports the largest relative loss difference and the relative
    difference of the parameter checksums after the last step."""
    from pipegoose_b200.distributed import ParallelMode

    S = min(args.seq_len, 1024)
    tp, pp = ctx.tensor_parallel_size, ctx.pipeline_parallel_size
    b_rep = max(args.batch_per_gpu, 1) * tp * pp
    gen = torch.Generator().manual_seed(77 + ctx.get_local_rank(ParallelMode.DATA))
    ids = torch.randint(0, 8192, (b_rep, S), generator=gen).to(args.device)
    out = {}
    for name, fused in (("fused", True), ("library", False)):
        torch.manual_seed(4321)
        model, optim, _ = _build_ours(args, ctx, torch, n_layer=2 * pp, vocab=8192, hf=args.hf, fused=fused)
        losses = []
        for _ in range(3):
            loss = _total_loss(model, ids, args.experts)
            optim.zero_grad()
            loss.backward()
            optim.step()
            losses.append(loss.detach().float())
        seen, chk = set(), torch.zeros((), dtype=torch.float64, device=args.device)
        for p in model.parameters():
            if id(p) not in seen:
                seen.add(id(p))
                chk += p.detach().double().abs().sum()
        losses = torch.stack(losses).double()
        if dist.get_world_size() > 1:
            dist.all_reduce(chk)
            dist.all_reduce(losses)   # (pipelined models report the loss on every rank; sums are compared like for like)
        out[name] = (losses, chk)
        del model, optim
    (lf, cf), (ll, cl) = out["fused"], out["library"]
    loss_err = float(((lf - ll).abs() / ll.abs().clamp(min=1e-9)).max())
    param_err = float((cf - cl).abs() / cl.abs().clamp(min=1e-9))
    # bf16 kernels with different summation orders: losses agree to ~1e-3 relative; a protocol bug (a lost tile, a
    # stale buffer, a double-counted gradient) shows up orders of magnitude above that
    ok = bool(loss_err < 2e-2 and param_err < 1e-3 and torch.isfinite(lf).all())
    return {"numerics_ok": ok, "max_rel_err_loss": loss_err, "rel_err_param_checksum": param_err,
            "losses_fused": [float(x) / dist.get_world_size() for x in lf],
            "losses_library": [float(x) / dist.get_world_size() for x in ll],
            "what": "3 steps, 2-layer model of the benchmark width, fused NVLink engines vs NCCL + plain kernels"}


def run_ours(args):
    import torch
    import torch.distributed as dist

    from pipegoose_b200 import ops
    from pipegoose_b200.distributed import ParallelContext, ParallelMode

    tp, pp, dp = layout_of(args)
    ctx = ParallelContext.from_torch(tensor_parallel_size=tp, pipeline_parallel_size=pp, data_parallel_size=dp,
                                     backend="nccl" if args.device == "cuda" else "gloo")
    rank = ctx.get_global_rank()
    dev = torch.device("cuda", torch.cuda.current_device()) if args.device == "cuda" else torch.device("cpu")
    numerics = None
    if args.gpus > 1 and not args.no_self_check:
        try:
            numerics = numerics_self_check(args, ctx, torch, dist)
        except Exception as e:  # a failing check is reported, it does not hide the benchmark number
            import traceback

            traceback.print_exc()
            numerics = {"numerics_ok": False, "error": f"{type(e).__name__}: {e}"[:300]}
        if args.device == "cuda":
            torch.cuda.empty_cache()
    torch.manual_seed(1234)
    model, optim, cfg = _build_ours(args, ctx, torch, hf=args.hf)

    S = args.seq_len
    b_rep = args.batch_per_gpu * tp * pp  # sequences per model replica (DP rank)
    gen = torch.Generator().manual_seed(1000 + ctx.get_local_rank(ParallelMode.DATA))
    n_host = args.steps + args.warmup + 1
    host_ids = [torch.randint(0, cfg.vocab_size, (b_rep, S), generator=gen) for _ in range(n_host)]
    if args.device == "cuda":
        host_ids = [t.pin_memory() for t in host_ids]
    dev_ids = host_ids[0].to(dev)

    def step_device(i):
        loss = _total_loss(model, dev_ids, args.experts)
        optim.zero_grad()
        loss.backward()
        optim.step()
        return loss

    last = {}

    def step_e2e(i):
        ids = host_ids[i % n_host].to(dev, non_blocking=True)
        loss = _total_loss(model, ids, args.experts)
        optim.zero_grad()
        loss.backward()
        optim.step()
        last["loss"] = loss.item()  # device -> host read of the step's result (0 on non-final pipeline stages)

    for i in range(args.warmup):
        step_e2e(i)
    sampler = ClockSampler(torch.cuda.current_device() if args.device == "cuda" else 0)
    if rank == 0 and args.device == "cuda":
        sampler.start()
    ops.reset_launch_count()
    ms_dev = timed_region(torch, dist, args.steps, step_device)
    launches = ops.launch_count()
    ms_e2e = timed_region(torch, dist, args.steps, step_e2e)
    if rank == 0:
        sampler.stop()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, torch, model, last["loss"])
    tokens_per_step = args.batch_per_gpu * args.gpus * S
    result = {
        "metric": f"{args.model} training tokens/sec (whole job, device-timed, max over ranks)",
        "value": tokens_per_step * args.steps / (ms_dev / 1e3),
        "unit": "tokens/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "bf16" if args.device == "cuda" else "fp32 (cpu dry run)",
        "data": "synthetic token ids (uniform random), random-init weights",
        "impl": "pipegoose_b200",
        "config": config_of(args, tp, pp, dp),
        "impl_notes": {"optimizer": "fused Adam, fp32 master weights + moments, ZeRO-1 slices when dp > 1",
                       "model_class": "transformers.BloomForCausalLM converted in place by TensorParallel" if args.hf
                       else "pipegoose_b200.models"},
        "e2e": {
            "value": tokens_per_step * args.steps / (ms_e2e / 1e3), "unit": "tokens/s",
            "ms_per_step": ms_e2e / args.steps,
            "h2d_bytes_per_step": int(host_ids[0].numel() * host_ids[0].element_size()),
            "d2h_bytes_per_step": 4,
        },
        "gpu_launches": launches,
        "final_loss": last.get("loss"),
        "mfu_vs_measured_sustained": None,
        "clocks": sampler.summary() if rank == 0 else None,
    }
    result["peak_mem_gb"] = _peak_mem_gb(torch, args)
    if numerics is not None:
        result["numerics"] = numerics
        result["numerics_ok"] = numerics.get("numerics_ok")
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        flops = model.flops_per_token(S) * tokens_per_step / args.gpus
        result["mfu_vs_measured_sustained"] = flops / (ms_dev / args.steps / 1e3) / (peaks["bf16_tflops_sustained"] * 1e12)
    except Exception:
        pass
    if rank == 0:
        print(json.dumps(result), flush=True)
    ctx.destroy()


# --------------------------------------------------------------------------------------------
# reference arm: the unmodified reference installed under baseline/_ref, stock code path
# --------------------------------------------------------------------------------------------
def _build_reference(args, n_layer=None, vocab=None):
    """The reference's stock path: transformers Bloom -> [ExpertParallel] -> TensorParallel -> DataParallel ->
    DistributedOptimizer(torch.optim.Adam).  Returns ``None`` (after printing the JSON "unavailable" line) when the
    reference cannot be imported, else ``(ctx, model, optim, fwd, cfg, (tp, pp, dp), note)``."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "pipegoose")):
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref/pipegoose not installed (see DESIGN.md)"}))
        return None
    sys.path.insert(0, os.path.join(ROOT, "baseline", "shims"))
    sys.path.insert(0, ref_dir)
    try:
        import hf_fx_shim

        hf_fx_shim.install()
        import torch
        from pipegoose.distributed.parallel_context import ParallelContext
        from pipegoose.nn import DataParallel, TensorParallel
        from pipegoose.optim import DistributedOptimizer
        from transformers import BloomConfig, BloomForCausalLM
    except Exception as e:  # pragma: no cover
        print(json.dumps({"impl": "reference", "unavailable": f"import failed: {type(e).__name__}: {e}"[:300]}))
        return None

    tp, pp, dp = layout_of(args)
    note = None
    if pp > 1:
        # The reference's pipeline engine cannot run in this image: nn/pipeline_parallel/partitioner.py traces the model
        # with transformers.utils.fx, which transformers 5 removed (BASELINE.md section 3), and its RPC runtime was never
        # finished (SURVEY section 8).  The closest layout its stock code does run is the same model with the pipeline
        # dimension folded into data parallelism: tp x (pp*dp) + ZeRO-1, same global batch.
        note = (f"reference pipeline engine not runnable (transformers.utils.fx removed in transformers 5): ran tp{tp} x "
                f"dp{dp * pp} + ZeRO-1 on the same global batch instead of tp{tp} x pp{pp} x dp{dp}")
        dp, pp = dp * pp, 1
    cuda = args.device == "cuda"
    if cuda:
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    # The reference issues collectives on CPU tensors during bring-up (parallel_context.py:263-287), which a
    # pure "nccl" group rejects; torch's per-device backend string gives it gloo for those and NCCL for CUDA
    # tensors.  This is an argument of the reference's public API, not a change to it.
    ctx = ParallelContext.from_torch(tensor_parallel_size=tp, pipeline_parallel_size=1, data_parallel_size=dp,
                                     backend="cpu:gloo,cuda:nccl" if cuda else "gloo")
    if cuda:
        ctx.set_device()
    dev = torch.device("cuda", torch.cuda.current_device()) if cuda else torch.device("cpu")
    h, L, nh, V = MODEL_SIZES[args.model]
    L, V = n_layer or L, vocab or V
    torch.manual_seed(1234)
    cfg = BloomConfig(hidden_size=h, n_layer=L, n_head=nh, vocab_size=V)
    import contextlib

    with (dev if _init_on_gpu(args) else contextlib.nullcontext()):   # same rule in both arms
        model = BloomForCausalLM(cfg)
    if cuda or os.environ.get("PIPEGOOSE_B200_BENCH_CPU_BF16") == "1":   # the env switch: dtype flow of the dry run = GPU run
        model = model.to(torch.bfloat16)
    loss_terms = None
    if args.experts > 0:
        # the reference's Switch-MoE path: ExpertParallel (experts sharded over the TENSOR group, tokens replicated,
        # all-reduce combine, nn/expert_parallel/experts.py:41-82) + ExpertLoss's auxiliary terms
        from pipegoose.nn.expert_parallel import ExpertParallel, SwitchNoisePolicy, Top1Router
        from pipegoose.nn.expert_parallel.expert_context import ExpertContext

        # (the reference's router computes its gate in fp32 — routers.py:109 `self.gate(inputs.float())` — so the router
        #  keeps its fp32 parameters next to the bf16 model)
        router = Top1Router(SwitchNoisePolicy(), args.experts, h, expert_capacity=(1.25, 2.0))
        layers = list(range(0, L, max(args.moe_every, 1)))
        model = ExpertParallel(model, num_experts=args.experts, mapping=layers, router=router,
                               parallel_context=ctx).parallelize()

        def loss_terms(loss):   # ExpertLoss.__call__ (nn/expert_parallel/loss.py:26-31) with this benchmark's weights
            store = ExpertContext.get_instance()
            return loss + 0.01 * sum(store.pop_all_aux_loss()) + 0.001 * sum(store.pop_all_z_loss())
    model = TensorParallel(model, ctx).parallelize()
    model = DataParallel(model, ctx).parallelize()
    optim = torch.optim.Adam(model.parameters(), lr=args.lr)
    optim = DistributedOptimizer(optim, ctx)
    if cuda:
        model.to("cuda")
    model.train()

    def fwd(ids):
        mask = torch.ones_like(ids)
        loss = model(input_ids=ids, attention_mask=mask, labels=ids).loss
        return loss_terms(loss) if loss_terms is not None else loss

    return ctx, model, optim, fwd, cfg, (tp, pp, dp), note, dev


def run_reference(args):
    built = _build_reference(args)
    if built is None:
        return
    import torch
    import torch.distributed as dist
    from pipegoose.distributed.parallel_mode import ParallelMode

    ctx, model, optim, fwd, cfg, (tp, pp, dp), note, dev = built
    cuda = args.device == "cuda"
    rank = ctx.get_global_rank()

    S = args.seq_len
    b_rep = args.batch_per_gpu * tp
    gen = torch.Generator().manual_seed(1000 + ctx.get_local_rank(ParallelMode.DATA))
    n_host = args.steps + args.warmup + 1
    host_ids = [torch.randint(0, cfg.vocab_size, (b_rep, S), generator=gen) for _ in range(n_host)]
    if cuda:
        host_ids = [t.pin_memory() for t in host_ids]
    dev_ids = host_ids[0].to(dev)

    def step_device(i):
        loss = fwd(dev_ids)
        optim.zero_grad()
        loss.backward()
        optim.step()

    last = {}

    def step_e2e(i):
        ids = host_ids[i % n_host].to(dev, non_blocking=True)
        loss = fwd(ids)
        optim.zero_grad()
        loss.backward()
        optim.step()
        last["loss"] = loss.item()

    for i in range(args.warmup):
        step_e2e(i)
    sampler = ClockSampler(torch.cuda.current_device() if cuda else 0)
    if rank == 0 and cuda:
        sampler.start()
    ms_dev = timed_region(torch, dist, args.steps, step_device)
    ms_e2e = timed_region(torch, dist, args.steps, step_e2e)
    if rank == 0:
        sampler.stop()
    tokens_per_step = args.batch_per_gpu * args.gpus * S
    result = {
        "impl": "reference",
        "metric": f"{args.model} training tokens/sec (whole job, device-timed, max over ranks)",
        "value": tokens_per_step * args.steps / (ms_dev / 1e3), "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if cuda else "fp32 (cpu dry run)",
        "data": "synthetic token ids (uniform random), random-init weights",
        "config": config_of(args, tp, pp, dp),
        "impl_notes": {"optimizer": "torch.optim.Adam via the reference's DistributedOptimizer",
                       "model_class": "transformers.BloomForCausalLM"},
        "e2e": {"value": tokens_per_step * args.steps / (ms_e2e / 1e3), "unit": "tokens/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(host_ids[0].numel() * host_ids[0].element_size()), "d2h_bytes_per_step": 4},
        "gpu_launches": 0,
        "final_loss": last.get("loss"),
        "clocks": sampler.summary() if rank == 0 else None,
    }
    result["peak_mem_gb"] = _peak_mem_gb(torch, args)
    if note is not None:
        result["note"] = note
    if rank == 0:
        print(json.dumps(result), flush=True)
    try:
        dist.barrier()
        dist.destroy_process_group()
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="bloom-560m")
    ap.add_argument("--seq-len", type=int, default=1024)
    ap.add_argument("--batch-per-gpu", type=int, default=8)
    ap.add_argument("--lr", type=float, default=1e-4)
    # non-default layouts (both arms): BASELINE.json configs #3-#5
    ap.add_argument("--tp", type=int, default=0, help="tensor parallel size (0: 1 GPU -> 1, else 2)")
    ap.add_argument("--pp", type=int, default=1, help="pipeline stages (1F1B)")
    ap.add_argument("--microbatches", type=int, default=8)
    ap.add_argument("--experts", type=int, default=0, help="Switch-MoE experts (sharded over the tensor group)")
    ap.add_argument("--moe-every", type=int, default=2, help="every n-th block gets a MoE MLP")
    ap.add_argument("--hf", action="store_true",
                    help="ours arm: feed a transformers BloomForCausalLM (the reference's input) instead of pipegoose_b200.models")
    ap.add_argument("--no-self-check", action="store_true", help="skip the N>1 numerics self-check (fused vs library engines)")
    ap.add_argument("--init-device", default="auto", choices=["auto", "cpu", "cuda"],
                    help="where the random weights are created (auto: on the GPU for the >= 1.7B configs)")
    ap.add_argument("--device", default="cuda", choices=["cuda", "cpu"],
                    help="cpu: dry run of this script on gloo with a tiny model (no benchmark value)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="our arm: write the last timed step's loss and a fixed sample of the updated weights as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is implemented for --impl ours only")
    args.warmup = max(args.warmup, 3)
    _env_defaults()
    world = int(os.environ["WORLD_SIZE"])
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            # convenience: re-launch under torchrun (a port picked as free can be taken before torchrun binds it: retry)
            for attempt in range(3):
                cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                       "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), os.path.abspath(__file__)] + sys.argv[1:]
                res = subprocess.run(cmd, stderr=subprocess.PIPE, text=True)
                sys.stderr.write(res.stderr)
                if res.returncode == 0 or "EADDRINUSE" not in res.stderr:
                    raise SystemExit(res.returncode)
            raise SystemExit(res.returncode)
        raise SystemExit(f"WORLD_SIZE={world} does not match --gpus {args.gpus}")
    if args.impl == "reference":
        try:
            run_reference(args)
        except Exception as e:  # the reference's own code path failed on this layout: report it, do not crash the driver
            import traceback

            traceback.print_exc()
            if int(os.environ.get("RANK", "0")) == 0:
                print(json.dumps({"impl": "reference", "n_gpus": args.gpus,
                                  "unavailable": f"reference failed at run time: {type(e).__name__}: {e}"[:300]}), flush=True)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
