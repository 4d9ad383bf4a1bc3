#!/usr/bin/env python
"""Headline benchmark: Llama-2-13B training throughput (tokens/s, whole job) on N B200s of one node.

Metric / config come from BASELINE.json: Llama-2 13B, fleet hybrid parallel (dp x mp x pp as N allows), bf16,
synthetic tokens, random-init weights.  Parallel layout per N: 1 -> single GPU; 2 -> mp2; 4 -> dp2 x mp2;
8 -> dp2 x mp2 x pp2.  Weak scaling: 4 sequences of 4096 tokens per GPU per step.

  python bench.py --gpus 1 --steps 5 --warmup 3
  python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR   -> also writes the last step's loss and sampled parameters as .npy
                                                                       files; inputs are seeded, so two builds compare file by file
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus 8 ...
  python bench.py --impl reference ...   -> {"impl": "reference", "unavailable": ...}
  python bench.py --impl library ...     -> same model and engine with the spec's hot ops on LIBRARY kernels (cuBLAS GEMMs, cuDNN / flash
                                            SDPA attention, NCCL collectives and p2p): the "NCCL + cuBLAS baseline" the fused paths are
                                            compared against on the same box.  It is NOT the reference framework.

Besides tokens/s the JSON line carries `exposed_comm`: device-measured milliseconds per step in which the compute stream waited on
communication (pipeline mailbox waits counted by the wait kernels, NCCL collectives / gradient all-reduce bracketed by CUDA events on
the compute stream) and, for the fused all-gather->GEMM / GEMM->reduce-scatter kernels, a calibrated estimate (fused kernel time minus
the same GEMM without the collective, times the calls per step).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--model", default="llama2-13b")
    ap.add_argument("--seq", type=int, default=4096)
    ap.add_argument("--seqs-per-gpu", type=int, default=4)
    ap.add_argument("--micro-batch", type=int, default=0, help="sequences per micro-batch (0 = per-layout default)")
    ap.add_argument("--layers", type=int, default=0, help="debug only: override layer count (result is then marked invalid)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--layout", default="", help="dp,mp,pp override of the per-N layout (experiments)")
    ap.add_argument("--pp-schedule", default="ZBH1", help="pipeline schedule when pp > 1: ZBH1 (zero bubble, default) | 1F1B | FThenB | VPP")
    ap.add_argument("--vpp", type=int, default=1, help="virtual pipeline chunks per rank (with --pp-schedule VPP)")
    ap.add_argument("--no-comm-calibration", action="store_true")
    ap.add_argument("--recompute-skip", type=int, default=-1,
                    help="N=1 only: number of trailing decoder layers that keep their activations (default: as many as fit in HBM)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the last step's loss and a fixed sample of the updated parameters as DIR/<name>.npy")
    args = ap.parse_args()
    # auto-tuner trials (paddle_b200.distributed.launch --auto_tuner_json / distributed.auto_tuner.AutoTuner.tune): the candidate arrives in the
    # environment and overrides the layout flags; sharding candidates are not a bench.py layout and leave the flags untouched
    tune = os.environ.get("B200_TUNE_CFG")
    if tune:
        c = json.loads(tune)
        if c.get("sharding", 1) == 1:
            args.layout = f"{c['dp']},{c['mp']},{c['pp']}"
            args.micro_batch = int(c.get("micro_batch", args.micro_batch))
            args.pp_schedule = c.get("pp_schedule", args.pp_schedule) if c.get("pp", 1) > 1 else args.pp_schedule
            args.vpp = int(c.get("vpp", args.vpp))
            if c.get("recompute") == "none":
                args.recompute_skip = -1
    return args


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
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
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


DEFAULT_RECOMPUTE_SKIP = 40   # measured: with the memory-lean fused blocks all 40 layers keep their activations in 164 GB (of 179 GB)


def layout_for(n):
    # (dp, mp, pp): sub-meshes of the 8-GPU dp2 x mp2 x pp2 layout BASELINE.json names; at 4 GPUs dp2 x mp2 measured 14 % faster
    # than mp2 x pp2 (no pipeline bubble, larger micro-batches)
    return {1: (1, 1, 1), 2: (1, 2, 1), 4: (2, 2, 1), 8: (2, 2, 2)}.get(n, (n, 1, 1))


DUMP_BUDGET_BYTES = 48 << 20   # all parameter samples together; stays under 64 MB whatever the model size


def dump_outputs(out_dir, loss, model):
    """Write what a caller of the training step holds after the last timed step, so that two builds can be compared output for
    output: `loss.npy` (float64) and, per parameter, `<parameter name>.npy` (float32) with the whole parameter when it is small,
    otherwise the values at positions drawn by a generator seeded with the parameter's index (the same positions in every run)."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    loss = loss.detach().float().item() if isinstance(loss, torch.Tensor) else float(loss)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([loss], dtype=np.float64))
    params = list(model.named_parameters())
    per_param = max(1, DUMP_BUDGET_BYTES // 4 // max(1, len(params)))
    for i, (name, p) in enumerate(params):
        flat = p.detach().as_subclass(torch.Tensor).reshape(-1)
        if flat.numel() > per_param:
            idx = torch.randint(0, flat.numel(), (per_param,), generator=torch.Generator().manual_seed(i)).sort().values
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), flat.float().cpu().numpy())


def exposed_comm_report(regions, args, cfg, mp, pp, dp, accumulate, n, local_rank, ms_per_step):
    """Max over ranks of the per-step exposed communication (see the module docstring); adds the calibrated in-kernel part of the fused
    tensor-parallel GEMMs when they are in use."""
    import torch
    import torch.distributed as dist

    keys = ["pp_mailbox_wait", "pp_recv_wait", "grad_all_reduce", "mp_all_gather", "mp_reduce_scatter", "mp_all_reduce"]
    vec = torch.tensor([float(regions.get(k, 0.0)) for k in keys], device="cuda", dtype=torch.float64)
    fused = None
    if mp > 1 and args.impl == "ours" and not args.no_comm_calibration:
        try:
            fused = calibrate_fused_mp(args, cfg, mp, pp, accumulate)
        except Exception as e:  # noqa: BLE001
            fused = {"error": str(e)[:200]}
    extra = torch.tensor([float((fused or {}).get("ms_per_step", 0.0))], device="cuda", dtype=torch.float64)
    dist.all_reduce(vec, op=dist.ReduceOp.MAX)
    dist.all_reduce(extra, op=dist.ReduceOp.MAX)
    rep = {k: round(float(v), 3) for k, v in zip(keys, vec.tolist()) if v > 0}
    out = {"unit": "ms/step, max over ranks, device-timed", "regions": rep}
    if fused is not None:
        fused["ms_per_step"] = round(float(extra.item()), 3)
        out["fused_mp_gemm_collective"] = fused
    total = sum(rep.values()) + float(extra.item())
    out["total_ms_per_step"] = round(total, 3)
    out["fraction_of_step"] = round(total / ms_per_step, 4)
    if "pp_mailbox_wait" in rep or "pp_recv_wait" in rep:
        out["note"] = "pipeline waits include the schedule's bubble (idle stages), not only transfer time"
    return out


def calibrate_fused_mp(args, cfg, mp, pp, accumulate):
    """Exposed part of the in-kernel collectives: time each fused tensor-parallel GEMM (all-gather->GEMM, GEMM->reduce-scatter) against
    the same GEMM on already-gathered / not-scattered operands, on the model's shapes, and scale by the calls per step."""
    import torch

    from paddle_b200.distributed import fleet
    from paddle_b200.kernels import gemm as KG
    from paddle_b200.parallel import symm

    hcg = fleet.get_hybrid_communicate_group()
    grp = hcg.get_model_parallel_group()
    sc = symm.context_for(grp)
    if sc is None:
        return {"ms_per_step": 0.0, "note": "fused kernels not in use"}
    h, f = cfg.hidden_size, cfg.intermediate_size
    rows = args.micro_batch * args.seq            # tokens per micro-batch (full sequence inside the tensor-parallel region)
    dev = torch.device("cuda")
    dt = torch.bfloat16
    layers_local = cfg.num_hidden_layers // pp
    shapes = {"qkv": (h, 3 * h // mp), "gate_up": (h, 2 * f // mp), "o": (h // mp, h), "down": (f // mp, h)}
    res, total = {}, 0.0

    def t(fn, it=6):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.distributed.barrier()
        a.record()
        for _ in range(it):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / it

    for name in ("qkv", "gate_up"):          # forward: all-gather -> GEMM ; backward dX: GEMM -> reduce-scatter
        k, nn_ = shapes[name]
        w = torch.randn(k, nn_, device=dev, dtype=dt) * 0.02
        xs = torch.randn(rows // mp, 1, k, device=dev, dtype=dt)
        xf = torch.randn(rows, k, device=dev, dtype=dt)
        dy = torch.randn(rows, 1, nn_, device=dev, dtype=dt)
        ag = t(lambda: sc.allgather_gemm(xs, w)) - t(lambda: KG.gemm(xf, w))
        rs = t(lambda: sc.gemm_reduce_scatter(dy, w, b_is_nk=True)) - t(lambda: KG.gemm(dy.view(rows, nn_), w, b_is_nk=True))
        res[name] = {"ag_gemm_minus_gemm_ms": round(ag, 4), "gemm_rs_minus_gemm_ms": round(rs, 4)}
        total += max(ag, 0.0) + max(rs, 0.0)
    for name in ("o", "down"):               # forward: GEMM -> reduce-scatter ; backward dX: all-gather -> GEMM
        k, nn_ = shapes[name]
        w = torch.randn(k, nn_, device=dev, dtype=dt) * 0.02
        x = torch.randn(rows, 1, k, device=dev, dtype=dt)
        dys = torch.randn(rows // mp, 1, nn_, device=dev, dtype=dt)
        dyf = torch.randn(rows, nn_, device=dev, dtype=dt)
        rs = t(lambda: sc.gemm_reduce_scatter(x, w)) - t(lambda: KG.gemm(x.view(rows, k), w))
        ag = t(lambda: sc.allgather_gemm(dys, w, b_is_nk=True)) - t(lambda: KG.gemm(dyf, w, b_is_nk=True))
        res[name] = {"gemm_rs_minus_gemm_ms": round(rs, 4), "ag_gemm_minus_gemm_ms": round(ag, 4)}
        total += max(ag, 0.0) + max(rs, 0.0)
    calls = layers_local * accumulate
    return {"ms_per_step": total * calls, "per_layer_per_microbatch_ms": round(total, 4), "calls_per_step": calls, "detail": res}


def main():
    args = parse()
    if args.impl == "reference":
        print(json.dumps({"impl": "reference", "unavailable": "PaddlePaddle cannot be built offline: third_party/ submodules are empty "
                                                              "and build dependency 'opteinsum' is not in /opt/wheelhouse (see DESIGN.md)"}))
        return 0

    if args.impl not in ("ours", "library"):
        print(json.dumps({"impl": args.impl, "unavailable": "unknown --impl (ours | library | reference)"}))
        return 0
    if args.impl == "library":   # must be set before paddle_b200 reads the flags
        os.environ.update({"FLAGS_b200_gemm_backend": "cublas", "FLAGS_b200_flash_attention": "0", "FLAGS_b200_p2p_collectives": "0",
                           "FLAGS_b200_pp_mailbox": "0", "FLAGS_b200_fused_wgrad": "0", "B200_DISABLE_SYMM": "1"})
    os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")   # 164 of 179 GB live at N=1: avoid fragmentation
    import torch

    import paddle_b200 as paddle
    from paddle_b200 import kernels
    from paddle_b200.distributed import env, fleet
    from paddle_b200.models import llama as L

    n = args.gpus
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if n > 1 and world != n:
        print(json.dumps({"error": f"--gpus {n} needs torchrun with {n} ranks (WORLD_SIZE={world})"}))
        return 1
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    paddle.set_device(f"gpu:{local_rank}")
    dp, mp, pp = layout_for(n)
    if args.layout:
        dp, mp, pp = (int(v) for v in args.layout.split(","))
        assert dp * mp * pp == n, "layout must multiply to --gpus"
    if n > 1:
        strategy = fleet.DistributedStrategy()
        strategy.hybrid_configs = {"dp_degree": dp, "mp_degree": mp, "pp_degree": pp}
        fleet.init(is_collective=True, strategy=strategy)
    rank = env.get_rank()

    cfg = L.llama2_13b() if args.model == "llama2-13b" else L.llama2_7b()
    if args.layers:
        cfg.num_hidden_layers = args.layers
    cfg.max_position_embeddings = args.seq
    cfg.tensor_parallel_degree = mp
    cfg.sequence_parallel = mp > 1
    # single GPU: 13B params + AdamW state fill HBM -> full activation recompute; model-parallel runs keep activations
    cfg.recompute = (n == 1)
    if n == 1:   # 156 GB of weights + optimizer state leave room for the activations of a few layers (~0.7 GB each)
        cfg.recompute_skip_layers = args.recompute_skip if args.recompute_skip >= 0 else DEFAULT_RECOMPUTE_SKIP
    paddle.seed(1234 + rank)
    paddle.set_default_dtype("bfloat16")

    if args.micro_batch <= 0:
        # measured on B200: without a pipeline, larger micro-batches give fuller GEMM waves (mp2: 4 sequences fit the activations of all
        # layers); with pp > 1 the bubble (pp-1)/(accumulate+pp-1) dominates, so keep as many micro-batches as possible.
        # single GPU: split master weights (bf16 + int16 residual) free 26 GB, enough to keep the activations of 2 sequences per micro-batch
        # with no recompute: M = 8192 rows turn the 4.3-wave N=5120 GEMMs (320 tiles on 74 CTA pairs) into 8.6 waves
        args.micro_batch = 4 if (pp == 1 and mp > 1) else 2
    seqs_per_replica = args.seqs_per_gpu * mp * pp
    global_batch = seqs_per_replica * dp
    accumulate = seqs_per_replica // args.micro_batch

    if pp > 1:
        from paddle_b200.distributed.fleet.pipeline import PipelineLayer

        vpp = args.vpp if args.pp_schedule.upper() in ("VPP", "FTHENB") and args.vpp > 1 else 1
        strategy.pipeline_configs = {"accumulate_steps": accumulate, "micro_batch_size": args.micro_batch, "schedule_mode": args.pp_schedule}
        model = PipelineLayer(layers=L.pipeline_layer_descs(cfg), num_stages=pp, loss_fn=L.LlamaPretrainingCriterion(cfg),
                              seg_method="layer:LlamaDecoderLayer", num_virtual_pipeline_stages=vpp if vpp > 1 else None)
    else:
        model = L.LlamaForCausalLM(cfg)
    n_params_local = sum(p.numel() for p in model.parameters())
    assert all(p.dtype == torch.bfloat16 for p in model.parameters()), "model parameters must be bf16"
    decay_fn = lambda name: not any(k in name for k in ("norm", "bias"))  # noqa: E731
    opt = paddle.optimizer.AdamW(learning_rate=1e-5, beta1=0.9, beta2=0.95, epsilon=1e-8, parameters=model.parameters(), weight_decay=0.1,
                                 grad_clip=paddle.nn.ClipGradByGlobalNorm(1.0), multi_precision=True, moment_dtype="bfloat16",
                                 apply_decay_param_fun=decay_fn)
    if n > 1:
        model = fleet.distributed_model(model)
        opt = fleet.distributed_optimizer(opt)
    else:
        opt.enable_flat_arena()

    vocab, seq = cfg.vocab_size, args.seq
    steps_total = args.warmup + args.steps
    # synthetic token stream in pinned host memory (one fresh batch per step: e2e copies it H2D every step)
    # every rank of one model replica (its mp and pp group) must see the same tokens: the stream is seeded by the dp index only
    dp_rank = fleet.get_hybrid_communicate_group().get_data_parallel_rank() if n > 1 else 0
    gen = torch.Generator().manual_seed(4321 + dp_rank)
    host = torch.randint(0, vocab, (steps_total * 2 + 2, seqs_per_replica, seq + 1), dtype=torch.int64, generator=gen).pin_memory()
    h2d_bytes = seqs_per_replica * (seq + 1) * 8
    dev_batches = [host[i].cuda(non_blocking=True) for i in range(2)]

    def train_step(tokens, read_loss):
        """One optimizer step over `accumulate` micro-batches; public-API calls only."""
        nonlocal accumulate
        if pp > 1:
            loss = model.train_batch([tokens[:, :-1], tokens[:, 1:]], opt)
        else:
            loss_acc = None
            for mb in range(accumulate):
                sl = slice(mb * args.micro_batch, (mb + 1) * args.micro_batch)
                loss = model(tokens[sl, :-1], tokens[sl, 1:]) / accumulate
                loss.backward()
                loss_acc = loss.detach() if loss_acc is None else loss_acc + loss.detach()
            opt.step()
            opt.clear_grad()
            loss = loss_acc
        return float(loss.item()) if read_loss else loss

    def barrier():
        if n > 1:
            paddle.distributed.barrier()
        torch.cuda.synchronize()

    from paddle_b200.distributed import comm_timer

    def pp_wait(reset=True):
        fn = getattr(model, "exposed_wait", None)
        return fn(reset) if (pp > 1 and fn is not None) else None

    def timed(nsteps, e2e, offset, measure_comm=False):
        barrier()
        if measure_comm:
            comm_timer.enable(True)
            pp_wait(True)
        sampler = ClockSampler(local_rank)
        sampler.start()
        kernels.reset_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record()
        last = None
        for i in range(nsteps):
            if e2e:
                tok = host[offset + i].cuda(non_blocking=True)       # H2D of this step's inputs from pinned memory
                last = train_step(tok.as_subclass(paddle.Tensor), read_loss=True)  # D2H read of the loss
            else:
                last = train_step(dev_batches[i % 2].as_subclass(paddle.Tensor), read_loss=False)
        ev1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = ev0.elapsed_time(ev1)
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)   # explicit: the default dtype is bf16 here
        if n > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        clocks = sampler.stop()
        if measure_comm:
            regions = comm_timer.summary()
            comm_timer.enable(False)
            w = pp_wait(True)
            ex = {k: round(v["ms"] / nsteps, 3) for k, v in regions.items()}
            if w is not None:
                ex["pp_mailbox_wait"] = round(w["wait_ms"] / nsteps, 3)
            timed.exposed = ex
        return float(t.item()), wall, kernels.launch_count(), clocks, last

    # warm-up (also materialises optimizer state and tensor maps).  Single GPU: if keeping every layer's activations does not
    # fit (allocator fragmentation on a different box), fall back to recomputing more layers instead of failing the run.
    def set_recompute_skip(k):
        layers = list(model.llama.layers)
        for j, l in enumerate(layers):
            l._skip_recompute = j >= len(layers) - k
        cfg.recompute_skip_layers = k

    w_done = 0
    while w_done < args.warmup:
        try:
            train_step(dev_batches[w_done % 2].as_subclass(paddle.Tensor), read_loss=False)
            w_done += 1
        except torch.OutOfMemoryError:
            if n != 1 or (int(getattr(cfg, "recompute_skip_layers", 0)) <= 0 and args.micro_batch <= 1):
                raise
            opt.clear_grad()
            torch.cuda.empty_cache()
            if args.micro_batch > 1:          # first give up micro-batch size, then start recomputing layers
                args.micro_batch //= 2
                accumulate = seqs_per_replica // args.micro_batch
            else:
                set_recompute_skip(max(0, int(cfg.recompute_skip_layers) - 8))
            w_done = 0
    ms, wall, launches, clocks, last = timed(args.steps, e2e=False, offset=0, measure_comm=n > 1)
    tokens_per_step = global_batch * seq
    value = tokens_per_step * args.steps / (ms / 1e3)
    out = {
        "metric": "tokens/sec (whole job, device-timed, max over ranks) Llama-2-13B fleet hybrid parallel training step",
        "value": round(value, 1), "unit": "tokens/s", "n_gpus": n, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms / args.steps, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic tokens (pinned host), random-init weights",
        "config": {"model": "Llama-2-13B" if args.model == "llama2-13b" and not args.layers else f"{args.model} layers={cfg.num_hidden_layers}",
                   "hidden": cfg.hidden_size, "layers": cfg.num_hidden_layers, "heads": cfg.num_attention_heads, "ffn": cfg.intermediate_size,
                   "vocab": vocab, "global_batch": global_batch, "seq_len": seq, "micro_batch": args.micro_batch, "accumulate_steps": accumulate,
                   "parallelism": f"dp{dp}xmp{mp}xpp{pp}", "sequence_parallel": bool(cfg.sequence_parallel), "recompute": (f"full on {cfg.num_hidden_layers - min(cfg.num_hidden_layers, int(getattr(cfg, 'recompute_skip_layers', 0)))} of {cfg.num_hidden_layers} layers"
                                 if cfg.recompute else "none"),
                   "optimizer": "AdamW fp32 master weights, bf16 moments, global-norm clip 1.0 (fused, device-side)",
                   "l2": "working set (weights+optimizer state >= 26 GB per GPU) >> 126 MB L2; no explicit flush needed",
                   "params_per_gpu": n_params_local, "recompute_skip_layers": int(getattr(cfg, "recompute_skip_layers", 0))},
        "gpu_launches": int(launches), "clocks": clocks, "wall_s": round(wall, 3),
    }
    if args.impl == "library":
        out["impl"] = "library"
        out["config"]["library_arm"] = "same model/engine; GEMM = cuBLAS (torch.matmul), attention = PyTorch SDPA (cuDNN / flash), mp/dp collectives and pipeline p2p = NCCL; no fused GEMM+collective kernels, no peer-memory mailbox"
    if pp > 1:
        out["config"]["pp_schedule"] = str(getattr(model, "schedule_mode", args.pp_schedule))
        out["config"]["pp_transport"] = model.transport_name() if hasattr(model, "transport_name") else None
    if n > 1:
        out["exposed_comm"] = exposed_comm_report(getattr(timed, "exposed", {}), args, cfg, mp, pp, dp, accumulate, n, local_rank, ms / args.steps)
    if args.layers:
        out["invalid"] = "debug run with reduced layer count"
    if not args.no_e2e:
        ms2, wall2, _, _, last = timed(args.steps, e2e=True, offset=2)
        out["e2e"] = {"value": round(tokens_per_step * args.steps / (ms2 / 1e3), 1), "unit": "tokens/s", "h2d_bytes_per_step": h2d_bytes,
                      "d2h_bytes_per_step": 4, "ms_per_step": round(ms2 / args.steps, 2), "last_loss": last}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")))
    except Exception:
        pass
    flops_per_token = 6 * 13.0e9 + 6 * cfg.num_hidden_layers * cfg.hidden_size * seq  # fwd+bwd model FLOPs (attention counted causal: half of 12 L h s)
    out["peak_mem_gb"] = round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)
    out["model_tflops_per_gpu"] = round(value * flops_per_token / n / 1e12, 1)
    if peaks.get("bf16_tflops_sustained"):
        out["mfu_of_measured_sustained_peak"] = round(out["model_tflops_per_gpu"] / peaks["bf16_tflops_sustained"], 3)
    if args.dump_outputs and rank == 0:   # with several ranks: rank 0's loss and its share of the parameters
        dump_outputs(args.dump_outputs, last, model)
    if rank == 0:
        print(json.dumps(out))
    if n > 1:
        env.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
