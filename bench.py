#!/usr/bin/env python3
"""Headline benchmark of the B200 HSTU hot path (contract: see the task statement / DESIGN.md section "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload hstu_large|attn]

Workload `hstu_large` (default; BASELINE.json metric "user-seqs/sec HSTU-large L=8192 d=256 bf16"):
  a 16-layer STU stack, D=256, H=8, dqk=dv=32, bf16, over a synthetic jagged batch of `--batch` user sequences per GPU
  with Lmax=8192 (lengths ~ U[0.9 Lmax, Lmax), 1..20 targets: the reference bench recipe, hstu_attention_bench.py:194-248).
  One step = forward + backward of the whole stack + (N>1) NCCL all-reduce of the parameter gradients (one bucket per
  layer, overlapped with the remaining backward) + fused AdamW step.  value = sequences / second over all ranks.
Workload `attn`: the reference microbench (B=512, H=4, d in {64,128}, fwd+bwd of hstu_mha only).

`--impl triton` (workload attn only) times the reference's own Triton kernel (`triton_hstu_mha`, sort_by_length=True,
enable_tma=False, autotuned; fetched into the git-ignored baseline/_ref/ by scripts/fetch_triton_baseline.py) on the same
seeded inputs with the same CUDA-event method: the GPU comparator the north-star names.
`--impl reference` times the CPU port of the reference eager path (oracle/) on the host cores on a bounded sample of
the same workload (the Python reference itself cannot travel to the GPU box).  Rank 0 only.

`--dump-outputs DIR` (GPU workloads) writes, after the timed steps, what the last step returned to its caller as
DIR/<name>.npy in float32 (at most 64 MB in all; row-sampled with a fixed seed where an output is larger), so that two builds
can be compared output for output on identical seeded inputs.  Two runs of the same build do not agree bit for bit: the
attention backward's dQ accumulation order varies (2e-5 relative), and AdamW on bf16 weights amplifies that over the steps.
Measured on one B200 (1000 W power limit), default workload, rel-L2 between two runs: after 3 steps up to 1.1e-2 on y and
5e-3 on the parameter gradients; the loss agrees to 2e-6.

bench.py writes nothing into the source tree: it loads the library that `python -m generative_recommenders_b200.build`
(or __graft_entry__.build()) left there and does not compile.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "triton"])
    ap.add_argument("--workload", default="hstu_large", choices=["hstu_large", "attn", "ml20m", "amzn_books"])
    ap.add_argument("--batch", type=int, default=16, help="user sequences per GPU per step")
    ap.add_argument("--lmax", type=int, default=8192)
    ap.add_argument("--layers", type=int, default=16)
    ap.add_argument("--attn-dim", type=int, default=128, help="head dim of the attn microbench workload")
    ap.add_argument("--attn-heads", type=int, default=4)
    ap.add_argument("--attn-impl", type=int, default=0, help="0 auto, 1 generic kernels, 2 force tcgen05")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch sequences per GPU (default, what the driver's scaling run measures); strong: --batch "
                         "sequences in total, sharded over the ranks balanced by sum(len^2) (distributed.shard_sequences)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last step as DIR/<name>.npy (float32, <= 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    return args


# ----------------------------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------------------------
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def ncu_traffic(cfg):
    """DRAM bytes per launch of the attention backward kernel from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by scripts/ncu_traffic.py) -- only if it was taken on this attention shape."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        d = json.load(open(path))
        if d.get("attn_shape") == cfg.get("attn_shape"):
            return d["kernels"]["attn_bwd"]["dram_bytes"], f"profiles/ncu_traffic.json ({d['source']}; {d['workload']})"
    except Exception:
        pass
    return None, None


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        clocks, maxc, reasons = [], None, set()
        for r in self.rows:
            try:
                clocks.append(float(r[1]))
                maxc = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        clocks.sort()
        med = clocks[len(clocks) // 2] if clocks else None
        return {"sm_mhz": med, "sm_max_mhz": maxc, "reasons": sorted(reasons), "samples": len(clocks)}


def synth_lengths(batch, lmax, device, seed):
    from generative_recommenders_b200.common import apply_sampling, generate_sparse_seq_len

    torch.manual_seed(seed)
    lengths = generate_sparse_seq_len(batch, lmax, 0.95, device)
    lengths = apply_sampling(lengths, 2.0, lmax)
    nt = torch.randint(1, 21, (batch,), device=device, dtype=lengths.dtype)
    nt = torch.where(nt > lengths, lengths, nt).to(torch.int32)
    off = torch.zeros(batch + 1, dtype=torch.int64, device=device)
    off[1:] = torch.cumsum(lengths, 0)
    return lengths, nt, off


def attn_inputs(L, heads, d, dev):
    """q|k|v as views of one [L, H, 3d] buffer, uniform(-0.01, 0.01), dO ~ N(0,1): hstu_attention_bench.py:222-248."""
    torch.manual_seed(2002)
    x = torch.empty(L, heads, 3 * d, device=dev, dtype=torch.bfloat16).uniform_(-0.01, 0.01)
    do = torch.randn(L, heads, d, device=dev, dtype=torch.bfloat16)
    return x, do


DUMP_BYTES = 64_000_000  # all files of --dump-outputs together
DUMP_SEED = 12345  # row sample of outputs that do not fit whole


def dump_outputs(out_dir, whole, sampled):
    """Write every tensor of `whole` entirely and of every tensor of `sampled` a seeded sample of rows (dim 0), as many as
    the rest of DUMP_BYTES allows, as out_dir/<name>.npy in float32.  The sample depends only on the row count and
    DUMP_SEED, so two runs with the same arguments write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {name: t.detach().float().cpu() for name, t in whole.items()}
    header = 128  # .npy header of one file (format 1.0)
    left = DUMP_BYTES - sum(a.numel() * 4 + header for a in arrays.values()) - header * len(sampled)
    for name, t in sampled.items():
        rows = t.shape[0]
        row_bytes = 4 * (t.numel() // max(rows, 1))
        keep = min(rows, max(0, left // len(sampled)) // max(row_bytes, 1))
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(DUMP_SEED))[:keep].sort().values
        arrays[name] = t.detach()[idx.to(t.device)].float().cpu()
    total = 0
    for name, a in arrays.items():
        path = os.path.join(out_dir, f"{name}.npy")
        np.save(path, a.numpy())
        total += os.path.getsize(path)
    assert total <= DUMP_BYTES, (total, DUMP_BYTES)
    return total


def attn_flops(lengths, heads, dqk, dv):
    """Reference FLOP model (hstu_attention_bench.py:35-59): causal-halved, 2 FLOP per MAC."""
    s2 = float((lengths.double() ** 2).sum())
    f1 = 2.0 * heads * dqk * s2 / 2.0
    f2 = 2.0 * heads * dv * s2 / 2.0
    return dict(fwd=f1 + f2, bwd=3 * f1 + 2 * f2)


def attn_bytes(lengths, heads, dqk, dv, elt=2):
    """Algorithmic bytes, every tensor touched once (SURVEY.md section 8d)."""
    rows = float(lengths.double().sum())
    return dict(fwd=elt * rows * heads * (2 * dqk + 2 * dv), bwd=elt * rows * heads * (4 * dqk + 3 * dv))


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from generative_recommenders_b200 import _lib
    from generative_recommenders_b200.modules.stu import STULayer, STULayerConfig, STUStack
    from generative_recommenders_b200.ops.hstu_attention import hstu_mha

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    last = {} if args.dump_outputs and rank == 0 else None  # outputs of the latest step, for --dump-outputs
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
    _lib.lib()
    D, H, dh, layers = 256, 8, 32, args.layers
    # the same seeded lengths on every rank (weak scaling: identical sum of len^2 per GPU, so the curve measures the collective
    # and not a straggler); the activations / gradients differ per rank (seeded below)
    lengths, nt, off = synth_lengths(args.batch, args.lmax, dev, 1001)
    torch.cuda.manual_seed(4321 + rank)  # dropout masks: CUDA generator, different per rank
    seqs_total = args.batch * world
    if args.scaling == "strong" and world > 1:
        # fixed global batch: this rank keeps its shard of the SAME seeded batch (balanced by attention cost)
        from generative_recommenders_b200.distributed import shard_sequences

        mine = shard_sequences(lengths.tolist(), world)[rank]
        idx = torch.tensor(mine, device=dev, dtype=torch.long)
        lengths, nt = lengths[idx], nt[idx]
        off = torch.zeros(len(mine) + 1, dtype=torch.int64, device=dev)
        off[1:] = torch.cumsum(lengths, 0)
        seqs_total = args.batch
    L = int(off[-1])

    if args.workload == "hstu_large":
        torch.manual_seed(7)  # identical initial weights on every rank (DDP broadcast equivalent)
        stack = STUStack([STULayer(STULayerConfig(embedding_dim=D, num_heads=H, hidden_dim=dh, attention_dim=dh,
                                                  output_dropout_ratio=0.2, target_aware=True, recompute_normed_x=True,
                                                  recompute_uvqk=True, recompute_y=True, sort_by_length=True))
                          for _ in range(layers)]).to(dev).to(torch.bfloat16)
        params = [p for p in stack.parameters()]
        opt = torch.optim.AdamW(params, lr=1e-4, fused=True)
        torch.manual_seed(100 + rank)
        x_dev = torch.randn(L, D, device=dev, dtype=torch.bfloat16)
        # e2e: the step's inputs live in pinned host memory and are copied in every step
        x_host = x_dev.cpu().pin_memory()
        off_host, nt_host, len_host = off.cpu().pin_memory(), nt.cpu().pin_memory(), lengths.cpu().pin_memory()
        h2d_bytes = x_host.numel() * 2 + off_host.numel() * 8 + nt_host.numel() * 4 + len_host.numel() * 4
        from generative_recommenders_b200.distributed import LayerBucketAllReduce

        # gradients live in one flat bf16 buffer (p.grad are views); for N > 1 one in-place NCCL all-reduce (AVG) per STU layer
        # is launched on a side stream as soon as that layer's grads are final.  Same code path at N = 1 (no collective).
        reducer = LayerBucketAllReduce(list(stack._stu_layers), world, dev)

        def step(e2e: bool):
            if e2e:
                x = x_host.to(dev, non_blocking=True)
                o_ = off_host.to(dev, non_blocking=True)
                n_ = nt_host.to(dev, non_blocking=True)
                l_ = len_host.to(dev, non_blocking=True)
            else:
                x, o_, n_, l_ = x_dev, off, nt, lengths
            reducer.zero_grad()
            y = stack(x=x, x_lengths=l_, x_offsets=o_, max_seq_len=args.lmax, num_targets=n_)
            loss = y.float().square().mean()
            loss.backward()
            reducer.wait()
            opt.step()
            if last is not None:
                last["y"], last["loss"] = y, loss
            if e2e:
                return float(loss.item())  # device -> host read of the step result
            return loss

        units_per_step = seqs_total / world
        d2h_bytes = 4
        cfg = {"workload": f"HSTU-large stack fwd+bwd+AdamW: {layers} layers, D=256, H=8, dqk=dv=32, bf16, Lmax={args.lmax}, "
                           f"{args.batch} user sequences{'/GPU' if args.scaling == 'weak' else ' in total (sharded by sum len^2)'} (lengths U[0.9,1.0)*Lmax, 1-20 targets, seed 1001 on every rank; activations seeded per rank), dropout 0.2",
               "global_batch": seqs_total, "seq_len": args.lmax, "rows_per_gpu": L,
               "parallelism": f"dp{world} (batch-sharded, per-layer in-place bf16 NCCL all-reduce of the flat gradient bucket overlapped with backward)",
               "l2": f"inputs + activations per step ({L * D * 2 * 6 / 1e6:.0f} MB+) exceed the 126 MB L2; no explicit flush"}
        cfg["attn_shape"] = {"batch": args.batch, "lmax": args.lmax, "heads": H, "d": dh}
        aflops = attn_flops(lengths, H, dh, dh)
        abytes = attn_bytes(lengths, H, dh, dh)
        per_step_calls = layers
    else:
        d = args.attn_dim
        Ha = args.attn_heads
        x, do = attn_inputs(L, Ha, d, dev)
        q, k, v = torch.split(x, [d, d, d], dim=-1)
        q.requires_grad_(True), k.requires_grad_(True), v.requires_grad_(True)
        alpha = 1.0 / d
        x_host = x.detach().cpu().pin_memory()
        h2d_bytes = x_host.numel() * 2

        def step(e2e: bool):
            if e2e:
                xx = x_host.to(dev, non_blocking=True)
                qq, kk, vv = torch.split(xx, [d, d, d], dim=-1)
                qq.requires_grad_(True), kk.requires_grad_(True), vv.requires_grad_(True)
            else:
                qq, kk, vv = q, k, v
                q.grad = k.grad = v.grad = None
            o = hstu_mha(args.lmax, alpha, qq, kk, vv, off, num_targets=nt, sort_by_length=True, impl=args.attn_impl)
            o.backward(do)
            if last is not None:
                last.update(out=o, dq=qq.grad, dk=kk.grad, dv=vv.grad)
            if e2e:
                return float(o[0, 0, 0].item())
            return o

        units_per_step = args.batch
        d2h_bytes = 2
        cfg = {"workload": f"hstu_mha fwd+bwd microbench (hstu_attention_bench.py recipe): B={args.batch}, H={Ha}, d={d}, "
                           f"Lmax={args.lmax}, bf16, alpha=1/d, targets<=20", "global_batch": args.batch * world,
               "seq_len": args.lmax, "rows_per_gpu": L, "parallelism": f"dp{world} (independent shards)",
               "l2": f"q,k,v,o,grads = {L * Ha * d * 2 * 11 / 1e6:.0f} MB per step > 126 MB L2" }
        cfg["attn_shape"] = {"batch": args.batch, "lmax": args.lmax, "heads": Ha, "d": d}
        aflops = attn_flops(lengths, Ha, d, d)
        abytes = attn_bytes(lengths, Ha, d, d)
        per_step_calls = 1

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed_run(e2e: bool, steps: int, warmup: int, with_kernel_timing: bool):
        for _ in range(warmup):
            step(e2e)
        sync_all()
        _lib.enable_timing(with_kernel_timing)
        launches0 = _lib.LAUNCHES
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step(e2e)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            dist.barrier()
        events = _lib.timed_events()
        _lib.enable_timing(False)
        return ms, _lib.LAUNCHES - launches0, events

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches, events = timed_run(False, args.steps, args.warmup, True)
    clocks = sampler.stop() if sampler else None
    ms_e2e, _, _ = timed_run(True, args.steps, 1, False)
    if last is not None:
        if args.workload == "hstu_large":
            # the training step returns the loss and leaves the stack output and the parameter gradients to its caller
            whole = {"loss": last["loss"]}
            whole.update({f"grad.{n}": p.grad for n, p in stack.named_parameters()})
            dump_outputs(args.dump_outputs, whole, {"y": last["y"]})
        else:
            dump_outputs(args.dump_outputs, {}, {k: last[k] for k in ("out", "dq", "dk", "dv")})

    value = units_per_step * world * args.steps / (ms * 1e-3)
    value_e2e = units_per_step * world * args.steps / (ms_e2e * 1e-3)
    peaks = measured_peaks()
    kt = {}
    for name, evs in (events or {}).items():
        kt[name] = sum(a.elapsed_time(b) for a, b in evs) / max(1, len(evs))  # ms per call
    out = {
        "metric": "user-seqs/sec HSTU-large L=8192 d=256 bf16 fwd+bwd" if args.workload == "hstu_large" else
                  "user-seqs/sec hstu_mha fwd+bwd microbench",
        "value": value, "unit": "sequences/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": cfg,
        "e2e": {"value": value_e2e, "unit": "sequences/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "clocks": clocks,
    }
    if "attn_bwd" in kt and "attn_fwd" in kt:
        tf_b = aflops["bwd"] / (kt["attn_bwd"] * 1e-3) / 1e12
        tf_f = aflops["fwd"] / (kt["attn_fwd"] * 1e-3) / 1e12
        peak = peaks["tflops_sustained"]
        traffic, traffic_src = ncu_traffic(cfg)
        out["roofline"] = {
            "kernel": "hstu_attn_bwd (dK/dV + dQ kernels of one layer call)", "bound": "tensor", "achieved": tf_b, "peak": peak,
            "unit": "TFLOP/s", "frac": tf_b / peak, "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peaks["source"] + ", sustained bf16",
            "ms_per_launch": kt["attn_bwd"], "algorithmic_flops_per_launch": aflops["bwd"],
            "fwd": {"achieved": tf_f, "frac": tf_f / peak, "ms_per_launch": kt["attn_fwd"],
                    "algorithmic_flops_per_launch": aflops["fwd"],
                    "hbm_gbs_algorithmic": abytes["fwd"] / (kt["attn_fwd"] * 1e-3) / 1e9},
            "bwd_hbm_gbs_algorithmic": abytes["bwd"] / (kt["attn_bwd"] * 1e-3) / 1e9, "hbm_peak_gbs": peaks["hbm_gbs"],
            "attn_share_of_step": (kt["attn_bwd"] + kt["attn_fwd"]) * per_step_calls / (ms / args.steps),
            # what bounds the kernel below the tensor peak at this head dim: measured by timing-only ablations, not assumed
            "bound_evidence": "profiles/r02_ablations.txt (d = 32 backward: tcgen05 issue rate of its N = 32 MMAs, 1464 clk per "
                              "128 x 128 tile = 0.67 of the bf16 peak for this tiling; forward: serial chain of a TMEM score slot)",
        }
    out["kernel_ms_per_call"] = {k: round(v, 4) for k, v in sorted(kt.items())}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args, seconds_budget=20.0)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(out))


# ----------------------------------------------------------------------------------------------------------------
# research-path configs of BASELINE.json (2: ML-20M HSTU-large, 3: Amazon-Books HSTU-large): item embedding -> 16 research
# blocks (relative position / time bias attention) -> sampled-softmax loss -> backward -> AdamW, synthetic data
# ----------------------------------------------------------------------------------------------------------------
RESEARCH_CFG = {
    # configs/ml-20m/hstu-sampled-softmax-n128-large-final.gin, configs/amzn-books/hstu-sampled-softmax-n512-large-final.gin
    # (SURVEY.md section 8 table): D, layers, H, dqk = dv, n = max_sequence_length + gr_output_length + 1, batch, negatives, items
    "ml20m": dict(D=256, layers=16, H=8, d=32, n=211, B=128, R=128, V=131263, name="ML-20M HSTU-large"),
    "amzn_books": dict(D=64, layers=16, H=8, d=8, n=61, B=128, R=512, V=695763, name="Amazon-Books HSTU-large"),
}


def run_research(args):
    from generative_recommenders_b200 import _lib
    from generative_recommenders_b200.modules.research_hstu import (RelativeBucketedTimeAndPositionBasedBias,
                                                                    SequentialTransductionUnitJagged)
    from generative_recommenders_b200.modules.sampled_softmax import LocalNegativesSampler, SampledSoftmaxLoss

    c = RESEARCH_CFG[args.workload]
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    _lib.lib()
    torch.manual_seed(7)
    D, H, d, n, B, R, V = c["D"], c["H"], c["d"], c["n"], c["B"], c["R"], c["V"]
    emb = torch.nn.Embedding(V, D)
    blocks = torch.nn.ModuleList([
        SequentialTransductionUnitJagged(embedding_dim=D, linear_hidden_dim=d, attention_dim=d, dropout_ratio=0.2,
                                         attn_dropout_ratio=0.0, num_heads=H, linear_activation="silu",
                                         relative_attention_bias_module=RelativeBucketedTimeAndPositionBasedBias(n, 128),
                                         normalization="rel_bias", linear_config="uvqk", concat_ua=False, epsilon=1e-6, max_length=n)
        for _ in range(c["layers"])])
    model = torch.nn.ModuleDict({"emb": emb, "blocks": blocks}).to(dev).to(torch.bfloat16)
    sampler = LocalNegativesSampler(V, model["emb"], list(range(V)), l2_norm=True, l2_norm_eps=1e-6).to(dev)
    loss_mod = SampledSoftmaxLoss(num_to_sample=R, softmax_temperature=0.05)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, fused=True)
    g = torch.Generator(device="cpu").manual_seed(1001)
    lengths = torch.randint(n // 2, n + 1, (B,), generator=g)
    off = torch.zeros(B + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(lengths, 0)
    L = int(off[-1])
    ids_host = torch.randint(1, V, (L,), generator=g).pin_memory()
    ts_host = torch.cumsum(torch.randint(0, 86400, (B, n), generator=g), dim=1).pin_memory()
    off_d = off.to(dev)
    mask = torch.tril(torch.ones(n, n, device=dev))
    ids_dev, ts_dev = ids_host.to(dev), ts_host.to(dev)
    nxt = torch.arange(1, L + 1, device=dev).clamp(max=L - 1)  # next-item supervision inside the flat row order (synthetic)
    w_dev = torch.ones(L, device=dev, dtype=torch.bfloat16)
    last = {} if args.dump_outputs else None  # outputs of the latest step, for --dump-outputs

    def step(e2e):
        ids = ids_host.to(dev, non_blocking=True) if e2e else ids_dev
        ts = ts_host.to(dev, non_blocking=True) if e2e else ts_dev
        opt.zero_grad(set_to_none=True)
        x = model["emb"](ids)
        for blk in model["blocks"]:
            x, _ = blk(x, off_d, ts, mask)
        sup_ids = ids[nxt]
        loss, _ = loss_mod.jagged_forward(output_embeddings=x, supervision_ids=sup_ids, supervision_embeddings=model["emb"](sup_ids),
                                          supervision_weights=w_dev, negatives_sampler=sampler)
        loss.backward()
        opt.step()
        if last is not None:
            last["x"], last["loss"] = x, loss
        return float(loss.item()) if e2e else loss

    def timed(e2e, steps, warmup, with_events):
        for _ in range(warmup):
            step(e2e)
        torch.cuda.synchronize(dev)
        _lib.enable_timing(with_events)
        l0 = _lib.LAUNCHES
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step(e2e)
        e1.record()
        torch.cuda.synchronize(dev)
        ev = _lib.timed_events()
        _lib.enable_timing(False)
        return e0.elapsed_time(e1), _lib.LAUNCHES - l0, ev

    sampler_c = ClockSampler(dev.index or 0)
    sampler_c.start()
    ms, launches, events = timed(False, args.steps, args.warmup, True)
    clocks = sampler_c.stop()
    ms_e2e, _, _ = timed(True, args.steps, 1, False)
    if last is not None:
        # the loss, the output embeddings of the last block and the gradients of the blocks; the item table's gradient (V x D)
        # is row-sampled like the embeddings
        whole = {"loss": last["loss"]}
        whole.update({f"grad.{n}": p.grad for n, p in model["blocks"].named_parameters() if p.grad is not None})
        dump_outputs(args.dump_outputs, whole, {"x": last["x"], "grad.emb.weight": model["emb"].weight.grad})
    kt = {k: round(sum(a.elapsed_time(b) for a, b in v) / max(1, len(v)), 4) for k, v in (events or {}).items()}
    print(json.dumps({
        "metric": f"user-seqs/sec {c['name']} (research path) fwd+bwd+AdamW", "value": B * args.steps / (ms * 1e-3), "unit": "sequences/s",
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{c['name']}: item embedding ({V} x {D}) -> {c['layers']} research HSTU blocks (D={D}, H={H}, dqk=dv={d}, "
                               f"n={n}, relative position + time bias) -> sampled softmax ({R} negatives, l2 norm, T=0.05), batch {B}, "
                               f"{L} rows, dropout 0.2, bf16", "global_batch": B, "seq_len": n, "rows_per_gpu": L,
                   "l2": "the whole working set fits the 126 MB L2 except the embedding table; launch-bound at this size"},
        "e2e": {"value": B * args.steps / (ms_e2e * 1e-3), "unit": "sequences/s", "h2d_bytes_per_step": ids_host.numel() * 8 + ts_host.numel() * 8,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "clocks": clocks, "kernel_ms_per_call": kt}))


# ----------------------------------------------------------------------------------------------------------------
# GPU comparator: the reference's own Triton kernel (unmodified, from baseline/_ref) on the same inputs
# ----------------------------------------------------------------------------------------------------------------
def run_triton(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if args.workload != "attn" or not os.path.isdir(os.path.join(ref_root, "generative_recommenders")):
        print(json.dumps({"impl": "triton", "unavailable": "needs --workload attn and baseline/_ref (scripts/fetch_triton_baseline.py)"}))
        return
    sys.path.insert(0, ref_root)
    try:
        # triton 3.6 no longer has the experimental TMA entry points the reference file names in its ENABLE_TMA branches.  Those
        # branches are statically dead here (enable_tma=False), but Triton's early-return checker resolves every attribute it
        # sees (code_generator.ContainsReturnChecker.visit_Attribute -> getattr) and would raise AttributeError: give the two names
        # a placeholder.  The kernels that run are the reference's own non-TMA kernels, unmodified.
        import triton.language as tl

        for name in ("_experimental_descriptor_load", "_experimental_descriptor_store"):
            if not hasattr(tl, name):
                setattr(tl, name, None)
        from generative_recommenders.ops.triton.triton_hstu_attention import triton_hstu_mha
    except Exception as e:  # noqa: BLE001
        print(json.dumps({"impl": "triton", "unavailable": f"import failed: {type(e).__name__}: {e}"[:300]}))
        return
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lengths, nt, off = synth_lengths(args.batch, args.lmax, dev, 1001)
    L = int(off[-1])
    d, Ha = args.attn_dim, args.attn_heads
    x, do = attn_inputs(L, Ha, d, dev)
    q, k, v = torch.split(x, [d, d, d], dim=-1)
    q.requires_grad_(True), k.requires_grad_(True), v.requires_grad_(True)
    alpha = 1.0 / d
    t_f, t_b = [], []

    def step(record):
        q.grad = k.grad = v.grad = None
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        o = triton_hstu_mha(args.lmax, alpha, q, k, v, off, num_targets=nt, max_attn_len=0, contextual_seq_len=0,
                            sort_by_length=True, enable_tma=False)
        e[1].record()
        o.backward(do)
        e[2].record()
        if record:
            t_f.append((e[0], e[1]))
            t_b.append((e[1], e[2]))

    t0 = time.perf_counter()
    try:
        for _ in range(max(1, args.warmup)):  # the first call autotunes (29 forward + 20 backward configurations)
            step(False)
        torch.cuda.synchronize()
        tune_s = time.perf_counter() - t0
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(args.steps):
            step(True)
        s1.record()
        torch.cuda.synchronize()
    except Exception as e:  # noqa: BLE001
        import traceback

        traceback.print_exc()
        cause = e.__cause__ or e.__context__
        print(json.dumps({"impl": "triton", "unavailable": (f"run failed: {type(e).__name__}: {str(e)[-1500:]}"
                                                            + (f" | cause: {type(cause).__name__}: {str(cause)[-800:]}" if cause else "")),
                          "config": {"attn_shape": {"batch": args.batch, "lmax": args.lmax, "heads": Ha, "d": d}}}))
        return
    ms = s0.elapsed_time(s1) / args.steps
    ms_f = sum(a.elapsed_time(b) for a, b in t_f) / len(t_f)
    ms_b = sum(a.elapsed_time(b) for a, b in t_b) / len(t_b)
    fl, by = attn_flops(lengths, Ha, d, d), attn_bytes(lengths, Ha, d, d)
    best = {}
    try:
        import generative_recommenders.ops.triton.triton_hstu_attention as T

        for name in ("_hstu_attn_fwd", "_hstu_attn_bwd"):
            cache = getattr(getattr(T, name), "cache", {})
            best[name] = [str(c) for c in cache.values()][:2]
    except Exception:  # noqa: BLE001
        pass
    import triton

    print(json.dumps({
        "impl": "triton", "metric": "user-seqs/sec hstu_mha fwd+bwd microbench", "value": args.batch / (ms * 1e-3),
        "unit": "sequences/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"reference triton_hstu_mha fwd+bwd (sort_by_length=True, enable_tma=False, autotuned, triton "
                               f"{triton.__version__}): B={args.batch}, H={Ha}, d={d}, Lmax={args.lmax}, bf16, alpha=1/d",
                   "attn_shape": {"batch": args.batch, "lmax": args.lmax, "heads": Ha, "d": d}, "rows_per_gpu": L},
        "kernel_ms_per_call": {"attn_fwd": round(ms_f, 4), "attn_bwd": round(ms_b, 4)},
        "tflops": {"fwd": fl["fwd"] / (ms_f * 1e-3) / 1e12, "bwd": fl["bwd"] / (ms_b * 1e-3) / 1e12},
        "hbm_gbs_algorithmic": {"fwd": by["fwd"] / (ms_f * 1e-3) / 1e9, "bwd": by["bwd"] / (ms_b * 1e-3) / 1e9},
        "autotune_seconds": round(tune_s, 1), "autotune_best": best,
    }))


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference eager path on the host cores
# ----------------------------------------------------------------------------------------------------------------
_REF_LAYER = None


def reference_layer():
    """The reference's OWN eager STULayer (unmodified Python, fetched into the git-ignored oracle/_ref/ by
    scripts/fetch_reference_eager.py; fbgemm_gpu's three jagged ops come from oracle/fbgemm_shim.py), HammerKernel.PYTORCH, fp32.
    None if oracle/_ref is absent (then the oracle port is timed instead)."""
    global _REF_LAYER
    if _REF_LAYER is None:
        ref_root = os.path.join(ROOT, "oracle", "_ref")
        if not os.path.isdir(os.path.join(ref_root, "generative_recommenders")):
            _REF_LAYER = False
            return None
        try:
            sys.path.insert(0, ref_root)
            from oracle import fbgemm_shim

            fbgemm_shim.install()
            import warnings

            warnings.filterwarnings("ignore")
            from generative_recommenders.common import HammerKernel as RefKernel
            from generative_recommenders.modules.stu import STULayer as RefLayer, STULayerConfig as RefConfig

            torch.manual_seed(7)
            layer = RefLayer(RefConfig(embedding_dim=256, num_heads=8, hidden_dim=32, attention_dim=32, output_dropout_ratio=0.0,
                                       causal=True, target_aware=True))
            layer.recursive_setattr("_hammer_kernel", RefKernel.PYTORCH) if hasattr(layer, "recursive_setattr") else \
                layer.set_hammer_kernel(RefKernel.PYTORCH)
            assert layer.hammer_kernel() == RefKernel.PYTORCH
            _REF_LAYER = layer
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"reference eager layer unavailable ({type(e).__name__}: {e}); timing the oracle port instead\n")
            _REF_LAYER = False
    return _REF_LAYER or None


def cpu_kind():
    return "reference" if reference_layer() is not None else "port"


def cpu_engine_name():
    return ("reference eager STULayer (unmodified generative_recommenders code from oracle/_ref + fbgemm shim, HammerKernel.PYTORCH)"
            if reference_layer() is not None else "oracle (fp32 CPU port of the reference eager path)")


def cpu_sample(args, layers_sampled: int, prefix: int = 0):
    """One sequence (the first of the seeded batch) -- or, if `prefix` > 0, its first `prefix` rows (a causal prefix of a user
    history is itself a valid, shorter history) -- through `layers_sampled` independent STU layers fwd+bwd in fp32 on CPU.
    Returns (seconds, rows processed, full length of the sequence)."""
    from oracle import hstu_oracle as O

    dev = torch.device("cpu")
    D, H, dh = 256, 8, 32
    torch.manual_seed(1001)
    lmax = args.lmax
    full = int(torch.randint(int(0.9 * lmax), lmax, (1,)).item())
    length = min(full, prefix) if prefix > 0 else full
    off = torch.tensor([0, length], dtype=torch.int64)
    nt = torch.tensor([min(7, length)], dtype=torch.int64)
    x = torch.randn(full, D, device=dev)[:length]
    Wd = 4 * H * dh
    params = {"_input_norm_weight": torch.ones(D), "_input_norm_bias": torch.zeros(D),
              "_uvqk_weight": torch.randn(D, Wd) * 0.05, "_uvqk_beta": torch.zeros(Wd),
              "_output_norm_weight": torch.ones(H * dh), "_output_norm_bias": torch.zeros(H * dh),
              "_output_weight": torch.randn(3 * H * dh, D) * 0.05}
    ref = reference_layer()
    t0 = time.perf_counter()
    for _ in range(layers_sampled):
        if ref is not None:
            xx = x.detach().clone().requires_grad_()
            n_pad = length if prefix > 0 else lmax  # the eager path pads to max_seq_len: a prefix is its own (shorter) problem
            y = ref(x=xx, x_lengths=torch.tensor([length]), x_offsets=off, max_seq_len=n_pad, num_targets=nt)
            y.backward(torch.ones_like(y))
        else:
            O.stu_layer_fwd_bwd_timed(x, off, lmax, nt, params, H, dh, dh)
    return time.perf_counter() - t0, length, full


def pick_cpu_threads(args, probe_rows: int):
    """The eager CPU path is partly memory-bound: on a many-core host all threads are not the fastest setting.  Time a short
    prefix with a few thread counts and keep the best, so that the CPU arm is the reference at its best on this host."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (cores, cores // 2, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    best, best_t = cores, float("inf")
    for c in cands:
        torch.set_num_threads(c)
        cpu_sample(args, 1, probe_rows)          # warm-up of this pool size
        t, _, _ = cpu_sample(args, 1, probe_rows)
        if t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best, cores


def cpu_baseline(args, seconds_budget: float):
    if args.workload != "hstu_large":
        return {"value": None, "unit": "sequences/s", "cores": os.cpu_count() or 1, "kind": cpu_kind(),
                "sample": "not measured for this workload"}
    cores, host_cores = pick_cpu_threads(args, max(256, min(1024, args.lmax // 8)))
    t1, length, _ = cpu_sample(args, 1)  # also the warm-up
    n = max(1, min(args.layers, int(seconds_budget / max(t1, 1e-3))))
    t, _, _ = cpu_sample(args, n)
    per_seq = t / n * args.layers
    return {"value": 1.0 / per_seq, "unit": "sequences/s", "cores": cores, "kind": cpu_kind(),
            "sample": f"{cpu_engine_name()}, fp32, 1 user sequence of length {length}, {n} of "
                      f"{args.layers} STU layers fwd+bwd in {t:.1f} s, scaled x{args.layers / n:.1f} to the full stack; "
                      f"{cores} threads (fastest of the probed settings on this {host_cores}-core host)"}


REFERENCE_ARM_BUDGET_S = 150.0  # wall time the K timed steps of the CPU arm may take together


def run_reference(args):
    """CPU arm: the oracle port of the reference eager path on all host threads.  One step = one STU layer fwd+bwd on one user
    sequence of the workload -- the whole sequence when K such steps fit the time budget, otherwise a causal prefix of it, scaled
    back with the cost model t(l) = a l^2 + b l fitted on two short prefixes during the (untimed) warm-up."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # calibration (untimed; also the warm-up of the thread pool and allocator)
    l1 = max(256, min(1024, args.lmax // 8))
    l2 = 2 * l1
    cores, host_cores = pick_cpu_threads(args, l2)
    cpu_sample(args, 1, l1)
    t1, l1, full = cpu_sample(args, 1, l1)
    t2, l2, _ = cpu_sample(args, 1, l2)
    a = max((t2 / l2 - t1 / l1) / (l2 - l1), 0.0)
    b = max(t1 / l1 - a * l1, 1e-9)
    model = lambda l: a * l * l + b * l  # noqa: E731
    per_step = REFERENCE_ARM_BUDGET_S / max(1, args.steps)
    prefix = full
    if model(full) > per_step:
        prefix = l2
        while prefix * 2 <= full and model(prefix * 2) <= per_step:
            prefix *= 2
    scale = model(full) / model(prefix) if prefix < full else 1.0
    for _ in range(min(args.warmup, 1)):
        cpu_sample(args, 1, prefix)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_sample(args, 1, prefix)
    dt = time.perf_counter() - t0
    per_seq = dt / args.steps * scale * args.layers
    value = 1.0 / per_seq
    what = (f"1 user sequence (length {full}) x 1 STU layer fwd+bwd per step" if prefix >= full else
            f"the first {prefix} rows of 1 user sequence (length {full}) x 1 STU layer fwd+bwd per step, scaled x{scale:.2f} to the "
            f"full length with t(l) = {a:.3e} l^2 + {b:.3e} l fitted on prefixes {l1}, {l2}")
    out = {
        "impl": "reference", "metric": "user-seqs/sec HSTU-large L=8192 d=256 bf16 fwd+bwd", "value": value,
        "unit": "sequences/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"HSTU-large stack fwd+bwd: {args.layers} layers, D=256, H=8, dqk=dv=32, Lmax={args.lmax} "
                               f"({cpu_engine_name()}; each step = a bounded sample, scaled to one sequence through the stack)"},
        "cpu_baseline": {"value": value, "unit": "sequences/s", "cores": cores, "kind": cpu_kind(),
                         "sample": f"{cpu_engine_name()}: {what}, fp32, {cores} threads (fastest of the probed settings on this {host_cores}-core host); "
                                   f"scaled x{args.layers} layers"},
        "e2e": {"value": value, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


if __name__ == "__main__":
    sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ next to the sources
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "triton":
        run_triton(a)
    elif a.workload in RESEARCH_CFG:
        run_research(a)
    else:
        run_ours(a)
