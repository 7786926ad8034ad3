#!/usr/bin/env python
"""bench.py - HSTU training sequences/sec (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE configs[1] - HSTU 4 blocks, d=128, h=4, seq_len=200, V=12,101 synthetic
Beauty-shaped items, B=128 sequences per GPU, bf16 tensor-core operands, dropout 0.2, Adam - one full training step =
embedding gather -> 4 HSTU blocks -> final LN -> tied logits + CE -> backward -> (all-reduce) -> Adam.

One JSON line on stdout (rank 0):  value = whole-job sequences/s with the batch already resident in HBM;
e2e = the same through the public nn.Module API with pinned-host inputs copied H2D and the loss read back D2H every
step; roofline = the HSTU block stack (fwd+bwd, 4 layers) against the measured bf16 peak; cpu_baseline = the oracle port
of the reference's CPU-eager path on this box's host cores (bounded sample).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = {
    # BASELINE.json configs[1] (the configuration the metric is quoted on) and configs[2] (the long-sequence regime)
    "cfg2": dict(model=dict(num_items=12101, max_seq_len=200, embed_dim=128, num_heads=4, num_blocks=4, dropout=0.2), batch=128,
                 cpu_batch=32, eager_batch=128),
    "cfg3": dict(model=dict(num_items=12101, max_seq_len=2048, embed_dim=256, num_heads=8, num_blocks=8, dropout=0.2), batch=32,
                 cpu_batch=1, eager_batch=4),
}
CFG = dict(CONFIGS["cfg2"]["model"])
METRIC = "hstu_train_sequences_per_sec"
UNIT = "sequences/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cuda_eager"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS), help="cfg2 = BASELINE configs[1] (default), cfg3 = configs[2]")
    ap.add_argument("--batch", type=int, default=None, help="sequences per GPU")
    ap.add_argument("--seq-len", type=int, default=None)
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of a captured CUDA graph")
    ap.add_argument("--cpu-batch", type=int, default=None)
    ap.add_argument("--eager-batch", type=int, default=None)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-eager", action="store_true")
    ap.add_argument("--skip-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (loss, parameters after the optimizer step) as "
                         "DIR/<name>.npy in float32.  That step starts from the initial parameters and optimizer state and its batch "
                         "and dropout seed follow from the arguments, so two runs or two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    c = CONFIGS[args.config]
    CFG.clear(); CFG.update(c["model"])
    args.batch = args.batch or c["batch"]
    args.seq_len = args.seq_len or CFG["max_seq_len"]
    args.cpu_batch = args.cpu_batch or c["cpu_batch"]
    args.eager_batch = args.eager_batch or c["eager_batch"]
    return args


# ------------------------------------------------------------------------------------------------ synthetic data
def synth_batch(B, L, V, seed):
    """SURVEY.md section 8(d): ids ~ Zipf(1.1) over 1..V, timestamps = 1.30e9 + cumsum(Exp(mean 3 days)), full-length
    sequences (throughput set), targets = ids shifted by one with a fresh last item."""
    g = torch.Generator().manual_seed(seed)
    w = torch.arange(1, V + 1, dtype=torch.float64).pow(-1.1)
    ids = torch.multinomial(w, B * (L + 1), replacement=True, generator=g).view(B, L + 1) + 1
    gaps = torch.empty(B, L).exponential_(1.0 / (3 * 86400.0), generator=g).long() + 1
    ts = 1_300_000_000 + torch.cumsum(gaps, 1)
    return ids[:, :L].contiguous(), ts.contiguous(), ids[:, 1:].contiguous()


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def usable_cpus() -> int:
    """Host threads this process may really use: min(affinity, cgroup CPU quota) - a 128-core host with a 16-CPU quota runs
    32x slower when torch spawns 128 threads."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:  # noqa: BLE001
        pass
    return max(1, n)


# ------------------------------------------------------------------------------------------------ CPU arm (oracle port)
def cpu_arm(batch, L, seconds, steps=None, warmup=1):
    """The reference's CPU-eager algorithm (oracle restatement, fp32, all host threads), full train-step fwd+bwd
    (+ Adam) on a bounded sample of the same workload.  bench.py executes oracle/ only in its baseline legs (this one,
    --impl reference, and the same-GPU eager arm)."""
    from oracle import hstu as oh
    from genrec_b200.hstu import HSTU
    threads = usable_cpus()
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    m = HSTU(**{**CFG, "max_seq_len": L, "dropout": 0.0})
    params = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    opt = torch.optim.Adam(list(params.values()), lr=1e-3, betas=(0.9, 0.98))
    ids, ts, tg = synth_batch(batch, L, CFG["num_items"], 123)

    def one():
        opt.zero_grad(set_to_none=True)
        _, loss = oh.hstu_forward(ids, ts, tg, params, CFG["num_heads"], CFG["num_blocks"])
        loss.backward()
        opt.step()
        return float(loss)

    for _ in range(warmup):
        one()
    times = []
    t_end = time.perf_counter() + seconds
    while (steps is None and time.perf_counter() < t_end and len(times) < 50) or (steps is not None and len(times) < steps):
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
        if steps is None and len(times) >= 3 and time.perf_counter() > t_end:
            break
    return dict(threads=threads, batch=batch, times=times, seq_per_s=batch / (sum(times) / len(times)),
                ms_per_step=1e3 * sum(times) / len(times))


def cuda_eager_arm(batch, L, dev, steps, warmup=2):
    """The reference's algorithm as plain PyTorch eager ON THE SAME GPU (oracle restatement, torch.autocast(bf16), dropout 0, Adam):
    the "beat this on the same box" number of BASELINE.md section 2.2 - the reference ships no kernel of its own."""
    from oracle import hstu as oh
    from genrec_b200.hstu import HSTU
    torch.manual_seed(0)
    m = HSTU(**{**CFG, "max_seq_len": L, "dropout": 0.0})
    params = {k: v.detach().clone().to(dev).requires_grad_(True) for k, v in m.state_dict().items()}
    opt = torch.optim.Adam(list(params.values()), lr=1e-3, betas=(0.9, 0.98))
    ids, ts, tg = (t.to(dev) for t in synth_batch(batch, L, CFG["num_items"], 123))

    def one():
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            _, loss = oh.hstu_forward(ids, ts, tg, params, CFG["num_heads"], CFG["num_blocks"])
        loss.float().backward()
        opt.step()
        return loss

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = one()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return dict(batch=batch, ms_per_step=ms, seq_per_s=batch / (ms * 1e-3), loss=float(loss))


def run_cuda_eager(args, rank, world, local_rank):
    if rank != 0:
        return
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    L = args.seq_len
    r = cuda_eager_arm(args.eager_batch, L, dev, max(1, args.steps), max(2, min(args.warmup, 3)))
    line = dict(impl="cuda_eager", metric=METRIC, value=r["seq_per_s"], unit=UNIT, n_gpus=1, steps=args.steps, warmup=args.warmup,
                ms_per_step=r["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16 autocast", data="synthetic",
                config=dict(workload=workload_name(L) + " - reference algorithm, PyTorch eager on cuda:0", batch_per_step=args.eager_batch))
    emit(line)


def workload_name(L):
    return (f"HSTU {CFG['num_blocks']} blocks d={CFG['embed_dim']} h={CFG['num_heads']} seq_len={L} V={CFG['num_items']}")


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; /root/reference does not travel
    to the GPU box), all host threads, same config/metric; rank 0 only."""
    if rank != 0:
        return
    L = args.seq_len
    r = cpu_arm(args.cpu_batch, L, seconds=0, steps=max(1, args.steps), warmup=max(1, min(args.warmup, 2)))
    cfg = dict(workload=workload_name(L) + " train step (fwd+bwd+Adam), CPU-eager fp32", batch_per_step=args.cpu_batch,
               same_config=False,
               mismatch=f"CPU arm: B={args.cpu_batch} per step, fp32, dropout 0, oracle port of the reference modules; "
                        f"GPU arm: B={args.batch} per GPU, bf16 operands, dropout {CFG['dropout']}")
    line = dict(impl="reference", metric=METRIC, value=r["seq_per_s"], unit=UNIT, n_gpus=args.gpus, steps=len(r["times"]),
                warmup=args.warmup, ms_per_step=r["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", config=cfg,
                cpu_baseline=dict(value=r["seq_per_s"], unit=UNIT, cores=r["threads"], kind="port",
                                  sample=f"{len(r['times'])} steps of B={args.cpu_batch} x L={L}"),
                e2e=dict(value=r["seq_per_s"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    emit(line)


# ------------------------------------------------------------------------------------------------ ours
def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from genrec_b200 import _lib
    from genrec_b200.hstu import HSTU
    from genrec_b200.optim import FlatAdam

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    _lib.ensure_device(dev)
    B, L, V = args.batch, args.seq_len, CFG["num_items"]
    K, W = args.steps, max(args.warmup, 3)
    torch.manual_seed(0)  # identical init on every rank (DDP broadcast equivalent)
    model = HSTU(**{**CFG, "max_seq_len": L}).to(dev).train()
    # plain loss.backward() every step: the head may accumulate straight into the flat gradient buffer (checked on the device)
    opt = FlatAdam(model, lr=1e-3, betas=(0.9, 0.98), unit_loss_grad=True, defer_weight_grads=os.environ.get("GRB_DEFER", "1") != "0")
    # --dump-outputs: the gradient reductions use float atomics, so two runs agree only to rounding after one step, and Adam amplifies
    # that difference with every further step.  The last timed step therefore starts again from the state before the first step (the
    # only training state that is bit-identical from run to run): parameters, bf16 mirror, Adam moments and step count.  Restoring
    # them adds one device copy to that step; without --dump-outputs the timed steps are unchanged.
    initial = [t.clone() for t in (opt.flat, opt.mirror, opt.m, opt.v, opt.state)] if args.dump_outputs else None

    nb = 8
    host = [tuple(t.pin_memory() for t in synth_batch(B, L, V, 1000 * rank + i)) for i in range(nb)]
    pool = [tuple(t.to(dev) for t in hb) for hb in host]
    ids_d, ts_d, tg_d = (torch.empty_like(t) for t in pool[0])
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()

    def train_step():
        _, loss = model(ids_d, ts_d, tg_d)
        loss.backward()
        opt.step()
        return loss

    def load_resident(i):
        for dst, src in zip((ids_d, ts_d, tg_d), pool[i % nb]):
            dst.copy_(src, non_blocking=True)

    def load_host(i):
        for dst, src in zip((ids_d, ts_d, tg_d), host[i % nb]):
            dst.copy_(src, non_blocking=True)

    # ---- warm-up (eager) then capture the whole step in a CUDA graph
    load_resident(0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(3):
            loss_static = train_step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    loss_static = None   # drop the eager autograd graph NOW: freeing side-stream blocks while capturing invalidates the capture
    l0 = _lib.launches()
    graph = None
    if not args.no_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                loss_static = train_step()
        except Exception as e:  # noqa: BLE001
            if rank == 0:
                print(f"[bench] CUDA graph capture failed ({type(e).__name__}: {e}); running eager", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()
    else:
        loss_static = train_step()
    launches_per_step = _lib.launches() - l0
    torch.cuda.synchronize()

    def run_step():
        nonlocal loss_static
        if graph is not None:
            graph.replay()
        else:
            loss_static = train_step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def restore_initial():
        for dst, src in zip((opt.flat, opt.mirror, opt.m, opt.v, opt.state), initial):
            dst.copy_(src)

    def timed(loader, sync_each, restart_last=False):
        for i in range(W):
            loader(i)
            run_step()
            if sync_each:
                loss_host.copy_(loss_static.detach(), non_blocking=True)
                torch.cuda.current_stream().synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        t0 = time.perf_counter()
        e0.record()
        marks[0].record()
        for i in range(K):
            if restart_last and i == K - 1:
                restore_initial()
            loader(W + i)
            run_step()
            if sync_each:
                loss_host.copy_(loss_static.detach(), non_blocking=True)
                torch.cuda.current_stream().synchronize()   # the trainer's per-step loss.item() (hstu_trainer.py:163)
            marks[i + 1].record()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        wall = (time.perf_counter() - t0) * 1e3
        per = sorted(marks[i].elapsed_time(marks[i + 1]) for i in range(K))
        pct = dict(p10=per[int(0.1 * (K - 1))], p50=per[K // 2], p90=per[int(0.9 * (K - 1) + 0.5)])
        t = torch.tensor([ms, wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t[0].item(), t[1].item(), pct

    try:
        gpu_index = int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank])
    except Exception:  # noqa: BLE001  (unset, or UUID-style entries)
        gpu_index = local_rank
    sampler = ClockSampler(gpu_index)
    if rank == 0:
        sampler.start()
    ms_dev, _, pct_dev = timed(load_resident, sync_each=False)
    clocks = sampler.stop() if rank == 0 else None
    ms_e2e, wall_e2e, pct_e2e = timed(load_host, sync_each=True, restart_last=initial is not None)
    final_loss = float(loss_static.detach().float().item())
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, loss_static, model)

    # ---- roofline of the HSTU block stack (fwd+bwd), device-timed inside a graph
    roof = None
    if rank == 0 and not args.skip_roofline:
        roof = block_roofline(model, B, L, dev, K)
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:      # reported baselines: single-GPU runs only (the other ranks would idle)
        try:
            r = cpu_arm(args.cpu_batch, L, args.cpu_seconds)
            cpu = dict(value=r["seq_per_s"], unit=UNIT, cores=r["threads"], kind="port",
                       sample=f"{len(r['times'])} train steps of B={args.cpu_batch} x L={L} (oracle port of the reference CPU-eager path, fp32)",
                       same_config=False, mismatch=f"B={args.cpu_batch} per step, fp32, dropout 0 (GPU arm: B={B}, bf16, dropout {CFG['dropout']})")
        except Exception as e:  # noqa: BLE001
            cpu = dict(value=None, unit=UNIT, cores=os.cpu_count(), kind="port", sample=f"failed: {e}")
    used_graph = graph is not None
    eager = None
    if rank == 0 and world == 1 and not args.skip_eager:
        used_graph = graph is not None
        graph = None
        torch.cuda.empty_cache()
        try:
            r = cuda_eager_arm(args.eager_batch, L, dev, steps=5 if args.config == "cfg2" else 2)
            eager = dict(value=r["seq_per_s"], unit=UNIT, ms_per_step=r["ms_per_step"], batch=r["batch"],
                         what="the reference's algorithm as PyTorch eager + autocast(bf16) on this same GPU (oracle restatement, dropout 0, Adam)")
        except Exception as e:  # noqa: BLE001
            eager = dict(value=None, unit=UNIT, what=f"failed: {type(e).__name__}: {e}")
    if world > 1:
        dist.barrier()      # rank 0 measured its extras alone: tear the process group down together
    if rank != 0:
        return
    gb = B * world
    h2d = sum(t.numel() * t.element_size() for t in host[0])
    line = dict(metric=METRIC, value=gb * K / (ms_dev * 1e-3), unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=ms_dev / K,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
                config=dict(workload=workload_name(L) + f" dropout={CFG['dropout']} full train step (emb, blocks, tied logits+CE, bwd, "
                                     f"{'all-reduce, ' if world > 1 else ''}Adam)", name=args.config,
                            global_batch=gb, batch_per_gpu=B, seq_len=L, parallelism=f"dp{world}",
                            cuda_graph=used_graph, dp_mode=opt.dp_mode,
                            l2="per-step working set (activations + logits, > 1 GB) exceeds the 126 MB L2; no explicit flush",
                            final_loss=final_loss, ms_per_step_pct=pct_dev),
                e2e=dict(value=gb * K / (ms_e2e * 1e-3), unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=4,
                         ms_per_step=ms_e2e / K, wall_ms_per_step=wall_e2e / K, ms_per_step_pct=pct_e2e),
                gpu_launches=launches_per_step * K, clocks=clocks, roofline=roof, cpu_baseline=cpu, cuda_eager_baseline=eager)
    emit(line)


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, loss, model):
    """The caller of a training step receives the loss and the updated parameters: loss.npy and param.<name>.npy, float32.
    Every parameter is written in full (36 MB at cfg3)."""
    import numpy as np
    arrays = {"loss": loss.detach()}
    arrays.update({f"param.{n}": p.detach() for n, p in model.named_parameters()})
    arrays = {k: v.float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the block stack's kernels for one fwd+bwd, from the committed ncu
# capture of the same command (profiles/*_step_dram_traffic.txt, scripts/step_traffic.py); keyed by (B, L, D, layers)
TRAFFIC_NCU = {(128, 200, 128, 4): 2.023e9,      # profiles/r2_step_cfg2_dram_traffic.txt
               (32, 2048, 256, 8): 38.780e9}     # profiles/r2_step_cfg3_dram_traffic.txt


def block_roofline(model, B, L, dev, K):
    """fwd+bwd of the HSTU block stack alone (no embedding / head / optimizer): algorithmic FLOPs (SURVEY.md section 8d:
    72 L D^2 + 6 D L (L+1) per sequence-layer) / CUDA-event time, vs the measured dense bf16 peak."""
    D, nl = CFG["embed_dim"], CFG["num_blocks"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak, which = (peaks["bf16_tflops"], "measured (burst)") if "bf16_tflops" in peaks else (1590.0, "fallback")
    ids, ts, _ = synth_batch(B, L, CFG["num_items"], 7)
    ids, ts = ids.to(dev), ts.to(dev)
    x0 = torch.randn(B, L, D, device=dev)
    dy = torch.randn(B, L, D, device=dev)
    import genrec_b200.functional as Fn
    from genrec_b200.hstu import _thresholds_on
    pad = (ids == 0).to(torch.uint8)
    meta = Fn.SeqMeta(pad, ts, model.layers[0].position_bias.bucket_of_delta(L, dev), _thresholds_on(dev), 64, 32,
                      model.layers[0].position_bias.uniform_of(L, dev))
    seed, seed_dev = model._seeds(dev)

    def fb():
        x = x0.detach().requires_grad_(True)
        y = x
        for layer in model.layers:
            y = layer(y, None, None, ts, _meta=meta, _seed=seed, _seed_dev=seed_dev)
        y.backward(dy)
        Fn.join_deferred(dev)      # the weight-gradient GEMMs belong to the stack's work: inside the timed region

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fb()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fb()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    model.zero_grad(set_to_none=False)
    flops = (72 * L * D * D + 6 * D * L * (L + 1)) * B * nl
    ach = flops / (ms * 1e-3) / 1e12
    # DRAM bytes (read + write) of the block stack's kernels for one fwd+bwd at the default geometry, summed from the ncu
    # captures profiles/r2_step_cfg{2,3}_dram_traffic.txt (scripts/step_traffic.py); not re-measured here (needs a profiler)
    traffic = TRAFFIC_NCU.get((B, L, D, nl))
    return dict(bound="tensor", kernel="hstu_block_stack_fwd_bwd", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak,
                peak_source=which, traffic=traffic, traffic_unit="bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                algorithmic_bytes_per_launch=(10 * L * D + 9 * L) * B * nl, ms_per_launch=ms, flops_per_launch=flops,
                unit_of_work=f"{nl} layers x B={B} sequences x L={L}")


_JSON_FD = None


def protect_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner at world > 1), so file descriptor 1
    is pointed at stderr for the whole run and the JSON line goes to the saved descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    args = parse()
    protect_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.impl == "cuda_eager":
        run_cuda_eager(args, rank, world, local_rank)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
