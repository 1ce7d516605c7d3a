#!/usr/bin/env python3
"""Benchmark of the NCF training hot path (BASELINE.json metric: NeuMF train samples/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]
                    [--dump-outputs DIR]

Workload at N=1: BASELINE.json configs[3] — NeuMF (factor 32, 3 tower layers: 256->128->64->32)
on the synthetic MovieLens-20M shape (138 493 users x 26 744 items, ~20M interactions, 4
negatives per positive), batch 65 536, Adam lr 1e-3.  It is the config the metric "train
samples/s @1/2/4/8 B200" is quoted on and it fits one GPU; configs[1] (ML-1M shape, batch 256) is
launch-latency-bound (SURVEY.md H3) and is a parity-test case (`--workload ml1m` runs it, and the
default line reports it under `small_config`).

A "step" is one pass of the hot path over one batch: the batch is laid out by the on-device epoch
stream (ncf_shuffle_epoch: shuffle + batching of this epoch's positives and sampled negatives), then
fused gather+forward+loss+backward (tcgen05 path at this batch size: weight images,
umma_tower_kernel, umma_wgrad_kernel), then Adam (touched rows + catch-up, or all rows when the
batch touches a large share of the tables).  Under torchrun (N>1) every rank owns a contiguous range
of the users and runs the same per-GPU batch on the samples of its own users (weak scaling; only the
item-table and tower gradients are all-reduced); the line then also carries `row_sharded`:
BASELINE configs[4] (10M x 1M tables, f=64) with the tables row-sharded and item rows exchanged by
all-to-all.  `--workload big` runs that configuration as the main workload.

The JSON line carries `value` (inputs resident in HBM), `e2e` (pinned HOST batches through the
public API — ncf_b200.trainer.HostFedTrainer on one GPU — with every step's H2D copies and loss
read-back inside the timed region), `roofline` of the dominant kernel (timed by CUDA events the
library records between its launches) with step-level / evaluation / sampler / NVLink views,
`cpu_baseline` (the reference's own NCF class from oracle/_ref — or the port in oracle/torch_port.py
when that directory is absent — on this box's host cores), `gpu_eager_reference` (the same reference
modules under torch eager on this GPU: the existing sm_100 path to beat) and the clocks sampled
during the timed region.  `--impl reference` times only the CPU reference.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (synthetic shape, factor_num, num_layers, batch)
    "ml20m": ("ml20m", 32, 3, 65536),
    "ml1m": ("ml1m", 8, 3, 256),
    "big": ("big", 64, 3, 65536),      # BASELINE configs[4]: row-sharded at N>1
}
METRIC, UNIT = "NeuMF train samples/s", "samples/s"
NVLINK_GBS = 900.0   # per direction per GPU (NVLink 5 / NVSwitch, B200_PROFILING.md)


def measured_tensor_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["bf16_tflops"])
    return 1590.0


def profile_traffic(kernel):
    """DRAM bytes per launch of the kernel from the committed `ncu --set full` capture of this
    command (profiles/traffic.json, re-measured per round), or None when no capture is on file."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        return json.loads(p.read_text()).get(kernel)
    return None


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML (a thread per rank for its own GPU, every 5 ms)
    from the start of the device-resident timed region to the end of the end-to-end one (the GPU is under
    load throughout: timed steps, per-phase passes, host-fed steps) — the same fields as the nvidia-smi
    clocks line of B200_PROFILING.md.  The polling itself costs nothing measurable, also at N=8
    (profiles/r02/clock_sampling_experiment.md: 0.361 ms/step with no thread, an idle thread, either query,
    both at 5 / 50 / 200 ms); what did cost 20 % in earlier runs was starting it (nvmlInit) between the
    barrier and the first timed step, which let the ranks enter the timed region at different times.  The
    line still carries the same loop after the samplers were stopped (`unsampled_loop`)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap"}

    def __init__(self, gpu_index, period=0.005, what="both", aligned=False):
        """`what`: "both" | "clock" | "reasons" | "idle" (the thread wakes but asks nothing); `aligned`: polls at
        multiples of the period on the machine's clock, i.e. at the same instants on every rank (experiments)."""
        self.period = float(os.environ.get("NCF_BENCH_CLOCK_PERIOD", period))
        self.what, self.aligned = what, aligned
        self.gpu, self.samples, self.mask, self.max_mhz = gpu_index, [], 0, None
        self._stop, self._thread, self._nvml = None, None, None

    def start(self):
        import threading
        if os.environ.get("NCF_BENCH_NO_CLOCKS") == "1":     # experiment knob: no NVML polling at all
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES when it lists indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                idx = int(vis.split(",")[self.gpu])
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
        except Exception:
            return
        self._stop = threading.Event()

        def loop():
            while not self._stop.is_set():
                try:
                    if self.what in ("both", "clock"):
                        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    if self.what in ("both", "reasons"):
                        self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    pass
                if self.aligned:
                    now = time.time()
                    self._stop.wait((int(now / self.period) + 1) * self.period - now)
                else:
                    self._stop.wait(self.period)

        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for bit, n in self.REASONS.items() if self.mask & bit),
                "samples": len(s)}


# ---- the reference's own implementation of the path (CPU arm, GPU-eager bar) --------------------------
class ReferenceTrainer:
    """The reference inner loop, verbatim in structure (scripts/train_neumf.py:86-90,106-118):
    `NCF(...)` + `nn.BCEWithLogitsLoss()` + `optim.Adam(model.parameters(), lr)`; per step
    zero_grad / forward / loss / backward / optimizer.step / loss.item().  The NCF class is the
    reference's own (oracle/_ref, kind "reference"); when that directory is absent the op-for-op
    port of oracle/torch_port.py (kind "port") stands in."""

    def __init__(self, U, I, f, L, device, lr=1e-3, seed=0):
        import torch
        from oracle import build_ref
        self.torch, self.device = torch, device
        ref = build_ref.load()
        torch.manual_seed(seed)
        if ref is not None:
            self.kind = "reference"
            self.model = ref.NCF(U, I, f, L, 0.0, "NeuMF-end").to(device)
            self.model.train()
            self.criterion = torch.nn.BCEWithLogitsLoss()
            self.optimizer = torch.optim.Adam(self.model.parameters(), lr=lr)
            self._port = None
        else:
            from oracle import torch_port as tp
            self.kind = "port"
            P = tp.init_params(U, I, f, L, "NeuMF-end", seed=seed)
            if device.type != "cpu":
                P = {k: v.detach().to(device).requires_grad_(True) for k, v in P.items()}
            self._port = tp.CpuTrainer(P, "NeuMF-end", lr=lr)

    def step(self, user, item, label):
        if self._port is not None:
            return self._port.step(user, item, label)
        self.model.zero_grad()
        prediction = self.model(user, item)
        loss = self.criterion(prediction, label)
        loss.backward()
        self.optimizer.step()
        return loss.item()


def reference_batches(U, I, B, n, device, seed=1):
    import torch
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        out.append((torch.randint(0, U, (B,), generator=g).to(device), torch.randint(0, I, (B,), generator=g).to(device),
                    (torch.rand(B, generator=g) < 0.2).float().to(device)))
    return out


def cpu_reference_run(workload, steps, warmup, budget_s=None):
    """Times the reference's CPU implementation of the path on this box's host cores on the same
    config: one step = one batch of the workload's size through forward, BCE, autograd backward (dense
    embedding grads) and dense Adam.  Returns (samples/s, ms/step, steps, threads, kind)."""
    import torch
    from ncf_b200.synth import SHAPES
    shape, f, L, B = WORKLOADS[workload]
    U, I, _, _ = SHAPES[shape]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    dev = torch.device("cpu")
    tr = ReferenceTrainer(U, I, f, L, dev)
    batches = reference_batches(U, I, B, 4, dev)
    for w in range(warmup):
        tr.step(*batches[w % 4])
    t0 = time.perf_counter()
    done = 0
    for k in range(steps):
        tr.step(*batches[k % 4])
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return done * B / dt, dt / done * 1e3, done, torch.get_num_threads(), tr.kind


def gpu_eager_reference_run(dev, hbm_peak):
    """The GPU bar to beat (SURVEY.md 2b/8d, BASELINE.md 3): the reference modules under torch eager
    on this B200 — configs[3] (this bench's workload, 20 steps) and configs[1] (ML-1M shape, f=8 L=3,
    batch 256, 300 steps).  Timed with CUDA events around the reference loop, `loss.item()` per step
    included as in the reference."""
    import torch
    from ncf_b200.synth import SHAPES
    out = {}
    for name, (wl, steps, warm) in {"config4_ml20m_b65536": ("ml20m", 20, 3), "config2_ml1m_b256": ("ml1m", 300, 30)}.items():
        shape, f, L, B = WORKLOADS[wl]
        U, I, _, _ = SHAPES[shape]
        tr = ReferenceTrainer(U, I, f, L, dev)
        batches = reference_batches(U, I, B, 8, dev)
        for w in range(warm):
            tr.step(*batches[w % 8])
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            tr.step(*batches[k % 8])
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        R = 2 * f + 2 * (f << (L - 1))
        out[name] = {"samples_per_s": B / (ms * 1e-3), "ms_per_step": ms, "steps": steps, "kind": tr.kind,
                     "step_level_hbm_frac": (4 * R * 7 + 24) * B / (ms * 1e-3) / 1e9 / hbm_peak}
        del tr
        torch.cuda.empty_cache()
    out["how"] = ("reference NCF + BCEWithLogitsLoss + dense optim.Adam + loss.item() per step under torch "
                  f"{torch.__version__} eager on this GPU (fp32, TF32 off = torch default)")
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    shape, f, L, B = WORKLOADS[args.workload]
    sps, ms, done, cores, kind = cpu_reference_run(args.workload, args.steps, max(1, args.warmup))
    line = {
        "impl": "reference", "metric": METRIC, "value": sps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": done, "warmup": max(1, args.warmup), "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.workload, 1),
        "cpu_baseline": {"value": sps, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{done} steps of batch {B} (uniform random indices of the workload's table "
                                   f"shape): the reference's NCF class, BCEWithLogitsLoss, autograd, dense optim.Adam "
                                   f"on torch CPU with {cores} threads"},
        "e2e": {"value": sps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def config_dict(workload, n_gpus, partitioned=True, tail=False):
    shape, f, L, B = WORKLOADS[workload]
    from ncf_b200.synth import SHAPES
    U, I, total, _ = SHAPES[shape]
    if workload == "big" and n_gpus > 1:
        par = f"row-sharded tables x{n_gpus} (item rows by all-to-all)"
    elif n_gpus == 1:
        par = "dp1"
    elif partitioned:
        par = (f"dp{n_gpus}: every rank owns 1/{n_gpus} of the users and trains on their samples; item tables + "
               f"tower replicated, " + ("reduced, stepped and broadcast by one kernel over peer memory (ncf_adam_p2p)"
                                        if tail else "their gradients all-reduced (NCCL)"))
    else:
        par = f"dp{n_gpus}: fully replicated tables, gradient all-reduce" + (
            " (exchange inside the Adam kernel over peer memory)" if os.environ.get("NCF_DP_P2P") == "1" else "")
    return {"workload": f"NeuMF f={f} L={L} (tower {f << L}->{f}) on synthetic {shape} shape "
                        f"({U} users x {I} items, ~{total} interactions, 4 neg/pos), batch {B} per GPU, Adam lr 1e-3",
            "batch_per_gpu": B, "global_batch": B * n_gpus, "parallelism": par,
            "l2": "state touched per step (tables + Adam moments + gradient buffers, ~400 MB at ml20m) "
                  "exceeds the 126 MB L2 and every step uses a different batch; no explicit flush"}


DUMP_ROWS = 16384       # embedding rows written per table by --dump-outputs (a fixed, seeded sample)


def dump_outputs(out_dir, ts, loss_before, user, item, label):
    """--dump-outputs: what the timed steps hand to their caller after the last one, as DIR/<name>.npy, so that
    two builds can be compared output for output (the inputs are seeded: same arguments, same inputs).
      loss                    float64 [1]  the loss the caller pops: the per-batch mean losses of the timed steps, summed
      <state_dict key>        float32      the parameters after the last step, flushed (every row at the Adam state of
                                           that step); of each embedding table the rows listed in rows_user / rows_item
      rows_user, rows_item    float64      the sampled row ids (DUMP_ROWS per table, seed 0, ascending)
      batch_user, batch_item  float64      the batch the last step trained on, as the epoch stream laid it out
      batch_label             float32
    Two runs of one build agree bit for bit on the batch and to ~2e-6 relative on the loss, but their parameters
    only to a median of 1e-6 .. 1e-4 of each array's largest magnitude (B200, default workload, 125 steps in all):
    the tcgen05 weight-gradient kernel sums in a run-dependent order and Adam amplifies gradients near zero.
    Compare builds with bounds of that kind (share of elements beyond a tolerance), not element by element."""
    import numpy as np
    import torch
    ts.flush()
    model = ts.model
    rng = np.random.default_rng(0)
    rows = {}
    for side, n in (("user", model.user_num), ("item", model.item_num)):
        rows[side] = np.sort(rng.choice(n, size=min(n, DUMP_ROWS), replace=False))
    arrays = {"loss": (ts.loss_accum - loss_before).cpu().numpy(),
              "rows_user": rows["user"].astype(np.float64), "rows_item": rows["item"].astype(np.float64),
              "batch_user": user.cpu().numpy().astype(np.float64), "batch_item": item.cpu().numpy().astype(np.float64),
              "batch_label": label.cpu().numpy().astype(np.float32)}
    for k, v in model.state_dict().items():
        side = "user" if k.startswith("embed_user") else "item" if k.startswith("embed_item") else None
        if side is not None:
            v = v[torch.from_numpy(rows[side]).to(v.device)]
        arrays[k] = v.detach().float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs would write {total} bytes"
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out / f"{k}.npy", a)


# ------------------------------------------------------------------------------------------------
def row_sharded_run(dev, world, rank, steps, warmup, tower_math, hbm_peak, dump_dir=None):
    """BASELINE configs[4]: NeuMF f=64 L=3 on 10M users x 1M items with the four tables (and their Adam
    state) row-sharded over the ranks; every rank draws `B` samples of its own users per step and item
    rows travel by all-to-all (ncf_b200.dist.RowShardedTrainer).  At N=1 the tables live on the one GPU
    and the step is the plain fused step (the weak-scaling base point)."""
    import torch
    import torch.distributed as dist
    from ncf_b200.dist import RowShardedTrainer, shard_rows
    from ncf_b200.models import NCF
    from ncf_b200.synth import SHAPES
    from ncf_b200.trainer import FusedTrainStep
    shape, f, L, B = WORKLOADS["big"]
    U, I = SHAPES["big"][0], SHAPES["big"][1]
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    Ul, Il = shard_rows(U, world, rank), shard_rows(I, world, rank)
    torch.manual_seed(0)
    with torch.device(dev):
        model = NCF(Ul, Il, f, L, 0.0, "NeuMF-end")
    model.tower_math = tower_math
    need = (warmup + steps) * B
    bu = torch.randint(0, Ul, (need,), device=dev, generator=g) * world + rank
    zipf = torch.rand(need, device=dev, generator=g).pow(3.0)                      # popularity skew
    bi = (zipf * I).long().clamp_(0, I - 1)
    bl = (torch.rand(need, device=dev, generator=g) < 0.2).float()
    if world > 1:
        tr = RowShardedTrainer(model, U, I, lr=1e-3, max_batch=B)
        step = tr.step
    else:
        tr = FusedTrainStep(model, "adam", 1e-3, max_batch=B)
        step = tr.step
    sl = lambda k: slice(k * B, (k + 1) * B)
    for k in range(warmup):
        step(bu[sl(k)], bi[sl(k)], bl[sl(k)])
    loss_before = tr.loss_accum.clone() if dump_dir else None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(warmup, warmup + steps):
        step(bu[sl(k)], bi[sl(k)], bl[sl(k)])
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dump_dir:
        last = sl(warmup + steps - 1)
        dump_outputs(dump_dir, tr, loss_before, bu[last], bi[last], bl[last])
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * steps * B / (ms * 1e-3)
    d = f << (L - 1)
    R = 2 * f + 2 * d
    res = {"metric": METRIC, "value": value, "unit": UNIT, "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
           "n_gpus": world, "scaling": "weak",
           "config": config_dict("big", world),
           "resident_gb_per_gpu": torch.cuda.max_memory_allocated(dev) / 1e9,
           "hbm": {"bytes_per_sample": 4 * R * 7 + 24, "achieved_gbs_per_gpu": (4 * R * 7 + 24) * value / world / 1e9,
                   "frac": (4 * R * 7 + 24) * value / world / 1e9 / hbm_peak}}
    if world > 1:
        stats = tr.wire_stats()
        out_bytes = stats["bytes_out_per_step"]
        res["nvlink"] = {"bytes_out_per_gpu_per_step": out_bytes, "peak_gbs_per_direction": NVLINK_GBS,
                         "achieved_gbs": out_bytes / (ms / steps * 1e-3) / 1e9,
                         "frac": out_bytes / (ms / steps * 1e-3) / 1e9 / NVLINK_GBS, **stats}
    del tr, model, bu, bi, bl
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from ncf_b200 import ops
    from ncf_b200.models import NCF
    from ncf_b200.synth import make_interactions
    from ncf_b200.trainer import EpochStream, FusedTrainStep

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the ncf_b200 hot path has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    hbm_peak, peak_src = measured_peaks()
    K, W = args.steps, max(4, args.warmup)     # >= 4: two eager steps, then each of the two step graphs replayed once

    if args.workload == "big":
        res = row_sharded_run(dev, world, rank, K, W, args.tower_math, hbm_peak, args.dump_outputs)
        if rank == 0:
            line = {**res, "higher_is_better": True, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "e2e": None, "gpu_launches": (17 if world > 1 else 8) * K, "roofline": None, "cpu_baseline": None}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    st = main_workload(args, dev, world, rank, local, hbm_peak, peak_src, K, W)
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    row_sharded = None
    if args.workload == "ml20m" and not args.no_row_sharded:
        row_sharded = row_sharded_run(dev, world, rank, steps=10, warmup=3, tower_math=args.tower_math,
                                      hbm_peak=hbm_peak)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    B = WORKLOADS[args.workload][3]
    extras = world == 1 and args.workload == "ml20m" and not args.no_extras
    # ---- CPU baseline: bounded sample on this box's host cores (rank 0, N=1 only) ---------------------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        sps, ms, done, cores, kind = cpu_reference_run(args.workload, steps=40, warmup=1, budget_s=15.0)
        cpu_baseline = {"value": sps, "unit": UNIT, "cores": cores, "kind": kind,
                        "sample": f"{done} steps of batch {B} ({ms:.0f} ms/step) of the same config: the reference's "
                                  f"NCF class + BCEWithLogitsLoss + autograd (dense embedding grads) + dense optim.Adam "
                                  f"on torch CPU, {cores} threads"}
    roofline = st["roofline"]
    sampler = sampler_run(dev, hbm_peak) if extras else None
    if roofline is not None and sampler is not None:
        roofline["sampler"] = sampler["roofline"]
    line = {
        "metric": METRIC, "value": st["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": st["ms_total"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_dict(args.workload, world, st["dp_partitioned"], st["dp_tail"]),
        "e2e": {"value": st["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": B * 20, "d2h_bytes_per_step": 8,
                "ms_per_step": st["e2e_ms"] / K,
                "launch": st["e2e_launch"],
                "note": "value's timer is CUDA events on the stream, e2e's is the host clock around the same number of "
                        "steps; the two agree within run-to-run noise when the copies are hidden"},
        # our kernels inside the timed region: per step everything but the shuffle, which lays out a whole window
        "gpu_launches": (st["launches_per_step"] - 1) * K + K // st["window"],
        "launch": (f"CUDA-graph windows of {st['window']} steps (one shuffle launch + one graph launch per window, as "
                   f"ncf_b200.trainer.train_epoch runs an epoch)" if st["window"] > 1 else
                   "one shuffle launch + one CUDA-graph launch per step"),
        "clocks": st["clocks"],
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "eval": st["eval_info"],
        "sampler": sampler,
        "small_config": small_config_run(dev) if extras else None,
        "kd_config": kd_config_run(dev) if extras else None,
        "gpu_eager_reference": gpu_eager_reference_run(dev, hbm_peak) if extras else None,
        "unsampled_loop": st["unsampled"],
        "row_sharded": row_sharded,
        "tower_math": args.tower_math,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main_workload(args, dev, world, rank, local, hbm_peak, peak_src, K, W):
    """The ml20m / ml1m workload: device-resident timing, per-phase timing, end-to-end timing and
    evaluation.  Returns plain numbers only, so that every tensor is released when it returns."""
    import torch
    import torch.distributed as dist

    from ncf_b200 import ops
    from ncf_b200.models import NCF
    from ncf_b200.synth import make_interactions
    from ncf_b200.trainer import EpochStream, FusedTrainStep

    import gc
    gc.disable()      # no collector pauses inside the host-clocked regions (re-enabled by the caller's return)
    shape, f, L, B = WORKLOADS[args.workload]
    inter = make_interactions(shape, device=dev)
    U, I = inter.user_num, inter.item_num
    torch.manual_seed(0)
    model = NCF(U, I, f, L, 0.0, "NeuMF-end").to(dev)
    model.tower_math = args.tower_math
    ts = FusedTrainStep(model, "adam", 1e-3, max_batch=B)
    dp = None
    pos_user, pos_item, p_off = inter.pos_user, inter.pos_item, 0
    if world > 1:
        from ncf_b200.dist import ReplicatedDataParallel
        dp = ReplicatedDataParallel(ts)
        if dp.partition_users:
            # the rank's own users: the synthetic positives are sorted by user, so they are one slice
            p_lo = int(torch.searchsorted(pos_user, torch.tensor(dp.user_lo, device=dev)))
            p_hi = int(torch.searchsorted(pos_user, torch.tensor(dp.user_hi, device=dev)))
            pos_user, pos_item, p_off = pos_user[p_lo:p_hi].contiguous(), pos_item[p_lo:p_hi].contiguous(), p_lo
    # the epoch stream of this rank: negatives for its positives, shuffled, laid out window by window
    stream = EpochStream(pos_user, pos_item, U, I, num_ng=4, seed=20250605, p_offset=p_off)
    stream.begin_epoch(0)
    # the timed steps run as CUDA-graph windows of G steps, the scheme ncf_b200.trainer.train_epoch uses (one
    # shuffle launch lays out the G batches of a window, one graph launch runs its G steps): G = the largest
    # divisor of K up to 64 whose two warm-up windows still fit into this rank's epoch stream;
    # NCF_BENCH_WINDOW=1 = one shuffle + one graph launch per step
    own_stream = dp is None or dp.partition_users          # else: the ranks take consecutive slices of one stream
    avail = stream.S // B // (1 if own_stream else world)  # steps this rank can draw from the epoch
    if world > 1:                                          # every rank must capture the same windows
        t_av = torch.tensor([avail], dtype=torch.int64, device=dev)
        dist.all_reduce(t_av, op=dist.ReduceOp.MIN)
        avail = int(t_av.item())
    want = int(os.environ.get("NCF_BENCH_WINDOW", "0"))
    G = 1
    if not args.no_graph:
        for g in range(min(64, K), 0, -1):
            if K % g == 0 and (want in (0, g)) and W + K + (2 * g if g > 1 else 0) <= avail:
                G = g
                break
    n_batches = W + K + (2 * G if G > 1 else 0)     # + one warm-up replay of each of the two window graphs
    need = n_batches * B
    q0 = 0 if own_stream else rank * need
    if q0 + need > stream.S:
        raise SystemExit(f"workload too small for {n_batches} steps of {B} on {world} ranks")
    # two rotating device batches: step k reads buffer k%2 while nothing else touches it
    bufs = [(torch.empty(B, dtype=torch.int64, device=dev), torch.empty(B, dtype=torch.int64, device=dev),
             torch.empty(B, dtype=torch.float32, device=dev)) for _ in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    step_fn = ts.step if dp is None else dp.step
    graphs = [None, None]

    def one_step(k):
        u, i, y = bufs[k & 1]
        stream.fill(q0 + k * B, B, u, i, y)          # shuffle + batching of the reference DataLoader, on the device
        if graphs[k & 1] is not None:
            graphs[k & 1].replay()                   # the step over this buffer as one CUDA-graph launch
        else:
            step_fn(u, i, y)

    # ---- device-resident timing ------------------------------------------------------------------
    # the first warm-up steps run eagerly (they load every kernel), then the step over each of the two
    # batch buffers is captured once (at N>1 with its exchange) and replayed; with G > 1 the timed region
    # then runs windows of G steps (two window buffers, one graph each, each replayed once as warm-up)
    use_step_graph = not args.no_graph and (dp is None or (dp.partition_users and os.environ.get("NCF_DP_GRAPH", "1") != "0"))
    use_e2e_graph = use_step_graph
    if dp is not None and os.environ.get("NCF_BENCH_STEP_GRAPH", "1") == "0":
        use_step_graph = False      # experiment knob: eager launches in the device-resident loop at N>1
    for k in range(W):
        one_step(k)
        if k == 1 and use_step_graph:
            barrier()
            graphs = [ts.capture(*bufs[j], B, step_fn if dp is not None else None) for j in range(2)]
    wgraphs = None
    if G > 1 and use_step_graph:
        wbufs = [(torch.empty(G * B, dtype=torch.int64, device=dev), torch.empty(G * B, dtype=torch.int64, device=dev),
                  torch.empty(G * B, dtype=torch.float32, device=dev)) for _ in range(2)]
        for wb in wbufs:
            stream.fill(q0, G * B, *wb)      # valid ids for the capture pass
        barrier()
        wgraphs = [ts.capture(*wbufs[j], B, step_fn if dp is not None else None) for j in range(2)]

    def run_window(kw, first_step):
        """Steps [first_step + kw*G, first_step + (kw+1)*G): one shuffle launch + one graph launch."""
        u, i, y = wbufs[kw & 1]
        stream.fill(q0 + (first_step + kw * G) * B, G * B, u, i, y)
        wgraphs[kw & 1].replay()

    if wgraphs is not None:
        run_window(0, W)
        run_window(1, W)
    T0 = W + (2 * G if wgraphs is not None else 0)     # first timed step
    loss_before = ts.loss_accum.clone() if args.dump_outputs else None
    sampler = ClockSampler(local)
    sampler.start()     # BEFORE the barrier: nvmlInit takes a different time on every rank, and a rank that enters the
    barrier()           # timed region late is waited for by all the others at the first exchange of the window
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # At N>1 the loop waits for the device every 4th step, as a loop that reads its loss every few steps does: with
    # all eight ranks running ahead unsynchronised the steps were measured 8 % slower (0.543 vs 0.497 ms at N=8; at
    # N=2 graph replays cost the same either way: 0.394 vs 0.400 ms - profiles/r02/dp_loop_modes.md)
    sync_every = int(os.environ.get("NCF_BENCH_SYNC_EVERY", "4" if world > 1 else "0"))
    def timed_steps():
        if wgraphs is not None:
            for kw in range(K // G):
                run_window(kw, T0)
            return
        for k in range(W, W + K):
            one_step(k)
            if sync_every and (k - W + 1) % sync_every == 0:
                torch.cuda.current_stream().synchronize()

    e0.record()
    timed_steps()
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs:
        if wgraphs is not None:     # the last window's buffers; its last B samples are the last step's batch
            last = [t[(G - 1) * B:] for t in wbufs[(K // G - 1) & 1]]
        else:
            last = bufs[(W + K - 1) & 1]
        dump_outputs(args.dump_outputs, ts, loss_before, *last)
    value = world * K * B / (ms_total * 1e-3)
    dense = ts.dense_adam(B * world)
    umma = B >= 8192 and f >= 32
    # kernels per step (replayed from a CUDA graph or launched one by one, the same kernels):
    # shuffle_epoch + [prepare] + (images, tower, wgrad | split, tile) + (flat, stamp | rows); the tower's Adam
    # update and the step counter are folded into the last of them
    launches_per_step = 1 + (0 if dense else 1) + (3 if umma else 2) + (2 if dense else 1)
    if dp is not None and not dp.partition_users and dp.sharded is not None:
        launches_per_step = 1 + 3 + 2       # images, tower, wgrad, adam_range (or adam_p2p), stamp
    if dp is not None and dp.tail is not None:
        launches_per_step = 1 + 3 + 1 + 2   # shuffle, images, tower, wgrad, adam_p2p, adam_flat (users), stamp
        if getattr(dp.tail["barrier"], "__self__", None).__class__.__name__ == "PeerBarrier":
            launches_per_step += 2          # the two peer-memory rank barriers around adam_p2p

    # materialise the timed batches once more for the per-phase and end-to-end passes
    bu = torch.empty(need, dtype=torch.int64, device=dev)
    bi = torch.empty(need, dtype=torch.int64, device=dev)
    bl = torch.empty(need, dtype=torch.float32, device=dev)
    stream.fill(q0, need, bu, bi, bl)
    sl = lambda k: slice(k * B, (k + 1) * B)

    # ---- per-phase timing of the local work of the same steps (events between the phases) ---------------
    import ctypes as C
    from ncf_b200 import _lib
    lib = _lib.load()
    names = ["shuffle_epoch", "adam_prepare", "train_step_grads", "adam_step"]
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(K)]
    u_lo, u_hi = (dp.user_lo, dp.user_hi) if (dp is not None and dp.partition_users) else (0, U)
    B_norm = B * world if (dp is not None and dp.partition_users) else B
    if dp is not None and dp.sharded is not None:
        phases, kernel_ms, tile_path = None, {}, "tcgen05" if umma else "mma.sync"
    else:
        def phase_prepare(u, i):
            if not dense:
                ops.adam_prepare(ts._m, ts._g, ts._s, u, i, ts.lr)

        def phase_grads(u, i, y):
            ops.train_step_grads_norm(ts._m, ts._g, u, i, y, B_norm, ts.loss_accum, ts.workspace)

        tail = dp.tail if dp is not None else None

        def phase_adam():
            if dense:   # with the peer-memory tail the local part of the optimiser is the user tables only
                ops.adam_step_dense_range(ts._m, ts._g, ts._s, u_lo, u_hi, ts.lr,
                                          parts=ops.PART_USERS if tail is not None else 7)
                if tail is not None:
                    tail["g"].zero_()
            else:
                ops.adam_step(ts._m, ts._g, ts._s, ts.lr)

        ts.flush()
        barrier()
        for k in range(K):
            u, i, y = bufs[k & 1]
            ev[k][0].record()
            stream.fill(q0 + (W + k) * B, B, u, i, y)
            ev[k][1].record()
            phase_prepare(u, i)
            ev[k][2].record()
            phase_grads(u, i, y)
            ev[k][3].record()
            phase_adam()
            ev[k][4].record()
        torch.cuda.synchronize()
        phases = {n: sum(ev[k][j].elapsed_time(ev[k][j + 1]) for k in range(K)) / K for j, n in enumerate(names)}
        # per-kernel times inside ncf_train_step_grads (CUDA events recorded by the library between its
        # launches; profiling mode synchronises after each step, so it is outside the timed region)
        kernel_ms = {}
        lib.ncf_profile_enable(1)
        for k in range(K):
            u, i, y = bu[sl(W + k)], bi[sl(W + k)], bl[sl(W + k)]
            phase_prepare(u, i)
            phase_grads(u, i, y)
            phase_adam()
            ms = (C.c_float * 16)()
            nm = C.create_string_buffer(16 * 32)
            n = lib.ncf_profile_read(ms, nm, 16, 32)
            for j in range(n):
                key = nm.raw[j * 32:(j + 1) * 32].split(b"\0")[0].decode()
                kernel_ms[key] = kernel_ms.get(key, 0.0) + ms[j] / K
        lib.ncf_profile_enable(0)
        tile_path = {0: "none", 1: "generic", 2: "mma.sync", 3: "tcgen05"}[lib.ncf_last_tile_path()]
    # the data-parallel step in place (N>1): wall time between CUDA events around the real dp.step calls, next to the
    # sum of the local phases above -> what the collective and the wait for the slowest rank add
    dp_in_place = None
    if dp is not None:
        barrier()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tms = []
        for k in range(K):
            u, i, y = bufs[k & 1]
            stream.fill(q0 + (W + k) * B, B, u, i, y)
            d0.record()
            dp.step(u, i, y)
            d1.record()
            torch.cuda.synchronize()           # every step starts with all ranks idle: no run-ahead skew
            tms.append(d0.elapsed_time(d1))
        dp_in_place = {"dp_step_ms_synchronised": max_over_ranks(sorted(tms)[len(tms) // 2]),
                       "overlap": dp.comm_stream is not None,
                       "note": "median over steps of one dp.step between CUDA events with a host sync after every step"}
    # the step's exchange alone (N>1): the replicated gradient tail [item GMF | item MLP | tower]
    nvlink = None
    if dp is not None and dp.tail is not None:
        # reduce + Adam + broadcast of the tail in one kernel over peer memory, between its two rank barriers
        tl = dp.tail
        m0, v0 = tl["m"].clone(), tl["v"].clone()
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(10):
            tl["barrier"]()
            ops.adam_p2p(tl["gptrs"], tl["pptrs"], tl["m"], tl["v"], tl["lo"], rank, ts.state.step, 0.0, grad_scale=1.0)
            tl["barrier"]()
        c1.record()
        barrier()
        tl["m"].copy_(m0); tl["v"].copy_(v0)           # lr = 0 left the parameters alone; restore the moments
        ex_ms = max_over_ranks(c0.elapsed_time(c1) / 10)
        per_bytes = tl["per"] * 4
        wire = (world - 1) * per_bytes                  # gradient slices read from the peers = parameter slices written to them
        nvlink = {"exchange": "ncf_adam_p2p: reduce + Adam + broadcast of [item GMF | item MLP | tower] over peer memory, "
                              "between two rank barriers (ncf_peer_barrier)",
                  "buffer_bytes": tl["g"].numel() * 4, "ms": ex_ms, "bytes_in_per_gpu": wire, "bytes_out_per_gpu": wire,
                  "achieved_gbs": wire / (ex_ms * 1e-3) / 1e9, "peak_gbs_per_direction": NVLINK_GBS,
                  "frac": wire / (ex_ms * 1e-3) / 1e9 / NVLINK_GBS, "share_of_step": ex_ms / (ms_total / K)}
    elif dp is not None:
        buf = ts.grads.flat[dp.n_user_flat:] if dp.partition_users else ts.grads.flat
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(10):
            dist.all_reduce(buf, op=dist.ReduceOp.SUM)
        c1.record()
        barrier()
        buf.zero_()
        ar_ms = max_over_ranks(c0.elapsed_time(c1) / 10)
        wire = 2.0 * (world - 1) / world * buf.numel() * 4          # bytes out (= in) per GPU of a ring / NVLS all-reduce
        nvlink = {"collective": "all_reduce(sum) of " + ("[item GMF | item MLP | tower] gradients"
                                                           if dp.partition_users else "the whole flat gradient buffer"),
                  "buffer_bytes": buf.numel() * 4, "ms": ar_ms, "bytes_out_per_gpu": wire,
                  "achieved_gbs": wire / (ar_ms * 1e-3) / 1e9, "peak_gbs_per_direction": NVLINK_GBS,
                  "frac": wire / (ar_ms * 1e-3) / 1e9 / NVLINK_GBS, "share_of_step": ar_ms / (ms_total / K)}

    # ---- end to end: host buffers, H2D + D2H inside the timed region -----------------------------------
    hu = bu.cpu().pin_memory(); hi = bi.cpu().pin_memory(); hl = bl.cpu().pin_memory()
    du = torch.empty(B, dtype=torch.int64, device=dev)
    di = torch.empty(B, dtype=torch.int64, device=dev)
    dl = torch.empty(B, dtype=torch.float32, device=dev)
    host_loss = torch.zeros(1, dtype=torch.float64).pin_memory()

    # ncf_b200.trainer.HostFedTrainer — the step over static device buffers is a CUDA graph (at N>1 with
    # the step's NCCL all-reduce captured in it) and the next batch's H2D copies run on a copy stream while
    # the current step computes; every step still copies its own inputs from pinned host memory and reads
    # its loss back.
    hf = None
    if use_e2e_graph:
        from ncf_b200.trainer import HostFedTrainer
        for k in range(2):  # every kernel loaded before capture
            du.copy_(hu[sl(k)]); di.copy_(hi[sl(k)]); dl.copy_(hl[sl(k)])
            step_fn(du, di, dl)
        barrier()
        # at N>1 the exchange is captured too.  8 buffer sets on one GPU: the host may fall 3 ms behind before the
        # GPU idles; at N>1 the two sets the multi-GPU runs of this round were measured with
        hf = HostFedTrainer(ts, B, step_fn if dp is not None else None, depth=8 if dp is None else 2)
        nb = W + K
        hf.prefetch(hu[sl(0)], hi[sl(0)], hl[sl(0)])

    def e2e_step(k):
        if hf is not None:
            hf.launch()
            j = (k + 1) % nb
            hf.prefetch(hu[sl(j)], hi[sl(j)], hl[sl(j)])   # overlaps with the step just launched
            # the reference reads loss.item() every step: so do we, up to depth-1 steps behind, so that the GPU has
            # the next steps queued while the host reads an older loss (the last ones are read before the clock stops)
            return hf.wait() if hf.in_flight == hf.depth else None
        du.copy_(hu[sl(k)], non_blocking=True)
        di.copy_(hi[sl(k)], non_blocking=True)
        dl.copy_(hl[sl(k)], non_blocking=True)
        if dp is None:
            ts.step(du, di, dl)
        else:
            dp.step(du, di, dl)
        host_loss.copy_(ts.loss_accum, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the reference reads loss.item() every step
        return float(host_loss[0])

    for k in range(W):
        e2e_step(k)
    barrier()
    t0 = time.perf_counter()
    for k in range(W, W + K):
        e2e_step(k)
    if hf is not None:
        while hf.in_flight:
            hf.wait()
    barrier()
    clocks = sampler.stop()     # sampled from the start of the device-resident region to the end of the end-to-end one
    if world > 1:               # every rank watched its own GPU: keep the slowest one in view as well
        allc = [None] * world
        dist.all_gather_object(allc, clocks)
        mhz = [c["sm_mhz"] for c in allc if c["sm_mhz"] is not None]
        clocks["all_ranks"] = {"sm_mhz_min_of_medians": min(mhz) if mhz else None,
                               "sm_mhz_per_rank": [c["sm_mhz"] for c in allc],
                               "reasons": sorted({r for c in allc for r in c["reasons"]})}
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e_value = world * K * B / (e2e_ms * 1e-3)
    used_graph = hf is not None
    del hf
    # the device-resident loop once more with no NVML polling anywhere in the job (N>1 only; see ClockSampler)
    unsampled = None
    if dp is not None:
        for k in range(2):
            one_step(k)
        barrier()
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record()
        timed_steps()
        u1.record()
        barrier()
        ums = max_over_ranks(u0.elapsed_time(u1))
        unsampled = {"value": world * K * B / (ums * 1e-3), "ms_per_step": ums / K,
                     "note": "the timed loop repeated after the clock samplers were stopped"}

    if dp is not None and os.environ.get("NCF_BENCH_CLOCK_EXPERIMENT") == "1":
        # what exactly about the clock sampling slows the coupled ranks down: printed to stderr, not part of the line
        out = {}
        for name, kw in (("none", None), ("idle_thread_5ms", dict(what="idle")), ("clock_only_5ms", dict(what="clock")),
                         ("reasons_only_5ms", dict(what="reasons")), ("both_5ms", dict()),
                         ("both_5ms_aligned", dict(aligned=True)), ("both_50ms", dict(period=0.05)),
                         ("both_200ms", dict(period=0.2)), ("none_again", None)):
            smp = ClockSampler(local, **kw) if kw is not None else None
            barrier()
            if smp is not None:
                smp.start()
            time.sleep(0.3)
            barrier()
            best = None
            for rep in range(3):
                x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                barrier()
                x0.record()
                timed_steps()
                x1.record()
                barrier()
                ms = max_over_ranks(x0.elapsed_time(x1)) / K
                best = ms if best is None else min(best, ms)
            got = smp.stop() if smp is not None else None
            out[name] = {"ms_per_step_best_of_3": best, "samples": got["samples"] if got else 0}
        if rank == 0:
            print("CLOCK_EXPERIMENT " + json.dumps(out), file=sys.stderr, flush=True)

    # ---- evaluation throughput (second half of the metric: eval users/s): every rank scores its own users ----
    from ncf_b200.metrics import evaluate
    ts.flush()
    model.eval()
    tu, tc = inter.test_users, inter.test_cands
    if dp is not None and dp.partition_users:
        keep = (tu >= dp.user_lo) & (tu < dp.user_hi)
        tu, tc = tu[keep].contiguous(), tc[keep].contiguous()
    elif dp is not None:
        lo = rank * (tu.numel() // world)
        hi_ = tu.numel() if rank == world - 1 else lo + tu.numel() // world
        tu, tc = tu[lo:hi_].contiguous(), tc[lo:hi_].contiguous()
    with torch.no_grad():
        evaluate(model, tu, tc, 10)
        barrier()
        times = []
        for _ in range(5):   # median of 5: an occasional 2x outlier was seen on this pool
            ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ee0.record()
            res = evaluate(model, tu, tc, 10)
            ee1.record()
            barrier()
            times.append(max_over_ranks(ee0.elapsed_time(ee1)))
    ev_ms = sorted(times)[len(times) // 2]
    n_users = int(inter.test_users.numel())
    d = f << (L - 1)
    eval_bytes_user = 4 * (f + d) * 101 + 808          # SURVEY.md 8d: user row once + 100 candidate rows + indices
    eval_info = {"users_per_s": n_users / (ev_ms * 1e-3), "ms": ev_ms, "users": n_users, "candidates": 100,
                 "hr10_rank0": float(res.hit.float().mean().item()),
                 "roofline": {"bound": "hbm", "bytes_per_user": eval_bytes_user,
                              "achieved_gbs_per_gpu": eval_bytes_user * n_users / world / (ev_ms * 1e-3) / 1e9,
                              "peak": hbm_peak, "frac": eval_bytes_user * n_users / world / (ev_ms * 1e-3) / 1e9 / hbm_peak}}

    # ---- roofline of the dominant kernel (rank 0's local work) --------------------------------------------
    tensor_peak = measured_tensor_peak()
    R = 2 * f + 2 * d
    macs = sum((f << (L - k)) * (f << (L - k - 1)) for k in range(L)) + 2 * f   # tower + predict, per sample
    roofline = None
    if rank == 0 and phases is not None:
        dom = max(phases, key=phases.get)
        nu = len(torch.unique(bufs[0][0])); ni = len(torch.unique(bufs[0][1]))
        # algorithmic bytes per launch (SURVEY.md 8d; DESIGN.md section 3)
        adam_rows = ((u_hi - u_lo) + I) if dense else (nu + ni)
        alg_bytes = {
            "shuffle_epoch": 20 * B + 24 * B,                  # batch out (2 x int64 + f32) + sources in
            "train_step_grads": (4 * R + 24) * B,              # row gather + indices + label/logit
            "adam_step": 8 * 4 * (f + d) * adam_rows,          # g, p, m, v read + p, m, v, 0 written
            "adam_prepare": 0 if dense else 16 * B + 6 * 4 * (f + d) * (nu + ni),
        }
        hbm = {n: {"algorithmic_bytes": alg_bytes[n], "ms": phases[n],
                   "achieved_gbs": alg_bytes[n] / max(phases[n], 1e-9) / 1e6,
                   "frac": alg_bytes[n] / max(phases[n], 1e-9) / 1e6 / hbm_peak} for n in phases}
        if dom == "train_step_grads" and "tower" in kernel_ms:
            # tcgen05 path: ncf_train_step_grads = weight images + umma_tower_kernel (forward and
            # backward-data of the tower, fused with gather / loss / scatter) + umma_wgrad_kernel.
            # The dominant kernel is the tower kernel: algorithmic FLOPs = 4 * MACs per sample.
            flops = 4.0 * macs * B
            achieved = flops / (kernel_ms["tower"] * 1e-3) / 1e12
            t_ms = kernel_ms["tower"]
            kbytes = (4 * R + 24) * B + 4 * R * B          # SURVEY 8d share of this kernel: gather + indices + row-gradient REDs
            lb_hbm = kbytes / (hbm_peak * 1e9) * 1e3        # ms lower bounds of one launch
            lb_tensor = flops / (tensor_peak * 1e12) * 1e3
            lb_3xtf32 = flops / (tensor_peak / 6.0 * 1e12) * 1e3
            tensor_view = {"achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved / tensor_peak,
                           "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst). The kernel computes in fp32-parity "
                                          "3xTF32 on tcgen05 (kind::tf32 runs at half the bf16 rate and every "
                                          "algorithmic MAC costs 3 MMAs), so its own ceiling is peak / 6",
                           "frac_of_3xtf32_ceiling": achieved / (tensor_peak / 6.0),
                           "algorithmic_flops_per_launch": flops}
            # which roof binds: with the contract's peaks (HBM copy bandwidth, dense bf16 rate) the kernel's algorithmic
            # bytes take longer than its algorithmic flops, so the headline object is the HBM one; the tensor view
            # (and the 3xTF32 ceiling, under which the two roofs nearly meet) rides along
            roofline = {"bound": "hbm", "kernel": "umma_tower_kernel (inside ncf_train_step_grads)",
                        "achieved": kbytes / (t_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": kbytes / (t_ms * 1e-3) / 1e9 / hbm_peak, "traffic": profile_traffic("umma_tower_kernel"),
                        "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": kbytes,
                        "algorithmic_bytes_note": "(4R + 24) B gathered rows + indices + 4R B row-gradient REDs, R = 2f + 2d "
                                                  "(SURVEY 8d per-sample figure, this kernel's share); the activation / delta "
                                                  "scratch it also writes for the weight-gradient kernel is not counted",
                        "launch_ms": t_ms,
                        "bound_analysis": {"lower_bound_ms_hbm": lb_hbm, "lower_bound_ms_tensor_bf16_peak": lb_tensor,
                                           "lower_bound_ms_tensor_3xtf32": lb_3xtf32,
                                           "note": "binding roof under MEASURED_PEAKS = HBM; counting the three TF32 "
                                                   "products per MAC at the tf32 rate the tensor roof is the higher one"},
                        "tensor_view": tensor_view,
                        "frac_of_3xtf32_ceiling": achieved / (tensor_peak / 6.0),
                        "kernel_ms": kernel_ms,
                        "wgrad": {"kernel": "umma_wgrad_kernel", "launch_ms": kernel_ms.get("wgrad"),
                                  "achieved_tflops": 2.0 * macs * B / (kernel_ms["wgrad"] * 1e-3) / 1e12,
                                  "traffic": profile_traffic("umma_wgrad_kernel")}}
        elif dom == "train_step_grads" and f >= 32:
            flops = 6.0 * macs * B
            achieved = flops / (phases[dom] * 1e-3) / 1e12
            roofline = {"bound": "tensor", "kernel": "ncf_mma_tile_kernel (ncf_train_step_grads)",
                        "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                        "frac": achieved / tensor_peak, "traffic": profile_traffic(dom),
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst); the kernel runs fp32-parity "
                                       "3xTF32 on mma.sync, i.e. 3 TF32 MMAs per algorithmic MAC",
                        "algorithmic_flops_per_launch": flops, "launch_ms": phases[dom]}
        else:
            roofline = {"bound": "hbm", "kernel": dom, "achieved": hbm[dom]["achieved_gbs"], "peak": hbm_peak,
                        "unit": "GB/s", "frac": hbm[dom]["frac"], "traffic": profile_traffic(dom), "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": alg_bytes[dom], "launch_ms": phases[dom]}
        roofline["phase_ms"] = phases
        roofline["tile_path"] = tile_path
        roofline["adam_mode"] = "all rows (ncf_adam_step_dense)" if dense else "touched rows + catch-up"
        roofline["hbm_view"] = hbm
        roofline["hbm_peak_gbs"] = hbm_peak
        roofline["step_level"] = {"bytes_per_sample": 4 * R * 7 + 24,
                                  "achieved_gbs_per_gpu": (4 * R * 7 + 24) * value / world / 1e9,
                                  "frac": (4 * R * 7 + 24) * value / world / 1e9 / hbm_peak}
        roofline["eval"] = eval_info["roofline"]
        roofline["nvlink"] = nvlink
        roofline["dp_in_place"] = dp_in_place

    e2e_launch = ("HostFedTrainer: cuda-graph step" + (" (NCCL all-reduce captured)" if dp is not None else "")
                  + f", next batches' H2D overlapped, {8 if dp is None else 2} buffer sets, each step's loss read up to "
                  f"{7 if dp is None else 1} steps behind") if used_graph else "eager"
    gc.enable()
    return dict(value=value, ms_total=ms_total, e2e_value=e2e_value, e2e_ms=e2e_ms, clocks=clocks, e2e_launch=e2e_launch,
                unsampled=unsampled,
                launches_per_step=launches_per_step, roofline=roofline, eval_info=eval_info,
                window=(G if wgraphs is not None else 1),
                dp_partitioned=(dp.partition_users if dp is not None else True),
                dp_tail=(dp is not None and dp.tail is not None))


def sampler_run(dev, hbm_peak):
    """ng_sample on the GPU for a full epoch of the ml20m shape: CSR build once + one sampler launch.
    Algorithmic bytes per positive (SURVEY.md 8d): 8 + 4*num_ng*(1 + ceil(log2 n_u))."""
    import math
    import torch
    from ncf_b200.synth import make_interactions
    from ncf_b200.trainer import EpochStream
    inter = make_interactions("ml20m", device=dev)
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    e[0].record()
    stream = EpochStream(inter.pos_user, inter.pos_item, inter.user_num, inter.item_num, num_ng=4, seed=1)
    e[1].record()
    stream.begin_epoch(0)
    e[2].record()
    stream.begin_epoch(1)
    e[3].record()
    torch.cuda.synchronize()
    P = stream.P
    n_u = P / inter.user_num
    bytes_pos = 8 + 4 * 4 * (1 + math.ceil(math.log2(max(n_u, 2))))
    ms = e[2].elapsed_time(e[3])
    return {"positives": int(P), "negatives_per_epoch": int(P * 4), "csr_build_ms": e[0].elapsed_time(e[1]),
            "ng_sample_ms": ms, "negatives_per_s": P * 4 / (ms * 1e-3),
            "roofline": {"bound": "hbm", "bytes_per_positive": bytes_pos, "achieved_gbs": bytes_pos * P / (ms * 1e-3) / 1e9,
                         "peak": hbm_peak, "frac": bytes_pos * P / (ms * 1e-3) / 1e9 / hbm_peak,
                         "note": "binary-search probes are dependent 4-byte loads: latency-bound, not bandwidth-bound"}}


def small_config_run(dev, epochs_steps: int = 2048):
    """BASELINE configs[1] for reference: NeuMF f=8 L=3 on the synthetic ML-1M shape at the
    reference batch 256 — launch-latency-bound (SURVEY.md H3), so it runs as CUDA-graph windows of
    64 steps through the same public API (EpochStream + FusedTrainStep + train_epoch machinery):
    on-device negative sampling, shuffle, fused steps, no host sync.  Reported beside the headline."""
    import torch
    from ncf_b200.models import NCF
    from ncf_b200.synth import make_interactions
    from ncf_b200.trainer import EpochStream, FusedTrainStep
    inter = make_interactions("ml1m", device=dev)
    torch.manual_seed(0)
    model = NCF(inter.user_num, inter.item_num, 8, 3, 0.0, "NeuMF-end").to(dev)
    B, W = 256, 64
    ts = FusedTrainStep(model, "adam", 1e-3, max_batch=B)
    stream = EpochStream(inter.pos_user, inter.pos_item, inter.user_num, inter.item_num, num_ng=4, seed=1)
    t_s0 = time.perf_counter()
    stream.begin_epoch(0)
    torch.cuda.synchronize()
    sample_ms = (time.perf_counter() - t_s0) * 1e3
    wu = torch.empty(W * B, dtype=torch.int64, device=dev)
    wi = torch.empty(W * B, dtype=torch.int64, device=dev)
    wl = torch.empty(W * B, dtype=torch.float32, device=dev)
    stream.fill(0, W * B, wu, wi, wl)
    for k in range(W):  # eager warm-up window (loads every kernel before capture)
        ts.step(wu[k * B:(k + 1) * B], wi[k * B:(k + 1) * B], wl[k * B:(k + 1) * B])
    graph = ts.capture(wu, wi, wl, B)
    n_windows = max(1, epochs_steps // W)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for w in range(n_windows):
        stream.fill((w + 1) * W * B, W * B, wu, wi, wl)
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    steps = n_windows * W
    return {"workload": "NeuMF f=8 L=3, synthetic ml1m shape, batch 256, Adam, CUDA-graph windows of 64 steps",
            "samples_per_s": steps * B / (ms * 1e-3), "us_per_step": ms * 1e3 / steps, "steps": steps,
            "ng_sample_ms_per_epoch": sample_ms, "negatives_per_epoch": int(stream.P * 4)}


def kd_config_run(dev, steps: int = 1024):
    """BASELINE configs[2]: response distillation on the ML-1M shape at the reference batch 256 — frozen teacher
    NeuMF f=64 L=3, student NeuMF f=8 L=2, alpha 0.5 (src/distillation/response.py:15-32, scripts/train_student.py:
    131-160).  Ours: FusedTrainStep(teacher=...) in CUDA-graph windows of 64 steps (teacher forward + fused student
    step with the KD term in the loss epilogue).  Beside it the reference's own ResponseDistillation + optim.Adam
    under torch eager on this GPU (oracle/_ref; skipped when that directory is absent)."""
    import torch
    from ncf_b200.models import NCF
    from ncf_b200.synth import SHAPES, make_interactions
    from ncf_b200.trainer import EpochStream, FusedTrainStep
    inter = make_interactions("ml1m", device=dev)
    U, I = inter.user_num, inter.item_num
    B, W = 256, 64
    torch.manual_seed(0)
    teacher = NCF(U, I, 64, 3, 0.0, "NeuMF-end").to(dev).eval()
    student = NCF(U, I, 8, 2, 0.0, "NeuMF-end").to(dev)
    ts = FusedTrainStep(student, "adam", 1e-3, max_batch=B, teacher=teacher, alpha=0.5)
    stream = EpochStream(inter.pos_user, inter.pos_item, U, I, num_ng=4, seed=1)
    stream.begin_epoch(0)
    wu = torch.empty(W * B, dtype=torch.int64, device=dev)
    wi = torch.empty(W * B, dtype=torch.int64, device=dev)
    wl = torch.empty(W * B, dtype=torch.float32, device=dev)
    stream.fill(0, W * B, wu, wi, wl)
    for k in range(W):
        ts.step(wu[k * B:(k + 1) * B], wi[k * B:(k + 1) * B], wl[k * B:(k + 1) * B])
    graph = ts.capture(wu, wi, wl, B)
    n_windows = max(1, steps // W)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for w in range(n_windows):
        stream.fill((w + 1) * W * B, W * B, wu, wi, wl)
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    out = {"workload": "response distillation, teacher NeuMF f=64 L=3 -> student NeuMF f=8 L=2, synthetic ml1m shape, "
                       "batch 256, alpha 0.5, Adam, CUDA-graph windows of 64 steps",
           "samples_per_s": n_windows * W * B / (ms * 1e-3), "us_per_step": ms * 1e3 / (n_windows * W)}
    del graph, ts
    from oracle import build_ref
    ref = build_ref.load()
    if ref is not None:
        torch.manual_seed(0)
        rt = ref.NCF(U, I, 64, 3, 0.0, "NeuMF-end").to(dev).eval()
        rs = ref.NCF(U, I, 8, 2, 0.0, "NeuMF-end").to(dev)
        kd = ref.response.ResponseDistillation(rt, rs, temperature=2.0, alpha=0.5)
        kd.train()
        opt = torch.optim.Adam(rs.parameters(), lr=1e-3)
        batches = reference_batches(U, I, B, 8, dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 300
        for k in range(30 + n):
            if k == 30:
                torch.cuda.synchronize()
                e0.record()
            u, i, y = batches[k % 8]
            opt.zero_grad()
            loss = kd(u, i, y)
            loss.backward()
            opt.step()
            loss.item()
        e1.record()
        torch.cuda.synchronize()
        rms = e0.elapsed_time(e1) / n
        out["gpu_eager_reference"] = {"samples_per_s": B / (rms * 1e-3), "us_per_step": rms * 1e3, "steps": n,
                                      "kind": "reference"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="ml20m")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-row-sharded", action="store_true", help="skip the configs[4] sub-result")
    ap.add_argument("--no-extras", action="store_true", help="skip small_config / sampler / gpu_eager_reference")
    ap.add_argument("--no-graph", action="store_true", help="end-to-end steps launched eagerly instead of as a CUDA graph")
    ap.add_argument("--tower-math", choices=["fp32", "tf32"], default="fp32",
                    help="fp32 = 3xTF32 parity mode (headline); tf32 = single-pass opt-in mode")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the outputs of --impl ours on one GPU")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
