#!/usr/bin/env python3
"""bench.py — scan-pairs/sec of the DeLORA hot path on B200 (BASELINE.json metric).

Workload (BASELINE.json configs[1]): batch = 8 synthetic 64x2048 KITTI-shaped scan pairs per GPU
(N ~ 128.5k raw points per scan), one "step" = 2x8 spherical projections + 2x8 normal images +
list/cell-index build + fused SE(3) transform / exact NN / point-to-plane + plane-to-plane loss
forward and backward to the 3x4 transform, for the whole batch.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

* `value`     : pairs/s with the raw scans already resident in HBM (CUDA events, max over ranks).
                R input sets are rotated so that a set is re-read only after > L2-size traffic.
* `e2e`       : the same step driven from pinned HOST buffers through the public pipeline object:
                per step H2D of the raw scans + transforms (copy stream, double-buffered against
                the compute stream) and D2H of the losses + transform gradients.
* `roofline`  : dominant kernel (by measured time inside the timed region), algorithmic bytes /
                its measured duration against the measured HBM peak (MEASURED_PEAKS.json).
* `roofline_encoder`: the tcgen05 encoder (fprop + dgrad + wgrad) timed alone against the measured sustained bf16 peak.
* `ts` / `train_step` / `train_scaling`: BASELINE configs[2] / configs[3], the full training step (batch 16 per GPU)
                with the gradient all-reduce overlapped with the backward; `ar_exposed_ms` = step - step without the
                collective; `cudnn_fp32_ms` / `cudnn_bf16_ms` = the reference's nn.Conv2d stack on the same box (N = 1).
* `cpu_baseline` / `--impl reference`: the oracle port of the reference's CPU path
                (oracle/delora_oracle.py: torch-CPU + numpy + scipy cKDTree) on the host cores.
* `--dump-outputs DIR`: what the last timed step returned on rank 0, `DIR/losses.npy` [8, 8] and
                `DIR/grad_T.npy` [8, 12] (float32).  The inputs are seeded, so two builds run with the same
                arguments can be compared output for output.
Multi-GPU: one process per GPU (torchrun), pairs sharded across ranks, no data-path collective
(weak scaling: 8 pairs per GPU); barrier + max over ranks for the timing.
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it

PAIRS_PER_GPU = 8
H, W, W_RAW = 64, 2048, 2048
ROTATE = 4
METRIC = "scan-pairs/sec on 64x2048 KITTI range images (projection + normals + exact-NN point-to-plane/plane-to-plane loss fwd/bwd)"


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_bf16_peak():
    """Sustained bf16 TFLOP/s (a kernel timed inside a long step): MEASURED_PEAKS.json, else the guide's fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        if "bf16_tflops_sustained" in p:
            return float(p["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)"


# fp32 work of the normals kernel per pixel: 77 taps x (3 sub + 1 gate test + 1 count + 3 sums + 6 second moments = 28 flops,
# FMAs counted as 2) + ~250 for the 3x3 Jacobi eigen-solve, orientation and gates (SURVEY.md 8(d): H*W*(77*~30 + ~250))
NORMALS_FLOP_PER_PIXEL = 77 * 30 + 250


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled through NVML every 5 ms while the timed regions run
    (the B200_PROFILING.md `nvidia-smi --query-gpu=clocks.sm,...` line, without the process spawn)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device_index):
        super().__init__(daemon=True)
        self.samples, self.reason_bits, self._stop_evt, self.handle, self.max_mhz = [], 0, threading.Event(), None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as e:                      # clocks are evidence, not a dependency of the run
            self.error = repr(e)

    def run(self):
        if self.handle is None:
            return
        nv = self.nv
        while not self._stop_evt.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                pass
            self._stop_evt.wait(0.005)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": self.max_mhz, "samples": len(sm),
                "reasons": sorted(name for bit, name in self.REASONS.items() if self.reason_bits & bit)}


def make_inputs(rank, n_sets):
    """Host (pinned) raw scans for `n_sets` rotating input sets of PAIRS_PER_GPU pairs each."""
    from delora_b200 import synthetic
    sets = []
    base = rank * PAIRS_PER_GPU * n_sets
    raw = [synthetic.make_pair(base + i, w_raw=W_RAW) for i in range(PAIRS_PER_GPU * n_sets)]
    n_max = max(max(p[0].shape[1], p[1].shape[1]) for p in raw)
    from delora_b200.pipeline import ScanPairPipeline
    layout = ScanPairPipeline.staging_layout(PAIRS_PER_GPU, 3, n_max)
    for s in range(n_sets):
        # one pinned staging buffer per set, laid out like the pipeline's `inputs`: a step's scans, counts and
        # transforms cross the host link as ONE copy
        flat = torch.zeros((layout["bytes"],), dtype=torch.uint8).pin_memory()
        pts, cnt, tr = ScanPairPipeline.input_views(flat, layout)
        for i in range(PAIRS_PER_GPU):
            s1, s2, _, t_pred = raw[s * PAIRS_PER_GPU + i]
            pts[i, :, :s1.shape[1]] = s1
            pts[PAIRS_PER_GPU + i, :, :s2.shape[1]] = s2
            cnt[i], cnt[PAIRS_PER_GPU + i] = s1.shape[1], s2.shape[1]
            tr[i] = t_pred[:3, :].reshape(12)
        sets.append((pts, cnt, tr, flat))
    return sets, n_max, raw


def barrier(world):
    if world > 1:
        torch.distributed.barrier()


def max_over_ranks(x, world, device):
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=device)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t[0])


def cpu_threads():
    """Threads for the CPU arm.  Measured on the B200 box's host (2 x Xeon 8562Y+, 128 hardware threads;
    profiles/r01_cpu_threads.log): 8 -> 4.00 s/pair, 16 -> 3.53, 32 -> 4.22, 64 -> 5.40, 128 -> 23.4.
    The reference's many small torch ops oversubscribe badly, so its best setting (16) is used."""
    return max(1, min(os.cpu_count() or 1, 16))


def cpu_reference_step(raw_pair, cfg):
    """One pair through the oracle port of the reference's CPU path (fwd + bwd to the transform)."""
    from oracle import delora_oracle as orc
    s1, s2, _, t_pred = raw_pair
    return orc.pair_forward_backward(s1, s2, t_pred, cfg)


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path (its Python modules
    cannot travel to the GPU box, so this is the oracle port: same torch-CPU / numpy / cKDTree
    calls), all host threads, one scan pair per step."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    from delora_b200 import synthetic
    cores = cpu_threads()
    torch.set_num_threads(cores)
    cfg = synthetic.fov_config(h=H, w=W)
    pairs = [synthetic.make_pair(i, w_raw=W_RAW) for i in range(2)]
    # Bounded sample: a pair costs ~3.5 s on the host, so the warm-up is capped at 2 pairs and the timed part at as
    # many of the K requested steps (1 pair each) as fit into --cpu-budget-s; value = pairs / time of what ran.
    t_w = time.perf_counter()
    n_warm = max(1, min(args.warmup, 2))
    for i in range(n_warm):
        cpu_reference_step(pairs[i % 2], cfg)
    t_pair = (time.perf_counter() - t_w) / n_warm
    n_timed = max(1, min(args.steps, int(args.cpu_budget_s / max(t_pair, 1e-3))))
    t0 = time.perf_counter()
    for i in range(n_timed):
        cpu_reference_step(pairs[i % 2], cfg)
    dt = time.perf_counter() - t0
    value = n_timed / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "steps_timed": n_timed, "warmup_run": n_warm,
        "ms_per_step": 1e3 * dt / n_timed,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1] shape: 64x2048 scan pairs, projection+normals+ICP loss fwd/bwd; "
                               "1 pair per step on the host CPU", "pairs_per_step": 1, "H": H, "W": W},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port",
                         "sample": f"{n_timed} of the {args.steps} requested steps x 1 pair, bounded by "
                                   f"--cpu-budget-s={args.cpu_budget_s:g} (oracle port of the reference CPU path, "
                                   f"torch {torch.__version__} CPU, {cores} of {os.cpu_count()} threads = best of a sweep)"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def train_leg(args, rank, world, device, raw, n_max):
    """BASELINE configs[2] (1 GPU) / configs[3] (DDP, 16 pairs per GPU): projection + normals + tcgen05 encoder fwd/bwd +
    heads + fused ICP loss + gradient all-reduce (overlapped, parallel_grad.py) + Adam; CUDA events, max over ranks.
    Also measured here, on the same inputs: the step without the collective (-> exposed all-reduce time), the blocking
    flat all-reduce, the encoder alone (-> tensor-core roofline) and, on rank 0 at N = 1, the reference's own
    nn.Conv2d stack on cuDNN in fp32 and under bf16 autocast (BASELINE.md §3 'reference on the same box')."""
    from delora_b200 import synthetic
    from delora_b200.train_step import SyntheticTrainStep
    tcfg = synthetic.fov_config(h=H, w=W, device=device)
    tb = args.train_batch
    tpts = torch.zeros((2 * tb, 3, n_max), dtype=torch.float32)
    tcnt = torch.zeros((2 * tb,), dtype=torch.int32)
    for i in range(tb):
        s1, s2, _, _ = raw[i % len(raw)]
        tpts[i, :, :s1.shape[1]] = s1
        tpts[tb + i, :, :s2.shape[1]] = s2
        tcnt[i], tcnt[tb + i] = s1.shape[1], s2.shape[1]
    tpts, tcnt = tpts.to(device), tcnt.to(device)

    def timed(ts, steps):
        for _ in range(3):
            ts.step()
        torch.cuda.synchronize()
        barrier(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss, _ = ts.step()
        e1.record()
        torch.cuda.synchronize()
        barrier(world)
        return max_over_ranks(e0.elapsed_time(e1), world, device) / steps, float(loss)

    def build(**kw):
        torch.manual_seed(1234)
        ts = SyntheticTrainStep(tcfg, tb, n_max, **kw)
        ts.load(tpts, tcnt)
        return ts

    ts = build(use_tensor_cores=True, grad_sync="bucketed")
    ms, loss = timed(ts, args.train_steps)
    transport = getattr(ts.sync, "transport", "none") if world > 1 else "none"
    transport_note = getattr(ts.sync, "transport_note", "")
    if world > 1 and getattr(ts.sync, "peer", None) is not None:
        # a rank that missed a peer-memory collective (20 s limit inside the kernel) invalidates the timing: every
        # rank then repeats the measurement over NCCL and the line says so
        bad = torch.tensor([int(ts.sync.peer.status.item() != 0)], dtype=torch.int32, device=device)
        torch.distributed.all_reduce(bad, op=torch.distributed.ReduceOp.MAX)
        if int(bad.item()):
            del ts
            ts = build(use_tensor_cores=True, grad_sync="bucketed-nccl")
            ms, loss = timed(ts, args.train_steps)
            transport, transport_note = "nccl", "peer-memory collective timed out on some rank; re-measured over NCCL"
    out = {"ms_per_step": ms, "pairs_per_s": world * tb / (ms * 1e-3), "n_gpus": world, "batch_per_gpu": tb,
           "loss": loss, "encoder_gflop_per_step": 3 * 96.17 * tb,
           "workload": f"full training step, batch {tb}/GPU, 64x{W}: projection + normals + tcgen05 encoder fwd/bwd "
                       "(bf16) + heads + fused ICP loss fwd/bwd (fp32) + Adam"
                       + (" + per-bucket all-reduce of 11.88 M fp32 gradients overlapped with the backward (transport: "
                          + transport + ")" if world > 1 else "")}
    if world > 1:
        out["allreduce_transport"] = transport
        if transport_note:
            out["allreduce_transport_note"] = transport_note
    if world == 1:
        # encoder alone: forward + backward of the trunk on fixed images -> achieved bf16 TFLOP/s vs the measured peak
        enc = ts.model._tensor_core_path()
        with torch.no_grad():
            from delora_b200 import ops
            image, _ = ops.project(ts.points, ts.n_points, H, W, ts.hf, ts.vf)
        img1, img2 = image[:tb].contiguous(), image[tb:].contiguous()
        sel = torch.randn(tb, 512, device=device)

        def enc_step():
            ts.optimizer.zero_grad(set_to_none=True)
            (enc.pooled_features(img1, img2) * sel).sum().backward()
            ts.sync.finish()
        for _ in range(2):
            enc_step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.train_steps):
            enc_step()
        e1.record()
        torch.cuda.synchronize()
        out["encoder_ms"] = e0.elapsed_time(e1) / args.train_steps
        del enc
    del ts
    if world > 1:
        ts = build(use_tensor_cores=True, grad_sync="none")
        ms_none, _ = timed(ts, args.train_steps)
        del ts
        ts = build(use_tensor_cores=True, grad_sync="flat")
        ms_flat, _ = timed(ts, args.train_steps)
        del ts
        out.update({"ms_without_allreduce": ms_none, "allreduce_exposed_ms": ms - ms_none,
                    "ms_blocking_flat_allreduce": ms_flat})
        if transport != "nccl":
            ts = build(use_tensor_cores=True, grad_sync="bucketed-nccl")
            ms_nccl, _ = timed(ts, args.train_steps)
            del ts
            out.update({"ms_bucketed_nccl": ms_nccl, "allreduce_exposed_ms_nccl": ms_nccl - ms_none})
    elif rank == 0 and args.cudnn_steps > 0:
        ts = build(use_tensor_cores=False)
        out["cudnn_fp32_ms"], _ = timed(ts, args.cudnn_steps)
        del ts
        ts = build(use_tensor_cores=False, autocast_bf16=True)
        out["cudnn_bf16_ms"], _ = timed(ts, args.cudnn_steps)
        del ts
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        # NCCL's own log lines (e.g. "NCCL version ...") go to stderr: stdout carries exactly one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        torch.distributed.init_process_group("nccl", device_id=device)
    from delora_b200 import synthetic
    from delora_b200.pipeline import ScanPairPipeline
    cfg = synthetic.fov_config(h=H, w=W)
    hf, vf = cfg["horizontal_field_of_view"], cfg["kitti"]["vertical_field_of_view"]

    global ROTATE
    ROTATE = max(1, args.rotate)
    sets, n_max, raw = make_inputs(rank, ROTATE)
    pipes = [ScanPairPipeline(PAIRS_PER_GPU, n_max, H, W, hf, vf, device=device) for _ in range(ROTATE)]
    for p, (pts, cnt, tr, flat) in zip(pipes, sets):
        p.inputs.copy_(flat)
    torch.cuda.synchronize()

    # ---------------- device-resident throughput (`value`) + per-operator times -------------
    K, Wm = args.steps, args.warmup
    for i in range(Wm):
        pipes[i % ROTATE].step()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    sampler = ClockSampler(local)
    sampler.start()
    barrier(world)
    torch.cuda.synchronize()
    # `value`: the pipeline as a user runs it -- two sub-batches of pairs on two streams (pipeline.py), whose kernels
    # overlap; the timed region is bracketed on the launching stream, which step() forks from and joins into
    t_wall = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        last = pipes[i % ROTATE].step()
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    t_wall = time.perf_counter() - t_wall
    total_ms = max_over_ranks(e0.elapsed_time(e1), world, device)
    if args.dump_outputs and rank == 0:
        # the step's output buffers are overwritten by the passes below: copy them out now
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in zip(("losses", "grad_T"), last):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy().astype(np.float32))
    # per-operator durations (-> `kernels`, `roofline`): K more steps of the same inputs on ONE stream with CUDA events
    # around every operator -- with overlapping sub-batches an operator's duration is not separable
    for i in range(K):
        pipes[i % ROTATE].step(events=ev[i])
    torch.cuda.synchronize()
    one_stream_ms = ev[0][0].elapsed_time(ev[K - 1][3]) / K
    op_ms = {name: sum(ev[i][j].elapsed_time(ev[i][j + 1]) for i in range(K)) / K
             for j, name in enumerate(ScanPairPipeline.OPERATORS)}
    value = world * PAIRS_PER_GPU * K / (total_ms * 1e-3)
    counts = (pipes[0].pts_grid[:, :, 3].view(torch.int32) >= 0).sum(dim=1).float().mean().item()
    losses0 = pipes[0].losses[0].tolist()

    # ---------------- end to end from pinned host buffers (`e2e`) -----------------------------
    copy_stream = torch.cuda.Stream(device=device)
    compute = torch.cuda.current_stream()
    out_host = [(torch.empty((PAIRS_PER_GPU, 8), dtype=torch.float32).pin_memory(),
                 torch.empty((PAIRS_PER_GPU, 12), dtype=torch.float32).pin_memory()) for _ in range(ROTATE)]
    h2d_done = [torch.cuda.Event() for _ in range(ROTATE)]
    slot_free = [torch.cuda.Event() for _ in range(ROTATE)]

    def h2d(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(slot_free[slot])
            pipes[slot].inputs.copy_(sets[slot][3], non_blocking=True)     # scans + counts + transforms, one copy
            h2d_done[slot].record(copy_stream)

    def e2e_loop(n):
        for s in range(ROTATE):
            slot_free[s].record(compute)
        h2d(0)
        for i in range(n):
            slot = i % ROTATE
            if i + 1 < n:
                h2d((i + 1) % ROTATE)                     # prefetch the next step's scans
            compute.wait_event(h2d_done[slot])
            losses, grad_t = pipes[slot].step()
            out_host[slot][0].copy_(losses, non_blocking=True)
            out_host[slot][1].copy_(grad_t, non_blocking=True)
            slot_free[slot].record(compute)

    e2e_loop(max(3, Wm))
    torch.cuda.synchronize()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(compute)
    e2e_loop(K)
    e1.record(compute)
    torch.cuda.synchronize()
    barrier(world)
    e2e_ms = max_over_ranks(e0.elapsed_time(e1), world, device)
    clocks = sampler.stop()
    e2e_value = world * PAIRS_PER_GPU * K / (e2e_ms * 1e-3)
    h2d_bytes = sets[0][3].numel()
    d2h_bytes = sum(t.numel() * t.element_size() for t in out_host[0])
    assert abs(out_host[0][0][0, 1].item() - losses0[1]) <= 1e-6 * abs(losses0[1]) + 1e-12

    # ---------------- full training step (BASELINE configs[2]/[3]: batch 16 per GPU, bf16 tensor-core encoder) ----
    train = None
    if args.train_steps > 0:
        try:
            train = train_leg(args, rank, world, device, raw, n_max)
        except Exception as e:                      # second leg: never takes the headline down
            train = {"error": repr(e)[:300]}

    # ---------------- streaming inference (BASELINE configs[4]), informational, rank 0 only ----------------
    stream = None
    if args.stream_frames > 0 and rank == 0:
        try:
            from delora_b200.deploy.stream import OdometryStream
            from delora_b200.models.model import OdometryModel
            scfg = synthetic.fov_config(h=H, w=W, device=device)
            scfg.update({"pre_feature_extraction": False, "resnet_outputs": 1000, "use_dropout": False,
                         "layers": [2, 2, 2, 2], "factor_fewer_resnet_channels": 1, "activation_fct": "tanh",
                         "use_single_mlp_at_output": False, "use_tensor_core_encoder": True})
            torch.manual_seed(4321)
            smodel = OdometryModel(scfg).to(device).eval()
            frames = [raw[i % len(raw)][i // len(raw) % 2] for i in range(min(len(raw) * 2, 32))]
            lat = {}
            import gc
            gc.collect()
            gc.freeze()            # keep the collector away from the (large, static) bench heap while frames are timed
            for graph in (True, False):
                st = OdometryStream(smodel, scfg, "kitti", n_max, use_cuda_graph=graph)
                for i in range(8):                                   # first frame, capture, warm-up
                    st.push(frames[i % len(frames)])
                ts_ = []
                for i in range(args.stream_frames):
                    t0 = time.perf_counter()
                    st.push(frames[i % len(frames)])
                    ts_.append((time.perf_counter() - t0) * 1e3)
                worst = max(range(len(ts_)), key=lambda j: ts_[j])
                srt = sorted(ts_)
                lat[graph] = (srt[len(srt) // 2], srt[min(len(srt) - 1, int(0.99 * len(srt)))], srt[-1], worst)
                del st
            stream = {"workload": f"inference stream, batch 1, 64x{W}, N~{n_max}: pinned host scan -> H2D -> 1 projection "
                                  "(previous range image cached) + tcgen05 encoder forward + heads + quaternion->T "
                                  "-> D2H of T, host-timed per frame (perf_counter around push(), includes the sync)",
                      "frames": args.stream_frames, "ms_per_frame_p50": lat[True][0], "ms_per_frame_p99": lat[True][1],
                      "frames_per_s": 1e3 / lat[True][0], "cuda_graph": True,
                      "ms_per_frame_max": lat[True][2], "slowest_frame_index": lat[True][3],
                      "eager_ms_per_frame_p50": lat[False][0], "eager_ms_per_frame_p99": lat[False][1]}
            gc.unfreeze()
            del smodel
        except Exception as e:                      # informational leg: never takes the headline down
            stream = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel ----------------------------------------
    peak, peak_src = measured_peaks()
    alg = pipes[0].algorithmic_bytes(k_points=counts)
    dom = max(op_ms, key=op_ms.get)
    kernels = {name: {"ms": op_ms[name], "algorithmic_bytes": alg[name],
                      "achieved_gbs": alg[name] / (op_ms[name] * 1e-3) / 1e9,
                      "frac_of_hbm_peak": alg[name] / (op_ms[name] * 1e-3) / 1e9 / peak}
               for name in op_ms}
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tdoc = json.load(f)
        traffic = tdoc.get(dom)
        # the three operators are instruction-issue bound, not HBM bound (DESIGN.md 4.1-4.3): next to the HBM
        # fraction report how full the issue slots are -- warp instructions per launch (ncu, profiles/) over
        # the slots the measured duration offers (SMs x 4 schedulers x SM clock)
        sm_clock = (clocks.get("sm_mhz") or 1965.0) * 1e6
        for name, wi in (tdoc.get("_warp_instructions") or {}).items():
            if name in kernels and wi:
                kernels[name]["warp_instructions"] = wi
                kernels[name]["issue_slot_frac"] = wi / (kernels[name]["ms"] * 1e-3 * 148 * 4 * sm_clock)
    sm_clock_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
    fp32_peak_tflops = 148 * 128 * 2 * sm_clock_hz / 1e12                 # FFMA lanes x 2 flops at the clock sampled under load
    if dom == "normals":
        # the dominant kernel is bound by the FP32 pipe, not by HBM (SURVEY.md 8(d), DESIGN.md 4.2): the roofline is
        # its fp32 work over the fp32 peak; the HBM figure stays as a note
        flops = 2 * PAIRS_PER_GPU * H * W * NORMALS_FLOP_PER_PIXEL
        ach = flops / (op_ms[dom] * 1e-3) / 1e12
        roofline = {"kernel": dom, "bound": "fp32", "achieved": ach, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
                    "frac": ach / fp32_peak_tflops, "traffic": traffic,
                    "peak_source": f"148 SMs x 128 FMA lanes x 2 x {sm_clock_hz / 1e6:.0f} MHz (SM clock sampled during the run)",
                    "flops_per_launch": flops,
                    "hbm": {"achieved_gbs": kernels[dom]["achieved_gbs"], "peak_gbs": peak, "frac": kernels[dom]["frac_of_hbm_peak"],
                            "peak_source": peak_src},
                    "issue_slot_frac": kernels[dom].get("issue_slot_frac"),
                    "counters_measured_at": (tdoc.get("_measured_at") if traffic is not None else None),
                    "measured_in": "second timed pass of the same K steps on ONE stream (CUDA events around every operator; "
                                   "its step time is `ms_per_step_one_stream`): the `value` pass runs two sub-batches of "
                                   "pairs on two streams whose kernels overlap, so operator durations are not separable there",
                    "note": "fp32 flops (SURVEY 8(d): 77 taps x ~30 + ~250 per pixel) / CUDA-event duration of the launch; "
                            "`hbm` = algorithmic bytes over the measured copy bandwidth for the same launch; "
                            "`issue_slot_frac` / `traffic` come from the ncu capture of the commit named in counters_measured_at"}
    else:
        roofline = {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["achieved_gbs"], "peak": peak,
                    "unit": "GB/s", "frac": kernels[dom]["frac_of_hbm_peak"], "traffic": traffic,
                    "peak_source": peak_src, "issue_slot_frac": kernels[dom].get("issue_slot_frac"),
                    "counters_measured_at": (tdoc.get("_measured_at") if traffic is not None else None),
                    "measured_in": "second timed pass of the same K steps on one stream (`ms_per_step_one_stream`)",
                    "note": "algorithmic bytes (SURVEY 8(d) formulas at the measured mean K valid pixels/scan) / "
                            "CUDA-event duration of the launch; see `kernels` for every operator"}
    roofline_encoder = None
    if train and "encoder_ms" in train:
        bf_peak, bf_src = measured_bf16_peak()
        ach = train["encoder_gflop_per_step"] / train["encoder_ms"]            # GFLOP / ms = TFLOP/s
        step_ach = train["encoder_gflop_per_step"] / train["ms_per_step"]
        roofline_encoder = {"bound": "tensor", "achieved": ach, "peak": bf_peak, "unit": "TFLOP/s", "frac": ach / bf_peak,
                            "peak_source": bf_src, "ms": train["encoder_ms"],
                            "over_whole_step": {"achieved": step_ach, "frac": step_ach / bf_peak, "ms": train["ms_per_step"]},
                            "note": "encoder forward + backward (20 convolutions: fprop, dgrad, wgrad; 3 x 96.17 GFLOP per "
                                    "sample) timed alone with CUDA events; `over_whole_step` divides the same flops by the "
                                    "full training step (projection, normals, loss, heads, Adam included)"}

    # ---------------- CPU baseline: oracle port on a bounded sample --------------------------
    cores = cpu_threads()
    torch.set_num_threads(cores)
    cpu_n = args.cpu_pairs
    out, cpu_dt, cpu_value = {"loss_po2pl": None, "loss_pl2pl": None}, 0.0, None
    if cpu_n > 0:
        out = cpu_reference_step(raw[0], cfg)             # warm-up (allocator, thread pools) + the parity check below
        t0 = time.perf_counter()
        for i in range(cpu_n):
            cpu_reference_step(raw[i % len(raw)], cfg)
        cpu_dt = time.perf_counter() - t0
        cpu_value = cpu_n / cpu_dt

    tshort = None
    if train and "ms_per_step" in train:
        # BASELINE configs[2] / configs[3] in short keys (kept at the front AND repeated as the last key of the line so
        # that a truncated record still carries them): ms per step, whole-job pairs/s, exposed all-reduce time
        tshort = {"n": world, "ms": round(train["ms_per_step"], 4), "pairs_per_s": round(train["pairs_per_s"], 1),
                  "ar_exposed_ms": (round(train["allreduce_exposed_ms"], 4) if "allreduce_exposed_ms" in train else None),
                  "enc_frac_of_bf16_peak": (round(roofline_encoder["frac"], 4) if roofline_encoder else None)}
    line = {
        "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": total_ms / K, "ms_per_step_one_stream": one_stream_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "ts": tshort,
        "config": {"workload": "BASELINE configs[1]: batch=8 synthetic 64x2048 clouds per GPU, "
                               "projection+normals+point-to-plane/plane-to-plane loss fwd/bwd",
                   "pairs_per_gpu": PAIRS_PER_GPU, "H": H, "W": W, "points_per_scan": n_max,
                   "concurrency": f"{pipes[0].concurrency} sub-batches of pairs per step, each on its own stream "
                                  "(ScanPairPipeline default; forked from / joined into the timed stream)",
                   "valid_pixels_per_scan": counts, "parallelism": f"dp{world} (pairs sharded, no collective)",
                   "l2": f"{ROTATE} rotating input sets (~{ROTATE * 185} MB of inputs+intermediates > 126 MB L2); "
                         "no flush kernels inside the timed region"},
        "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_ms / K,
                "h2d_gbs": h2d_bytes / (e2e_ms / K * 1e-3) / 1e9,
                "how": "pinned host scans -> H2D on a copy stream (prefetch 1 step ahead) -> pipeline.step() -> "
                       "D2H of losses[B,8] + grad_T[B,12]",
                "bound": "host link: the raw fp32 scans (12 B/point) cross PCIe every step; when h2d_gbs is ~50 the "
                         "copy, not the kernels, sets this number"},
        "gpu_launches": K * pipes[0].launches_per_step,
        "roofline": roofline, "roofline_encoder": roofline_encoder, "kernels": kernels,
        "cpu_baseline": {"value": cpu_value, "unit": "pairs/s", "cores": cores, "kind": "port",
                         "sample": f"{cpu_n} pairs at 64x2048 through oracle.pair_forward_backward "
                                   f"(torch {torch.__version__} CPU + scipy cKDTree), {cores} of {os.cpu_count()} host threads "
                                   f"(best of a sweep), {cpu_dt:.1f} s"},
        "train_step": train,
        "inference_stream": stream,
        "clocks": clocks, "wall_s_timed_region": t_wall,
        "check": {"loss_po2pl": losses0[1], "loss_pl2pl": losses0[2], "pairs": losses0[3],
                  "cpu_loss_po2pl": out["loss_po2pl"], "cpu_loss_pl2pl": out["loss_pl2pl"]},
        "train_scaling": tshort,
    }
    print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-pairs", type=int, default=3, help="pairs timed for the cpu_baseline leg (0 = skip)")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0,
                    help="--impl reference: wall-clock budget of the timed CPU steps (a pair costs seconds)")
    ap.add_argument("--stream-frames", type=int, default=200,
                    help="frames of the informational streaming-inference leg (0 = skip)")
    ap.add_argument("--train-steps", type=int, default=10, help="steps of the full-training-step leg (0 = skip)")
    ap.add_argument("--cudnn-steps", type=int, default=3,
                    help="steps of the reference-on-GPU bar (torch nn.Conv2d / cuDNN, fp32 and bf16 autocast; N = 1; 0 = skip)")
    ap.add_argument("--train-batch", type=int, default=16)
    ap.add_argument("--rotate", type=int, default=ROTATE, help="rotating input sets (1 only for profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the losses and transform gradients of the last timed step to DIR/*.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
