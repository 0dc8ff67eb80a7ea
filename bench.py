#!/usr/bin/env python
"""bench.py -- particle-steps/sec of the filtering recursion on B200 (contract: task statement section 4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c1|c2] [--impl b200|reference] [--dump-outputs DIR]

A "step" is ONE pass of the hot path over one batch of synthetic trajectories: the whole
``forward_loop`` of the named BASELINE config (T filter steps for N trajectories).

  value  particle-steps/s of the recursion with its inputs (hoisted observation features, controls)
         resident in HBM; noise is drawn on the device inside the timed region, as torchfilter does.
  e2e    the same metric through the public API ``filter.forward_loop(observations=, controls=)``
         with PINNED HOST buffers: H2D of the raw observations (images included), the observation
         encoders, the recursion, and the D2H read of the estimates are all inside the timed region.
  roofline      the dominant kernel (the per-particle MLP chain) timed live with CUDA events on its
                stream: algorithmic FLOPs (BASELINE.md section 4: 189,824 / particle-step, hoisted
                minimum) / launch time vs the measured bf16 peak of MEASURED_PEAKS.json.
  cpu_baseline  the oracle port (eager PyTorch, CPU, all host threads) on a bounded sample.
  gpu_eager_baseline  the same oracle port with eager PyTorch on this B200 (BASELINE.md section 5.4: "the reference on
                this box" -- launch-bound, ~150-200 library kernels per filter step).
  training      BASELINE config C4 at the same rank count: one BPTT step (forward over 15 filter steps, backward,
                gradient all-reduce over NCCL, Adam) captured in ONE CUDA graph per rank; ms/step max over ranks.

--dump-outputs DIR (c1, c2, c3): after the timed steps of ``value``, rank 0 writes what the last of them computed as
DIR/<name>.npy (float32): the estimates of every filter step, and the belief the filter holds afterwards (particle
states and log-weights; for the EKF, the fused covariances).  The device noise is seeded, so with the same arguments the
inputs are identical from run to run and two builds can be compared output for output.

Multi-GPU: trajectories are sharded, N per rank is fixed (weak scaling), no data-path collective.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import torch  # noqa: E402

WORKLOADS = {
    # name: (model class, state_dim, N per GPU, particles, T, BASELINE.json config string)
    "c3": ("PushUnimodalParticleFilter", 2, 4096, 1000, 100,
           "Push task unimodal weighted-fusion PF, 4096 trajectories x 1000 particles x 100 steps"),
    "c1": ("PushCrossmodalParticleFilter", 2, 32, 30, 50,
           "Push task crossmodal PF eval (state_dim=2, 30 particles), 32 trajectories x 50 steps"),
    "c2": ("DoorCrossmodalKalmanFilter", 3, 256, 1, 100,
           "Door task crossmodal EKF eval (state_dim=3), 256 trajectories x 100 steps"),
    "c4": ("PushCrossmodalParticleFilter", 2, 8192, 30, 15,
           "Push crossmodal PF BPTT training step (fwd+bwd, subsequence 16, 8192 trajectories), gradient allreduce"),
    "c5": ("PushUnimodalParticleFilter", 2, 16384, 0, 10,
           "Particle-count sweep 1K-1M particles x 16K trajectories, trajectory-sharded"),
}
# bounded CPU sample (trajectories, steps) of the big workloads: a few seconds of host work per timed run
CPU_SAMPLE = {"c3": (64, 20), "c4": (256, 15)}
GPU_EAGER_SAMPLE = {"c3": (512, 20), "c1": (32, 50), "c2": (256, 100)}  # eager-torch oracle on the GPU (launch-bound)
FLOP_PER_PARTICLE_STEP = {2: 189_824.0, 3: 190_336.0}  # BASELINE.md section 4 (hoisted minimum)
DUMP_LIMIT_BYTES = 64_000_000  # C3's estimates + final particle set: 52.4 MB


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback"}


def ncu_traffic(capture):
    """dram read + write bytes per launch of a kernel from the committed ncu --set full capture
    (profiles/r0N_ncu_metrics.json, written by tools/ncu_extract.py from the .ncu-rep files), or None."""
    d = None
    for rnd in ("r02", "r01"):  # the newest committed capture of this kernel
        path = os.path.join(REPO, "profiles", f"{rnd}_ncu_metrics.json")
        if os.path.exists(path):
            with open(path) as f:
                d = json.load(f).get(capture)
            if d:
                break
    if not d or "dram_read" not in d or "dram_write" not in d:
        return None
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    return sum(d[k]["value"] * scale.get(d[k]["unit"], 1.0) for k in ("dram_read", "dram_write"))


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) == 6 and parts[0].isdigit():
                self.samples.append(parts)

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(self.samples[0][1]), "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
def build_inputs(workload, seed=0):
    from multimodalfilter_b200.synthetic import synthetic_trajectories

    name, sd, N, M, T, _ = WORKLOADS[workload]
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=seed)
    return states, obs, controls


def dump_outputs(directory, outputs):
    """Write every tensor of ``outputs`` (name -> tensor) as ``directory/<name>.npy`` in float32."""
    import numpy as np

    arrays = {name: t.detach().float().cpu().numpy() for name, t in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"outputs of {total} bytes exceed the dump limit of {DUMP_LIMIT_BYTES}"
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def run_cpu_oracle(workload, n_sample, t_sample, repeats=1, warm=True, device="cpu"):
    """The reference's path (oracle port: eager PyTorch, on the host cores or -- device="cuda:k" -- on the GPU) on a
    bounded sample of the workload.  Returns (particle-steps/s, description, seconds)."""
    from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories
    from oracle import crossmodal_port as port

    name, sd, _, M, _, _ = WORKLOADS[workload]
    filt = fill_parameters(getattr(port, name)(), seed=0).eval().to(device)
    is_pf = hasattr(filt, "num_particles")
    if is_pf:
        filt.num_particles = M
    states, obs, controls = synthetic_trajectories(t_sample + 1, n_sample, sd, seed=0)
    states, controls = states.to(device), controls.to(device)
    obs = {k: v.to(device) for k, v in obs.items()}
    cov = (torch.eye(sd, device=device) * 0.1)[None].expand(n_sample, sd, sd)
    on_gpu = str(device) != "cpu"
    best = None
    if warm:  # first call pays for thread-pool start-up, allocator growth and oneDNN primitive creation: not timed
        with torch.no_grad():
            nw = min(n_sample, 4)
            filt.initialize_beliefs(mean=states[0][:nw], covariance=cov[:nw])
            filt.forward_loop(observations={k: v[1:3, :nw] for k, v in obs.items()}, controls=controls[1:3, :nw])
    for _ in range(repeats):
        torch.manual_seed(0)
        t0 = time.perf_counter()
        with torch.no_grad():
            filt.initialize_beliefs(mean=states[0], covariance=cov)
            filt.forward_loop(observations={k: v[1:] for k, v in obs.items()}, controls=controls[1:])
        if on_gpu:
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    units = n_sample * (M if is_pf else 1) * t_sample
    where = "GPU (eager, library kernels)" if on_gpu else "CPU"
    sample = f"{name} oracle port, eager PyTorch {where} fp32, forward_loop incl. observation encoders, N={n_sample} M={M} T={t_sample}"
    return units / best, sample, best


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name, sd, N, M, T, cfg = WORKLOADS[args.workload]
    n_s, t_s = CPU_SAMPLE.get(args.workload, (min(N, 32), min(T, 50)))
    torch.set_num_threads(os.cpu_count() or 1)
    times = []
    for i in range(args.warmup + args.steps):
        rate, sample, dt = run_cpu_oracle(args.workload, n_s, t_s)
        if i >= args.warmup:
            times.append(dt)
    units = n_s * (M if "Particle" in name else 1) * t_s
    ms = 1e3 * sum(times) / len(times)
    value = units / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "particle-steps/sec", "value": value, "unit": "particle-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg, "bounded_sample": sample},
        "cpu_baseline": {"value": value, "unit": "particle-steps/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def time_resample_modes(N, Mp, sd, dev, reps=12):
    """mmf_pf_normalize_resample stand-alone at the workload's shape, every resampling mode: CUDA events around each
    launch on the launching stream, L2 flushed (a 256 MB write) between launches, median.  Algorithmic bytes (BASELINE.md
    section 4): log-weights read + written 8, states read + written 8 sd, float64 uniform 8 (multinomial only)."""
    from multimodalfilter_b200 import _lib, ops

    g = torch.Generator(device=dev).manual_seed(0)
    states = torch.randn(N, Mp, sd, device=dev, generator=g)
    logw = torch.randn(N, Mp, device=dev, generator=g)  # log-normal weights, effective sample size ~ M / e
    u_m = torch.rand(N, Mp, device=dev, dtype=torch.float64, generator=g)
    u_s = torch.rand(N, device=dev, dtype=torch.float64, generator=g)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {}
    for name, mode, u in (("multinomial", _lib.RESAMPLE_MULTINOMIAL_STRICT, u_m), ("multinomial_fast", _lib.RESAMPLE_MULTINOMIAL_FAST, u_m),
                          ("systematic", _lib.RESAMPLE_SYSTEMATIC_STRICT, u_s), ("systematic_fast", _lib.RESAMPLE_SYSTEMATIC_FAST, u_s)):
        ts = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.pf_normalize_resample(states, logw, mode=mode, uniforms=u)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = sorted(ts[2:])[len(ts[2:]) // 2]
        bytes_ = N * Mp * (8 + 8 * sd + (8 if u is u_m else 0))
        out[name] = {"avg_launch_ms": ms, "achieved": bytes_ / (ms / 1e3) / 1e9, "unit": "GB/s", "bytes": bytes_}
    return out


def setup_ranks(args):
    """One process per GPU (torch.distributed.run sets RANK / LOCAL_RANK / WORLD_SIZE); NCCL process group when N > 1."""
    import torch.distributed as dist

    from multimodalfilter_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.load().mmf_device_check())
    return world, rank, local_rank, dev


def run_c4(ctx, steps, warmup, precision):
    """BASELINE config C4: one BPTT training step = forward over 15 filter steps + backward + gradient all-reduce + Adam,
    on N=8192 trajectories x 30 particles per GPU; the whole step (the NCCL all-reduce included: it is issued as
    ncclAllReduce on the capture stream, multimodalfilter_b200.distributed.StreamAllReduce) is ONE CUDA graph per rank.
    The observation encoders are hoisted and frozen (their features are inputs, as in the primary timed region of the eval
    configs): at this batch size a backward through three CNNs x 8192 x 15 images would need ~220 GB of activations and is
    the cuDNN-bound "next" row, not the recursion.  Trainable: both measurement heads, the observation halves of their
    first shared Linear, and the modality weight model's fusion layers; the dynamics is frozen as in the reference's
    curricula (ref: scripts/push_task/train_push.py:154,213).  Gradients live in one flat buffer (views), so the
    collective is a single in-place all-reduce with no concatenate / copy-back.  Returns the result record."""
    import torch.distributed as dist

    from multimodalfilter_b200 import ops
    from multimodalfilter_b200.crossmodal import models as M_
    from multimodalfilter_b200.distributed import FlatGradients, StreamAllReduce, max_over_ranks
    from multimodalfilter_b200.synthetic import fill_parameters

    world, rank, local_rank, dev = ctx
    name, sd, N, Mp, T, cfg = WORKLOADS["c4"]
    filt = fill_parameters(M_.PushCrossmodalParticleFilter(), seed=0).to(dev)
    filt.train()
    filt.num_particles = Mp
    filt.precision = precision or "bf16x3"
    mm = filt.measurement_model
    wm = mm.crossmodal_weight_model
    trainable = [p for h in mm.measurement_models for p in list(h.state_layers.parameters()) + list(h.shared_layers.parameters())]
    trainable += list(wm.fusion_layers.parameters())
    for p in filt.parameters():
        p.requires_grad_(False)
    for p in trainable:
        p.requires_grad_(True)
    grads = FlatGradients(trainable)
    # The step's only collective.  Default at N > 1: the step is TWO CUDA graphs (zero + forward + backward | scale + Adam)
    # with torch.distributed's NCCL all-reduce of the flat gradient buffer enqueued between them on the same stream.
    # MMF_NCCL_IN_GRAPH=1 (opt-in): ncclAllReduce issued on the capture stream (distributed.StreamAllReduce), the whole
    # step one graph.
    in_graph = world > 1 and os.environ.get("MMF_NCCL_IN_GRAPH") == "1"
    reduce_ = StreamAllReduce(dev) if in_graph else None
    # fused: one multi-tensor kernel instead of ~10 launches per tensor; capturable: the step lives in a CUDA graph
    opt = torch.optim.Adam(trainable, lr=1e-4, fused=True, capturable=True)
    g = torch.Generator(device=dev).manual_seed(rank)
    feats = [torch.randn(T, N, 64, device=dev, generator=g), torch.randn(T, N, 128, device=dev, generator=g)]
    wm_feats = torch.randn(T, N, 192, device=dev, generator=g)
    controls = torch.randn(T, N, 7, device=dev, generator=g)
    targets = torch.randn(T, N, sd, device=dev, generator=g)
    mean0 = torch.randn(N, sd, device=dev, generator=g)
    cov = (torch.eye(sd, device=dev) * 0.1)[None].expand(N, sd, sd).contiguous()

    def forward_backward():
        grads.zero()
        filt.initialize_beliefs(mean=mean0, covariance=cov)
        # what forward_loop does in train mode: the per-trajectory pieces (weight-model fusion layers, the heads'
        # observation rows, the dynamics rows) once over all T * N rows, then the per-particle kernels step by step
        modw = wm.fusion_layers(wm_feats.reshape(T * N, -1)).reshape(T, N, -1)
        ests = filt.forward_loop_train_hoisted(feats, modw, controls)
        loss = torch.mean((ests - targets) ** 2)
        loss.backward()
        if in_graph:
            reduce_(grads.flat)  # ncclAllReduce (avg) on this stream
        return loss

    def exchange():  # between the two graphs: the process group's all-reduce, stream-ordered after backward
        if world > 1 and not in_graph:
            dist.all_reduce(grads.flat, op=dist.ReduceOp.SUM)

    def update():
        if world > 1 and not in_graph:
            grads.flat.mul_(1.0 / world)
        opt.step()

    def step():
        loss = forward_backward()
        exchange()
        update()
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    graph, static_loss, eager_ms, launch = None, None, None, "eager"
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):  # every backward runs on `side`: autograd's AccumulateGrad nodes stay there
        for _ in range(max(3, warmup)):  # also warms the NCCL communicator on this stream before any capture
            step()
        side.synchronize()
        assert grads.intact(), "a parameter gradient left the flat buffer"
        ops.PROFILE.reset(enabled=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step()
        e1.record()
        prof = ops.PROFILE.collect()
        ops.PROFILE.reset(enabled=False)
        eager_ms = e0.elapsed_time(e1)
        graph2 = None
        if not os.environ.get("MMF_BENCH_NO_GRAPH"):
            try:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    static_loss = forward_backward()
                    if world == 1 or in_graph:
                        update()
                if world > 1 and not in_graph:
                    graph2 = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph2, stream=side):
                        update()
                graph.replay()  # first replay outside the timed region
                if graph2 is not None:
                    exchange()
                    graph2.replay()
                side.synchronize()
                launch = ("one CUDA graph per training step" if world == 1 else
                          "one CUDA graph per training step (ncclAllReduce inside)" if in_graph else
                          "two CUDA graphs per training step (zero + forward + backward | scale + Adam), the NCCL all-reduce "
                          "enqueued between them on the same stream")
            except Exception as exc:
                print(f"[bench] rank {rank}: CUDA-graph capture of the training step failed ({type(exc).__name__}: {exc})",
                      file=sys.stderr, flush=True)
                if world == 1:  # a failed capture leaves the generator / stream state unusable: start over without it
                    os.environ["MMF_BENCH_NO_GRAPH"] = "1"
                    os.execv(sys.executable, [sys.executable] + sys.argv)
                raise
    torch.cuda.current_stream().wait_stream(side)
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk, torch.cuda.stream(side):
        start.record()
        for _ in range(steps):
            if graph is not None:
                graph.replay()
                if graph2 is not None:
                    exchange()
                    graph2.replay()
            else:
                loss = step()
        if graph is not None:
            loss = static_loss
        stop.record()
        side.synchronize()
        barrier()
    ms = max_over_ranks(start.elapsed_time(stop), dev) / steps
    units = N * Mp * T
    kern = {k: {"avg_ms": v["avg_ms"], "share_of_eager_step": v["total_ms"] / eager_ms} for k, v in prof["kernels"].items()}
    record = {
        "metric": "particle-steps/sec", "value": world * units / (ms / 1e3), "unit": "particle-steps/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": filt.precision, "data": "synthetic",
        "config": {"workload": cfg, "id": "c4", "model": name, "trajectories_per_gpu": N, "particles": Mp,
                   "filter_steps_per_pass": T, "phases": "forward + backward + grad all-reduce + Adam",
                   "encoders": "hoisted and frozen (features are inputs)", "final_loss": float(loss.detach()),
                   "launch": launch, "eager_ms_per_step": eager_ms,
                   "allreduce": {"elements": int(grads.flat.numel()), "bytes": int(grads.flat.numel()) * 4,
                                 "ranks": world, "how": ("none (1 rank)" if world == 1 else
                                                        "ncclAllReduce (avg, fp32, in place on the flat gradient buffer) "
                                                        "captured on the step's stream" if in_graph else
                                                        "torch.distributed NCCL all_reduce (sum, fp32, in place on the flat "
                                                        "gradient buffer) between the step's two graphs")}},
        "clocks": clk.summary(), "gpu_launches": prof["launches"] * steps, "kernels": kern,
        "e2e": {"value": world * units / (ms / 1e3), "unit": "particle-steps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 4, "note": "training step is device-resident; loss scalar read back"},
    }
    if reduce_ is not None:
        reduce_.close()
    del graph, graph2
    return record


def bptt_arm(args):
    import torch.distributed as dist

    ctx = setup_ranks(args)
    record = run_c4(ctx, args.steps, args.warmup, args.precision)
    if ctx[1] == 0:
        print(json.dumps(record), flush=True)
    if ctx[0] > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------
def sweep_arm(args):
    """BASELINE config C5: particle-count sweep M = 1K ... 1M at 16K trajectories (sharded over the ranks).
    16K x 1M particles do not fit one GPU (196 GB of state), so the trajectories are TILED (tile-of-trajectories outer,
    time inner: legal because trajectories are independent); a "step" here times a bounded number of tiles per M
    (up to 2 tiles x 10 filter steps -- BASELINE.md's step count --, a tile holds up to 134 M particles) and reports
    particle-steps/s per M -- tiles are independent and identical, so the rate of the full 16K-trajectory sweep point is
    the same number.  value = geometric mean.  The trajectories are sharded over the ranks (strong scaling: 16K total)."""
    import torch.distributed as dist

    from multimodalfilter_b200 import _lib
    from multimodalfilter_b200.crossmodal import models as M_
    from multimodalfilter_b200.synthetic import fill_parameters

    world, rank, local_rank, dev = setup_ranks(args)
    name, sd, N_total, _, T, cfg = WORKLOADS["c5"]
    n_rank = N_total // world
    filt = fill_parameters(M_.MODEL_TYPES["push"][name](), seed=0).to(dev).eval()
    filt.precision = args.precision or "bf16x3"
    filt.resample_mode = args.resample_mode
    plan = filt.fused_plan()
    g = torch.Generator(device=dev).manual_seed(rank)
    points = []
    for Mp in (1024, 4096, 16384, 65536, 262144, 1048576):
        n_tile = max(1, min(n_rank, (1 << 27) // Mp))
        tiles = min(2 if Mp < 262144 else 1, max(1, n_rank // n_tile))
        filt.num_particles = Mp
        mean = torch.randn(n_tile, sd, device=dev, generator=g)
        cov = (torch.eye(sd, device=dev) * 0.1)[None].expand(n_tile, sd, sd).contiguous()
        feats = [torch.randn(T, n_tile, 64, device=dev, generator=g), torch.randn(T, n_tile, 128, device=dev, generator=g)]
        controls = torch.randn(T, n_tile, 7, device=dev, generator=g)

        def one_pass():
            with torch.no_grad():
                for _ in range(tiles):
                    filt.initialize_beliefs(mean=mean, covariance=cov)
                    for t in range(T):
                        filt.forward(observations=None, controls=controls[t], _hoisted=([f[t] for f in feats], None))

        for _ in range(max(1, args.warmup)):
            one_pass()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            one_pass()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        rate = world * tiles * n_tile * Mp * T / (float(ms) / 1e3)
        points.append({"particles": Mp, "trajectories_per_tile": n_tile, "tiles_timed": tiles, "ms": float(ms),
                       "particle_steps_per_s": rate})
        del mean, cov, feats, controls
        filt.particle_states = filt.particle_log_weights = None
        torch.cuda.empty_cache()
    if rank == 0:
        import math
        value = math.exp(sum(math.log(p["particle_steps_per_s"]) for p in points) / len(points))
        print(json.dumps({
            "metric": "particle-steps/sec", "value": value, "unit": "particle-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sum(p["ms"] for p in points),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": filt.precision,
            "data": "synthetic",
            "config": {"workload": cfg, "id": "c5", "model": name, "trajectories_total": N_total,
                       "filter_steps_per_tile": T, "resample": args.resample_mode,
                       "note": "value = geometric mean over the sweep; bounded tiles per point, see sweep"},
            "sweep": points,
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=None, choices=["fp32", "bf16x3", "bf16"])
    ap.add_argument("--resample-mode", default="multinomial")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (workloads c1, c2, c3)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("c4", "c5")):
        ap.error("--dump-outputs covers the forward workloads c1, c2 and c3 of --impl b200")
    if os.environ.get("MMF_BENCH_WATCHDOG_S"):  # diagnosis of a hung rank: dump every thread's stack and exit
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["MMF_BENCH_WATCHDOG_S"]), exit=True)
    assert args.warmup >= 3 or args.impl == "reference" or os.environ.get("MMF_BENCH_ALLOW_SHORT"), "W >= 3 warm-up steps"

    if args.impl == "reference":
        return reference_arm(args)
    if args.workload == "c4":
        return bptt_arm(args)
    if args.workload == "c5":
        return sweep_arm(args)

    import torch.distributed as dist

    from multimodalfilter_b200 import _lib, ops
    from multimodalfilter_b200.crossmodal import models as M_
    from multimodalfilter_b200.synthetic import fill_parameters

    ctx = setup_ranks(args)
    world, rank, local_rank, dev = ctx

    name, sd, N, Mp, T, cfg = WORKLOADS[args.workload]
    task = "push" if name.startswith("Push") else "door"
    filt = fill_parameters(M_.MODEL_TYPES[task][name](), seed=0).to(dev).eval()
    is_pf = hasattr(filt, "num_particles")
    precision = args.precision or "bf16x3"
    if is_pf:
        filt.num_particles = Mp
        filt.precision = precision
        filt.resample_mode = args.resample_mode
    units_per_pass = N * (Mp if is_pf else 1) * T

    # every rank owns its own N trajectories (seeded by rank): weak scaling, no data-path collective
    states, obs, controls = build_inputs(args.workload, seed=rank)
    cov = (torch.eye(sd, device=dev) * 0.1)[None].expand(N, sd, sd).contiguous()
    host_obs = {k: v[1:].contiguous().pin_memory() for k, v in obs.items()}
    host_controls = controls[1:].contiguous().pin_memory()
    host_mean0 = states[0].contiguous().pin_memory()
    h2d_bytes = sum(v.numel() * v.element_size() for v in host_obs.values()) + host_controls.numel() * 4 + host_mean0.numel() * 4
    host_out = torch.empty((T, N, sd), dtype=torch.float32).pin_memory()
    d2h_bytes = host_out.numel() * 4

    dev_obs = {k: v.to(dev) for k, v in host_obs.items()}
    dev_controls = host_controls.to(dev)
    dev_mean0 = host_mean0.to(dev)

    # ---- device-resident pass: hoisted features computed once, outside the timed region ---------------
    if is_pf:
        plan = filt.fused_plan()
        assert plan is not None
        with torch.no_grad():
            feats, modw = filt.hoist_observations(plan, dev_obs, T, N)
        del dev_obs
        torch.cuda.empty_cache()

        def resident_pass():
            with torch.no_grad():
                filt.initialize_beliefs(mean=dev_mean0, covariance=cov)
                est = filt.forward_loop_hoisted(feats, modw, dev_controls)  # graph replay when the problem is small
            return est
    else:
        filters = list(filt.filter_models)
        with torch.no_grad():
            zr = [f.sense_sequence(dev_obs, T, N) for f in filters]
            z = torch.stack([a[0] for a in zr])
            r = torch.stack([a[1] for a in zr])
            beta = filt._sequence_weights(dev_obs, T, N, dev).transpose(0, 1).contiguous()
        del dev_obs
        torch.cuda.empty_cache()

        def resident_pass():
            with torch.no_grad():
                filt.initialize_beliefs(mean=dev_mean0, covariance=cov)
                means, covs = filt._advance(filters, dev_controls, z, r)
                return ops.kf_fuse_crossmodal(means, covs, beta)  # fused means, fused covariances

    def e2e_pass():
        with torch.no_grad():
            # PF: forward_loop takes the pinned host observations and streams them in behind the encoders
            o = host_obs if is_pf else {k: v.to(dev, non_blocking=True) for k, v in host_obs.items()}
            c = host_controls.to(dev, non_blocking=True)
            m0 = host_mean0.to(dev, non_blocking=True)
            filt.initialize_beliefs(mean=m0, covariance=cov)
            est = filt.forward_loop(observations=o, controls=c)
            host_out.copy_(est, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        barrier()
        ops.PROFILE.reset(enabled=profile)
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = None
        with ClockSampler(local_rank) as clk:
            start.record()
            for _ in range(steps):
                out = fn()
            stop.record()
            barrier()
        ms = start.elapsed_time(stop)
        prof = ops.PROFILE.collect() if profile else None
        ops.PROFILE.reset(enabled=False)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / steps, clk.summary(), prof, out

    # inputs per pass (>= 100 MB of particle state + features) exceed nothing like L2 reuse across passes:
    # every step rewrites the N*M particle set (C3: 49 MB states+weights per step, new noise each step).
    torch.manual_seed(rank)  # the device noise of every pass: the same draws from run to run
    ms_resident, clocks, prof, last = timed(resident_pass, args.steps, args.warmup, profile=True)
    if args.dump_outputs and rank == 0:
        if is_pf:
            dump_outputs(args.dump_outputs, {"estimates": last, "particle_states": filt.particle_states,
                                             "particle_log_weights": filt.particle_log_weights})
        else:
            dump_outputs(args.dump_outputs, {"estimates": last[0], "covariances": last[1]})
    # kernel-level numbers: the same kernels launched step by step (one C call per kernel, CUDA events around each on the
    # launching stream) instead of through the whole-sequence call, which offers no place to put an event
    ms_profiled = None
    if is_pf:
        filt.whole_loop = False
        saved_graph, filt.graph_max_particles = filt.graph_max_particles, 0
        ms_profiled, _, prof_k, _ = timed(resident_pass, args.steps, 1, profile=True)
        filt.whole_loop, filt.graph_max_particles = True, saved_graph
        prof["kernels"].update(prof_k["kernels"])
    # same step / warm-up counts as `value` (small workloads capture their CUDA graph on the second call: warm-up)
    ms_e2e, clocks_e2e, _, _ = timed(e2e_pass, args.steps, args.warmup)

    # ---- the HBM-bound kernel of the step, stand-alone, per resampling mode (north star: >= 60 % of the HBM roofline) ----
    hbm_modes = None
    if is_pf and args.workload == "c3":
        hbm_modes = time_resample_modes(N, Mp, sd, dev)

    value = world * units_per_pass / (ms_resident / 1e3)
    e2e_value = world * units_per_pass / (ms_e2e / 1e3)

    line = {
        "metric": "particle-steps/sec", "value": value, "unit": "particle-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_resident, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if precision == "fp32" else precision,
        "data": "synthetic",
        "config": {"workload": cfg, "id": args.workload, "model": name, "trajectories_per_gpu": N, "particles": Mp,
                   "filter_steps_per_pass": T, "resample": args.resample_mode if is_pf else None,
                   "precision": precision,
                   "recursion": ("one launch for all T steps (k_pf_loop_small: a CTA per trajectory, particle set in shared memory, "
                                 "layers on mma.sync with split bf16 operands; fp32 CUDA cores at precision fp32)"
                                 if is_pf and _lib.load().mmf_pf_forward_loop_persistent(N, Mp) else
                                 "mmf_pf_forward_loop: 1 + 2 T launches" if is_pf else "k_ekf_loop: one launch for all T steps"),
                   "l2": "working set per filter step (particle states + weights + noise, C3: 115 MB) exceeds nothing "
                         "cached across passes: inputs larger than L2 over a pass; no explicit flush"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "particle-steps/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes, "clocks": clocks_e2e},
        "gpu_launches": prof["launches"] if prof else 0,
    }

    # ---- BASELINE config C4 at the same rank count: the path's only collective (gradient all-reduce) ----------------
    if args.workload == "c3" and not os.environ.get("MMF_BENCH_NO_TRAINING"):
        del feats, modw
        filt.particle_states = filt.particle_log_weights = None
        torch.cuda.empty_cache()
        try:
            tr = run_c4(ctx, args.steps, args.warmup, args.precision)
            line["training"] = {k: tr[k] for k in ("value", "unit", "n_gpus", "ms_per_step", "steps", "dtype", "config", "clocks")}
            line["training"]["kernels"] = tr["kernels"]
        except Exception as exc:  # the forward line above is measured: a failing training record must not take it down
            print(f"[bench] rank {rank}: training record failed ({type(exc).__name__}: {exc})", file=sys.stderr, flush=True)
            line["training"] = {"unavailable": f"{type(exc).__name__}: {exc}"[:300]}
    if rank == 0:
        peaks = measured_peaks()
        line["config"]["e2e_timing"] = "same steps / warm-up as value"
        if is_pf and prof and prof["kernels"].get("pf_predict_measure"):
            k = prof["kernels"]["pf_predict_measure"]
            flops = FLOP_PER_PARTICLE_STEP[sd] * N * Mp
            achieved = flops / (k["avg_ms"] / 1e3) / 1e12
            line["roofline"] = {
                "kernel": "k_particle_chain (mmf_pf_predict_measure)", "bound": "tensor", "achieved": achieved,
                "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"],
                "traffic": ncu_traffic("prof_chain_ws") if args.workload == "c3" and precision == "bf16x3" else None, "traffic_unit": "dram bytes per launch (ncu --set full, C3 step)",
                "peak_source": f"{peaks['source']} bf16 sustained", "avg_launch_ms": k["avg_ms"],
                "share_of_step": k["avg_ms"] * T / ms_resident,
                "timed_in": "a pass that launches the kernels step by step (CUDA events per launch); value / ms_per_step "
                            "come from the whole-sequence call (mmf_pf_forward_loop)", "ms_per_step_profiled_pass": ms_profiled,
                "other_kernels": {n: {"avg_ms": v["avg_ms"], "count_per_pass": v["count"] / args.steps,
                                      "share": v["avg_ms"] * v["count"] / args.steps / ms_resident}
                                  for n, v in prof["kernels"].items() if n not in ("pf_predict_measure", "pf_forward_loop")},
            }
            nr = prof["kernels"].get("pf_normalize_resample")
            if nr:
                systematic = args.resample_mode.startswith("systematic")
                bytes_ = N * Mp * (8 + 8 * sd + (0 if systematic else 8))  # logw r/w, states r/w, fp64 uniform (BASELINE.md section 4)
                line["roofline"]["hbm_kernel"] = {
                    "kernel": "mmf_pf_normalize_resample inside the step", "mode": args.resample_mode, "bound": "hbm",
                    "achieved": bytes_ / (nr["avg_ms"] / 1e3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": bytes_ / (nr["avg_ms"] / 1e3) / 1e9 / peaks["hbm_gbs"], "avg_launch_ms": nr["avg_ms"]}
                if hbm_modes:
                    for m in hbm_modes.values():
                        m["frac"] = m["achieved"] / peaks["hbm_gbs"]
                    line["roofline"]["hbm_kernel"]["standalone_by_mode"] = hbm_modes
        elif prof and prof["kernels"].get("ekf_loop"):
            k = prof["kernels"]["ekf_loop"]
            bytes_ = 340.0 * N * T  # BASELINE.md section 4: 340 B / trajectory-step (K=2, sd=3)
            achieved = bytes_ / (k["avg_ms"] / 1e3) / 1e9
            line["roofline"] = {"kernel": "k_ekf_loop", "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"],
                                "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": None,
                                "avg_launch_ms": k["avg_ms"],
                                "note": "latency/parallelism-bound by construction at N=256 (SURVEY.md section 7.6)"}
        if not args.no_cpu_baseline:
            torch.set_num_threads(os.cpu_count() or 1)
            n_s, t_s = CPU_SAMPLE.get(args.workload, (min(N, 32), min(T, 50)))
            rate, sample, dt = run_cpu_oracle(args.workload, n_s, t_s)
            line["cpu_baseline"] = {"value": rate, "unit": "particle-steps/s", "cores": torch.get_num_threads(),
                                    "kind": "port", "sample": sample, "seconds": dt}
            if world == 1:
                # BASELINE.md section 5.4: the oracle with eager torch on this B200 -- "the reference on this box"
                try:
                    n_g, t_g = GPU_EAGER_SAMPLE.get(args.workload, (min(N, 256), min(T, 50)))
                    rate, sample, dt = run_cpu_oracle(args.workload, n_g, t_g, device=str(dev))
                    line["gpu_eager_baseline"] = {"value": rate, "unit": "particle-steps/s", "kind": "port", "sample": sample,
                                                  "seconds": dt, "speedup_e2e": e2e_value / rate}
                except Exception as exc:  # the oracle is test infrastructure: never let it take the bench line down
                    line["gpu_eager_baseline"] = {"unavailable": f"{type(exc).__name__}: {exc}"[:300]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
