#!/usr/bin/env python
"""bench.py -- rendered frames/sec of the ENeRF render-time hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c4|c5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Workloads (BASELINE.json configs; one "step" = one full frame through the drop-in Network.forward):
  c2 (default, the metric's configuration, README.md:114 of the reference): 512x640, 3 source views, 48+8 depth
     planes, 2-level cascade, render_if [False, True]                                   -> enerf_b200.network
  c4: 1024x1024 ZJU-MoCap shape, 4 source views, 48+8 planes, rays masked by mask_at_box -> enerf_b200.network_human
  c5: 1920x1088 ENeRF-Outdoor shape (1080 is not /32), 6 source views, 3 foreground layers + background,
      planes [32,8] (+ background [16,4]), samples [2,1]                                 -> enerf_b200.network_composite
Random-init weights with randomised BN statistics, synthetic inputs (enerf_b200/synthetic.py).

Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  roofline          the fused MLP + compositing ray kernel (the north-star kernel): algorithmic FLOPs / CUDA-event time
  roofline_families the same arithmetic for the tcgen05 convolution stacks and the cost volumes
  cpu_baseline      the CPU oracle (port of the reference's PyTorch path) on this box's host cores (bounded sample)
  library_baseline  the same oracle port run on cuda:0 = the reference's formulation on torch's cuDNN/cuBLAS kernels
  e2e               the same metric through the public API with HOST (pinned) inputs and outputs
  fp32_mode         the exact FP32-pipe mode next to the default (TF32 tensor-core operands, fp32 accumulate)
  config.single_frame_fps  one frame at a time, device resident (how run.py:57-76 measures); `value` is the
                    throughput with `frames_in_flight_per_gpu` frames rendered concurrently
At N > 1 `value` is frame-parallel sequence rendering (every rank renders its own frames; no data-path collective)
and, for c2, `config.intra_frame` holds the north-star layout measured in the same run: row-band sharding of the
level-1 cost volume / CostRegNet / rays with ONE NCCL all-gather (latency of a single frame, Amdahl bound beside it).
`--impl reference` times the reference's CPU path (the oracle port: the Python reference tree cannot travel to the
GPU box) on the same config and prints the same line with "impl": "reference".
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

import torch  # noqa: E402

PUBLISHED_FPS = 21.78          # BASELINE.md section 1: RTX 3090, trained weights, DTU (README.md:121); c2 only
DTYPE = "tf32-operands/fp32-accumulate"

WORKLOADS = {
    "c2": dict(H=512, W=640, S=3, planes=(48, 8), kind="plain",
               metric="rendered frames/sec @512x640, 3 src views, 48/8 planes",
               desc="512x640, 3 src views, 48+8 planes, 2-level cascade, render_if [F,T] (BASELINE.json configs[1])"),
    "c4": dict(H=1024, W=1024, S=4, planes=(48, 8), kind="human",
               metric="rendered frames/sec @1024x1024, 4 src views, 48/8 planes, masked rays",
               desc="1024x1024 ZJU-MoCap shape, 4 src views, 48+8 planes, network_human with mask_at_box (BASELINE.json configs[3])"),
    "c5": dict(H=1088, W=1920, S=6, planes=(32, 8), kind="composite",
               metric="rendered frames/sec @1920x1088, 6 src views, 3 foreground layers + background",
               desc="1920x1088 (1080 padded to /32) ENeRF-Outdoor shape, 6 src views, network_composite: 3 fg layers [32,8] planes "
                    "+ background [16,4], samples [2,1], both levels rendered (BASELINE.json configs[4])"),
}


def stage_work(h, w, s, d0, d1, ray_fraction=1.0):
    """Per-frame algorithmic work of each stage of the plain / human network (BASELINE.md section 2, the
    reference formulation; bytes = each tensor read once / written once, SURVEY.md section 8d)."""
    px = h * w
    sc, sv = px / (512 * 640), s / 3.0
    return {
        "feature_net": {"flops": 14896.0 * s * px, "bytes": (11.8 + 55.1) * 1e6 * sc * sv},
        "cost_volume_0": {"flops": 0.2e9 * sc * sv, "bytes": (7.9 * sv + 31.5 * d0 / 48) * 1e6 * sc},
        "cost_reg_0": {"flops": 357.75 * d0 * px, "bytes": (31.5 + 8.8) * 1e6 * sc * d0 / 48},
        "cost_volume_1": {"flops": 0.3e9 * sc * sv, "bytes": (15.8 * sv + 41.9 * d1 / 8) * 1e6 * sc},
        "cost_reg_1": {"flops": 4212.0 * d1 * px, "bytes": (41.9 + 23.6) * 1e6 * sc * d1 / 8},
        "render_rays_1": {"flops": 2.0 * px * ray_fraction * (15576.0 * s + 4224.0),
                          "bytes": (10.5 + 21.0 + (31.5 + 11.8) * sv + 0.7 + 7.9) * 1e6 * sc * ray_fraction},
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[0]))
                mx = max(mx, float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained"), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def build_problem(workload, seed=2):
    """(cfg, net on CPU in eval mode, CPU batch in the reference's contract, info)."""
    from enerf_b200 import config as cfg_mod, synthetic
    wl = WORKLOADS[workload]
    if wl["kind"] == "composite":
        cfg, batch = synthetic.c5_case(seed=seed)
        cfg_mod.set_cfg(cfg)
        from enerf_b200.network_composite import Network
    elif wl["kind"] == "human":
        cfg, batch = synthetic.c4_case(seed=seed)
        cfg_mod.set_cfg(cfg)
        from enerf_b200.network_human import Network
    else:
        cfg = cfg_mod.set_cfg(cfg_mod.make_cfg(volume_planes=list(wl["planes"]), render_if=[False, True]))
        batch = synthetic.make_batch(wl["H"], wl["W"], wl["S"], cfg, seed=seed)
        batch.pop("rays_0", None)      # level 0 is not rendered (render_if False): the reference never reads it either
        from enerf_b200.network import Network
    torch.manual_seed(0)
    net = Network().eval()
    synthetic.randomize_bn_(net, seed=1)
    return cfg, net, batch, wl


def oracle_forward(kind):
    from oracle import enerf_oracle as O
    from oracle import enerf_oracle_composite as OC
    if kind == "composite":
        return lambda sd, cfg, batch: OC.forward(sd, cfg, batch)
    return lambda sd, cfg, batch: O.forward(sd, cfg, batch, human=(kind == "human"))


def cpu_reference_run(kind, cfg, sd, batch, frames, warmup=1, budget_s=240.0):
    """The reference's CPU PyTorch path (oracle port) on this box's host cores.  torch's CPU conv / grid_sample
    kernels slow down badly when oversubscribed (128 threads: 34 s/frame on the GPU box), so the thread count is
    the best of a short probe over {16, 32, 64, all}.  Returns (fps, out, threads, frames actually timed)."""
    fwd = oracle_forward(kind)
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (16, 32, 64, ncpu) if c <= ncpu}) or [ncpu]
    best, best_t, out = None, float("inf"), None
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            t0 = time.perf_counter()
            out = fwd(sd, cfg, batch)                      # first call at this thread count doubles as warm-up
            t1 = time.perf_counter()
            if t1 - t0 > 20.0:                             # large workloads (c4 / c5): one frame per candidate is enough
                dt = t1 - t0
            else:
                out = fwd(sd, cfg, batch)
                dt = time.perf_counter() - t1
            if dt < best_t:
                best, best_t = c, dt
            if dt > 3 * best_t:
                break                                      # oversubscribed: larger counts only get worse
        torch.set_num_threads(best)
        frames = max(1, min(frames, int(budget_s / max(best_t, 1e-3))))
        for _ in range(max(0, min(warmup, 2) - 1)):
            fwd(sd, cfg, batch)
        t0 = time.perf_counter()
        for _ in range(frames):
            out = fwd(sd, cfg, batch)
        dt = time.perf_counter() - t0
    return frames / dt, out, best, frames


def run_reference_arm(args, rank):
    if rank != 0:
        return
    cfg, net, batch, wl = build_problem(args.workload)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    fps, out, n_thr, frames = cpu_reference_run(wl["kind"], cfg, sd, batch, args.steps, warmup=args.warmup)
    if args.dump_outputs:
        dump_outputs(host_outputs(out), args.dump_outputs)
    line = {
        "impl": "reference", "metric": wl["metric"], "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": frames,
        "warmup": min(args.warmup, 2), "ms_per_step": 1000.0 / fps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": fps / PUBLISHED_FPS if args.workload == "c2" else None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"]},
        "note": "reference CPU PyTorch path restated in oracle/ (the Python reference tree does not travel to the GPU box); "
                f"requested steps {args.steps}, timed {frames} (bounded to ~4 min of CPU work)",
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": os.cpu_count(), "threads": n_thr, "kind": "port",
                         "sample": f"{frames} full frames, torch {torch.__version__} CPU, {n_thr} threads (best of a probe over 16/32/64/all)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_REAL_STDOUT = None


def _protect_stdout():
    """Everything the process (NCCL banners included) writes to fd 1 goes to stderr; the single JSON
    line is written to the original stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def to_dev(batch, dev):
    return {k: (v.to(dev) if torch.is_tensor(v) and k != "bbox" else v) for k, v in batch.items()}


DUMP_BYTES = 60 * 10**6       # array data of --dump-outputs: keeps the directory under 64 MB with the .npy headers


def host_outputs(out):
    """The tensors of a forward's output dict on the host: float64 stays float64 and integer outputs become float64
    (exact), everything else float32."""
    res = {}
    for k, v in out.items():
        if torch.is_tensor(v):
            v = v.detach().cpu()
            wide = v.dtype == torch.float64 or not (v.is_floating_point() or v.dtype == torch.bool)
            res[k] = v.double() if wide else v.float()
    return res


def dump_outputs(outs, path):
    """Writes every array of ``outs`` as <path>/<name>.npy.  When they hold more than DUMP_BYTES together, each array is
    cut to the same fraction of its elements: flattened, at sorted indices drawn with a fixed seed, so that runs and
    builds with the same arguments dump the same elements."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    total = sum(v.numel() * v.element_size() for v in outs.values())
    frac = min(1.0, DUMP_BYTES / total) if total else 1.0
    for k, v in outs.items():
        if frac < 1.0:
            flat = v.reshape(-1)
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:int(flat.numel() * frac)]
            v = flat[idx.sort().values]
        np.save(os.path.join(path, k + ".npy"), v.numpy())
    print(f"[bench] {len(outs)} output(s) written to {path}" + (f" (seeded sample of {frac:.3f} of each)" if frac < 1.0 else ""),
          file=sys.stderr)


def timed_events(fn, steps, flush_buf=None):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        if flush_buf is not None:
            flush_buf.zero_()            # L2 flush between timed iterations (not timed)
        a.record()
        fn()
        b.record()
    return ev


def main():
    _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip fp32_mode / library_baseline / intra_frame (profiling runs)")
    ap.add_argument("--graph", type=int, default=1, help="replay the forward as a CUDA graph (0 = eager launches)")
    ap.add_argument("--inflight", type=int, default=4, help="frames rendered concurrently per GPU (one CUDA graph + stream each); "
                    "1 = strictly one frame at a time (latency mode)")
    ap.add_argument("--host-rays", type=int, default=0, help="1: ship rays_1 from the host like the reference's data layer (default: generate on device)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the output tensors of the last one as DIR/<name>.npy "
                    "(float32 / float64, 64 MB at most: larger outputs are replaced by a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    from enerf_b200 import dist as edist
    rank, local, world = edist.init_from_env()
    if args.impl == "reference":
        run_reference_arm(args, rank)
        if world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    from enerf_b200 import capi, config as cfg_mod, synthetic
    import torch.distributed as dist
    from enerf_b200.pipeline import GraphedNetwork, StreamedRenderer

    # rank r renders its own frame of the sequence (different image content, same rig)
    cfg, net, batch, wl = build_problem(args.workload, seed=2 + (rank if world > 1 else 0) * 10)
    kind, H, W, S = wl["kind"], wl["H"], wl["W"], wl["S"]
    sd_cpu = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.to(dev)
    # the data layer's rays_{i} (10.5 MB/frame at c2) are not shipped: rays are generated on device from tar_ext / tar_ixt
    # (SURVEY 8f row f3); `--host-rays 1` restores the reference's batch contract
    batch_full = dict(batch)                       # the CPU oracle still takes the reference's full batch
    if not args.host_rays:
        for k in [k for k in batch if k.startswith("rays_")]:
            batch.pop(k)
    gbatch = to_dev(batch, dev)
    # network_human: the reference's boolean indexing implies a host read-back of the masked-ray count; the drop-in's
    # `static_mask` mode keeps the count on the device (kernels sized for the full frame stop at it), which makes the
    # forward graph-capturable.  Outputs are the reference's, with depth / weights padded to the full ray count.
    if kind == "human":
        net.static_mask = bool(args.graph)
    graphable = bool(args.graph)

    flush_buf = torch.empty(256 * 1024 * 1024 // 4, device=dev)   # 256 MiB > 126 MB L2
    l0 = capi.LAUNCHES
    with torch.no_grad():
        net(gbatch)
    launches_per_forward = capi.LAUNCHES - l0
    # `inflight` frames are rendered concurrently (sequence rendering): replica j has its own captured graph (with its
    # own scratch buffers), stream and static inputs / outputs; a step = one frame on every replica
    nfl = max(1, args.inflight) if graphable else 1
    main_stream = torch.cuda.current_stream()
    replicas = []
    for j in range(nfl):
        st = torch.cuda.Stream(device=dev) if j > 0 else main_stream
        with torch.cuda.stream(st):
            g = GraphedNetwork(net, gbatch) if graphable else None
        replicas.append((st, g, torch.cuda.Event()))
    torch.cuda.synchronize()

    def one_frame():
        with torch.no_grad():
            return replicas[0][1].replay() if replicas[0][1] is not None else net(gbatch)

    def step():
        """one frame per replica, concurrently; all joined back on the main stream"""
        if nfl == 1:
            return one_frame()
        fork = torch.cuda.Event()
        fork.record(main_stream)
        for st, g, done in replicas:
            if st is not main_stream:
                st.wait_event(fork)
            with torch.cuda.stream(st):
                out_j = g.replay()
                if st is not main_stream:
                    done.record(st)
        for st, g, done in replicas[1:]:
            main_stream.wait_event(done)
        return out_j

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    # ---- headline: device-resident throughput ----
    last = {}

    def timed_step():
        last["out"] = step()

    for _ in range(args.warmup):
        step()
    sync_all()
    with ClockSampler(local) as clk:
        sync_all()
        ev = timed_events(timed_step, args.steps, flush_buf)
        sync_all()
    if args.dump_outputs and rank == 0:
        dump_outputs(host_outputs(last["out"]), args.dump_outputs)
    times = [a.elapsed_time(b) for a, b in ev]
    (total_ms,) = max_over_ranks([sum(times)])
    frames_per_step = nfl * world
    ms_per_step = total_ms / args.steps
    value = frames_per_step * 1000.0 / ms_per_step
    times.sort()
    # one frame at a time (nothing else in flight): how run.py:57-76 measures
    for _ in range(3):
        one_frame()
    sync_all()
    ev1 = timed_events(one_frame, min(args.steps, 20), flush_buf)
    sync_all()
    (lat_ms,) = max_over_ranks([sum(a.elapsed_time(b) for a, b in ev1) / len(ev1)])

    # ---- end to end through the public API with HOST buffers: every frame pays its own H2D (pinned) and D2H (pinned);
    #      StreamedRenderer overlaps copy-in / forward / copy-out of adjacent frames ----
    probe_h = torch.empty(64 * 1024 * 1024, dtype=torch.uint8).pin_memory()
    probe_d = torch.empty(64 * 1024 * 1024, dtype=torch.uint8, device=dev)
    pe = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    probe_d.copy_(probe_h, non_blocking=True)
    torch.cuda.synchronize()
    pe[0].record()
    for _ in range(4):
        probe_d.copy_(probe_h, non_blocking=True)
    pe[1].record()
    for _ in range(4):
        probe_h.copy_(probe_d, non_blocking=True)
    pe[2].record()
    torch.cuda.synchronize()
    host_link = {"h2d_gbs": 4 * 64 / 1024 / (pe[0].elapsed_time(pe[1]) * 1e-3), "d2h_gbs": 4 * 64 / 1024 / (pe[1].elapsed_time(pe[2]) * 1e-3)}
    del probe_h, probe_d
    host_in = {k: (v.clone().pin_memory() if torch.is_tensor(v) and k != "bbox" else v) for k, v in batch.items()}
    h2d = sum(v.numel() * v.element_size() for k, v in host_in.items() if torch.is_tensor(v) and k != "bbox")
    depth = max(2, args.inflight)
    streamed = StreamedRenderer(net, host_in, dev, depth=depth, use_graph=graphable)
    d2h_box = {}

    def on_frame(i, host_out):
        d2h_box["bytes"] = sum(v.numel() * v.element_size() for v in host_out.values() if torch.is_tensor(v))

    streamed.render([host_in] * 4, on_frame)
    sync_all()
    e2e_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    e2e_ev[0].record()
    streamed.render([host_in] * args.steps, on_frame)
    e2e_ev[1].record()
    sync_all()
    e2e_ms = e2e_ev[0].elapsed_time(e2e_ev[1]) / args.steps
    # the plain synchronous loop of run.py:57-76 (copy, forward, copy, sync) for comparison
    sync_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    host_out = None
    n_sync = min(args.steps, 20)
    sync_ev[0].record()
    for _ in range(n_sync):
        with torch.no_grad():
            o = net(to_dev({k: v for k, v in host_in.items()}, dev))
            if host_out is None:
                host_out = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in o.items() if torch.is_tensor(v)}
            for k, v in o.items():
                if torch.is_tensor(v):
                    host_out[k].copy_(v, non_blocking=True)
        torch.cuda.synchronize()
    sync_ev[1].record()
    sync_all()
    e2e_sync_ms = sync_ev[0].elapsed_time(sync_ev[1]) / n_sync
    te = max_over_ranks([e2e_ms, e2e_sync_ms])
    e2e_fps = world * 1000.0 / te[0]     # every rank pushes its own frames end to end
    e2e_sync_fps = world * 1000.0 / te[1]
    d2h = d2h_box.get("bytes", 0)
    del streamed

    # ---- N > 1, c2: the north-star intra-frame layout in the same run (row bands + halo, one all-gather) ----
    intra = None
    if world > 1 and kind == "plain" and not args.no_extras:
        _, _, batch0, _ = build_problem(args.workload, seed=2)       # every rank renders ITS BAND OF THE SAME frame (rank 0's)
        gb0 = to_dev({k: v for k, v in batch0.items() if not k.startswith("rays_")}, dev)
        intra = edist.measure_intra_frame(net, gb0, rank, world, dev, steps=min(args.steps, 20), warmup=args.warmup,
                                          flush_buf=flush_buf, single_frame_ms=lat_ms)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    roofline, families, acc, stage_rates = None, None, {}, None
    if kind != "composite":
        # ---- one profiled pass: per-stage CUDA events (explains `value`, feeds the rooflines) ----
        net.profile = True
        reps = min(10, args.steps)
        for _ in range(reps):
            flush_buf.zero_()
            with torch.no_grad():
                net(gbatch)
            torch.cuda.synchronize()
            for k, v in net.stage_times_ms().items():
                acc[k] = acc.get(k, 0.0) + v / reps
        net.profile = False
        frac_rays = float(batch["mask_at_box"].float().mean()) if kind == "human" else 1.0
        work = stage_work(H, W, S, *wl["planes"], ray_fraction=frac_rays)
        stage_rates = {k: {"ms": round(acc[k], 4), "tflops": round(work[k]["flops"] / (acc[k] * 1e-3) / 1e12, 2),
                           "alg_gbs": round(work[k]["bytes"] / (acc[k] * 1e-3) / 1e9, 1)} for k in work if k in acc}
        traffic_db = {}
        for name in ("r2_traffic.json", "r1_traffic.json"):     # dram__bytes_{read,write}.sum per launch, ncu --set full (c2)
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath):
                traffic_db = json.load(open(tpath))
                traffic_db["_src"] = f"profiles/{name}"
                break

        def tensor_entry(stages, kernel, tkey):
            fl = sum(work[s]["flops"] for s in stages)
            by = sum(work[s]["bytes"] for s in stages)
            ms = sum(acc[s] for s in stages)
            ach = fl / (ms * 1e-3) / 1e12
            tj = traffic_db.get(tkey) if args.workload == "c2" else None
            return {"bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"],
                    "tf32_dense_frac": ach / (peaks["bf16_tflops"] / 2.0), "kernel": kernel, "ms": ms, "algorithmic_flops": fl,
                    "algorithmic_bytes": by, "traffic": ((tj["dram_read_MB"] + tj["dram_write_MB"]) * 1e6 if tj else None),
                    "traffic_src": traffic_db.get("_src") if tj else None, "peak_src": peaks["src"]}

        def hbm_entry(stages, kernel, tkey):
            by = sum(work[s]["bytes"] for s in stages)
            ms = sum(acc[s] for s in stages)
            ach = by / (ms * 1e-3) / 1e9
            tj = traffic_db.get(tkey) if args.workload == "c2" else None
            return {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "kernel": kernel,
                    "ms": ms, "algorithmic_bytes": by, "traffic": ((tj["dram_read_MB"] + tj["dram_write_MB"]) * 1e6 if tj else None),
                    "traffic_src": traffic_db.get("_src") if tj else None, "peak_src": peaks["src"]}

        roofline = tensor_entry(["render_rays_1"], "render_rays_tc_kernel (fused gather + MLP + compositing)", "render_rays_tc")
        roofline["note"] = ("algorithmic FLOPs (reference formulation, BASELINE.md section 2) / CUDA-event time of the launch; tensor peak = measured "
                            "bf16 burst (the contract's denominator); the kernel computes in TF32 (half that rate)")
        families = {
            "tc_conv": tensor_entry(["feature_net", "cost_reg_0", "cost_reg_1"], "tc_conv*_kernel family (FeatureNet + both CostRegNets, "
                                    "incl. their FP32 conv0.0 / lateral kernels)", "tc_conv_family"),
            "cost_volume": hbm_entry(["cost_volume_0", "cost_volume_1"], "cost_volume_kernel<C> (warp + variance, both levels)", "cost_volume_family"),
            "render_rays": dict(roofline),
        }

    # ---- CPU baseline + parity: the oracle port on this box's host cores, bounded sample ----
    cpu_baseline, parity = None, None
    rgb_key = "rgb_level1"
    if not args.no_cpu_baseline and world == 1:
        frames = 3 if args.workload == "c2" else 1
        fps_cpu, ref_out, n_thr, frames = cpu_reference_run(kind, cfg, sd_cpu, batch_full, frames, warmup=1)
        cpu_baseline = {"value": fps_cpu, "unit": "frames/s", "cores": os.cpu_count(), "threads": n_thr, "kind": "port",
                        "sample": f"{frames} full frame(s) of the same workload; oracle/ (torch {torch.__version__} CPU ops), {n_thr} threads "
                                  "(best of a probe over 16/32/64/all)"}
        with torch.no_grad():
            o = net(gbatch)
        tgt = torch.rand(ref_out[rgb_key].shape, generator=torch.Generator().manual_seed(5))
        n_valid = ref_out["depth_level1"].shape[1]          # masked path: the compact length (static_mask pads behind it)
        parity = {"psnr_ours_vs_oracle_db": synthetic.psnr(o[rgb_key].cpu(), ref_out[rgb_key]),
                  "delta_psnr_db": synthetic.psnr(o[rgb_key].cpu(), tgt) - synthetic.psnr(ref_out[rgb_key], tgt),
                  "max_abs_rgb": (o[rgb_key].cpu() - ref_out[rgb_key]).abs().max().item(),
                  "max_abs_depth": (o["depth_level1"].cpu()[:, :n_valid] - ref_out["depth_level1"]).abs().max().item()}

    # ---- the exact mode and the library-kernel baseline (same box, same batch) ----
    fp32_mode, library_baseline = None, None
    if not args.no_extras and world == 1:
        net.precision = "fp32"
        getattr(net, "invalidate_packed", lambda: None)()
        with torch.no_grad():
            o32 = net(gbatch)
            g32 = GraphedNetwork(net, gbatch) if graphable else None
            run32 = (g32.replay if g32 is not None else (lambda: net(gbatch)))
            for _ in range(3):
                run32()
            torch.cuda.synchronize()
            ev32 = timed_events(run32, min(args.steps, 20), flush_buf)
            torch.cuda.synchronize()
        ms32 = sum(a.elapsed_time(b) for a, b in ev32) / len(ev32)
        fp32_mode = {"single_frame_fps": 1000.0 / ms32, "ms": ms32, "dtype": "f32 (FP32-pipe kernels only, ENERF_B200_PRECISION=fp32)"}
        if parity is not None:
            fp32_mode["psnr_vs_oracle_db"] = synthetic.psnr(o32[rgb_key].cpu(), ref_out[rgb_key])
            fp32_mode["max_abs_rgb"] = (o32[rgb_key].cpu() - ref_out[rgb_key]).abs().max().item()
        del g32
        net.precision = "tf32"
        getattr(net, "invalidate_packed", lambda: None)()
        # the reference's formulation on torch's library kernels (cuDNN convs, cuBLAS GEMMs, ATen grid_sample) on this GPU:
        # the oracle port is pure torch, so it runs on cuda:0 unchanged.  TF32 off = the reference's fp32 numerics.
        try:
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            fwd = oracle_forward(kind)
            sd_dev = {k: v.to(dev) for k, v in sd_cpu.items()}
            lb = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in batch_full.items()}
            with torch.no_grad():
                for _ in range(2):
                    fwd(sd_dev, cfg, lb)
                torch.cuda.synchronize()
                n_lib = 5 if args.workload == "c2" else 2
                evl = timed_events(lambda: fwd(sd_dev, cfg, lb), n_lib, flush_buf)
                torch.cuda.synchronize()
            ms_lib = sum(a.elapsed_time(b) for a, b in evl) / len(evl)
            library_baseline = {"value": 1000.0 / ms_lib, "unit": "frames/s", "ms": ms_lib, "kind": "port on cuda:0",
                                "what": f"oracle/ (the reference's PyTorch formulation) on torch {torch.__version__} library kernels "
                                        "(cuDNN / cuBLAS / ATen, fp32, TF32 off), eager, device-resident batch, sync per frame as run.py:62-66"}
            del sd_dev, lb
        except Exception as e:  # noqa: BLE001
            library_baseline = {"unavailable": f"{type(e).__name__}: {e}"[:300]}

    line = {
        "metric": wl["metric"], "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": value / PUBLISHED_FPS if args.workload == "c2" else None, "dtype": DTYPE, "data": "synthetic",
        "config": {"workload": wl["desc"],
                   "single_frame_fps": 1000.0 / lat_ms * world, "single_frame_latency_ms": lat_ms,
                   "single_frame_note": "one frame at a time per GPU, device resident, CUDA-event timed: the reference's own method "
                                        "(run.py:57-76); `value` is the throughput with frames_in_flight_per_gpu frames rendered concurrently",
                   "frames_per_step": frames_per_step, "parallelism": (f"frames x{world} (no data-path collective)" if world > 1 else "single"),
                   "cuda_graph": graphable, "frames_in_flight_per_gpu": nfl,
                   "rays": "host (batch rays_i)" if args.host_rays else "generated on device from tar_ext/tar_ixt",
                   "l2": "256 MiB buffer written between timed iterations (L2 flush)", "timing": "CUDA events per step, max over ranks",
                   "p50_ms": times[len(times) // 2], "p95_ms": times[min(len(times) - 1, int(0.95 * len(times)))],
                   "vs_baseline_note": "published 21.78 FPS is RTX 3090 + trained weights (README.md:121)" if args.workload == "c2" else None},
        "clocks": clk.summary(),
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": te[0],
                "api": f"enerf_b200.pipeline.StreamedRenderer.render (copy-in / compute / copy-out streams, {depth} frames in flight, "
                       f"{'CUDA-graph' if graphable else 'eager'} forward)",
                "sync_loop_value": e2e_sync_fps, "sync_loop_note": "run.py:57-76 style: copy in, Network.forward, copy out, synchronize"},
        "gpu_launches": launches_per_forward * nfl,
        "roofline": roofline,
        "roofline_families": families,
        "cpu_baseline": cpu_baseline,
        "library_baseline": library_baseline,
        "fp32_mode": fp32_mode,
        "stages_ms": {k: round(v, 4) for k, v in acc.items()} or None,
        "stage_rates": stage_rates,
        "host_link": host_link,
    }
    if intra is not None:
        line["config"]["intra_frame"] = intra
    if parity:
        line["parity"] = parity
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
