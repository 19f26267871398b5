#!/usr/bin/env python
"""bench.py -- frames/sec of the volumetric renderer hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision fp16|fp32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is ONE 512x512 frame of the north-star synthetic workload (SURVEY.md section 8d "512x512x128"): head+torso model of the
May configs with bound=4 (3 cascades), all-ones occupancy bitfield, dt_gamma=0, max_steps=128 -> every one of the 262,144
rays composites exactly 128 samples (33,554,432 field evaluations per frame; asserted), plus the 2-D torso field on the lower
image half.  Random-init weights of the exact architecture, synthetic pose/cond (no datasets or checkpoints here).

value  : frames/s, whole job (all ranks), inputs (pose, cond feature window, background) resident in HBM, device-timed with
         CUDA events over exactly K steps between barrier + synchronize; max over ranks.
e2e    : the same metric through the public API with HOST inputs: per step pinned pose+cond -> H2D, cond encoder, fused
         frame, RGB8 frame -> D2H into pinned memory, all inside the timed region.
roofline: dominant kernel = the field kernel (grid gathers + MLPs); achieved = samples/frame x 1536 B (SURVEY.md 8d algorithmic
         gather bytes per head sample) / its CUDA-event time per frame (events recorded inside gf_render_frame on the launch
         stream); peak = MEASURED_PEAKS.json hbm_gbs.  The tables (16 MB) are L2-resident, so this is an "HBM-equivalent"
         gather rate as the metric asks; tensor-pipe fraction is reported beside it.
cpu_baseline: the CPU oracle (port of the reference path, OpenMP + numpy, all host threads) on a bounded sample of the SAME
         frame (rays x 128 samples), extrapolated to frames/s.
--dump-outputs DIR: after the timed steps, what the last timed step returned to its caller (the RGB8 frame and the frame counters)
         is written as DIR/<name>.npy in float32 / float64.  The inputs depend only on the arguments, so two builds can be compared
         output for output.
--impl reference: the reference's CPU implementation timed on the host cores (rank 0 only): the oracle port of the RAD-NeRF
         path on a bounded sample per step; the vanilla AD-NeRF (modules/nerfs) port is reported in `adnerf_cpu`.
"""
import os as _os
# The CPU legs alternate OpenMP regions (C oracle) and OpenBLAS GEMMs (numpy) ~10^3 times per frame sample.  With libgomp's default
# ACTIVE wait policy its idle threads spin between regions and starve the BLAS threads (measured: 6 ms instead of 29 us per GEMM).
# Must be set before libgomp is loaded, i.e. before torch/numpy are imported.
_os.environ.setdefault("OMP_WAIT_POLICY", "passive")
_os.environ.setdefault("GOMP_SPINCOUNT", "0")
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

METRIC = "512x512 frames/sec (head+torso), 128 samples/ray"
HEAD_SAMPLE_BYTES = 1536          # SURVEY.md 8d: 16 lvl x 8 corners x 8 B + 16 lvl x 4 corners x 8 B
HEAD_SAMPLE_FLOP = 178688
TORSO_PIXEL_BYTES = 512
H = W = 512
MAX_STEPS = 128
WORKLOAD = ("RAD-NeRF head+torso (May cfg architecture), 512x512 rays x 128 samples = 33,554,432 field evaluations/frame "
            "(bound=4, 3 cascades, all-ones bitfield, dt_gamma=0, max_steps=128) + torso field on the lower image half")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi sampler (B200_PROFILING.md clocks line).  Started before the warm-up (nvidia-smi takes ~0.5 s to come up);
    only samples whose timestamp falls inside [mark_begin, mark_end] -- the timed region -- are reported."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines, self.t0, self.t1 = gpu_index, None, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        import datetime
        sm, mx, reasons, power = [], None, set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if self.t0 is not None and not (self.t0 - 0.03 <= ts <= self.t1 + 0.03):
                    continue
                sm.append(float(f[2])); mx = float(f[3]); power.append(float(f[4]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------ CPU legs
def host_threads():
    """Threads for the CPU legs.  The port's host loop issues ~128 small numpy/OpenMP regions per frame sample; beyond a few dozen
    threads their fork/join cost dominates (measured on the 128-core GPU host: 2048 rays took 280 s with 128 threads), so the legs
    use min(cores, 32) and report that number."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("GF_CPU_THREADS", "32"))))


def _cpu_port_once(n_rays, threads):
    import numpy as np
    import torch
    from threadpoolctl import threadpool_limits
    torch.set_num_threads(threads)
    from geneface_b200 import synthetic
    from oracle import field as OF
    model, hp = synthetic.build_model(torso=True, bitfield='F', seed=0, sigma_scale=0.25, bound=4, device='cpu')
    sd = synthetic.state_to_numpy(model)
    fi = synthetic.frame_inputs(H, W, device='cpu')
    ro, rd = OF.get_rays(fi['pose'][0].numpy(), fi['intrinsics'], H, W)
    sel = np.linspace(0, H * W - 1, n_rays).astype(np.int64)
    ro, rd = np.ascontiguousarray(ro[sel]), np.ascontiguousarray(rd[sel])
    fo = OF.FieldOracle(sd, bound=4.0)
    OF.MATMUL_DTYPE = np.float32          # timing leg: fp32 GEMMs like the reference's CPU tensors
    with threadpool_limits(limits=threads):
        t0 = time.perf_counter()
        cf = OF.cal_cond_feat(sd, fi['cond'].numpy())
        ws, depth, img, nears, fars, ns = OF.render_head(fo, sd, ro, rd, cf, sd['density_bitfield'], 3, 128, sd['aabb_infer'], hp['min_near'], 0.0, MAX_STEPS)
        bgc = OF.get_bg_coords(H, W)[sel]
        bg, _, _, _ = OF.render_torso_mix(OF.TorsoOracle(sd), sd, bgc, fi['poses6'].numpy(), fi['bg_color'][0].numpy()[sel], img, ws)
        OF.finish(img, ws, depth, nears, fars, bg)
        dt = time.perf_counter() - t0
    OF.MATMUL_DTYPE = np.float64
    assert int(ns.min()) == MAX_STEPS == int(ns.max())
    return dt


CPU_SAMPLE_RAYS = 8192            # FIXED bounded sample of the CPU legs (of 262,144 rays): the ratio against it is repeatable


def cpu_port_fps(n_rays=CPU_SAMPLE_RAYS, threads=None, warm=True):
    """The CPU oracle (port of the reference RAD-NeRF path) on a BOUNDED, FIXED sample of the benchmark frame: `n_rays` rays
    (evenly spread over the image) x 128 samples (head + torso + mix), after one small untimed call (library load, page faults)."""
    threads = threads or host_threads()
    os.environ["OMP_NUM_THREADS"] = str(threads)
    if warm:
        _cpu_port_once(256, threads)
    dt = _cpu_port_once(n_rays, threads)
    fps = 1.0 / (dt * (H * W) / n_rays)
    return fps, dt, threads, f"{n_rays} of 262144 rays x 128 samples of the same frame (head+torso), {dt:.1f} s of CPU work on {threads} threads, extrapolated"


def adnerf_cpu_fps(threads=None):
    """Vanilla AD-NeRF port (BASELINE.json configs[0]: 64x64, 64 coarse + 128 fine samples, 1 frame)."""
    try:
        from oracle import adnerf_port
    except Exception as e:  # noqa: BLE001
        return {"unavailable": str(e)}
    return adnerf_port.time_frame(threads or host_threads())


def run_reference_arm(args, rank):
    """--impl reference: the reference path on the host CPU (rank 0 only)."""
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    t0 = time.perf_counter()
    for _ in range(max(1, warm)):
        _cpu_port_once(256, host_threads())                         # warm-up steps: library load, page faults, thread pools
        if time.perf_counter() - t0 > 30:
            break
    fps_list = []
    for _ in range(steps):
        fps, dt, threads, sample = cpu_port_fps(CPU_SAMPLE_RAYS, warm=False)
        fps_list.append(fps)
    k = len(fps_list)
    value = k / sum(1.0 / f for f in fps_list)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": k, "warmup": 1,
            "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "cpu_sample_rays": CPU_SAMPLE_RAYS, "impl": "CPU port (oracle/) of the reference path", "l2": "n/a (CPU)"},
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "adnerf_cpu": adnerf_cpu_fps(), "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------ GPU arm
CONFIGS = {
    # name: (torso, bitfield, sigma_scale, bound, max_steps, dt_gamma, description)
    "headline": (True, 'F', 0.25, 4, 128, 0.0, WORKLOAD),
    "may_head": (False, 'S', 4.0, 1, 16, 1 / 256, "BASELINE.json configs[1]: RAD-NeRF head (lm3d_radnerf, May cfg) 512x512: bound=1, max_steps=16, dt_gamma=1/256, sphere bitfield"),
    "may_torso": (True, 'S', 4.0, 1, 16, 1 / 256, "BASELINE.json configs[2]: RAD-NeRF head+torso (lm3d_radnerf_torso, May cfg) 512x512: bound=1, max_steps=16, dt_gamma=1/256, sphere bitfield"),
}


def profile_record():
    """ncu-derived numbers of the dominant kernels, written by scripts/ncu_field_json.py from a `ncu --set full` capture of
    this very command and committed under profiles/ (the JSON line never carries a hand-typed counter)."""
    for name in ("r02_field_ncu.json",):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            try:
                return json.load(open(p)), "profiles/" + name
            except Exception:  # noqa: BLE001
                pass
    return None, None


def gather_ubench():
    """scripts/ubench/l2_gather_bw: measured ceiling of 8-byte gathers served by L2/L1 on THIS GPU (a few ms)."""
    exe = os.path.join(ROOT, "scripts", "ubench", "l2_gather_bw")
    if not os.path.exists(exe):
        return None
    try:
        r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001
        return {"unavailable": repr(e)[:120]}


def gather_probe_gbs(model, fi, dev, precision):
    """The field's grid gathers WITHOUT the MLPs on one full round of the benchmark frame (8,388,608 samples: 262,144 rays x 32 slots, in
    the slot-major order of k_march_chunk), through `gf_gather_probe` = the producer warps' own gather code at full occupancy: the
    measured ceiling of this access pattern on this GPU.  Same accounting as roofline.achieved (1,536 B per sample)."""
    import numpy as np
    import torch
    from geneface_b200 import _lib, utils
    N, S = H * W, 32
    rays = utils.get_rays(fi['pose'], fi['intrinsics'], H, W)
    o, d = rays['rays_o'][0], rays['rays_d'][0]
    # every ray enters the bound-4 box at t ~ 1.35 and takes 128 steps of 2 sqrt(3) / 128: slots 0..31 of the first round
    dt = 2 * np.sqrt(3.0) / MAX_STEPS
    t = 1.36 + dt * torch.arange(1, S + 1, device=dev, dtype=torch.float32)
    pts = o[:, None, :] + d[:, None, :] * t[None, :, None]                                     # [N, S, 3] ray-major
    pts = pts.view(N // 32, 32, S, 3).permute(0, 2, 1, 3).reshape(-1, 3).contiguous()          # slot-major inside each 32-ray block
    M = pts.shape[0]
    cf = model.cal_cond_feat(fi['cond'])
    _, _, amb = model.field_forward(pts, torch.zeros_like(pts), cf, precision=precision)
    out = torch.empty(M, 2, device=dev)
    L = _lib.lib()
    handle = model.gf_model()
    for _ in range(2):
        _lib.check(L.gf_gather_probe(handle, _lib.ptr(pts), _lib.ptr(amb), M, _lib.ptr(out), _lib.stream_ptr()))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        _lib.check(L.gf_gather_probe(handle, _lib.ptr(pts), _lib.ptr(amb), M, _lib.ptr(out), _lib.stream_ptr()))
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return {"gbs": M * HEAD_SAMPLE_BYTES / (ms / 1000.0) / 1e9, "ms_per_round": ms, "samples": M,
            "what": "gf_gather_probe: the producers' gather code alone (no MLP, full occupancy) over one 8.4 M-sample round of this frame"}


def dump_outputs(directory, arrays):
    """Write each array as DIR/<name>.npy: integer and float64 data as float64, everything else as float32."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype in (np.int64, np.uint64, np.float64) else np.float32)
        np.save(os.path.join(directory, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("GF_BENCH_PRECISION", "fp16"), choices=["fp16", "fp32"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS) + ["seq300", "train"],
                    help="headline = the BASELINE.json metric's workload (the driver's line); the others are BASELINE.json configs 1/2/3/4")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-may", action="store_true", help="skip the May-configuration / AD-NeRF context measurements")
    ap.add_argument("--eager", action="store_true", help="per-frame eager launches instead of CUDA-graph replay (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (frame configurations only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config in ("seq300", "train")):
        ap.error("--dump-outputs applies to the GPU frame configurations (%s)" % ", ".join(sorted(CONFIGS)))
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    args.warmup = max(args.warmup, 3)
    if args.config == "seq300":
        return run_seq300(args, rank, world, local)
    if args.config == "train":
        return run_train(args, rank, world, local)

    import ctypes
    import numpy as np
    import torch
    import torch.distributed as dist
    from geneface_b200 import _lib, sequence, synthetic
    from geneface_b200.utils import get_audio_features, orbit_pose

    assert torch.cuda.is_available(), "bench.py (ours) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    torso, bitfield, sigma_scale, bound, max_steps, dt_gamma, workload = CONFIGS[args.config]
    headline = args.config == "headline"
    model, hp = synthetic.build_model(torso=torso, bitfield=bitfield, seed=0 if rank == 0 else 100 + rank, sigma_scale=sigma_scale, bound=bound, device=dev)
    bcast_bytes = sequence.broadcast_model_(model, src=0)      # parameters reach every rank through ONE NCCL broadcast
    fi = synthetic.frame_inputs(H, W, device=dev)
    N = H * W
    n_frames = args.steps + args.warmup
    first = rank * n_frames                                    # weak scaling: every rank renders its own K frames of the sequence
    poses = torch.stack([torch.from_numpy(orbit_pose(3.35, 10.0 * np.sin(2 * np.pi * (first + f) / 100.0))) for f in range(n_frames)])
    g = torch.Generator().manual_seed(1234)
    conds_all = torch.randn(300 * world + 8 + n_frames * world, 1, 204, generator=g)
    conds = torch.stack([get_audio_features(conds_all, 2, first + f, 5) for f in range(n_frames)])       # [F,5,1,204]
    poses_h, conds_h = poses.pin_memory(), conds.pin_memory()
    bg = fi['bg_color']
    handle = model.gf_model()
    L = _lib.lib()
    rgb8 = torch.empty(N, 3, dtype=torch.uint8, device=dev)
    counters = torch.zeros(4, dtype=torch.int64, device=dev)

    # resident arm: every frame's packed inputs (condition window + 22 scalars) already sit in HBM; a step = one device-side row copy
    # into the graph's input buffer + ONE CUDA-graph replay of {condition encoder, gf_render_frame} (or the eager launches with --eager)
    packed_d = sequence.pack_frame_inputs(poses, conds, fi['intrinsics'], torso).to(dev)
    fg = sequence.FrameGraph(model, H, W, conds.shape[1:], bg, rgb8, precision=args.precision, max_steps=max_steps, dt_gamma=dt_gamma, torso=torso,
                             want=('rgb8', 'counters'), extra_out={'counters': counters})

    def frame_resident(f):
        fg.inputs.copy_(packed_d[f], non_blocking=True)
        if args.eager:
            with torch.no_grad():
                fg._frame()
        else:
            fg.replay()

    # end to end = the public sequence API (geneface_b200.sequence.SequenceRenderer, the replacement of the frame loop of
    # inference/nerfs/base_nerf_infer.py:131-179) with HOST inputs: poses + condition windows in host memory, per frame one H2D copy of
    # the packed row, the graph replay, and the RGB8 frame D2H into a pinned ring on a copy stream (frame k+1 renders while frame k
    # drains); the call returns when every frame is resident in host memory.  Host-side packing is inside the call, hence timed.
    seq = sequence.SequenceRenderer(model, H, W, fi['intrinsics'], precision=args.precision, max_steps=max_steps, dt_gamma=dt_gamma, torso=torso,
                                    graph=not args.eager)
    host_ring = torch.empty(args.steps, H, W, 3, dtype=torch.uint8).pin_memory()

    def sequence_e2e():
        seq.render(poses_h, conds_h, bg, args.warmup, args.warmup + args.steps, out_rgb8=host_ring)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up + workload assertions ----
    sampler = ClockSampler(local)
    sampler.start()
    for f in range(args.warmup):
        frame_resident(f)
    torch.cuda.synchronize()
    c = counters.cpu().numpy()
    samples_per_frame, torso_px, s_total, launches = int(c[0]), int(c[1]), int(c[2]), int(c[3])
    if headline:
        assert samples_per_frame == N * MAX_STEPS == 33554432, f"workload must evaluate 262144 x 128 samples, got {samples_per_frame}"
        assert s_total == MAX_STEPS and torso_px > 0
    seq.render(poses_h, conds_h, bg, 0, min(args.warmup, 3, args.steps), out_rgb8=host_ring)        # warm the e2e path too (graph capture, ring)

    # ---- timed: resident inputs ----
    barrier()
    sampler.mark_begin()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for k in range(args.steps):
        frame_resident(args.warmup + k)
    ev1.record()
    barrier()
    ms_res = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"rgb8": rgb8.view(H, W, 3), "counters": counters})
    # ---- timed: end to end (host inputs, host result), 3 repeats of the K-frame sequence, median ----
    e2e_ms = []
    for rep in range(3):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sequence_e2e()
        e1.record()
        barrier()
        e2e_ms.append(e0.elapsed_time(e1))
    sampler.mark_end()
    clocks = sampler.stop()
    # ---- dominant-kernel time (events inside gf_render_frame; eager launches so that the events bracket each field launch) ----
    _lib.check(L.gf_profile_enable(handle, 1))
    field_ms = []
    for k in range(min(5, args.steps)):
        fg.inputs.copy_(packed_d[args.warmup + k], non_blocking=True)
        with torch.no_grad():
            fg._frame()
        torch.cuda.synchronize()
        tot, n = ctypes.c_float(0), ctypes.c_int(0)
        _lib.check(L.gf_profile_field_ms(handle, ctypes.byref(tot), ctypes.byref(n)))
        field_ms.append(tot.value)
    _lib.check(L.gf_profile_enable(handle, 0))
    field_ms_per_frame = float(np.median(field_ms))
    n_field_launches = n.value

    t = torch.tensor([ms_res] + e2e_ms, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_res, e2e_ms = float(t[0]), [float(v) for v in t[1:]]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_e2e = sorted(e2e_ms)[1]
    peaks = load_peaks()
    value = world * args.steps / (ms_res / 1000.0)
    e2e = world * args.steps / (ms_e2e / 1000.0)
    achieved = samples_per_frame * HEAD_SAMPLE_BYTES / (field_ms_per_frame / 1000.0) / 1e9
    tflops = samples_per_frame * HEAD_SAMPLE_FLOP / (field_ms_per_frame / 1000.0) / 1e12
    prof, prof_src = profile_record()
    rounds = max(1, n_field_launches)
    roof = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "traffic": (prof or {}).get("dram_bytes_per_round") if args.precision == "fp16" and headline else None, "traffic_source": prof_src,
            "algorithmic_bytes_per_launch": samples_per_frame // rounds * HEAD_SAMPLE_BYTES,
            "kernel": "k_tc_amb+k_tc_sigcol" if args.precision == "fp16" else "k_field_fp32", "kernel_ms_per_frame": field_ms_per_frame,
            "field_launches_per_frame": rounds, "kernel_share_of_step": field_ms_per_frame / (ms_res / args.steps), "peak_source": peaks["source"],
            "tensor_tflops": tflops, "tensor_frac_of_bf16_peak": tflops / peaks["bf16_tflops"],
            "note": "algorithmic gather bytes (1536 B/sample: 16 levels x 8 corners x 8 B + 16 x 4 x 8 B); the 16 MB tables are L2-resident so DRAM traffic "
                    "(sample lists + the 72 B/sample hand-off between the two field kernels) is far below this; one launch = one round of <= 32 slots/ray; "
                    "gather_ceiling = the same accounting measured by scripts/ubench/l2_gather_bw on this GPU"}
    ub = gather_ubench()
    if ub and "coherent64_2tables" in ub:
        roof["gather_ceiling"] = ub
        roof["frac_of_l2_gather"] = achieved / ub["coherent64_2tables"]
        roof["frac_of_l2_random_gather"] = achieved / ub["random_16MB_2tables"]
    if headline and args.precision == "fp16":
        try:
            with torch.no_grad():
                gp = gather_probe_gbs(model, fi, dev, args.precision)
            roof["gather_probe"] = gp
            roof["frac_of_gather_ceiling"] = achieved / gp["gbs"]
        except Exception as e:  # noqa: BLE001
            roof["gather_probe"] = {"unavailable": repr(e)[:200]}
    if prof:
        roof["ncu"] = {k: prof[k] for k in prof if k != "dram_bytes_per_round"}
    line = {
        "metric": METRIC if headline else "512x512 frames/sec, " + args.config, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16" if args.precision == "fp16" else "f32", "data": "synthetic",
        "config": {"workload": workload, "name": args.config,
                   "frames_per_rank": args.steps, "sharding": "frames, rank-block; one NCCL parameter broadcast (%d B), no per-frame communication" % bcast_bytes,
                   "l2": "per-round sample lists (335 MB) exceed L2; the 16 MB grid tables are the algorithm's own hot set; no explicit flush",
                   "launch": "eager" if args.eager else "CUDA graph replay per frame", "cpu_sample_rays": CPU_SAMPLE_RAYS,
                   "precision": args.precision, "samples_per_frame": samples_per_frame, "torso_pixels": torso_px, "s_total": s_total},
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": int(packed_d[0].numel() * 4),
                "d2h_bytes_per_step": int(host_ring[0].numel()), "api": "geneface_b200.sequence.SequenceRenderer.render (pipelined frames)",
                "repeats_ms": e2e_ms, "stat": "median of 3 warmed repeats of the K-frame sequence"},
        "gpu_launches": launches * args.steps,
        "roofline": roof,
        "clocks": clocks,
    }
    if not args.no_cpu_baseline and world == 1 and headline:
        try:
            fps, dt, threads, sample = cpu_port_fps()
            line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample}
        except Exception as e:  # noqa: BLE001  (the GPU line must still be printed)
            line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": host_threads(), "kind": "port", "sample": "failed: " + repr(e)[:200]}
    if not args.no_ref_cuda and world == 1:
        try:
            line["reference_cuda"], line["parity"] = reference_cuda_fps(model, hp, fi, dev, torso, dt_gamma, max_steps, args.precision)
        except Exception as e:  # noqa: BLE001
            line["reference_cuda"] = {"unavailable": repr(e)[:300]}
    if not args.no_may and world == 1 and headline:
        for name in ("may_head", "may_torso"):
            try:
                line[name] = may_cfg_fps(dev, name, args.precision, not args.no_ref_cuda)
            except Exception as e:  # noqa: BLE001
                line[name] = {"unavailable": repr(e)[:300]}
        try:
            line["adnerf_gpu"] = adnerf_gpu_fps(dev)
        except Exception as e:  # noqa: BLE001
            line["adnerf_gpu"] = {"unavailable": repr(e)[:200]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def adnerf_gpu_fps(dev):
    """Context number (BASELINE.json configs[0] on the GPU): the vanilla AD-NeRF frame -- 64x64 rays, 64 coarse + 128 fine samples,
    8x256 backbone -- through geneface_b200.adnerf; `adnerf_cpu` in the reference arm is its CPU twin."""
    import torch
    from geneface_b200 import adnerf
    torch.manual_seed(0)
    m = adnerf.ADNeRF(dict(cond_dim=64, hidden_size=256)).to(dev).eval()
    Hh = Ww = 64
    focal = 1200.0 * Hh / 450.0
    c2w = torch.tensor([[1.0, 0, 0, 0], [0, 1.0, 0, 0], [0, 0, 1.0, 0.6]], device=dev)
    cond = torch.randn(8, 16, 29, generator=torch.Generator().manual_seed(1)).to(dev)
    bc = torch.ones(Hh, Ww, 3, device=dev)

    def frame():
        with torch.no_grad():
            cf = m.cal_cond_feat(cond, with_att=True)
            return adnerf.render_dynamic_face(Hh, Ww, focal, Ww / 2, Hh / 2, chunk=4096, c2w=c2w, cond=cf, near=0.3, far=0.9, network_fn=m,
                                              N_samples=64, N_importance=128, perturb=0., bc_rgb=bc)
    for _ in range(3):
        frame()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20
    e0.record()
    for _ in range(n):
        out = frame()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    return {"value": 1000.0 / ms, "unit": "frames/s", "ms_per_frame": ms, "finite": bool(torch.isfinite(out[0]).all()),
            "workload": "vanilla AD-NeRF 64x64, 64 coarse + 128 fine samples/ray, random weights (BASELINE.json configs[0])"}


def may_cfg_fps(dev, name, precision, with_ref):
    """Context numbers (BASELINE.json configs[1] and [2]): the reference's own deployment configuration -- May head / head+torso,
    bound=1, max_steps=16, dt_gamma=1/256, sphere occupancy -- rendered by the same fused path through one CUDA-graph replay per
    frame, beside the reference's own render() on the same GPU."""
    import torch
    from geneface_b200 import sequence, synthetic
    torso, bitfield, sigma_scale, bound, max_steps, dt_gamma, workload = CONFIGS[name]
    model, hp = synthetic.build_model(torso=torso, bitfield=bitfield, seed=0, sigma_scale=sigma_scale, bound=bound, device=dev)
    fi = synthetic.frame_inputs(H, W, device=dev)
    counters = torch.zeros(4, dtype=torch.int64, device=dev)
    rgb8 = torch.empty(H * W, 3, dtype=torch.uint8, device=dev)
    fg = sequence.FrameGraph(model, H, W, fi['cond'].shape, fi['bg_color'], rgb8, precision=precision, max_steps=max_steps, dt_gamma=dt_gamma,
                             torso=torso, want=('rgb8', 'counters'), extra_out={'counters': counters})
    row = sequence.pack_frame_inputs(fi['pose'].cpu(), fi['cond'][None].cpu(), fi['intrinsics'], torso).to(dev)[0]
    res = {"unit": "frames/s", "workload": workload}
    for mode in ("graph", "eager"):
        def frame():
            fg.inputs.copy_(row, non_blocking=True)
            if mode == "graph":
                fg.replay()
            else:
                with torch.no_grad():
                    fg._frame()
        for _ in range(5):
            frame()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 100
        e0.record()
        for _ in range(n):
            frame()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        if mode == "graph":
            res.update({"value": 1000.0 / ms, "ms_per_frame": ms})
        else:
            res["eager_ms_per_frame"] = ms
    c = counters.cpu().numpy()
    res.update({"samples_per_frame": int(c[0]), "torso_pixels": int(c[1]), "launches_per_frame": int(c[3])})
    if with_ref:
        try:
            res["reference_cuda"], res["parity"] = reference_cuda_fps(model, hp, fi, dev, torso, dt_gamma, max_steps, precision)
        except Exception as e:  # noqa: BLE001
            res["reference_cuda"] = {"unavailable": repr(e)[:300]}
    return res


def reference_cuda_fps(model, hp, fi, dev, torso, dt_gamma, max_steps, precision):
    """Context number AND parity check on the timed workload: the reference's OWN `RADNeRF(Torso).render()` (unmodified Python from
    oracle/_ref/pyref on the unmodified compiled extensions oracle/_ref/*.so, fp32 torch GEMMs) on the same GPU, same weights, same
    frame -- the 'kernel to beat' (BASELINE.md B-REF-CUDA).  Its image is compared with the fused frame of the benchmarked precision:
    worst per-pixel scaled error |a-b| / (1e-5 + |b|) of rgb / depth / weights, and equality of the per-ray sample counts.
    Not part of the product path."""
    import numpy as np
    import torch
    from oracle import ref_model
    if not ref_model.available():
        return {"unavailable": "oracle/_ref not built"}, None
    ns = ref_model.load()
    ref = ref_model.build(model.state_dict(), hp, torso=torso, device=dev)
    rays = ns.utils.get_rays(fi['pose'], fi['intrinsics'], H, W, -1)
    bgc = ns.utils.get_bg_coords(H, W, dev)
    poses6 = ns.utils.convert_poses(fi['pose'])
    times = []
    for it in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res_r = ref_model.render(ref, rays['rays_o'], rays['rays_d'], fi['cond'], bgc, poses6, fi['bg_color'], dt_gamma, max_steps, trace=(it == 0))
        e1.record()
        torch.cuda.synchronize()
        if it == 0:
            first = res_r                      # traced call (weights_sum / n_marched observed); untimed
        else:
            times.append(e0.elapsed_time(e1))
    ms = sorted(times)[len(times) // 2]
    with torch.no_grad():
        ours = model.render(rays['rays_o'], rays['rays_d'], fi['cond'], bgc, poses6, bg_color=fi['bg_color'], dt_gamma=dt_gamma, max_steps=max_steps,
                            precision=precision)
    torch.cuda.synchronize()

    def worst(a, b):
        a, b = a.reshape(-1).double(), b.reshape(-1).double()
        return float(((a - b).abs() / (1e-5 + b.abs())).nan_to_num(0.0).max())
    parity = {"vs": "the reference's own render() on identical rays and weights (fp32)", "precision": precision,
              "rgb_worst": worst(ours['rgb_map'], first['rgb_map']), "depth_worst": worst(ours['depth_map'], first['depth_map']),
              "weights_worst": worst(ours['weights_sum_eval'], first['weights_sum']), "bar": 1e-3}
    if max_steps == MAX_STEPS and dt_gamma == 0.0:
        parity["n_samples_equal"] = bool(torch.equal(ours['n_samples'], first['n_marched']))
    parity["ok"] = _within_bar(ours, first)          # |a-b| <= 1e-5 + 1e-3 |b| on every pixel of rgb / depth / weights
    return ({"value": 1000.0 / ms, "unit": "frames/s", "ms_per_frame": ms,
             "what": "the reference's own render() (unmodified Python + compiled extensions, torch fp32 GEMMs), same GPU, same frame; median of 3"}, parity)


def _within_bar(ours, ref, rel=1e-3, abs_=1e-5):
    """|a-b| <= abs + rel*|b| per pixel (the tests' criterion; the scaled error above can read slightly over `rel` near the abs floor)."""
    import torch
    ok = True
    for k, k2 in (("rgb_map", "rgb_map"), ("depth_map", "depth_map"), ("weights_sum_eval", "weights_sum")):
        a, b = ours[k].reshape(-1).double(), ref[k2].reshape(-1).double()
        d = (a - b).abs()
        ok = ok and bool((torch.isnan(a) & torch.isnan(b) | (d <= abs_ + rel * b.abs())).all())
    return ok


def run_seq300(args, rank, world, local):
    """BASELINE.json configs[3]: ONE 300-frame 512x512 head+torso (May cfg) sequence, frames sharded across the ranks in the reference's
    rank-block partition (STRONG scaling: total work fixed).  Wall-clock on the device timeline from the first launch to the last
    frame's RGB8 resident in pinned host memory (max over ranks); PNG encoding of the rank's frames is timed separately."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from geneface_b200 import egress, sequence, synthetic
    from geneface_b200.utils import get_audio_features, orbit_pose
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    F = 300
    torso, bitfield, sigma_scale, bound, max_steps, dt_gamma, workload = CONFIGS["may_torso"]
    model, hp = synthetic.build_model(torso=torso, bitfield=bitfield, seed=0 if rank == 0 else 100 + rank, sigma_scale=sigma_scale, bound=bound, device=dev)
    bcast = sequence.broadcast_model_(model, src=0)
    fi = synthetic.frame_inputs(H, W, device=dev)
    poses = torch.stack([torch.from_numpy(orbit_pose(3.35, 10.0 * np.sin(2 * np.pi * f / 100.0))) for f in range(F)])
    conds_all = torch.randn(F, 1, 204, generator=torch.Generator().manual_seed(1234))
    conds = torch.stack([get_audio_features(conds_all, 2, f, 5) for f in range(F)]).pin_memory()
    start, end = sequence.partition_frames(F, world, rank)
    seq = sequence.SequenceRenderer(model, H, W, fi['intrinsics'], precision=args.precision, max_steps=max_steps, dt_gamma=dt_gamma, torso=torso,
                                    graph=not args.eager)
    host = torch.empty(end - start, H, W, 3, dtype=torch.uint8).pin_memory()
    seq.render(poses, conds, fi['bg_color'], start, min(end, start + 4), out_rgb8=host)            # warm-up: graph capture
    times = []
    for rep in range(3):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        seq.render(poses, conds, fi['bg_color'], start, end, out_rgb8=host)
        times.append(time.perf_counter() - t0)
    t = torch.tensor(times, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    png = None
    if rank == 0:
        import tempfile
        with tempfile.TemporaryDirectory() as d:
            t0 = time.perf_counter()
            with egress.PngSequenceWriter(d, workers=min(16, os.cpu_count() or 1)) as wr:
                for k in range(end - start):
                    wr.submit(start + k, host[k].numpy())
            png = {"frames": end - start, "seconds": time.perf_counter() - t0, "workers": min(16, os.cpu_count() or 1)}
            png["frames_per_s"] = png["frames"] / png["seconds"]
        secs = sorted(float(v) for v in t)[1]
        print(json.dumps({"metric": "300-frame 512x512 head+torso sequence, wall-clock to last frame in pinned host memory", "value": F / secs,
                          "unit": "frames/s", "seconds": secs, "repeats_s": [float(v) for v in t], "n_gpus": world, "frames": F, "scaling": "strong",
                          "higher_is_better": True, "dtype": "f16" if args.precision == "fp16" else "f32", "data": "synthetic",
                          "config": {"workload": workload, "name": "seq300", "partition": "rank-block (base_nerf_infer.py:150-155)", "broadcast_bytes": bcast,
                                     "launch": "eager" if args.eager else "CUDA graph replay per frame"},
                          "png_egress": png}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_train(args, rank, world, local):
    """BASELINE.json configs[4]: train step, 4096 rays: march_rays_train + field + composite + hash-grid backward (scripts/bench_train.py)."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import bench_train
    line = bench_train.run(steps=args.steps, warmup=args.warmup, local=local)
    line["amp"] = bench_train.run(steps=args.steps, warmup=args.warmup, local=local, amp=True)
    # the MLPs on the gf_tl_* tcgen05 operators (fp16 operands, fp32 accumulation: the arithmetic of the amp arm) -- BASELINE.json's 4096 rays and the
    # May configuration's own training batch (n_rays = 65536)
    line["tc_mlp"] = bench_train.run(steps=args.steps, warmup=args.warmup, local=local, mlp="tc", no_ref=True)
    line["tc_mlp_65536"] = bench_train.run(steps=max(5, args.steps // 2), warmup=args.warmup, local=local, rays=65536, mlp="tc", no_ref=True)
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
