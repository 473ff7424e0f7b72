#!/usr/bin/env python
"""bench.py -- rasterizer forward+backward frames/s at BASELINE.json's headline configuration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[1] -- ~100k mesh-bound splats, 1920x1080, SH degree 3, fused
binding + rasterizer forward + backward, one camera per step per GPU.  media/306 cannot travel to the GPU box, so the
splats are the seeded synthetic avatar of gaussianavatars_b200/synthetic.py, calibrated against media/306 through
the oracle (DESIGN.md "Workload calibration").

One "step" = one frame: per-face frame of the posed mesh, fused forward, backward down to the raw parameters and
the mesh vertices (+ for N>1 one NCCL all-reduce of the flat 59-float per-splat gradient buffer; frames shard by
camera, "scaling": "weak").
  value  : frames/s, all inputs resident in HBM (camera block, posed mesh, dL/dimage), the step replayed as ONE CUDA
           graph (gaussianavatars_b200/graph.py: the forward runs sync-free on a fixed instance capacity, overflow is
           checked after the timed loop), L2 flushed between steps, timed per step with CUDA events on the launching
           stream, max over ranks.
  eager  : the same step through the eager `render()` + autograd (what a caller of the drop-in surface gets).
  e2e    : the same metric with HOST inputs: every step uploads the camera block and the uint8 ground-truth image from
           pinned memory (copy nodes at the head of the graph), computes an L1 loss, runs backward and copies the loss
           scalar back to pinned memory, which the host reads one step later (the data flow of the reference training
           step, train.py:113-170).
  parity_check : one frame of this very workload compared with the CPU oracle (image, radii, all gradients).
  baseline_b3  : SURVEY 8(d) baseline 3 -- the reference's eager binding getters on the GPU + the unfused operator
           surface + the reference's full instance list (exact_binning=1), forward+backward, same GPU, same run.  It
           is a PROXY for the absent upstream CUDA rasterizer (same kernels underneath, minus the fusion and the
           culling), not a measurement of it.
  roofline / cpu_baseline : see DESIGN.md "Measurement".

--dump-outputs DIR: after the timed steps, rank 0 writes what the last of them computed -- the image, the radii and
the gradients of the raw splat parameters and of the posed mesh vertices -- as DIR/<name>.npy (float32).  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

P_SPLATS = 100_000
WIDTH, HEIGHT = 1920, 1080
SH_DEGREE = 3
N_CAMERAS = 16  # distinct orbit views cycled through
DUMP_BYTES = 63_900_000  # --dump-outputs: all arrays together, room left for the .npy headers within 64 MB
# names of the gradients of MeshBoundGaussians.parameters(), in its order
PARAM_NAMES = ("xyz", "rotation", "scaling", "opacity", "features_dc", "features_rest")
METRIC = "rasterizer fwd+bwd frames/sec @100k splats 1080p"
WORKLOAD = "avatar-100k-splats-1920x1080-sh3-fused-binding-fwd+bwd (BASELINE configs[1], synthetic media/306 stand-in)"


class Pipe:
    debug = False
    compute_cov3D_python = False
    convert_SHs_python = False


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip cpu_baseline and parity_check")
    ap.add_argument("--no-graph", action="store_true", help="time the eager render() + autograd step instead of the CUDA graph")
    ap.add_argument("--no-baseline-b3", action="store_true", help="skip SURVEY 8(d) baseline 3 (eager getters + unfused + exact list)")
    ap.add_argument("--exact-binning", action="store_true", help="emit the reference's full instance list")
    # other BASELINE.json configs (parity/scale cases, not the headline line): e.g. config 4 =
    #   --gpus 8 --splats 500000 --width 2048 --height 2048 --cameras 64
    ap.add_argument("--collective", default="auto", choices=["auto", "nccl", "nvls", "nvls2"],
                    help="N>1 gradient reduction.  nccl: one ncclAllReduce after backward.  nvls2: this library's two-shot "
                         "NVLS all-reduce kernel (multimem.ld_reduce + multimem.st, csrc/nvls.cu) on the symmetric-memory "
                         "gradient buffer, captured inside the step's graph.  nvls: push-style multimem.red fused into "
                         "preprocess_bwd (eager only; loses at N=8, every replica receives N x the buffer).  auto = "
                         "nvls2 when the fabric has multicast and its self-test passes on every rank, else nccl "
                         "(DESIGN.md section 6)")
    ap.add_argument("--reduce", default="deferred", choices=["deferred", "sync"],
                    help="N>1: deferred = the all-reduce of step i's gradient buffer runs as a forked branch of step i+1's "
                         "graph (two graphs / two buffers used alternately; the K-th reduction is drained inside the timed "
                         "region); sync = the collective sits after backward inside the same graph.  The sync figure is "
                         "measured and reported either way (`sync_collective`)")
    ap.add_argument("--side-at", default="start", choices=["start", "backward"],
                    help="deferred reduction: fork the reduction branch at the start of the frame or after its forward")
    ap.add_argument("--nvls-ctas", type=int, default=0, help="CTAs of the two-shot NVLS kernel (0 = library default)")
    ap.add_argument("--shard", default="round_robin", choices=["cost", "round_robin"],
                    help="N>1 camera sharding: cost = cameras sorted by their instance count (one forward each in warm-up) "
                         "and dealt so that the cameras of one step have neighbouring costs (dist.shard_frames_by_cost); "
                         "round_robin = r, r+N, ...")
    ap.add_argument("--splats", type=int, default=None)
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--cameras", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (native arm)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native path")
    global P_SPLATS, WIDTH, HEIGHT, N_CAMERAS, WORKLOAD
    if a.splats or a.width or a.height or a.cameras:
        P_SPLATS = a.splats or P_SPLATS
        WIDTH, HEIGHT = a.width or WIDTH, a.height or HEIGHT
        N_CAMERAS = a.cameras or N_CAMERAS
        WORKLOAD = f"avatar-{P_SPLATS}-splats-{WIDTH}x{HEIGHT}-sh3-fused-binding-fwd+bwd ({N_CAMERAS} cameras; non-headline config)"
    return a


def make_cameras(n):
    from gaussianavatars_b200 import synthetic as syn

    cams = []
    for i in range(n):
        az = -60.0 + 120.0 * (i + 0.5) / n  # +-60 degree arc (SURVEY.md 8d config 3)
        c = syn.orbit_camera(WIDTH, HEIGHT, r=1.0, fovy_deg=20.0, azimuth_deg=az, elevation_deg=5.0 * math.sin(i))
        c.timestep = i
        cams.append(c)
    return cams


def algorithmic_bytes(P, N, W, H, F):
    """SURVEY.md 8(d) per-unit figures (SH3, fused, training mode) -- compulsory traffic per frame, by stage."""
    c_in = 240
    return {
        "preprocess": P * c_in + P * (48 + 28),
        "scan": P * 8,
        "emit_keys": P * 48 + N * 12,
        "sort": N * 24,
        "tile_ranges": N * 8,
        "blend_fwd": N * 40 + H * W * (12 + 8),
        "blend_bwd": H * W * 20 + N * 40 + P * 44,
        "preprocess_bwd": P * 44 + P * (c_in + 76) + P * 236 + F * 52,
    }


# ---------------------------------------------------------------------------------------------------------------
# clocks sampler (recipe: B200_PROFILING.md "clocks DURING the timed region")
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores (bench.py's cpu_baseline and --impl reference)
# ---------------------------------------------------------------------------------------------------------------
def host_cpus():
    """CPUs this process can actually use: the smaller of the affinity mask and the cgroup CPU quota.  The GPU boxes
    show 128 logical CPUs under a quota of 16 (cpu.max = 1600000 100000); 128 OpenMP threads throttled onto 16 CPUs'
    worth of time made the eager binding getters 700x slower (3.5 s instead of 5 ms per frame, profiles/r02/
    cpu_threads_probe.jsonl), and the C oracle shares torch's OpenMP runtime, so one number serves both."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, -(-int(txt[0]) // int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, -(-quota // period)))
            break
        except Exception:
            continue
    return max(1, n)


def cpu_frames(params, verts, faces, cams, frames, threads=None):
    """Runs `frames` full fwd+bwd frames of the same workload through the CPU oracle (eager torch binding getters +
    C rasterizer, OpenMP over all host cores).  Returns (seconds per frame list, binding seconds per frame list)."""
    import numpy as np

    from oracle import binding as ob
    from oracle import rasterizer as orc

    # torch.distributed.run exports OMP_NUM_THREADS=1 to its workers: say explicitly how many threads this arm gets
    # (host_cpus(): what the container may really use).
    cpus = threads or host_cpus()
    torch.set_num_threads(cpus)
    orc.set_threads(cpus)
    bg = np.ones(3, np.float32)
    gout = torch.randn(3, HEIGHT, WIDTH, generator=torch.Generator().manual_seed(1)).numpy()
    from gaussianavatars_b200 import synthetic as syn

    times, bind_times = [], []
    for i in range(frames):
        cam = cams[i % len(cams)]
        t0 = time.perf_counter()
        v = syn.pose_mesh(verts, cam.timestep)
        fr = ob.update_mesh_properties(v, faces)
        b = params["binding"].long()
        xyz = ob.get_xyz(params["_xyz"], b, fr["face_center"], fr["face_orien_mat"], fr["face_scaling"])
        sc = ob.get_scaling(params["_scaling"], b, fr["face_scaling"])
        ro = ob.get_rotation(params["_rotation"], b, fr["face_orien_quat"])
        op = ob.get_opacity(params["_opacity"])
        sh = ob.get_features(params["_features_dc"], params["_features_rest"]).contiguous()
        t1 = time.perf_counter()
        kw = dict(shs=sh.numpy(), sh_degree=SH_DEGREE, scales=sc.numpy(), rotations=ro.numpy())
        st = orc.forward(xyz.numpy(), op.numpy(), cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(),
                         cam.camera_center.numpy(), WIDTH, HEIGHT, cam.tanfovx, cam.tanfovy, bg, **kw)
        orc.backward(st, gout, xyz.numpy(), cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(),
                     cam.camera_center.numpy(), cam.tanfovx, cam.tanfovy, bg, **kw)
        t2 = time.perf_counter()
        times.append(t2 - t0)
        bind_times.append(t1 - t0)
    return times, bind_times


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path.  The rasterizer submodule is absent from
    /root/reference (unbuildable), so this is the oracle PORT (cpu_baseline.kind = "port") on all host cores."""
    if rank != 0:
        return
    from gaussianavatars_b200 import synthetic as syn

    verts, faces = syn.head_mesh()
    params = syn.avatar_splats(P_SPLATS, n_faces=faces.shape[0], seed=0, sh_degree=SH_DEGREE)
    cams = make_cameras(N_CAMERAS)
    cores = host_cpus()
    steps = args.steps   # one frame per step
    warm = max(1, min(args.warmup, 2))
    cpu_frames(params, verts, faces, cams, warm)
    t, _ = cpu_frames(params, verts, faces, cams, steps)
    sec = sum(t) / len(t)
    fps = 1.0 / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "splats": P_SPLATS, "width": WIDTH, "height": HEIGHT, "sh_degree": SH_DEGREE},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} full frames (binding getters + rasterizer fwd+bwd), OpenMP x{cores}; "
                                   "the port is the parity CHECKER being timed (scalar C, one tile per task), "
                                   "not a tuned CPU renderer"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist

    from gaussianavatars_b200 import _native as N
    from gaussianavatars_b200 import dist as gdist
    from gaussianavatars_b200 import rasterizer as R
    from gaussianavatars_b200 import synthetic as syn
    from gaussianavatars_b200.model import MeshBoundGaussians
    from gaussianavatars_b200.renderer import render

    assert torch.cuda.is_available(), "bench.py (native arm) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    N.lib()
    if args.nvls_ctas > 0:
        N.tune(N.TUNE_NVLS_CTAS, args.nvls_ctas)
    R.set_exact_binning(args.exact_binning)
    R.keep_last_state(True)

    verts, faces = syn.head_mesh()
    params = syn.avatar_splats(P_SPLATS, n_faces=faces.shape[0], seed=0, sh_degree=SH_DEGREE)
    pc = MeshBoundGaussians(params, SH_DEGREE, verts, faces, pose_fn=syn.pose_mesh, device=dev, requires_grad=True)
    # N > 1: caller-owned gradient buffers (dist.SymmetricGradBuffer).  bufs[0] doubles as the buffer of the synchronous
    # step; the pair serves the two alternating graphs of the deferred reduction.
    symm, bufs, collective_note = None, None, None
    if world > 1:
        def agree(ok):
            flag = torch.tensor([1.0 if ok else 0.0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            return float(flag) != 0.0

        def make(mode, n):
            why, made = None, []
            try:
                made = [gdist.SymmetricGradBuffer(pc, mode=mode) for _ in range(n)]
                ok = all(b.enabled for b in made) and (mode != "two_shot" or all(b.self_test() for b in made))
                if not ok:
                    why = next((getattr(b, "error", None) for b in made if getattr(b, "error", None)), "self-test failed")
            except Exception as e:
                ok, why = False, f"{type(e).__name__}: {e}"
            return (made if agree(ok) else None), why

        if args.collective == "nvls":      # push-style multimem.red from the backward kernel: eager only
            made, why = make("push", 1)
            if made is None:
                raise RuntimeError(f"--collective nvls unavailable: {why or 'another rank failed'}")
            symm = made[0]
        else:
            if args.collective in ("auto", "nvls2"):
                bufs, why = make("two_shot", 2)
                if bufs is None:
                    if args.collective == "nvls2":
                        raise RuntimeError(f"--collective nvls2 unavailable: {why or 'another rank failed'}")
                    collective_note = f"nvls2 unavailable ({why or 'another rank failed'}): nccl"
            if bufs is None:
                bufs, why = make("plain", 2)
                if bufs is None:
                    raise RuntimeError(f"gradient buffers could not be created: {why}")
            symm = bufs[0]
        pc.symm_grad = symm
    cams_host = make_cameras(N_CAMERAS)
    shard_note = "all cameras on the one GPU"
    mine_idx = gdist.shard_frames(N_CAMERAS, rank, world)
    if world > 1:
        shard_note = "round robin"
        if args.shard == "cost" and N_CAMERAS >= world:
            # one forward per camera (every rank renders all of them once: identical counts), then cost-sorted dealing
            costs = []
            with torch.no_grad():
                for c in cams_host:
                    pc.update_mesh_properties(syn.pose_mesh(pc.verts_rest, c.timestep).contiguous())
                    render(c.to(dev), pc, Pipe, torch.ones(3, device=dev))
                    torch.cuda.synchronize(dev)
                    costs.append(int(R.last_frame_info().get("num_rendered", 0)))
            t = torch.tensor(costs, dtype=torch.int64, device=dev)
            dist.broadcast(t, 0)
            costs = [int(x) for x in t.tolist()]
            mine_idx = gdist.shard_frames_by_cost(costs, rank, world)
            pc.face_center = pc.face_orien_mat = pc.face_scaling = None
            shard_note = (f"cost-sorted dealing: cameras ordered by instance count ({min(costs)}..{max(costs)}), step j renders "
                          f"cameras j*{world}..j*{world}+{world - 1} of that order, one per rank")
    my_cams = [cams_host[i] for i in mine_idx] or cams_host
    cams_dev = [c.to(dev) for c in my_cams]
    # posed meshes (output of the FLAME LBS, upstream of the path) are inputs resident in HBM; the per-face frame
    # (SURVEY.md 8a rows a1/a2) is recomputed inside every step by the library's face-frame kernel
    # requires_grad: --bind_to_mesh training optimises the FLAME parameters (scene/flame_gaussian_model.py:186-207), so
    # the step includes dL/d(face frame) and the face-frame backward down to the vertices
    posed = [syn.pose_mesh(pc.verts_rest, c.timestep).contiguous().requires_grad_(True) for c in my_cams]
    bg = torch.ones(3, device=dev)
    gout = torch.randn(3, HEIGHT, WIDTH, generator=torch.Generator().manual_seed(1)).to(dev) / (3 * HEIGHT * WIDTH)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # 2x the 126 MB L2

    def zero_grads():
        for p in pc.parameters():
            p.grad = None
        for v in posed:
            v.grad = None

    def step_eager(i):
        """HBM-resident step through the eager drop-in surface: render() + autograd."""
        cam = cams_dev[i % len(cams_dev)]
        zero_grads()
        pc.update_mesh_properties(posed[i % len(posed)])
        out = render(cam, pc, Pipe, bg)
        if symm is not None:
            symm.begin()
            out["render"].backward(gout)
            symm.end()
        else:
            out["render"].backward(gout)
            gdist.allreduce_splat_grads(pc)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- warm-up (eager): learns the capacity / depth hints, builds the face CSR ---------------------------------
    for i in range(max(args.warmup, 3)):
        step_eager(i)
    barrier()
    _, _, _, n_inst = R.export_last_binning()
    R.keep_last_state(False)

    # ---- timed region: HBM-resident, L2 flushed between steps, per-step CUDA events -------------------------
    K = args.steps

    def timed_pass(step, stage_events: bool, tail=None):
        N.stage_timing(stage_events)
        N.stage_times(reset=True)
        N.host_times(reset=True)
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        l0 = N.launch_count()
        barrier()
        with ClockSampler(local_rank) as clk_:
            w0 = time.perf_counter()
            for i in range(K):
                flush_buf.fill_(i & 0xFF)  # L2 flush (outside the step's event pair)
                starts[i].record()
                step(i)
                ends[i].record()
            if tail is not None:   # work the K steps left pending (the K-th deferred reduction): timed, added
                starts.append(torch.cuda.Event(enable_timing=True))
                ends.append(torch.cuda.Event(enable_timing=True))
                starts[-1].record()
                tail()
                ends[-1].record()
            barrier()
            w1 = time.perf_counter()
        st_ = N.stage_times(reset=True)
        hu_ = N.host_times(reset=True)
        N.stage_timing(False)
        return sum(s.elapsed_time(e) for s, e in zip(starts, ends)), N.launch_count() - l0, clk_, w1 - w0, st_, hu_

    # eager passes FIRST (before any NCCL kernel is captured into a graph: afterwards the eager all-reduce of a fresh
    # buffer per step took 9.8 ms at N = 2, profiles/r02/bench_n2_first.json -- buffer registration churn)
    # pass A -- the eager drop-in surface, K flushed steps (launch count of one eager step = kernels per frame)
    ms_eager, launches_eager, _, _, _, host_us = timed_pass(step_eager, False)
    # pass B -- eager again with the library's per-stage CUDA events switched on (two event records per stage per step
    # perturb the pipeline, so they stay out of the other passes): per-kernel durations for the roofline line and stage_ms
    ms_instrumented, _, _, _, stage, _ = timed_pass(step_eager, True)
    launches = launches_eager  # a graph replay launches the same kernels (they were captured from this very step)

    # ---- the step as ONE CUDA graph --------------------------------------------------------------------------------
    from gaussianavatars_b200.graph import GraphedFrame, camera_block

    cam_blocks_dev = [camera_block(c) for c in cams_dev]
    c0 = my_cams[0]
    from gaussianavatars_b200.graph import pair_with_deferred_reduce

    use_graph = not args.no_graph and (symm is None or symm.mode != "push")
    frames = []          # the resident step: one graph, or the alternating pair of the deferred reduction
    graph_note = None
    n_common = max(1, N_CAMERAS // world)   # warm-up frames issue collectives: every rank must run the same number

    def sync_hooks():
        """(before_backward, after_backward) of a step whose collective sits after backward in the same graph."""
        return (None, None) if world == 1 else (symm.begin, symm.end)

    def attach_sync():
        if world > 1:
            pc.symm_grad = symm

    def capture_agreed(build):
        """build() -> captured frame(s); None (+ reason) if any rank could not (a captured collective cannot meet an
        eager one, so every rank must take the same path)."""
        got, why = None, None
        try:
            got = build()
        except Exception as e:  # e.g. a fabric on which the collective cannot be captured
            got, why = None, f"{type(e).__name__}: {e}"
        if world > 1 and not agree(got is not None):
            got, why = None, why or "another rank could not capture the step"
        return got, why

    def build_sync():
        attach_sync()
        before, after = sync_hooks()
        fr = GraphedFrame(pc, WIDTH, HEIGHT, c0.FoVx, c0.FoVy, bg, loss="dL_dimage", warm_cameras=cam_blocks_dev[:n_common],
                          before_backward=before, after_backward=after)
        fr.set_inputs(camera=cam_blocks_dev[0], verts=posed[0].detach(), dL_dimage=gout)
        fr.capture()
        return [fr]

    def build_deferred():
        pair = []
        for k in range(2):
            fr = GraphedFrame(pc, WIDTH, HEIGHT, c0.FoVx, c0.FoVy, bg, loss="dL_dimage",
                              warm_cameras=cam_blocks_dev[:n_common])
            fr.set_inputs(camera=cam_blocks_dev[0], verts=posed[0].detach(), dL_dimage=gout)
            pair.append(fr)
        pair_with_deferred_reduce(pair, bufs, side_work_at=args.side_at)
        for fr in pair:
            fr.capture()
        return pair

    last_eager = {}

    def step_resident(i):
        if not frames:
            last_eager["out"] = step_eager(i)
            return
        fr = frames[i % len(frames)]
        fr.set_inputs(camera=cam_blocks_dev[i % len(cam_blocks_dev)], verts=posed[i % len(posed)].detach())
        fr.run()

    def drain():
        """Deferred reduction: the gradients of the last of K steps are still unreduced -- reduce them now."""
        bufs[(K - 1) % 2].reduce()

    sync_line, deferred = None, False
    if use_graph:
        frames, why = capture_agreed(build_sync)
        if frames is None:
            frames, use_graph, graph_note = [], False, f"graph capture failed ({why}); eager step timed"
    if use_graph and world > 1 and args.reduce == "deferred" and bufs is not None:
        # the synchronous form first (reported beside the headline), then the deferred pair
        for i in range(max(args.warmup, 3)):
            step_resident(i)
        barrier()
        ms_sync, _, _, _, _, _ = timed_pass(step_resident, False)
        sync_line = ms_sync   # max over ranks below
        pair, why = capture_agreed(build_deferred)
        if pair is None:
            graph_note = f"deferred-reduction pair not capturable ({why}); synchronous step timed"
            attach_sync()
        else:
            frames, deferred = pair, True

    for i in range(max(args.warmup, 3)):
        step_resident(i)
    barrier()

    # the headline number: nothing but the K steps (+ the drained K-th reduction) inside the event pairs
    ms_total, _, clk, wall_timed, _, _ = timed_pass(step_resident, False, tail=drain if deferred else None)
    overflow_steps = any(fr.overflowed(wait=True) for fr in frames)
    if args.dump_outputs and rank == 0:
        if frames:
            fr = frames[(K - 1) % len(frames)]
            image, radii, grad_verts = fr.image, fr.radii, fr.verts.grad
        else:
            out = last_eager["out"]
            image, radii, grad_verts = out["render"], out["radii"], posed[(K - 1) % len(posed)].grad
        dump_outputs(args.dump_outputs, {"image": image, "radii": radii, "grad_verts": grad_verts,
                                         **{"grad_" + n: p.grad for n, p in zip(PARAM_NAMES, pc.parameters())}})

    # ---- warm-L2 variant (no flush), whole-loop events: what a training loop actually sees -------------------
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step_resident(i)
    if deferred:
        drain()
    e1.record()
    barrier()
    ms_warm = e0.elapsed_time(e1)

    # ---- e2e: host-resident inputs -----------------------------------------------------------------------------------
    gt_host = [torch.randint(0, 256, (3, HEIGHT, WIDTH), dtype=torch.uint8) for _ in range(2)]
    gt_pin = [t.pin_memory() for t in gt_host]
    cam_host_blocks = [camera_block(c).pin_memory() for c in my_cams]
    h2d_bytes = gt_host[0].numel() + cam_host_blocks[0].numel() * 4
    losses = []
    if use_graph:
        # two graphs, each reading its own pinned ground-truth staging buffer (a loader fills one while the GPU reads
        # the other); camera block staged in pinned memory per step; loss scalar copied back by the graph, read late
        e2e_frames = []
        if not deferred:
            attach_sync()
        for k in range(2):
            before_, after_ = (None, None) if deferred else sync_hooks()
            f_ = GraphedFrame(pc, WIDTH, HEIGHT, c0.FoVx, c0.FoVy, bg, loss="l1_u8", host_inputs=True,
                              warm_cameras=cam_host_blocks[:n_common], before_backward=before_, after_backward=after_)
            f_.gt_stage.copy_(gt_host[k])   # the loader's job: decoded frames land in the two pinned staging buffers
            f_.cam_stage.copy_(cam_host_blocks[0])
            f_.set_inputs(verts=posed[0].detach())
            f_.upload_staged()
            e2e_frames.append(f_)
        e2e_frames[0].prefetch_for(e2e_frames[1])
        e2e_frames[1].prefetch_for(e2e_frames[0])
        if deferred:   # each graph's forked branch also all-reduces the other frame's gradient buffer
            pair_with_deferred_reduce(e2e_frames, bufs, side_work_at=args.side_at)
        for f_ in e2e_frames:
            f_.capture()
        done = [torch.cuda.Event() for _ in range(2)]

        def step_e2e(i):
            f_, nxt = e2e_frames[i % 2], e2e_frames[(i + 1) % 2]
            # the NEXT step's camera block goes into the other frame's pinned staging (140 bytes; its ground truth is
            # already in that frame's pinned staging buffer): this step's graph uploads both on a forked branch while
            # it computes.  The last reader of that staging was graph i-2, finished (we waited for done[i-2]).
            nxt.cam_stage.copy_(cam_host_blocks[(i + 1) % len(cam_host_blocks)])
            f_.set_inputs(verts=posed[i % len(posed)].detach())
            f_.run()
            done[i % 2].record()
            if i > 0:  # read the PREVIOUS step's loss: every step's result reaches the host inside the timed region
                done[(i - 1) % 2].synchronize()
                losses.append(float(e2e_frames[(i - 1) % 2].loss_host))

        def finish_e2e(last):
            if deferred:
                drain()
            done[last % 2].synchronize()
            losses.append(float(e2e_frames[last % 2].loss_host))
    else:
        from gaussianavatars_b200 import l1_loss_u8

        copy_stream = torch.cuda.Stream(device=dev)
        loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ready = [torch.cuda.Event() for _ in range(2)]

        def step_e2e(i):
            cam = my_cams[i % len(my_cams)]
            zero_grads()
            with torch.cuda.stream(copy_stream):
                gt_u8 = gt_pin[i % 2].to(dev, non_blocking=True)
            blk = cam_host_blocks[i % len(my_cams)].to(dev, non_blocking=True)
            dcam = syn.SyntheticCamera(cam.image_width, cam.image_height, cam.FoVx, cam.FoVy, blk[0:16].view(4, 4),
                                       blk[16:32].view(4, 4), blk[32:35], cam.timestep)
            pc.update_mesh_properties(posed[i % len(posed)])
            out = render(dcam, pc, Pipe, bg)
            torch.cuda.current_stream(dev).wait_stream(copy_stream)
            gt_u8.record_stream(torch.cuda.current_stream(dev))
            loss = l1_loss_u8(out["render"], gt_u8)
            if symm is not None:
                symm.begin()
                loss.backward()
                symm.end()
            else:
                loss.backward()
                gdist.allreduce_splat_grads(pc)
            loss_host[i % 2].copy_(loss.detach(), non_blocking=True)
            loss_ready[i % 2].record()
            if i > 0:
                loss_ready[(i - 1) % 2].synchronize()
                losses.append(float(loss_host[(i - 1) % 2]))

        def finish_e2e(last):
            loss_ready[last % 2].synchronize()
            losses.append(float(loss_host[last % 2]))

    if use_graph:   # step 0's own inputs (every later step's arrive through the previous step's graph)
        e2e_frames[0].cam_stage.copy_(cam_host_blocks[0])
        e2e_frames[0].upload_staged()
    for i in range(4):
        step_e2e(i)
    barrier()
    losses.clear()
    e0.record()
    for i in range(K):
        step_e2e(i)
    finish_e2e(K - 1)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    assert len(losses) == K and all(math.isfinite(v) for v in losses)
    if use_graph:
        overflow_steps = overflow_steps or any(f_.overflowed(wait=True) for f_ in e2e_frames)

    # ---- baseline 3 (SURVEY 8d): eager getters + unfused surface + the reference's full instance list, same GPU ----
    b3 = None
    if world == 1 and not args.no_baseline_b3:
        R.set_exact_binning(True)
        pc_b3 = MeshBoundGaussians(params, SH_DEGREE, verts, faces, pose_fn=syn.pose_mesh, device=dev, requires_grad=True)

        def step_b3(i):
            for p in pc_b3.parameters():
                p.grad = None
            for v in posed:
                v.grad = None
            pc_b3.update_mesh_properties(posed[i % len(posed)])
            out = render(cams_dev[i % len(cams_dev)], pc_b3, Pipe, bg, fused=False)
            out["render"].backward(gout)

        for i in range(5):
            step_b3(i)
        ms_b3, launches_b3, _, _, _, _ = timed_pass(step_b3, False)
        _, _, _, _, stage_b3, _ = timed_pass(step_b3, True)
        lib_ms_b3 = sum(v[0] / max(v[1], 1) for v in stage_b3.values())
        R.set_exact_binning(args.exact_binning)
        b3 = {"value": K / (ms_b3 / 1e3), "unit": "frames/s", "ms_per_step": ms_b3 / K, "gpu_launches_per_step": launches_b3 / K,
              "rasterizer_kernels_ms": lib_ms_b3, "eager_binding_and_autograd_ms": ms_b3 / K - lib_ms_b3,
              "instances_per_frame": int(R.last_frame_info().get("num_rendered", 0)),
              "what": "SURVEY 8(d) baseline 3: the reference's eager binding getters (PyTorch ops on the GPU, autograd "
                      "through them) + this repo's UNFUSED operator surface + exact_binning=1 (the reference's full "
                      "3-sigma instance list), fwd+bwd, L2 flushed.  A structural proxy for the absent upstream "
                      "diff_gaussian_rasterization CUDA path, NOT a measurement of it."}
        del pc_b3

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    per_rank = None
    if world > 1:   # every rank's own clock over the same K steps: skew between ranks is part of a max-over-ranks metric
        mine_t = torch.tensor([ms_total / K, ms_eager / K, ms_e2e / K, float(len(my_cams))], dtype=torch.float64, device=dev)
        allt = [torch.zeros_like(mine_t) for _ in range(world)]
        dist.all_gather(allt, mine_t)
        per_rank = {"ms_per_step": [round(float(t[0]), 4) for t in allt], "eager_ms_per_step": [round(float(t[1]), 4) for t in allt],
                    "e2e_ms_per_step": [round(float(t[2]), 4) for t in allt], "cameras": [int(t[3]) for t in allt]}
    ms_total, ms_warm, ms_e2e = max_over_ranks(ms_total), max_over_ranks(ms_warm), max_over_ranks(ms_e2e)
    ms_eager, ms_instrumented = max_over_ranks(ms_eager), max_over_ranks(ms_instrumented)
    if sync_line is not None:
        ms_sync = max_over_ranks(sync_line)
        sync_line = {"value": world * K / (ms_sync / 1e3), "unit": "frames/s", "ms_per_step": ms_sync / K,
                     "what": "collective after backward inside the same graph (on the critical path)"}
    if rank != 0:
        finish(world, dev)
        return

    fps = world * K / (ms_total / 1e3)
    F = faces.shape[0]
    alg = algorithmic_bytes(P_SPLATS, n_inst, WIDTH, HEIGHT, F)
    stage_ms = {k: (v[0] / max(v[1], 1)) for k, v in stage.items()}
    dom = max(stage_ms, key=lambda k: stage_ms[k])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg[dom] / (stage_ms[dom] * 1e-3) / 1e9
    traffic = traffic_source = None
    secondary = None  # the path is not HBM-bound at this size (SURVEY 8d): report the limiter ncu names beside the roofline
    headline_shape = (P_SPLATS, WIDTH, HEIGHT) == (100_000, 1920, 1080)
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        if headline_shape:  # the capture is of the headline workload: meaningless for any other --splats/--width
            traffic = tj.get(dom, {}).get("dram_bytes_per_launch")
            traffic_source = "static: " + str(tj.get(dom, {}).get("source", "committed ncu --set full capture of this workload"))
            if tj.get(dom, {}).get("issue_active_per_cycle") is not None:
                secondary = {"bound": "issue slots / fma pipe", "issue_active_per_cycle": tj[dom]["issue_active_per_cycle"],
                             "fma_pipe_active_pct": tj[dom].get("fma_pipe_active_pct"),
                             "warps_active_per_scheduler": tj[dom].get("warps_active_per_scheduler"),
                             "registers": tj[dom].get("registers"), "source": tj[dom].get("source")}
    except Exception:
        pass
    frame_alg = sum(alg.values())
    line = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "splats": P_SPLATS, "width": WIDTH, "height": HEIGHT, "sh_degree": SH_DEGREE,
                   "faces": F, "instances_per_frame": int(n_inst), "binning": "exact" if args.exact_binning else "culled",
                   "frames_per_step_per_gpu": 1, "parallelism": f"frame-sharded dp{world}",
                   "step": (("one CUDA-graph replay (face frame + fused fwd + bwd" +
                             ("" if world == 1 else
                              "; forked branch: all-reduce of the PREVIOUS step's gradient buffer -- two graphs and two "
                              "buffers used alternately, the K-th reduction drained inside the timed region" if deferred
                              else " + gradient all-reduce") + ")") + (f" [{graph_note}]" if graph_note else ""))
                           if use_graph else (graph_note or "eager render() + autograd"),
                   "grad_collective": ("none" if world == 1 else
                                       "nccl all-reduce of the caller-owned flat buffer" if symm.mode == "plain" else
                                       "nvls multimem.red fused in preprocess_bwd" if symm.mode == "push" else
                                       "nvls two-shot all-reduce kernel (multimem.ld_reduce + multimem.st) on the "
                                       "symmetric flat buffer, between two signal-pad barriers, inside the graph"),
                   "reduction": "none" if world == 1 else ("deferred by one replay" if deferred else "synchronous"),
                   "camera_sharding": shard_note,
                   **({"reduction_branch": f"forked at {args.side_at}, nvls ctas {args.nvls_ctas or 'default'}"} if deferred else {}),
                   **({"collective_note": collective_note} if collective_note else {}),
                   "l2": "flushed between steps (256 MiB fill outside the per-step event pair)"},
        "warm_l2": {"value": world * K / (ms_warm / 1e3), "unit": "frames/s", "ms_per_step": ms_warm / K},
        "eager": {"value": world * K / (ms_eager / 1e3), "unit": "frames/s", "ms_per_step": ms_eager / K,
                  "what": "same step through the eager render() + autograd (sync mode LATE), L2 flushed"},
        "e2e": {"value": world * K / (ms_e2e / 1e3), "unit": "frames/s", "ms_per_step": ms_e2e / K,
                "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 4,
                "path": ("two GraphedFrame(host_inputs=True, loss='l1_u8') prefetching each other's inputs from pinned "
                         "staging inside their graphs") if use_graph else "eager render() + l1_loss_u8"},
        **({"sync_collective": sync_line} if sync_line else {}),
        **({"per_rank": per_rank} if per_rank else {}),
        "gpu_launches": int(launches),
        "graph_overflow": bool(overflow_steps),
        "clocks": clk.summary(),
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak,
                     "peak_source": "measured" if peaks else "fallback", "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_source, "secondary": secondary,
                     "algorithmic_bytes_per_launch": alg[dom], "avg_launch_ms": stage_ms[dom],
                     "frame": {"algorithmic_bytes": frame_alg,
                               "achieved_gbs": frame_alg / ((ms_total / K) * 1e-3) / 1e9,
                               "frac": frame_alg / ((ms_total / K) * 1e-3) / 1e9 / peak}},
        "stage_ms": {k: round(v, 4) for k, v in stage_ms.items()},
        "stage_ms_note": "per-stage CUDA events, measured in a separate eager pass over the same K flushed steps "
                         f"({ms_instrumented / K:.4f} ms/step with the events on); 'scan' = per-splat depth sort + offsets scan",
        "host_us_in_forward": {k: round(v, 1) for k, v in host_us.items()},
        "wall_s_timed_region": wall_timed,
    }
    if b3 is not None:
        line["baseline_b3"] = b3
    if world == 1 and not args.no_cpu_baseline:
        line.update(cpu_and_parity(params, verts, faces, cams_host, pc, posed, cams_dev, bg, gout, dev))
    print(json.dumps(line), flush=True)
    finish(world, dev)


def dump_outputs(directory, tensors):
    """Writes each tensor as <directory>/<name>.npy in float32 (float64 stays float64).  When together they would exceed
    DUMP_BYTES, every one is flattened and keeps the same share of its elements, chosen with a fixed seed and kept in
    their original order, so that two runs of the same configuration write the same elements."""
    import numpy as np

    host = {}
    for name, t in tensors.items():
        if t is None:
            raise RuntimeError(f"--dump-outputs: the timed step produced no {name}")
        a = t.detach().cpu().numpy()
        host[name] = a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False)
    total = sum(a.nbytes for a in host.values())
    share = min(1.0, DUMP_BYTES / total) if total else 1.0
    os.makedirs(directory, exist_ok=True)
    for name, a in host.items():
        if share < 1.0:
            n = max(1, int(a.size * share))
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def finish(world, dev):
    """Multi-rank teardown.  With CUDA graphs that captured NCCL kernels still alive, dist.destroy_process_group()
    never returned on the 2-GPU box (both ranks had printed their results; the launcher then waited for its 900 s
    limit).  Nothing is left to clean up that the process exit does not release: meet once, flush, leave."""
    if world == 1:
        return
    import torch.distributed as dist

    torch.cuda.synchronize(dev)
    dist.barrier()
    torch.cuda.synchronize(dev)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


def cpu_and_parity(params, verts, faces, cams_host, pc, posed, cams_dev, bg, gout, dev):
    """cpu_baseline (the oracle port timed on the host cores, + the 1-thread binding time of SURVEY 8d baseline 2) and
    parity_check: frame 0 of this workload, eager fused route on the GPU vs the oracle (oracle/fused_reference.py)."""
    import numpy as np

    from gaussianavatars_b200 import synthetic as syn
    from gaussianavatars_b200.renderer import render
    from oracle import binding as ob
    from oracle import fused_reference as fr

    out = {}
    cores = host_cpus()
    cpu_frames(params, verts, faces, cams_host, 1)
    frames = 6
    t, tb = cpu_frames(params, verts, faces, cams_host, frames)
    sec = sum(t) / len(t)
    # SURVEY 8(d) baseline 2: the reference's PyTorch-only CPU transform path (binding getters), one thread
    default_threads = torch.get_num_threads()
    torch.set_num_threads(1)
    b = params["binding"].long()
    tb1 = []
    for i in range(5):
        t0 = time.perf_counter()
        fr_ = ob.update_mesh_properties(syn.pose_mesh(verts, i), faces)
        ob.get_xyz(params["_xyz"], b, fr_["face_center"], fr_["face_orien_mat"], fr_["face_scaling"])
        ob.get_scaling(params["_scaling"], b, fr_["face_scaling"])
        ob.get_rotation(params["_rotation"], b, fr_["face_orien_quat"])
        ob.get_opacity(params["_opacity"])
        ob.get_features(params["_features_dc"], params["_features_rest"])
        tb1.append(time.perf_counter() - t0)
    torch.set_num_threads(cores)
    out["cpu_baseline"] = {"value": 1.0 / sec, "unit": "frames/s", "cores": cores, "kind": "port",
                           "sample": f"{frames} full frames of the same workload (eager torch binding getters + "
                                     f"C oracle rasterizer fwd+bwd, OpenMP x{cores}); the port is the parity CHECKER "
                                     "being timed (scalar C, one tile per task), not a tuned CPU renderer",
                           "machine_cpus": os.cpu_count(), "torch_threads": default_threads,
                           "binding_ms_per_frame": 1e3 * sum(tb) / len(tb),
                           "binding_ms_per_frame_1thread": 1e3 * sorted(tb1)[len(tb1) // 2]}
    # parity of the benchmarked frame
    cam = cams_host[0]
    for p in pc.parameters():
        p.grad = None
    v = posed[0].detach().clone().requires_grad_(True)
    pc.update_mesh_properties(v)
    o = render(cams_dev[0], pc, Pipe, bg)
    o["render"].backward(gout)
    torch.cuda.synchronize(dev)
    ref = fr.fused_frame(params, posed[0].detach().cpu(), faces, cam, WIDTH, HEIGHT, bg.cpu(), SH_DEGREE, dL_dimage=gout.cpu())
    d = np.abs(o["render"].detach().cpu().numpy().astype(np.float64) - ref["image"])
    grads = {k: getattr(pc, k).grad.cpu().numpy() for k in fr.RAW}
    grads["means2D"] = o["viewspace_points"].grad.cpu().numpy()
    grads["verts"] = v.grad.cpu().numpy()
    worst = {}
    for k, gc in grads.items():
        gr = ref["grads"][k].astype(np.float64)
        scale = float(np.abs(gr).max()) + 1e-300
        e = np.abs(gc.astype(np.float64).reshape(gr.shape) - gr)
        tol = 2e-5 * scale + 1e-3 * np.abs(gr)
        worst[k] = {"max_abs_over_max_ref": float(e.max() / scale), "beyond_atol_rtol": int((e > tol).sum()), "n": int(e.size)}
    out["parity_check"] = {
        "frame": "camera 0 of this workload, eager fused route vs oracle/fused_reference.py (eager getters under torch "
                 "autograd -> C oracle)",
        "image_max_abs": float(d.max()), "image_values_over_1e-4": int((d > 1e-4).sum()), "image_values": int(d.size),
        "radii_mismatches": int((o["radii"].cpu().numpy() != ref["radii"]).sum()),
        "grad_gate": "|d| <= 2e-5 max|ref| + 1e-3 |ref|", "grads": worst,
        "oracle_instances_exact_list": ref["N"], "tile_list_max": ref["tile_list_max"]}
    return out


if __name__ == "__main__":
    main()
