"""One training frame of the hot path as ONE CUDA graph.

    frame = GraphedFrame(pc, width, height, fovx, fovy, bg, loss="l1_u8")
    frame.set_inputs(camera=cam, verts=posed_vertices, gt_u8=ground_truth)     # device or pinned-host tensors
    frame.run()                                                                # enqueue one replay
    pc._xyz.grad, frame.verts.grad, frame.loss ...                             # static result tensors

What is captured (the data flow of the reference training step, train.py:113-170, with the fused route of
`render()`): [H2D copy of the camera block and the uint8 ground truth] -> per-face frame of the posed mesh
(scene/flame_gaussian_model.py:137-147) -> fused binding + rasterizer forward (gaussian_renderer/__init__.py:19-101) ->
loss (utils/loss_utils.py:17-63) -> backward down to the raw splat parameters and the mesh vertices -> [D2H copy of
the loss scalar].  ~25 launches, memsets and copies become one `cudaGraphLaunch`: the host is off the step.

The forward inside the graph runs with `GAB200_SYNC_NONE` (include/gab200_rasterizer.h): the instance capacity is
fixed at capture time from the frames rendered eagerly before it (x `headroom`).  A replay that needs more than the
capacity renders from a truncated instance list -- memory-safe, wrong -- and raises the slot's sticky device flag;
`run(check=True)` waits for the replay, and on overflow grows the capacity, re-captures and replays: its results are
then exactly those of an eager `render()`.  `run(check=False)` never touches the host; call `overflowed()` whenever
convenient (bench.py does after its timed loop).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import rasterizer as R
from .renderer import render
from .rasterizer import l1_loss_u8
from .training import binding_regularizers, photometric_loss


class _Pipe:
    debug = False
    compute_cov3D_python = False
    convert_SHs_python = False


class _GraphCamera:
    """Camera whose matrices are views into the graph's static camera block."""

    def __init__(self, W, H, fovx, fovy, block):
        self.image_width, self.image_height, self.FoVx, self.FoVy = W, H, fovx, fovy
        self.world_view_transform = block[0:16].view(4, 4)
        self.full_proj_transform = block[16:32].view(4, 4)
        self.camera_center = block[32:35]


def camera_block(cam) -> torch.Tensor:
    """(35,) float32: world_view_transform (16) | full_proj_transform (16) | camera_center (3) of a camera object."""
    return torch.cat((cam.world_view_transform.reshape(-1).float(), cam.full_proj_transform.reshape(-1).float(),
                      cam.camera_center.reshape(-1).float()))


def pair_with_deferred_reduce(frames, buffers, side_work_at: str = "start"):
    """Two frames of one model used alternately, each with its own caller-owned gradient buffer
    (dist.SymmetricGradBuffer, mode "two_shot" or "plain"): frame k's backward fills buffers[k], and a forked branch of
    frame k's graph all-reduces buffers[1-k] -- the gradients of the PREVIOUS step -- while frame k computes.  After
    replay i the reduced gradients of step i-1 are in buffers[1-k] (`reduced_grads(frames, buffers, k)`), those of
    step i become available after replay i+1 or `buffers[k].reduce()`.  The collective leaves the critical path; the
    price is that an optimizer consuming reduced gradients runs one replay behind (DESIGN.md section 6).
    Call before capture()."""
    if len(frames) != 2 or len(buffers) != 2:
        raise ValueError("a deferred-reduction pair is two frames and two buffers")
    for k, f in enumerate(frames):
        mine, other = buffers[k], buffers[1 - k]

        def before(f=f, mine=mine):
            f.pc.symm_grad = mine
            mine.begin()

        f.before_backward = before
        f.after_backward = lambda mine=mine: mine.end(reduce=False)
        f.side_work = other.reduce
        f.side_work_at = side_work_at
        if f._side is None:
            f._side = torch.cuda.Stream(device=f.device)
    return frames


def reduced_grads(buffers, k):
    """Views (in pc.parameters() order) of the all-reduced gradients available after replaying frame k of a
    deferred-reduction pair: those of the step before."""
    return buffers[1 - k].all_views[0]


class GraphedFrame:
    def __init__(self, pc, width: int, height: int, fovx: float, fovy: float, bg: torch.Tensor, loss: str = "l1_u8",
                 lambda_dssim: float = 0.2, host_inputs: bool = False, capacity: Optional[int] = None,
                 headroom: float = 1.25, after_backward=None, warm_cameras=None, regularizers: Optional[dict] = None,
                 before_backward=None, side_work=None, side_work_at: str = "start", flame=None, flame_param=None,
                 warm_timesteps=None):
        """loss: "l1_u8" (L1 vs a uint8 ground truth), "photometric" ((1-l) L1 + l (1-SSIM) vs a uint8 ground truth) or
        "dL_dimage" (the caller supplies dL/dimage in `self.dL_dimage`).
        host_inputs: the frame owns pinned STAGING tensors (`cam_stage` (35,) float32, `gt_stage` (3,H,W) uint8) that a
        loader fills, and the graph ends with a D2H copy of the loss to `loss_host`.  How the staged inputs reach the
        device: (a) `set_inputs()` with HOST tensors uploads them on this frame's copy stream and `run()` makes the
        replay wait for them on the GPU; or (b) two frames used alternately prefetch for each other INSIDE their graphs
        (`a.prefetch_for(b); b.prefetch_for(a)` before capture): a forked branch of a's graph copies b's staging
        tensors into b's device buffers while a computes, so the upload of step i+1 runs under step i with no event
        between graphs.  (An H2D node at the HEAD of the consuming graph is what does not work: measured, a 140-byte
        camera copy queued on the copy engine behind the 6 MB ground truth of the next step and delayed every replay
        by the full 124 us of that transfer; and ordering uploads against replays with cross-stream events costs
        ~40 us per step, profiles/r02/e2e_loop_probe.json.)
        after_backward: optional callable run inside the capture after backward (e.g. the gradient all-reduce).
        before_backward: the same, right before backward (e.g. attach this frame's gradient buffer to the model).
        side_work: optional callable captured on a FORKED branch of the graph that runs concurrently with the whole
        frame and is joined at its end -- e.g. the all-reduce of the PREVIOUS step's gradient buffer
        (dist.SymmetricGradBuffer.reduce of the other frame of an alternating pair), which then costs no step time.
        warm_cameras: camera blocks (35,) rendered eagerly before the capture to size the instance capacity.
        regularizers: keyword arguments of `binding_regularizers` (threshold_xyz, lambda_scale, ...; {} = the
        reference's defaults): the position / scale terms of train.py:134-146 are added to the loss inside the graph.
        flame / flame_param: a FusedFlameHead and its parameters (io.load_flame_param's layout).  The graph then starts
        from a device timestep (`set_inputs(timestep=t)`) instead of posed vertices: FLAME forward -> face frame -> ...
        -> backward -> FLAME backward, and after each replay the `.grad` of every flame_param tensor that requires grad
        is the graph's static (T,k) gradient (one non-zero row).  warm_timesteps: the timesteps of the eager frames
        that size the instance capacity.  FLAME gradients are not all-reduced, so this mode refuses a process group of
        more than one rank."""
        if loss not in ("l1_u8", "photometric", "dL_dimage"):
            raise ValueError("loss must be 'l1_u8', 'photometric' or 'dL_dimage'")
        self.pc, self.W, self.H, self.fovx, self.fovy = pc, int(width), int(height), float(fovx), float(fovy)
        self.loss_kind, self.lambda_dssim, self.host_inputs = loss, float(lambda_dssim), bool(host_inputs)
        self.after_backward = after_backward
        self.before_backward = before_backward   # e.g. SymmetricGradBuffer.begin
        self.side_work = side_work
        self.side_work_at = side_work_at   # "start": beside the whole frame; "backward": forked after the forward
        self.regularizers = regularizers
        if regularizers is not None and loss == "dL_dimage":
            raise ValueError("regularizers need a scalar loss ('l1_u8' or 'photometric')")
        self.headroom = float(headroom)
        dev = pc._xyz.device
        self.device = dev
        self.bg = bg.to(dev).float().contiguous()
        self.cam = torch.zeros(35, dtype=torch.float32, device=dev)
        self.camera = _GraphCamera(self.W, self.H, self.fovx, self.fovy, self.cam)
        if (flame is None) != (flame_param is None):
            raise ValueError("flame and flame_param go together")
        if flame is not None and torch.distributed.is_available() and torch.distributed.is_initialized() \
                and torch.distributed.get_world_size() > 1:
            raise RuntimeError("GraphedFrame(flame=...) does not all-reduce the FLAME-parameter gradients: with "
                               f"{torch.distributed.get_world_size()} ranks the replicas would diverge")
        self.flame, self.flame_param = flame, flame_param
        if flame is None:
            self.verts = pc.verts_rest.detach().clone().contiguous().requires_grad_(True)
            self.timestep = None
        else:   # posed by the graph itself: `verts` is the FLAME output of the last replay
            self.verts = None
            self.timestep = torch.zeros(1, dtype=torch.int32, device=dev)
        self._warm_t = list(warm_timesteps) if warm_timesteps is not None else None
        self.gt = torch.zeros((3, self.H, self.W), dtype=torch.uint8, device=dev) if loss != "dL_dimage" else None
        self.dL_dimage = torch.zeros((3, self.H, self.W), dtype=torch.float32, device=dev) if loss == "dL_dimage" else None
        self.cam_host = torch.zeros(35, dtype=torch.float32).pin_memory() if host_inputs else None  # staging
        self.cam_stage = self.cam_host
        self.gt_stage = (torch.zeros((3, self.H, self.W), dtype=torch.uint8).pin_memory()
                         if host_inputs and self.gt is not None else None)
        self._prefetch_target = None
        self._gt_ready = self._done = None   # events ordering the ground-truth upload against the replays
        self.loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
        self.loss = None
        self.image = self.radii = self.viewspace_points = None
        self.graph = None
        self.slot = None
        self.replays = 0
        self.captures = 0
        self._side = torch.cuda.Stream(device=dev) if (host_inputs or side_work is not None) else None
        self._uploads = bool(host_inputs)
        self._capacity = capacity
        self._warm = list(warm_cameras) if warm_cameras is not None else None

    # ---- inputs ------------------------------------------------------------------------------------------------
    def set_inputs(self, camera=None, verts=None, gt_u8=None, dL_dimage=None, timestep=None):
        """Copies new inputs into the static buffers (device tensors) / staging buffers (host_inputs).  `timestep`
        (an int or an int32 tensor) is the FLAME frame of a graph built with flame=; `verts` is the posed mesh of one
        built without."""
        if self.flame is not None and verts is not None:
            raise ValueError("this GraphedFrame poses the mesh with FLAME: pass timestep=, not verts=")
        if self.flame is None and timestep is not None:
            raise ValueError("timestep= needs a GraphedFrame built with flame= and flame_param=")
        if timestep is not None:
            if isinstance(timestep, torch.Tensor):
                self.timestep.copy_(timestep.reshape(1), non_blocking=True)
            else:
                self.timestep.fill_(int(timestep))
        if camera is not None:
            blk = camera if isinstance(camera, torch.Tensor) else camera_block(camera)
            if blk.device.type == "cpu" and self._uploads:
                if not blk.is_pinned():      # stage pageable memory (after any upload still reading the staging copy)
                    self._side.synchronize()
                    self.cam_host.copy_(blk)
                    blk = self.cam_host
                self._upload(self.cam, blk)
            else:
                self.cam.copy_(blk, non_blocking=True)
        if verts is not None:
            with torch.no_grad():
                self.verts.copy_(verts.reshape(self.verts.shape), non_blocking=True)
        if gt_u8 is not None:
            if gt_u8.device.type == "cpu" and self._uploads:
                self._upload(self.gt, gt_u8)
            else:
                self.gt.copy_(gt_u8, non_blocking=True)
        if dL_dimage is not None:
            self.dL_dimage.copy_(dL_dimage, non_blocking=True)

    def prefetch_for(self, other: "GraphedFrame"):
        """This frame's graph will, on a forked branch, copy `other`'s pinned staging tensors (cam_stage, gt_stage)
        into `other`'s device inputs while it computes.  Call before capture()."""
        if not (self.host_inputs and other.host_inputs):
            raise ValueError("prefetching needs host_inputs=True on both frames")
        self._prefetch_target = other
        return self

    def upload_staged(self):
        """Eager upload of this frame's own staging tensors (the first step of a prefetching pair)."""
        self.cam.copy_(self.cam_stage, non_blocking=True)
        if self.gt_stage is not None:
            self.gt.copy_(self.gt_stage, non_blocking=True)

    def _upload(self, dst, src_host):
        """H2D on the copy stream: after the last replay that read `dst`, concurrently with the main stream."""
        if self._done is not None:
            self._side.wait_event(self._done)
        with torch.cuda.stream(self._side):
            dst.copy_(src_host, non_blocking=True)
            self._gt_ready = torch.cuda.Event()
            self._gt_ready.record(self._side)

    # ---- the step body (run eagerly for warm-up, then captured) --------------------------------------------------
    def _params(self):
        ps = list(self.pc.parameters())
        if self.flame_param is not None:
            ps += [t for t in self.flame_param.values() if isinstance(t, torch.Tensor) and t.requires_grad]
        return ps

    def _body(self):
        pc = self.pc
        for p in self._params():
            p.grad = None
        if self.flame is None:
            self.verts.grad = None
        other = self._prefetch_target
        forked = other is not None or self.side_work is not None
        if forked:   # forked branch: runs while this frame computes
            cur = torch.cuda.current_stream(self.device)
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                if other is not None:   # the other frame's next inputs travel
                    other.cam.copy_(other.cam_stage, non_blocking=True)
                    if other.gt_stage is not None:
                        other.gt.copy_(other.gt_stage, non_blocking=True)
                if self.side_work is not None and self.side_work_at == "start":
                    self.side_work()
        if self.flame is not None:
            self.verts = self.flame.mesh_at(self.flame_param, self.timestep)
        pc.update_mesh_properties(self.verts)
        out = render(self.camera, pc, _Pipe, self.bg)
        img = out["render"]
        if self.loss_kind in ("l1_u8", "photometric"):
            loss = l1_loss_u8(img, self.gt) if self.loss_kind == "l1_u8" else photometric_loss(img, self.gt, self.lambda_dssim)
            if self.regularizers is not None:
                lx, ls = binding_regularizers(pc._xyz, pc._scaling, out["radii"], getattr(pc, "binding", None),
                                              getattr(pc, "face_scaling", None), **self.regularizers)
                loss = loss + lx + ls
            self._fork_side_at_backward()
            if self.before_backward is not None:
                self.before_backward()
            loss.backward()
        else:
            loss = None
            self._fork_side_at_backward()
            if self.before_backward is not None:
                self.before_backward()
            img.backward(self.dL_dimage)
        if self.after_backward is not None:
            self.after_backward()
        if loss is not None:
            self.loss = loss.detach()
            self.loss_host.copy_(self.loss, non_blocking=True)
        if forked:   # join the branch (a captured fork must end inside the graph)
            torch.cuda.current_stream(self.device).wait_stream(self._side)
        self.image, self.radii, self.viewspace_points = img.detach(), out["radii"], out["viewspace_points"]

    def _fork_side_at_backward(self):
        if self.side_work is not None and self.side_work_at == "backward":
            self._side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(self._side):
                self.side_work()

    # ---- capture ---------------------------------------------------------------------------------------------------
    def _learn_capacity(self):
        """Eager frames (sync modes EXACT then LATE) over the warm-up cameras: their instance counts size the graph."""
        hints = R.hints_of(self.pc)
        key = (self.device, self.W, self.H, self.pc._xyz.shape[0])
        n_max, lo, hi = 0, 0xFFFFFFFF, 0
        blocks = self._warm if self._warm else [self.cam.clone()]
        steps = [None]
        if self.flame is not None:
            steps = self._warm_t if self._warm_t else [self.timestep.clone()]
        # eager frames on a side stream (torch's recipe for whole-step capture): nothing autograd creates here may be
        # tied to the legacy default stream
        cur = torch.cuda.current_stream(self.device)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for rep in range(2):
                for blk, ts in [(b, t) for b in blocks for t in steps]:
                    self.cam.copy_(blk)
                    if ts is not None:
                        self.set_inputs(timestep=ts)
                    self._body()
                    info = hints.last or {}
                    n_max = max(n_max, int(info.get("num_rendered", 0)))
                    d = hints.get(key)[1]
                    if d[1] > d[0]:  # union of the (already widened) depth-key ranges: one bucket grid fits every camera
                        lo, hi = min(lo, d[0]), max(hi, d[1])
        cur.wait_stream(side)
        torch.cuda.synchronize(self.device)
        # release what the eager frames left on the model / on this object (tensors with autograd history)
        self.pc.face_center = self.pc.face_orien_mat = self.pc.face_scaling = None
        self.image = self.radii = self.viewspace_points = self.loss = None
        if self.flame is not None:
            self.verts = None
        return n_max, ((lo, hi) if hi > lo else (0, 0))

    def capture(self, capacity: Optional[int] = None):
        dev = self.device
        n_max, depth = self._learn_capacity()
        if capacity is None:
            capacity = self._capacity if self._capacity else int(n_max * self.headroom) + 16384
        self.slot = R.CaptureSlot(dev, capacity, depth)
        self.graph = torch.cuda.CUDAGraph()
        R._capture_slot = self.slot
        try:
            with torch.cuda.graph(self.graph):
                self._body()
                self.slot.flag_host.copy_(self.slot.flag, non_blocking=True)
        finally:
            R._capture_slot = None
        # the tensors autograd left in .grad during the capture ARE the graph's outputs: remember them, a second
        # GraphedFrame of the same model re-points .grad at its own when it captures
        self.grads = [p.grad for p in self._params()]
        self.flat_grad = getattr(self.pc, "flat_grad", None)
        self.captures += 1
        return self

    # ---- replay ----------------------------------------------------------------------------------------------------
    def run(self, check: bool = False):
        if self.graph is None:
            self.capture()
        if self._gt_ready is not None:   # a ground-truth upload is in flight on the copy stream
            torch.cuda.current_stream(self.device).wait_event(self._gt_ready)
            self._gt_ready = None
        self.graph.replay()
        self.replays += 1
        if self._uploads:
            self._done = torch.cuda.Event()
            self._done.record()
        for p, g in zip(self._params(), self.grads):
            p.grad = g
        self.pc.flat_grad = self.flat_grad
        if check and self.overflowed(wait=True):
            self.regrow()
            self.graph.replay()
            self.replays += 1
            for p, g in zip(self._params(), self.grads):
                p.grad = g
            self.pc.flat_grad = self.flat_grad
            if self.overflowed(wait=True):
                raise RuntimeError("GraphedFrame: the frame still overflows its instance capacity after re-capture")
        return self

    def overflowed(self, wait: bool = True) -> bool:
        """True if any replay since the last (re-)capture needed more than the captured capacity."""
        if self.slot is None:
            return False
        if wait:
            torch.cuda.current_stream(self.device).synchronize()
        return bool(int(self.slot.flag_host[0]) != 0)

    def counters(self) -> dict:
        """Frame counters of the most recent finished replay (host copy; synchronise first for an exact answer)."""
        c = self.slot.counters
        return dict(num_rendered=int(c[R.N.CTR_NUM_RENDERED]) & 0xFFFFFFFF, capacity=int(c[R.N.CTR_CAPACITY]) & 0xFFFFFFFF,
                    bucket_overflow=int(c[R.N.CTR_BUCKET_OVERFLOW]), listed=int(c[R.N.CTR_NUM_LISTED]) & 0xFFFFFFFF)

    def regrow(self):
        """Re-capture with the capacity the overflowing frame asked for (x headroom) and a fresh depth range."""
        torch.cuda.synchronize(self.device)
        need = self.counters()["num_rendered"]
        cap = max(int(need * self.headroom) + 16384, int(self.slot.capacity * 1.5))
        self.graph = None
        self.capture(capacity=cap)
