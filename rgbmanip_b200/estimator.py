"""Drop-in for ``models.pose_estimator.AdaPose.interface_v5.AdaPoseEstimator_v5`` (RGBManip).

Same constructor (``env, cfg, logger``), same ``estimate`` / ``predict`` signatures and return values
(interface_v5.py:39-56,213-374): host numpy in, ``np.ndarray [num_envs, 8, 3]`` float64 world-frame box corners
out, the ``unit cube + 10`` sentinel for environments whose mask is empty in either view or whose fit is not
finite.  The per-env Python loop of the reference is replaced by chunked batches on the device pipeline
(:class:`rgbmanip_b200.engine.Engine`); there is no CPU fallback.

Deliberate deviations from the live reference, all documented in DESIGN.md:
  * inference runs in eval mode (the reference never calls ``.eval()``: SURVEY.md finding 0.3-1);
  * the random 1024-pixel subset is drawn by a counter-based hash on the device instead of the global numpy
    RNG (same distribution; pass ``choose=`` to replay the reference's stream exactly);
  * ``draw_result`` (interface_v5.py:364) and the view-2 decode branch are dead work and are not computed;
  * float64 HOST frames are demoted to float32 while they are staged for upload.  The reference's float64 frames are the
    simulator's float32 renders stored in ``np.zeros`` queues (rl_pose.py:94,196), for which this is lossless; for other
    float64 data it moves the crop by <= 6e-8.  ``cfg["keep_float64"] = True`` (or passing float64 CUDA tensors) keeps
    the cv2-in-double interpolation of interface_v5.py:148;
  * uint8 RGB is accepted as a 4x smaller upload and means ``rgb / 255`` (torchvision ToTensor semantics).

Inputs may be numpy arrays, torch host tensors (pinned or pageable) or CUDA tensors (zero-copy).  The batch is cut into equal
chunks of at most ``max_envs`` environments; uploads of chunk i+1 overlap the kernels of chunk i, pageable host memory goes
through pinned staging buffers, a small first chunk (``cfg["first_chunk_envs"]``, default 16) followed by doubling ones starts
the kernels early, and of every host frame only the rows under its crop window are uploaded (``cfg["window_upload"]``, default
on: the masks go first, the device returns the windows, see ``_upload_window_rows``).
"""
from __future__ import annotations

import numpy as np
import torch

from . import weights as W
from .engine import Engine

try:  # inside an RGBManip checkout the real base class is importable; keep isinstance() relations intact
    from models.pose_estimator.base_estimator import BasePoseEstimator  # type: ignore
except Exception:  # pragma: no cover - stand-alone use
    class BasePoseEstimator:  # mirrors models/pose_estimator/base_estimator.py:5-21
        def __init__(self, env, cfg, logger):
            self.env = env
            self.cfg = cfg
            self.logger = logger

        def append_picture(self, pic, pose):
            pass

        def estimate(self):
            pass


DEFAULT_BBOX = np.asarray([[0, 0, 0], [0, 0, 1], [0, 1, 0], [0, 1, 1],
                           [1, 0, 0], [1, 0, 1], [1, 1, 0], [1, 1, 1]], dtype=np.float64) + 10.0


def chunk_bounds(N, max_envs, first=0):
    """[lo, hi) chunk boundaries of a batch of N environments: equal chunks of at most ``max_envs`` (every chunk size is replayed
    as a CUDA graph; a short tail chunk would miss both the graph and the whole-wave sizing).  ``first`` > 0 (frames coming
    from the host): a small chunk goes ahead and the following ones double in size (first, 2 first, 4 first, ...) until the
    equal split takes over -- the upload of chunk i+1 then fits under the kernels of chunk i, so only the first small upload is
    exposed instead of a full chunk's (at 8 GPUs a shard is 128 envs = 1 GB of fp32 frames against 43 ms of kernels)."""
    bounds, lo = [], 0
    size = min(int(first), max_envs)
    if size > 0 and N > max_envs:
        while size < max_envs and N - lo - size >= size:
            bounds.append((lo, lo + size))
            lo += size
            size = min(2 * size, max_envs)
    rest = N - lo
    if rest > 0:
        nch = -(-rest // max_envs)
        base, rem = divmod(rest, nch)
        for i in range(nch):
            hi = lo + base + (1 if i < rem else 0)
            bounds.append((lo, hi))
            lo = hi
    return bounds


AUTO_CHUNK_MAX = 74       # envs per chunk an auto-sized workspace grows to: 148 frames = whole waves of 128-row tiles on 148 SMs, 18 GB

_BOX_SIGNS = np.array([[1, 1, 1], [1, 1, -1], [-1, 1, 1], [-1, 1, -1], [1, -1, 1], [1, -1, -1], [-1, -1, 1], [-1, -1, -1]], np.float64)


_PNP_POOL = None


def _pnp_one(nocs, pts2d, scale, valid, K, E1):
    """One environment of :func:`pnp_box_tail` -> [8,3] float64."""
    import cv2
    ts = np.float64(scale)
    if not valid or not np.isfinite(ts):
        return DEFAULT_BBOX          # NaN scale: the reference's box is NaN too and fails its finite check -> sentinel
    temp = nocs * ts                                         # float32 array * np.float64 scalar, as in the reference
    try:
        ok, rv, tv, _ = cv2.solvePnPRansac(temp, pts2d, K, np.zeros(4), flags=cv2.SOLVEPNP_EPNP, reprojectionError=3.0)
        if ok:
            crit = (cv2.TERM_CRITERIA_MAX_ITER + cv2.TERM_CRITERIA_EPS, 20, 1e-6)
            rv, tv = cv2.solvePnPRefineVVS(temp, pts2d, K, None, rv, tv, criteria=crit)
        Rm, _ = cv2.Rodrigues(rv)
    except cv2.error:
        return DEFAULT_BBOX
    size = 2 * np.max(np.abs(nocs), axis=0) * ts
    sRT = np.eye(4).astype(np.float32)                       # float32 matrix, no scale in it (interface_v5.py:359-361)
    sRT[:3, :3] = Rm
    sRT[:3, 3] = np.asarray(tv).flatten()
    cam = sRT @ np.vstack([(_BOX_SIGNS * (size / 2)).T, np.ones((1, 8), np.float32)])
    cam = cam[:3] / cam[3]
    with np.errstate(all="ignore"):
        try:
            inv = np.linalg.inv(E1)
        except np.linalg.LinAlgError:
            return DEFAULT_BBOX
    if np.isfinite(inv).all() and np.isfinite(cam).all():
        return (inv[:3, :3] @ cam + inv[:3, 3:4]).T
    return DEFAULT_BBOX


def pnp_box_tail(nocs, pts2d, scale, valid, K, E1):
    """Host tail of branch C, per environment as the reference runs it: ``estimatePnPRansac`` (align.py:104-115) with size = the
    median scale of the triangulated matches, then the box + world transform + finite check of interface_v5.py:350-374.  The
    PnP is the reference's own OpenCV call (its RANSAC lives inside cv2 and seeds its generator per call, so the result does not
    depend on the thread); everything before it ran on the device.  The environments are independent and cv2 releases the GIL:
    they go through a host thread pool (18 ms per environment on one thread is what bounds this branch).
    nocs [n,P,3] f32, pts2d [n,P,2] f32, scale [n] f64, valid [n], K [n,3,3], E1 [n,4,4] -> [n,8,3] float64."""
    global _PNP_POOL
    n = len(scale)
    if n <= 1:
        return np.stack([np.asarray(_pnp_one(nocs[e], pts2d[e], scale[e], valid[e], K[e], E1[e]), np.float64) for e in range(n)]).reshape(n, 8, 3)
    if _PNP_POOL is None:
        import os
        from concurrent.futures import ThreadPoolExecutor
        _PNP_POOL = ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1), thread_name_prefix="adapose-pnp")
    out = list(_PNP_POOL.map(lambda e: _pnp_one(nocs[e], pts2d[e], scale[e], valid[e], K[e], E1[e]), range(n)))
    return np.stack([np.asarray(o, np.float64) for o in out])


class AdaPoseEstimator_v5(BasePoseEstimator):
    ARCH = "v5"          # which network sits behind the interface (weights.param_table)

    def __init__(self, env, cfg, logger, state_dict=None, device=None, max_envs=None, precision=None, devices=None, **engine_kw):
        super().__init__(env, cfg, logger)
        self.cfg = cfg
        self._replicas = None
        engine_kw = dict(engine_kw, arch=self.ARCH)
        regress = bool(cfg.get("direct_regression", True))
        self._branch_c = (not regress) and not cfg.get("use_depth", True)
        if self._branch_c:
            # branch C (interface_v5.py:339-349): matching / triangulation / median scale run on the device, the PnP tail is the
            # reference's own OpenCV call on the host (align.py:104-115; its RANSAC lives inside cv2: "parity unpinned" there)
            import cv2  # noqa: F401  (fail at construction, not in the middle of an episode)
            engine_kw = dict(engine_kw, use_depth=False)
        if state_dict is None:
            if cfg.get("load", False):
                # same failure mode as the reference: a missing checkpoint raises from torch.load (interface_v5.py:55-56)
                state_dict = W.load_checkpoint(cfg["checkpoint_path"], regress_pose=regress, arch=self.ARCH)
            else:
                state_dict = W.init_state_dict(int(cfg.get("seed", 0)), regress_pose=regress, arch=self.ARCH)
        devices = devices if devices is not None else cfg.get("devices")
        if devices == "all":
            devices = list(range(torch.cuda.device_count()))
        if devices is not None and len(devices) > 1:
            # Single-process multi-GPU (SURVEY 8(b)/(e)): the reference builds ONE estimator in ONE process (train.py:238-240), so
            # an unmodified vec-env host reaches every GPU of the box through this object -- no torchrun.  One replica (engine,
            # weights, workspace, streams) per device, each driven by its own host thread; the ctypes calls and torch's CUDA calls
            # release the GIL, and a chunk is one CUDA-graph replay, so the host threads stay out of each other's way.
            from concurrent.futures import ThreadPoolExecutor
            devs = [torch.device(d if isinstance(d, (str, torch.device)) else f"cuda:{int(d)}") for d in devices]
            import threading
            self._tls = threading.local()
            self._pool = ThreadPoolExecutor(max_workers=len(devs), thread_name_prefix="adapose-gpu")
            def mk(d):
                from .dist import bind_to_gpu_numa
                bind_to_gpu_numa(d)          # this replica's pinned staging buffers land on the GPU's NUMA node
                kw = {k: v for k, v in engine_kw.items() if k != "arch"}
                return type(self)(env, {k: v for k, v in cfg.items() if k != "devices"}, logger, state_dict=state_dict,
                                  device=d, max_envs=max_envs, precision=precision, **kw)
            self._replicas = list(self._pool.map(mk, devs))
            self.device = devs[0]
            self.estimator = self._replicas[0].estimator     # the attribute the reference exposes (interface_v5.py:48)
            self._seed = int(cfg.get("sample_seed", 0))
            self._calls = 0
            return
        if devices is not None and len(devices) == 1:
            device = devices[0] if isinstance(devices[0], (str, torch.device)) else f"cuda:{int(devices[0])}"
        device = device or cfg.get("device", "cuda:%d" % torch.cuda.current_device() if torch.cuda.is_available() else "cuda:0")
        self.device = torch.device(device)
        # chunk capacity: an explicit ``max_envs`` / ``max_envs_per_chunk`` is final; otherwise the workspace starts at 16 environments
        # and grows with the batches it sees, up to AUTO_CHUNK_MAX per chunk (a drop-in user never sizes anything)
        self._auto_chunk = max_envs is None and "max_envs_per_chunk" not in cfg
        self._engine_args = dict(device=self.device, precision=precision or cfg.get("precision", "fp16f8"), regress_pose=regress,
                                 img_size=int(cfg.get("img_size", 224)), **engine_kw)
        self.estimator = Engine(state_dict, max_envs=int(max_envs or cfg.get("max_envs_per_chunk", 16)), **self._engine_args)
        self._seed = int(cfg.get("sample_seed", 0))
        self._calls = 0
        self._copy_stream = None
        self._stage_bufs = {}
        self._slot_free = [None, None]
        self._win_state = {}
        self._window_upload = bool(cfg.get("window_upload", True))
        self.h2d_bytes = 0          # bytes copied host -> device so far (bench.py reports the per-step figure)
        self._keep_f64 = bool(cfg.get("keep_float64", False))
        self._first_chunk = int(cfg.get("first_chunk_envs", 16))

    def _ensure_capacity(self, N):
        """Auto-sized workspace: rebuild the engine with a larger chunk capacity the first time a bigger batch shows up.  A
        multi-device estimator grows every replica to its share of N (the contiguous block :meth:`_estimate_multi` gives it)."""
        if self._replicas is not None:
            from .dist import shard_range
            world = len(self._replicas)
            self._on_replicas(lambda r: self._replicas[r]._ensure_capacity(len(range(*shard_range(int(N), r, world)[:2]))))
            return
        eng = self.estimator
        want = min(max(int(N), 1), AUTO_CHUNK_MAX)
        if not self._auto_chunk or want <= eng.E:
            return
        sd = eng.sd
        torch.cuda.synchronize(self.device)
        eng.close()
        self.estimator = eng = None
        self._stage_bufs, self._win_state, self._slot_free = {}, {}, [None, None]
        torch.cuda.empty_cache()
        self.estimator = Engine(sd, max_envs=want, **self._engine_args)

    def one_device_chunk(self, N):
        """Chunk capacity (environments) a one-device estimator of this configuration has for a batch of N environments: the
        explicit ``max_envs`` / ``max_envs_per_chunk``, else the auto-sized 16 .. AUTO_CHUNK_MAX.  The view ring keys its random
        draws by these chunks, so that a ring sharded over several devices draws what a one-device ring draws."""
        rep = self._replicas[0] if self._replicas is not None else self
        if not rep._auto_chunk:
            return rep.estimator.E
        return max(16, min(int(N), AUTO_CHUNK_MAX))

    def _on_replicas(self, fn, which=None):
        """``fn(r)`` for every replica index r (or those in ``which``), concurrently on the per-device host threads -> results in
        order.  Pool threads are not tied to a replica: a thread re-pins itself to the GPU's NUMA node when its replica changes."""
        def run(r):
            if getattr(self._tls, "bound", None) != r:
                from .dist import bind_to_gpu_numa
                bind_to_gpu_numa(self._replicas[r].device)
                self._tls.bound = r
            return fn(r)
        return list(self._pool.map(run, range(len(self._replicas)) if which is None else which))

    # -- helpers ---------------------------------------------------------------------------------
    _RGB_OK = (torch.uint8, torch.float32, torch.float64)
    _MASK_OK = (torch.uint8, torch.bool, torch.float32, torch.float64)

    @staticmethod
    def _as_tensor(a):
        return a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))

    def _pinned(self, key, slot, shape, dtype):
        """Reusable page-locked staging buffer (two slots per input: the host copy of chunk i+1 overlaps the upload of chunk i)."""
        k = (key, slot)
        buf = self._stage_bufs.get(k)
        if buf is None or buf.dtype != dtype or buf.shape[1:] != tuple(shape[1:]) or buf.shape[0] < shape[0]:
            buf = torch.empty((max(shape[0], self.estimator.E),) + tuple(shape[1:]), dtype=dtype).pin_memory()
            self._stage_bufs[k] = buf
        return buf[:shape[0]]

    def _upload(self, key, slot, t, dtype=None):
        """Host or device tensor -> device tensor of ``dtype`` on the current (copy) stream.  Pageable host memory goes
        through the pinned staging buffers (a multi-threaded host copy that also converts the dtype), so the PCIe copy is
        asynchronous and overlaps the previous chunk's kernels."""
        if t.is_cuda:
            t = t if dtype is None or t.dtype == dtype else t.to(dtype)
            return t.to(self.device, non_blocking=True).contiguous()
        dtype = dtype or t.dtype
        if t.is_pinned() and t.dtype == dtype and t.is_contiguous():
            return t.to(self.device, non_blocking=True)
        buf = self._pinned(key, slot, t.shape, dtype)
        buf.copy_(t)
        return buf.to(self.device, non_blocking=True)

    def _rgb_dtype(self, t):
        if t.dtype == torch.float64 and not t.is_cuda and not self._keep_f64:
            return torch.float32        # see the class docstring: float64 host frames are demoted while staging
        if t.dtype in self._RGB_OK:
            return t.dtype
        if t.dtype in (torch.float16, torch.bfloat16):
            return torch.float32
        raise TypeError(f"unsupported image dtype {t.dtype}: pass float RGB in [0, 1] (what the simulator renders) or uint8 in [0, 255]")

    # -- reference API ---------------------------------------------------------------------------
    def _stage_chunk(self, batches, choose, lo, hi, stream, slot):
        """Issue the host->device copies of envs [lo, hi) on ``stream`` (no-ops for tensors already on the device)."""
        K_b, rgb1_b, m1_b, E1_b, rgb2_b, m2_b, E2_b = batches
        ev_free = self._slot_free[slot]
        if ev_free is not None:
            ev_free.synchronize()       # the uploads that last used this slot's pinned buffers have completed
        with torch.cuda.stream(stream):
            t = dict(K=self._upload("K", slot, K_b[lo:hi], torch.float64), E1=self._upload("E1", slot, E1_b[lo:hi], torch.float64),
                     E2=self._upload("E2", slot, E2_b[lo:hi], torch.float64))
            for name, src in (("m1", m1_b), ("m2", m2_b)):
                m = src[lo:hi]
                if m.dtype not in self._MASK_OK:
                    m = m != 0          # integer segmentation ids: any non-zero id is foreground (never a cast that can wrap to 0)
                if m.dtype == torch.bool:
                    m = m.view(torch.uint8)
                t[name] = self._upload(name, slot, m)
            if rgb1_b.is_cuda or not self._window_upload or hi == lo:
                for name, src in (("rgb1", rgb1_b), ("rgb2", rgb2_b)):
                    t[name] = self._upload(name, slot, src[lo:hi], self._rgb_dtype(src))
                    self.h2d_bytes += 0 if src.is_cuda else t[name].numel() * t[name].element_size()
            else:
                self._upload_window_rows(t, (rgb1_b, rgb2_b), lo, hi, stream, slot)
            self.h2d_bytes += sum(t[k].numel() * t[k].element_size() for k in ("m1", "m2") if not (m1_b.is_cuda))
            t["c1"] = t["c2"] = None
            if choose is not None:
                t["c1"] = self._upload("c1", slot, choose[0][lo:hi], torch.int32)
                t["c2"] = self._upload("c2", slot, choose[1][lo:hi], torch.int32)
            ev = torch.cuda.Event()
            ev.record(stream)
            self._slot_free[slot] = ev
        return t, ev

    def _upload_window_rows(self, t, rgbs, lo, hi, stream, slot):
        """Host frames: upload only the image rows the crop window of each frame covers.  The masks (already queued on ``stream``)
        give the windows on the device (adp_mask_windows = the mask pass of the preprocessing); they are read back (a few
        hundred bytes) and every frame contributes rows [rmin, rmax) -- a contiguous block of the host frame -- to a persistent
        device frame buffer.  adp_preprocess reads nothing outside the window, so the stale rest of the buffer is never seen.
        A 480 x 640 fp32 frame is 3.7 MB, the rows of a typical 160-pixel window 1.2 MB."""
        from . import _lib as L
        eng = self.estimator
        n = hi - lo
        st = self._win_state.get(slot)
        if st is None:
            st = dict(win=torch.zeros((2 * eng.E, 4), dtype=torch.int32, device=self.device),
                      ws=torch.zeros((2 * eng.E, 4), dtype=torch.int32, device=self.device),
                      valid=torch.zeros(2 * eng.E, dtype=torch.uint8, device=self.device),
                      host=torch.zeros((2 * eng.E, 5), dtype=torch.int32).pin_memory(), frames={}, done=None)
            self._win_state[slot] = st
        cs = L.C.c_void_p(stream.cuda_stream)
        for v, key in enumerate(("m1", "m2")):
            m = t[key]
            code = {torch.uint8: L.DT_U8, torch.float32: L.DT_F32, torch.float64: L.DT_F64}[m.dtype]
            L.check(eng.lib.adp_mask_windows(L.ptr(m), code, n, m.shape[1], m.shape[2], L.ptr(st["ws"][v * n:]), L.ptr(st["win"][v * n:]),
                                             L.ptr(st["valid"][v * n:]), cs), "mask_windows")
        st["host"][:2 * n, :4].copy_(st["win"][:2 * n], non_blocking=True)
        st["host"][:2 * n, 4].copy_(st["valid"][:2 * n], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(stream)
        if st["done"] is not None:
            stream.wait_event(st["done"])        # the preprocessing that last read this slot's frame buffers has run
        ev.synchronize()
        wins = st["host"][:2 * n].tolist()
        for v, (name, src) in enumerate((("rgb1", rgbs[0]), ("rgb2", rgbs[1]))):
            dt = self._rgb_dtype(src)
            key = (v, dt, tuple(src.shape[1:]))
            buf = st["frames"].get(key)
            if buf is None:
                buf = torch.zeros((eng.E,) + tuple(src.shape[1:]), dtype=dt, device=self.device)
                st["frames"] = {k: b for k, b in st["frames"].items() if k[0] != v}      # one buffer per view and slot
                st["frames"][key] = buf
            direct = src.is_pinned() and src.dtype == dt
            stage = None if direct else self._pinned(name, slot, (n,) + tuple(src.shape[1:]), dt)
            row_bytes = src.shape[2] * src.shape[3] * buf.element_size()
            for f in range(n):
                r0, r1, _, _, ok = wins[v * n + f]
                if not ok:
                    continue
                if direct:
                    buf[f, r0:r1].copy_(src[lo + f, r0:r1], non_blocking=True)
                else:        # pageable (or float64) source: only these rows pass through the pinned staging buffer
                    stage[f, r0:r1].copy_(src[lo + f, r0:r1])
                    buf[f, r0:r1].copy_(stage[f, r0:r1], non_blocking=True)
                self.h2d_bytes += (r1 - r0) * row_bytes
            t[name] = buf[:n]
        t["_slot"] = slot

    def _chunk_bounds(self, N, on_host):
        return chunk_bounds(N, self.estimator.E, self._first_chunk if on_host else 0)

    def estimate(self, camera_intrinsic_batch, rgb1_batch, view1_mask_batch, view1_extrinsic_batch,
                 rgb2_batch, view2_mask_batch, view2_extrinsic_batch, choose=None, return_tensor=False, ransac_idx=None,
                 env_offset=0, sample_seed=None):
        """interface_v5.py:213-227.  Extra keyword arguments (all optional): ``choose`` / ``ransac_idx`` replay the reference's
        random draws; ``return_tensor`` returns the CUDA tensor without the device->host copy; ``env_offset`` is the global
        index of the first environment when the caller shards a larger batch (the device pixel sampler is keyed by
        (seed, global env index), so shards reproduce the unsharded result); ``sample_seed`` fixes that seed for one call
        (default: a per-call counter)."""
        if self._replicas is not None:
            return self._estimate_multi((camera_intrinsic_batch, rgb1_batch, view1_mask_batch, view1_extrinsic_batch,
                                         rgb2_batch, view2_mask_batch, view2_extrinsic_batch), choose, return_tensor, ransac_idx,
                                        env_offset, sample_seed)
        self._ensure_capacity(len(camera_intrinsic_batch))
        eng = self.estimator
        eng.check_error_flag(wait=False)        # a flag read posted by an earlier tensor-returning call
        batches = tuple(self._as_tensor(a) for a in (camera_intrinsic_batch, rgb1_batch, view1_mask_batch, view1_extrinsic_batch,
                                                     rgb2_batch, view2_mask_batch, view2_extrinsic_batch))
        K_b, rgb1_b, m1_b, _, rgb2_b, m2_b, _ = batches
        N = K_b.shape[0]
        for rgb, m in ((rgb1_b, m1_b), (rgb2_b, m2_b)):
            if rgb.dim() != 4 or rgb.shape[-1] != 3 or tuple(m.shape) != tuple(rgb.shape[:3]) or rgb.shape[0] != N:
                raise ValueError(f"expected rgb [N,H,W,3] and mask [N,H,W] for N = {N}, got {tuple(rgb.shape)} and {tuple(m.shape)}")
        if choose is not None:
            choose = tuple(self._as_tensor(c) for c in choose)
            for c in choose:
                if c.shape[0] != N or c.shape[1] != eng.P or bool((c < 0).any()) or bool((c >= eng.S * eng.S).any()):
                    raise ValueError(f"choose must be [N, {eng.P}] pixel indices in [0, {eng.S * eng.S})")
        out = torch.empty((N, 8, 3), dtype=torch.float64, device=self.device)
        self._calls += 1
        seed = (self._seed + 7919 * self._calls) if sample_seed is None else int(sample_seed)
        with torch.cuda.device(self.device):
            compute = torch.cuda.current_stream(self.device)
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(self.device)
            copy = self._copy_stream
            copy.wait_stream(compute)
            bounds = self._chunk_bounds(N, on_host=not rgb1_b.is_cuda)
            nxt = self._stage_chunk(batches, choose, *bounds[0], copy, 0) if bounds else None
            for i, (lo, hi) in enumerate(bounds):
                t, ev = nxt
                compute.wait_event(ev)
                for v in t.values():          # allocated on the copy stream, consumed on the compute stream
                    if isinstance(v, torch.Tensor) and v.is_cuda:
                        v.record_stream(compute)          # (harmless for the persistent window-upload frame buffers)
                ridx = None
                if ransac_idx is not None:      # [N,128,5] sample indices of the RANSAC fit (branch B parity replay)
                    ridx = self._as_tensor(ransac_idx[lo:hi]).to(torch.int32).to(self.device)
                box = eng.run_chunk(t["K"], t["rgb1"], t["m1"], t["E1"], t["rgb2"], t["m2"], t["E2"],
                                    seed=seed, choose1=t["c1"], choose2=t["c2"], ransac_idx=ridx, env0=int(env_offset) + lo)
                if self._branch_c:
                    out[lo:hi].copy_(self._pnp_tail(box, t["K"], t["E1"]))
                else:
                    out[lo:hi].copy_(box)
                if "_slot" in t:          # the slot's persistent frame buffers may be overwritten once this chunk's kernels ran
                    done = torch.cuda.Event()
                    done.record(compute)
                    self._win_state[t["_slot"]]["done"] = done
                # this chunk's kernels are queued: the host-side staging of the next chunk (and its upload) overlaps them
                nxt = self._stage_chunk(batches, choose, *bounds[i + 1], copy, (i + 1) & 1) if i + 1 < len(bounds) else None
            # watchdog + fp16 range flag (set by the last backbone layer on inf/NaN features, every chunk): read with the boxes
            eng.post_error_flag()
            if return_tensor:
                return out              # checked at the next call (or by an explicit check_error_flag())
            res = out.cpu().numpy()
        eng.check_error_flag()
        return res

    def _pnp_tail(self, r, K, E1):
        """Host tail of branch C for one chunk of environments -> [n,8,3] float64 boxes on the device."""
        box = pnp_box_tail(r["nocs1"].cpu().numpy(), r["pts2d1"].cpu().numpy(), r["scale"].cpu().numpy(), r["valid"].cpu().numpy(),
                           K.cpu().numpy().reshape(-1, 3, 3), E1.cpu().numpy().reshape(-1, 4, 4))
        return torch.from_numpy(box).to(self.device)

    def estimate_nocs_single_view(self, camera_intrinsic_batch, rgb_batch, mask_batch, choose=None, env_offset=0, sample_seed=None):
        """BASELINE configs[0..1]: one view per environment -> (nocs [N,1024,3] float32, choose [N,1024] int32, valid [N] bool)
        as numpy arrays.  This is the per-view part of the reference forward (preprocessing, PSPNet, ``instance_color`` +
        ``nocs_head``, network_v5.py:432-444); a full pose needs two views (interface_v5.py:256-257).  ``env_offset`` /
        ``sample_seed`` as in :meth:`estimate`: a multi-device estimator runs one contiguous block per replica with the global
        env index as the sampler key, so the result equals the one-device result bit for bit."""
        if self._replicas is not None:
            return self._single_view_multi(camera_intrinsic_batch, rgb_batch, mask_batch, choose, env_offset, sample_seed)
        self._ensure_capacity(len(camera_intrinsic_batch))
        eng = self.estimator
        K_b, rgb_b, m_b = (self._as_tensor(a) for a in (camera_intrinsic_batch, rgb_batch, mask_batch))
        N = K_b.shape[0]
        nocs = torch.empty((N, eng.P, 3), dtype=torch.float32, device=self.device)
        chs = torch.empty((N, eng.P), dtype=torch.int32, device=self.device)
        val = torch.empty((N,), dtype=torch.uint8, device=self.device)
        self._calls += 1
        seed = (self._seed + 7919 * self._calls) if sample_seed is None else int(sample_seed)
        with torch.cuda.device(self.device):
            for lo, hi in chunk_bounds(N, eng.E):
                m = m_b[lo:hi]
                if m.dtype not in self._MASK_OK:
                    m = m != 0
                if m.dtype == torch.bool:
                    m = m.view(torch.uint8)
                c = None if choose is None else self._as_tensor(choose[lo:hi]).to(torch.int32).to(self.device)
                n_, c_, v_ = eng.single_view_nocs(self._upload("rgb1", 0, rgb_b[lo:hi], self._rgb_dtype(rgb_b)),
                                                  self._upload("m1", 0, m), self._upload("K", 0, K_b[lo:hi], torch.float64), hi - lo,
                                                  seed=seed, choose=c, env0=int(env_offset) + lo)
                nocs[lo:hi].copy_(n_); chs[lo:hi].copy_(c_); val[lo:hi].copy_(v_)
                torch.cuda.current_stream(self.device).synchronize()       # the pinned staging slot is reused by the next chunk
            out = (nocs.cpu().numpy(), chs.cpu().numpy(), val.cpu().numpy().astype(bool))
        eng.check_error_flag()
        return out

    def _estimate_multi(self, batches, choose, return_tensor, ransac_idx, env_offset, sample_seed):
        """Contiguous blocks of environments, one per replica / device, run concurrently; the [n,8,3] results come back to the
        first device (peer copies) or the host.  Same sampler seed and global env indices on every replica: the result equals
        the one-GPU result of the same call bit for bit."""
        from .dist import shard_range
        N = len(batches[0])
        world = len(self._replicas)
        self._calls += 1
        seed = (self._seed + 7919 * self._calls) if sample_seed is None else int(sample_seed)

        def run(r):
            lo, hi, _ = shard_range(N, r, world)
            if hi <= lo:
                return None
            sl = lambda a: None if a is None else a[lo:hi]
            ch = None if choose is None else (choose[0][lo:hi], choose[1][lo:hi])
            return self._replicas[r].estimate(*[a[lo:hi] for a in batches], choose=ch, return_tensor=True, ransac_idx=sl(ransac_idx),
                                              env_offset=int(env_offset) + lo, sample_seed=seed)
        parts = [p for p in self._on_replicas(run) if p is not None]
        if return_tensor:
            if not parts:
                return torch.empty((0, 8, 3), dtype=torch.float64, device=self.device)
            return torch.cat([p.to(self.device) for p in parts])
        res = np.concatenate([p.cpu().numpy() for p in parts]) if parts else np.zeros((0, 8, 3))
        self.check_error_flag()
        return res

    def _single_view_multi(self, K_b, rgb_b, m_b, choose, env_offset, sample_seed):
        """:meth:`estimate_nocs_single_view` over the replicas: the blocks of :meth:`_estimate_multi`, gathered in env order."""
        from .dist import shard_range
        N = len(K_b)
        world = len(self._replicas)
        self._calls += 1
        seed = (self._seed + 7919 * self._calls) if sample_seed is None else int(sample_seed)

        def run(r):
            lo, hi, _ = shard_range(N, r, world)
            if hi <= lo:
                return None
            return self._replicas[r].estimate_nocs_single_view(K_b[lo:hi], rgb_b[lo:hi], m_b[lo:hi],
                                                               choose=None if choose is None else choose[lo:hi],
                                                               env_offset=int(env_offset) + lo, sample_seed=seed)
        parts = [p for p in self._on_replicas(run) if p is not None]
        if not parts:
            rep = self._replicas[0].estimator
            return np.zeros((0, rep.P, 3), np.float32), np.zeros((0, rep.P), np.int32), np.zeros((0,), bool)
        return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))

    def check_error_flag(self):
        """Synchronise and raise if the pipeline watchdog or the fp16 range guard fired (the tensor-returning paths defer it)."""
        for rep in (self._replicas or [self]):
            rep.estimator.check_error_flag()

    def estimate_tensor(self, *args, **kw):
        """Same as :meth:`estimate` but returns the [N,8,3] float64 CUDA tensor without the device->host copy."""
        return self.estimate(*args, return_tensor=True, **kw)

    def predict(self, camera_intrinsic, rgb1, view1_mask, view1_extrinsic, rgb2, view2_mask, view2_extrinsic):
        """Single environment (interface_v5.py:229-374) -> [8,3]."""
        f = lambda a: (a if isinstance(a, torch.Tensor) else np.asarray(a))[None]
        return self.estimate(f(camera_intrinsic), f(rgb1), f(view1_mask), f(view1_extrinsic),
                             f(rgb2), f(view2_mask), f(view2_extrinsic))[0]


class AdaPoseEstimator_baseline(AdaPoseEstimator_v5):
    """``name: adapose_baseline`` (train.py:242-244 -> interface_baseline.py:37-56): the same interface, preprocessing and pose
    fit around StereoPoseNet_with_depth_baseline (network_baseline.py:523-669), whose stereo term is 4 blocks of cross-view
    attention over the sampled point features (fusion.py:53-82) followed by a per-point depth MLP instead of the plane-sweep
    cost volume and its 3-D U-Net."""
    ARCH = "baseline"
