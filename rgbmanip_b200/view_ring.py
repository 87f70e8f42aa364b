"""Device-resident view ring + per-view feature cache (SURVEY.md 8(f)-1).

Replaces the host queues of the reference's RL controller, ``models/controller/rl_pose.py``:
``reset_queue`` (:85-97), ``add_view`` (:118-150) and ``get_estimation`` (:189-223).  The reference keeps every frame of
every environment as float64 on the host (``[max_steps, N, 480, 640, 3]``: 151 GB at 4096 envs), re-walks the ring in
Python on every step and pushes BOTH views of every environment through the estimator again.  Here

* ``add_view`` uploads only the new frame, runs preprocessing + the backbone ONCE for it and keeps what the stereo head
  needs per (ring slot, env) on the device: the 32 x 224 x 224 feature map (fp32 + the fp16 twin the volume builder
  gathers), K', the 1024 sampled pixels, validity, extrinsic.  The mask box of :130-150 comes out of the preprocess
  kernel's bounding-box pass (including the quirk at :132: once ANY environment sees the object, every environment's
  slot counts as available);
* ``get_estimation`` pairs the views with the reference's rule (the k-th available view of an env goes to batch slot
  k % 2, so slot 0 = last even-indexed, slot 1 = last odd-indexed available view), gathers the two cached feature maps
  of every environment and runs only volume -> U-Net -> decode -> fit.  One backbone pass per controller step instead of
  two (81.8 vs 138.9 GFLOP per estimate).

Differences from the reference, by construction: the random 1024-pixel subset of a view is drawn once, when the view
is added (the reference redraws it at every estimate; same distribution), and frames themselves are not retained.

Over a multi-device estimator (``devices``: a list or ``"all"``) ``ViewRing`` is a :class:`ShardedViewRing`: every replica
keeps the ring of its contiguous block of environments on its own device, the shards run on the estimator's per-device host
threads, and the random draws are keyed as a one-device ring keys them (:func:`ring_pieces`), so the queues and boxes do
not depend on the device count.
"""
from __future__ import annotations

import numpy as np
import torch

MUG_CORNER_ORDER = [0, 2, 4, 6, 1, 3, 5, 7]      # rl_pose.py:220-221


def ring_pieces(key, lo, hi, cap):
    """Launch schedule of the environments [lo, hi) (global indices) of a ring whose random draws are keyed by chunks of
    ``key`` environments -- chunk c is [c key, (c + 1) key), the launches of a one-device ring of that capacity -- on a device
    that runs at most ``cap`` environments per launch.  -> [(p_lo, p_hi, key_lo)]: the range is cut at every key-chunk
    boundary and then at ``cap``; key_lo is the start of the key chunk the piece lies in.  A piece's draws are keyed by
    key_lo (the seed) and p_lo - key_lo (the position of its first environment inside the key chunk)."""
    out, a = [], int(lo)
    while a < hi:
        k0 = a // key * key
        b = min(int(hi), k0 + key, a + cap)
        out.append((a, b, k0))
        a = b
    return out


class ViewRing:
    def __new__(cls, estimator, *args, **kw):
        if cls is ViewRing and getattr(estimator, "_replicas", None) is not None:
            cls = ShardedViewRing
        return super().__new__(cls)

    def __init__(self, estimator, num_envs: int, max_steps: int, height: int = 480, width: int = 640, env0: int = 0,
                 key_envs: int | None = None):
        """``env0`` / ``key_envs`` describe a shard of a :class:`ShardedViewRing`: the global index of its first environment and
        the chunk size its random draws are keyed by.  Default: the whole batch, keyed by this estimator's own chunks."""
        self.estimator = estimator
        if hasattr(estimator, "_ensure_capacity"):
            estimator._ensure_capacity(num_envs)         # an auto-sized estimator grows its chunk capacity to the ring's batch
            if key_envs is not None and not estimator.estimator.regress_pose:
                estimator._ensure_capacity(key_envs)     # a whole key chunk per launch: see _boxes
        eng = estimator.estimator
        if getattr(eng, "branch_c", False) or getattr(eng, "arch", "v5") != "v5":
            raise NotImplementedError("the view ring drives the cost-volume head with the direct-regression fit (every shipped config) "
                                      "or the RANSAC + Umeyama fit (direct_regression=False, use_depth=True)")
        self.num_envs, self.max_steps, self.h, self.w = int(num_envs), int(max_steps), int(height), int(width)
        self.env0, self._key = int(env0), key_envs
        self.device = eng.device
        T, N, S, P = self.max_steps, self.num_envs, eng.S, eng.P
        dev = self.device
        self.feat = torch.zeros((T, N, S, S, 32), dtype=torch.float32, device=dev)
        self.feat16 = torch.zeros((T, N, S, S, 32), dtype=torch.float16, device=dev) if eng.feat16 is not None else None
        self.Kp = torch.zeros((T, N, 9), dtype=torch.float64, device=dev)
        self.choose = torch.zeros((T, N, P), dtype=torch.int32, device=dev)
        self.valid = torch.zeros((T, N), dtype=torch.uint8, device=dev)
        self.extrinsic = torch.zeros((T, N, 16), dtype=torch.float64, device=dev)
        self.intrinsic = torch.zeros((T, N, 9), dtype=torch.float64, device=dev)
        self.pose = torch.zeros((T, N, 7), dtype=torch.float64, device=dev)
        self.bbox = torch.zeros((T, N, 4), dtype=torch.float64, device=dev)
        self.avail = torch.zeros((T, N), dtype=torch.float64, device=dev)
        self.avail_num = torch.zeros((N,), dtype=torch.int32, device=dev)
        self._hw = torch.tensor([self.h, self.w, self.h, self.w], dtype=torch.float64, device=dev)
        self.accumulate_steps = 0          # advanced by the caller after add_view, as in the reference (rl_pose.py:116)
        self._adds = 0

    @property
    def eng(self):
        return self.estimator.estimator          # looked up per call: an auto-sized estimator may rebuild its engine

    # ---- queue state in the reference's host format (small arrays: observations / rewards read them) ----
    @property
    def available(self):
        return self.avail.cpu().numpy()

    @property
    def available_num(self):
        return self.avail_num.cpu().numpy()

    @property
    def bbox_queue(self):
        return self.bbox.cpu().numpy()

    @property
    def pose_queue(self):
        return self.pose.cpu().numpy()

    def reset_queue(self):
        """rl_pose.py:85-97."""
        for t in (self.feat, self.feat16, self.Kp, self.choose, self.valid, self.extrinsic, self.intrinsic, self.pose, self.bbox,
                  self.avail, self.avail_num):
            if t is not None:
                t.zero_()
        self.accumulate_steps = 0

    def _dev(self, a, dtype=None):
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        return t.to(self.device, non_blocking=True).contiguous()

    def add_view(self, image, cam_pose):
        """rl_pose.py:118-150: ``image`` is the env's camera dict (``image["camera0"]["Color" | "Mask" | "Intrinsic" |
        "Extrinsic"]``, one entry per environment), ``cam_pose`` [N,7]."""
        self._mark_available(self._add_frames(image, cam_pose))
        self._check_error_flag()

    def _add_frames(self, image, cam_pose):
        """Everything of add_view but the availability: frames -> preprocess + backbone -> this ring's slot of the feature
        cache and queues.  The arguments hold every environment (global indices); this ring takes [env0, env0 + num_envs).
        -> device bool: does any of those environments see the object?"""
        cam = image["camera0"]
        color, mask, K, E = cam["Color"], cam["Mask"], cam["Intrinsic"], cam["Extrinsic"]
        eng, N, slot = self.eng, self.num_envs, self.accumulate_steps % self.max_steps
        g0, g1 = self.env0, self.env0 + N
        self._adds += 1
        key = eng.F if self._key is None else 2 * self._key       # a one-device ring preprocesses 2 x max_envs frames per launch
        with torch.cuda.device(self.device):
            any_pixel = torch.zeros((), dtype=torch.bool, device=self.device)
            for lo, hi, key_lo in ring_pieces(key, g0, g1, eng.F):   # the frame buffers hold 2 x max_envs frames: full-size backbone launches
                n = hi - lo
                l, h = lo - g0, hi - g0
                c = color[lo:hi]
                c = c if isinstance(c, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(c))
                # same staging policy as estimate(): float64 host frames are demoted to float32, uint8 means value / 255
                rgb_d = self._dev(c, self.estimator._rgb_dtype(c))
                mask_d = self._dev(mask[lo:hi])
                if mask_d.dtype not in (torch.uint8, torch.bool, torch.float32, torch.float64):
                    mask_d = (mask_d != 0).to(torch.uint8)       # segmentation ids: a cast could wrap 256 to 0
                K_d = self._dev(K[lo:hi], torch.float64)
                eng.preprocess(0, rgb_d, mask_d, K_d, n, seed=(self.estimator._seed + 104729 * self._adds + key_lo), frame_id0=lo - key_lo)
                eng.run_backbone(n)                       # ONE view: frames [0, n)
                self.feat[slot, l:h].copy_(eng.feat[:n])
                if self.feat16 is not None:
                    self.feat16[slot, l:h].copy_(eng.feat16[:n])
                self.Kp[slot, l:h].copy_(eng.Kp[:n])
                self.choose[slot, l:h].copy_(eng.choose[:n])
                self.valid[slot, l:h].copy_(eng.valid[:n])
                bb = eng.bbox_ws[:n].to(torch.float64)    # {ymin, xmin, ymax, xmax}; ymax < 0 <=> empty mask
                empty = bb[:, 2] < 0
                any_pixel = any_pixel | (~empty).any()
                box = torch.div(bb, self._hw)             # tensor divisor: a true IEEE division, as numpy's (scalar division multiplies by 1/x)
                box[empty] = torch.tensor([2.0, 2.0, 0.0, 0.0], dtype=torch.float64, device=self.device)   # (2H/H, 2W/W, 0, 0): :141-144
                self.bbox[slot, l:h].copy_(box)
            self.extrinsic[slot].copy_(self._dev(E[g0:g1], torch.float64).reshape(N, 16))
            self.intrinsic[slot].copy_(self._dev(K[g0:g1], torch.float64).reshape(N, 9))
            self.pose[slot].copy_(self._dev(cam_pose[g0:g1], torch.float64).reshape(N, 7))
        return any_pixel

    def _mark_available(self, any_pixel):
        """:132 tests the pixel count over ALL environments: one visible object marks every environment's slot available.
        ``any_pixel``: a device bool, or a host bool combined over the shards of a sharded ring."""
        slot = self.accumulate_steps % self.max_steps
        with torch.cuda.device(self.device):
            flag = torch.as_tensor(any_pixel, device=self.device)
            self.avail[slot] = flag.to(torch.float64)
            self.avail_num += flag.to(torch.int32)

    def _check_error_flag(self):
        self.eng.check_error_flag()

    def pair_slots(self):
        """[2, N] ring indices feeding estimate()'s view 1 / view 2 (-1: that batch slot stays empty); rl_pose.py:199-208."""
        av = self.avail > 0
        k = torch.cumsum(av.to(torch.int64), 0) - 1
        ring = torch.arange(self.max_steps, device=self.device)[:, None]
        out = []
        for par in (0, 1):
            m = av & ((k % 2) == par)
            out.append(torch.where(m, ring, torch.full_like(ring, -1)).max(0).values)
        return torch.stack(out)

    def get_estimation(self, return_tensor: bool = False, ransac_idx=None):
        """rl_pose.py:189-223 -> [N,8,3] float64 world-frame boxes (sentinel where an env has no valid view pair).
        ``ransac_idx`` ([N,128,5] int32, optional) replays given RANSAC draws of the Umeyama fit (direct_regression=False);
        by default they come from the device hash, as in ``estimate()``."""
        with torch.cuda.device(self.device):
            out = self._boxes(ransac_idx)
            if self.estimator.cfg.get("task_name") == "mugs":
                out = out[:, MUG_CORNER_ORDER]
            if return_tensor:
                return out
            res = out.cpu().numpy()
        self._check_error_flag()
        return res

    def _boxes(self, ransac_idx=None):
        """The [num_envs,8,3] boxes of this ring's environments on its device, corners in the estimator's order.
        ``ransac_idx`` holds every environment (global indices), as the arguments of add_view do."""
        eng, N, g0 = self.eng, self.num_envs, self.env0
        E = eng.E
        key = E if self._key is None else self._key
        # the Umeyama fit's device RANSAC draws are keyed by the seed and an env's position in the launch: a piece that starts
        # inside its key chunk is launched behind lo - key_lo placeholder environments (no valid view), so that every
        # environment keeps the position it has in the one-device launch
        pad_to_key = not eng.regress_pose and ransac_idx is None
        out = torch.empty((N, 8, 3), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            sl = self.pair_slots()
            for lo, hi, key_lo in ring_pieces(key, g0, g0 + N, E):
                pad = lo - key_lo if pad_to_key else 0
                n = hi - lo + pad
                assert n <= E, (n, E)
                g = torch.arange(lo - pad, hi, device=self.device)
                real = g >= lo
                idx = g.clamp(min=lo) - g0
                ext = []
                for v in (0, 1):
                    s = sl[v, idx]
                    have = (s >= 0) & real
                    sc = s.clamp(min=0)
                    o = v * E
                    eng.feat[o:o + n].copy_(self.feat[sc, idx])
                    if self.feat16 is not None:
                        eng.feat16[o:o + n].copy_(self.feat16[sc, idx])
                    eng.Kp[o:o + n].copy_(self.Kp[sc, idx])
                    eng.choose[o:o + n].copy_(self.choose[sc, idx])
                    eng.valid[o:o + n].copy_(self.valid[sc, idx] * have.to(torch.uint8))
                    ext.append(self.extrinsic[sc, idx].contiguous())
                ridx = None
                if ransac_idx is not None and not eng.regress_pose:
                    ridx = torch.as_tensor(np.ascontiguousarray(ransac_idx[lo:hi])).to(torch.int32).to(self.device)
                eng.stereo(n, ext[0], ext[1], ransac_idx=ridx, seed=7919 * self._adds + key_lo)
                out[lo - g0:hi - g0].copy_(eng.bbox[pad:n])
        return out


class ShardedViewRing(ViewRing):
    """:class:`ViewRing` over a multi-device estimator (what ``ViewRing(estimator, ...)`` builds for one).  Replica r keeps a
    ring of the contiguous block ``dist.shard_range(num_envs, r, world)`` -- the block ``estimate()`` gives it -- on its own
    device; the shards run concurrently on the estimator's per-device host threads.  Both kinds of random draws (pixel
    subsets, device RANSAC samples) are keyed by the chunks of a one-device estimator of the same configuration, so every
    queue, pixel subset and box equals the one-device ring's.  The queue properties are gathered in env order; tensors come
    back on the first device."""

    def __init__(self, estimator, num_envs: int, max_steps: int, height: int = 480, width: int = 640):
        from .dist import shard_range
        self.estimator = estimator
        self.num_envs, self.max_steps, self.h, self.w = int(num_envs), int(max_steps), int(height), int(width)
        self.device = estimator.device
        self.accumulate_steps = 0
        world = len(estimator._replicas)
        key = estimator.one_device_chunk(self.num_envs)
        blocks = {r: shard_range(self.num_envs, r, world)[:2] for r in range(world)}
        self._ranks = [r for r, (lo, hi) in blocks.items() if hi > lo]        # fewer environments than devices: empty blocks idle
        self.shards = estimator._on_replicas(
            lambda r: ViewRing(estimator._replicas[r], blocks[r][1] - blocks[r][0], max_steps, height, width, env0=blocks[r][0],
                               key_envs=key), self._ranks)
        self._shard = dict(zip(self._ranks, self.shards))

    def _gather(self, name, dim=1):
        """A per-shard queue tensor, concatenated in env order on the first device."""
        return torch.cat([getattr(s, name).to(self.device) for s in self.shards], dim)

    @property
    def available(self):
        return np.concatenate([s.available for s in self.shards], 1)

    @property
    def available_num(self):
        return np.concatenate([s.available_num for s in self.shards], 0)

    @property
    def bbox_queue(self):
        return np.concatenate([s.bbox_queue for s in self.shards], 1)

    @property
    def pose_queue(self):
        return np.concatenate([s.pose_queue for s in self.shards], 1)

    @property
    def choose(self):
        """[T,N,P] int32 pixel subsets of the cached views."""
        return self._gather("choose")

    @property
    def extrinsic(self):
        """[T,N,16] float64 extrinsics of the cached views."""
        return self._gather("extrinsic")

    def reset_queue(self):
        for s in self.shards:
            s.reset_queue()
        self.accumulate_steps = 0

    def add_view(self, image, cam_pose):
        for s in self.shards:
            s.accumulate_steps = self.accumulate_steps
        # the :132 quirk couples the environments: the visibility flags of all shards (one per device, read back) are OR-ed
        # before any shard marks its slot available
        seen = self.estimator._on_replicas(lambda r: bool(self._shard[r]._add_frames(image, cam_pose)), self._ranks)
        any_pixel = any(seen)
        for s in self.shards:
            s._mark_available(any_pixel)
        self._check_error_flag()

    def pair_slots(self):
        return torch.cat([s.pair_slots().to(self.device) for s in self.shards], 1)

    def _boxes(self, ransac_idx=None):
        parts = self.estimator._on_replicas(lambda r: self._shard[r]._boxes(ransac_idx), self._ranks)
        return torch.cat([p.to(self.device) for p in parts])

    def _check_error_flag(self):
        self.estimator.check_error_flag()


def attach(control_interface, estimator=None):
    """Swap the queue methods of a live ``ControlInterface`` (rl_pose.py:14) for a device ring; observations keep reading
    ``pose_queue`` / ``bbox_queue`` / ``available`` as numpy arrays."""
    ci = control_interface
    ring = ViewRing(estimator or ci.estimator, ci.num_envs, ci.max_steps)

    def sync():
        ci.pose_queue, ci.bbox_queue = ring.pose_queue, ring.bbox_queue
        ci.available, ci.available_num = ring.available, ring.available_num

    def reset_queue():
        ring.reset_queue()
        ci.accumulate_steps = 0
        ci.pred_bbox = np.zeros((ci.max_steps, ci.num_envs, 8, 3))
        ci.gt_bbox = np.zeros((ci.max_steps, ci.num_envs, 8, 3))
        sync()

    def add_view(image, cam_pose):
        ring.accumulate_steps = ci.accumulate_steps
        ring.add_view(image, cam_pose)
        sync()

    ci.reset_queue, ci.add_view, ci.get_estimation = reset_queue, add_view, ring.get_estimation
    ci.view_ring = ring
    reset_queue()
    return ring
