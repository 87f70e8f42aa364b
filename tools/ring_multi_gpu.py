"""BASELINE config 5 as a user of the reference runs it: ONE process, one estimator over every GPU (``devices``), a 5-slot
view ring over all environments and the 60-96-96-32-12 ELU actor -- the RL controller step ``add_view -> get_estimation ->
act_inference`` (rl_pose.py:118-223, module.py:89-91).

    python tools/ring_multi_gpu.py OUT_DIR [--envs 4096] [--devices all] [--share 512] [--steps 5] [--unique 64]

Runs, each after filling the ring with 5 views:
  * ``multi_host`` / ``multi_device``: ``--envs`` environments over ``--devices`` (skipped when fewer than two GPUs are
    visible).  Host frames are what the vec env hands over, float32 numpy (uint8 when the host cannot hold float32 frames;
    the JSON says which); device-resident frames live on the first GPU and reach the others by peer copies.
  * ``one_host`` / ``one_device``: the per-GPU share (``--share`` envs) on ``devices=[0]``, the yardstick of the scaling.
Reports ms per phase and per step (host clock, every device synchronised at the end of each phase), estimates/s
(num_envs per step), peak device memory per GPU, the scaling multi / (world x one-GPU share) and the GPUs' name and power
limit read with nvidia-smi in the same run.  Writes OUT_DIR/ring_multi_gpu.json.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rgbmanip_b200 import synth, weights  # noqa: E402

CFG = {"name": "adapose_v5", "task_name": "one_drawer_cabinet", "load": False, "img_size": 224, "use_depth": True,
       "n_pts": 1024, "direct_regression": True, "real_world": False}
ACTOR_DIMS = [60, 96, 96, 32, 12]       # cfg/controller/rl.yaml pi_hid_sizes, 12 actions; 60 = 5 slots x 12


def gpu_info():
    q = "index,name,power.limit,power.max_limit,clocks.max.sm,memory.total"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    return [dict(zip(q.split(","), [x.strip() for x in line.split(",")])) for line in out.stdout.strip().splitlines()]


def actor_state_dict():
    g = torch.Generator().manual_seed(0)
    sd = {}
    for i, (a, b) in enumerate(zip(ACTOR_DIMS[:-1], ACTOR_DIMS[1:])):
        sd[f"actor.{2 * i}.weight"] = torch.randn((b, a), generator=g) / a ** 0.5
        sd[f"actor.{2 * i}.bias"] = torch.zeros(b)
    return sd


def host_frames(n, unique, rgb_dtype):
    """Two camera steps of n environments (tiled from `unique` distinct scenes), as numpy the vec env hands over."""
    b = synth.make_batch(n, seed=0, special=True, n_unique=unique)
    views = []
    for rgb, m, E in ((b.rgb1, b.mask1, b.E1), (b.rgb2, b.mask2, b.E2)):
        if rgb_dtype == np.uint8:
            rgb = (np.clip(rgb, 0, 1) * 255).round().astype(np.uint8)
        views.append({"camera0": {"Color": rgb, "Mask": m.astype(np.uint8), "Intrinsic": b.K, "Extrinsic": E}})
    return views


def to_device(views, dev):
    return [{"camera0": {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in c["camera0"].items()}} for c in views]


def run(devices, n, views, steps):
    from rgbmanip_b200.actor import DeviceActor
    from rgbmanip_b200.estimator import AdaPoseEstimator_v5
    from rgbmanip_b200.view_ring import ViewRing
    devs = [torch.device(f"cuda:{d}") for d in devices]
    for d in devs:
        torch.empty(1, device=d)                  # the allocator of a device keeps statistics once it is in use
        torch.cuda.reset_peak_memory_stats(d)
    est = AdaPoseEstimator_v5(None, dict(CFG), None, state_dict=weights.init_state_dict(0), devices=list(devices))
    ring = ViewRing(est, n, 5)
    actor = DeviceActor(actor_state_dict(), ring, activation="elu")
    pose = np.zeros((n, 7))
    sync = lambda: [torch.cuda.synchronize(d) for d in devs]
    phases = {"add_view": [], "get_estimation": [], "act_inference": [], "step": []}

    def step(t, record):
        t0 = time.perf_counter()
        ring.add_view(views[t % 2], pose)          # ends with the error-flag check of every replica (synchronises)
        ring.accumulate_steps = min(ring.accumulate_steps + 1, ring.max_steps)
        sync()
        t1 = time.perf_counter()
        boxes = ring.get_estimation()              # numpy [n,8,3], as the controller receives it
        t2 = time.perf_counter()
        act, obs = actor.act_inference()
        sync()
        t3 = time.perf_counter()
        if record:
            for k, v in (("add_view", t1 - t0), ("get_estimation", t2 - t1), ("act_inference", t3 - t2), ("step", t3 - t0)):
                phases[k].append(v * 1e3)
        return boxes, act

    for t in range(5 + 1):                         # fill the 5 slots, then one warm step of the steady state
        step(t, False)
    for t in range(steps):
        boxes, act = step(6 + t, True)
    ms = {k: float(np.median(v)) for k, v in phases.items()}
    res = {"devices": [str(d) for d in devs], "num_envs": n, "steps": steps, "ms_median": ms,
           "ms_all": {k: [round(x, 3) for x in v] for k, v in phases.items()},
           "estimates_per_s": n / (ms["step"] / 1e3),
           "peak_mem_gb": [torch.cuda.max_memory_allocated(d) / 1e9 for d in devs],
           "sentinel_boxes": int((boxes[:, 0, 0] >= 9.5).sum()), "actions_finite": bool(torch.isfinite(act).all())}
    del actor, ring, est
    gc.collect()                                   # the replicas' engines sit in reference cycles: free them before the next run
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("out_dir")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--devices", default="all", help="'all' or a comma-separated list of GPU indices")
    ap.add_argument("--share", type=int, default=512, help="environments of the one-GPU run (default: 4096 / 8)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--unique", type=int, default=64, help="distinct scenes tiled over the environments")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ring_multi_gpu.py measures on CUDA devices; none is visible")
    devices = list(range(torch.cuda.device_count())) if args.devices == "all" else [int(d) for d in args.devices.split(",")]
    os.makedirs(args.out_dir, exist_ok=True)
    out = {"gpus": gpu_info(), "torch": torch.__version__, "args": {k: v for k, v in vars(args).items() if k != "out_dir"}}
    # host frames: 2 steps x envs x 480 x 640 x 3 float32 (30 GB at 4096 envs) plus the masks; uint8 if the host has no room
    need = 2 * args.envs * 480 * 640 * (3 * 4 + 1)
    avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    rgb_dtype = np.float32 if need < 0.6 * avail else np.uint8
    out["host_frames"] = {"rgb_dtype": np.dtype(rgb_dtype).name, "host_available_bytes": avail,
                          "bytes": 2 * args.envs * 480 * 640 * (3 * np.dtype(rgb_dtype).itemsize + 1)}
    if len(devices) >= 2:
        views = host_frames(args.envs, args.unique, rgb_dtype)
        out["multi_host"] = run(devices, args.envs, views, args.steps)
        views = to_device(views, f"cuda:{devices[0]}")
        out["multi_device"] = run(devices, args.envs, views, args.steps)
        del views
    else:
        out["multi_host"] = out["multi_device"] = None
        out["multi_skipped"] = f"{len(devices)} GPU visible: the multi-device runs need two or more"
    views = host_frames(args.share, args.unique, rgb_dtype)
    out["one_host"] = run(devices[:1], args.share, views, args.steps)
    out["one_device"] = run(devices[:1], args.share, to_device(views, f"cuda:{devices[0]}"), args.steps)
    if out["multi_host"] is not None:
        w = len(devices)
        out["scaling"] = {k: out[f"multi_{k}"]["estimates_per_s"] / (w * out[f"one_{k}"]["estimates_per_s"]) for k in ("host", "device")}
    path = os.path.join(args.out_dir, "ring_multi_gpu.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    summary = {k: (v["ms_median"], round(v["estimates_per_s"])) for k, v in out.items() if isinstance(v, dict) and "ms_median" in v}
    print(json.dumps({"gpus": [(g["name"], g["power.limit"]) for g in out["gpus"]], "runs": summary, "scaling": out.get("scaling")}))
    print("wrote", path)


if __name__ == "__main__":
    main()
