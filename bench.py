"""Headline benchmark: pose estimates / second at num_envs=1024 (BASELINE.json), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--num-envs 1024] [--precision fp16f8|fp16x2|bf16x3|bf16]
                    [--dump-outputs DIR]

A step = one pass of the hot path (preprocess -> backbone x2 views -> plane-sweep volume -> 3-D U-Net -> decode ->
fit) over ALL num_envs environments of synthetic input.  With N > 1 (torchrun) the environments are sharded
contiguously over the ranks (no data-path collective) and the per-env poses are all-gathered over NCCL; the total
stays num_envs, i.e. strong scaling, as the metric is defined at num_envs=1024.

`value`  : device-resident inputs, CUDA-event timing of exactly K steps, max over ranks.
`e2e`    : the same metric through AdaPoseEstimator_v5.estimate() with pinned HOST float32 inputs, host->device copies and
           the device->host read of the boxes inside the timed region.  `e2e_variants` repeats it with what the RL caller
           really passes (pageable float64 numpy, rl_pose.py:194-218) and with uint8 frames.
`parity_in_bench` : before anything is timed, the 8 golden environments of tests/golden/e2e.npz (boxes produced by the
           reference itself) run through THIS estimator object -- bench chunk size, CUDA-graph replay -- and must agree to
           0.5 px / 0.5 deg / 1 mm.  `shard_identity`: after the timed region the sharded result (all ranks, all-gathered) is
           compared with a one-rank run of the same environments on rank 0.
`configs`: the other BASELINE.json configurations (single-view NOCS at N=64, the 4-view mug ring at N=256, the
           observation + actor step of the N=4096 / 8-GPU configuration as this rank's share) -- reported beside the headline.
`--impl reference`: the reference's own CPU implementation (oracle/_ref: a run-time copy of the unmodified reference staged
           by __graft_entry__.build(); the oracle port if that copy is absent) timed on the host cores on a bounded sample.
`--dump-outputs DIR`: after the timed steps, the boxes of the last timed step (what estimate() hands its caller, all num_envs
           environments) go to DIR/boxes.npy as float64.  Inputs, weights and the per-call sampler seeds depend only on the
           arguments, so two builds run with the same arguments can be compared box for box.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from rgbmanip_b200 import synth, weights  # noqa: E402

GF_BACKBONE_PER_FRAME = 57.0177e9       # SURVEY.md A.3 (2 * MACs of every conv of the PSPNet backbone)
GF_BACKBONE_TC_PER_FRAME = 57.0177e9 - 0.0128e9 - 0.0066e9     # minus the pyramid 1x1 convs (CUDA cores); everything else is tcgen05
# executed on the tensor cores: up_1 / up_2 run as low-resolution per-tap GEMMs (engine._build_backbone), a quarter of their 3x3 FLOPs
GF_BACKBONE_EXECUTED_PER_FRAME = GF_BACKBONE_TC_PER_FRAME - 0.75 * (14.7968e9 + 3.6992e9)
GF_COSTREG_PER_VIEW = 24.4506e9
# HBM-bound stages, algorithmic bytes per environment (DESIGN.md section 5 derives them):
#   volume + 3-D U-Net, materialised-volume variant (SURVEY 8(d)): 302.7 MB per reference view
#   decode gather: 3 x 3 x 26 voxels x 16 B of the last U-Net tensor per sampled pixel (the `prob` conv is evaluated only
#   there) + 24 depths x 4 bilinear corners x 128 B of fp32 source features + 128 B reference features + outputs
BYTES_VOLUME_COSTREG_PER_ENV = 302.7e6
BYTES_DECODE_GATHER_PER_ENV = 1024 * (3 * 3 * 26 * 16 + 24 * 4 * 128 + 128 + 4 + 4 + 2 * 128 * 2)
# "profile constants": figures of an ncu capture of one chunk (not of this run); the launch list they come from is committed
NCU_PROFILE = {"fp16f8": {"dram_bytes_per_frame": 13312.8e6 / 148, "tensor_pipe_active": 0.660, "src": "profiles/r02d_chunk_launches.csv"},
               "fp16x2": {"dram_bytes_per_frame": 11141.8e6 / 148, "tensor_pipe_active": 0.720, "src": "profiles/r01_chunk_by_kernel.csv"},
               "bf16x3": {"dram_bytes_per_frame": 18958.8e6 / 128, "tensor_pipe_active": 0.712, "src": "profiles/r01_bf16x3_backbone_tc_summary.csv"}}
CFG = {"name": "adapose_v5", "task_name": "one_drawer_cabinet", "load": False, "img_size": 224, "use_depth": True,
       "n_pts": 1024, "direct_regression": True, "real_world": False}
DEFAULT_BBOX = np.asarray([[0, 0, 0], [0, 0, 1], [0, 1, 0], [0, 1, 1], [1, 0, 0], [1, 0, 1], [1, 1, 0], [1, 1, 1]], dtype=np.float64) + 10.0
TOL_PX, TOL_DEG, TOL_MM = 0.5, 0.5, 1.0
DUMP_MAX_BYTES = 64 << 20


def workload_name(n):
    return (f"adapose_v5 estimate(), num_envs={n}, 2 views/env, 480x640 fp32 RGB + u8 mask -> [N,8,3] world boxes "
            "(BASELINE configs[3]; all four adapose_* yamls share this architecture)")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def dump_output(out_dir, name, t):
    """Write one output as out_dir/<name>.npy.  Beyond DUMP_MAX_BYTES only a fixed, seeded sample of its rows (environments),
    in ascending order, is written, so that the file stays comparable between runs with the same arguments."""
    a = t.cpu().numpy()
    row = max(1, a[:1].nbytes)
    keep = (DUMP_MAX_BYTES - 4096) // row          # 4 KB for the .npy header
    if len(a) > keep:
        a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), a)


def dist_setup():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo")
    return rank, world, local


# ------------------------------------------------------------------------------------------------ box metrics (checker)
def _box_pose(box):
    c = box.mean(0)
    ax = np.stack([box[0] - box[2], box[0] - box[4], box[0] - box[1]], 1)      # corner order of utils.py:40-58
    return c, ax / np.maximum(np.linalg.norm(ax, axis=0, keepdims=True), 1e-12)


def box_errors(a, b, K, E1, min_z=0.5):
    """(keypoint reprojection error [px] of the 8 corners + centre in view 1 (points nearer than min_z to the camera plane are
    compared in mm only: f/z diverges there, see tests/test_gpu_e2e.py MIN_Z), rotation [deg], centre [mm], max corner [mm])."""
    ca, Ra = _box_pose(a)
    cb, Rb = _box_pose(b)

    def proj(pts):
        pc = (E1[:3, :3] @ pts.T).T + E1[:3, 3]
        return (K @ pc.T).T[:, :2] / pc[:, 2:3], pc[:, 2]
    pa, za = proj(np.vstack([a, ca[None]]))
    pb, zb = proj(np.vstack([b, cb[None]]))
    ok = (za > min_z) & (zb > min_z)
    px = float(np.abs(pa[ok] - pb[ok]).max()) if ok.any() else 0.0
    cosang = np.clip((np.trace(Ra.T @ Rb) - 1.0) / 2.0, -1.0, 1.0)
    box_errors.compared += int(ok.sum())
    box_errors.total += int(ok.size)
    return px, float(np.degrees(np.arccos(cosang))), float(np.linalg.norm(ca - cb) * 1e3), float(np.linalg.norm(a - b, axis=1).max() * 1e3)


box_errors.compared = box_errors.total = 0      # keypoints that entered the pixel metric / all keypoints seen (the rest: mm only)


def parity_check(est, copies):
    """The golden environments of tests/golden/e2e.npz through the bench-configured estimator (its chunk size, graph replay)."""
    gpath = os.path.join(ROOT, "tests", "golden", "e2e.npz")
    if not os.path.exists(gpath):
        return {"skipped": "tests/golden/e2e.npz not found"}
    g = np.load(gpath)
    base = synth.make_batch(8, seed=0)
    c1 = np.zeros((8, 1024), np.int32); c2 = np.zeros((8, 1024), np.int32)
    for e in range(8):
        if g["valid"][e]:
            c1[e], c2[e] = g[f"env{e}_choose1"], g[f"env{e}_choose2"]
    idx = np.arange(copies) % 8
    args = [torch.from_numpy(np.ascontiguousarray(a[idx])).to(est.device) for a in base.args()]
    args[2], args[5] = args[2].to(torch.uint8), args[5].to(torch.uint8)
    choose = (c1[idx], c2[idx])
    eng = est.estimator
    for _ in range(3):                   # eager, capture, replay
        boxes = est.estimate(*args, choose=choose)
    worst = np.zeros(4)
    sentinel_ok = True
    box_errors.compared = box_errors.total = 0
    for i, e in enumerate(idx):
        if not g["valid"][e]:
            sentinel_ok &= bool(np.array_equal(boxes[i], DEFAULT_BBOX))
            continue
        worst = np.maximum(worst, box_errors(boxes[i], g["boxes"][e], base.K[e], base.E1[e]))
    # the gate is north_star's three quantities (keypoints, rotation, translation = box centre); the worst corner distance is
    # reported beside them (it adds the size error of ~1 m random-init boxes)
    ok = bool(worst[0] < TOL_PX and worst[1] < TOL_DEG and worst[2] < TOL_MM and sentinel_ok)
    out = {"envs": int(copies), "fixture": "tests/golden/e2e.npz (boxes from the unmodified reference, 8 envs tiled)",
           "chunk_sizes": sorted({hi - lo for lo, hi in est._chunk_bounds(copies, False)}),
           "graph_replayed": bool(eng._graphs), "max_px": float(worst[0]), "max_deg": float(worst[1]), "max_centre_mm": float(worst[2]),
           "max_corner_mm": float(worst[3]), "sentinels_bit_exact": sentinel_ok,
           "keypoints_in_px_metric": box_errors.compared, "keypoints_total": box_errors.total,
           "tolerance": {"px": TOL_PX, "deg": TOL_DEG, "mm": TOL_MM}, "ok": ok}
    if not ok:
        raise SystemExit("parity_in_bench failed: " + json.dumps(out))
    return out


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_rate(n_envs, seed=0):
    """The reference's per-env loop on the host cores -> (estimates/s, threads, seconds, kind)."""
    torch.set_num_threads(os.cpu_count())
    batch = synth.make_batch(n_envs + 1, seed=seed, special=False)
    from oracle import ref_stage
    if ref_stage.root() is not None:
        est, _ = ref_stage.load(seed=0)
        with torch.no_grad():
            np.random.seed(0)
            est.estimate(*batch.slice(0, 1).args())          # warm-up env
            t0 = time.perf_counter()
            est.estimate(*batch.slice(1, n_envs + 1).args())
            dt = time.perf_counter() - t0
        return n_envs / dt, torch.get_num_threads(), dt, "reference"
    from oracle import adapose_oracle as O
    sd = weights.init_state_dict(0)
    np.random.seed(0)
    O.estimate(sd, CFG, *batch.slice(0, 1).args())
    t0 = time.perf_counter()
    O.estimate(sd, CFG, *batch.slice(1, n_envs + 1).args())
    dt = time.perf_counter() - t0
    return n_envs / dt, torch.get_num_threads(), dt, "port"


def cpu_single_view(n_frames=3):
    """BASELINE configs[0]: adapose_drawer forward, batch 1, ONE view, PyTorch on CPU: preprocessing + PSPNet + NOCS head of the
    reference (the full estimate needs two views: interface_v5.py:256-257) -> frames/s."""
    torch.set_num_threads(os.cpu_count())
    batch = synth.make_batch(n_frames + 1, seed=3, special=False)
    from oracle import ref_stage
    if ref_stage.root() is None:
        return None
    est, _ = ref_stage.load(seed=0)
    net = est.estimator.module

    def one(e):
        view, choose, _, _ = est.prepare_model_input(batch.rgb1[e], batch.mask1[e], batch.K[e], 224)
        with torch.no_grad():
            feat = net.img_extractor(view[None].float())
            emb = feat.view(1, feat.shape[1], -1)[:, :, torch.from_numpy(np.asarray(choose)).long()]
            return net.nocs_head(net.instance_color(emb))
    np.random.seed(0)
    one(0)
    t0 = time.perf_counter()
    for e in range(1, n_frames + 1):
        one(e)
    dt = time.perf_counter() - t0
    return {"value": n_frames / dt, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "reference",
            "what": "BASELINE configs[0]: batch 1, one 480x640 view -> crop, PSPNet, instance_color + nocs_head on the CPU", "frames": n_frames}


def cpu_legs_subprocess(n_envs):
    """The CPU legs run in a child process that cannot see the GPUs: the reference moves its tensors with .cuda() and wraps the
    net in nn.DataParallel, so with a visible device it would not be the CPU arm any more."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu-sample", "--cpu-sample", str(n_envs)],
                       env=env, capture_output=True, text=True, timeout=900)
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("CPU legs failed:\n" + r.stdout[-2000:] + r.stderr[-4000:])


def run_cpu_sample(args):
    rate, threads, dt, kind = cpu_reference_rate(args.cpu_sample)
    print(json.dumps({"rate": rate, "threads": threads, "dt": dt, "kind": kind, "single_view": cpu_single_view()}), flush=True)


def run_reference(args, rank, world):
    if rank != 0:
        return
    sample = 6
    vals = []
    kind = threads = None
    for i in range(args.warmup + args.steps):
        rate, threads, dt, kind = cpu_reference_rate(sample, seed=i)
        if i >= args.warmup:
            vals.append((rate, dt))
    rate = sample * len(vals) / sum(d for _, d in vals)
    note = ("the unmodified reference (oracle/_ref) on the CPU: per-env loop of AdaPoseEstimator_v5.estimate, eval mode"
            if kind == "reference" else "reference's per-env CPU loop (oracle port, torch CPU fp32 eval mode)")
    line = {"metric": "pose estimates/sec at num_envs=1024", "value": rate, "unit": "estimates/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(d for _, d in vals) / len(vals),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "impl": "reference",
            "config": {"workload": workload_name(args.num_envs), "note": note + "; cost is linear in num_envs"},
            "cpu_baseline": {"value": rate, "unit": "estimates/s", "cores": threads, "kind": kind,
                             "sample": f"{sample} envs per step of the {args.num_envs}-env workload (per-env loop, linear)"},
            "e2e": {"value": rate, "unit": "estimates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def instrumented_pass(eng, n_env, E1, E2):
    """One extra, untimed-for-the-headline pass with a CUDA-event pair around every launch group."""
    ev = lambda: torch.cuda.Event(enable_timing=True)
    rec = []

    def timed(name, kind, fn):
        a, b = ev(), ev()
        a.record(); fn(); b.record()
        rec.append((name, kind, a, b))

    for name, op in eng.backbone_ops:
        timed(name, getattr(op, "kind", "aux"), lambda op=op: op(2 * n_env))
    marks = []

    def mark(name):
        e = ev(); e.record(); marks.append((name, e))
    start = ev(); start.record()
    eng.stereo(n_env, E1, E2, mark=mark, o2=n_env)
    torch.cuda.synchronize()
    out = {}
    for name, kind, a, b in rec:
        d = out.setdefault(kind, {"ms": 0.0, "launches": 0})
        d["ms"] += a.elapsed_time(b); d["launches"] += 1
    per_op = {name: a.elapsed_time(b) for name, kind, a, b in rec}
    prev = start
    for name, e in marks:
        per_op["stereo." + name] = prev.elapsed_time(e)
        prev = e
    return out, per_op


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--num-envs", type=int, default=1024)
    ap.add_argument("--chunk", type=int, default=74,
                    help="envs per chunk (= what an auto-sized estimator grows to); 74 = num_SMs / 2: 148 frames per backbone launch = whole "
                         "waves of 128-row tiles on 148 SMs.  Measured A/B on one box: chunk 148 gives the same device-resident rate "
                         "(3373-3400 vs 3369-3377) but 5 %% less end to end (3232-3278 vs 3411)")
    ap.add_argument("--precision", default="fp16f8")
    ap.add_argument("--unique", type=int, default=32)
    ap.add_argument("--cpu-sample", type=int, default=16)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU legs (profiling runs)")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configurations and the e2e variants")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the boxes of the last timed step to DIR/boxes.npy (float64 [num_envs, 8, 3]; a seeded sample of the "
                         "environments if that exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl in ("reference", "cpu-sample"):
        ap.error("--dump-outputs writes the outputs of the device path, not of the CPU reference arm")
    if args.impl in ("reference", "cpu-sample"):
        os.environ["CUDA_VISIBLE_DEVICES"] = ""         # the CPU arm must not see a GPU (see cpu_legs_subprocess); set before CUDA initialises
    if args.impl == "cpu-sample":
        run_cpu_sample(args)
        return
    rank, world, local = dist_setup()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the product path has no CPU fallback)"
    import torch.distributed as dist
    from rgbmanip_b200 import _lib
    from rgbmanip_b200.dist import shard_range
    from rgbmanip_b200.estimator import AdaPoseEstimator_v5
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from rgbmanip_b200.dist import bind_to_gpu_numa
    numa_bound = bind_to_gpu_numa(dev) if world > 1 else False     # pinned host frames on the GPU's own NUMA node
    lib = _lib.load()
    N = args.num_envs
    lo, hi, per = shard_range(N, rank, world)
    n_loc = hi - lo
    # synthetic inputs: `unique` distinct envs (the same on every rank), global env g = unique env g % unique; this rank's shard is
    # resident in HBM and mirrored in pinned host memory
    base = synth.make_batch(args.unique, seed=100, special=True)
    order = ("K", "rgb1", "mask1", "E1", "rgb2", "mask2", "E2")
    base_t = {}
    for name, arr in zip(order, base.args()):
        t = torch.from_numpy(np.ascontiguousarray(arr))
        base_t[name] = t.to(torch.uint8) if name.startswith("mask") else t
    idx = (lo + np.arange(n_loc)) % args.unique
    host = {k: v[idx].contiguous().pin_memory() for k, v in base_t.items()}
    devt = {k: v.to(dev) for k, v in host.items()}
    est = AdaPoseEstimator_v5(None, dict(CFG), None, state_dict=weights.init_state_dict(0), device=dev, max_envs=args.chunk,
                              precision=args.precision)
    eng = est.estimator
    gathered = torch.zeros((world * per, 8, 3), dtype=torch.float64, device=dev)

    def gather(out):
        if world == 1:
            return out
        pad = out if n_loc == per else torch.cat([out, out.new_zeros((per - n_loc, 8, 3))])
        dist.all_gather_into_tensor(gathered, pad)
        return gathered[:N]

    last = {}

    def step_device():
        last["boxes"] = gather(est.estimate(*[devt[k] for k in order], return_tensor=True, env_offset=lo))
        return last["boxes"]

    def step_host(src=host):
        return gather(est.estimate(*[src[k] for k in order], return_tensor=True, env_offset=lo)).cpu()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        l0 = lib.adp_launch_count()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = a.elapsed_time(b)
        launches = lib.adp_launch_count() - l0
        if world > 1:
            t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        return ms, wall, launches

    # ---- parity gate inside the measurement: the golden envs through this very estimator (chunk size, graph replay)
    parity = parity_check(est, 2 * args.chunk) if rank == 0 else None
    barrier()

    sampler = ClockSampler(local)
    sampler.start()
    ms, wall, launches = timed(step_device, args.steps, args.warmup)
    clocks = sampler.stop()
    value = N * args.steps / (ms / 1e3)
    eng.check_error_flag()
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, "boxes", last["boxes"])     # before the next gather reuses its buffer

    e2e = None
    h2d = sum(host[k].numel() * host[k].element_size() for k in order)
    if not args.no_e2e:
        b0 = est.h2d_bytes
        ms_h, wall_h, _ = timed(step_host, max(1, args.steps), 2)
        h2d_real = (est.h2d_bytes - b0) // (max(1, args.steps) + 2)
        e2e = {"value": N * max(1, args.steps) / wall_h, "unit": "estimates/s", "h2d_bytes_per_step": int(h2d_real),
               "host_input_bytes_per_step": int(h2d),
               "h2d_note": "of every host frame only the rows under its crop window are uploaded (masks first, windows read back from the device)",
               "d2h_bytes_per_step": int(n_loc * 24 * 8), "timed": "host wall clock around estimate() + all-gather + D2H; pinned fp32 host inputs",
               "chunks": [h - l for l, h in est._chunk_bounds(n_loc, True)]}

    # ---- sharded result == one-rank result (same sampler seed; the sampler is keyed by the global env index)
    SEED = 424242
    mine = gather(est.estimate(*[devt[k] for k in order], return_tensor=True, env_offset=lo, sample_seed=SEED)).clone()
    identity = None
    if rank == 0:
        if world > 1:
            gidx = np.arange(N) % args.unique
            full = [base_t[k][gidx].to(dev) for k in order]
            alone = est.estimate(*full, return_tensor=True, sample_seed=SEED)
            del full
            what = f"{world}-rank sharded + all-gathered boxes vs a 1-rank run of the same {N} envs on rank 0"
        else:
            alone = est.estimate(*[host[k] for k in order], return_tensor=True, sample_seed=SEED)     # other chunking (host path)
            what = ("device-resident run (equal chunks) vs the host-input run (small first chunk + equal chunks) of the same "
                    f"{N} envs: an environment's box does not depend on how the batch is cut")
        diff = (mine - alone).abs()
        diff = torch.where(torch.isnan(diff), torch.zeros_like(diff), diff)
        identity = {"what": what, "envs": int(N), "bit_identical_envs": int((diff.reshape(N, -1).max(1).values == 0).sum()),
                    "max_abs_diff_m": float(diff.max()), "checksum": float(torch.nan_to_num(mine).sum())}
        torch.cuda.empty_cache()
    barrier()

    variants, configs = {}, {}
    if not args.no_extra:
        # ---- e2e with the RL caller's real input format: pageable float64 numpy (rl_pose.py:194-218), bounded to 256 envs
        nv = min(n_loc, 256)
        if nv:
            f64 = {k: (host[k][:nv].numpy().astype(np.float64) if k.startswith(("rgb", "mask")) else host[k][:nv].numpy().copy()) for k in order}
            run = lambda: est.estimate(*[f64[k] for k in order])
            run()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(2):
                run()
            dt = (time.perf_counter() - t0) / 2
            variants["pageable_float64_numpy"] = {"value": nv * world / dt, "unit": "estimates/s", "num_envs": nv * world, "host_bytes_per_step": int(sum(v.nbytes for v in f64.values())),
                                                  "note": "what rl_pose.py passes; staged through pinned buffers and demoted to float32 on the way (host-copy bound)"}
            del f64
            u8 = {k: ((host[k] * 255).round().to(torch.uint8).pin_memory() if k.startswith("rgb") else host[k]) for k in order}
            b0 = est.h2d_bytes
            ms_u, wall_u, _ = timed(lambda: step_host(u8), 2, 1)
            variants["pinned_uint8"] = {"value": N * 2 / wall_u, "unit": "estimates/s", "num_envs": N,
                                        "h2d_bytes_per_step": int((est.h2d_bytes - b0) // 3)}
            est._window_upload = False
            b0 = est.h2d_bytes
            ms_w, wall_w, _ = timed(step_host, 2, 1)
            est._window_upload = True
            variants["pinned_float32_whole_frames"] = {"value": N * 2 / wall_w, "unit": "estimates/s", "num_envs": N,
                                                       "h2d_bytes_per_step": int((est.h2d_bytes - b0) // 3),
                                                       "note": "window_upload off: every frame uploaded whole (the round-1 behaviour)"}
            del u8
        # ---- the whole box from ONE process (cfg["devices"]): what an unmodified vec-env host gets without torchrun
        if world == 1 and torch.cuda.device_count() > 1:
            ndev = torch.cuda.device_count()
            est_m = AdaPoseEstimator_v5(None, dict(CFG, devices=list(range(ndev))), None, state_dict=weights.init_state_dict(0),
                                        max_envs=args.chunk, precision=args.precision)
            run = lambda: est_m.estimate(*[host[k] for k in order])
            for _ in range(3):
                run()
            t0 = time.perf_counter()
            for _ in range(3):
                out_m = run()
            dt = (time.perf_counter() - t0) / 3
            ref_m = est.estimate(*[host[k] for k in order], sample_seed=est_m._seed + 7919 * est_m._calls)
            variants["single_process_all_gpus"] = {"value": N / dt, "unit": "estimates/s", "devices": ndev, "num_envs": N,
                                                   "bit_identical_to_one_gpu": bool(np.array_equal(out_m, ref_m)),
                                                   "note": "AdaPoseEstimator_v5(cfg['devices']=[0..n)): one engine per GPU, one host thread each, pinned fp32 host inputs"}
            del est_m
            torch.cuda.empty_cache()
        # ---- BASELINE configs[1]: N = 64, one view per env: backbone + NOCS
        n64 = min(64, n_loc)
        if n64:
            a = [devt["K"][:n64], devt["rgb1"][:n64], devt["mask1"][:n64]]
            f = lambda: est.estimate_nocs_single_view(*a)
            f(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(5):
                f()
            dt = (time.perf_counter() - t0) / 5
            configs["single_view_nocs_n64"] = {"value": n64 / dt, "unit": "frames/s", "ms_per_step": dt * 1e3, "num_envs": n64,
                                               "what": "BASELINE configs[1]: 64 envs, one view each: preprocess + PSPNet + NOCS head, device-resident frames, NOCS read back"}
        # ---- BASELINE configs[2] (N = 256 mug ring, 4 views) and configs[4] (this rank's share of the N = 4096 observation step)
        from rgbmanip_b200.actor import DeviceActor
        from rgbmanip_b200.view_ring import ViewRing

        def ring_bench(n_ring, task, with_actor):
            est.cfg["task_name"] = task
            ring = ViewRing(est, n_ring, 5)
            ridx = torch.arange(n_ring, device=dev) % n_loc
            views = [{"camera0": {"Color": devt[f"rgb{v}"][ridx], "Mask": devt[f"mask{v}"][ridx], "Intrinsic": devt["K"][ridx],
                                  "Extrinsic": devt[f"E{v}"][ridx]}} for v in (1, 2)]
            pose = torch.zeros((n_ring, 7), dtype=torch.float64, device=dev)
            actor = None
            if with_actor:
                g = torch.Generator().manual_seed(0)
                dims = [60, 96, 96, 32, 12]                    # cfg/controller/rl.yaml pi_hid_sizes, 12 actions
                sd = {}
                for i, (a_, b_) in enumerate(zip(dims[:-1], dims[1:])):
                    sd[f"actor.{2 * i}.weight"] = torch.randn((b_, a_), generator=g) / a_ ** 0.5
                    sd[f"actor.{2 * i}.bias"] = torch.zeros(b_)
                actor = DeviceActor(sd, ring, activation="elu")
            state = {"t": 0}

            def step():
                ring.add_view(views[state["t"] % 2], pose)
                ring.accumulate_steps = min(ring.accumulate_steps + 1, ring.max_steps)
                state["t"] += 1
                out = ring.get_estimation(return_tensor=True)
                if actor is not None:
                    actor.act_inference()
                return out
            for _ in range(4):
                step()                               # 4 views in the ring
            ms_r, _, _ = timed(step, 3, 0)
            pairs = ring.pair_slots()
            res = {"ms_per_step": ms_r / 3, "value": n_ring * world * 3 / (ms_r / 1e3), "unit": "estimates/s", "num_envs": n_ring * world,
                   "views_in_ring": int((ring.avail > 0).sum(0).max()), "cache_gb": ring.feat.numel() * 6 / 1e9}
            if not with_actor:       # the reference-equivalent cost: both paired views through the whole network again
                a2 = [views[0]["camera0"]["Intrinsic"], views[0]["camera0"]["Color"], views[0]["camera0"]["Mask"], views[0]["camera0"]["Extrinsic"],
                      views[1]["camera0"]["Color"], views[1]["camera0"]["Mask"], views[1]["camera0"]["Extrinsic"]]
                rec = lambda: est.estimate(*a2, return_tensor=True)[:, [0, 2, 4, 6, 1, 3, 5, 7]]
                ms_c, _, _ = timed(rec, 3, 2)
                res["recomputed"] = {"ms_per_step": ms_c / 3, "value": n_ring * world * 3 / (ms_c / 1e3), "unit": "estimates/s"}
            del ring, actor, views
            torch.cuda.empty_cache()
            est.cfg["task_name"] = CFG["task_name"]
            return res
        n_mug = max(1, 256 // world)
        configs["mug_ring_n256"] = dict(ring_bench(n_mug, "mugs", False),
                                        what="BASELINE configs[2]: adapose_mug, 4 views per env in the device ring, pairing rule of rl_pose.py:199-208, "
                                             "stereo estimate + fit + mug corner permutation; `value` = one new frame per env with the cached "
                                             "features of the other view, `recomputed` = both paired frames through the whole network (reference-equivalent)")
        n_obs = 4096 // 8                               # per-GPU share of the 8-GPU configuration
        configs["obs_step_n4096_share"] = dict(ring_bench(n_obs, "one_drawer_cabinet", True),
                                               what=f"BASELINE configs[4]: open_drawer observation step at num_envs=4096 on 8 GPUs = {n_obs} envs per GPU; this line "
                                                    f"runs that share on each of the {world} rank(s): add_view (preprocess + backbone of the new frame) + "
                                                    "get_estimation (stereo head on cached features) + get_observation + actor forward (60-96-96-32-12 ELU)")

        # ---- the other fit branches and the transformer variant (SURVEY 8(f)-4), 256 envs device-resident, for the record
        if world == 1:
            from rgbmanip_b200.estimator import AdaPoseEstimator_baseline
            n_v = min(256, n_loc)
            a_v = [devt[k][:n_v] for k in ("K", "rgb1", "mask1", "E1", "rgb2", "mask2", "E2")]
            variants_fit = {}
            for label, cls, extra, arch in (("branch_b_ransac_umeyama", AdaPoseEstimator_v5, {"direct_regression": False, "use_depth": True}, "v5"),
                                            ("branch_c_nocs_matching_pnp", AdaPoseEstimator_v5, {"direct_regression": False, "use_depth": False}, "v5"),
                                            ("transformer_variant_adapose_baseline", AdaPoseEstimator_baseline, {"name": "adapose_baseline"}, "baseline")):
                cfg_v = dict(CFG, **extra)
                sd_v = weights.init_state_dict(0, regress_pose=cfg_v["direct_regression"], arch=arch)
                est_v = cls(None, cfg_v, None, state_dict=sd_v, device=dev, max_envs=min(args.chunk, n_v), precision=args.precision)
                f_v = lambda: est_v.estimate(*a_v, return_tensor=True)
                ms_v, wall_v, _ = timed(f_v, 2, 2)
                variants_fit[label] = {"value": n_v * 2 / wall_v, "unit": "estimates/s", "num_envs": n_v, "ms_per_step": wall_v * 1e3 / 2}
                est_v.estimator.close()
                del est_v
                torch.cuda.empty_cache()
            variants_fit["branch_c_nocs_matching_pnp"]["note"] = ("device part (NOCS of both views, matching, triangulation, median scale) + the "
                                                                  "reference's cv2.solvePnPRansac per environment on a host thread pool (~18 ms per environment and thread), which is the bound")
            configs["other_branches_n256"] = variants_fit

    # ---- per-kernel-class timing of one chunk, live, on the launching stream
    n_chunk = min(eng.E, n_loc)
    E1c = devt["E1"][:n_chunk].contiguous(); E2c = devt["E2"][:n_chunk].contiguous()
    eng.run_chunk(devt["K"][:n_chunk], devt["rgb1"][:n_chunk], devt["mask1"][:n_chunk], E1c, devt["rgb2"][:n_chunk], devt["mask2"][:n_chunk], E2c)
    # three instrumented passes, per-op median: a single pass right after the previous leg catches the GPU mid clock ramp
    passes = [instrumented_pass(eng, n_chunk, E1c, E2c) for _ in range(3)]
    per_op = {k: float(np.median([p[1][k] for p in passes])) for k in passes[0][1]}
    classes = {k: {"ms": float(np.median([p[0][k]["ms"] for p in passes])), "launches": passes[0][0][k]["launches"]} for k in passes[0][0]}
    pk = peaks()
    frames = 2 * n_chunk
    npass = {"fp16f8": 1.5, "fp16x2": 2, "bf16x3": 3, "bf16": 1}[eng.precision]
    tc_ms = classes.get("tc", {}).get("ms", 0.0)
    tc_flops = GF_BACKBONE_TC_PER_FRAME * frames
    roof = None
    prof = NCU_PROFILE.get(eng.precision)
    if tc_ms > 0:
        ach = tc_flops / (tc_ms / 1e3) / 1e12
        roof = {"bound": "tensor", "kernel": "tc_conv_kernel (tcgen05 implicit-GEMM, backbone 2-D convs) + the two upconv_blend launches that "
                                             "complete the restructured up_1 / up_2 stages", "achieved": ach,
                "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tf_sustained"],
                "traffic": prof["dram_bytes_per_frame"] * frames if prof else None,
                "traffic_note": ("PROFILE CONSTANT, not measured in this run: dram__bytes_read+write of the launch group in the ncu capture "
                                 f"{prof['src']}, scaled to this chunk") if prof else "no ncu capture of this precision mode committed yet",
                "tensor_pipe_active_ncu": prof["tensor_pipe_active"] if prof else None,
                "peak_source": pk["src"] + " (sustained: timed inside a long step)",
                "algorithmic_flops_per_launch_group": tc_flops, "launches": classes["tc"]["launches"],
                "executed_flops_per_launch_group": GF_BACKBONE_EXECUTED_PER_FRAME * frames,
                "tensor_pipe_work_frac": ach * npass / pk["tf_sustained"] * GF_BACKBONE_EXECUTED_PER_FRAME / GF_BACKBONE_TC_PER_FRAME,
                "note": f"algorithmic FLOPs (SURVEY A.3) / summed CUDA-event time of the {classes['tc']['launches']} launches of one chunk "
                        f"({frames} frames); precision {eng.precision} issues {npass} fp16-equivalent MMA pass(es) per algorithmic FLOP"
                        + (" (the wide layers run the low-order weight term as an fp8 MMA at twice the rate)" if eng.precision == "fp16f8" else "")
                        + "; `achieved` counts the reference's FLOPs (conv 3x3 over the upsampled maps), `executed_flops...` what the GEMMs "
                          "really issue after up_1 / up_2 were restructured (upsampling and channel mixing commute)"}
    cr_ms = sum(v for k, v in per_op.items() if k.startswith("stereo.cr."))
    vol_ms = per_op.get("stereo.volume", 0.0)
    dg_ms = per_op.get("stereo.decode_gather", 0.0)
    hbm = {}
    if cr_ms + vol_ms > 0:
        gbs = BYTES_VOLUME_COSTREG_PER_ENV * n_chunk / ((cr_ms + vol_ms) / 1e3) / 1e9
        hbm["volume_costreg"] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                                 "ms_per_chunk": cr_ms + vol_ms, "algorithmic_bytes_per_env": BYTES_VOLUME_COSTREG_PER_ENV,
                                 "variant": "materialised fp16 volume (SURVEY 8(d): 302.7 MB per reference view)"}
    if dg_ms > 0:
        gbs = BYTES_DECODE_GATHER_PER_ENV * n_chunk / (dg_ms / 1e3) / 1e9
        hbm["decode_gather"] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                                "ms_per_chunk": dg_ms, "algorithmic_bytes_per_env": BYTES_DECODE_GATHER_PER_ENV,
                                "note": "bytes the gather formulation must touch (16 B voxels of the last U-Net tensor, fp32 feature corners); "
                                        "most of it is L2-resident, so this is an L2-path figure quoted against the HBM peak"}
    kernels = {k: {"ms_per_chunk": v["ms"], "launches": v["launches"]} for k, v in classes.items()}
    kernels["chunk_envs"] = n_chunk
    kernels["costreg_tflops"] = GF_COSTREG_PER_VIEW * n_chunk / (cr_ms / 1e3) / 1e12 if cr_ms > 0 else None
    kernels["stereo_ms"] = {k[7:]: v for k, v in per_op.items() if k.startswith("stereo.")}

    if rank == 0:
        cpu = {"value": 0.0, "unit": "estimates/s", "cores": 0, "kind": "skipped", "sample": "--no-cpu"}
        if not args.no_cpu:
            c = cpu_legs_subprocess(args.cpu_sample)
            cpu = {"value": c["rate"], "unit": "estimates/s", "cores": c["threads"], "kind": c["kind"],
                   "sample": f"{args.cpu_sample} envs of the workload through the reference's per-env loop on the host cores ({c['dt']:.1f} s)"}
            if c.get("single_view") is not None:
                configs["cpu_single_view_b1"] = c["single_view"]
        line = {"metric": "pose estimates/sec at num_envs=1024", "value": value, "unit": "estimates/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16" if eng.precision.startswith("bf16") else "fp16",
                "data": f"synthetic ({args.unique} seeded envs tiled to {N})",
                "config": {"workload": workload_name(N),
                           "precision": eng.precision, "chunk_envs": eng.E, "sharding": f"env-sharded dp{world}, NCCL all-gather of poses",
                           "l2": "inputs (>= 8 GB per step) exceed the 126 MB L2; no explicit flush needed",
                           "sampling": "device hash sampler for the 1024-pixel subset, keyed by the global env index",
                           "host_threads_bound_to_gpu_numa_node": bool(numa_bound)},
                "roofline": roof, "roofline_hbm": hbm, "cpu_baseline": cpu,
                "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "kernels": kernels,
                "parity_in_bench": parity, "shard_identity": identity, "e2e_variants": variants, "configs": configs,
                "wall_s_timed_region": wall}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
