"""The view ring, the device actor and single-view NOCS over a multi-device estimator (``devices``: one replica per GPU in
one process) against the same calls on one device and the reference controller's queue state.

Up to four GPUs are used.  On a one-GPU machine the estimator gets two replicas on that GPU: each replica still owns its
engine, its ring shard and its host thread, which is everything the sharding changes."""
import os

import numpy as np
import pytest
import torch

from oracle import adapose_oracle as O
from oracle import view_ring_oracle as V
from rgbmanip_b200 import synth, weights

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore")]

ATOL = 2e-5      # metres: the ring tests' tolerance (identical inputs still differ by the atomicAdd order of per-env means)


def _devices():
    n = torch.cuda.device_count()
    return list(range(min(n, 4))) if n >= 2 else [0, 0]


def _estimator(max_envs, devices=None, task="one_drawer_cabinet", direct=True):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from rgbmanip_b200.estimator import AdaPoseEstimator_v5
    cfg = {"name": "adapose_v5", "task_name": task, "load": False, "img_size": 224, "use_depth": True, "n_pts": 1024,
           "direct_regression": direct, "real_world": False}
    return AdaPoseEstimator_v5(None, cfg, None, state_dict=weights.init_state_dict(0, regress_pose=direct), max_envs=max_envs,
                               devices=devices)


def _rings(N, T, max_envs, direct=True):
    from rgbmanip_b200.view_ring import ShardedViewRing, ViewRing
    one, multi = _estimator(max_envs, direct=direct), _estimator(max_envs, _devices(), direct=direct)
    r1, rm = ViewRing(one, N, T), ViewRing(multi, N, T)
    assert isinstance(rm, ShardedViewRing) and not isinstance(r1, ShardedViewRing)
    return r1, rm


def _assert_queues_equal(a, b):
    np.testing.assert_array_equal(a.available, b.available)
    np.testing.assert_array_equal(a.available_num, b.available_num)
    np.testing.assert_array_equal(a.bbox_queue, b.bbox_queue)
    np.testing.assert_array_equal(a.pose_queue, b.pose_queue)
    np.testing.assert_array_equal(a.pair_slots().cpu().numpy(), b.pair_slots().cpu().numpy())
    np.testing.assert_array_equal(a.choose.cpu().numpy(), b.choose.cpu().numpy())


def _add(ring, rgb, mask, K, E, pose):
    ring.add_view({"camera0": {"Color": rgb, "Mask": mask, "Intrinsic": K, "Extrinsic": E}}, pose)
    ring.accumulate_steps += 1


def _synthetic_steps(N):
    """The controller-like sequence of test_gpu_view_ring.test_ring_estimation_equals_estimator_on_paired_frames."""
    frames = []
    for s in range(3):
        b = synth.make_batch(N, seed=20 + s, special=False)
        frames.append((b.rgb1.astype(np.float64), b.mask1.astype(np.float64), b.K, b.E1))
        frames.append((b.rgb2.astype(np.float64), b.mask2.astype(np.float64), b.K, b.E2))
    frames[2] = (frames[2][0], np.where(np.arange(N)[:, None, None] == 1, 0.0, frames[2][1]), frames[2][2], frames[2][3])
    return frames


def test_sharded_queue_state_matches_reference_controller(golden_dir):
    from rgbmanip_b200.view_ring import ViewRing
    g = np.load(os.path.join(golden_dir, "view_ring.npz"))
    est = _estimator(2, _devices())
    ring = ViewRing(est, 3, 5)
    assert len(ring.shards) >= 2 and ring.device == est.device
    q = V.ViewQueues(3, 5)
    for t, (color, mask, K, E, pose) in enumerate(V.view_ring_script()):
        _add(ring, color / 100.0, mask, K, E, pose)
        q.add_view(color, mask, K, E, pose)
        q.accumulate_steps += 1
        np.testing.assert_array_equal(ring.available, g[f"s{t}_available"])
        np.testing.assert_array_equal(ring.available_num, g[f"s{t}_available_num"])
        np.testing.assert_array_equal(ring.bbox_queue, g[f"s{t}_bbox_queue"])
        np.testing.assert_array_equal(ring.pose_queue, g[f"s{t}_pose_queue"])
        sl = ring.pair_slots().cpu().numpy()
        np.testing.assert_array_equal(sl, q.pair_slots())
        ext = ring.extrinsic.cpu().numpy()
        for v, key in ((0, "E1"), (1, "E2")):
            got = np.array([ext[sl[v, e], e, 0] if sl[v, e] >= 0 else 0.0 for e in range(3)])
            np.testing.assert_array_equal(got, g[f"s{t}_{key}"])


def test_sharded_ring_equals_one_device_ring():
    """5 environments, max_envs = 2: the key chunks of both the pixel sampler (4 frames) and the RANSAC / stereo launches
    (2 envs) straddle a shard boundary.  Pixel subsets and queues are bit-equal at every step, boxes within ATOL."""
    N = 5
    r1, rm = _rings(N, 3, 2)
    bit_equal = True
    for t, (rgb, mask, K, E) in enumerate(_synthetic_steps(N)):
        pose = np.full((N, 7), float(t))
        _add(r1, rgb, mask, K, E, pose)
        _add(rm, rgb, mask, K, E, pose)
        _assert_queues_equal(r1, rm)
        a, b = r1.get_estimation(), rm.get_estimation()
        np.testing.assert_allclose(b, a, rtol=0, atol=ATOL)
        bit_equal &= np.array_equal(a, b)
        t_ = rm.get_estimation(return_tensor=True)
        assert t_.device == rm.device and tuple(t_.shape) == (N, 8, 3)
    assert not np.array_equal(a[0], O.DEFAULT_BBOX)
    print(f"sharded ring over {len(rm.shards)} replicas: boxes bit-equal to one device: {bit_equal}")


def test_quirk_132_one_visible_env_in_the_last_shard_marks_every_env():
    """rl_pose.py:132: one environment that sees the object marks every environment's slot available -- also when that
    environment lives on another device than the rest."""
    N = 5
    r1, rm = _rings(N, 4, 2)
    q = V.ViewQueues(N, 4)
    b = synth.make_batch(N, seed=7, special=False)
    blind = np.zeros_like(b.mask1)
    only_last = blind.copy()
    only_last[N - 1] = b.mask1[N - 1]
    lo_last = rm.shards[-1].env0
    assert lo_last > 0 and lo_last <= N - 1                  # env N-1 lives in the last shard, env 0 in another
    for t, m in enumerate((blind, only_last, blind)):
        pose = np.full((N, 7), float(t))
        for ring in (r1, rm):
            _add(ring, b.rgb1, m, b.K, b.E1, pose)
        q.add_view(b.rgb1, m, b.K, b.E1, pose)
        q.accumulate_steps += 1
        _assert_queues_equal(r1, rm)
        np.testing.assert_array_equal(rm.available, q.available)
        np.testing.assert_array_equal(rm.available_num, q.available_num)
        np.testing.assert_array_equal(rm.bbox_queue, q.bbox_queue)
    assert rm.available[1].tolist() == [1.0] * N and rm.available[0].sum() == 0 and rm.available[2].sum() == 0


def test_sharded_branch_b_equals_one_device_ring():
    """direct_regression=False: the RANSAC + Umeyama fit with given draws and with device-drawn ones."""
    N = 5
    r1, rm = _rings(N, 4, 2, direct=False)
    b = synth.make_batch(N, seed=31, special=False)
    for rgb, m, E in ((b.rgb1, b.mask1, b.E1), (b.rgb2, b.mask2, b.E2)):
        for ring in (r1, rm):
            _add(ring, rgb, m, b.K, E, np.zeros((N, 7)))
    _assert_queues_equal(r1, rm)
    ridx = np.random.default_rng(3).integers(0, 1024, size=(N, 128, 5)).astype(np.int32)
    a = r1.get_estimation(ransac_idx=ridx)
    assert not np.array_equal(a[0], O.DEFAULT_BBOX)
    np.testing.assert_allclose(rm.get_estimation(ransac_idx=ridx), a, rtol=0, atol=ATOL)
    a = r1.get_estimation()
    np.testing.assert_allclose(rm.get_estimation(), a, rtol=0, atol=ATOL)
    assert not np.array_equal(a[N - 1], O.DEFAULT_BBOX)


def test_sharded_device_actor_matches_reference(golden_dir):
    from rgbmanip_b200.actor import DeviceActor
    from rgbmanip_b200.view_ring import ViewRing
    g = np.load(os.path.join(golden_dir, "actor.npz"))
    sd = {k: g[k] for k in g.files if k.startswith("actor.")}
    ring = ViewRing(_estimator(2, _devices()), 3, 5)
    actor = DeviceActor(sd, ring)
    assert actor.dims == [60, 96, 96, 32, 12]
    for t, (color, mask, K, E, pose) in enumerate(V.view_ring_script()):
        if t >= 5:
            break
        _add(ring, color, mask, K, E, pose * 0.1)
        act, obs = actor.act_inference()
        assert act.device == ring.device and tuple(obs.shape) == (3, 60)
        np.testing.assert_array_equal(obs.cpu().numpy(), g[f"s{t}_obs"])
        np.testing.assert_allclose(act.cpu().numpy(), g[f"s{t}_act"], rtol=0, atol=2e-5)
    with pytest.raises(IndexError):
        actor.act_inference(accumulate_steps=6)


def test_attach_with_a_multi_device_estimator():
    from rgbmanip_b200 import view_ring

    class FakeController:                     # the attributes ControlInterface.__init__ sets (rl_pose.py:22-44)
        pass

    ci = FakeController()
    ci.estimator = _estimator(2, _devices())
    ci.num_envs, ci.max_steps, ci.accumulate_steps = 3, 5, 3
    ring = view_ring.attach(ci)
    assert isinstance(ring, view_ring.ShardedViewRing)
    assert ci.accumulate_steps == 0 and ci.pose_queue.shape == (5, 3, 7) and ci.available.sum() == 0
    b = synth.make_batch(3, seed=4, special=False)
    for rgb, m, E in ((b.rgb1, b.mask1, b.E1), (b.rgb2, b.mask2, b.E2)):
        ci.add_view({"camera0": {"Color": rgb, "Mask": m, "Intrinsic": b.K, "Extrinsic": E}}, np.full((3, 7), 0.5))
        ci.accumulate_steps += 1
    assert ci.available[:2].sum() == 6 and list(ci.available_num) == [2, 2, 2]
    assert np.all(ci.pose_queue[:2] == 0.5) and np.all(ci.bbox_queue[:2, :, 2] > ci.bbox_queue[:2, :, 0])
    box = ci.get_estimation()
    ch = ring.choose.cpu().numpy()
    want = ci.estimator.estimate(b.K, b.rgb1, b.mask1, b.E1, b.rgb2, b.mask2, b.E2, choose=(ch[0], ch[1]))
    np.testing.assert_allclose(box, want, rtol=0, atol=ATOL)
    ci.reset_queue()
    assert ci.available.sum() == 0 and ci.accumulate_steps == 0


def test_fewer_envs_than_devices():
    N = 1
    r1, rm = _rings(N, 3, 2)
    assert len(rm.shards) == 1 < len(rm.estimator._replicas)
    b = synth.make_batch(N, seed=5, special=False)
    for rgb, m, E in ((b.rgb1, b.mask1, b.E1), (b.rgb2, b.mask2, b.E2)):
        for ring in (r1, rm):
            _add(ring, rgb, m, b.K, E, np.ones((N, 7)))
        _assert_queues_equal(r1, rm)
        np.testing.assert_allclose(rm.get_estimation(), r1.get_estimation(), rtol=0, atol=ATOL)


def test_single_view_nocs_multi_device_equals_one_device():
    """BASELINE config 2 from one process: the blocks of estimate(), the global env index as the sampler key."""
    N = 7                                         # more than a chunk of 2 on every replica
    b = synth.make_batch(N, seed=9, special=True)
    one, multi = _estimator(2), _estimator(2, _devices())
    for call in range(2):
        a = one.estimate_nocs_single_view(b.K, b.rgb1, b.mask1)
        c = multi.estimate_nocs_single_view(b.K, b.rgb1, b.mask1)
        for x, y in zip(a, c):
            np.testing.assert_array_equal(x, y)
    assert a[2].any() and a[0].shape == (N, 1024, 3)
    ch = np.random.default_rng(1).integers(0, 224 * 224, size=(N, 1024)).astype(np.int32)
    a = one.estimate_nocs_single_view(b.K, b.rgb1, b.mask1, choose=ch)
    c = multi.estimate_nocs_single_view(b.K, b.rgb1, b.mask1, choose=ch)
    for x, y in zip(a, c):
        np.testing.assert_array_equal(x, y)
