"""The launch schedule of a view ring sharded over devices (rgbmanip_b200.view_ring.ring_pieces), on the CPU: every
environment is covered once, and its random draws are keyed as a one-device ring of the same configuration keys them."""
import pytest

from rgbmanip_b200.dist import shard_range
from rgbmanip_b200.view_ring import ring_pieces


def _one_device_keys(num_envs, key):
    """env -> (seed offset, frame id): a one-device ring launches chunks [lo, lo + key) with seed offset lo and frame ids
    counted from 0 inside the chunk (view_ring.py before sharding: ``for lo in range(0, N, eng.F)``)."""
    out = {}
    for lo in range(0, num_envs, key):
        for g in range(lo, min(num_envs, lo + key)):
            out[g] = (lo, g - lo)
    return out


CASES = [  # (num_envs, world, key chunk, replica capacity)
    (5, 2, 2, 2),           # the GPU test's setup: a key chunk straddles the shard boundary
    (5, 2, 4, 4),           # add_view of the same ring: chunks of 2 x max_envs frames
    (3, 4, 2, 2),           # fewer environments than devices: an empty shard
    (3, 8, 16, 16),
    (100, 8, 74, 16),       # auto-sized: the replicas' 13-env shards run with a smaller capacity than the key chunk
    (4096, 8, 74, 74),      # the 8-GPU controller step
    (4096, 8, 148, 148),
    (1000, 3, 74, 74),      # uneven shards
    (1000, 7, 74, 20),
    (17, 5, 6, 4),
    (1, 1, 16, 16),
]


@pytest.mark.parametrize("num_envs,world,key,cap", CASES)
def test_shard_pieces_reproduce_the_one_device_keys(num_envs, world, key, cap):
    want = _one_device_keys(num_envs, key)
    seen = {}
    for r in range(world):
        lo, hi, _ = shard_range(num_envs, r, world)
        pieces = ring_pieces(key, lo, hi, cap)
        if hi <= lo:
            assert pieces == []
            continue
        assert pieces[0][0] == lo and pieces[-1][1] == hi
        for (a, b, k0), nxt in zip(pieces, pieces[1:] + [None]):
            assert 0 < b - a <= cap                       # fits the replica's launch
            assert k0 <= a and b <= k0 + key              # inside one key chunk
            if nxt is not None:
                assert nxt[0] == b                        # contiguous, in env order
            for g in range(a, b):
                assert g not in seen
                seen[g] = (k0, g - k0)                    # seed offset = key-chunk start, frame id = a - k0 + position
    assert seen == want


def test_one_device_schedule_is_the_plain_chunking():
    for n, key in ((1, 4), (4, 4), (9, 4), (148, 148), (4096, 148)):
        assert ring_pieces(key, 0, n, key) == [(lo, min(n, lo + key), lo) for lo in range(0, n, key)]


def test_padded_branch_b_launch_fits_a_key_chunk():
    """Device RANSAC draws (direct_regression=False) are keyed by the position inside the launch: a piece is launched behind
    a_lo - key_lo placeholders, which needs a_lo - key_lo + length <= key <= the replica's capacity."""
    for num_envs, world, key in ((5, 2, 2), (100, 8, 74), (4096, 8, 74), (17, 5, 6)):
        for r in range(world):
            lo, hi, _ = shard_range(num_envs, r, world)
            for a, b, k0 in ring_pieces(key, lo, hi, key):
                assert b - k0 <= key
