"""Pair layout of the many-videos driver (geometry_from_features_batch).  Runs without a GPU."""
import numpy as np
import pytest

from evenvizion_b200.processing.video_processing import PairLayout

RAGGED = [3, 0, 5, 1, 5, 0, 2]          # pairs per video: empty (one-frame) videos, a one-pair video, ties


def _input_order(n):
    return [(v, k) for v in range(len(n)) for k in range(n[v])]


def test_step_major_layout_on_ragged_videos():
    lay = PairLayout(RAGGED, step_major=True)
    P = sum(RAGGED)
    assert len(lay.video) == len(lay.k) == len(lay.inverse) == P
    # videos by pair count, longest first, ties in input order: 2, 4, 0, 6, 3 (1 and 5 have no pairs)
    rank = [2, 4, 0, 6, 3]
    expect = [(v, k) for k in range(max(RAGGED)) for v in rank if RAGGED[v] > k]
    assert list(zip(lay.video.tolist(), lay.k.tolist())) == expect
    assert lay.step_off.tolist() == [0, 5, 9, 12, 14, 16]
    # the chains still running at step k are a prefix of those at step k - 1
    sizes = np.diff(lay.step_off)
    assert sizes.tolist() == [5, 4, 3, 2, 2]
    for k in range(len(sizes)):
        a, b = lay.step_off[k], lay.step_off[k + 1]
        assert (lay.k[a:b] == k).all()
        assert lay.video[a:b].tolist() == rank[:sizes[k]]
    assert lay.seg_off.tolist() == [0, 3, 3, 8, 9, 14, 14, 16]
    # inverse permutation: processing order -> input order (video-major, videos in input order)
    back = list(zip(lay.video[lay.inverse].tolist(), lay.k[lay.inverse].tolist()))
    assert back == _input_order(RAGGED)
    parts = lay.split(np.arange(P))
    assert [len(x) for x in parts] == RAGGED
    for v, x in enumerate(parts):
        assert (lay.video[x] == v).all() and lay.k[x].tolist() == list(range(RAGGED[v]))


def test_video_major_layout_is_input_order():
    lay = PairLayout(RAGGED, step_major=False)
    assert list(zip(lay.video.tolist(), lay.k.tolist())) == _input_order(RAGGED)
    assert lay.inverse.tolist() == list(range(sum(RAGGED)))
    assert lay.seg_off.tolist() == [0, 3, 3, 8, 9, 14, 14, 16]
    assert lay.step_off is None


@pytest.mark.parametrize("step_major", [True, False])
@pytest.mark.parametrize("n", [[], [0], [0, 0], [1], [7], [1, 0, 1]])
def test_layout_degenerate_batches(n, step_major):
    lay = PairLayout(n, step_major)
    P = sum(n)
    assert len(lay.k) == P and lay.seg_off[-1] == P and len(lay.seg_off) == len(n) + 1
    assert sorted(zip(lay.video[lay.inverse].tolist(), lay.k[lay.inverse].tolist())) == _input_order(n)
    if step_major:
        assert lay.step_off[0] == 0 and lay.step_off[-1] == P and len(lay.step_off) == max(n, default=0) + 1


def test_layout_random_ragged():
    rng = np.random.default_rng(0)
    n = rng.integers(0, 40, 50).tolist()
    lay = PairLayout(n, True)
    sizes = np.diff(lay.step_off)
    assert (np.diff(sizes) <= 0).all()                                   # non-increasing active prefix
    assert sizes.tolist() == [sum(1 for x in n if x > k) for k in range(max(n))]
    assert list(zip(lay.video[lay.inverse].tolist(), lay.k[lay.inverse].tolist())) == _input_order(n)
