"""systematic_ancestors (CPU): systematic resampling within each camera's filters, survivors in place, copies in the slots of
the filters not drawn."""
import numpy as np
import pytest


def _plain_counts(w, u):
    """Systematic resampling as usually written: M pointers (u + k) / M into the cumulative normalised weights."""
    M = len(w)
    c = np.cumsum(np.asarray(w, dtype=np.float64) / np.sum(w))
    counts = np.zeros(M, dtype=int)
    i = 0
    for k in range(M):
        p = (u + k) / M
        while i < M - 1 and c[i] <= p:
            i += 1
        counts[i] += 1
    return counts


def _check_layout(anc, idx, counts):
    """Ancestors within group idx: drawn filters keep their slot, copies fill the undrawn slots in ascending order."""
    a = anc[idx]
    assert np.isin(a, idx).all(), "an ancestor outside the group"
    drawn = counts > 0
    assert np.array_equal(a[drawn], idx[drawn]), "a drawn filter lost its slot"
    extra = np.repeat(idx, np.maximum(counts - 1, 0))
    assert np.array_equal(a[~drawn], extra), "copies not in ascending order of the free slots"
    got = np.bincount(np.searchsorted(idx, a), minlength=idx.size)
    assert np.array_equal(got, counts), "ancestor counts"
    moved = a != idx
    assert not np.isin(a[moved], idx[moved]).any(), "a source is also overwritten"


@pytest.mark.parametrize("seed", range(6))
def test_counts_match_systematic_resampling(pkg, seed):
    rng = np.random.default_rng(seed)
    B = 64
    w = rng.gamma(0.5, size=B)
    u = float(rng.random())
    anc = pkg.systematic_ancestors(w, u)
    assert anc.dtype == np.int32 and anc.shape == (B,)
    _check_layout(anc, np.arange(B), _plain_counts(w, u))


@pytest.mark.parametrize("seed", range(4))
def test_groups_are_resampled_separately(pkg, seed):
    rng = np.random.default_rng(100 + seed)
    K, M = 5, 7
    cam = rng.permutation(np.repeat(np.arange(K), M))   # groups interleaved over the filters
    w = rng.exponential(size=K * M)
    w[rng.random(K * M) < 0.3] = 0.0
    for c in range(K):   # no group with zero weight
        w[np.flatnonzero(cam == c)[0]] += 0.5
    u = float(rng.random())
    anc = pkg.systematic_ancestors(w, u, camera_of=cam)
    assert np.array_equal(cam[anc], cam)
    for c in range(K):
        idx = np.flatnonzero(cam == c)
        _check_layout(anc, idx, _plain_counts(w[idx], u))


@pytest.mark.parametrize("value", [1.0, 0.1, 3e-7, 12345.678])
@pytest.mark.parametrize("u", [0.0, 0.5, 0.999999])
def test_equal_weights_give_the_identity(pkg, value, u):
    B = 97
    assert np.array_equal(pkg.systematic_ancestors(np.full(B, value), u), np.arange(B))
    cam = np.arange(B) % 4
    assert np.array_equal(pkg.systematic_ancestors(np.full(B, value), u, camera_of=cam), np.arange(B))


def test_one_weight_takes_every_slot(pkg):
    w = np.zeros(10)
    w[6] = 2.0
    assert np.array_equal(pkg.systematic_ancestors(w, 0.25), np.full(10, 6))


@pytest.mark.parametrize("w", [[1.0, -0.5, 1.0], [1.0, np.nan, 1.0], [1.0, np.inf, 1.0], [0.0, 0.0, 0.0]])
def test_bad_weights_raise(pkg, w):
    with pytest.raises(ValueError):
        pkg.systematic_ancestors(np.array(w), 0.5)


def test_zero_group_and_bad_offset_raise(pkg):
    with pytest.raises(ValueError):   # camera 1's weights sum to 0
        pkg.systematic_ancestors([1.0, 1.0, 0.0, 0.0], 0.5, camera_of=[0, 0, 1, 1])
    for u in (-0.1, 1.0, np.nan):
        with pytest.raises(ValueError):
            pkg.systematic_ancestors(np.ones(4), u)
    with pytest.raises(ValueError):
        pkg.systematic_ancestors(np.ones(4), 0.5, camera_of=[0, 1])
