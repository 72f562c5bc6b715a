"""CPU checks of the seeded sampler's restatement (tests/sampling_oracle.py): its draws follow softmax of the top-k
filtered, temperature-scaled logits, draws of consecutive steps are independent, its kept set is the reference's, and
its hash is the dropout hash of csrc/kernels.cuh."""
import numpy as np
import pytest
import torch
from scipy import stats

import sampling_oracle as SO
from oracle import valle_oracle as O

N_SEEDS = 100_000  # x 2 consecutive steps = 200k (seed, step) pairs per configuration


def _row(V=1025):
    g = torch.Generator().manual_seed(7)
    return torch.randn(V, generator=g) * 1.5


def _draws(z, top_k, T):
    """draws at steps (t, t + 1) of N_SEEDS random seeds: [N_SEEDS, 2]"""
    rng = np.random.default_rng(11)
    seeds = rng.integers(0, 2 ** 64, size=N_SEEDS, dtype=np.uint64)
    t0 = rng.integers(0, 4000, size=N_SEEDS).astype(np.uint64)
    out = np.empty((N_SEEDS, 2), dtype=np.int64)
    for c in range(0, N_SEEDS, 4000):
        for j in range(2):
            out[c:c + 4000, j] = SO.seeded_draw(z, seeds[c:c + 4000], t0[c:c + 4000] + np.uint64(j), top_k, T)
    return out


def _pooled(ids, p, min_expected=5.0):
    """observed / expected counts over the ids, categories with a small expectation pooled into one"""
    n = ids.size
    obs = np.bincount(ids, minlength=p.size).astype(np.float64)
    exp = p * n
    big = exp >= min_expected
    o, e = list(obs[big]), list(exp[big])
    if (~big & (p > 0)).any():
        o.append(obs[~big].sum())
        e.append(exp[~big].sum())
    return np.array(o), np.array(e)


@pytest.mark.parametrize("top_k", [5, -100])
@pytest.mark.parametrize("T", [1.0, 0.7])
def test_seeded_draws_follow_the_filtered_softmax_and_are_independent(top_k, T):
    z = _row()
    p = torch.softmax(O.top_k_top_p_filtering((z / T).view(1, -1), top_k=top_k).double(), -1)[0].numpy()
    d = _draws(z, top_k, T)
    assert p[d.reshape(-1)].min() > 0, "an id outside the kept set was drawn"
    obs, exp = _pooled(d.reshape(-1), p)
    chi = stats.chisquare(obs, exp * obs.sum() / exp.sum())
    assert chi.pvalue > 1e-3, (chi.statistic, chi.pvalue, len(obs))
    # consecutive steps of one seed: ids grouped into ~equal-mass classes, then a contingency test
    order = np.argsort(-p)
    cls = np.zeros(p.size, dtype=np.int64)
    cls[order] = np.minimum((np.cumsum(p[order]) - p[order]) * 8, 7).astype(np.int64)
    a, b = cls[d[:, 0]], cls[d[:, 1]]
    n_cls = int(cls.max()) + 1
    table = np.zeros((n_cls, n_cls))
    np.add.at(table, (a, b), 1)
    table = table[table.sum(1) > 0][:, table.sum(0) > 0]
    ind = stats.chi2_contingency(table)
    assert ind.pvalue > 1e-3, (ind.statistic, ind.pvalue, table.shape)


@pytest.mark.parametrize("T", [1.0, 0.7, 1.3])
def test_kept_set_is_the_reference_filter_including_ties(T):
    z = _row()
    top = torch.topk(z, 5).indices.tolist()
    rest = [i for i in (100, 200, 300, 400) if i not in top][:3]
    kth = float(z[top[4]])
    z[rest[0]], z[rest[1]] = kth, kth                    # two more ids tie with the 5th largest value
    z[rest[2]] = torch.nextafter(torch.tensor(kth), torch.tensor(-1e9))  # one just below it
    for top_k in (1, 5, 7, 1025, 2000, 0, -100):
        want = torch.isfinite(O.top_k_top_p_filtering((z / T).view(1, -1), top_k=top_k))[0].numpy()
        got = SO.kept(z, top_k, T)
        assert np.array_equal(got, want), top_k
    assert SO.kept(z, 5, T).sum() == 7


def test_seeded_draw_keys_ties_to_the_lowest_id_and_respects_top_k_one():
    z = _row()
    for s in range(50):
        assert SO.seeded_draw(z, s, s, 1, 1.0) == int(torch.argmax(z))
    keys = SO.seeded_keys(z, 3, 9, -100, 1.0)
    assert np.isfinite(keys).all() and keys.dtype == np.float32


def test_hash_is_the_dropout_hash():
    """thresholding mix64 as drop_keep does reproduces the dropout-mask restatement of test_backward_gpu"""
    from test_backward_gpu import _keep_mask
    n = 1 << 16
    for seed, stream, p in ((0x1234567890ABCDEF % (1 << 62), 7, 0.1), (987654321, (3 << 2) | 2, 0.5), (2 ** 64 - 1, 0, 0.3)):
        h = SO.mix64(seed, stream, np.arange(n, dtype=np.uint64))
        keep = (h >> np.uint64(32)) >= np.uint64(int(p * 4294967296.0))
        assert np.array_equal(keep, _keep_mask(seed, stream, n, p).numpy())
