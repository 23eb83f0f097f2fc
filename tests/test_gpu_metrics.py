"""Evaluation metrics on the device (`fr_topk_metrics`, `fr_by_user_metrics`) against the host metrics, the goldens
and numpy restatements; `ItemSets` construction on the host (CPU tests at the end)."""
import numpy as np
import pytest

from conftest import load_golden

import foodrec_b200  # noqa: F401
from foodrec_b200 import metrics as M

ALL = ("recall", "recall2", "ndcg", "precision", "map")


def _cuda(x, dtype=None):
    import torch
    t = torch.as_tensor(np.asarray(x))
    return (t.to(dtype) if dtype is not None else t).cuda()


def _host_columns(top, pos):
    """The per-user `[n, K]` arrays `metrics.topk_metrics` averages, with its dtypes and summation order, in
    `TOPK_METRICS` order (recall2: the hit count), and the list lengths."""
    hits = M.hit_matrix(top, pos)
    pos_len = np.fromiter((len(p) for p in pos), dtype=np.int64, count=hits.shape[0])
    n, K = hits.shape
    ranks = np.arange(1, K + 1)
    cum = np.cumsum(hits, axis=1)
    cut = np.minimum(pos_len, K)
    disc, ideal = M._ndcg_tables(K)
    idcg = ideal[np.minimum(np.arange(K)[None, :], (cut - 1)[:, None])]
    ndcg = np.cumsum(np.where(hits, disc, 0), axis=1) / idcg
    pre = cum / ranks
    ap = (np.cumsum(pre * hits.astype(np.float32), axis=1) / np.minimum(ranks[None, :], cut[:, None])).astype(np.float32)
    return [cum / pos_len.reshape(-1, 1), cum, ndcg, pre, ap], pos_len


def host_per_user(top, pos, topk):
    """`metrics.topk_metrics` without the mean: `[n, 5, len(topk)]` fp64."""
    cols, _ = _host_columns(top, pos)
    c = np.asarray(topk) - 1
    return np.stack([x[:, c].astype(np.float64) for x in cols], axis=1)


def host_means_unrounded(top, pos, topk):
    """The host's unrounded means, averaged exactly as `topk_metrics` averages them (fp32 for ndcg and map)."""
    cols, pos_len = _host_columns(top, pos)
    out = {}
    for m, x in zip(ALL, cols):
        v = x.sum(axis=0) / pos_len.sum() if m == "recall2" else x.mean(axis=0)
        for k in topk:
            out[f"{m}@{k}"] = float(v[k - 1])
    return out


def near_rounding_boundary(v, tol=1e-6):
    x = v * 1e4
    return abs((x - np.floor(x)) - 0.5) * 1e-4 < tol


def random_case(rng, n, n_items, K=50, pad=True, dup_cols=True, dup_pos=True):
    top = np.stack([rng.permutation(n_items)[:K] for _ in range(n)]).astype(np.int64)
    pos = [rng.choice(n_items, size=int(rng.integers(1, 70)), replace=False).tolist() for _ in range(n)]
    for r in range(n):      # make some hits likely: copy a few positives into the ranked list
        h = rng.choice(len(pos[r]), size=min(len(pos[r]), int(rng.integers(0, 8))), replace=False)
        top[r, rng.choice(K, size=h.size, replace=False)] = np.asarray(pos[r])[h]
    if pad:
        rows = rng.choice(n, size=n // 10, replace=False)
        for r in rows:
            top[r, int(rng.integers(1, K)):] = -1
    if dup_cols:
        rows = rng.choice(n, size=n // 10, replace=False)
        top[rows, 7] = top[rows, 3]
    if dup_pos:
        for r in rng.choice(n, size=n // 10, replace=False):
            pos[r] = pos[r] + pos[r][:1]
    return top, pos


# ------------------------------------------------------------------------------------------------ full sort (GPU)
@pytest.mark.gpu
def test_topk_goldens_through_device():
    import torch
    g = load_golden("primitives.npz")
    ptr, idx = g["rank/pos_ptr"], g["rank/pos_idx"]
    pos = [idx[ptr[u]:ptr[u + 1]].tolist() for u in range(len(ptr) - 1)]
    # precision@20 of this golden is exactly 11/800 = 0.01375, a rounding boundary: numpy's sequential fp64 sum lands
    # just below it (0.0137), the device's fp64 fold may land just above; the same explicit exception as for random cases
    unrounded = host_means_unrounded(g["rank/topi"], pos, (5, 10, 20, 50))
    exempt = {k for k, v in unrounded.items() if near_rounding_boundary(v)}
    assert "precision@20" in exempt
    for dt in (torch.int64, torch.int32):
        res = M.topk_metrics_device(_cuda(g["rank/topi"], dt), pos)
        for k, v in zip(g["rank/metric_keys"], g["rank/metric_vals"]):
            if str(k) in exempt:
                assert abs(res[str(k)] - v) <= 1.0001e-4, (k, res[str(k)], v)
            else:
                assert res[str(k)] == v, (k, res[str(k)], v)
        toy_top = np.array([[4, 1, 7], [0, 2, 9], [5, 6, 3], [8, 8, 1]])          # row 3 repeats a column
        toy = M.topk_metrics_device(_cuda(toy_top, dt), [[1], [9, 0], [2], [1, 8, 4]], topk=(1, 3))
        for k, v in zip(g["rank/toy_keys"], g["rank/toy_vals"]):
            assert toy[str(k)] == v, (k, toy[str(k)], v)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_topk_random_per_user_bit_equal_and_dict_equal(seed):
    import torch
    rng = np.random.default_rng(seed)
    n = 3000 + 517 * seed
    top, pos = random_case(rng, n, 4000)
    topk = (1, 5, 10, 20, 50) if seed % 2 else (5, 10, 20, 50)
    want_pu = host_per_user(top, pos, topk)
    host = M.topk_metrics(top, pos, metrics=ALL, topk=topk)
    unrounded = host_means_unrounded(top, pos, topk)
    for k in host:                                  # the restatement is the host's arithmetic
        assert round(unrounded[k], 4) == host[k], k
    for dt in (torch.int32, torch.int64):
        got, pu = M.topk_metrics_device(_cuda(top, dt), pos, metrics=ALL, topk=topk, return_per_user=True)
        pu = pu.cpu().numpy()
        assert pu.shape == want_pu.shape
        assert np.array_equal(pu, want_pu), np.argwhere(pu != want_pu)[:5]
        # numpy averages ndcg / map in fp32, the device every metric in fp64: a rounded value may differ only where the
        # unrounded host value lies within 1e-6 of a rounding boundary (and then by one step of the last digit)
        exempt = {k for k in host if near_rounding_boundary(unrounded[k])}
        assert set(got) == set(host)
        assert {k: v for k, v in got.items() if k not in exempt} == {k: v for k, v in host.items() if k not in exempt}
        assert all(abs(got[k] - host[k]) <= 1.0001e-4 for k in exempt), {k: (got[k], host[k]) for k in exempt}


@pytest.mark.gpu
def test_topk_large_means_are_fp64_means_of_per_user_values():
    import torch
    rng = np.random.default_rng(7)
    n, I, K = 200_000, 100_000, 50
    top = torch.randint(0, I, (n, K), generator=torch.Generator().manual_seed(3)).to(torch.int32)
    lens = rng.integers(1, 30, size=n)
    ptr = np.concatenate([[0], np.cumsum(lens)])
    idx = rng.integers(0, I, size=int(ptr[-1]))
    top_np = top.numpy()
    for r in range(0, n, 3):                          # plant hits in a third of the rows
        top_np[r, r % K] = idx[ptr[r]]
    sets = M.ItemSets.from_csr(ptr, idx, "cuda")
    topk = (5, 10, 20, 50)
    sums, pu = M.topk_metrics_sums(top.cuda(), sets, topk, per_user=True)
    sums, pu = sums.cpu().numpy(), pu.cpu().numpy()
    mean_dev = sums[:-1].reshape(5, 4) / n
    mean_ref = pu.mean(axis=0)
    assert np.abs(mean_dev - mean_ref).max() <= 1e-12
    assert sums[-1] == lens.sum()
    pos = [idx[ptr[r]:ptr[r + 1]] for r in range(n)]
    assert np.array_equal(pu, host_per_user(top_np, pos, topk))


@pytest.mark.gpu
def test_topk_repeatable_and_graph_capturable():
    import torch
    rng = np.random.default_rng(11)
    top, pos = random_case(rng, 5000, 3000)
    sets = M.ItemSets.from_lists(pos, "cuda")
    t = _cuda(top)
    a, pa = M.topk_metrics_sums(t, sets, per_user=True)
    b, pb = M.topk_metrics_sums(t, sets, per_user=True)
    assert torch.equal(a, b) and torch.equal(pa, pb)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c, _ = M.topk_metrics_sums(t, sets)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(c, a)


@pytest.mark.gpu
def test_topk_invalid_arguments_raise():
    import torch
    from foodrec_b200 import _lib
    rng = np.random.default_rng(5)
    top, pos = random_case(rng, 64, 500, K=50)
    t = _cuda(top)
    with pytest.raises(_lib.FoodRecError):
        M.topk_metrics_device(t, pos, topk=(0, 5))
    with pytest.raises(_lib.FoodRecError):
        M.topk_metrics_device(t, pos, topk=(51,))
    with pytest.raises(_lib.FoodRecError):
        M.topk_metrics_device(t, pos, topk=tuple(range(1, 10)))
    with pytest.raises(_lib.FoodRecError):
        M.topk_metrics_device(torch.zeros((64, 65), dtype=torch.int64, device="cuda"), pos, topk=(5,))
    with pytest.raises(_lib.FoodRecError):
        M.topk_metrics_device(t[:10], pos)                       # row count mismatch
    with pytest.raises(_lib.FoodRecError):
        M.topk_metrics_device(torch.from_numpy(top), pos)        # CPU tensor
    with pytest.raises(ValueError):
        M.topk_metrics_device(t, pos, metrics=("hit",))
    # the C entry point itself: null pointer, K > 64, cutoff outside 1..K
    sets = M.ItemSets.from_lists(pos, "cuda")
    ws, (disc, ideal) = M._device_state(t.device, 50)
    sums = torch.empty(64, dtype=torch.float64, device="cuda")
    cut = np.array([5, 10], dtype=np.int32)
    args = [t.data_ptr(), 1, 64, 50, sets.ptr.data_ptr(), sets.idx.data_ptr(), sets.length.data_ptr(), cut.ctypes.data,
            2, disc.data_ptr(), ideal.data_ptr(), sums.data_ptr(), None, ws.data_ptr(), _lib.stream_ptr()]
    assert _lib.lib.fr_topk_metrics(*args) == 0
    for i, v in ((0, None), (4, None), (3, 65)):
        bad = list(args)
        bad[i] = v
        assert _lib.lib.fr_topk_metrics(*bad) == -1
    bad_cut = np.array([5, 51], dtype=np.int32)
    assert _lib.lib.fr_topk_metrics(*args[:7], bad_cut.ctypes.data, *args[8:]) == -1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ by user (GPU)
def ragged_segments(rng, n, distinct=True):
    n_pos = rng.integers(1, 201, size=n)
    n_neg = rng.integers(0, 2001, size=n)
    n_pos[:5], n_neg[:5] = [1, 3, 1, 10, 2], [0, 5, 12, 4, 17]          # segments shorter than 20
    n_pos[5], n_neg[5] = 40, 5000                                       # longer than the shared-memory stage
    n_pos[6], n_neg[6] = 7, 31000                                       # 30 000+ candidates
    lens = n_pos + n_neg
    ptr = np.concatenate([[0], np.cumsum(lens)])
    segs = []
    for L in lens:
        if distinct:
            segs.append((rng.permutation(int(L)).astype(np.float32) - L / 2) / 64)
        else:
            segs.append(rng.integers(0, 6, size=int(L)).astype(np.float32))
    return np.concatenate(segs).astype(np.float32), ptr, n_pos


def stable_by_user(scores, ptr, n_pos, neg_num, cutoffs):
    """`by_user_metrics` restated with the stable descending order (per-user rows)."""
    rows = []
    for r in range(len(n_pos)):
        pred = scores[ptr[r]:ptr[r + 1]]
        p, L = int(n_pos[r]), len(pred)
        order = np.argsort(pred, kind="stable")[::-1]
        auc = sum(float(np.sum(pred[p:] < pred[i])) for i in range(p)) / (p * neg_num)
        hit = order < p
        rec, nd = [], []
        for c in cutoffs:
            h = hit[:c]
            rec.append(h.sum() / p)
            dcg = sum(1.0 / np.log2(t + 2) for t in np.flatnonzero(h))
            nd.append(dcg / sum(1.0 / np.log2(t + 2) for t in range(min(c, L, p))))
        rows.append([auc] + rec + nd)
    return np.array(rows)


@pytest.mark.gpu
def test_by_user_ragged_matches_host_and_oracle():
    import torch
    from oracle import ranking
    rng = np.random.default_rng(2)
    scores, ptr, n_pos = ragged_segments(rng, 160)
    got = M.by_user_metrics_device(_cuda(scores), ptr, n_pos, neg_num=500)
    host = M.by_user_metrics(scores, ptr, n_pos, neg_num=500)
    orc = ranking.by_user_eval([scores[ptr[r]:ptr[r + 1]] for r in range(len(n_pos))], n_pos.tolist(), neg_num=500)
    assert list(got) == list(host)
    for k in host:
        assert abs(got[k] - host[k]) <= 1e-12, (k, got[k], host[k])
        assert abs(got[k] - orc[k]) <= 1e-12, (k, got[k], orc[k])
    # device ptr / n_pos, other cutoffs, per-user rows against the restatement
    cut = (1, 5, 20, 64)
    got2, pu = M.by_user_metrics_device(_cuda(scores), _cuda(ptr), _cuda(n_pos, torch.int32), neg_num=500,
                                        cutoffs=cut, return_per_user=True)
    want = stable_by_user(scores, ptr, n_pos, 500, cut)
    assert np.abs(pu.cpu().numpy() - want).max() <= 1e-12
    assert abs(got2["AUC"] - got["AUC"]) == 0.0


@pytest.mark.gpu
def test_by_user_ties_follow_the_stable_order():
    rng = np.random.default_rng(9)
    scores, ptr, n_pos = ragged_segments(rng, 60, distinct=False)
    cut = (3, 10, 20)
    got, pu = M.by_user_metrics_device(_cuda(scores), ptr, n_pos, neg_num=100, cutoffs=cut, return_per_user=True)
    want = stable_by_user(scores, ptr, n_pos, 100, cut)
    assert np.abs(pu.cpu().numpy() - want).max() <= 1e-12
    mean = want.mean(axis=0)
    keys = ["AUC"] + [f"Recall@{c}" for c in cut] + [f"NDCG@{c}" for c in cut]
    for i, k in enumerate(keys):
        assert abs(got[k] - mean[i]) <= 1e-12, k


@pytest.mark.gpu
def test_by_user_repeatable_and_invalid_arguments():
    import torch
    from foodrec_b200 import _lib
    rng = np.random.default_rng(4)
    scores, ptr, n_pos = ragged_segments(rng, 40)
    s = _cuda(scores)
    a = M.by_user_metrics_device(s, ptr, n_pos, return_per_user=True)
    b = M.by_user_metrics_device(s, ptr, n_pos, return_per_user=True)
    assert a[0] == b[0] and torch.equal(a[1], b[1])
    with pytest.raises(_lib.FoodRecError):
        M.by_user_metrics_device(torch.from_numpy(scores), ptr, n_pos)             # CPU tensor
    with pytest.raises(_lib.FoodRecError):
        M.by_user_metrics_device(s, ptr, n_pos, cutoffs=(10, 65))
    with pytest.raises(_lib.FoodRecError):
        M.by_user_metrics_device(s, ptr, n_pos, cutoffs=())
    with pytest.raises(_lib.FoodRecError):
        M.by_user_metrics_device(s, ptr, n_pos, neg_num=0)
    with pytest.raises(_lib.FoodRecError):
        M.by_user_metrics_device(s, ptr[:-1], n_pos)
    with pytest.raises(_lib.FoodRecError):
        M.by_user_metrics_device(s.double(), ptr, n_pos)
    cut = np.array([10], dtype=np.int32)
    out = torch.empty(3, dtype=torch.float64, device="cuda")
    ws, _ = M._device_state(s.device)
    assert _lib.lib.fr_by_user_metrics(None, None, None, 4, 10, cut.ctypes.data, 1, out.data_ptr(), None,
                                       ws.data_ptr(), _lib.stream_ptr()) == -1


# ------------------------------------------------------------------------------------------------ model level (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True])
def test_lightgcn_full_sort_device_metrics_equal_host(masked):
    import torch
    from test_gpu_clussl import Cfg
    from test_gpu_models import BASE
    from foodrec_b200 import evaluation as E
    from foodrec_b200.models.lightgcn import LightGCN
    from foodrec_b200.synth import make_dataset
    ds = make_dataset("C1")
    torch.manual_seed(999)
    m = LightGCN(Cfg({**BASE, "n_layers": 2, "reg_weight": 0.1}), ds).to("cuda")
    users = np.arange(ds.n_users)
    pos = [ds.testRatings[u] for u in users]
    hist = E.HistoryCSR(ds.train_coo_matrix, ds.n_users, "cuda") if masked else None
    host, top_h = E.evaluate_full_sort(m, users, pos, hist=hist)
    dev, top_d = E.evaluate_full_sort(m, users, pos, hist=hist, device_metrics=True)
    assert torch.is_tensor(top_d) and top_d.is_cuda
    assert np.array_equal(top_d.cpu().numpy(), top_h)
    assert dev == host, {k: (dev[k], host[k]) for k in host if dev[k] != host[k]}
    sets = M.ItemSets.from_lists(pos, "cuda")
    dev2, _ = E.evaluate_full_sort(m, users, sets, hist=hist, device_metrics=True, metrics=ALL)
    assert dev2 == E.evaluate_full_sort(m, users, pos, hist=hist, metrics=ALL)[0]
    with pytest.raises(ValueError):
        E.evaluate_full_sort(m, users, sets, hist=hist)


@pytest.mark.gpu
def test_schgn_full_sort_device_metrics_equal_host():
    import torch
    from test_gpu_schgn import CFG
    from test_gpu_clussl import Cfg
    from foodrec_b200 import evaluation as E
    from foodrec_b200.models.schgn import SCHGN
    from foodrec_b200.synth import make_dataset
    ds = make_dataset("C1")
    torch.manual_seed(5)
    m = SCHGN(Cfg(CFG), ds)
    with torch.no_grad():
        for p in (m.user_embed, m.item_embed, m.ingre_embed_first, m.health_embed):
            p.mul_(20.0)
    m = m.to("cuda").eval()
    users = list(range(0, 5000, 7))[:512]
    pos = [ds.testRatings[u] for u in users]
    host, top_h = E.evaluate_full_sort(m, users, pos)
    dev, top_d = E.evaluate_full_sort(m, users, pos, device_metrics=True)
    assert top_d.dtype == torch.int64 and top_d.is_cuda
    assert np.array_equal(top_d.cpu().numpy(), top_h)
    assert dev == host, {k: (dev[k], host[k]) for k in host if dev[k] != host[k]}


@pytest.mark.gpu
def test_evaluate_by_user_device_metrics_equal_host(mini_ds):
    import torch
    from test_gpu_models import load
    from foodrec_b200 import evaluation as E
    from foodrec_b200.models.lightgcn import LightGCN
    m, _ = load(LightGCN, "lightgcn_mini.npz", mini_ds, n_layers=2, reg_weight=0.1)
    rng = np.random.default_rng(0)
    users = np.arange(mini_ds.n_users)
    cands, n_pos = [], []
    for u in users:                        # negatives distinct from the positives: no tied scores (see the tie rule)
        p = mini_ds.testRatings[u]
        cands.append(np.concatenate([p, rng.choice(np.setdiff1d(np.arange(mini_ds.n_items), p), size=100,
                                                   replace=False)]))
        n_pos.append(len(p))
    ptr = np.concatenate([[0], np.cumsum([len(c) for c in cands])])
    host, s_h = E.evaluate_by_user(m, users, ptr, np.concatenate(cands), n_pos, neg_num=100)
    dev, s_d = E.evaluate_by_user(m, users, ptr, np.concatenate(cands), n_pos, neg_num=100, device_metrics=True)
    assert torch.is_tensor(s_d) and s_d.is_cuda
    assert np.array_equal(s_d.cpu().numpy(), s_h)
    assert list(dev) == list(host)
    for k in host:
        assert abs(dev[k] - host[k]) <= 1e-12, (k, dev[k], host[k])


# ------------------------------------------------------------------------------------------------ host (CPU)
def test_item_sets_from_lists_and_csr():
    s = M.ItemSets.from_lists([[3, 1, 3], [7], np.array([9, 2, 1])], "cpu")
    assert s.n == 3
    assert s.ptr_host.tolist() == [0, 2, 3, 6]
    assert s.idx_host.tolist() == [1, 3, 7, 1, 2, 9] and s.idx_host.dtype == np.int32
    assert s.length_host.tolist() == [3, 1, 3] and s.length_host.dtype == np.int32
    assert s.ptr.tolist() == [0, 2, 3, 6] and s.idx.tolist() == [1, 3, 7, 1, 2, 9] and s.length.tolist() == [3, 1, 3]
    c = M.ItemSets.from_csr([0, 3, 4], [5, 2, 5, 0], "cpu")
    assert c.ptr_host.tolist() == [0, 2, 3] and c.idx_host.tolist() == [2, 5, 0] and c.length_host.tolist() == [3, 1]
    c2 = M.ItemSets.from_csr([0, 3, 4], [5, 2, 5, 0], "cpu", length=[2, 1])
    assert c2.length_host.tolist() == [2, 1]
    rng = np.random.default_rng(0)
    pos = [rng.integers(0, 50, size=int(rng.integers(1, 20))).tolist() for _ in range(300)]
    s = M.ItemSets.from_lists(pos, "cpu")
    for r, p in enumerate(pos):
        assert s.idx_host[s.ptr_host[r]:s.ptr_host[r + 1]].tolist() == sorted(set(p))
        assert s.length_host[r] == len(p)


def test_item_sets_reject_empty_rows_and_bad_input():
    with pytest.raises(ValueError, match="row 1 has no items"):
        M.ItemSets.from_lists([[1], [], [2]], "cpu")
    with pytest.raises(ValueError):
        M.ItemSets.from_csr([0, 1, 1], [4], "cpu")
    with pytest.raises(ValueError):
        M.ItemSets.from_csr([0, 2, 1], [4, 5], "cpu")
    with pytest.raises(ValueError):
        M.ItemSets.from_csr([0, 1], [-3], "cpu")
    with pytest.raises(ValueError):
        M.ItemSets.from_csr([0, 1], [3], "cpu", length=[0])


def test_ndcg_tables_are_the_host_expression():
    K = 50
    ranks = np.arange(1, K + 1)
    disc = (1.0 / np.log2(ranks.astype(np.float32) + 1)).astype(np.float32)
    d, i = M._ndcg_tables(K)
    assert d.dtype == np.float32 and i.dtype == np.float32
    assert np.array_equal(d, disc) and np.array_equal(i, np.cumsum(disc))


def test_per_user_restatement_reproduces_host_metrics():
    rng = np.random.default_rng(3)
    for n in (400, 1000):
        top, pos = random_case(rng, n, 600)
        host = M.topk_metrics(top, pos, metrics=ALL)
        unrounded = host_means_unrounded(top, pos, (5, 10, 20, 50))
        assert {k: round(v, 4) for k, v in unrounded.items()} == host
