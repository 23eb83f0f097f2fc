"""Top-K ranking metrics with the reference's definitions, vectorised.

`topk_metrics` follows `TopKEvaluator.evaluate` (FoodRec/utils/topk_evaluator.py:68-115) and
FoodRec/common/matrics.py:9-102 (Recall, Recall2, NDCG, Precision, MAP; values rounded to 4 d.p.);
the hit matrix replaces the reference's python double loop (`i in m` over lists) by a sorted-key
membership test.  Host numpy, like the reference: it runs once per evaluation on `[n_users, 50]`.

`topk_metrics_device` / `by_user_metrics_device` compute the same metrics on the GPU from device results
(`fr_topk_metrics`, `fr_by_user_metrics`); `ItemSets` holds the held-out items there.
"""
from __future__ import annotations

import numpy as np


def hit_matrix(topk_index: np.ndarray, pos_items) -> np.ndarray:
    topk_index = np.asarray(topk_index, dtype=np.int64)
    n, K = topk_index.shape
    lens = np.fromiter((len(p) for p in pos_items), dtype=np.int64, count=n)
    flat = np.concatenate([np.asarray(p, dtype=np.int64) for p in pos_items]) if lens.sum() else np.zeros(0, np.int64)
    stride = int(max(topk_index.max(initial=0), flat.max(initial=0))) + 2
    keys = np.unique(np.repeat(np.arange(n, dtype=np.int64), lens) * stride + flat)
    q = np.arange(n, dtype=np.int64)[:, None] * stride + topk_index
    pos = np.searchsorted(keys, q)
    pos[pos >= keys.size] = max(keys.size - 1, 0)
    return (keys[pos] == q) & (topk_index >= 0) if keys.size else np.zeros_like(q, dtype=bool)


def _ndcg_tables(K: int):
    """fp32 discounts `1 / log2(rank + 1)` for ranks 1..K and their running sum (the ideal DCG)."""
    ranks = np.arange(1, K + 1)
    disc = (1.0 / np.log2(ranks.astype(np.float32) + 1)).astype(np.float32)
    return disc, np.cumsum(disc)


def topk_metrics(topk_index, pos_items, metrics=("recall", "ndcg", "precision", "map"), topk=(5, 10, 20, 50)):
    hits = hit_matrix(topk_index, pos_items)
    pos_len = np.fromiter((len(p) for p in pos_items), dtype=np.int64, count=hits.shape[0])
    n, K = hits.shape
    ranks = np.arange(1, K + 1)
    cum = np.cumsum(hits, axis=1)
    cut = np.minimum(pos_len, K)
    out = {}
    for m in metrics:
        m = m.lower()
        if m == "recall":
            v = (cum / pos_len.reshape(-1, 1)).mean(axis=0)
        elif m == "recall2":
            v = cum.sum(axis=0) / pos_len.sum()
        elif m == "precision":
            v = (cum / ranks).mean(axis=0)
        elif m == "ndcg":
            disc, ideal = _ndcg_tables(K)
            idcg = ideal[np.minimum(np.arange(K)[None, :], (cut - 1)[:, None])]
            dcg = np.cumsum(np.where(hits, disc, 0), axis=1)
            v = (dcg / idcg).mean(axis=0)
        elif m == "map":
            pre = cum / ranks
            sum_pre = np.cumsum(pre * hits.astype(np.float32), axis=1)
            den = np.minimum(ranks[None, :], cut[:, None])
            v = (sum_pre / den).astype(np.float32).mean(axis=0)
        else:
            raise ValueError(f"There is no user grouped topk metric named {m}!")
        for k in topk:
            out[f"{m}@{k}"] = round(float(v[k - 1]), 4)
    return out


def metrics_by_user(doc_list, rel_list):
    """Recall and NDCG of one ranked list (FoodRec/common/trainer.py:55-69)."""
    rel = set(rel_list)
    gains = [1.0 / np.log2(i + 2) for i, d in enumerate(doc_list) if d in rel]
    idcg = sum(1.0 / np.log2(i + 2) for i in range(min(len(doc_list), len(rel_list))))
    return len(gains) / len(rel_list), float(sum(gains)) / idcg


def by_user_metrics(scores: np.ndarray, ptr: np.ndarray, n_pos: np.ndarray, neg_num: int = 500):
    """The reference's by-user evaluation (FoodRec/common/trainer.py:49-69,231-282) on a flat score
    array: user `r` owns `scores[ptr[r]:ptr[r+1]]`, its first `n_pos[r]` entries are the positives.
    Returns {'AUC', 'Recall@10', 'Recall@20', 'NDCG@10', 'NDCG@20'} averaged over users."""
    disc = 1.0 / np.log2(np.arange(2, 22))
    rows = np.zeros((len(n_pos), 5))
    for r in range(len(n_pos)):
        pred = scores[ptr[r]:ptr[r + 1]]
        p = int(n_pos[r])
        order = np.argsort(pred)[::-1]
        neg = pred[p:]
        rows[r, 0] = sum(float(np.sum(neg < pred[i])) for i in range(p)) / (p * neg_num)
        hit = order[:20] < p
        for j, k in enumerate((10, 20)):
            h = hit[:k]
            rows[r, 1 + j] = h.sum() / p
            rows[r, 3 + j] = (disc[:len(h)] * h).sum() / disc[:min(len(h), p)].sum()
    m = rows.mean(axis=0)
    return {"AUC": m[0], "Recall@10": m[1], "Recall@20": m[2], "NDCG@10": m[3], "NDCG@20": m[4]}


# ------------------------------------------------------------------------------------- device metrics
# The same metrics computed on the GPU (`fr_topk_metrics`, `fr_by_user_metrics`, csrc/eval_metrics.cu) from results that
# are already there: only a few fp64 sums come back.  Per-user values have the host's dtypes and summation order, so
# they are bit-identical to the ones `topk_metrics` averages; the mean over users is taken in fp64 (numpy averages the
# fp32 ndcg / map columns in fp32), so a rounded value can differ from the host's only where the unrounded one lies
# within the host's fp32 averaging error of a rounding boundary.
TOPK_METRICS = ("recall", "recall2", "ndcg", "precision", "map")     # row order of the kernel's sums / per-user values
MAX_CUTOFFS = 8


class ItemSets:
    """Per-user item sets as a CSR on the device: `ptr` int64 `[n+1]`, `idx` int32 (sorted and unique per row) and
    `length` int32 `[n]`, the size of each list AS GIVEN (duplicates included -- `topk_metrics` divides by `len(p)`).
    Built once per split; `ptr_host` / `idx_host` / `length_host` keep the host arrays.  Rows without items are
    rejected: their recall is 0 / 0."""

    def __init__(self, ptr, idx, length, device):
        import torch
        self.ptr_host, self.idx_host, self.length_host = ptr, idx, length
        self.n = len(length)
        self.ptr = torch.from_numpy(ptr).to(device)
        self.idx = torch.from_numpy(idx).to(device)
        self.length = torch.from_numpy(length).to(device)

    @classmethod
    def from_csr(cls, ptr, idx, device, length=None):
        """`idx[ptr[r]:ptr[r+1]]` are the items of row r, in any order, repeats allowed; `length` defaults to the
        row sizes."""
        ptr = np.asarray(ptr, dtype=np.int64)
        idx = np.asarray(idx, dtype=np.int64)
        if ptr.ndim != 1 or ptr.size < 1 or ptr[0] != 0 or (np.diff(ptr) < 0).any() or ptr[-1] != idx.size:
            raise ValueError("ptr must start at 0, be non-decreasing and end at len(idx)")
        n = ptr.size - 1
        counts = np.diff(ptr)
        length = counts if length is None else np.asarray(length, dtype=np.int64)
        if length.shape != (n,):
            raise ValueError(f"length has shape {length.shape}, expected ({n},)")
        if (counts == 0).any() or (length < 1).any():
            raise ValueError(f"row {int(np.flatnonzero((counts == 0) | (length < 1))[0])} has no items")
        if idx.size and (idx.min() < 0 or idx.max() > np.iinfo(np.int32).max):
            raise ValueError("item ids must lie in [0, 2^31)")
        rows = np.repeat(np.arange(n, dtype=np.int64), counts)
        order = np.lexsort((idx, rows))
        rows, idx = rows[order], idx[order]
        keep = np.ones(idx.size, dtype=bool)
        keep[1:] = (rows[1:] != rows[:-1]) | (idx[1:] != idx[:-1])
        out_ptr = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(np.bincount(rows[keep], minlength=n), out=out_ptr[1:])
        return cls(out_ptr, idx[keep].astype(np.int32), length.astype(np.int32), device)

    @classmethod
    def from_lists(cls, pos_items, device):
        lens = np.fromiter((len(p) for p in pos_items), dtype=np.int64, count=len(pos_items))
        flat = np.concatenate([np.asarray(p, dtype=np.int64).reshape(-1) for p in pos_items]) if lens.sum() else \
            np.zeros(0, np.int64)
        ptr = np.zeros(len(lens) + 1, dtype=np.int64)
        np.cumsum(lens, out=ptr[1:])
        return cls.from_csr(ptr, flat, device)


_WS = {}
_NDCG = {}


def _device_state(device, K: int | None = None):
    """Per-device workspace of the metric kernels (zeroed once; the kernels leave its ticket zero) and the fp32
    NDCG tables for K columns."""
    import torch
    from . import _lib
    ws = _WS.get(device)
    if ws is None:
        ws = torch.zeros(int(_lib.lib.fr_eval_metrics_ws_bytes()) // 8 + 2, dtype=torch.float64, device=device)
        _WS[device] = ws
    if K is None:
        return ws, None
    tabs = _NDCG.get((device, K))
    if tabs is None:
        disc, ideal = _ndcg_tables(K)
        tabs = (torch.from_numpy(disc).to(device), torch.from_numpy(ideal).to(device))
        _NDCG[(device, K)] = tabs
    return ws, tabs


def _cutoffs(cutoffs, hi: int):
    from . import _lib
    c = np.asarray([int(k) for k in cutoffs], dtype=np.int32)
    if not 1 <= c.size <= MAX_CUTOFFS or (c < 1).any() or (c > hi).any():
        raise _lib.FoodRecError(f"cutoffs {list(cutoffs)}: 1..{MAX_CUTOFFS} values in [1, {hi}] expected")
    return c


def topk_metrics_sums(top, pos: ItemSets, topk=(5, 10, 20, 50), per_user: bool = False):
    """One `fr_topk_metrics` launch: device fp64 sums `[5, len(topk)]` (rows in `TOPK_METRICS` order) and the sum of
    the list lengths, plus optionally the per-user values `[n, 5, len(topk)]` fp64 (recall2: the hit count).  Nothing
    is synchronised."""
    import torch
    from . import _lib
    if not torch.is_tensor(top) or top.device.type != "cuda":
        raise _lib.FoodRecError("topk_metrics_device needs the top-K indices as a CUDA tensor (no CPU path)")
    if top.dim() != 2 or top.dtype not in (torch.int32, torch.int64):
        raise _lib.FoodRecError(f"top must be a 2-d int32 / int64 tensor, got {tuple(top.shape)} {top.dtype}")
    n, K = top.shape
    if pos.n != n:
        raise _lib.FoodRecError(f"{n} rows of top-K indices but {pos.n} item sets")
    if pos.ptr.device != top.device:
        raise _lib.FoodRecError(f"item sets live on {pos.ptr.device}, the indices on {top.device}")
    cut = _cutoffs(topk, K)
    top = top.contiguous()
    ws, (disc, ideal) = _device_state(top.device, K)
    sums = torch.empty(len(TOPK_METRICS) * cut.size + 1, dtype=torch.float64, device=top.device)
    pu = torch.empty((n, len(TOPK_METRICS), cut.size), dtype=torch.float64, device=top.device) if per_user else None
    _lib.check(_lib.lib.fr_topk_metrics(
        top.data_ptr(), int(top.dtype == torch.int64), n, K, pos.ptr.data_ptr(), pos.idx.data_ptr(),
        pos.length.data_ptr(), cut.ctypes.data, cut.size, disc.data_ptr(), ideal.data_ptr(), sums.data_ptr(),
        _lib.ptr(pu), ws.data_ptr(), _lib.stream_ptr()), "fr_topk_metrics")
    return sums, pu


def topk_metrics_device(top, pos, metrics=("recall", "ndcg", "precision", "map"), topk=(5, 10, 20, 50),
                        return_per_user: bool = False):
    """`topk_metrics` on the GPU: `top` is the `[n, K]` int32 / int64 CUDA tensor of ranked items (never copied to the
    host), `pos` an `ItemSets` on the same device or the lists of held-out items.  Returns the same dict (same keys,
    values rounded to 4 d.p.); with `return_per_user` also the `[n, 5, len(topk)]` fp64 per-user values."""
    names = [m.lower() for m in metrics]
    for m in names:
        if m not in TOPK_METRICS:
            raise ValueError(f"There is no user grouped topk metric named {m}!")
    if not isinstance(pos, ItemSets):
        pos = ItemSets.from_lists(pos, top.device)
    sums, pu = topk_metrics_sums(top, pos, topk, per_user=return_per_user)
    s = sums.cpu().numpy()                   # the only device -> host copy: 5 x len(topk) + 1 doubles
    nc = len(topk)
    v = s[:-1].reshape(len(TOPK_METRICS), nc)
    out = {}
    for m in names:
        row = TOPK_METRICS.index(m)
        mean = v[row] / s[-1] if m == "recall2" else v[row] / pos.n
        for i, k in enumerate(topk):
            out[f"{m}@{k}"] = round(float(mean[i]), 4)
    return (out, pu) if return_per_user else out


def by_user_metrics_device(scores, ptr, n_pos, neg_num: int = 500, cutoffs=(10, 20), return_per_user: bool = False):
    """`by_user_metrics` on the GPU (`fr_by_user_metrics`): `scores` is the flat fp32 CUDA tensor of candidate scores,
    user r owns `scores[ptr[r]:ptr[r+1]]` with its `n_pos[r]` positives first (`ptr`, `n_pos`: host arrays or device
    tensors).  Returns {'AUC', 'Recall@c', ..., 'NDCG@c', ...} averaged over users; with `return_per_user` also the
    `[n, 1 + 2 len(cutoffs)]` fp64 per-user rows.

    Ties: a positive's rank is its position in `np.argsort(pred, kind="stable")[::-1]`; the host's default argsort
    agrees wherever the positive's score ties no other candidate's."""
    import torch
    from . import _lib
    if not torch.is_tensor(scores) or scores.device.type != "cuda":
        raise _lib.FoodRecError("by_user_metrics_device needs the scores as a CUDA tensor (no CPU path)")
    if scores.dtype != torch.float32:
        raise _lib.FoodRecError(f"scores must be float32, got {scores.dtype}")
    dev = scores.device
    ptr = torch.as_tensor(ptr).to(device=dev, dtype=torch.int64).contiguous()
    n_pos = torch.as_tensor(n_pos).to(device=dev, dtype=torch.int32).contiguous()
    n = n_pos.numel()
    if ptr.numel() != n + 1:
        raise _lib.FoodRecError(f"ptr has {ptr.numel()} entries for {n} users")
    if int(neg_num) < 1:
        raise _lib.FoodRecError(f"neg_num={neg_num}")
    cut = _cutoffs(cutoffs, 64)
    scores = scores.contiguous()
    ws, _ = _device_state(dev)
    n_out = 1 + 2 * cut.size
    sums = torch.empty(n_out, dtype=torch.float64, device=dev)
    pu = torch.empty((n, n_out), dtype=torch.float64, device=dev) if return_per_user else None
    _lib.check(_lib.lib.fr_by_user_metrics(
        scores.data_ptr(), ptr.data_ptr(), n_pos.data_ptr(), n, int(neg_num), cut.ctypes.data, cut.size,
        sums.data_ptr(), _lib.ptr(pu), ws.data_ptr(), _lib.stream_ptr()), "fr_by_user_metrics")
    m = sums.cpu().numpy() / n
    out = {"AUC": float(m[0])}
    out.update({f"Recall@{c}": float(m[1 + i]) for i, c in enumerate(cut.tolist())})
    out.update({f"NDCG@{c}": float(m[1 + cut.size + i]) for i, c in enumerate(cut.tolist())})
    return (out, pu) if return_per_user else out
