"""Ranking on the tensor cores: fused score + (mask) + top-K for full-sort evaluation, cosine kNN item
graphs and centroid assignment.

Replaces `Trainer.evaluate`'s per-user `full_sort_predict` + `torch.topk`
(FoodRec/common/trainer.py:476-503), the LATTICE kNN utilities (FoodRec/utils/utils.py:118-183) and
the centroid-assignment loop of dataset_process/*_kmeans.ipynb.  Pipeline per call:
fp32 -> bf16 operands, `fr_gemm_topk_bf16` keeps `kc = k + slack` candidates per row from the bf16
tensor-core scores, `fr_rescore_topk_f32` re-scores those exactly in fp32, keeps the best k and CERTIFIES
each row: a dropped column's fp32 score is at most (smallest kept bf16 score) + |u' - u| max|i'| + |u| max|i' - i|
(u', i' the bf16-rounded rows), and if that is below the k-th re-scored value the row's result is the fp32 top-k.  Rows that fail are re-ranked with 64
candidates and, failing again, scored against every column in fp32 (`fr_exact_topk_f32`).  The result is the
fp32 `topk` (ties to the lower column) for every row -- a guarantee, not a heuristic.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

_L = _lib.lib
MAX_K = 64
# bench.py sets this to a list to collect (start_event, end_event, flops) per fused GEMM+top-K launch
PROFILE = None


class HistoryCSR:
    """Per-user sorted training items on the device (the optional full-sort mask, SURVEY.md D1)."""

    def __init__(self, train_coo, n_users: int, device):
        u = np.asarray(train_coo.row, dtype=np.int64)
        i = np.asarray(train_coo.col, dtype=np.int64)
        order = np.lexsort((i, u))
        ptr = np.zeros(n_users + 1, dtype=np.int64)
        np.cumsum(np.bincount(u, minlength=n_users), out=ptr[1:])
        self.ptr_host, self.idx_host = ptr, i[order].astype(np.int32)
        self.ptr = torch.from_numpy(ptr).to(device)
        self.idx = torch.from_numpy(self.idx_host).to(device)

    def mask_scores_(self, scores: torch.Tensor, users: torch.Tensor) -> torch.Tensor:
        """`scores[r, history(users[r])] = -inf` on a dense `[len(users), n_items]` block (for rankers
        whose scores are not a GEMM, e.g. SCHGN's pair scorer)."""
        users = users.to(self.ptr.device).long()
        lo, hi = self.ptr[users], self.ptr[users + 1]
        cnt = hi - lo
        rows = torch.repeat_interleave(torch.arange(users.numel(), device=cnt.device), cnt)
        off = torch.arange(rows.numel(), device=cnt.device) - torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
        scores[rows, self.idx[torch.repeat_interleave(lo, cnt) + off].long()] = float("-inf")
        return scores


_WS = {}


def _workspace(device, nbytes: int) -> torch.Tensor:
    """Scratch for the per-(row, quarter) candidate lists of the ranking kernel (reused across calls)."""
    ws = _WS.get(device)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        _WS[device] = ws
    return ws


def to_bf16(x: torch.Tensor, l2_normalise: bool = False) -> torch.Tensor:
    x = x.detach()
    if x.dtype != torch.float32 or not x.is_contiguous():
        x = x.float().contiguous()
    if x.device.type != "cuda":
        raise _lib.FoodRecError("to_bf16 needs a CUDA tensor (no CPU path)")
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    _lib.check(_L.fr_f32_to_bf16(x.data_ptr(), y.data_ptr(), x.shape[0], x.shape[1], int(l2_normalise),
                                 _lib.stream_ptr()), "fr_f32_to_bf16")
    return y


def _bf16_candidates(Ab, Bb, M, N, K, kc, scale, bias, row_ids, hist):
    """One launch of the fused tensor-core score + (mask) + top-`kc` kernel -> (bf16-pass scores, columns)."""
    dev = Ab.device
    cand_v = torch.empty((M, kc), dtype=torch.float32, device=dev)
    cand_i = torch.empty((M, kc), dtype=torch.int32, device=dev)
    ws = _workspace(dev, int(_L.fr_gemm_topk_ws_bytes(M)))
    prof = PROFILE
    if prof is not None:
        ev0 = torch.cuda.Event(enable_timing=True)
        ev0.record()
    _lib.check(_L.fr_gemm_topk_bf16(
        Ab.data_ptr(), M, Bb.data_ptr(), N, K, float(scale), _lib.ptr(bias),
        _lib.ptr(row_ids) if hist is not None else None, hist.ptr.data_ptr() if hist is not None else None,
        hist.idx.data_ptr() if hist is not None else None, kc, cand_v.data_ptr(), cand_i.data_ptr(),
        ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "fr_gemm_topk_bf16")
    if prof is not None:
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record()
        prof.append((ev0, ev1, 2.0 * M * N * K))
    return cand_v, cand_i


def _rescore(A, a_rows, B, K, scale, bias, metric, cand_v, cand_i, k, index_dtype, bmax):
    """fp32 re-score of the candidates -> (values, indices, certificate [M] uint8)."""
    M, kc = cand_i.shape
    dev = A.device
    out_v = torch.empty((M, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((M, k), dtype=index_dtype, device=dev)
    cert = torch.empty(M, dtype=torch.uint8, device=dev)
    _lib.check(_L.fr_rescore_topk_f32(A.data_ptr(), _lib.ptr(a_rows), B.data_ptr(), K, float(scale), _lib.ptr(bias), int(metric),
                                      cand_i.data_ptr(), cand_v.data_ptr(), kc, M, k, out_v.data_ptr(), out_i.data_ptr(),
                                      int(index_dtype == torch.int64), bmax.data_ptr(), cert.data_ptr(),
                                      _lib.stream_ptr()), "fr_rescore_topk_f32")
    return out_v, out_i, cert


def max_row_norm(B: torch.Tensor) -> torch.Tensor:
    """`[max_n |bf16(B_n)|, max_n |bf16(B_n) - B_n|]` as two device floats (the column factors of the
    certificate's rounding-error bound)."""
    out = torch.empty(2, dtype=torch.float32, device=B.device)
    _lib.check(_L.fr_max_row_norm(B.data_ptr(), B.shape[0], B.shape[1], out.data_ptr(), _lib.stream_ptr()), "fr_max_row_norm")
    return out


def exact_topk_rows(A, rows, B, k, *, scale=1.0, bias=None, metric=0, row_ids=None, hist=None, max_ws_bytes=1 << 30,
                    thr=None):
    """fp32 top-k of rows `A[rows]` against every row of B on the CUDA cores: the path for rows whose certificate
    failed.  Returns (values `[len(rows), k]`, int64 indices).

    `thr` (`[len(rows)]`, optional): a lower bound of each row's k-th best fp32 score.  With it the scoring pass keeps
    only the columns that reach the bound (`fr_exact_topk_thr_f32`: per-row lists instead of a dense `[rows, N]` score
    block and five passes over it); rows whose list overflows (massive ties) are redone densely (`fr_exact_topk_f32`)."""
    dev, N, K = A.device, B.shape[0], B.shape[1]
    rows = rows.to(torch.int64).contiguous()
    n = rows.numel()
    out_v = torch.empty((n, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((n, k), dtype=torch.int64, device=dev)
    if thr is not None and n:
        hr = (row_ids[rows] if row_ids is not None else rows).to(torch.int64).contiguous() if hist is not None else None
        ws = torch.empty(int(_L.fr_exact_topk_thr_ws_bytes(n)), dtype=torch.uint8, device=dev)
        over = torch.empty(1, dtype=torch.int32, device=dev)
        thr = thr.to(torch.float32).contiguous()
        _lib.check(_L.fr_exact_topk_thr_f32(
            A.data_ptr(), rows.data_ptr(), n, B.data_ptr(), N, K, float(scale), _lib.ptr(bias), int(metric),
            _lib.ptr(hr), hist.ptr.data_ptr() if hist is not None else None,
            hist.idx.data_ptr() if hist is not None else None, k, thr.data_ptr(), ws.data_ptr(), out_v.data_ptr(),
            out_i.data_ptr(), over.data_ptr(), _lib.stream_ptr()), "fr_exact_topk_thr_f32")
        if int(over.item()) == 0:
            return out_v, out_i
        # some list overflowed: those rows' outputs were left untouched -- redo every row densely (rare: massive ties)
    chunk = max(1, min(n, max_ws_bytes // (4 * N)))
    ws = torch.empty(chunk * N, dtype=torch.float32, device=dev)
    hrows = None
    if hist is not None:
        hrows = (row_ids[rows] if row_ids is not None else rows).to(torch.int64).contiguous()
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        _lib.check(_L.fr_exact_topk_f32(
            A.data_ptr(), rows[s:].data_ptr(), m, B.data_ptr(), N, K, float(scale), _lib.ptr(bias), int(metric),
            hrows[s:].data_ptr() if hrows is not None else None, hist.ptr.data_ptr() if hist is not None else None,
            hist.idx.data_ptr() if hist is not None else None, k, ws.data_ptr(), out_v[s:].data_ptr(), out_i[s:].data_ptr(),
            _lib.stream_ptr()), "fr_exact_topk_f32")
    return out_v, out_i


def gemm_topk(A: torch.Tensor, B: torch.Tensor, k: int, *, scale: float = 1.0, bias: torch.Tensor | None = None,
              row_ids: torch.Tensor | None = None, hist: HistoryCSR | None = None, slack: int | None = None,
              exact: bool = True, metric: int = 0, A_bf16: torch.Tensor | None = None,
              B_bf16: torch.Tensor | None = None, index_dtype=torch.int64, b_max_norm: torch.Tensor | None = None,
              stats: dict | None = None):
    """Row-wise top-k of `scale * A @ B.T + bias` (A `[M, K]`, B `[N, K]` fp32) -> (values `[M, k]`
    fp32, indices `[M, k]` `index_dtype`), descending.  `hist` + `row_ids` exclude each row's history columns.

    `exact=True` (default) returns the fp32 top-k, ties to the lower column: candidates from the bf16
    tensor-core pass are re-scored in fp32, every row is checked against the rounding-error certificate
    (`fr_rescore_topk_f32`), rows that fail are re-ranked with the widest candidate set and, if they fail
    again, scored exactly against every column (`fr_exact_topk_f32`).  `stats` (a dict) receives how many rows
    took each path.  `exact=False` returns the bf16-scored top-k without re-score.

    `slack` = extra candidates the tensor-core pass keeps per row (`kc = k + slack`).  Every extra candidate costs
    ~0.7 % of the kernel time (measured on the 1 M x 500 k shape: kc = 32 / 40 / 48 / 64 -> 14.2 / 15.0 / 15.8 / 17.7 ms
    per 125 000 rows) while the rows a narrow `kc` leaves uncertified cost a fixed 3.5 - 5 ms of fallback passes
    (`scripts/microbench_c4_slack.py`); with kc = k + 20 no row of that shape needs a fallback.  Default: 20 when the
    table is wide (N >= 131 072) and the launch short enough for the fixed cost to matter (< ~45 ms of tensor-core
    time), else 12."""
    if k < 1 or k > MAX_K:
        raise _lib.FoodRecError(f"k={k} outside [1, {MAX_K}]")
    if index_dtype not in (torch.int64, torch.int32):
        raise _lib.FoodRecError("index_dtype must be torch.int64 or torch.int32")
    M, K = A.shape
    N = B.shape[0]
    if K % 8 != 0:
        raise _lib.FoodRecError(f"inner dimension {K} must be a multiple of 8")
    dev = A.device
    A = A.detach().float().contiguous()
    B = B.detach().float().contiguous()
    Ab = A_bf16 if A_bf16 is not None else to_bf16(A)
    Bb = B_bf16 if B_bf16 is not None else to_bf16(B)
    kk = min(k, N)
    if slack is None:
        # (the fallback's fixed cost is a sweep over all N columns: it only outweighs the wider lists when N is large;
        #  on the 45 000-item C2 table kc = 32 / 40 / 64 give 4.17 / 4.37 / 4.17 ms, `scripts/microbench_eval_slack.py`)
        slack = 20 if (N >= 131072 and 2.0 * M * N * K < 45e-3 * 5.5e14) else 12       # ~550 TFLOP/s at K = 64 (DESIGN.md 3.4)
    kc = min(MAX_K, kk + max(int(slack), 0), N) if exact else kk
    if hist is not None:
        if row_ids is None:
            row_ids = torch.arange(M, device=dev)
        row_ids = row_ids.to(torch.int64).contiguous()
    if bias is not None:
        bias = bias.detach().float().contiguous()
    cand_v, cand_i = _bf16_candidates(Ab, Bb, M, N, K, kc, scale, bias, row_ids, hist)
    if not exact:
        return cand_v[:, :kk], cand_i[:, :kk].to(index_dtype)
    bmax = b_max_norm if b_max_norm is not None else max_row_norm(B)
    out_v, out_i, cert = _rescore(A, None, B, K, scale, bias, metric, cand_v, cand_i, kk, index_dtype, bmax)
    n_bad = int((cert == 0).sum().item())       # 4-byte read-back; rows beyond the certificate are rare
    n_wide = n_exact = 0
    if n_bad:
        bad = torch.nonzero(cert == 0).reshape(-1)
        kc2 = min(MAX_K, N)
        # second chance on the tensor cores: the widest candidate set for just these rows -- unless they are too few to
        # fill the tensor-core kernel (one 256-row block sweeps every column alone), where the exact fp32 kernel is faster
        if kc2 > kc and n_bad > 1024:
            n_wide = n_bad
            A_bad = A[bad].contiguous()
            rid_bad = row_ids[bad].contiguous() if hist is not None else None
            cv2, ci2 = _bf16_candidates(to_bf16(A_bad), Bb, n_bad, N, K, kc2, scale, bias, rid_bad, hist)
            v2, i2, cert2 = _rescore(A_bad, None, B, K, scale, bias, metric, cv2, ci2, kk, index_dtype, bmax)
            out_v[bad] = v2
            out_i[bad] = i2
            bad = bad[cert2 == 0]
        n_exact = int(bad.numel())
        if n_exact:
            # every member of the fp32 top-k scores at least the k-th best re-scored value; the margin covers the
            # different fp32 summation orders of the two kernels (K 2^-24 |a| max|b|, doubled)
            margin = max(1e-5, 2.0 * K * 2.0 ** -24)
            vk = out_v[bad, kk - 1]
            thr = vk - margin * (vk.abs() + (A[bad].norm(dim=1) * bmax[0] * abs(float(scale)) if metric == 0 else 0.0))
            v3, i3 = exact_topk_rows(A, bad, B, kk, scale=scale, bias=bias, metric=metric, row_ids=row_ids, hist=hist,
                                     thr=thr)
            out_v[bad] = v3
            out_i[bad] = i3.to(index_dtype)
    if stats is not None:
        stats.update(rows=M, kc=kc, uncertified=n_bad, widened=n_wide, exact_rows=n_exact)
    return out_v, out_i


# ------------------------------------------------------------------------------- full-sort evaluation
def full_sort_scores(user_all: torch.Tensor, item_all: torch.Tensor, users: torch.Tensor) -> torch.Tensor:
    """Dense fp32 `[n_batch_users, n_items]` scores -- only for API compatibility with
    `full_sort_predict`; `full_sort_topk` is the path that never materialises this matrix."""
    return user_all[users.reshape(-1).long()] @ item_all.t()


def full_sort_topk(user_all: torch.Tensor, item_all: torch.Tensor, users: torch.Tensor | None, k: int,
                   hist: HistoryCSR | None = None, **kw):
    """Top-k items for `users` (all users when None).  `hist=None` reproduces the reference (no mask)."""
    from . import ops
    if users is None:
        A, row_ids = user_all, None
    else:
        users = users.reshape(-1).to(torch.int64)
        A, row_ids = ops.gather_rows(user_all.detach(), users), users
    return gemm_topk(A, item_all, k, row_ids=row_ids, hist=hist, **kw)


def evaluate_full_sort(model, eval_users, pos_items, topk=(5, 10, 20, 50), metrics=("recall", "ndcg", "precision", "map"),
                       hist: HistoryCSR | None = None, batch_users: int = 65536, device_metrics: bool = False):
    """`Trainer.evaluate` (FoodRec/common/trainer.py:476-503): rank every eval user against all items and
    score with the reference's metric definitions.  Dot-product models propagate once and rank on the
    tensor cores; a model with its own `full_sort_topk` (SCHGN: fused pair scorer) is asked directly.

    `device_metrics=True` computes the metrics on the GPU (`metrics.topk_metrics_device`): the top-K indices stay
    there and are returned as a device tensor; `pos_items` may then be a `metrics.ItemSets` built once per split."""
    from . import metrics as M
    if not device_metrics and isinstance(pos_items, M.ItemSets):
        raise ValueError("an ItemSets is the device form of pos_items: pass device_metrics=True, or the lists")
    model.eval()
    with torch.no_grad():
        if hasattr(model, "full_sort_topk"):
            dev = next(model.parameters()).device
            users = torch.as_tensor(np.asarray(eval_users), device=dev)
            top = model.full_sort_topk(users, max(topk), hist=hist)[1]
            if device_metrics:
                return M.topk_metrics_device(top, pos_items, metrics=metrics, topk=topk), top
            top = top.cpu().numpy()
            return M.topk_metrics(top, pos_items, metrics=metrics, topk=topk), top
        user_all, item_all = model._tables()
        users = torch.as_tensor(np.asarray(eval_users), device=user_all.device)
        item_bf16, bmax = to_bf16(item_all), max_row_norm(item_all.detach().float().contiguous())
        tops = []
        for s in range(0, users.numel(), batch_users):     # int32 indices: half the device->host bytes of int64
            _, idx = full_sort_topk(user_all, item_all, users[s:s + batch_users], max(topk), hist=hist,
                                    B_bf16=item_bf16, b_max_norm=bmax, index_dtype=torch.int32)
            tops.append(idx)
        top = torch.cat(tops, 0)
        if device_metrics:
            return M.topk_metrics_device(top, pos_items, metrics=metrics, topk=topk), top
        top = top.cpu().numpy().astype(np.int64)
    return M.topk_metrics(top, pos_items, metrics=metrics, topk=topk), top


# ------------------------------------------------------------------------------------- kNN / centroids
def knn_topk(features: torch.Tensor, k: int, **kw):
    """Cosine-similarity kNN: `torch.topk(build_sim(x), k)` (FoodRec/utils/utils.py:119,132-135),
    self included.  Returns (`knn_val`, `knn_ind`) `[N, k]`."""
    x = features.detach().float()
    xn = (x / torch.norm(x, p=2, dim=-1, keepdim=True)).contiguous()
    return gemm_topk(xn, xn, k, **kw)


def knn_normalized_graph(features: torch.Tensor, k: int, norm_type: str = "sym"):
    """Sparse branch of `build_knn_normalized_graph` (FoodRec/utils/utils.py:170-180): COO
    `(edge_index [2, N k], edge_weight [N k])` with `get_sparse_laplacian` normalisation."""
    val, ind = knn_topk(features, k)
    n = features.shape[0]
    row = torch.arange(n, device=val.device).repeat_interleave(k)
    col = ind.reshape(-1)
    w = val.reshape(-1)
    deg = torch.zeros(n, dtype=w.dtype, device=w.device).index_add_(0, row, w)
    if norm_type == "sym":
        dis = deg.pow(-0.5)
        dis.masked_fill_(dis == float("inf"), 0)
        w = dis[row] * w * dis[col]
    elif norm_type == "rw":
        di = 1.0 / deg
        di.masked_fill_(di == float("inf"), 0)
        w = di[row] * w
    return torch.stack([row, col]), w


def centroid_topk(features: torch.Tensor, centres: torch.Tensor, k: int = 6, **kw):
    """k nearest (Euclidean) centres per item, nearest first: the notebook's
    `argsort([norm(x - c) for c in centres])[:10][:6]`.  Candidates from the bf16 GEMM with the
    `-|c|^2/2` column bias, final order from exact fp32 squared distances."""
    c = centres.detach().float().contiguous()
    bias = -0.5 * (c * c).sum(1)
    _, idx = gemm_topk(features, c, k, bias=bias, metric=1, **kw)
    return idx


# ------------------------------------------------------------------------------ by-user evaluation
def schgn_pair_scores(*, user_final, user_key, user_comp, user_hidden, W_item, W_prod, w_out, h_ingre, h_comp, codes,
                      nums, ingre_key, ingre_final, ingre_comp, img_key, comps, comp_keys, topk: int | None = None,
                      user_ids: torch.Tensor | None = None, hist: HistoryCSR | None = None):
    """SCHGN scores `[nu, n_items]` of `nu` users against every item from the user-independent tables
    (`models.schgn.SCHGN._item_side`): `fr_schgn_attend` + `fr_schgn_score`, FoodRec/models/schgn.py:159-206,
    233-268, 318-345.  Users are processed in blocks so the `[nu, I, 64]` attended-row scratch stays
    under ~1 GB.

    `topk=k`: returns `(values [nu, k], int64 indices [nu, k])` instead, with the selection fused into the scorer
    (`fr_schgn_score_topk`) -- the score block is never written; `hist` + `user_ids` mask each user's training items."""
    dev = user_final.device
    if dev.type != "cuda":
        raise _lib.FoodRecError("schgn_pair_scores needs CUDA tensors (no CPU path)")
    f32 = [user_final, user_key, user_comp, user_hidden, W_item, W_prod, w_out, h_ingre, h_comp, ingre_key,
           ingre_final, ingre_comp, img_key, comps, comp_keys]
    user_final, user_key, user_comp, user_hidden, W_item, W_prod, w_out, h_ingre, h_comp, ingre_key, ingre_final, \
        ingre_comp, img_key, comps, comp_keys = [t.detach().float().contiguous() for t in f32]
    nu, d = user_final.shape
    n_items, slots = codes.shape
    if codes.dtype != torch.int32 or nums.dtype != torch.int32:
        raise _lib.FoodRecError("ingredient codes / counts must be int32")
    if topk is not None:
        if not 1 <= topk <= MAX_K:
            raise _lib.FoodRecError(f"k={topk} outside [1, {MAX_K}]")
        out_v = torch.empty(nu, topk, dtype=torch.float32, device=dev)
        out_i = torch.empty(nu, topk, dtype=torch.int64, device=dev)
        if hist is not None:
            if user_ids is None:
                raise _lib.FoodRecError("a history mask needs the users' ids")
            user_ids = user_ids.to(device=dev, dtype=torch.int64).contiguous()
    else:
        scores = torch.empty(nu, n_items, dtype=torch.float32, device=dev)
    block = max(16, min(256, (1 << 30) // max(1, n_items * d * 4) // 16 * 16))
    if topk is not None:
        ws = torch.empty(int(_L.fr_schgn_score_topk_ws_bytes(min(block, nu), n_items, topk)), dtype=torch.uint8, device=dev)
    att = torch.empty(min(block, nu), n_items, d, dtype=torch.float32, device=dev)
    logits = torch.empty(min(block, nu), 4, n_items, dtype=torch.float32, device=dev)
    st = _lib.stream_ptr()
    for s in range(0, nu, block):
        n = min(block, nu - s)
        _lib.check(_L.fr_schgn_attend(
            user_key[s:].data_ptr(), user_comp[s:].data_ptr(), n, codes.data_ptr(), slots, nums.data_ptr(), n_items,
            ingre_key.data_ptr(), ingre_final.data_ptr(), ingre_comp.data_ptr(), img_key.data_ptr(),
            comp_keys.data_ptr(), h_ingre.data_ptr(), h_comp.data_ptr(), d, att.data_ptr(),
            logits.data_ptr(), st), "fr_schgn_attend")
        if topk is None:
            _lib.check(_L.fr_schgn_score(
                user_final[s:].data_ptr(), user_hidden[s:].data_ptr(), n, W_item.data_ptr(), W_prod.data_ptr(),
                w_out.data_ptr(), comps.data_ptr(), att.data_ptr(), logits.data_ptr(), n_items, d,
                scores[s:].data_ptr(), st), "fr_schgn_score")
        else:
            _lib.check(_L.fr_schgn_score_topk(
                user_final[s:].data_ptr(), user_hidden[s:].data_ptr(), n, W_item.data_ptr(), W_prod.data_ptr(),
                w_out.data_ptr(), comps.data_ptr(), att.data_ptr(), logits.data_ptr(), n_items, d,
                user_ids[s:].data_ptr() if hist is not None else None, hist.ptr.data_ptr() if hist is not None else None,
                hist.idx.data_ptr() if hist is not None else None, topk, ws.data_ptr(), out_v[s:].data_ptr(),
                out_i[s:].data_ptr(), st), "fr_schgn_score_topk")
    return scores if topk is None else (out_v, out_i)


def schgn_by_user_scores(cand_ptr, cand_items, *, user_final, user_key, user_comp, user_hidden, W_item, W_prod, w_out,
                         h_ingre, h_comp, codes, nums, ingre_key, ingre_final, ingre_comp, img_key, comps, comp_keys,
                         block_pairs: int = 1 << 22):
    """SCHGN scores of per-user candidate lists: user r (row r of the user tables) against `cand_items[cand_ptr[r]:
    cand_ptr[r+1]]`, each list scored as the reference scores it in one `inference_by_user` batch -- the component
    softmax groups the list's own logits (`.view(b, -1)` with b = the list length, FoodRec/models/schgn.py:198).
    `fr_schgn_attend_pairs` + `fr_schgn_score_pairs` over the tables of `models.schgn.SCHGN._item_side`, users in blocks
    of at most `block_pairs` pairs (one longer list forms a block alone) so the `[pairs, 64]` attended-row scratch stays
    under ~1 GB.  `cand_ptr` [n+1] is a host array from 0 to len(cand_items); returns the flat fp32 scores [len(cand_items)]
    in list order.  An item outside [0, n_items) raises `FoodRecError` (checked on the device: one 4-byte read-back)."""
    dev = user_final.device
    if dev.type != "cuda":
        raise _lib.FoodRecError("schgn_by_user_scores needs CUDA tensors (no CPU path)")
    f32 = [user_final, user_key, user_comp, user_hidden, W_item, W_prod, w_out, h_ingre, h_comp, ingre_key,
           ingre_final, ingre_comp, img_key, comps, comp_keys]
    user_final, user_key, user_comp, user_hidden, W_item, W_prod, w_out, h_ingre, h_comp, ingre_key, ingre_final, \
        ingre_comp, img_key, comps, comp_keys = [t.detach().float().contiguous() for t in f32]
    nu, d = user_final.shape
    n_items, slots = codes.shape
    if codes.dtype != torch.int32 or nums.dtype != torch.int32:
        raise _lib.FoodRecError("ingredient codes / counts must be int32")
    ptr = np.asarray(cand_ptr, dtype=np.int64).reshape(-1)
    items = torch.as_tensor(cand_items).reshape(-1).to(dev)
    if ptr.shape[0] != nu + 1:
        raise _lib.FoodRecError(f"cand_ptr has {ptr.shape[0]} entries for {nu} users")
    if nu == 0:
        return torch.empty(0, dtype=torch.float32, device=dev)
    if ptr[0] != 0 or ptr[-1] != items.numel():
        raise _lib.FoodRecError(f"cand_ptr runs from {ptr[0]} to {ptr[-1]}, cand_items holds {items.numel()} items")
    if (np.diff(ptr) < 1).any():
        raise _lib.FoodRecError("every candidate list must be non-empty (cand_ptr strictly increasing)")
    if items.dtype != torch.int32:       # an id beyond int32 must not wrap into range: map it to -1, which the kernel rejects
        items = torch.where((items >= 0) & (items < n_items), items, -1)
    items = items.to(torch.int32).contiguous()
    blocks, s = [], 0
    while s < nu:
        e = max(s + 1, int(np.searchsorted(ptr, ptr[s] + block_pairs, side="right")) - 1)
        blocks.append((s, min(e, nu)))
        s = min(e, nu)
    most = max(int(ptr[e] - ptr[s]) for s, e in blocks)
    most_users = max(e - s for s, e in blocks)
    ws = torch.empty(int(_L.fr_schgn_attend_pairs_ws_bytes(most_users, most, n_items)), dtype=torch.uint8, device=dev)
    att = torch.empty(most, d, dtype=torch.float32, device=dev)
    logits = torch.empty(4 * most, dtype=torch.float32, device=dev)
    scores = torch.empty(items.numel(), dtype=torch.float32, device=dev)
    ptr_d = torch.from_numpy(ptr).to(dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    st = _lib.stream_ptr()
    for s, e in blocks:
        n, q0, npairs = e - s, int(ptr[s]), int(ptr[e] - ptr[s])
        _lib.check(_L.fr_schgn_attend_pairs(
            user_key[s:].data_ptr(), user_comp[s:].data_ptr(), n, ptr_d[s:].data_ptr(), items[q0:].data_ptr(), npairs,
            codes.data_ptr(), slots, nums.data_ptr(), n_items, ingre_key.data_ptr(), ingre_final.data_ptr(),
            ingre_comp.data_ptr(), img_key.data_ptr(), comp_keys.data_ptr(), h_ingre.data_ptr(), h_comp.data_ptr(), d,
            ws.data_ptr(), ws.numel(), att.data_ptr(), logits.data_ptr(), status.data_ptr(), st), "fr_schgn_attend_pairs")
        _lib.check(_L.fr_schgn_score_pairs(
            user_final[s:].data_ptr(), user_hidden[s:].data_ptr(), n, ptr_d[s:].data_ptr(), items[q0:].data_ptr(), npairs,
            W_item.data_ptr(), W_prod.data_ptr(), w_out.data_ptr(), comps.data_ptr(), att.data_ptr(), logits.data_ptr(),
            n_items, d, scores[q0:].data_ptr(), st), "fr_schgn_score_pairs")
    if int(status.item()) != 0:          # cand_ptr was checked on the host: only an item can be out of range here
        raise _lib.FoodRecError(f"a candidate item is outside [0, {n_items})")
    return scores


def evaluate_by_user(model, users, cand_ptr, cand_items, n_pos, neg_num: int = 500, device_metrics: bool = False):
    """The reference's default evaluation (`eval_by_user: True`): every user is scored against its
    positives followed by `neg_num` sampled negatives (FoodRec/common/trainer.py:231-282,
    utils/dataloader.py:228-302).  The reference propagates once and then, PER USER, calls
    `inference_fast`, copies the scores to the host and argsorts them there; here all users' candidates
    are scored by one `fr_pair_scores` launch and read back once.  A model with its own `by_user_scores`
    (SCHGN: the fused pair scorer over candidate lists) is asked directly.

    `users [n]`, `cand_ptr [n+1]`, `cand_items [cand_ptr[-1]]` (positives first for each user), `n_pos [n]`
    are host arrays.  Returns the reference's metric dict.  `device_metrics=True` computes it on the GPU
    (`metrics.by_user_metrics_device`) and returns the scores as a device tensor instead of copying them back."""
    from . import metrics as M, ops
    users = np.asarray(users, dtype=np.int64)
    cand_ptr = np.asarray(cand_ptr, dtype=np.int64)
    cand_items = np.asarray(cand_items, dtype=np.int64)
    model.eval()
    with torch.no_grad():
        if hasattr(model, "by_user_scores"):
            dev = next(model.parameters()).device
            scores = model.by_user_scores(torch.from_numpy(users).to(dev), cand_ptr, torch.from_numpy(cand_items).to(dev))
        else:
            user_all, item_all = model._tables()
            dev = user_all.device
            rep = np.repeat(users, np.diff(cand_ptr))
            scores = ops.pair_scores(user_all, item_all, torch.from_numpy(rep).to(dev), torch.from_numpy(cand_items).to(dev))
        if device_metrics:
            return M.by_user_metrics_device(scores, cand_ptr, np.asarray(n_pos), neg_num), scores
        scores = scores.cpu().numpy()
    return M.by_user_metrics(scores, cand_ptr, np.asarray(n_pos), neg_num), scores
