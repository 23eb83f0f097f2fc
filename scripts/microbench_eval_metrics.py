"""Evaluation metrics: host numpy (`metrics.topk_metrics` / `metrics.by_user_metrics`) vs the device kernels
(`fr_topk_metrics` / `fr_by_user_metrics`), with the ranking that produces their input beside them.

Shapes: C2 full sort (70 000 users x 45 000 items, k = 50, history mask), the 1 M x 500 k sweep built as
`bench.py::_bench_eval_c4` builds it (k = 50 here), and C2 by-user (70 000 users x (held-out positives + 500 sampled
negatives)).  Host times include the device -> host copy of the indices / scores the host metrics need; device
`kernel_ms` is CUDA events around the metric launch (median of 20), `e2e_ms` a host clock around the whole call
including the final copy of the sums.  The full-sort kernel's bytes are the top-K indices plus the positives' CSR; at
C2 they fit the 126 MB L2 and are read from there after the first pass, at C4 (200 MB of indices) they do not.

    python scripts/microbench_eval_metrics.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import foodrec_b200  # noqa: F401
from foodrec_b200 import evaluation as E, metrics as M, ops
from foodrec_b200.synth import make_dataset

HBM_PEAK = 7.7e12       # B200 data sheet, bytes/s


def ev_ms(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def wall_ms(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def full_sort_case(name, U, I, hist, pos, k=50, host_iters=3):
    topk = (5, 10, 20, 50)
    run = lambda: E.gemm_topk(U, I, k, row_ids=torch.arange(U.shape[0], device=U.device), hist=hist,   # noqa: E731
                              index_dtype=torch.int32)[1]
    rank_ms = ev_ms(run, iters=5, warm=1)
    top = run()
    t0 = time.perf_counter()
    sets = M.ItemSets.from_lists(pos, top.device)
    build_ms = (time.perf_counter() - t0) * 1e3

    def host():
        return M.topk_metrics(top.cpu().numpy().astype(np.int64), pos, topk=topk)
    host_ts = []
    for _ in range(host_iters):
        t0 = time.perf_counter()
        want = host()
        host_ts.append((time.perf_counter() - t0) * 1e3)
    kernel_ms = ev_ms(lambda: M.topk_metrics_sums(top, sets, topk))
    e2e_ms = wall_ms(lambda: M.topk_metrics_device(top, sets, topk=topk))
    got = M.topk_metrics_device(top, sets, topk=topk)
    n = top.shape[0]
    nbytes = top.numel() * top.element_size() + (n + 1) * 8 + n * 4 + sets.idx.numel() * 4
    return {"case": name, "users": n, "k": k, "rank_ms": rank_ms, "host_metrics_ms": float(np.median(host_ts)),
            "device_kernel_ms": kernel_ms, "device_e2e_ms": e2e_ms, "item_sets_build_ms": build_ms,
            "kernel_bytes": nbytes, "kernel_GBps": nbytes / kernel_ms / 1e6,
            "kernel_frac_hbm_peak": nbytes / (kernel_ms * 1e-3) / HBM_PEAK,
            "speedup_e2e": float(np.median(host_ts)) / e2e_ms, "metrics_equal": got == want,
            "differences": {key: (got[key], want[key]) for key in want if got[key] != want[key]}}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": gpu[0] if gpu else torch.cuda.get_device_name(0), "cases": []}

    # ---- C2 full sort
    ds = make_dataset("C2", features=False)
    g = torch.Generator(device=dev).manual_seed(0)
    U = torch.randn(ds.n_users, 64, device=dev, generator=g) * 0.1
    I = torch.randn(ds.n_items, 64, device=dev, generator=g) * 0.1
    hist = E.HistoryCSR(ds.train_coo_matrix, ds.n_users, dev)
    res["cases"].append(full_sort_case("C2 full sort 70 000 x 45 000", U, I, hist, ds.testRatings))

    # ---- C2 by user: held-out positives first, then 500 sampled negatives
    rng = np.random.default_rng(0)
    n_pos = np.array([len(p) for p in ds.testRatings])
    neg = rng.integers(0, ds.n_items, size=(ds.n_users, 500))
    cand = np.concatenate([np.concatenate([np.asarray(p), neg[u]]) for u, p in enumerate(ds.testRatings)])
    ptr = np.concatenate([[0], np.cumsum(n_pos + 500)])
    rep = torch.from_numpy(np.repeat(np.arange(ds.n_users), n_pos + 500)).to(dev)
    cand_d = torch.from_numpy(cand).to(dev)
    score = lambda: ops.pair_scores(U, I, rep, cand_d)      # noqa: E731
    rank_ms = ev_ms(score, iters=10)
    scores = score()
    ptr_d, npos_d = torch.from_numpy(ptr).to(dev), torch.from_numpy(n_pos).to(dev, torch.int32)
    host_ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        want = M.by_user_metrics(scores.cpu().numpy(), ptr, n_pos, 500)
        host_ts.append((time.perf_counter() - t0) * 1e3)
    kernel_ms = ev_ms(lambda: M.by_user_metrics_device(scores, ptr_d, npos_d, 500))   # includes the 40-byte copy
    e2e_ms = wall_ms(lambda: M.by_user_metrics_device(scores, ptr_d, npos_d, 500))
    got = M.by_user_metrics_device(scores, ptr_d, npos_d, 500)
    with foodrec_b200._lib.kernel_profile() as prof:
        for _ in range(20):
            M.by_user_metrics_device(scores, ptr_d, npos_d, 500)
    n_launch, us = prof.result.get("by_user_metrics_kernel", (1, float("nan")))
    res["cases"].append({"case": "C2 by user 70 000 x (positives + 500)", "users": ds.n_users,
                         "candidates": int(ptr[-1]), "rank_ms": rank_ms, "host_metrics_ms": float(np.median(host_ts)),
                         "device_kernel_ms": us / n_launch / 1e3, "device_call_ms_events": kernel_ms,
                         "device_e2e_ms": e2e_ms, "speedup_e2e": float(np.median(host_ts)) / e2e_ms,
                         "max_abs_diff": max(abs(got[k] - float(want[k])) for k in want)})
    del scores, rep, cand_d, U, I, hist

    # ---- C4: 1 M users x 500 k items, 20-item history mask per user (bench.py::_bench_eval_c4), k = 50
    M_all, N = 1_000_000, 500_000
    I = torch.randn(N, 64, device=dev, generator=torch.Generator(device=dev).manual_seed(4)) * 0.1
    gu = torch.Generator(device=dev).manual_seed(1000)
    U = torch.randn(M_all, 64, device=dev, generator=gu) * 0.1
    hist_idx = torch.sort(torch.randint(0, N, (M_all, 20), device=dev, generator=gu), dim=1)[0].to(torch.int32).reshape(-1)

    class _Hist:
        ptr = torch.arange(0, 20 * M_all + 1, 20, device=dev, dtype=torch.int64)
        idx = hist_idx
    rng = np.random.default_rng(4)
    lens = 1 + rng.poisson(2.0, size=M_all)           # held-out positives per user, as synth draws them
    flat = rng.integers(0, N, size=int(lens.sum()))
    bounds = np.cumsum(lens)[:-1]
    pos = np.split(flat, bounds)
    res["cases"].append(full_sort_case("C4 full sort 1 000 000 x 500 000", U, I, _Hist, pos, host_iters=1))

    line = json.dumps(res)
    print(line)
    if out_path:
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
