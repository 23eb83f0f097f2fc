"""SCHGN by-user evaluation at C2: the fused candidate-list scorer (`SCHGN.by_user_scores`: `fr_schgn_attend_pairs` +
`fr_schgn_score_pairs`) and `evaluation.evaluate_by_user(..., device_metrics=True)` around it, with the full-sort
scorer's pair rate on the same model and the per-user `inference_by_user` loop beside them.

Model and dataset as `bench.py::_bench_schgn` builds them (seed 999, C2).  Candidates: every user's held-out positives,
then 500 negatives drawn without replacement from the items outside them (numpy seed 0), 35 M pairs in all.  Kernel
times are CUDA events around each launch (`_lib.kernel_profile`) over one scoring call; wall times are host clocks
around calls that end in a device synchronise (median of 5).  The `evaluate_by_user` wall time is split into the
scoring call, the host -> device copy of the int64 candidate ids and the rebuild of the item-side tables that
`model.eval()` causes (the rest is host-side conversion and the metric call).  The per-user loop runs 200 users and is extrapolated
linearly to all users.  Per-pair reciprocal and FMA counts follow from the shapes: 64 features x (ingredients + 4
component logits) tanh evaluations, each one reciprocal; the FMA count adds the attended-row sums and the 64 x 64 M_u x.

    python scripts/microbench_schgn_by_user.py [out.json]      (default: profiles/schgn_by_user.json)
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import foodrec_b200  # noqa: E402,F401
from foodrec_b200 import _lib, evaluation as E  # noqa: E402
from foodrec_b200.models.schgn import SCHGN  # noqa: E402
from foodrec_b200.synth import make_dataset  # noqa: E402
from bench import Cfg, SCHGN_CFG  # noqa: E402

NEG = 500
LOOP_USERS = 200


def wall_ms(fn, iters=5, warm=1):
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


def candidates(ds, rng):
    lists, n_pos = [], []
    for u in range(ds.n_users):
        p = np.asarray(ds.testRatings[u], dtype=np.int64)
        while True:
            draw = rng.integers(0, ds.n_items, NEG + 200)
            _, first = np.unique(draw, return_index=True)
            draw = draw[np.sort(first)]
            draw = draw[~np.isin(draw, p)][:NEG]
            if len(draw) == NEG:
                break
        lists.append(np.concatenate([p, draw]))
        n_pos.append(len(p))
    ptr = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int64)
    return ptr, np.concatenate(lists), np.asarray(n_pos)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "schgn_by_user.json")
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    ds = make_dataset("C2")
    torch.manual_seed(999)
    model = SCHGN(Cfg({**SCHGN_CFG, "device": str(dev)}), ds).to(dev).eval()
    ptr, items, n_pos = candidates(ds, np.random.default_rng(0))
    users = np.arange(ds.n_users)
    n_pairs = int(ptr[-1])
    users_d, items_d = torch.from_numpy(users).to(dev), torch.from_numpy(items).to(dev)
    score = lambda: model.by_user_scores(users_d, ptr, items_d)  # noqa: E731
    with torch.no_grad():
        score()                                                   # item-side tables, module load
        torch.cuda.synchronize()
        with _lib.kernel_profile() as prof:
            scores = score()
            torch.cuda.synchronize()
        score_ms = wall_ms(score)
        eval_ms = wall_ms(lambda: E.evaluate_by_user(model, users, ptr, items, n_pos, neg_num=NEG, device_metrics=True))
        metrics, _ = E.evaluate_by_user(model, users, ptr, items, n_pos, neg_num=NEG, device_metrics=True)
        # parts of that wall time: the pageable host -> device copy of the int64 candidate ids, and the item-side
        # tables, which `model.eval()` drops and the next call rebuilds
        h2d_ms = wall_ms(lambda: torch.from_numpy(items).to(dev))

        def rebuild():
            model.eval()
            model._item_side()
        rebuild_ms = wall_ms(rebuild)

        fs_users = torch.arange(256, device=dev)
        fs_ms = wall_ms(lambda: model.full_sort_scores(fs_users))
        with _lib.kernel_profile() as fs_prof:
            model.full_sort_scores(fs_users)
            torch.cuda.synchronize()

        # the existing per-user route: one `inference_by_user` batch per user, inputs already on the device
        t = lambda a: torch.from_numpy(np.asarray(a)).to(dev)  # noqa: E731
        batches = []
        for u in range(LOOP_USERS):
            x = items[ptr[u]:ptr[u + 1]]
            batches.append({"user_input": torch.full((len(x),), u, device=dev), "item_input": t(x),
                            "img_input": t(ds.embImage[x]), "ingre_num_input": t(ds.ingredientNum[x]),
                            "ingre_input": t(ds.ingredientCodeDict[x]), "cal_level_input": t(ds.cal_level[x])})
        loop_out = [model.inference_by_user(b) for b in batches[:5]]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop_out = [model.inference_by_user(b) for b in batches]
        torch.cuda.synchronize()
        loop_ms = (time.perf_counter() - t0) * 1e3
        loop_diff = max(float((scores[ptr[u]:ptr[u + 1]] - loop_out[u].reshape(-1)).abs().max()) for u in range(LOOP_USERS))
        loop_scale = max(float(o.abs().max()) for o in loop_out)
        score_abs_max, score_std = float(scores.abs().max()), float(scores.std())

    kern = {name: {"launches": n, "ms_total": us / 1e3} for name, (n, us) in prof.result.items()}
    fs_kern = {name: {"launches": n, "ms_total": us / 1e3} for name, (n, us) in fs_prof.result.items()}
    by_user_kernel_ms = sum(v["ms_total"] for v in kern.values())
    fs_kernel_ms = sum(v["ms_total"] for v in fs_kern.values())
    n_ingr = np.minimum(np.asarray(ds.ingredientNum)[items], np.asarray(ds.ingredientCodeDict).shape[1]).mean()
    d = 64
    rcp = d * (n_ingr + 4)
    fma = d * n_ingr * (4.5 + 2.0) + 4 * d * 4.5 + d * d + 4 * d
    res = {
        "gpu": gpu[0] if gpu else torch.cuda.get_device_name(0),
        "workload": f"C2 SCHGN by-user: {ds.n_users} users x (held-out positives + {NEG} negatives drawn without "
                    f"replacement outside them), {n_pairs} pairs",
        "pairs": n_pairs, "users": ds.n_users,
        "kernels_one_call": kern, "kernel_ms_one_call": by_user_kernel_ms,
        "by_user_scores_wall_ms": score_ms,
        "evaluate_by_user_device_metrics_wall_ms": eval_ms,
        "evaluate_by_user_parts_ms": {"by_user_scores": score_ms, "h2d_int64_candidate_ids": h2d_ms,
                                      "item_side_tables_rebuild_after_eval": rebuild_ms,
                                      "rest": eval_ms - score_ms - h2d_ms - rebuild_ms},
        "scores_abs_max": score_abs_max, "scores_std": score_std,
        "pairs_per_s_scoring_wall": n_pairs / (score_ms * 1e-3),
        "pairs_per_s_kernels": n_pairs / (by_user_kernel_ms * 1e-3),
        "full_sort": {"workload": f"256 users x {ds.n_items} items, dense scores (fr_schgn_attend + fr_schgn_score)",
                      "wall_ms": fs_ms, "kernels": fs_kern, "kernel_ms": fs_kernel_ms,
                      "pairs_per_s_wall": 256 * ds.n_items / (fs_ms * 1e-3),
                      "pairs_per_s_kernels": 256 * ds.n_items / (fs_kernel_ms * 1e-3)},
        "by_user_over_full_sort_pairs_per_s_kernels": (n_pairs / by_user_kernel_ms) / (256 * ds.n_items / fs_kernel_ms),
        "per_user_inference_by_user_loop": {
            "users_timed": LOOP_USERS, "ms": loop_ms,
            "extrapolated_ms_all_users": loop_ms / LOOP_USERS * ds.n_users,
            "kind": f"extrapolation: {LOOP_USERS} users timed, scaled linearly to {ds.n_users}",
            "max_abs_diff_vs_by_user_scores": loop_diff, "max_abs_score_of_these_users": loop_scale,
            "max_abs_diff_relative_to_max_abs_score": loop_diff / loop_scale},
        "per_pair_counts": {"mean_ingredients": float(n_ingr), "reciprocals": float(rcp), "fma_approx": float(fma)},
        "metrics": {k: float(v) for k, v in metrics.items()},
    }
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
