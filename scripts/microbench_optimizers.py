"""Fused optimizer steps (`fr_optim_step`: Adam, SGD, Adagrad, RMSprop) on HealthRec's C2 parameter set against
torch's fastest implementation of the same learner on the same tensors.

Workload: every trainable parameter of `CIKM_Model` on the C2 data (~211 M fp32 parameters, most of them the
raw-feature tables), random dense gradients, weight decay 1e-4 (the factory's `weight_decay` path).  The working
set (5.9 GB for Adam) is far beyond the 126 MB L2, so every step streams from HBM.  Time per step is CUDA events
around a loop of eager `step()` calls lasting at least 0.5 s (the steps are HBM-bound milliseconds, so the host
keeps the queue full); bytes per parameter are what the update must move (p, g read, p written, each state read
and written: Adam 28, SGD 12, Adagrad 20, RMSprop 20).  torch's comparison uses `fused=True` where torch has a
fused CUDA kernel for the learner and `foreach=True` otherwise.

    python scripts/microbench_optimizers.py [out.json]     (default profiles/optimizers.json)
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import foodrec_b200  # noqa: F401
from foodrec_b200 import train
from foodrec_b200.synth import make_dataset

HBM_PEAK = 7.7e12       # B200 data sheet, bytes/s
BYTES = {"Adam": 28, "SGD": 12, "Adagrad": 20, "RMSprop": 20}
LR = {"Adam": 1e-3, "SGD": 1e-3, "Adagrad": 1e-2, "RMSprop": 1e-2}
DESIGN_ADAM_MS = 1.40   # fr_adam_step on this parameter set before the optimizers shared one kernel (DESIGN.md 3.7)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def shapes():
    from bench import BATCH, Cfg
    from foodrec_b200.models.cikm_model import CIKM_Model
    ds = make_dataset("C2")
    cfg = Cfg(device="cuda", embedding_size=64, train_batch_size=BATCH, is_multimodal_model=True, end2end=False,
              use_health_level_multi_hot=True, num_attention_heads=2, num_hidden_layers=2, attention_probs_dropout_prob=0.5,
              hidden_act="gelu", n_layers=2, ui_layers=1, reg_weight=0.5, loss_kd=0.05, loss_health=0.1, kd_threshold=0.4,
              learning_rate=0.001)          # bench.py::_bench_healthrec
    torch.manual_seed(999)
    m = CIKM_Model(cfg, ds)
    return [tuple(p.shape) for p in m.parameters() if p.requires_grad]


def make_params(shp):
    gen = torch.Generator(device="cuda").manual_seed(0)
    ps = []
    for s in shp:
        p = torch.nn.Parameter(torch.randn(s, device="cuda", generator=gen) * 0.1)
        p.grad = torch.randn(s, device="cuda", generator=gen) * 0.01
        ps.append(p)
    return ps


def events_ms(step, min_s=0.5):
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    n = 8
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            step()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        if ms >= min_s * 1e3:
            return ms / n, n
        n *= 2


def torch_fastest(name, ps):
    """torch's fused CUDA kernel for the learner if it has one, else its foreach implementation."""
    cls = getattr(torch.optim, name)
    try:
        opt = cls(ps, lr=LR[name], weight_decay=1e-4, fused=True)
        opt.step()
        return opt, "fused"
    except (RuntimeError, TypeError, ValueError):
        return cls(ps, lr=LR[name], weight_decay=1e-4, foreach=True), "foreach"


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "optimizers.json")
    assert torch.cuda.is_available(), "needs a CUDA device"
    shp = shapes()
    n_par = sum(int(torch.Size(s).numel()) for s in shp)
    res = {"card": card(), "parameters": n_par, "tensors": len(shp), "hbm_peak_Bps": HBM_PEAK,
           "workload": "CIKM_Model (HealthRec) trainable parameters on the C2 data, random dense gradients, wd = 1e-4",
           "timing": "CUDA events around >= 0.5 s of eager step() calls", "rules": {}}
    for name in ("Adam", "SGD", "Adagrad", "RMSprop"):
        ps = make_params(shp)
        opt = getattr(train, "Fused" + name)(ps, lr=LR[name], weight_decay=1e-4)
        ms, n = events_ms(opt.step)
        del opt
        torch.cuda.empty_cache()
        tref, kind = torch_fastest(name, ps)
        ms_t, n_t = events_ms(tref.step)
        del tref, ps
        torch.cuda.empty_cache()
        b = BYTES[name] * n_par
        res["rules"][name] = {
            "bytes_per_param": BYTES[name], "bytes": b,
            "this_library": {"kernel": f"{name.lower()}_multi_kernel (fr_optim_step)", "ms": ms, "steps_timed": n,
                             "TBps": b / (ms * 1e-3) / 1e12, "frac_of_hbm_peak": b / (ms * 1e-3) / HBM_PEAK},
            "torch": {"impl": f"torch.optim.{name}({kind}=True)", "ms": ms_t, "steps_timed": n_t,
                      "TBps": b / (ms_t * 1e-3) / 1e12, "frac_of_hbm_peak": b / (ms_t * 1e-3) / HBM_PEAK},
            "speedup_vs_torch": ms_t / ms}
        print(name, json.dumps(res["rules"][name]), flush=True)
    a = res["rules"]["Adam"]["this_library"]["ms"]
    res["adam_vs_design_3_7"] = {"design_ms": DESIGN_ADAM_MS, "design_TBps": 4.2, "ms": a, "ratio": a / DESIGN_ADAM_MS}
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["adam_vs_design_3_7"]))


if __name__ == "__main__":
    main()
