"""The fused optimizers (`fr_optim_step`, `train.FusedAdam` / `FusedSGD` / `FusedAdagrad` / `FusedRMSprop`,
`train.build_optimizer`) and learning-rate schedules under CUDA-graph replay.

Tolerances follow the policy of `test_gpu_train_kernels.py`: one step of each rule against a float64 restatement
computed from the kernel's own fp32 inputs, bounded by a few units of fp32 roundoff per intermediate, propagated
through the formula.  Comparisons against torch's own optimizers on the GPU use a fixed tolerance (same arithmetic,
contraction into fma may differ by an ulp per operation); graph replay against eager calls of the same kernels is
bit-exact.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

U32 = 2.0 ** -24
ADAM, SGD, ADAGRAD, RMSPROP = 0, 1, 2, 3
RULES = {ADAM: "adam", SGD: "sgd", ADAGRAD: "adagrad", RMSPROP: "rmsprop"}
N_STATE = {ADAM: 2, SGD: 0, ADAGRAD: 1, RMSPROP: 1}
HYPER = dict(beta1=0.9, beta2=0.999, alpha=0.99)
EPS = {ADAM: 1e-8, SGD: 0.0, ADAGRAD: 1e-10, RMSPROP: 1e-8}


def _lib():
    from foodrec_b200 import _lib
    return _lib


def as64(t):
    return t.detach().cpu().double().numpy().reshape(-1)


def assert_within(got, ref, bound, what):
    got = as64(got)
    err = np.abs(got - ref)
    bad = ~(err <= bound)
    if bad.any():
        k = np.flatnonzero(bad)[0]
        pytest.fail(f"{what}: {int(bad.sum())} of {bad.size} out of bound; first at {k}: got {got[k]!r} "
                    f"ref {ref[k]!r} bound {bound[k]!r}")


class Dev:
    """Device scalars of one call sequence: lr (fp64), step (int32), scratch."""

    def __init__(self, lr, step0=0):
        self.lr = torch.full((1,), lr, dtype=torch.float64, device="cuda")
        self.step = torch.full((1,), step0, dtype=torch.int32, device="cuda")
        self.scal = torch.zeros(2, device="cuda")


def optim_call(rule, entries, dev, wd, eps=None, step=True, hyper=None):
    """`fr_optim_step` over `entries` = [(p, g, s0, s1) (None where unused), optionally with an explicit n]."""
    L = _lib()
    arr = (L.OptimTensor * max(len(entries), 1))()
    for a, e in zip(arr, entries):
        a.param, a.grad, a.state0, a.state1 = (None if x is None else x.data_ptr() for x in e[:4])
        a.n = e[4] if len(e) > 4 else e[0].numel()
    h = L.OptimHyper(**(hyper or dict(HYPER, eps=EPS[rule] if eps is None else eps, weight_decay=wd)))
    return L.lib.fr_optim_step(rule, arr, len(entries), C.byref(h), dev.lr.data_ptr(),
                               dev.step.data_ptr() if step else None, dev.scal.data_ptr(), L.stream_ptr())


def oracle(rule, p, g, s0, s1, t, lr, wd):
    """One step of torch's `_single_tensor_<rule>` in float64 from the kernel's fp32 inputs, and the bound of each
    fp32 result: (p', s0', s1'), (bp, bs0, bs1).  g' = g + wd p carries bg = 2u (|g| + wd |p|) (the product, the
    sum, wd's own rounding); each later operation adds one rounding, a rounded constant one more, and the bounds
    returned are twice the first-order sums (covers the second-order terms)."""
    eps = EPS[rule]
    gw = g + wd * p
    bg = 2 * U32 * (np.abs(g) + wd * np.abs(p)) if wd else np.zeros_like(g)
    zero = np.zeros_like(p)
    if rule == SGD:
        p1 = p - lr * gw
        bp = lr * (bg + 3 * U32 * np.abs(gw)) + U32 * np.abs(p1)
        return (p1, None, None), (2 * bp, None, None)
    if rule == ADAM:
        b1, b2 = HYPER["beta1"], HYPER["beta2"]
        w1, w2 = 1.0 - b1, 1.0 - b2
        m1 = s0 + w1 * (gw - s0)
        v1 = s1 * b2 + w2 * gw * gw
        bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
        step = lr / bc1
        den = np.sqrt(v1) / math.sqrt(bc2) + eps
        q = m1 / den
        p1 = p - step * q
        bm = 4 * U32 * (np.abs(s0) + np.abs(w1 * (gw - s0))) + w1 * bg
        bv = 4 * U32 * (s1 * b2 + w2 * gw * gw) + 2 * w2 * np.abs(gw) * bg
        with np.errstate(divide="ignore", invalid="ignore"):
            rel_den = np.where(v1 > 0, bv / (2 * v1), 0.0) + 3 * U32
        bp = step * (bm / den + np.abs(q) * (rel_den + 3 * U32)) + U32 * np.abs(p1)
        return (p1, m1, v1), (2 * bp, 2 * bm, 2 * bv)
    if rule == ADAGRAD:
        a1 = s0 + gw * gw
        ba = 2 * U32 * a1 + 2 * np.abs(gw) * bg
    else:
        al = HYPER["alpha"]
        a1 = s0 * al + (1.0 - al) * gw * gw
        ba = 4 * U32 * (s0 * al + (1.0 - al) * gw * gw) + 2 * (1.0 - al) * np.abs(gw) * bg
    den = np.sqrt(a1) + eps
    q = gw / den
    p1 = p - lr * q
    with np.errstate(divide="ignore", invalid="ignore"):
        rel_den = np.where(a1 > 0, ba / (2 * a1), 0.0) + 3 * U32
    bp = lr * (bg / den + np.abs(q) * (rel_den + 3 * U32)) + U32 * np.abs(p1)
    return (p1, a1, zero), (2 * bp, 2 * ba, zero)


def make_entry(rule, n, gen, off=0):
    """(p, g, s0, s1) of n fp32 elements (None for a state the rule lacks); with `off` > 0 each is a view `off`
    floats into its own buffer (4-byte aligned only).  Second moments and sums are >= 0."""
    def one(scale, sq=False):
        base = torch.randn(n + off, generator=gen) * scale
        if sq:
            base = base * base
        return base.cuda()[off:]
    p, g = one(1.0), one(1.0)
    if rule == ADAM:
        return p, g, one(0.3), one(0.2, sq=True)
    if rule == SGD:
        return p, g, None, None
    return p, g, one(0.5, sq=True), None


def snapshot(entries):
    return [None if e[0] is None or e[0].numel() == 0 else tuple(None if x is None else as64(x) for x in e[:4])
            for e in entries]


def check_step(rule, entries, before, t, lr, wd, what):
    for k, (e, b) in enumerate(zip(entries, before)):
        if b is None:
            continue
        p, g, s0, s1 = b
        z = np.zeros_like(p)
        (p1, a1, v1), (bp, ba, bv) = oracle(rule, p, g, z if s0 is None else s0, z if s1 is None else s1, t, lr, wd)
        assert_within(e[0], p1, bp, f"{what}: param of tensor {k}")
        if N_STATE[rule] > 0:
            assert_within(e[2], a1, ba, f"{what}: state0 of tensor {k}")
        if N_STATE[rule] > 1:
            assert_within(e[3], v1, bv, f"{what}: state1 of tensor {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("lr", [0.0, 1e-3])
@pytest.mark.parametrize("wd", [0.0, 1e-4, 0.5])
@pytest.mark.parametrize("rule", list(RULES), ids=list(RULES.values()))
def test_one_step_vs_fp64(rule, wd, lr):
    """Sizes on both sides of the 4096-element chunk (vector path against scalar tail), views 1..3 floats into
    their buffers (scalar path), and a tensor of 6 M elements whose chunks exceed the 8 x num_sms grid (the
    persistent grid strides).  Adam's step counter starts at 999 (bias corrections at t = 1000)."""
    gen = torch.Generator().manual_seed(rule * 100 + int(wd * 10) + int(lr * 1e4))
    entries = [make_entry(rule, n, gen) for n in (4095, 4096, 4097, 3 * 4096)]
    entries += [make_entry(rule, 5000, gen, off=o) for o in (1, 2, 3)]
    entries.append(make_entry(rule, 6_000_000, gen))
    assert (6_000_000 + 4095) // 4096 > 8 * torch.cuda.get_device_properties(0).multi_processor_count
    step0 = 999 if rule == ADAM else 0
    dev = Dev(lr, step0)
    before = snapshot(entries)
    assert optim_call(rule, entries, dev, wd) == 0, _lib().lib.fr_last_error()
    torch.cuda.synchronize()
    if rule in (ADAM, ADAGRAD):
        assert int(dev.step.item()) == step0 + 1
    check_step(rule, entries, before, step0 + 1, lr, wd, f"{RULES[rule]} wd={wd} lr={lr}")
    if lr == 0.0:
        for e, b in zip(entries, before):
            assert np.array_equal(as64(e[0]), b[0])


def ragged(rule, n_tensors, empty, gen):
    out = []
    for k in range(n_tensors):
        if k in empty:
            z = torch.empty(0, device="cuda")
            out.append((z, z, z if N_STATE[rule] else None, None))
        else:
            out.append(make_entry(rule, 1 + (k * 37) % 300, gen))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n_tensors,empty", [(65, {0, 63, 64}), (130, {0, 3, 63, 64, 127, 128})])
@pytest.mark.parametrize("rule", [SGD, ADAGRAD], ids=["sgd", "adagrad"])
def test_each_tensor_updated_once_per_call(rule, n_tensors, empty):
    """More than 64 tensors take several launches; empty tensors at the launch boundaries must not shift the
    cursor.  A tensor updated twice (or not at all) falls outside the one-step bound.  Two calls, so Adagrad's
    counter and accumulated sums are checked across calls."""
    gen = torch.Generator().manual_seed(n_tensors + rule)
    entries = ragged(rule, n_tensors, empty, gen)
    dev = Dev(1e-2)
    for call in (1, 2):
        for e in entries:
            if e[1].numel():
                e[1].copy_(torch.randn(e[1].numel(), generator=gen).cuda())
        before = snapshot(entries)
        assert optim_call(rule, entries, dev, 1e-4, step=rule == ADAGRAD) == 0, _lib().lib.fr_last_error()
        torch.cuda.synchronize()
        if rule == ADAGRAD:
            assert int(dev.step.item()) == call
        check_step(rule, entries, before, call, 1e-2, 1e-4, f"call {call}")


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["unknown_rule", "negative_eps", "negative_wd", "bad_beta", "null_state",
                                 "null_step", "negative_extent", "negative_lr", "nan_lr"])
def test_rejected_call_changes_nothing(bad):
    """A bad argument is rejected before anything runs (a bad tensor sits at position 100 of 130, past the first
    launch).  The learning rate lives on the device, so a negative or NaN lr is rejected by the prologue: no
    parameter, state or step moves, and the scratch says so (NaN)."""
    rule = ADAGRAD if bad in ("null_state", "negative_extent") else ADAM
    gen = torch.Generator().manual_seed(7)
    entries = ragged(rule, 130, {3, 64}, gen)
    p, g, s0, s1 = entries[100]
    if bad == "null_state":
        entries[100] = (p, g, None, None)
    if bad == "negative_extent":
        entries[100] = (p, g, s0, s1, -1)
    dev = Dev({"negative_lr": -1e-3, "nan_lr": float("nan")}.get(bad, 1e-3), 41)
    hyper = dict(HYPER, eps=-1e-8 if bad == "negative_eps" else 1e-8, weight_decay=-1e-4 if bad == "negative_wd" else 0.0)
    if bad == "bad_beta":
        hyper["beta2"] = 1.0
    keep = [tuple(x.clone() for x in e[:4] if x is not None) for e in entries]
    rc = optim_call(7 if bad == "unknown_rule" else rule, entries, dev, 0.0, step=bad != "null_step", hyper=hyper)
    torch.cuda.synchronize()
    if bad in ("negative_lr", "nan_lr"):
        assert rc == 0
        assert math.isnan(float(dev.scal[0]))
    else:
        assert rc != 0
        assert str(_lib().lib.fr_last_error(), "utf-8")
    assert int(dev.step.item()) == 41
    for e, k in zip(entries, keep):
        for x, y in zip([x for x in e[:4] if x is not None], k):
            assert torch.equal(x, y)


# ============================================================================================ optimizer classes
def fused(name, params, **kw):
    from foodrec_b200 import train
    return getattr(train, "Fused" + name)(params, **kw)


TORCH_CASES = [("Adam", dict(lr=2e-3, weight_decay=1e-4)), ("SGD", dict(lr=1e-2, weight_decay=1e-4)),
               ("Adagrad", dict(lr=1e-2, weight_decay=1e-4)), ("RMSprop", dict(lr=1e-3, weight_decay=1e-4))]
STATE_KEYS = {"Adam": ("exp_avg", "exp_avg_sq"), "SGD": (), "Adagrad": ("sum",), "RMSprop": ("square_avg",)}


def ragged_params():
    torch.manual_seed(3)
    shapes = [(4097, 64), (3,), (1000, 7), (64, 64), (5, 4096), (1,)]
    base = [torch.randn(s, device="cuda") for s in shapes]
    big = torch.randn(10_001, device="cuda")
    base.append(big[1:])                      # 4-byte-aligned only: the kernel's scalar path
    return base


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw", TORCH_CASES, ids=[c[0] for c in TORCH_CASES])
def test_fused_optimizer_follows_torch(name, kw):
    """Ten steps against `torch.optim.<name>(foreach=False)` (torch's `_single_tensor_*` arithmetic) over ragged
    tensor sizes, weight decay on, one all-zero and some partially zero gradients: parameters and state."""
    base = ragged_params()
    ref_p = [torch.nn.Parameter(b.clone()) for b in base]
    my_p = [torch.nn.Parameter(b.clone()) for b in base]
    ref = getattr(torch.optim, name)(ref_p, foreach=False, **kw)
    mine = fused(name, my_p, **kw)
    for step in range(10):
        for a, b in zip(ref_p, my_p):
            g = torch.randn_like(a) * (0.0 if step == 4 else 1.0)
            if step % 3 == 0:
                g[: g.shape[0] // 2] = 0
            a.grad, b.grad = g.clone(), g.clone()
        ref.step()
        mine.step()
        for a, b in zip(ref_p, my_p):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6), (step, float((a - b).abs().max()))
    for a, b in zip(ref_p, my_p):
        for k in STATE_KEYS[name]:
            assert torch.allclose(ref.state[a][k], mine.state[b][k], rtol=1e-5, atol=1e-7), (k, float((ref.state[a][k] - mine.state[b][k]).abs().max()))


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw", TORCH_CASES, ids=[c[0] for c in TORCH_CASES])
def test_lr_schedule_under_replay_equals_eager_steps(name, kw):
    """`step()` captured once; `LambdaLR(0.5 ** epoch)` stepped between replays (and `refresh_lr()` before each,
    as `GraphedTrainStep` does) must give the bits of the same sequence of eager `step()` calls."""
    base = ragged_params()
    pa = [torch.nn.Parameter(b.clone()) for b in base]
    pb = [torch.nn.Parameter(b.clone()) for b in base]
    grads = [torch.randn_like(b) for b in base]           # static gradient buffers
    for a, b, g in zip(pa, pb, grads):
        a.grad, b.grad = g, g
    oa, ob = fused(name, pa, **kw), fused(name, pb, **kw)
    sa = torch.optim.lr_scheduler.LambdaLR(oa, lambda e: 0.5 ** e)
    sb = torch.optim.lr_scheduler.LambdaLR(ob, lambda e: 0.5 ** e)
    oa.step()
    ob.step()                                             # the device state exists before the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ob.step()
    for _ in range(5):
        sa.step()
        sb.step()
        oa.step()
        ob.refresh_lr()
        graph.replay()
    torch.cuda.synchronize()
    assert ob.param_groups[0]["lr"] == kw["lr"] * 0.5 ** 5
    for a, b in zip(pa, pb):
        assert torch.equal(a, b)
        for k in STATE_KEYS[name]:
            assert torch.equal(oa.state[a][k], ob.state[b][k])
    # and the schedule took effect: a replay without the refresh would have used the capture-time lr
    pc = [torch.nn.Parameter(b.clone()) for b in base]
    for c, g in zip(pc, grads):
        c.grad = g
    oc = fused(name, pc, **kw)
    for _ in range(6):
        oc.step()
    assert any(not torch.equal(a, c) for a, c in zip(pa, pc))


def clussl_model(ds):
    from foodrec_b200.models.pricai_modelx import PRICAI_ModelX

    class Cfg(dict):
        def __getitem__(self, k):
            return self.get(k)
    cfg = Cfg(device="cuda", embedding_size=64, train_batch_size=64, is_multimodal_model=True, end2end=False,
              use_health_level_multi_hot=True, n_ri_layers=2, n_mm_layers=1, n_ui_layers=1, reg_weight=0.01,
              loss_cl=0.1, n_cluster=ds.cfg.n_cluster, learner="adam", learning_rate=0.01, weight_decay=1e-4)
    torch.manual_seed(999)
    return PRICAI_ModelX(cfg, ds).to("cuda"), cfg


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", [True, False])
def test_graphed_train_step_follows_an_lr_schedule(mini_ds, schedule):
    """The drop-in model on the mini dataset, `build_optimizer` (Adam, wd = 1e-4) and `GraphedTrainStep`.  Replay
    and eager steps differ in the last bits (fp32 atomics in the backward), so the check is deterministic instead:
    a `LambdaLR` whose factor drops to 0 after the first epoch leaves every parameter bit-identical over the
    following replays; without the scheduler the same replays move them."""
    from foodrec_b200.synth import sample_train_batches
    from foodrec_b200.train import FusedAdam, GraphedTrainStep, build_optimizer
    m, cfg = clussl_model(mini_ds)
    m.train()
    opt = build_optimizer(cfg, m.parameters())
    assert isinstance(opt, FusedAdam) and opt.param_groups[0]["weight_decay"] == 1e-4
    dev = [{k: torch.from_numpy(b[k]).cuda() for k in ("u_id", "pos_i_id", "neg_i_id")}
           for b in sample_train_batches(mini_ds, 64, 4, seed=2)]
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda e: 1.0 if e == 0 else 0.0) if schedule else None
    step = GraphedTrainStep(m, opt, dev[0], warmup=1)
    p0 = [p.detach().clone() for p in m.parameters()]
    for b in dev:
        step(b)
    torch.cuda.synchronize()
    moved = [not torch.equal(p, q) for p, q in zip(m.parameters(), p0)]       # parameters the loss reaches
    assert any(moved)
    if sched is not None:
        sched.step()
        assert opt.param_groups[0]["lr"] == 0.0
    p1 = [p.detach().clone() for p in m.parameters()]
    for b in dev:
        step(b)
    torch.cuda.synchronize()
    same = [torch.equal(p, q) for p, q in zip(m.parameters(), p1)]
    if schedule:
        assert all(same)
    else:
        assert not any(s for s, mv in zip(same, moved) if mv)


@pytest.mark.gpu
def test_graphed_train_step_refuses_a_frozen_lr_change(mini_ds):
    """torch's Adam (capturable, float lr) freezes lr into the graph: a replay after the lr changed raises."""
    from foodrec_b200.synth import sample_train_batches
    from foodrec_b200.train import GraphedTrainStep
    m, _ = clussl_model(mini_ds)
    m.train()
    opt = torch.optim.Adam(m.parameters(), lr=0.01, capturable=True)
    b = {k: torch.from_numpy(v).cuda() for k, v in sample_train_batches(mini_ds, 64, 1, seed=3)[0].items()
         if k in ("u_id", "pos_i_id", "neg_i_id")}
    step = GraphedTrainStep(m, opt, b, warmup=1)
    step(b)
    opt.param_groups[0]["lr"] = 0.005                     # what a scheduler's step() does
    with pytest.raises(RuntimeError, match="lr changed"):
        step(b)


@pytest.mark.gpu
def test_fused_adam_without_weight_decay_equals_fr_adam_step():
    """`FusedAdam(weight_decay=0)` runs `fr_optim_step` with the lr on the device; `fr_adam_step` takes it by
    value.  Both run the same kernels: three steps on copies of the same tensors agree bit for bit."""
    L = _lib()
    base = ragged_params()
    params = [torch.nn.Parameter(b.clone()) for b in base]
    opt = fused("Adam", params, lr=2e-3, betas=(0.8, 0.99), eps=1e-8)
    copies = [(b.clone(), torch.zeros_like(b), torch.zeros_like(b)) for b in base]
    step, scal = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(2, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(3):
        grads = [torch.randn(b.shape, device="cuda", generator=gen) for b in base]
        for p, g in zip(params, grads):
            p.grad = g
        opt.step()
        arr = (L.AdamTensor * len(base))()
        for a, (p, m, v), g in zip(arr, copies, grads):
            a.param, a.grad, a.exp_avg, a.exp_avg_sq, a.n = p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel()
        L.check(L.lib.fr_adam_step(arr, len(base), 2e-3, 0.8, 0.99, 1e-8, step.data_ptr(), scal.data_ptr(),
                                   L.stream_ptr()), "fr_adam_step")
    torch.cuda.synchronize()
    for p, (q, m, v) in zip(params, copies):
        assert torch.equal(p, q)
        assert torch.equal(opt.state[p]["exp_avg"], m) and torch.equal(opt.state[p]["exp_avg_sq"], v)


@pytest.mark.gpu
def test_negative_lr_from_a_scheduler_is_refused():
    params = [torch.nn.Parameter(torch.randn(10, device="cuda"))]
    opt = fused("SGD", params, lr=0.1)
    params[0].grad = torch.ones(10, device="cuda")
    opt.step()
    keep = params[0].detach().clone()
    opt.param_groups[0]["lr"] = -0.1
    with pytest.raises(ValueError):
        opt.step()
    assert torch.equal(params[0], keep)


# ================================================================================================= CPU only
@pytest.mark.parametrize("learner,cls", [("adam", "FusedAdam"), ("Adam", "FusedAdam"), ("SGD", "FusedSGD"),
                                         ("adagrad", "FusedAdagrad"), ("RMSprop", "FusedRMSprop"),
                                         ("lamb", "FusedAdam")])
def test_build_optimizer_maps_the_learner(learner, cls):
    import warnings
    from foodrec_b200 import train
    params = [torch.nn.Parameter(torch.zeros(3))]
    cfg = {"learner": learner, "learning_rate": 0.005, "weight_decay": 1e-4}
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        opt = train.build_optimizer(cfg, params)
    assert type(opt).__name__ == cls
    g = opt.param_groups[0]
    assert g["lr"] == 0.005
    known = learner.lower() in ("adam", "sgd", "adagrad", "rmsprop")
    assert g["weight_decay"] == (1e-4 if known else 0.0)       # the fallback passes lr only
    assert bool(caught) == (not known)


@pytest.mark.parametrize("name,kw", [("Adam", dict(amsgrad=True)), ("Adam", dict(maximize=True)),
                                     ("SGD", dict(momentum=0.9)), ("SGD", dict(nesterov=True)),
                                     ("Adagrad", dict(lr_decay=0.1)), ("Adagrad", dict(initial_accumulator_value=0.1)),
                                     ("RMSprop", dict(momentum=0.9)), ("RMSprop", dict(centered=True)),
                                     ("SGD", dict(lr=-1.0)), ("Adam", dict(weight_decay=-1.0)),
                                     ("RMSprop", dict(eps=-1.0))])
def test_unsupported_or_invalid_options_raise(name, kw):
    from foodrec_b200 import train
    with pytest.raises(ValueError):
        getattr(train, "Fused" + name)([torch.nn.Parameter(torch.zeros(3))], **kw)


def test_defaults_are_torchs():
    import inspect
    from foodrec_b200 import train
    for name in ("Adam", "SGD", "Adagrad", "RMSprop"):
        mine = inspect.signature(getattr(train, "Fused" + name)).parameters
        ref = inspect.signature(getattr(torch.optim, name)).parameters
        for k, v in mine.items():
            if k != "params":
                assert ref[k].default == v.default, (name, k)
