"""The kernels of a training step against float64 references at their edge shapes.

Every case runs the kernel on fp32 inputs and the same operation in float64 on the CPU from the same fp32 values
(`oracle/losses.py` in double, plain torch / numpy in double, or the formula written out), then checks each entry
against a bound that the reference computes.  Cases aim at the code paths that the model-level tests do not reach:
multi-batch Adam, zero-size tensors, the grid-stride loops, widths that leave lanes idle, empty groups, saturated
sigmoids, NULL outputs and single-block scans over more than one 1024-row chunk.

Tolerance policy (u = 2^-24, the unit roundoff of fp32):

* A dot product, mean or norm is bounded by `c * u * sum|terms|`, per entry or per row, where `sum|terms|` is taken
  from the float64 reference and c is the length of the longest chain of fp32 roundings in the kernel's summation
  tree (a lane's fma chain + the warp butterfly + the block and grid folds) plus a few roundings for the terms
  themselves.  That is the first-order worst-case bound gamma_c for recursive summation (Higham, *Accuracy and
  Stability of Numerical Algorithms*, 2nd ed., section 4.2): it holds for every input and every summation order,
  so it also covers sums whose order changes from run to run because they go through atomics; such sums are never
  compared for bit equality.  A bare rtol against the tensor's maximum is not used: it would hide errors in the
  small entries.
* Elementwise arithmetic (Adam) is bounded by a few u of each intermediate, propagated through the formula.
* Pure data movement (gather, spread, sum of one table) and left-to-right fp32 sums that the reference repeats in
  fp32 in the same order (sum_rows, spread_rows with accumulation) must be bit-exact, as must the integer scan.
* Where fp32 rounds a value that float64 keeps (a saturated sigmoid: 1 - sigmoid(30) = 9e-14 is 0 in fp32), an
  absolute floor of u times the magnitude the rounding can lose is added, and the case says so.

Distance correlation and InfoNCE have their edge cases in `test_gpu_losses.py` (bounds of DESIGN section 3.3).
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24


def _lib():
    from foodrec_b200 import _lib
    return _lib


def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def assert_within(got, ref, bound, what):
    got = np.asarray(got.detach().cpu() if torch.is_tensor(got) else got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    bound = np.broadcast_to(np.asarray(bound, dtype=np.float64), ref.shape)
    err = np.abs(got - ref)
    bad = ~(err <= bound)                       # NaN fails too
    if bad.any():
        k = np.flatnonzero(bad.reshape(-1))[0]
        pytest.fail(f"{what}: {int(bad.sum())} of {bad.size} entries out of bound; first at flat index {k}: "
                    f"got {got.reshape(-1)[k]!r} ref {ref.reshape(-1)[k]!r} bound {bound.reshape(-1)[k]!r}")


def as64(t):
    return t.detach().cpu().double().numpy()


def max_mult(idx):
    """Largest number of times one index occurs (the length of an atomic accumulation chain)."""
    idx = np.asarray(idx).reshape(-1)
    return int(np.bincount(idx).max()) if idx.size else 0


# ======================================================================================================== Adam
def adam_call(entries, lr, b1, b2, eps, step_dev, scal):
    """`fr_adam_step` over `entries` = [(p, g, m, v) or (None, None, None, None, n)]; returns the return code."""
    L = _lib()
    arr = (L.AdamTensor * max(len(entries), 1))()
    for a, e in zip(arr, entries):
        p, g, m, v = e[:4]
        a.param, a.grad, a.exp_avg, a.exp_avg_sq = (None if x is None else x.data_ptr() for x in (p, g, m, v))
        a.n = e[4] if len(e) > 4 else p.numel()
    rc = L.lib.fr_adam_step(arr, len(entries), float(lr), float(b1), float(b2), float(eps), step_dev.data_ptr(),
                            scal.data_ptr(), L.stream_ptr())
    return rc


def adam_oracle(p, g, m, v, t, lr, b1, b2, eps):
    """One step of `torch.optim.adam._single_tensor_adam` (amsgrad = False, weight_decay = 0) in float64 from the
    kernel's own current fp32 state, and an error bound for each fp32 result.

    The kernel evaluates m' = m + w1 (g - m), v' = v b2 + (w2 g) g, den = sqrt(v') / bc2s + eps,
    p' = p + (-lr / bc1) (m' / den), with w1 = 1 - b1, w2 = 1 - b2, b2, -lr / bc1 and bc2s = sqrt(1 - b2^t) each
    rounded once to fp32.  Counting one rounding per operation and per rounded constant:
      |m' - m'64| <= 3u |w1 (g - m)| + u |m'|               -> bm = 4u (|m| + |w1 (g - m)|)
      |v' - v'64| <= 2u v b2 + 3u w2 g^2 + u v'            -> bv = 4u (v b2 + w2 g^2)
      den: the sqrt halves v's relative error, then sqrt, division, add: <= (bv / (2 v') + 3u) den
      p':  |step| (bm / den + |q| (rel(den) + 3u)) + u |p'|, q = m' / den.
    The returned bounds are twice that, which covers the second-order terms."""
    p, g, m, v = (np.asarray(x, dtype=np.float64) for x in (p, g, m, v))
    w1, w2 = 1.0 - b1, 1.0 - b2
    m1 = m + w1 * (g - m)                   # exp_avg.lerp_(grad, 1 - beta1)
    v1 = v * b2 + w2 * g * g                # exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
    step = lr / bc1
    den = np.sqrt(v1) / math.sqrt(bc2) + eps
    q = m1 / den
    p1 = p - step * q                       # param.addcdiv_(exp_avg, denom, value=-step_size)
    bm = 4 * U32 * (np.abs(m) + np.abs(w1 * (g - m)))
    bv = 4 * U32 * (v * b2 + w2 * g * g)
    with np.errstate(divide="ignore", invalid="ignore"):
        rel_den = np.where(v1 > 0, bv / (2 * v1), 0.0) + 3 * U32
    bp = step * (bm / den + np.abs(q) * (rel_den + 3 * U32)) + U32 * np.abs(p1)
    return (p1, m1, v1), (2 * bp, 2 * bm, 2 * bv)


def make_adam_tensor(n, gen, off=0):
    """(p, g, m, v) of n fp32 elements; with `off` > 0 each is a view `off` floats into its own buffer (4-byte
    aligned only).  v >= 0 as a second moment is."""
    def one(scale, sq=False):
        base = torch.randn(n + off, generator=gen) * scale
        if sq:
            base = base * base
        return base.cuda()[off:]
    return one(1.0), one(1.0), one(0.3), one(0.2, sq=True)


def check_adam_step(entries, before, t, lr, b1, b2, eps, what):
    for k, (e, b) in enumerate(zip(entries, before)):
        if b is None:
            continue
        (p1, m1, v1), (bp, bm, bv) = adam_oracle(*b, t=t, lr=lr, b1=b1, b2=b2, eps=eps)
        assert_within(e[0], p1, bp, f"{what}: param of tensor {k}")
        assert_within(e[2], m1, bm, f"{what}: exp_avg of tensor {k}")
        assert_within(e[3], v1, bv, f"{what}: exp_avg_sq of tensor {k}")


def snapshot(entries):
    return [None if e[0] is None else tuple(as64(x) for x in e[:4]) for e in entries]


def ragged_entries(n_tensors, empty, gen):
    out = []
    for k in range(n_tensors):
        if k in empty:
            z = torch.empty(0, device="cuda")
            out.append((z, z, z, z))
        else:
            out.append(make_adam_tensor(1 + (k * 37) % 300, gen))
    return out


@pytest.mark.parametrize("n_tensors,empty", [
    (64, {0, 3, 63}),                   # one launch, 61 non-empty tensors
    (65, {0, 3, 63, 64}),               # the last slot empty: still one launch
    (70, {3}),                          # 69 non-empty: the second launch must start at tensor 65, not 64
    (130, {0, 3, 63, 64}),              # three batches
    (130, set(range(64, 128))),         # a run of 64 empty tensors between two non-empty ones
    (5, {0, 1, 2, 3, 4}),               # nothing but empty tensors: only the step counter moves
])
def test_adam_each_tensor_updated_once_per_call(n_tensors, empty):
    gen = torch.Generator().manual_seed(n_tensors + len(empty))
    entries = ragged_entries(n_tensors, empty, gen)
    step = torch.zeros(1, dtype=torch.int32, device="cuda")
    scal = torch.zeros(2, device="cuda")
    lr, b1, b2, eps = 1e-2, 0.9, 0.999, 1e-8
    for call in range(1, 3):            # the counter rises by exactly one per call, however many launches it took
        for e in entries:
            if e[1].numel():
                e[1].copy_(torch.randn(e[1].numel(), generator=gen).cuda())
        before = snapshot(entries)
        assert adam_call(entries, lr, b1, b2, eps, step, scal) == 0, _lib().lib.fr_last_error()
        torch.cuda.synchronize()
        assert int(step.item()) == call
        check_adam_step(entries, [None if b is None or b[0].size == 0 else b for b in before], call, lr, b1, b2, eps,
                        f"call {call}")


@pytest.mark.parametrize("lr,b1,b2,step0", [
    (1e-3, 0.9, 0.999, 0),
    (2e-3, 0.0, 0.9999, 999),           # beta1 = 0, and bias corrections at t = 1000
    (0.0, 0.9, 0.999, 7),               # lr = 0: parameters unchanged, moments still move
])
def test_adam_vector_path_scalar_tails_and_grid_stride(lr, b1, b2, step0):
    """Sizes on both sides of the 4096-element chunk (vector path against scalar tail), views 1..3 floats into
    their buffers (scalar path), and one tensor of 6 M elements: its 1465 chunks exceed the 8 x num_sms grid, so
    the persistent grid strides."""
    gen = torch.Generator().manual_seed(step0 + 11)
    entries = [make_adam_tensor(n, gen) for n in (4095, 4096, 4097, 3 * 4096)]
    entries += [make_adam_tensor(5000, gen, off=o) for o in (1, 2, 3)]
    entries.append(make_adam_tensor(6_000_000, gen))
    assert (6_000_000 + 4095) // 4096 > 8 * num_sms()
    step = torch.full((1,), step0, dtype=torch.int32, device="cuda")
    scal = torch.zeros(2, device="cuda")
    before = snapshot(entries)
    assert adam_call(entries, lr, b1, b2, 1e-8, step, scal) == 0, _lib().lib.fr_last_error()
    torch.cuda.synchronize()
    assert int(step.item()) == step0 + 1
    check_adam_step(entries, before, step0 + 1, lr, b1, b2, 1e-8, f"lr={lr} b1={b1} b2={b2} t={step0 + 1}")
    if lr == 0.0:
        for e, b in zip(entries, before):
            assert np.array_equal(as64(e[0]), b[0])


@pytest.mark.parametrize("bad", ["null_param", "null_exp_avg_sq", "negative_extent"])
def test_adam_rejected_call_changes_nothing(bad):
    """A bad tensor at position 100 of 130 (past the first batch of 64) is rejected before anything runs: every
    parameter, both moments and the step counter keep their bits."""
    gen = torch.Generator().manual_seed(5)
    entries = ragged_entries(130, {3, 64}, gen)
    p, g, m, v = entries[100]
    entries[100] = {"null_param": (None, g, m, v, p.numel()), "null_exp_avg_sq": (p, g, m, None, p.numel()),
                    "negative_extent": (p, g, m, v, -1)}[bad]
    step = torch.full((1,), 41, dtype=torch.int32, device="cuda")
    scal = torch.zeros(2, device="cuda")
    keep = [tuple(x.clone() for x in e[:4] if x is not None) for e in entries]
    scal0 = scal.clone()
    assert adam_call(entries, 1e-2, 0.9, 0.999, 1e-8, step, scal) != 0
    torch.cuda.synchronize()
    assert int(step.item()) == 41
    assert torch.equal(scal, scal0)
    for e, k in zip(entries, keep):
        for x, y in zip([x for x in e[:4] if x is not None], k):
            assert torch.equal(x, y)


def test_fused_adam_over_70_parameters_with_an_empty_one():
    """`train.FusedAdam` hands every parameter with a gradient to one call: 70 parameters, the fourth of zero size,
    take two launches.  Two steps, each against the one-step oracle from the optimizer's own state."""
    from foodrec_b200.train import FusedAdam
    gen = torch.Generator().manual_seed(70)
    shapes = [(1 + (k * 53) % 400,) if k != 3 else (0,) for k in range(70)]
    shapes[10] = (33, 7)
    params = [torch.nn.Parameter(torch.randn(s, generator=gen).cuda()) for s in shapes]
    opt = FusedAdam(params, lr=3e-3, betas=(0.8, 0.99), eps=1e-8)
    for t in (1, 2):
        for p in params:
            p.grad = torch.randn(p.shape, generator=gen).cuda()
        before = []
        for p in params:
            st = opt.state[p]
            m = as64(st["exp_avg"]) if st else np.zeros(p.numel())
            v = as64(st["exp_avg_sq"]) if st else np.zeros(p.numel())
            before.append((as64(p).reshape(-1), as64(p.grad).reshape(-1), m.reshape(-1), v.reshape(-1)))
        opt.step()
        torch.cuda.synchronize()
        for k, (p, b) in enumerate(zip(params, before)):
            (p1, m1, v1), (bp, bm, bv) = adam_oracle(*b, t=t, lr=3e-3, b1=0.8, b2=0.99, eps=1e-8)
            assert_within(p.reshape(-1), p1, bp, f"step {t}: parameter {k}")
            assert_within(opt.state[p]["exp_avg"].reshape(-1), m1, bm, f"step {t}: exp_avg {k}")
            assert_within(opt.state[p]["exp_avg_sq"].reshape(-1), v1, bv, f"step {t}: exp_avg_sq {k}")


# ================================================================================================== rank_loss
GAMMA = 1e-10


def expit(x):
    return np.where(x >= 0, 1.0 / (1.0 + np.exp(-np.abs(x))), np.exp(-np.abs(x)) / (1.0 + np.exp(-np.abs(x))))


def fold_depth(n_tasks, warps_per_block=8, blocks_per_sm=4):
    """Longest chain of fp32 additions when `n_tasks` warp tasks are folded as rank_loss_fwd_kernel folds them: a
    warp's strided tasks, then the warps of its block, then the block partials in order."""
    grid = max(1, min(-(-n_tasks // warps_per_block), blocks_per_sm * num_sms()))
    return -(-n_tasks // (grid * warps_per_block)) + warps_per_block + grid


def rank_case(d, B, groups, seed):
    """Inputs: an embedding table with `U` users then `I` items, B triples (the first ones scripted: score
    differences 0 (p == n), +-30, +-90; the rest random, with repeated ids), and regulariser groups."""
    gen = torch.Generator().manual_seed(seed)
    U, I = (20_000, 30_000) if B > 10_000 else (50, 70)
    emb = torch.randn(U + I, d, generator=gen) * 0.3
    u = torch.randint(0, U - 6, (B,), generator=gen)
    p = torch.randint(0, I - 6, (B,), generator=gen)
    n = torch.randint(0, I - 6, (B,), generator=gen)
    script = [None, 30.0, -30.0, 90.0, -90.0, 0.0]
    for k, s in enumerate(script[:B]):
        if s is None:
            n[k] = p[k]                               # p == n: score difference exactly 0
            continue
        ur, pr, nr = U - 1 - k, I - 1 - k, I - 6      # reserved rows: <E_u, E_p - E_n> = s exactly
        emb[ur] = 0
        emb[ur, 0] = 1.0
        emb[U + pr] = 0
        emb[U + pr, 0] = s
        emb[U + nr] = 0
        u[k], p[k], n[k] = ur, pr, nr
    tA = torch.randn(50, d, generator=gen) * 0.2
    tB = torch.randn(70, d, generator=gen) * 0.2
    tC = torch.randn(12, d, generator=gen) * 0.2      # row 11 is the padding row: counted forward, no gradient
    specs = {
        "none": [],
        "one": [("A", torch.randint(0, 50, (B,), generator=gen), -1)],
        "six": [("A", torch.randint(0, 50, (B,), generator=gen), -1),
                ("B", torch.randint(0, 70, (B,), generator=gen), -1),
                ("B", torch.empty(0, dtype=torch.long), -1),               # empty group between non-empty ones
                ("B", torch.randint(0, 70, (B,), generator=gen), -1),      # the same table in a second group
                ("C", torch.randint(0, 12, (B, 5), generator=gen), 11),    # padding index
                ("A", torch.tensor([7, 7, 0]), -1)],                       # repeated ids
    }[groups]
    if groups == "six":
        specs[4][1][0, :2] = 11                       # the padding index occurs
    return U, emb, u, p, n, dict(A=tA, B=tB, C=tC), specs


RANK_CASES = ([(d, 512, "six") for d in (8, 32, 48, 64, 128, 200)]
              + [(64, B, "six") for B in (1, 7, 50_000)]
              + [(200, 50_000, "one"), (48, 7, "none"), (8, 1, "one"), (128, 512, "none")])


@pytest.mark.parametrize("d,B,groups", RANK_CASES)
def test_rank_loss_vs_fp64(d, B, groups):
    from foodrec_b200 import ops
    U, emb, u, p, n, tabs, specs = rank_case(d, B, groups, seed=d * 7 + B)
    g_mf, g_reg = (0.0, 2.5) if (d + B) % 3 == 0 else (0.7, -1.3)      # upstream gradients != 1, one of them 0
    emb_d = emb.cuda().requires_grad_(True)
    tabs_d = {k: t.cuda().requires_grad_(True) for k, t in tabs.items()}
    mf, reg = ops.rank_loss(emb_d, U, u.cuda(), p.cuda(), n.cuda(),
                            [(tabs_d[k], i.cuda(), pad) for k, i, pad in specs], reg_den=float(B))
    (mf * g_mf + reg * g_reg).backward()
    torch.cuda.synchronize()

    E = emb.double().numpy()
    un, pn, nn_ = u.numpy(), p.numpy() + U, n.numpy() + U
    Eu, Ep, En = E[un], E[pn], E[nn_]
    lanes = -(-d // 32) + 5                            # a lane's fma chain + the warp butterfly
    # ---- BPR: x_b = <E_u, E_p - E_n>; the kernel rounds E_p - E_n (u) and sums d products over `lanes` levels
    x = (Eu * (Ep - En)).sum(1)
    bx = (lanes + 2) * U32 * (np.abs(Eu) * (np.abs(Ep) + np.abs(En))).sum(1)
    sg, sgc = expit(x), expit(-x)
    ell = -np.log(GAMMA + sg)
    n_tasks = B + sum(int(i.numel()) for _, i, _ in specs)
    depth = fold_depth(n_tasks)
    # |d ell / dx| <= 1; expf, the reciprocal, logf and gamma's rounding to fp32 cost <= 4u + 2u |ell| per term
    e_ell = bx + 4 * U32 + 2 * U32 * np.abs(ell)
    assert_within(mf, ell.mean(), (e_ell.sum() + depth * U32 * np.abs(ell).sum()) / B + U32 * abs(ell.mean()), "mf")
    # ---- d mf / d emb: coef_b = -sig (1 - sig) / ((gamma + sig) B).  fp32 rounds sig to 1 for x > 17, so 1 - sig
    # is known to 2^-25 absolute only (coef = 0 where float64 has 9e-14 / B at x = 30): the floor u / B
    coef = -(sg * sgc) / ((GAMMA + sg) * B)
    dcoef = 8 * U32 * np.abs(coef) + (bx + U32) / B
    w, wd = abs(g_mf) * np.abs(coef), abs(g_mf) * dcoef
    ref = np.zeros_like(E)
    mag = np.zeros_like(E)
    err = np.zeros_like(E)
    c = g_mf * coef
    np.add.at(ref, un, c[:, None] * (Ep - En))
    np.add.at(ref, pn, c[:, None] * Eu)
    np.add.at(ref, nn_, -c[:, None] * Eu)
    for rows, val in ((un, np.abs(Ep) + np.abs(En)), (pn, np.abs(Eu)), (nn_, np.abs(Eu))):
        np.add.at(mag, rows, w[:, None] * val)
        np.add.at(err, rows, wd[:, None] * val)
    mult = max_mult(np.concatenate([un, pn, nn_]))     # atomics into one entry: a chain of that length
    assert_within(emb_d.grad, ref, (mult + 4) * U32 * mag + err, "d emb")
    # ---- regulariser: reg = sum_g sqrt(S_g) / B, S_g = sum of the group's squared rows (padding rows included)
    norms = []
    reg_ref = {k: np.zeros(t.shape) for k, t in tabs.items()}
    reg_mag = {k: np.zeros(t.shape) for k, t in tabs.items()}
    hits = {k: [] for k in tabs}
    s_depth = lanes + 1 + depth
    for k, i, pad in specs:
        T = tabs[k].double().numpy()
        ids = i.reshape(-1).numpy()
        S = float((T[ids] ** 2).sum())
        nrm = math.sqrt(S)
        norms.append(nrm)
        if not ids.size:
            continue                                  # an empty group: norm 0, no gradient
        live = ids[ids != pad]
        sc = g_reg / (B * nrm)
        np.add.at(reg_ref[k], live, sc * T[live])
        np.add.at(reg_mag[k], live, abs(sc) * np.abs(T[live]))
        hits[k].append(live)
    reg_val = sum(norms) / B
    reg_bound = (sum((s_depth / 2 + 2 + len(norms)) * U32 * x for x in norms)) / B + U32 * reg_val
    assert_within(reg, reg_val, reg_bound, "reg")
    for k, t in tabs_d.items():
        used = [key for key, _, _ in specs if key == k]
        if not used:
            assert t.grad is None
            continue
        # sc carries S's relative error (<= s_depth u) halved by the sqrt, plus the division and the product; the
        # atomics into one entry add a chain as long as the number of rows that land there
        mult = max_mult(np.concatenate(hits[k])) if hits[k] else 0
        assert_within(t.grad, reg_ref[k], (s_depth / 2 + 4 + mult) * U32 * reg_mag[k], f"d table {k}")
    if groups == "six":
        assert float(tabs_d["C"].grad[11].abs().max()) == 0.0      # the padding row gets no gradient


# ======================================================================================= BPRLoss / EmbLoss
@pytest.mark.parametrize("n", [1, 31, 1024, 1025, 3_000_000])
def test_bpr_and_emb_loss_modules_vs_fp64(n):
    """The stand-alone kernels behind `BPRLoss` / `EmbLoss` (one block of 1024 threads, each thread strides
    ceil(n / 1024) terms, then two warp folds): the chain is ceil(n / 1024) + 10 additions long."""
    from foodrec_b200.common.loss import BPRLoss, EmbLoss
    gen = torch.Generator().manual_seed(n)
    pos, neg = torch.randn(n, generator=gen) * 3, torch.randn(n, generator=gen) * 3
    for k, s in enumerate([0.0, 30.0, -30.0, 90.0, -90.0][:n]):       # saturated sigmoids (pos - neg exact)
        pos[k], neg[k] = s / 2, -s / 2
    depth = -(-n // 1024) + 10
    pd, nd = pos.cuda().requires_grad_(True), neg.cuda().requires_grad_(True)
    out = BPRLoss()(pd, nd)
    (out * 1.9).backward()
    x = pos.double().numpy() - neg.double().numpy()
    sg, sgc = expit(x), expit(-x)
    ell = -np.log(GAMMA + sg)
    bx = U32 * np.abs(x)                               # pos - neg rounded once
    e_ell = bx + 4 * U32 + 2 * U32 * np.abs(ell)
    assert_within(out, ell.mean(), (e_ell.sum() + depth * U32 * np.abs(ell).sum()) / n + U32 * abs(ell.mean()), "bpr")
    coef = -(sg * sgc) / ((GAMMA + sg) * n) * 1.9
    bound = 9 * U32 * np.abs(coef) + 1.9 * (bx + U32) / n          # floor: fp32 1 - sigmoid, see rank_loss
    assert_within(pd.grad, coef, bound, "d pos")
    assert_within(nd.grad, -coef, bound, "d neg")

    es = [torch.randn(n, generator=gen) * s for s in (0.5, 1.0, 2.0)]
    ed = [e.cuda().requires_grad_(True) for e in es]
    reg = EmbLoss()(*ed)
    (reg.sum() * -0.6).backward()
    e64 = [e.double().numpy() for e in es]
    norms = [math.sqrt(float((e * e).sum())) for e in e64]
    # sqrt of a positive sum: relative error <= (depth + 1) u / 2 + u each; three norms added, then divided
    rel = (depth + 1) / 2 + 1
    assert_within(reg, [sum(norms) / n], [(rel + 3) * U32 * sum(norms) / n], "emb loss")
    for e, ref, nrm in zip(ed, e64, norms):
        g = -0.6 / n * ref / nrm
        assert_within(e.grad, g, (rel + 4) * U32 * np.abs(g), "d emb")


# ================================================================================================ cosine_mean
COS_CASES = [(n, d) for n in (1, 7, 200_000) for d in (4, 33, 64, 512) if (n, d) != (200_000, 512)] + [(20_000, 512)]


@pytest.mark.parametrize("n,d", COS_CASES)
@pytest.mark.parametrize("want", ["both", "A", "T"])
def test_cosine_mean_vs_fp64(n, d, want):
    """`cosine_similarity(A, T[idx]).mean()` against torch in float64: repeated idx, a zero row in A and in T
    (torch clamps each norm at eps = 1e-8, so the gradient there is finite and about 1 / eps), and a gradient for
    A only or T only (the NULL dT / dA paths)."""
    from foodrec_b200 import ops
    if want != "both" and n == 200_000 and d != 64:
        pytest.skip("the NULL-output paths are covered at the other sizes")
    gen = torch.Generator().manual_seed(n + d)
    rows = max(n // 2, 3)
    A = torch.randn(n, d, generator=gen)
    T = torch.randn(rows, d, generator=gen)
    idx = torch.randint(0, rows, (n,), generator=gen)
    A[n // 2] = 0                                     # a zero row in A
    T[idx[-1]] = 0                                    # and one in T
    if n > 3:
        idx[1] = idx[2]                               # repeated idx
    g = 1.7
    A64, T64 = A.double().requires_grad_(want != "T"), T.double().requires_grad_(want != "A")
    ref = torch.nn.functional.cosine_similarity(A64, T64[idx], dim=-1, eps=1e-8)
    (ref.mean() * g).backward()
    Ad = A.cuda().requires_grad_(want != "T")
    Td = T.cuda().requires_grad_(want != "A")
    out = ops.cosine_mean(Ad, Td, idx.cuda())
    (out * g).backward()
    torch.cuda.synchronize()

    a, t = A.double().numpy(), T.double().numpy()[idx.numpy()]
    x = np.maximum(np.linalg.norm(a, axis=1), 1e-8)
    y = np.maximum(np.linalg.norm(t, axis=1), 1e-8)
    cos = ref.detach().numpy()
    cd = -(-d // 32) + 5 + 1                          # a lane's fma chain + the warp butterfly
    # dot: cd u sum|a t| <= cd u |a||t|; each norm: (cd / 2 + 1) u relative; division and product: 2u
    e_cos = cd * U32 * (np.abs(a) * np.abs(t)).sum(1) / (x * y) + (cd + 4) * U32 * np.abs(cos)
    mdepth = -(-n // 1024) + 5 + 32                  # mean_kernel: strided chain, warp fold, 32 warp partials
    assert_within(out, cos.mean(), (e_cos.sum() + mdepth * U32 * np.abs(cos).sum()) / n + U32 * abs(cos.mean()), "mean")
    gn = g / n
    ax, ty = (x > 1e-8)[:, None], (y > 1e-8)[:, None]
    if want != "T":
        # dA = g/n (t / (x y) - c a / x^2): each term to (cd + 6) u, plus c's own error through a / x^2
        mag = gn * (np.abs(t) / (x * y)[:, None] + ax * (np.abs(cos)[:, None] * np.abs(a) / (x * x)[:, None]))
        bound = (cd + 6) * U32 * mag + gn * ax * e_cos[:, None] * np.abs(a) / (x * x)[:, None]
        assert_within(Ad.grad, A64.grad.numpy(), bound, "dA")
    else:
        assert Ad.grad is None
    if want != "A":
        per = gn * (np.abs(a) / (x * y)[:, None] + ty * (np.abs(cos)[:, None] * np.abs(t) / (y * y)[:, None]))
        per_e = gn * ty * e_cos[:, None] * np.abs(t) / (y * y)[:, None]
        mag = np.zeros(T.shape)
        err = np.zeros(T.shape)
        np.add.at(mag, idx.numpy(), per)
        np.add.at(err, idx.numpy(), per_e)
        mult = max_mult(idx.numpy())
        assert_within(Td.grad, T64.grad.numpy(), (cd + 6 + mult) * U32 * mag + err, "dT")
    else:
        assert Td.grad is None


# ================================================================================ gather / scatter-add / pairs
def grid_threads():
    return 16 * num_sms() * 256                       # grid1d's cap in csrc/gather.cu


@pytest.mark.parametrize("d", [4, 12, 64, 2048])
@pytest.mark.parametrize("size", ["empty", "one", "strided"])
def test_gather_and_scatter_add_rows(d, size):
    """Gather is bit-exact; its adjoint (fp32 atomics) is within (k - 1) u sum|g| of the float64 sum of the k
    gradient rows that land on one table row.  "strided": more float4 / float work items than the capped grid has
    threads, so both loops stride."""
    from foodrec_b200 import ops
    n = {"empty": 0, "one": 1, "strided": (3 * grid_threads()) // (2 * (d // 4)) + 3}[size]
    rows = max(n // 3, 5)
    gen = torch.Generator().manual_seed(d + n)
    tab = torch.randn(rows, d, generator=gen)
    idx = torch.randint(0, rows, (n,), generator=gen)      # repeated indices (n >= 3 rows per index on average)
    td = tab.cuda().requires_grad_(True)
    out = ops.gather_rows(td, idx.cuda())
    assert out.shape == (n, d)
    assert torch.equal(out.cpu(), tab[idx])
    g = torch.randn(n, d, generator=gen)
    out.backward(g.cuda())
    ref = np.zeros((rows, d))
    mag = np.zeros((rows, d))
    np.add.at(ref, idx.numpy(), g.double().numpy())
    np.add.at(mag, idx.numpy(), np.abs(g.double().numpy()))
    assert_within(td.grad, ref, max(max_mult(idx.numpy()) - 1, 0) * U32 * mag, "scatter-add")


@pytest.mark.parametrize("d", [1, 33, 64])
@pytest.mark.parametrize("n", [0, 1, 100_003])
def test_pair_scores_vs_fp64(d, n):
    from foodrec_b200 import ops
    gen = torch.Generator().manual_seed(d * 3 + n)
    Ut, It = torch.randn(300, d, generator=gen), torch.randn(500, d, generator=gen)
    user, item = torch.randint(0, 300, (n,), generator=gen), torch.randint(0, 500, (n,), generator=gen)
    out = ops.pair_scores(Ut.cuda(), It.cuda(), user.cuda(), item.cuda())
    assert out.shape == (n,)
    a, b = Ut.double().numpy()[user.numpy()], It.double().numpy()[item.numpy()]
    cd = -(-d // 32) + 5 + 1
    assert_within(out, (a * b).sum(1), cd * U32 * np.abs(a * b).sum(1), "pair scores")


# ================================================================================== sum_rows / spread_rows
def _ptrs(ts):
    return (C.c_void_p * max(len(ts), 1))(*[None if t is None else t.data_ptr() for t in ts])


@pytest.mark.parametrize("n_tabs", [1, 2, 3, 4])
@pytest.mark.parametrize("rows", [0, 1, 777])
@pytest.mark.parametrize("d", [12, 64])
def test_sum_rows_bit_exact(n_tabs, rows, d):
    """out[r] = tab_0[r] + tab_1[r] + ... left to right in fp32 over tables of different heights."""
    L = _lib()
    gen = torch.Generator().manual_seed(n_tabs * 1000 + rows + d)
    tabs = [torch.randn(rows + (0, 5, 17, 3)[v], d, generator=gen) for v in range(n_tabs)]
    tabs_d = [t.cuda() for t in tabs]
    buf = torch.full((rows + 1, d), float("nan"), device="cuda")     # one row past the end must stay untouched
    L.check(L.lib.fr_sum_rows(_ptrs(tabs_d), n_tabs, d, rows, buf.data_ptr(), L.stream_ptr()), "fr_sum_rows")
    ref = tabs[0][:rows].numpy().copy()
    for t in tabs[1:]:
        ref = ref + t[:rows].numpy()                   # numpy float32: one correctly rounded add per table
    out = buf.cpu().numpy()
    assert np.array_equal(out[:rows], ref)
    assert np.isnan(out[rows]).all()


@pytest.mark.parametrize("n_tabs", [1, 2, 3, 4])
@pytest.mark.parametrize("rows", [0, 1, 777])
@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("src_mask", [False, True])
def test_spread_rows_bit_exact(n_tabs, rows, accumulate, src_mask):
    """d_tab_v[r] = g[r] for r < rows and 0 above (accumulate = 0), or d_tab_v[r] += g[r] for r < rows with every
    row >= rows untouched (accumulate = 1); the per-table row masks are written (0) or OR-ed (1) from `src_mask`
    (NULL = every source row active)."""
    L = _lib()
    d = 12
    gen = torch.Generator().manual_seed(n_tabs * 100 + rows + 10 * accumulate + src_mask)
    heights = [rows + (0, 5, 17, 3)[v] for v in range(n_tabs)]
    g = torch.randn(rows, d, generator=gen)
    sm = (torch.rand(rows, generator=gen) < 0.5).to(torch.uint8)
    if src_mask:
        g[sm == 0] = 0                                # the mask's promise: inactive rows of g are zero
    dst = [torch.randn(h, d, generator=gen) for h in heights]
    masks = [(torch.rand(h, generator=gen) < 0.5).to(torch.uint8) for h in heights]
    dst_d, masks_d = [t.cuda() for t in dst], [m.cuda() for m in masks]
    # device copies held until the call has run (a temporary's block could be handed to the next copy)
    g_d = g.cuda() if rows else torch.zeros(1, d, device="cuda")     # rows = 0: a valid pointer that is never read
    sm_d = sm.cuda() if (src_mask and rows) else None
    rows_total = (C.c_int64 * n_tabs)(*heights)
    L.check(L.lib.fr_spread_rows(g_d.data_ptr(), d, rows, _ptrs(dst_d), rows_total, n_tabs, accumulate,
                                 None if sm_d is None else sm_d.data_ptr(), _ptrs(masks_d), L.stream_ptr()),
            "fr_spread_rows")
    torch.cuda.synchronize()
    src_m = sm.numpy() if src_mask else np.ones(rows, np.uint8)
    for v in range(n_tabs):
        ref = dst[v].numpy().copy()
        mref = masks[v].numpy().copy()
        if accumulate:
            ref[:rows] = ref[:rows] + g.numpy()
            mref[:rows] |= src_m
        else:
            ref[:] = 0
            ref[:rows] = g.numpy()
            mref[:] = 0
            mref[:rows] = src_m
        assert np.array_equal(dst_d[v].cpu().numpy(), ref), f"table {v}"
        assert np.array_equal(masks_d[v].cpu().numpy(), mref), f"mask {v}"


# ============================================================================================= csr_from_coo
@pytest.mark.parametrize("n_rows", [1, 1023, 1024, 1025, 5000])
@pytest.mark.parametrize("nnz", [0, 7, 50_000])
def test_csr_from_coo_vs_bincount(n_rows, nnz):
    """Row pointers of an unsorted COO with the first, the last and a middle row empty (the scan covers several
    1024-row chunks from n_rows = 1025 on), against np.bincount + cumsum, exactly."""
    L = _lib()
    gen = np.random.default_rng(n_rows * 7 + nnz)
    if n_rows >= 3:
        live = np.setdiff1d(np.arange(1, n_rows - 1), [n_rows // 2])
        rows = gen.choice(live, size=nnz)
    else:
        rows = np.zeros(nnz, dtype=np.int64)
    rows = rows.astype(np.int64)
    row_ptr = torch.full((n_rows + 1,), -7, dtype=torch.int32, device="cuda")
    scratch = torch.full((n_rows,), 123, dtype=torch.int32, device="cuda")
    coo = torch.from_numpy(rows).cuda()
    L.check(L.lib.fr_csr_from_coo(coo.data_ptr() if nnz else None, nnz, n_rows, row_ptr.data_ptr(), scratch.data_ptr(),
                                  L.stream_ptr()), "fr_csr_from_coo")
    ref = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n_rows))])
    assert np.array_equal(row_ptr.cpu().numpy(), ref)
