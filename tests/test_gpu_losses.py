"""GPU parity of the fused loss kernels against reference goldens and the oracle."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from test_gpu_clussl import close

pytestmark = pytest.mark.gpu


def test_rank_loss_matches_reference_modules():
    from foodrec_b200 import ops
    from oracle import losses
    torch.manual_seed(3)
    U, I, d, B = 50, 70, 64, 97
    emb = (torch.randn(U + I, d) * 0.3).requires_grad_(True)
    uw, iw = (torch.randn(U, d) * 0.2).requires_grad_(True), (torch.randn(I, d) * 0.2).requires_grad_(True)
    gw = (torch.randn(11, d) * 0.2).requires_grad_(True)
    u, p, n = torch.randint(0, U, (B,)), torch.randint(0, I, (B,)), torch.randint(0, I, (B,))
    ing = torch.randint(0, 11, (B, 20))
    mf = losses.bpr_from_tables(emb[:U], emb[U:], u, p, n)
    gpad = torch.nn.functional.embedding(ing, gw, padding_idx=10)
    reg = losses.emb_loss(uw[u], iw[p], iw[n], gpad)
    (mf * 0.7 + reg.sum() * 1.3).backward()
    c = lambda t: t.detach().cuda().requires_grad_(True)
    emb_d, uw_d, iw_d, gw_d = c(emb), c(uw), c(iw), c(gw)
    mf_d, reg_d = ops.rank_loss(emb_d, U, u.cuda(), p.cuda(), n.cuda(),
                                [(uw_d, u.cuda()), (iw_d, p.cuda()), (iw_d, n.cuda()), (gw_d, ing.cuda(), 10)],
                                reg_den=float(B))
    (mf_d * 0.7 + reg_d * 1.3).backward()
    close(mf_d, mf.detach().numpy())
    close(reg_d, reg.detach().numpy()[0])
    for a, b in ((emb_d, emb), (uw_d, uw), (iw_d, iw), (gw_d, gw)):
        close(a.grad, b.grad.numpy(), rtol=2e-5)
    assert float(gw_d.grad[10].abs().max()) == 0.0  # padding row gets no gradient


def test_bpr_and_embloss_golden():
    from foodrec_b200 import ops
    g = load_golden("primitives.npz")
    # BPR on scores: build rows whose dot products reproduce the golden scores exactly
    pos, neg = torch.from_numpy(g["bpr/pos"]), torch.from_numpy(g["bpr/neg"])
    B = pos.numel()
    emb = torch.zeros(1 + 2 * B, 32)
    emb[0, 0] = 1.0
    emb[1:1 + B, 0] = pos
    emb[1 + B:, 0] = neg
    z = torch.zeros(B, dtype=torch.long)
    e1, e2, e3 = (torch.from_numpy(g[k]) for k in ("emb/e1", "emb/e2", "emb/e3"))
    embs = [torch.nn.functional.pad(e, (0, 0, 0, 0))[:, :].contiguous() for e in (e1, e2, e3)]
    tabs = [torch.cat([e[:, :32], e[:, 32:]], 0).cuda() for e in embs]  # [2n, 32]: same Frobenius norm
    mf, reg = ops.rank_loss(emb.cuda(), 1, z.cuda(), torch.arange(B).cuda(), (torch.arange(B) + B).cuda(),
                            [(t, torch.arange(t.shape[0]).cuda()) for t in tabs], reg_den=float(e3.shape[0]))
    close(mf, g["bpr/out"])
    close(reg, g["emb/out"][0])


def test_loss_modules_called_directly_match_reference_golden():
    """`model.mf_loss(pos, neg)` / `model.reg_loss(e1, e2, e3)` as reference code calls them (FoodRec/common/loss.py:31-34,
    44-50): values against the reference-run golden, gradients against the same formula in torch-CPU."""
    from foodrec_b200.common.loss import BPRLoss, EmbLoss
    g = load_golden("primitives.npz")
    pos, neg = torch.from_numpy(g["bpr/pos"]), torch.from_numpy(g["bpr/neg"])
    pd, nd = pos.cuda().requires_grad_(True), neg.cuda().requires_grad_(True)
    out = BPRLoss()(pd, nd)
    close(out, g["bpr/out"])
    out.backward()
    pc, nc = pos.clone().requires_grad_(True), neg.clone().requires_grad_(True)
    (-torch.log(1e-10 + torch.sigmoid(pc - nc)).mean()).backward()
    close(pd.grad, pc.grad.numpy(), rtol=2e-5)
    close(nd.grad, nc.grad.numpy(), rtol=2e-5)
    es = [torch.from_numpy(g[k]) for k in ("emb/e1", "emb/e2", "emb/e3")]
    ed = [e.cuda().requires_grad_(True) for e in es]
    reg = EmbLoss()(*ed)
    assert tuple(reg.shape) == (1,)
    close(reg, g["emb/out"])
    (reg.sum() * 1.7).backward()
    ec = [e.clone().requires_grad_(True) for e in es]
    (sum(torch.norm(e, p=2) for e in ec) / ec[-1].shape[0] * 1.7).backward()
    for a, b in zip(ed, ec):
        close(a.grad, b.grad.numpy(), rtol=2e-5)
    with pytest.raises(Exception):
        BPRLoss()(pos, neg)          # CPU tensors: no fallback


def test_distance_correlation_golden_and_grad():
    """Against the reference golden (fp32, CPU) and against the same formula evaluated in fp64.

    The reference's fp32 result carries noise of its own: its diagonal
    D_ii = sqrt(max(r_i - 2 x_i.x_i + r_i, 0) + 1e-8) is BLAS rounding (1e-4..3e-4 instead of 1e-4),
    the diagonal carries ~n/(n + 0.01 n^2) of dcov_xx, and autograd multiplies that noise by
    1/(2 D_ii) = 5000 before it cancels.  So: tight bound against fp64, loose against fp32."""
    from foodrec_b200 import ops
    from oracle import losses
    g = load_golden("primitives.npz")
    x = torch.from_numpy(g["dcor/x"]).cuda().requires_grad_(True)
    y = torch.from_numpy(g["dcor/y"]).cuda().requires_grad_(True)
    d = ops.correlation_distance(x, y)
    d.sum().backward()
    close(d, g["dcor/out"].reshape(1), rtol=1e-4)
    close(x.grad, g["dcor/gx"], rtol=3e-3)
    close(y.grad, g["dcor/gy"], rtol=3e-3)
    x64 = torch.from_numpy(g["dcor/x"]).double().requires_grad_(True)
    y64 = torch.from_numpy(g["dcor/y"]).double().requires_grad_(True)
    d64 = losses.correlation_distance(x64, y64)
    d64.sum().backward()
    close(d, d64.detach().numpy().reshape(1), rtol=1e-5)
    close(x.grad, x64.grad.numpy(), rtol=1e-4)
    close(y.grad, y64.grad.numpy(), rtol=1e-4)


THREE = ((0, 1), (0, 2), (2, 1))
DCOR_CASES = ([(100, 64, THREE, None), (1024, 64, THREE, None)]
              # d = 32 instantiations; n % 4 != 0 takes the scalar Dm stores and W fetches, n < 64 a partial tile
              + [(n, 32, THREE, None) for n in (1, 2, 3, 63, 65, 97, 2048)]
              + [(97, 32, ((0, 1),), None),         # two views, one pair
                 (65, 64, ((1, 0),), None),         # a reversed pair
                 (63, 64, THREE, 1)])               # view 1 needs no gradient (its d_tab is NULL)


def _dcor_id(case):
    n, d, pairs, frozen = case
    if d == 64 and pairs == THREE and frozen is None and n in (100, 1024):
        return str(n)                                     # the original cases keep their ids
    return f"{n}-d{d}-" + "".join(f"{a}{b}" for a, b in pairs) + ("" if frozen is None else f"-frozen{frozen}")


@pytest.mark.parametrize("n,d,pairs,frozen", DCOR_CASES, ids=[_dcor_id(c) for c in DCOR_CASES])
def test_three_view_dcor_vs_oracle(n, d, pairs, frozen):
    from foodrec_b200 import ops
    from oracle import losses
    torch.manual_seed(n)
    rows = 3000
    V = 1 + max(max(ab) for ab in pairs)
    tabs = [(torch.randn(rows + k * 10, d) * 0.1) for k in range(V)]
    idx = torch.randint(0, rows, (n,))
    if n > 17:
        idx[5] = idx[17]  # duplicate rows in the batch (same item as pos and neg)
    w = torch.tensor([0.3, 1.0, -0.5][:len(pairs)] if len(pairs) > 1 else [-0.7])   # per-term upstream gradients
    refs = {}
    for dt in (torch.float32, torch.float64):
        ts = [t.detach().clone().to(dt).requires_grad_(k != frozen) for k, t in enumerate(tabs)]
        views = [t[idx] for t in ts]
        ref = torch.stack([losses.correlation_distance(views[a], views[b]) for a, b in pairs]).reshape(-1)
        (ref * w.to(dt)).sum().backward()
        refs[dt] = (ref.detach().numpy(), [None if t.grad is None else t.grad.numpy() for t in ts])
    tabs_d = [t.cuda().requires_grad_(k != frozen) for k, t in enumerate(tabs)]
    out = ops.dcor_terms(tabs_d, idx.cuda(), list(pairs))
    (out * w.cuda()).sum().backward()
    # n <= 2: two points are always perfectly distance-correlated, so each term is 1 up to the 1e-8 / 1e-10
    # stabilisers and its float64 gradient is O(1e-8) (exactly 0 at n = 1).  Against distances of order 1 fp32 keeps
    # none of those stabilisers (half an ulp of 1 is 6e-8), so the kernel's gradient there is the cancellation
    # noise of a few u times the O(1) partial derivatives it sums: the floor 1e-5 sum|w| is two orders above that.
    atol = 1e-5 * float(w.abs().sum()) if n <= 2 else 0.0
    close(out, refs[torch.float64][0], rtol=1e-5)
    original = d == 64 and pairs == THREE and frozen is None
    if original:
        close(out, refs[torch.float32][0], rtol=1e-4)
    for k, (td, g64, g32) in enumerate(zip(tabs_d, refs[torch.float64][1], refs[torch.float32][1])):
        if k == frozen:
            assert td.grad is None
            continue
        close(td.grad, g64, rtol=1e-4, atol=atol)
        if original:
            close(td.grad, g32, rtol=1e-2)  # the fp32 autograd reference is itself ~5e-3 noisy at n=1024 (see above)


def test_dcor_backward_into_aliased_gradient():
    """`fr_dcor_bwd` may be handed the same gradient table for two views (the header allows aliasing): the atomics
    then add both views' gradients into it.  Views 0 and 1 are two tables of one height sharing d_tab, view 2 has
    its own; compared with the float64 sum of the two views' gradients."""
    from foodrec_b200 import ops
    from oracle import losses
    torch.manual_seed(21)
    n, rows = 97, 500
    tabs = [torch.randn(rows, 32) * 0.1, torch.randn(rows, 32) * 0.1, torch.randn(rows + 9, 32) * 0.1]
    idx = torch.randint(0, rows, (n,))
    w = torch.tensor([0.3, 1.0, -0.5])
    ts = [t.double().requires_grad_(True) for t in tabs]
    views = [t[idx] for t in ts]
    ref = torch.stack([losses.correlation_distance(views[a], views[b]) for a, b in THREE]).reshape(-1)
    (ref * w.double()).sum().backward()
    tabs_d = [t.cuda() for t in tabs]
    idx_d = idx.cuda()
    out, state = ops._dcor_forward(tabs_d, idx_d, list(THREE), 1.0)
    close(out[:3], ref.detach().numpy(), rtol=1e-5)
    shared, own = torch.zeros(rows, 32, device="cuda"), torch.zeros(rows + 9, 32, device="cuda")
    ops._dcor_backward(tabs_d, idx_d, list(THREE), state, w.cuda(), [shared, shared, own])
    close(shared, (ts[0].grad + ts[1].grad).numpy(), rtol=1e-4)
    close(own, ts[2].grad.numpy(), rtol=1e-4)


def test_info_nce_golden():
    from foodrec_b200 import ops
    g = load_golden("primitives.npz")
    h = torch.from_numpy(g["nce/h"]).cuda().requires_grad_(True)
    c = ops.info_nce(h)
    c.backward()
    close(c, g["nce/out"])
    close(h.grad, g["nce/gh"], rtol=1e-4)


NCE_ORIGINAL = [(1024, 0.5, True, 64), (130, 0.2, True, 64), (257, 0.5, False, 64)]


NCE_CASES = NCE_ORIGINAL + [
    (1024, 0.5, True, 32), (257, 0.5, False, 32),         # the d = 32 instantiations
    (2, 0.5, True, 64), (3, 2.0, False, 32),              # b = 1
    (66, 0.05, True, 32), (131, 2.0, True, 64),           # b = 33, 65
    (1400, 0.05, True, 64), (1401, 2.0, False, 32),       # b = 700
]


@pytest.mark.parametrize("rows,temperature,norm,d", NCE_CASES,     # the original cases keep their ids
                         ids=["-".join(map(str, c[:3] if c in NCE_ORIGINAL else c)) for c in NCE_CASES])
def test_info_nce_vs_oracle(rows, temperature, norm, d):
    """Fused NT-Xent (one Gram matrix) vs the reference's four-block formulation restated in the oracle, in float64
    (and in fp32 for the original cases), including an odd trailing row (ignored, zero gradient), the
    un-normalised variant, small and large temperatures and an upstream gradient != 1."""
    from foodrec_b200 import ops
    from oracle import losses
    torch.manual_seed(rows)
    g = 1.7
    h = (torch.randn(rows, d) * (1.0 if norm else 0.3)).requires_grad_(True)
    ref = losses.info_nce(h, temperature=temperature, hidden_norm=norm)
    (ref * g).backward()
    h64 = h.detach().double().requires_grad_(True)
    ref64 = losses.info_nce(h64, temperature=temperature, hidden_norm=norm)
    (ref64 * g).backward()
    hd = h.detach().cuda().requires_grad_(True)
    out = ops.info_nce(hd, temperature=temperature, hidden_norm=norm)
    (out * g).backward()
    # b = 1: after the mask each row's only logit is its positive, so loss and gradient are exactly 0 in exact
    # arithmetic; a logsumexp rounded by an ulp of |G| <= 1 / temperature would leave ~1e-7, hence the floor
    atol = 1e-6 * g if rows // 2 == 1 else 0.0
    close(out, ref64.detach().numpy(), rtol=1e-5, atol=atol)
    close(hd.grad, h64.grad.numpy(), rtol=1e-4, atol=atol)
    if (rows, temperature, norm, d) in NCE_ORIGINAL:
        close(out, ref.detach().numpy())
        close(hd.grad, h.grad.numpy(), rtol=2e-5)


def test_cosine_mean_vs_torch():
    """HealthRec's KD cosine term: fused gather + cosine + mean vs `F.cosine_similarity(A, T[idx]).mean()`."""
    from foodrec_b200 import ops
    torch.manual_seed(8)
    A = torch.randn(1024, 64).requires_grad_(True)
    T = torch.randn(5000, 64).requires_grad_(True)
    idx = torch.randint(0, 5000, (1024,))
    idx[3] = idx[9]
    ref = torch.nn.functional.cosine_similarity(A, T[idx], dim=-1).mean()
    (ref * 1.7).backward()
    Ad, Td = A.detach().cuda().requires_grad_(True), T.detach().cuda().requires_grad_(True)
    out = ops.cosine_mean(Ad, Td, idx.cuda())
    (out * 1.7).backward()
    close(out, ref.detach().numpy())
    close(Ad.grad, A.grad.numpy(), rtol=2e-5)
    close(Td.grad, T.grad.numpy(), rtol=2e-5)
