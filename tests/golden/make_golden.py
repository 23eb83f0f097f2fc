"""Generate the golden fixtures in this directory by EXECUTING THE REFERENCE (CPU, this container).

Run from the repo root:  python tests/golden/make_golden.py
Needs /root/reference (read-only mount); the GPU box does not have it, which is why the outputs are
committed.  Two compatibility shims are applied, neither touching arithmetic (SURVEY.md 8c):
scipy >= 1.13 dropped the private `dok_matrix._update`, and `matplotlib` is not installed.
"""
import os
import sys
import types

import numpy as np
import scipy.sparse as sp
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")

torch.set_num_threads(10)      # fp32 reductions depend on it; tests/test_oracle_golden.py runs with the same count
sp.dok_matrix._update = lambda self, d: [self.__setitem__(k, v) for k, v in d.items()]
_m, _mp = types.ModuleType("matplotlib"), types.ModuleType("matplotlib.pyplot")
_m.pyplot = _mp
sys.modules["matplotlib"], sys.modules["matplotlib.pyplot"] = _m, _mp

sys.path.insert(0, ROOT)
from oracle.schgn import install_pyg_stub  # noqa: E402

install_pyg_stub()  # torch_geometric is not installable offline: GCNConv alone is a restatement (oracle/schgn.py)

from FoodRec.common.loss import BPRLoss, EmbLoss  # noqa: E402
from FoodRec.common.trainer import metrics_by_user, get_auc_fast  # noqa: E402
from FoodRec.models.cikm_model import CIKM_Model  # noqa: E402
from FoodRec.models.lightgcn import LightGCN  # noqa: E402
from FoodRec.models.pricai_modelx import PRICAI_ModelX  # noqa: E402
from FoodRec.models.schgn import SCHGN  # noqa: E402
from FoodRec.utils import utils as ref_utils  # noqa: E402
from FoodRec.utils.topk_evaluator import TopKEvaluator  # noqa: E402

import foodrec_b200  # noqa: E402
from foodrec_b200.synth import make_dataset, sample_train_batches  # noqa: E402


class Cfg(dict):
    """Missing keys read as None, like FoodRec/utils/configurator.py:121-125."""

    def __getitem__(self, k):
        return self.get(k)


BASE = dict(device="cpu", embedding_size=64, train_batch_size=64, is_multimodal_model=True, end2end=False,
            use_health_level_multi_hot=True, num_attention_heads=2, num_hidden_layers=2,
            attention_probs_dropout_prob=0.0, hidden_act="gelu", metrics=["Recall", "NDCG", "Precision", "MAP"],
            topk=[5, 10, 20, 50])
CFGS = {
    "CIKM_Model": dict(n_layers=2, ui_layers=1, reg_weight=0.5, loss_kd=0.05, loss_health=0.1, kd_threshold=0.4),
    "PRICAI_ModelX": dict(n_ri_layers=2, n_mm_layers=1, n_ui_layers=1, reg_weight=0.01, loss_cl=0.1, knn_k=10,
                          mm_image_weight=0.1),
    "LightGCN": dict(n_layers=2, reg_weight=0.1),
    "SCHGN": dict(inner_size=256, hidden_dropout_prob=0.5, attention_probs_dropout_prob=0.5, regs=0.01, reg_image=1,
                  reg_w=0.05, reg_g=0.01, reg_health=0.01, ssl=0.008, SCHGN_ssl=True, neg_sample_num=4),
}


def coo_arrays(t):
    t = t.coalesce() if not t.is_coalesced() else t
    return t._indices().numpy().astype(np.int64), t._values().numpy().astype(np.float32)


def raw_coo(t):
    # reference tensors are flagged uncoalesced but hold sorted, duplicate-free entries
    return t._indices().numpy().astype(np.int64), t._values().numpy().astype(np.float32)


def to_t(batch):
    out = {}
    for k, v in batch.items():
        out[k] = torch.from_numpy(np.asarray(v))
    return out


def sd_np(model):
    return {"sd/" + k: v.detach().numpy() for k, v in model.state_dict().items()}


def grads_np(model, names):
    g = {}
    for n, p in model.named_parameters():
        if n in names and p.grad is not None:
            g["grad/" + n] = p.grad.detach().numpy().copy()
    return g


SCALE_ROWS = 256      # sampled rows per table in the larger-scale goldens (whole tables would be tens of MB)


def clussl_at_scale(scale):
    """The reference's CLUSSL (`PRICAI_ModelX`) executed on the synthetic C1 / Foodcom-scale C3 data (BASELINE.json
    configs[0] / configs[2] sizes): one batch of 512 from the seed-999 initial state.  Stored: every loss term (fp64
    print of the fp32 values), `SCALE_ROWS` sampled rows of each forward table and of each parameter gradient (the rows
    the batch touches first), the batch, and sampled rows of the initial parameters (so a test can verify it starts
    from the same state without shipping the tables)."""
    ds = make_dataset(scale)
    batch = sample_train_batches(ds, 512, 1, seed=3)[0]
    cfg = Cfg({**BASE, **CFGS["PRICAI_ModelX"], "n_cluster": ds.cfg.n_cluster, "train_batch_size": 512})
    torch.manual_seed(999)
    m = PRICAI_ModelX(cfg, ds)
    rng = np.random.default_rng(17)
    g = {}
    names = ("user_embedding.weight", "item_embedding.weight", "ingre_embedding.weight",
             "image_prototype_embedding.weight", "text_prototype_embedding.weight")
    touched = {"user_embedding.weight": np.unique(batch["u_id"]),
               "item_embedding.weight": np.unique(np.concatenate([batch["pos_i_id"], batch["neg_i_id"]]))}
    params = dict(m.named_parameters())
    rows = {}
    for k in names:
        n = params[k].shape[0]
        t = touched.get(k, np.empty(0, np.int64))[:SCALE_ROWS // 2]
        rows[k] = np.unique(np.concatenate([t, rng.choice(n, size=min(n, SCALE_ROWS - t.size), replace=False)]))
        g[f"rows/{k}"] = rows[k]
        g[f"sd_rows/{k}"] = params[k].detach().numpy()[rows[k]].copy()
        g[f"sd_sum/{k}"] = np.array(params[k].detach().double().sum().item())
    ua, ia, (vi, vt, vg) = m.forward()
    g["fwd/user_all"] = ua.detach().numpy()[rows["user_embedding.weight"]].copy()
    g["fwd/item_all"] = ia.detach().numpy()[rows["item_embedding.weight"]].copy()
    g["fwd/item_image"] = vi.detach().numpy()[rows["item_embedding.weight"]].copy()
    g["fwd/item_text"] = vt.detach().numpy()[rows["item_embedding.weight"]].copy()
    g["fwd/item_ingre"] = vg.detach().numpy()[rows["item_embedding.weight"]].copy()
    m.zero_grad()
    losses = m.calculate_loss(to_t(batch))
    sum(losses).backward()
    g["loss"] = np.array([float(x) for x in losses], dtype=np.float64)
    for k in names:
        g[f"grad/{k}"] = params[k].grad.detach().numpy()[rows[k]].copy()
        g[f"grad_absmax/{k}"] = np.array(float(params[k].grad.abs().max()))
    for k in ("u_id", "pos_i_id", "neg_i_id"):
        g[f"batch/{k}"] = batch[k]
    np.savez_compressed(os.path.join(HERE, f"clussl_{scale.lower()}.npz"), **g)
    return len(g)


def healthrec_c1():
    """BASELINE.json configs[0]: the reference's HealthRec (`CIKM_Model`) executed on the synthetic C1 data (5 000 users,
    3 000 items, 50 000 interactions, d = 64, 2 + 1 layers) on the CPU: one batch of 512 from the seed-999 initial state,
    transformer dropout off (`eval()`).  Stored like `clussl_at_scale`: loss terms, sampled rows of the forward tables,
    of the table gradients and of the initial parameters, the two projection gradients in full, the batch."""
    ds = make_dataset("C1")
    batch = sample_train_batches(ds, 512, 1, seed=3)[0]
    cfg = Cfg({**BASE, **CFGS["CIKM_Model"], "train_batch_size": 512})
    torch.manual_seed(999)
    m = CIKM_Model(cfg, ds)
    m.eval()
    rng = np.random.default_rng(19)
    params = dict(m.named_parameters())
    tables = ("user_embedding.weight", "item_embedding.weight", "ingre_embedding.weight")
    touched = {"user_embedding.weight": np.unique(batch["u_id"]),
               "item_embedding.weight": np.unique(np.concatenate([batch["pos_i_id"], batch["neg_i_id"]]))}
    g, rows = {}, {}
    for k in tables:
        n = params[k].shape[0]
        t = touched.get(k, np.empty(0, np.int64))[:SCALE_ROWS // 2]
        rows[k] = np.unique(np.concatenate([t, rng.choice(n, size=min(n, SCALE_ROWS - t.size), replace=False)]))
        g[f"rows/{k}"] = rows[k]
        g[f"sd_rows/{k}"] = params[k].detach().numpy()[rows[k]].copy()
    for k, v in m.state_dict().items():
        if v.dtype.is_floating_point:
            g[f"sd_sum/{k}"] = np.array(v.double().sum().item())
    ua, ia, ing = m.forward()
    g["fwd/user_all"] = ua.detach().numpy()[rows["user_embedding.weight"]].copy()
    g["fwd/item_all"] = ia.detach().numpy()[rows["item_embedding.weight"]].copy()
    ing_rows = rows["ingre_embedding.weight"][rows["ingre_embedding.weight"] < ing.shape[0]]
    g["rows/ingre_ir"] = ing_rows
    g["fwd/ingre_ir"] = ing.detach().numpy()[ing_rows].copy()
    m.zero_grad()
    losses = m.calculate_loss(to_t(batch))
    sum(losses).backward()
    g["loss"] = np.array([float(x) for x in losses], dtype=np.float64)
    for k in tables:
        g[f"grad/{k}"] = params[k].grad.detach().numpy()[rows[k]].copy()
        g[f"grad_absmax/{k}"] = np.array(float(params[k].grad.abs().max()))
    for k in ("image_trs.weight", "text_trs.weight"):
        g[f"grad_full/{k}"] = params[k].grad.detach().numpy().copy()
    for k, v in batch.items():
        g[f"batch/{k}"] = np.asarray(v)
    np.savez_compressed(os.path.join(HERE, "healthrec_c1.npz"), **g)
    return len(g)


def schgn_c1():
    """The reference's SCHGN class executed on the synthetic C1 data (GCNConv from oracle/schgn.py, dropout = identity):
    one batch of 256 from the seed-999 initial state -- loss terms, every small parameter's gradient in full, sampled
    rows of the table gradients and of the GCN output, full-sort scores of three users."""
    ds = make_dataset("C1")
    cfg = Cfg({**BASE, **CFGS["SCHGN"], "train_batch_size": 256})
    torch.manual_seed(999)
    m = SCHGN(cfg, ds)
    m.eval()
    real_dropout = torch.nn.functional.dropout
    torch.nn.functional.dropout = lambda x, p=0.5, training=True, inplace=False: x
    rng = np.random.default_rng(23)
    g = {}
    for k, v in m.state_dict().items():
        if v.dtype.is_floating_point:
            g[f"sd_sum/{k}"] = np.array(v.double().sum().item())
    x = torch.cat([m.user_embed, m.item_embed, m.ingre_embed_first, m.health_embed], 0)
    gcn = m.new_gcn(x, torch.cat([m.g2i_edges, m.i2u_edges], 0).t().contiguous()).detach().numpy()
    g["rows/gcn"] = np.sort(rng.choice(gcn.shape[0], size=SCALE_ROWS, replace=False))
    g["gcn/out"] = gcn[g["rows/gcn"]].copy()
    batch = sample_train_batches(ds, 256, 1, seed=3, schgn=True)[0]
    m.zero_grad()
    losses = m.calculate_loss(to_t(batch))
    sum(losses).backward()
    g["loss"] = np.array([float(x) for x in losses], dtype=np.float64)
    for n_, p_ in m.named_parameters():
        if p_.grad is None:
            continue
        gr = p_.grad.detach().numpy()
        if gr.size <= 64 * 256:
            g[f"grad_full/{n_}"] = gr.copy()
        else:
            rows = np.sort(rng.choice(gr.shape[0], size=min(SCALE_ROWS, gr.shape[0]), replace=False))
            g[f"rows/{n_}"], g[f"grad/{n_}"] = rows, gr[rows].copy()
            g[f"grad_absmax/{n_}"] = np.array(float(np.abs(gr).max()))
    for k in ("masked_ingre_seq", "neg_ingre_seq", "u_id"):
        g[f"batch/{k}"] = np.asarray(batch[k])
    with torch.no_grad():
        for u in (0, 7, 4999):
            g[f"full_sort/{u}"] = m.full_sort_predict({"u_id": torch.tensor([u])}).numpy()
    torch.nn.functional.dropout = real_dropout
    np.savez_compressed(os.path.join(HERE, "schgn_c1.npz"), **g)
    return len(g)


def lightgcn_c1():
    """The reference's LightGCN executed on the synthetic C1 data: one batch of 512 from the seed-999 initial state."""
    ds = make_dataset("C1")
    batch = sample_train_batches(ds, 512, 1, seed=3)[0]
    cfg = Cfg({**BASE, **CFGS["LightGCN"], "train_batch_size": 512})
    torch.manual_seed(999)
    m = LightGCN(cfg, ds)
    rng = np.random.default_rng(29)
    g = {}
    for k, v in m.state_dict().items():
        if v.dtype.is_floating_point:
            g[f"sd_sum/{k}"] = np.array(v.double().sum().item())
    ru = np.unique(np.concatenate([np.unique(batch["u_id"])[:SCALE_ROWS // 2], rng.choice(ds.n_users, SCALE_ROWS // 2, replace=False)]))
    ri = np.unique(np.concatenate([np.unique(batch["pos_i_id"])[:SCALE_ROWS // 2], rng.choice(ds.n_items, SCALE_ROWS // 2, replace=False)]))
    g["rows/user"], g["rows/item"] = ru, ri
    ua, ia = m.forward()
    g["fwd/user_all"], g["fwd/item_all"] = ua.detach().numpy()[ru].copy(), ia.detach().numpy()[ri].copy()
    m.zero_grad()
    losses = m.calculate_loss(to_t(batch))
    sum(losses).backward()
    g["loss"] = np.array([float(x) for x in losses], dtype=np.float64)
    params = dict(m.named_parameters())
    g["grad/user_embedding.weight"] = params["user_embedding.weight"].grad.detach().numpy()[ru].copy()
    g["grad_absmax/user_embedding.weight"] = np.array(float(params["user_embedding.weight"].grad.abs().max()))
    for k in ("image_trs.weight", "image_trs.bias"):
        g[f"grad_full/{k}"] = params[k].grad.detach().numpy().copy()
    for k in ("u_id", "pos_i_id", "neg_i_id"):
        g[f"batch/{k}"] = batch[k]
    np.savez_compressed(os.path.join(HERE, "lightgcn_c1.npz"), **g)
    return len(g)


def main():
    torch.manual_seed(999)
    np.random.seed(999)
    ds = make_dataset("mini")
    batches = sample_train_batches(ds, 64, 2, seed=11)
    out = {}

    # ---------------- CLUSSL
    cfg = Cfg({**BASE, **CFGS["PRICAI_ModelX"], "n_cluster": ds.cfg.n_cluster})
    torch.manual_seed(999)
    m = PRICAI_ModelX(cfg, ds)
    g = sd_np(m)
    for name in ("norm_adj_matrix", "image_norm_adj", "text_norm_adj", "ingre_norm_adj"):
        idx, val = raw_coo(getattr(m, name))
        g[f"adj/{name}/idx"], g[f"adj/{name}/val"] = idx, val
    ua, ia, (vi, vt, vg) = m.forward()
    g.update({"fwd/user_all": ua.detach().numpy(), "fwd/item_all": ia.detach().numpy(),
              "fwd/item_image": vi.detach().numpy(), "fwd/item_text": vt.detach().numpy(),
              "fwd/item_ingre": vg.detach().numpy()})
    for b, batch in enumerate(batches):
        m.zero_grad()
        losses = m.calculate_loss(to_t(batch))
        sum(losses).backward()
        g[f"loss/{b}"] = np.array([float(x) for x in losses], dtype=np.float64)
        for k, v in grads_np(m, {"user_embedding.weight", "item_embedding.weight", "ingre_embedding.weight",
                                  "image_prototype_embedding.weight",
                                  "text_prototype_embedding.weight"}).items():
            g[f"{k}/{b}"] = v
        for k in ("u_id", "pos_i_id", "neg_i_id"):
            g[f"batch/{b}/{k}"] = batch[k]
    cand = np.concatenate([np.array(ds.validRatings[3]), np.arange(40, 90)])
    sc = m.inference_fast({"user_input": torch.full((len(cand),), 3), "item_input": torch.from_numpy(cand)}, ua, ia)
    g["infer/cand"], g["infer/scores"] = cand, sc.detach().numpy()
    np.savez_compressed(os.path.join(HERE, "clussl_mini.npz"), **g)
    out["clussl"] = len(g)

    # ---------------- SCHGN (reference class executed; GCNConv from oracle/schgn.py; dropout = identity)
    cfg = Cfg({**BASE, **CFGS["SCHGN"]})
    torch.manual_seed(999)
    m = SCHGN(cfg, ds)
    m.eval()
    real_dropout = torch.nn.functional.dropout
    torch.nn.functional.dropout = lambda x, p=0.5, training=True, inplace=False: x
    g = sd_np(m)
    g["edges/g2i"], g["edges/i2u"] = m.g2i_edges.numpy(), m.i2u_edges.numpy()
    x = torch.cat([m.user_embed, m.item_embed, m.ingre_embed_first, m.health_embed], 0)
    g["gcn/out"] = m.new_gcn(x, torch.cat([m.g2i_edges, m.i2u_edges], 0).t().contiguous()).detach().numpy()
    sbatches = sample_train_batches(ds, 64, 2, seed=11, schgn=True)
    for b, batch in enumerate(sbatches):
        m.zero_grad()
        losses = m.calculate_loss(to_t(batch))
        sum(losses).backward()
        g[f"loss/{b}"] = np.array([float(x) for x in losses], dtype=np.float64)
        for n_, p_ in m.named_parameters():
            if p_.grad is not None:
                g[f"grad/{n_}/{b}"] = p_.grad.detach().numpy().copy()
        for k in ("masked_ingre_seq", "pos_ingre_seq", "neg_ingre_seq"):
            g[f"batch/{b}/{k}"] = batch[k]
    with torch.no_grad():
        for u in (0, 7, 200):
            g[f"full_sort/{u}"] = m.full_sort_predict({"u_id": torch.tensor([u])}).numpy()
        cand = np.concatenate([np.array(ds.validRatings[3]), np.arange(40, 90)])
        g["by_user/cand"] = cand
        g["by_user/scores"] = m.inference_by_user({
            "user_input": torch.full((len(cand),), 3), "item_input": torch.from_numpy(cand),
            "img_input": torch.from_numpy(ds.embImage[cand]), "ingre_num_input": torch.from_numpy(ds.ingredientNum[cand]),
            "ingre_input": torch.from_numpy(ds.ingredientCodeDict[cand]),
            "cal_level_input": torch.from_numpy(ds.cal_level[cand])}).numpy()
    torch.nn.functional.dropout = real_dropout
    np.savez_compressed(os.path.join(HERE, "schgn_mini.npz"), **g)
    out["schgn"] = len(g)

    # ---------------- HealthRec
    cfg = Cfg({**BASE, **CFGS["CIKM_Model"]})
    torch.manual_seed(999)
    m = CIKM_Model(cfg, ds)
    m.eval()  # transformer dropout off; the propagation path has no train/eval difference
    g = sd_np(m)
    for name in ("norm_adj_matrix", "ri_norm_adj"):
        idx, val = raw_coo(getattr(m, name))
        g[f"adj/{name}/idx"], g[f"adj/{name}/val"] = idx, val
    ua, ia, ing = m.forward()
    g.update({"fwd/user_all": ua.detach().numpy(), "fwd/item_all": ia.detach().numpy(),
              "fwd/ingre_ir": ing.detach().numpy()})
    for b, batch in enumerate(batches):
        m.zero_grad()
        losses = m.calculate_loss(to_t(batch))
        sum(losses).backward()
        g[f"loss/{b}"] = np.array([float(x) for x in losses], dtype=np.float64)
        for k, v in grads_np(m, {"user_embedding.weight", "item_embedding.weight",
                                  "ingre_embedding.weight", "image_trs.weight", "text_trs.weight"}).items():
            g[f"{k}/{b}"] = v
    np.savez_compressed(os.path.join(HERE, "healthrec_mini.npz"), **g)
    out["healthrec"] = len(g)

    # ---------------- LightGCN
    cfg = Cfg({**BASE, **CFGS["LightGCN"]})
    torch.manual_seed(999)
    m = LightGCN(cfg, ds)
    g = sd_np(m)
    ua, ia = m.forward()
    g.update({"fwd/user_all": ua.detach().numpy(), "fwd/item_all": ia.detach().numpy()})
    for b, batch in enumerate(batches):
        m.zero_grad()
        losses = m.calculate_loss(to_t(batch))
        sum(losses).backward()
        g[f"loss/{b}"] = np.array([float(x) for x in losses], dtype=np.float64)
        for k, v in grads_np(m, {"user_embedding.weight", "image_trs.weight", "image_trs.bias"}).items():
            g[f"{k}/{b}"] = v
    np.savez_compressed(os.path.join(HERE, "lightgcn_mini.npz"), **g)
    out["lightgcn"] = len(g)

    # ---------------- primitives: losses, contrastive, kNN utilities, top-k, metrics
    gen = torch.Generator().manual_seed(5)
    g = {}
    pos, neg = torch.randn(97, generator=gen), torch.randn(97, generator=gen)
    g["bpr/pos"], g["bpr/neg"] = pos.numpy(), neg.numpy()
    g["bpr/out"] = BPRLoss()(pos, neg).numpy()
    e1, e2, e3 = (torch.randn(n, 64, generator=gen) for n in (33, 33, 17))
    g["emb/e1"], g["emb/e2"], g["emb/e3"] = e1.numpy(), e2.numpy(), e3.numpy()
    g["emb/out"] = EmbLoss()(e1, e2, e3).numpy()
    stub = types.SimpleNamespace()
    x, y = torch.randn(128, 64, generator=gen) * 0.1, torch.randn(128, 64, generator=gen) * 0.1
    x.requires_grad_(True)
    y.requires_grad_(True)
    dc = PRICAI_ModelX.correlation_distance(stub, x, y)
    dc.backward()
    g["dcor/x"], g["dcor/y"], g["dcor/out"] = x.detach().numpy(), y.detach().numpy(), dc.detach().numpy()
    g["dcor/gx"], g["dcor/gy"] = x.grad.numpy(), y.grad.numpy()
    h = (torch.randn(96, 64, generator=gen)).requires_grad_(True)
    cl = PRICAI_ModelX.CL_loss(stub, h)
    cl.backward()
    g["nce/h"], g["nce/out"], g["nce/gh"] = h.detach().numpy(), cl.detach().numpy(), h.grad.numpy()
    feat = torch.randn(80, 24, generator=gen)
    sim = ref_utils.build_sim(feat)
    nb = ref_utils.build_knn_neighbourhood(sim, 7)
    lap = ref_utils.compute_normalized_laplacian(nb)
    dl = ref_utils.build_knn_normalized_graph(sim, 7, is_sparse=False, norm_type="sym")
    g["knn/feat"], g["knn/sim"], g["knn/nb"], g["knn/lap"], g["knn/dense_sym"] = (
        feat.numpy(), sim.numpy(), nb.numpy(), lap.numpy(), dl.numpy())
    g["knn/dense_rw"] = ref_utils.get_dense_laplacian(nb, "rw").numpy()
    v, i = torch.topk(sim, 7, dim=-1)
    g["knn/topk_val"], g["knn/topk_ind"] = v.numpy(), i.numpy()
    # centroid assignment: the notebook's loop (allrecipes_kmeans.ipynb code cell 0-1) on mini features
    centres = ds.image_center
    lists = []
    for each_embedding in ds.embImage[:64].astype(np.float64):
        distances = [np.linalg.norm(each_embedding - arr) for arr in centres.astype(np.float64)]
        lists.append(list(np.argsort(distances)[:10]))
    g["centroid/top6"] = np.array([c[:6] for c in lists], dtype=np.int64)
    # ranking: torch.topk as Trainer.evaluate applies it, then TopKEvaluator
    U, I = 40, 300
    ue, ie = torch.randn(U, 64, generator=gen) * 0.1, torch.randn(I, 64, generator=gen) * 0.1
    scores = ue @ ie.t()
    _, topi = torch.topk(scores, 50, dim=-1)
    rng = np.random.default_rng(3)
    pos_items = [sorted(rng.choice(I, size=int(rng.integers(1, 9)), replace=False).tolist()) for _ in range(U)]
    ev = TopKEvaluator(Cfg(BASE))
    res = ev.evaluate([topi[u] for u in range(U)], (list(range(U)), pos_items, [len(p) for p in pos_items]))
    g["rank/ue"], g["rank/ie"], g["rank/topi"] = ue.numpy(), ie.numpy(), topi.numpy()
    g["rank/pos_ptr"] = np.cumsum([0] + [len(p) for p in pos_items])
    g["rank/pos_idx"] = np.concatenate(pos_items)
    g["rank/metric_keys"] = np.array(sorted(res.keys()))
    g["rank/metric_vals"] = np.array([res[k] for k in sorted(res.keys())], dtype=np.float64)
    toy = TopKEvaluator(Cfg({**BASE, "topk": [1, 3]})).evaluate(
        [torch.tensor([4, 1, 7]), torch.tensor([0, 2, 9]), torch.tensor([5, 6, 3]), torch.tensor([8, 8, 1])],
        ([0, 1, 2, 3], [[1], [9, 0], [2], [1, 8, 4]], [1, 2, 1, 3]))
    g["rank/toy_keys"] = np.array(sorted(toy.keys()))
    g["rank/toy_vals"] = np.array([toy[k] for k in sorted(toy.keys())], dtype=np.float64)
    r, n = metrics_by_user([3, 0, 9, 1, 7], range(2))
    g["rank/by_user"] = np.array([r, n, get_auc_fast(range(2), np.array([0.9, 0.1, 0.5, 0.3, 0.05, 0.7]), 4)])
    np.savez_compressed(os.path.join(HERE, "primitives.npz"), **g)
    out["primitives"] = len(g)
    for scale in ("C1", "C3"):
        out["clussl_" + scale] = clussl_at_scale(scale)
    out["healthrec_C1"] = healthrec_c1()
    out["schgn_C1"] = schgn_c1()
    out["lightgcn_C1"] = lightgcn_c1()
    print(out)
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
