"""Pin the CPU oracle to outputs of the reference itself (tests/golden/*.npz, made by
tests/golden/make_golden.py in the build container).  CPU only."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import adjacency, knn, losses, propagation, ranking

RTOL = 1e-5
# The goldens were written with 10 torch intra-op threads.  Several compared values (SCHGN's attention-weight
# gradients among them) are fp32 sums with heavy cancellation that move by up to 1e-4 relative with the number of
# threads a reduction is split over, so the oracle runs with the same count on every host.
GOLDEN_THREADS = 10


@pytest.fixture(autouse=True)
def golden_thread_count():
    prev = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(prev)


def close(a, b, rtol=RTOL, atol=1e-7):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = max(np.abs(b).max(), 1e-30)
    assert a.shape == b.shape
    assert np.abs(a - b).max() <= rtol * scale + atol, (np.abs(a - b).max(), scale)


def coo_equal(t, idx, val):
    t = t.coalesce()
    order = np.lexsort((idx[1], idx[0]))
    assert np.array_equal(t.indices().numpy(), idx[:, order])
    assert np.array_equal(t.values().numpy(), val[order])  # bit-exact fp32


def T(x):
    return torch.from_numpy(np.asarray(x))


def test_adjacency_bit_exact(mini_ds):
    g = load_golden("clussl_mini.npz")
    ds = mini_ds
    coo_equal(adjacency.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items),
              g["adj/norm_adj_matrix/idx"], g["adj/norm_adj_matrix/val"])
    coo_equal(adjacency.norm_adj_item_side(ds.rIngre_triples, ds.n_items, ds.num_ingredients),
              g["adj/ingre_norm_adj/idx"], g["adj/ingre_norm_adj/val"])
    coo_equal(adjacency.norm_adj_item_side(ds.image_cluster_triples, ds.n_items, ds.cfg.n_cluster),
              g["adj/image_norm_adj/idx"], g["adj/image_norm_adj/val"])
    coo_equal(adjacency.norm_adj_item_side(ds.text_cluster_triples, ds.n_items, ds.cfg.n_cluster),
              g["adj/text_norm_adj/idx"], g["adj/text_norm_adj/val"])


def _clussl(ds, g, grad=False):
    S_ui = adjacency.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items)
    S_g = adjacency.norm_adj_item_side(ds.rIngre_triples, ds.n_items, ds.num_ingredients)
    S_v = adjacency.norm_adj_item_side(ds.image_cluster_triples, ds.n_items, ds.cfg.n_cluster)
    S_t = adjacency.norm_adj_item_side(ds.text_cluster_triples, ds.n_items, ds.cfg.n_cluster)
    P = {k: T(g["sd/" + k]).clone().requires_grad_(grad) for k in (
        "user_embedding.weight", "item_embedding.weight", "ingre_embedding.weight",
        "image_prototype_embedding.weight", "text_prototype_embedding.weight")}
    out = propagation.clussl_forward(
        S_ui, S_g, S_v, S_t, P["user_embedding.weight"], P["item_embedding.weight"],
        P["ingre_embedding.weight"], P["image_prototype_embedding.weight"],
        P["text_prototype_embedding.weight"], ds.n_users, ds.n_items, ds.num_ingredients,
        ds.cfg.n_cluster, 2, 1)
    return P, out


def test_clussl_forward_loss_grad(mini_ds):
    g = load_golden("clussl_mini.npz")
    P, (ua, ia, (vi, vt, vg)) = _clussl(mini_ds, g)
    for got, key in ((ua, "user_all"), (ia, "item_all"), (vi, "item_image"), (vt, "item_text"), (vg, "item_ingre")):
        close(got.numpy(), g["fwd/" + key])
    for b in range(2):
        P, out = _clussl(mini_ds, g, grad=True)
        u, p, n = (T(g[f"batch/{b}/{k}"]) for k in ("u_id", "pos_i_id", "neg_i_id"))
        terms = losses.clussl_loss(out, P["user_embedding.weight"], P["item_embedding.weight"], u, p, n, 0.01, 0.1)
        close([float(t) for t in terms], g[f"loss/{b}"])
        sum(terms).sum().backward()
        for k, v in P.items():
            # padding_idx row of ingre_embedding receives no gradient in nn.Embedding
            # distance-correlation backward cancels heavily in fp32: two orderings of the same
            # ops differ by ~1e-4 of the gradient's max, so grads are held to 5e-4 (losses to 1e-5)
            got = v.grad.numpy().copy()
            close(got, g[f"grad/{k}/{b}"], rtol=5e-4)
    close(ranking.inference_scores(ua, ia, torch.full((len(g["infer/cand"]),), 3), T(g["infer/cand"])).numpy(),
          g["infer/scores"])


@pytest.mark.parametrize("scale", ["C1", "C3"])
def test_clussl_oracle_matches_reference_run_at_scale(scale):
    """The oracle against the REFERENCE executed at C1 and at the Foodcom-scale C3 (BASELINE.json configs[2]):
    `tests/golden/clussl_{c1,c3}.npz` hold the reference's loss terms and sampled rows of its forward tables and
    parameter gradients for one batch of 512 from the seed-999 initial state.  The drop-in's constructor must start from
    bit-identical parameters; losses and tables agree to 1e-6.  Gradients fed by `correlation_distance` agree to
    1e-5 .. 5e-5 only -- that IS the fp32 run-to-run spread of the reference's own arithmetic (same torch ops, another
    summation order inside BLAS), the yardstick the GPU tolerances are stated against."""
    import foodrec_b200  # noqa: F401
    from foodrec_b200.models.pricai_modelx import PRICAI_ModelX
    from foodrec_b200.synth import make_dataset
    g = load_golden(f"clussl_{scale.lower()}.npz")
    ds = make_dataset(scale)

    class Cfg(dict):
        def __getitem__(self, k):
            return self.get(k)
    cfg = Cfg(device="cpu", embedding_size=64, train_batch_size=512, is_multimodal_model=True, end2end=False,
              use_health_level_multi_hot=True, n_ri_layers=2, n_mm_layers=1, n_ui_layers=1, reg_weight=0.01, loss_cl=0.1,
              n_cluster=ds.cfg.n_cluster)
    torch.manual_seed(999)
    sd = {k: v.clone() for k, v in PRICAI_ModelX(cfg, ds).state_dict().items()}
    names = [k[len("sd_rows/"):] for k in g if k.startswith("sd_rows/")]
    for k in names:                                      # same seed => the reference's own initial parameters
        assert np.array_equal(sd[k].numpy()[g["rows/" + k]], g["sd_rows/" + k]), k
        assert float(sd[k].double().sum()) == float(g["sd_sum/" + k]), k
    P = {k: sd[k].clone().requires_grad_(True) for k in names}
    S = [adjacency.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items),
         adjacency.norm_adj_item_side(ds.rIngre_triples, ds.n_items, ds.num_ingredients),
         adjacency.norm_adj_item_side(ds.image_cluster_triples, ds.n_items, ds.cfg.n_cluster),
         adjacency.norm_adj_item_side(ds.text_cluster_triples, ds.n_items, ds.cfg.n_cluster)]
    order = ("user_embedding.weight", "item_embedding.weight", "ingre_embedding.weight",
             "image_prototype_embedding.weight", "text_prototype_embedding.weight")
    out = propagation.clussl_forward(*S, *(P[k] for k in order), ds.n_users, ds.n_items, ds.num_ingredients,
                                     ds.cfg.n_cluster, 2, 1)
    u, p, n = (torch.from_numpy(g["batch/" + k]) for k in ("u_id", "pos_i_id", "neg_i_id"))
    terms = losses.clussl_loss(out, P["user_embedding.weight"], P["item_embedding.weight"], u, p, n, 0.01, 0.1)
    sum(terms).sum().backward()
    assert np.allclose([float(t) for t in terms], g["loss"], rtol=1e-6, atol=0)
    ru, ri = g["rows/user_embedding.weight"], g["rows/item_embedding.weight"]
    views = out[2]
    for got, rows, key in ((out[0], ru, "user_all"), (out[1], ri, "item_all"), (views[0], ri, "item_image"),
                           (views[1], ri, "item_text"), (views[2], ri, "item_ingre")):
        a, b = got.detach().numpy()[rows], g["fwd/" + key]
        assert np.abs(a - b).max() <= 1e-6 * np.abs(b).max(), key
    for k in order:
        a, b = P[k].grad.numpy()[g["rows/" + k]], g["grad/" + k]
        tol = 1e-6 if k == "user_embedding.weight" else 2e-4
        assert np.abs(a - b).max() <= tol * float(g["grad_absmax/" + k]), k


def test_healthrec_forward(mini_ds, mini_batches):
    g = load_golden("healthrec_mini.npz")
    ds = mini_ds
    S_ui = adjacency.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items)
    S_ri = adjacency.norm_adj_item_side(ds.rIngre_triples, ds.n_items, ds.num_ingredients)
    coo_equal(S_ri, g["adj/ri_norm_adj/idx"], g["adj/ri_norm_adj/val"])
    uw, iw, gw = (T(g["sd/" + k]) for k in ("user_embedding.weight", "item_embedding.weight", "ingre_embedding.weight"))
    ua, ia, ing = propagation.healthrec_forward(S_ui, S_ri, uw, iw, gw, ds.n_users, ds.n_items,
                                               ds.num_ingredients, 2, 1)
    close(ua.numpy(), g["fwd/user_all"])
    close(ia.numpy(), g["fwd/item_all"])
    close(ing.numpy(), g["fwd/ingre_ir"])
    for b, batch in enumerate(mini_batches):
        u, p, n = (T(batch[k]) for k in ("u_id", "pos_i_id", "neg_i_id"))
        mf = losses.bpr_from_tables(ua, ia, u, p, n)
        reg = 0.5 * losses.emb_loss(uw[u], iw[p], iw[n], gw[T(batch["pos_ingre_code"])],
                                    gw[T(batch["neg_ingre_code"])])
        close([float(mf), float(reg)], g[f"loss/{b}"][[0, 3]])


def test_healthrec_oracle_matches_reference_run_at_c1():
    """BASELINE.json configs[0] (HealthRec on C1, CPU): the oracle's propagation, BPR and regulariser against the
    reference's own run (`tests/golden/healthrec_c1.npz`), from the same-seed initial parameters of the drop-in's
    constructor (checked bit for bit against the reference's)."""
    import foodrec_b200  # noqa: F401
    from foodrec_b200.models.cikm_model import CIKM_Model
    from foodrec_b200.synth import make_dataset
    g = load_golden("healthrec_c1.npz")
    ds = make_dataset("C1")

    class Cfg(dict):
        def __getitem__(self, k):
            return self.get(k)
    torch.manual_seed(999)
    m = CIKM_Model(Cfg(device="cpu", embedding_size=64, train_batch_size=512, is_multimodal_model=True, end2end=False,
                       use_health_level_multi_hot=True, num_attention_heads=2, num_hidden_layers=2,
                       attention_probs_dropout_prob=0.0, hidden_act="gelu", n_layers=2, ui_layers=1, reg_weight=0.5,
                       loss_kd=0.05, loss_health=0.1, kd_threshold=0.4), ds)
    sd = m.state_dict()
    for k in [x[len("sd_sum/"):] for x in g if x.startswith("sd_sum/")]:
        assert float(sd[k].double().sum()) == float(g["sd_sum/" + k]), k
    uw, iw, gw = (sd[k] for k in ("user_embedding.weight", "item_embedding.weight", "ingre_embedding.weight"))
    S_ui = adjacency.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items)
    S_ri = adjacency.norm_adj_item_side(ds.rIngre_triples, ds.n_items, ds.num_ingredients)
    ua, ia, ing = propagation.healthrec_forward(S_ui, S_ri, uw, iw, gw, ds.n_users, ds.n_items, ds.num_ingredients, 2, 1)
    close(ua.numpy()[g["rows/user_embedding.weight"]], g["fwd/user_all"])
    close(ia.numpy()[g["rows/item_embedding.weight"]], g["fwd/item_all"])
    close(ing.numpy()[g["rows/ingre_ir"]], g["fwd/ingre_ir"])
    u, p, n = (T(g["batch/" + k]) for k in ("u_id", "pos_i_id", "neg_i_id"))
    mf = losses.bpr_from_tables(ua, ia, u, p, n)
    reg = 0.5 * losses.emb_loss(uw[u], iw[p], iw[n], gw[T(g["batch/pos_ingre_code"])], gw[T(g["batch/neg_ingre_code"])])
    close([float(mf), float(reg)], g["loss"][[0, 3]])


def test_lightgcn_forward(mini_ds, mini_batches):
    g = load_golden("lightgcn_mini.npz")
    ds = mini_ds
    S_ui = adjacency.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items)
    ego = T(g["sd/image_embedding.weight"]) @ T(g["sd/image_trs.weight"]).t() + T(g["sd/image_trs.bias"])
    ua, ia = propagation.lightgcn_forward(S_ui, T(g["sd/user_embedding.weight"]), ego, ds.n_users, ds.n_items, 2)
    close(ua.numpy(), g["fwd/user_all"])
    close(ia.numpy(), g["fwd/item_all"])
    for b, batch in enumerate(mini_batches):
        u, p, n = (T(batch[k]) for k in ("u_id", "pos_i_id", "neg_i_id"))
        close(float(losses.bpr_from_tables(ua, ia, u, p, n)), g[f"loss/{b}"][0])


def test_loss_primitives():
    g = load_golden("primitives.npz")
    close(losses.bpr_loss(T(g["bpr/pos"]), T(g["bpr/neg"])).numpy(), g["bpr/out"])
    close(losses.emb_loss(T(g["emb/e1"]), T(g["emb/e2"]), T(g["emb/e3"])).numpy(), g["emb/out"])
    x, y = T(g["dcor/x"]).requires_grad_(True), T(g["dcor/y"]).requires_grad_(True)
    d = losses.correlation_distance(x, y)
    d.backward()
    close(d.detach().numpy(), g["dcor/out"])
    close(x.grad.numpy(), g["dcor/gx"], rtol=1e-4)
    close(y.grad.numpy(), g["dcor/gy"], rtol=1e-4)
    h = T(g["nce/h"]).requires_grad_(True)
    c = losses.info_nce(h)
    c.backward()
    close(c.detach().numpy(), g["nce/out"])
    close(h.grad.numpy(), g["nce/gh"], rtol=1e-4)


def test_knn_utilities(mini_ds):
    g = load_golden("primitives.npz")
    sim = knn.build_sim(T(g["knn/feat"]))
    close(sim.numpy(), g["knn/sim"])
    nb, val, ind = knn.knn_neighbourhood(T(g["knn/sim"]), 7)
    assert np.array_equal(ind.numpy(), g["knn/topk_ind"])
    close(nb.numpy(), g["knn/nb"])
    close(knn.normalized_laplacian(nb).numpy(), g["knn/lap"])
    close(knn.normalized_laplacian(nb).numpy(), g["knn/dense_sym"])
    got = knn.centroid_topk(mini_ds.embImage[:64], mini_ds.image_center, 6)
    assert np.array_equal(got, g["centroid/top6"])
    from foodrec_b200.synth import topk_nearest_centres
    assert np.array_equal(topk_nearest_centres(mini_ds.embImage[:64], mini_ds.image_center, 6), g["centroid/top6"])


def test_ranking_and_metrics():
    g = load_golden("primitives.npz")
    ue, ie = T(g["rank/ue"]), T(g["rank/ie"])
    _, topi = ranking.full_sort_topk(ue, ie, torch.arange(ue.shape[0]), 50)
    assert np.array_equal(topi.numpy(), g["rank/topi"])
    ptr, idx = g["rank/pos_ptr"], g["rank/pos_idx"]
    pos = [idx[ptr[u]:ptr[u + 1]].tolist() for u in range(len(ptr) - 1)]
    res = ranking.topk_metrics(g["rank/topi"], pos)
    for k, v in zip(g["rank/metric_keys"], g["rank/metric_vals"]):
        assert res[str(k)] == v, (k, res[str(k)], v)
    toy = ranking.topk_metrics(np.array([[4, 1, 7], [0, 2, 9], [5, 6, 3], [8, 8, 1]]),
                               [[1], [9, 0], [2], [1, 8, 4]], topk=(1, 3))
    for k, v in zip(g["rank/toy_keys"], g["rank/toy_vals"]):
        assert toy[str(k)] == v, (k, toy[str(k)], v)
    r, n = ranking.metrics_by_user([3, 0, 9, 1, 7], [0, 1])
    a = ranking.auc_fast(2, np.array([0.9, 0.1, 0.5, 0.3, 0.05, 0.7]), 4)
    close([r, n, a], g["rank/by_user"])


def test_history_mask_oracle():
    torch.manual_seed(0)
    ue, ie = torch.randn(5, 8), torch.randn(30, 8)
    ptr = np.array([0, 3, 3, 10, 12, 15])
    idx = np.random.default_rng(0).integers(0, 30, size=15)
    _, top = ranking.full_sort_topk(ue, ie, torch.arange(5), 6, ptr, idx)
    for u in range(5):
        assert not set(top[u].tolist()) & set(idx[ptr[u]:ptr[u + 1]].tolist())


def test_schgn_oracle_matches_reference_run(mini_ds):
    """oracle/schgn.py vs tests/golden/schgn_mini.npz (the reference's SCHGN class executed with the
    GCNConv stand-in; dropout = identity): losses, every parameter gradient, full-sort and by-user scores."""
    from foodrec_b200.synth import sample_train_batches
    from oracle import schgn as O
    g = load_golden("schgn_mini.npz")
    P = {k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd/")}
    ei = O.schgn_edge_index(mini_ds)
    assert torch.equal(ei, torch.from_numpy(np.concatenate([g["edges/g2i"], g["edges/i2u"]], 0)).t())
    sizes = (mini_ds.n_users, mini_ds.n_items, mini_ds.num_ingredients, mini_ds.num_calories_level)
    assert torch.equal(torch.cat(O.gcn_tables(P, ei, sizes), 0), torch.from_numpy(g["gcn/out"]))
    cfg = dict(regs=0.01, reg_image=1, reg_w=0.05, reg_g=0.01, reg_health=0.01, ssl=0.008, num_hidden_layers=2,
               num_attention_heads=2)
    for b, batch in enumerate(sample_train_batches(mini_ds, 64, 2, seed=11, schgn=True)):
        for k in ("masked_ingre_seq", "neg_ingre_seq"):
            assert np.array_equal(batch[k], g[f"batch/{b}/{k}"])
        Pg = {k: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in P.items()}
        losses = O.calculate_loss(Pg, {k: torch.from_numpy(np.asarray(v)) for k, v in batch.items()}, cfg, ei, sizes)
        np.testing.assert_allclose([float(x.detach()) for x in losses], g[f"loss/{b}"], rtol=1e-6)
        sum(losses).backward()
        for k, ref in g.items():
            if k.startswith("grad/") and k.endswith(f"/{b}") and "key.bias" not in k:  # d/d(key bias) == 0 exactly
                got = Pg[k[5:-2]].grad.numpy()
                assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max() + 1e-12, k
    for u in (0, 7, 200):
        s = O.full_sort_scores(P, mini_ds, u, ei, sizes)
        np.testing.assert_allclose(s.numpy(), g[f"full_sort/{u}"], rtol=0, atol=1e-7)


def test_schgn_oracle_matches_reference_run_at_c1():
    """oracle/schgn.py vs tests/golden/schgn_c1.npz (the reference's SCHGN class executed on C1 with the GCNConv
    stand-in; dropout = identity), from the drop-in constructor's same-seed state (every floating tensor's sum checked
    against the reference's): GCN output rows, the three loss terms, every small parameter's gradient, sampled rows of
    the table gradients, full-sort scores of three users."""
    import foodrec_b200  # noqa: F401
    from foodrec_b200.models.schgn import SCHGN
    from foodrec_b200.synth import make_dataset, sample_train_batches
    from oracle import schgn as O
    g = load_golden("schgn_c1.npz")
    ds = make_dataset("C1")

    class Cfg(dict):
        def __getitem__(self, k):
            return self.get(k)
    torch.manual_seed(999)
    m = SCHGN(Cfg(device="cpu", embedding_size=64, train_batch_size=256, is_multimodal_model=True, end2end=False,
                  use_health_level_multi_hot=True, num_attention_heads=2, num_hidden_layers=2, hidden_act="gelu",
                  inner_size=256, hidden_dropout_prob=0.5, attention_probs_dropout_prob=0.5, regs=0.01, reg_image=1,
                  reg_w=0.05, reg_g=0.01, reg_health=0.01, ssl=0.008, SCHGN_ssl=True, neg_sample_num=4), ds)
    P = {k: v.detach().clone() for k, v in m.state_dict().items()}
    for k in [x[len("sd_sum/"):] for x in g if x.startswith("sd_sum/")]:
        assert float(P[k].double().sum()) == float(g["sd_sum/" + k]), k
    ei = O.schgn_edge_index(ds)
    sizes = (ds.n_users, ds.n_items, ds.num_ingredients, ds.num_calories_level)
    gcn = torch.cat(O.gcn_tables(P, ei, sizes), 0).numpy()
    assert np.abs(gcn[g["rows/gcn"]] - g["gcn/out"]).max() <= 1e-6 * np.abs(g["gcn/out"]).max()
    cfg = dict(regs=0.01, reg_image=1, reg_w=0.05, reg_g=0.01, reg_health=0.01, ssl=0.008, num_hidden_layers=2,
               num_attention_heads=2)
    batch = sample_train_batches(ds, 256, 1, seed=3, schgn=True)[0]
    for k in ("masked_ingre_seq", "neg_ingre_seq", "u_id"):
        assert np.array_equal(np.asarray(batch[k]), g["batch/" + k])
    Pg = {k: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in P.items()}
    losses_ = O.calculate_loss(Pg, {k: torch.from_numpy(np.asarray(v)) for k, v in batch.items()}, cfg, ei, sizes)
    np.testing.assert_allclose([float(x.detach()) for x in losses_], g["loss"], rtol=1e-6)
    sum(losses_).backward()
    for k, ref in g.items():
        if k.startswith("grad_full/") and "key.bias" not in k:       # d/d(key bias) == 0 exactly
            got = Pg[k[len("grad_full/"):]].grad.numpy()
            assert np.abs(got - ref).max() <= 2e-5 * np.abs(ref).max() + 1e-12, k
        if k.startswith("grad/"):
            name = k[len("grad/"):]
            got = Pg[name].grad.numpy()[g["rows/" + name]]
            assert np.abs(got - ref).max() <= 2e-5 * float(g["grad_absmax/" + name]) + 1e-12, k
    for u in (0, 7, 4999):
        s = O.full_sort_scores(P, ds, u, ei, sizes)
        np.testing.assert_allclose(s.numpy(), g[f"full_sort/{u}"], rtol=0, atol=2e-6)


def test_lightgcn_oracle_matches_reference_run_at_c1():
    """The oracle's LightGCN forward and BPR term against the reference executed on C1 (`lightgcn_c1.npz`), from the
    drop-in constructor's same-seed state (sums checked against the reference's)."""
    import foodrec_b200  # noqa: F401
    from foodrec_b200.models.lightgcn import LightGCN
    from foodrec_b200.synth import make_dataset
    g = load_golden("lightgcn_c1.npz")
    ds = make_dataset("C1")

    class Cfg(dict):
        def __getitem__(self, k):
            return self.get(k)
    torch.manual_seed(999)
    sd = LightGCN(Cfg(device="cpu", embedding_size=64, train_batch_size=512, is_multimodal_model=True, end2end=False,
                      use_health_level_multi_hot=True, n_layers=2, reg_weight=0.1), ds).state_dict()
    for k in [x[len("sd_sum/"):] for x in g if x.startswith("sd_sum/")]:
        assert float(sd[k].double().sum()) == float(g["sd_sum/" + k]), k
    S_ui = adjacency.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items)
    ego = sd["image_embedding.weight"] @ sd["image_trs.weight"].t() + sd["image_trs.bias"]
    ua, ia = propagation.lightgcn_forward(S_ui, sd["user_embedding.weight"], ego, ds.n_users, ds.n_items, 2)
    close(ua.numpy()[g["rows/user"]], g["fwd/user_all"])
    close(ia.numpy()[g["rows/item"]], g["fwd/item_all"])
    u, p, n = (T(g["batch/" + k]) for k in ("u_id", "pos_i_id", "neg_i_id"))
    close(float(losses.bpr_from_tables(ua, ia, u, p, n)), g["loss"][0])
