"""By-user scoring of SCHGN over per-user candidate lists (`SCHGN.by_user_scores`: `fr_schgn_attend_pairs` +
`fr_schgn_score_pairs`) against the reference run, the CPU restatement and the drop-in's own `inference_by_user`, and
`evaluation.evaluate_by_user` on SCHGN."""
import numpy as np
import pytest
import torch

from test_gpu_schgn import c1_model, golden_model  # noqa: F401  (c1_model is a fixture)

pytestmark = pytest.mark.gpu

# list lengths that expose a wrong `.view(b, -1)` mapping (1-3, not multiples of 4) and tile edges of the scorer (256)
LENGTHS = [1, 2, 3, 4, 5, 7, 255, 256, 257, 503, 1100]


def _csr(lists):
    ptr = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int64)
    return ptr, np.concatenate(lists).astype(np.int64)


def _oracle(m, ds):
    """Per-list scores of the CPU restatement: the list passed alone as one `compute_score` batch."""
    from oracle import schgn as O
    P = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    tables = O.gcn_tables(P, O.schgn_edge_index(ds), (ds.n_users, ds.n_items, ds.num_ingredients, ds.num_calories_level))
    emb = torch.cat([P["ingre_embed_first"], P["ingre_embed_second"]], 0)
    f = lambda a: torch.from_numpy(np.asarray(a))  # noqa: E731

    def score(user, items):
        items = np.asarray(items, dtype=np.int64)
        with torch.no_grad():
            return O.compute_score(P, tables, torch.full((len(items),), int(user), dtype=torch.long), f(items),
                                   f(ds.ingredientCodeDict[items]).long(), f(ds.ingredientNum[items]).long(),
                                   f(ds.embImage[items]), f(ds.cal_level[items]).long(), emb)[0].reshape(-1)
    return score


def _c1_lists(ds, n_users=64, seed=0):
    """64 users: the lengths of LENGTHS, then random ones; one list repeats an item, item 17 is in every list."""
    rng = np.random.default_rng(seed)
    lens = LENGTHS + list(rng.integers(1, 600, n_users - len(LENGTHS)))
    users = rng.choice(ds.n_users, n_users, replace=False)
    lists = [rng.integers(0, ds.n_items, n) for n in lens]
    for x in lists:
        x[len(x) // 2] = 17
    lists[9][5] = lists[9][200]                                   # repeated item inside one list (length 503)
    return users, lists


def test_reference_run_user3_alone_and_among_other_lists(mini_ds):
    m, g = golden_model(mini_ds)
    cand = g["by_user/cand"]
    alone = m.by_user_scores(torch.tensor([3]), [0, len(cand)], torch.from_numpy(cand).cuda())
    assert alone.shape == (len(cand),) and alone.dtype == torch.float32
    assert np.abs(alone.cpu().numpy() - g["by_user/scores"]).max() <= 2e-6
    rng = np.random.default_rng(1)
    lists = [rng.integers(0, mini_ds.n_items, 13), cand, rng.integers(0, mini_ds.n_items, 6)]
    ptr, items = _csr(lists)
    mid = m.by_user_scores(torch.tensor([5, 3, 9]), ptr, torch.from_numpy(items).cuda())[ptr[1]:ptr[2]]
    assert float((mid - alone).abs().max()) <= 1e-6
    assert np.abs(mid.cpu().numpy() - g["by_user/scores"]).max() <= 2e-6


def test_c1_lists_match_oracle(c1_model):
    m, ds = c1_model
    users, lists = _c1_lists(ds)
    ptr, items = _csr(lists)
    got = m.by_user_scores(torch.from_numpy(users), ptr, torch.from_numpy(items).cuda()).cpu()
    score = _oracle(m, ds)
    refs = [score(u, x) for u, x in zip(users, lists)]
    scale = max(float(r.abs().max()) for r in refs)
    for r, (u, ref) in enumerate(zip(users, refs)):
        err = float((got[ptr[r]:ptr[r + 1]] - ref).abs().max())
        assert err <= 1e-5 * scale + 2e-6, (r, len(ref), err, scale)
    assert float(torch.cat(refs).std()) > 100 * 2e-6          # the comparison is not vacuous


def test_c1_lists_match_inference_by_user(c1_model):
    m, ds = c1_model
    users, lists = _c1_lists(ds, seed=3)
    ptr, items = _csr(lists)
    got = m.by_user_scores(torch.from_numpy(users), ptr, torch.from_numpy(items).cuda())
    t = lambda a: torch.from_numpy(np.asarray(a)).cuda()  # noqa: E731
    for r in (0, 1, 2, 3, 4, 5, 7, 8, 10, 20, 63):
        x = lists[r]
        with torch.no_grad():
            want = m.inference_by_user({
                "user_input": torch.full((len(x),), int(users[r]), device="cuda"), "item_input": t(x),
                "img_input": t(ds.embImage[x]), "ingre_num_input": t(ds.ingredientNum[x]),
                "ingre_input": t(ds.ingredientCodeDict[x]), "cal_level_input": t(ds.cal_level[x])}).reshape(-1)
        assert float((got[ptr[r]:ptr[r + 1]] - want).abs().max()) <= 2e-6, r


def test_blocks_and_neighbours_do_not_change_scores(c1_model):
    """Per-user projections are cuBLAS GEMMs whose summation order depends on the batch size: 1e-6, not bitwise."""
    m, ds = c1_model
    users, lists = _c1_lists(ds, seed=5)
    ptr, items = _csr(lists)
    u, it = torch.from_numpy(users), torch.from_numpy(items).cuda()
    full = m.by_user_scores(u, ptr, it)
    assert torch.equal(full, m.by_user_scores(u, ptr, it))                       # repeatable, bit for bit
    small = m.by_user_scores(u, ptr, it, block_pairs=300)                        # many blocks; 1100 alone
    assert float((small - full).abs().max()) <= 1e-6
    for r in (0, 2, 9, 10, 40):
        one = m.by_user_scores(u[r:r + 1], [0, len(lists[r])], torch.from_numpy(lists[r]).cuda())
        assert float((one - full[ptr[r]:ptr[r + 1]]).abs().max()) <= 1e-6, r
    # a list of every item in order is the full-sort row (L = n_items in both mappings)
    every = m.by_user_scores(u[:2], [0, ds.n_items, 2 * ds.n_items], torch.arange(ds.n_items).repeat(2).cuda())
    assert float((every.view(2, -1) - m.full_sort_scores(u[:2].cuda())).abs().max()) <= 1e-6


def test_evaluate_by_user_metrics(c1_model):
    from foodrec_b200 import evaluation as E, metrics as M
    m, ds = c1_model
    rng = np.random.default_rng(7)
    users = np.arange(0, ds.n_users, 71)[:64]
    lists, n_pos = [], []
    for u in users:                       # distinct candidates: no tied scores (see the tie rule of the metrics)
        p = np.unique(ds.testRatings[u])
        lists.append(np.concatenate([p, rng.choice(np.setdiff1d(np.arange(ds.n_items), p), 100, replace=False)]))
        n_pos.append(len(p))
    ptr, items = _csr(lists)
    host, s_h = E.evaluate_by_user(m, users, ptr, items, n_pos, neg_num=100)
    score = _oracle(m, ds)
    ref = torch.cat([score(u, x) for u, x in zip(users, lists)]).numpy()
    want = M.by_user_metrics(ref, ptr, np.asarray(n_pos), 100)
    assert list(host) == list(want)
    for k in want:
        assert abs(host[k] - want[k]) <= 1e-6, (k, host[k], want[k])
    dev, s_d = E.evaluate_by_user(m, users, ptr, items, n_pos, neg_num=100, device_metrics=True)
    assert s_d.is_cuda and np.array_equal(s_d.cpu().numpy(), s_h)
    for k in host:
        assert abs(dev[k] - host[k]) <= 1e-12, (k, dev[k], host[k])


def test_scores_follow_a_parameter_update(mini_ds):
    from foodrec_b200 import evaluation as E
    from foodrec_b200.train import mark_parameters_updated
    m, _ = golden_model(mini_ds)
    rng = np.random.default_rng(2)
    users = np.array([0, 7, 31])
    lists = [rng.choice(mini_ds.n_items, n, replace=False) for n in (9, 22, 5)]
    ptr, items = _csr(lists)
    n_pos = [2, 3, 1]
    _, before = E.evaluate_by_user(m, users, ptr, items, n_pos, neg_num=20)
    with torch.no_grad():            # in place through `.data`, as a graph replay or fused optimizer leaves `_version`
        for p in (m.item_embed, m.W_concat.weight, m.W_concat.bias, m.W_att_comp.weight):
            p.data.mul_(1.5)
    mark_parameters_updated(m)
    _, after = E.evaluate_by_user(m, users, ptr, items, n_pos, neg_num=20)
    assert np.abs(after - before).max() > 1e-3
    score = _oracle(m, mini_ds)
    for r, (u, x) in enumerate(zip(users, lists)):
        assert np.abs(after[ptr[r]:ptr[r + 1]] - score(u, x).numpy()).max() <= 2e-6, r


def test_bad_lists_are_rejected(mini_ds):
    from foodrec_b200 import _lib
    m, _ = golden_model(mini_ds)
    n = mini_ds.n_items
    u = torch.tensor([1, 2])
    ok = m.by_user_scores(u, [0, 3, 5], torch.tensor([0, 1, 2, 3, 4], device="cuda"))
    for bad in ([0, 1, 2, n, 4], [0, 1, -1, 3, 4]):
        with pytest.raises(_lib.FoodRecError):                                   # checked on the device
            m.by_user_scores(u, [0, 3, 5], torch.tensor(bad, device="cuda", dtype=torch.int32))
    with pytest.raises(_lib.FoodRecError):                                       # would wrap into range as int32
        m.by_user_scores(u, [0, 3, 5], torch.tensor([0, 1, 2, 3, 2 ** 32 + 1], device="cuda"))
    with pytest.raises(_lib.FoodRecError):                                       # empty list
        m.by_user_scores(u, [0, 5, 5], torch.tensor([0, 1, 2, 3, 4], device="cuda"))
    with pytest.raises(_lib.FoodRecError):                                       # ptr / items mismatch
        m.by_user_scores(u, [0, 3, 6], torch.tensor([0, 1, 2, 3, 4], device="cuda"))
    with pytest.raises(_lib.FoodRecError):
        m.by_user_scores(u, [0, 3], torch.tensor([0, 1, 2], device="cuda"))
    empty = m.by_user_scores(u[:0], [0], torch.zeros(0, dtype=torch.int64, device="cuda"))
    assert empty.shape == (0,) and empty.is_cuda
    # the C ABI checks the lists on the device and reports through a status word: a non-increasing ptr, a ptr that
    # misses n_pairs, an item out of range
    L = _lib.lib
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    GUARD = 1 << 16

    def attend(ptr, items):
        """-> (return code, status, whether any byte outside the attended pairs' outputs changed).  The workspace is
        followed by a zeroed guard region; att / logits start out as a sentinel."""
        nu, n_pairs = len(ptr) - 1, len(items)
        t = m._scorer_tables(torch.arange(1, nu + 1, device="cuda"))
        f = {k: v.float().contiguous() for k, v in t.items() if k not in ("codes", "nums")}
        need = int(L.fr_schgn_attend_pairs_ws_bytes(nu, n_pairs, n))
        ws = torch.zeros(need + GUARD, dtype=torch.uint8, device="cuda")
        att = torch.full((n_pairs, 64), 7.0, device="cuda")
        logits = torch.full((4 * n_pairs,), 7.0, device="cuda")
        p = torch.tensor(ptr, device="cuda", dtype=torch.int64)
        it = torch.tensor(items, device="cuda", dtype=torch.int32)
        status.zero_()
        rc = L.fr_schgn_attend_pairs(
            f["user_key"].data_ptr(), f["user_comp"].data_ptr(), nu, p.data_ptr(), it.data_ptr(), n_pairs,
            t["codes"].data_ptr(), t["codes"].shape[1], t["nums"].data_ptr(), n, f["ingre_key"].data_ptr(),
            f["ingre_final"].data_ptr(), f["ingre_comp"].data_ptr(), f["img_key"].data_ptr(), f["comp_keys"].data_ptr(),
            f["h_ingre"].data_ptr(), f["h_comp"].data_ptr(), 64, ws.data_ptr(), need, att.data_ptr(), logits.data_ptr(),
            status.data_ptr(), _lib.stream_ptr())
        untouched = bool((ws[need:] == 0).all()) and bool((att == 7.0).all()) and bool((logits == 7.0).all())
        return rc, int(status.item()), untouched
    six = list(range(6))
    assert attend([0, 4, 2, 6], six) == (0, 1, True)
    assert attend([0, 2, 4, 5], six) == (0, 1, True)
    assert attend([0, 2, 2, 6], six) == (0, 1, True)
    assert attend([0, 2, 4, 6], [0, 1, 2, n, 4, 5])[:2] == (0, 2)
    rc, st, untouched = attend([0, 2, 4, 6], six)
    assert (rc, st, untouched) == (0, 0, False)                                  # a valid call does write its outputs
    # lists that each pass their own check but overlap: [0, 1000) and four times [1, 1000).  Their per-item counts add
    # up to 4996 pairs, so grouping them would write ~32 KB past the 1000-pair grp array, beyond the workspace
    assert attend([0, 1000, 1, 1000, 1, 1000, 1, 1000, 1, 1000], [i % n for i in range(1000)]) == (0, 1, True)
    assert torch.equal(m.by_user_scores(u, [0, 3, 5], torch.tensor([0, 1, 2, 3, 4], device="cuda")), ok)
