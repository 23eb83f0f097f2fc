"""CPU-only checks of the host side: the C-ABI library loads and exports every declared symbol,
the graph builder reproduces the reference's adjacency bit for bit, segment plans are well formed,
and the drop-in models initialise to the reference's `state_dict` under the same seed."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden

import foodrec_b200  # noqa: F401
from foodrec_b200 import _lib, graph as G


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "foodrec_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = sorted(set(re.findall(r"\b(fr_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 10
    for n in names:
        assert hasattr(_lib.lib, n), f"libfoodrec_b200.so does not export {n}"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature in _lib.py"
    assert _lib.lib.fr_version() >= 100


def test_error_reporting_without_gpu():
    import ctypes as C
    rp = np.array([0, 3, 2], dtype=np.int32)  # not monotone
    a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
    rc = _lib.lib.fr_spmm_plan_sizes(rp.ctypes.data, 2, 32, C.byref(a), C.byref(b), C.byref(c))
    assert rc == -1
    assert b"monotone" in _lib.lib.fr_last_error()
    with pytest.raises(_lib.FoodRecError):
        _lib.check(rc, "plan")


def _csr_matches(g, idx, val):
    rows = np.repeat(np.arange(g.n_rows), np.diff(g.row_ptr_host))
    order = np.lexsort((idx[1], idx[0]))
    assert np.array_equal(rows, idx[0][order])
    assert np.array_equal(g.col.numpy().astype(np.int64), idx[1][order])
    assert np.array_equal(g.val.numpy(), val[order])  # bit-exact fp32


def test_graph_builder_bit_exact_vs_reference(mini_ds):
    ds, g = mini_ds, load_golden("clussl_mini.npz")
    _csr_matches(G.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items, "cpu"),
                 g["adj/norm_adj_matrix/idx"], g["adj/norm_adj_matrix/val"])
    _csr_matches(G.norm_adj_item_side(ds.rIngre_triples, ds.n_items, ds.num_ingredients, "cpu"),
                 g["adj/ingre_norm_adj/idx"], g["adj/ingre_norm_adj/val"])
    _csr_matches(G.norm_adj_item_side(ds.image_cluster_triples, ds.n_items, ds.cfg.n_cluster, "cpu"),
                 g["adj/image_norm_adj/idx"], g["adj/image_norm_adj/val"])
    _csr_matches(G.norm_adj_item_side(ds.text_cluster_triples, ds.n_items, ds.cfg.n_cluster, "cpu"),
                 g["adj/text_norm_adj/idx"], g["adj/text_norm_adj/val"])


def _fold_shape(k):
    """csrc/spmm.cu::fold_shape: rows of up to 16 segments fold in one level, longer ones in ~sqrt(k) children."""
    if k <= 16:
        return k, 0
    per = 1
    while per * per < k:
        per += 1
    return per, -(-k // per)


def _interpret_plan(g, rp, col, val, X):
    """What `spmm_group_kernel` computes from the plan, restated in numpy: per-segment partial sums, then the fold
    entries in fixed order (children into their parent's slots, parents / single-level entries into the row)."""
    seg, lr = g.seg_host[:g.n_seg], g.long_rows_host[:g.n_long]
    Y = np.zeros((len(rp) - 1, X.shape[1]), np.float64)
    part = np.full((max(g.n_part, 1), X.shape[1]), np.nan)
    arrived = np.zeros(max(g.n_long, 1), np.int64)
    written = np.zeros(len(rp) - 1, np.int64)

    def publish(entry, slot, acc):
        first, n_parts, pbase, row = lr[entry]
        assert 0 <= slot < n_parts and np.isnan(part[pbase + slot]).all()
        part[pbase + slot] = acc
        arrived[entry] += 1
        if arrived[entry] < n_parts:
            return
        tot = part[pbase:pbase + n_parts].sum(0)
        if row >= 0:
            Y[row] = tot
            written[row] += 1
        else:
            parent = -row - 1
            publish(parent, entry - lr[parent][0], tot)
    for r, st, ln, lid in seg:
        acc = (val[st:st + ln, None] * X[col[st:st + ln]]).sum(0) if ln else np.zeros(X.shape[1])
        if lid < 0:
            Y[r] = acc
            written[r] += 1
        else:
            publish(lid, r, acc)             # a long-row segment carries its slot in the first field
    assert (written == 1).all() and (arrived == lr[:, 1]).all() if g.n_long else (written == 1).all()
    return Y


@pytest.mark.parametrize("degs", [[0, 1, 128, 129, 0, 1000, 5, 256, 0], [], [0, 0], [4000], [64 * 16, 64 * 16 + 1, 70000, 3, 64 * 290],
                                  [3000, 200] + [1] * 262144 + [2000, 65]])   # >= 262 144 rows: long segments ordered by position
def test_segment_plan_covers_every_nonzero_once(degs):
    rp = np.concatenate([[0], np.cumsum(degs)]).astype(np.int32)
    rng = np.random.default_rng(len(degs))
    n_cols = 37
    col = rng.integers(0, n_cols, int(rp[-1])).astype(np.int32)
    val = rng.standard_normal(int(rp[-1])).astype(np.float32)
    g = G.PropGraph(rp, col, val, n_cols, "cpu")
    seg = g.seg_host[:g.n_seg]
    assert g.n_seg == sum(max(1, -(-d // G.SEG)) for d in degs)
    seen = np.zeros(int(rp[-1]), dtype=np.int32)
    rows_seen = set()
    lr = g.long_rows_host[:g.n_long]

    def row_of(entry):                       # a child entry names its parent, the parent (or a single-level entry) the row
        return int(lr[entry][3]) if lr[entry][3] >= 0 else row_of(-int(lr[entry][3]) - 1)
    for r, s, l, lid in seg:
        if lid >= 0:                         # (slot, start, len, entry): the row comes from the fold entry
            assert 0 <= r < lr[lid][1]
            r = row_of(lid)
        assert 0 <= l <= G.SEG and rp[r] <= s and s + l <= rp[r + 1]
        seen[s:s + l] += 1
        rows_seen.add(int(r))
        assert (lid >= 0) == (degs[r] > G.SEG)
    assert (seen == 1).all() and rows_seen == set(range(len(degs)))
    ks = [-(-d // G.SEG) for d in degs if d > G.SEG]
    assert g.n_long == sum(1 + (_fold_shape(k)[1] if _fold_shape(k)[1] else 0) for k in ks)
    assert g.n_part == sum(k + _fold_shape(k)[1] for k in ks)
    slots = np.zeros(max(g.n_part, 1), np.int32)
    for k, (first, nparts, pbase, row) in enumerate(lr):
        slots[pbase:pbase + nparts] += 1
        mine = seg[seg[:, 3] == k]
        if row >= 0 and not (k > 0 and lr[k - 1][3] == -(k + 1)):          # a single-level row: every slot once
            assert sorted(mine[:, 0].tolist()) == list(range(nparts)) and nparts <= 16
        elif row >= 0:                                                   # a parent: its children precede it, contiguously
            assert first + nparts == k and (lr[first:k, 3] == -(k + 1)).all() and len(mine) == 0
        else:                                                            # a child
            parent = -row - 1
            assert lr[parent][3] >= 0 and lr[parent][0] <= k < parent
            assert sorted(mine[:, 0].tolist()) == list(range(nparts))
            # slot j of the entry is segment first + j of the row
            r0 = lr[parent][3]
            assert all(int(st) == rp[r0] + (first + int(sl)) * G.SEG for sl, st in mine[:, :2])
    assert (slots[:g.n_part] == 1).all()
    # order of the long-row block: row after row for small graphs, by relative position inside the row from 262 144 rows up
    long_seg = seg[seg[:, 3] >= 0]
    if len(long_seg):
        rows_l = np.array([row_of(e) for e in long_seg[:, 3]])
        idx_in_row = (long_seg[:, 1] - rp[rows_l]) // G.SEG
        k_of = -(-np.asarray(degs)[rows_l] // G.SEG)
        if len(degs) >= 262144:
            assert (np.diff((idx_in_row << 16) // k_of) >= 0).all() and len(set(rows_l[:4].tolist())) > 1
        else:
            assert (np.diff(rows_l) >= 0).all()
    # whole-row segments come sorted by descending length
    single = seg[seg[:, 3] < 0][:, 2]
    assert (np.diff(single) <= 0).all()
    # the plan, interpreted the way the kernel walks it, is the product
    X = rng.standard_normal((n_cols, 8))
    import scipy.sparse as sp
    ref = sp.csr_matrix((val.astype(np.float64), col, rp), shape=(len(degs), n_cols)) @ X if len(degs) else np.zeros((0, 8))
    np.testing.assert_allclose(_interpret_plan(g, rp, col, val.astype(np.float64), X), ref, rtol=1e-9, atol=1e-9)


def test_gcn_normalisation_matches_oracle(mini_ds):
    from oracle import adjacency
    ei = adjacency.schgn_edge_index(mini_ds)
    n = mini_ds.n_users + mini_ds.n_items + mini_ds.num_ingredients + mini_ds.num_calories_level
    src, dst, w = adjacency.gcn_norm_edges(ei, n)
    g = G.gcn_normalised(ei[0].numpy(), ei[1].numpy(), n, "cpu")
    import scipy.sparse as sp
    ref = sp.coo_matrix((w.numpy(), (dst.numpy(), src.numpy())), shape=(n, n)).tocsr()
    ref.sum_duplicates()
    got = g.to_scipy()
    got.sum_duplicates()
    assert abs(got - ref).max() < 1e-7
    assert abs(g.T.to_scipy() - ref.T).max() < 1e-7


class Cfg(dict):
    def __getitem__(self, k):
        return self.get(k)


BASE = dict(device="cpu", embedding_size=64, train_batch_size=64, is_multimodal_model=True, end2end=False,
            use_health_level_multi_hot=True, num_attention_heads=2, num_hidden_layers=2,
            attention_probs_dropout_prob=0.0, hidden_act="gelu")


def test_clussl_same_seed_same_state_dict(mini_ds):
    from foodrec_b200.models.pricai_modelx import PRICAI_ModelX
    g = load_golden("clussl_mini.npz")
    cfg = Cfg({**BASE, "n_ri_layers": 2, "n_mm_layers": 1, "n_ui_layers": 1, "reg_weight": 0.01, "loss_cl": 0.1,
               "n_cluster": mini_ds.cfg.n_cluster})
    torch.manual_seed(999)
    m = PRICAI_ModelX(cfg, mini_ds)
    sd = m.state_dict()
    ref_keys = sorted(k[3:] for k in g if k.startswith("sd/"))
    assert sorted(sd.keys()) == ref_keys
    for k in ref_keys:
        assert np.array_equal(sd[k].numpy(), g["sd/" + k]), k


def test_healthrec_and_lightgcn_same_seed_same_state_dict(mini_ds):
    from foodrec_b200.models.cikm_model import CIKM_Model
    from foodrec_b200.models.lightgcn import LightGCN
    for cls, fname, extra in ((CIKM_Model, "healthrec_mini.npz",
                               dict(n_layers=2, ui_layers=1, reg_weight=0.5, loss_kd=0.05, loss_health=0.1,
                                    kd_threshold=0.4)),
                              (LightGCN, "lightgcn_mini.npz", dict(n_layers=2, reg_weight=0.1))):
        g = load_golden(fname)
        torch.manual_seed(999)
        m = cls(Cfg({**BASE, **extra}), mini_ds)
        sd = m.state_dict()
        ref_keys = sorted(k[3:] for k in g if k.startswith("sd/"))
        assert sorted(sd.keys()) == ref_keys, set(sd.keys()) ^ set(ref_keys)
        for k in ref_keys:
            assert np.array_equal(sd[k].numpy(), g["sd/" + k]), (cls.__name__, k)


SCHGN_CFG = dict(inner_size=256, hidden_dropout_prob=0.5, attention_probs_dropout_prob=0.5, regs=0.01, reg_image=1,
                 reg_w=0.05, reg_g=0.01, reg_health=0.01, ssl=0.008, SCHGN_ssl=True, neg_sample_num=4)


def test_schgn_same_seed_same_state_dict_and_edges(mini_ds):
    """Parameter names, order, shapes and RNG consumption follow FoodRec/models/schgn.py:46-122."""
    from foodrec_b200.models.schgn import SCHGN
    g = load_golden("schgn_mini.npz")
    torch.manual_seed(999)
    m = SCHGN(Cfg({**BASE, **SCHGN_CFG}), mini_ds)
    sd = m.state_dict()
    ref_keys = [k[3:] for k in g if k.startswith("sd/")]
    assert list(sd.keys()) == ref_keys
    for k in ref_keys:
        assert np.array_equal(sd[k].numpy(), g["sd/" + k]), k
    assert np.array_equal(m.g2i_edges.numpy(), g["edges/g2i"])
    assert np.array_equal(m.i2u_edges.numpy(), g["edges/i2u"])
    assert not m.ingre_embed_second.requires_grad


def test_masked_ingredient_task_shapes(mini_ds):
    from foodrec_b200.synth import sample_train_batches
    b = sample_train_batches(mini_ds, 64, 1, seed=3, schgn=True)[0]
    G = mini_ds.num_ingredients
    real = np.arange(20)[None, :] < b["pos_ingre_num"][:, None]
    hidden = b["masked_ingre_seq"] == G + 1
    assert (hidden <= real).all() and hidden.any()
    assert np.array_equal(b["pos_ingre_seq"], b["pos_ingre_code"])
    assert np.array_equal(b["neg_ingre_seq"][~hidden], b["pos_ingre_code"][~hidden])
    # a sampled negative is never one of the recipe's own ingredients (dataloader.py:117-143)
    for r, c in zip(*np.nonzero(hidden)):
        assert b["neg_ingre_seq"][r, c] not in set(b["pos_ingre_code"][r, :b["pos_ingre_num"][r]])
    assert b["pos_img"].dtype == np.float64


def test_public_header_is_plain_c():
    """The drop-in boundary is a C ABI: the header must compile as C99 (no C++-isms, no torch types)."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    hdr = os.path.join(ROOT, "include", "foodrec_b200.h")
    res = subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-x", "c", hdr], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    code = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)     # declarations only (comments cite torch call sites)
    assert "torch" not in code.lower() and "at::" not in code and "std::" not in code


def test_device_sampler_exclusion_lists_host_side(mini_ds):
    """Host part of `train.DeviceBatchSampler`: the per-user exclusion CSR is train + valid + test items, sorted,
    duplicate-free (what `get_random_neg` tests against, dataloader.py:145-151); epoch length = ceil(n / B)."""
    from foodrec_b200.train import DeviceBatchSampler
    s = DeviceBatchSampler(mini_ds, 64, "cpu", seed=1)
    ptr, idx = s.excl_ptr.numpy(), s.excl_idx.numpy()
    coo = mini_ds.train_coo_matrix
    for u in (0, 3, 100, mini_ds.n_users - 1):
        want = set(coo.col[coo.row == u].tolist()) | set(mini_ds.validRatings[u]) | set(mini_ds.testRatings[u])
        got = idx[ptr[u]:ptr[u + 1]]
        assert (np.diff(got) > 0).all() and set(got.tolist()) == want
    assert ptr[-1] == idx.shape[0] and len(s) == -(-coo.nnz // 64)
    assert len(DeviceBatchSampler(mini_ds, 64, "cpu", drop_last=True)) == coo.nnz // 64


def test_device_sampler_reference_shaped_heldout_structures(mini_ds):
    """The reference's `validRatings` is positional (paired with `valid_users`; users without validation rows are
    skipped, FoodRec/utils/dataset.py:32,115-135) and its sampler reads `validTestRatings` (dict user -> set,
    dataset.py:35,93-113; dataloader.py:145-151).  Held-out items must land on the right users either way."""
    import copy
    from foodrec_b200.train import DeviceBatchSampler
    ds = copy.copy(mini_ds)
    keep = [u for u in range(ds.n_users) if u % 3 != 1]                 # a third of the users have no validation rows
    ds.valid_users = np.asarray(keep)
    ds.validRatings = [mini_ds.validRatings[u] for u in keep]
    coo = ds.train_coo_matrix

    def check(s):
        ptr, idx = s.excl_ptr.numpy(), s.excl_idx.numpy()
        for u in (0, 1, 2, 4, 100, ds.n_users - 1):
            want = set(coo.col[coo.row == u].tolist()) | set(mini_ds.testRatings[u])
            if u % 3 != 1:
                want |= set(mini_ds.validRatings[u])
            assert set(idx[ptr[u]:ptr[u + 1]].tolist()) == want, u
    check(DeviceBatchSampler(ds, 64, "cpu"))
    ds2 = copy.copy(ds)
    ds2.validTestRatings = {u: set(mini_ds.testRatings[u]) | (set(mini_ds.validRatings[u]) if u % 3 != 1 else set())
                            for u in range(ds.n_users)}
    ds2.validRatings = ds2.testRatings = None                           # the dict alone must be enough
    check(DeviceBatchSampler(ds2, 64, "cpu"))
    ds3 = copy.copy(ds)
    ds3.valid_users = None                                              # positional lists without owners: refuse to guess
    with pytest.raises(ValueError):
        DeviceBatchSampler(ds3, 64, "cpu")


def test_device_graph_builder_matches_host_builder():
    """`graph.symmetric_normalised_device` (torch ops, used for the C5-shaped stress graph) reproduces the host
    builder bit for bit (same de-duplication, fp64 degree products cast to fp32)."""
    rng = np.random.default_rng(3)
    u, i = rng.integers(0, 300, 5000), rng.integers(300, 420, 5000)
    a = G.symmetric_normalised(u, i, 420, "cpu")
    b = G.symmetric_normalised_device(torch.from_numpy(u), torch.from_numpy(i), 420)
    assert np.array_equal(a.row_ptr_host, b.row_ptr_host) and torch.equal(a.col, b.col) and torch.equal(a.val, b.val)
    assert np.array_equal(a.seg_host, b.seg_host)


# The parts of the reference's `FoodRec/` tree that model discovery touches: the lookup of its `get_model`
# (FoodRec/utils/utils.py:27-40, `importlib` on `models.<name.lower()>`) and a `models` package holding modules of the
# same names as the drop-ins, so the test also fails if the reference's own files won.
_REFERENCE_LAYOUT = {
    "utils/__init__.py": "",
    "utils/utils.py": (
        "import importlib\n"
        "import importlib.util\n\n\n"
        "def get_model(model_name):\n"
        "    module_path = '.'.join(['models', model_name.lower()])\n"
        "    if importlib.util.find_spec(module_path, __name__):\n"
        "        model_module = importlib.import_module(module_path, __name__)\n"
        "    return getattr(model_module, model_name)\n"),
    "models/__init__.py": "",
    **{f"models/{name.lower()}.py": f"class {name}:\n    pass\n"
       for name in ("PRICAI_ModelX", "CIKM_Model", "LightGCN", "SCHGN", "BM3")},
}


def test_unmodified_get_model_resolves_the_dropins(tmp_path):
    """Zero-edit discovery (SURVEY.md 8b): with `dropin/` ahead of `FoodRec/` on sys.path the reference's
    `get_model` returns the B200 classes for the four hot-path models and still finds the reference's other models
    through the overlay's `__path__`."""
    import subprocess
    import sys
    REFERENCE = str(tmp_path / "FoodRec")
    for rel, src in _REFERENCE_LAYOUT.items():
        path = os.path.join(REFERENCE, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            f.write(src)
    code = (
        "import sys, types\n"
        f"sys.path[:0] = [{os.path.join(ROOT, 'dropin')!r}, {REFERENCE!r}, {os.path.dirname(REFERENCE)!r}]\n"   # bm3.py imports `FoodRec.common...`
        "from utils.utils import get_model\n"
        "for name, mod in (('PRICAI_ModelX', 'pricai_modelx'), ('CIKM_Model', 'cikm_model'), ('LightGCN', 'lightgcn'), ('SCHGN', 'schgn')):\n"
        "    cls = get_model(name)\n"
        "    import foodrec_b200, importlib\n"
        "    want = getattr(importlib.import_module('foodrec_b200.models.' + mod), name)\n"
        "    assert cls is want, (name, cls, want)\n"
        "    assert 'multi-modal-food-recommendation_b200' in sys.modules[cls.__module__].__file__\n"
        "bm3 = get_model('BM3')\n"                       # not overridden: the reference's own file
        f"assert sys.modules[bm3.__module__].__file__.startswith({REFERENCE!r}), sys.modules[bm3.__module__].__file__\n"
        "print('ok')\n")
    res = subprocess.run([sys.executable, "-c", code], cwd=REFERENCE, capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.strip().endswith("ok"), res.stderr[-2000:]
