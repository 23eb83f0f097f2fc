"""SCHGN on the B200 kernels -- drop-in for FoodRec/models/schgn.py.

What runs where:

* the heterogeneous GCN (`tanh(GCNConv(x))`, schgn.py:241-250) is one dense `lin` GEMM plus one fused
  propagate + bias + tanh launch of the CSR kernel on a plan built once (`schgn_gcn.GraphConv`).
  The reference evaluates it twice per training batch (once per `compute_score` call, identical
  inputs) and once per user in `full_sort_predict`; here it is evaluated once per batch and, for
  evaluation, once per parameter version;
* `full_sort_predict` (schgn.py:318-345: python loops over every item, the whole `[I, Dv]` image
  matrix re-uploaded and projected, a full GCN -- per user) runs the fused pair scorer
  `fr_schgn_attend` + `fr_schgn_score` (csrc/schgn_score.cu) over item-side tables that are computed
  once: one launch pair scores up to 16 users against every item.  `full_sort_topk` is the batched
  entry point;
* the per-pair scorer on a training batch (B x 20 x 64) and the masked-ingredient encoder are
  batch-sized dense torch, outside the hot path (SURVEY.md section 2); their row gathers go through
  `fr_gather_rows` / `fr_scatter_add_rows`.

Parameter names, shapes and creation order are the reference's, so `state_dict`s interchange and
`torch.manual_seed(s)` reproduces its initial weights.  The reference's component attention reads
its `[4b]` logits back with `.view(b, -1)` (schgn.py:198), which mixes samples of the batch; that is
reproduced here, on both paths, because results must match.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _lib, ops
from ..common.abstract_recommender import GeneralRecommender
from ..common.encoder import Encoder
from .schgn_gcn import GraphConv, truncated_normal_

# (attribute, in, out, bias, fan used for the weight std, init the bias?)  -- creation order matters
_HEADS = (
    ("W_att_ingre", 3, 1, True, 4, True),   # ingredient-level attention over [ingredient; user; image]
    ("h_att_ingre", 1, 0, False, 0, False),
    ("W_att_comp", 2, 1, True, 3, True),    # component-level attention over [user; component]
    ("h_att_comp", 1, 0, False, 0, False),
    ("W_concat", 3, 1, True, 4, True),      # [user; item; user * item] -> hidden
    ("output_mlp", 1, 0, False, 2, False),
)


def _sq(t):
    return torch.sum(t ** 2)


def _rows(table, idx):
    """`table[idx]` for an index tensor of any shape through the gather kernel: its backward is one
    scatter-add launch instead of torch's sort-based `index_put_` (1 ms per gather on the C2 tables,
    84 % of the eager step before this)."""
    return ops.gather_rows(table, idx.reshape(-1)).view(*idx.shape, table.shape[1])


class SCHGN(GeneralRecommender):
    def __init__(self, config, dataset):
        super().__init__(config, dataset)
        self.config, self.dataset = config, dataset
        self.n_cold = dataset.cold_num
        self.n_health = dataset.num_calories_level
        self.n_ingredients = dataset.num_ingredients
        self.img_size = dataset.image_size
        e = self.emb_size = config["embedding_size"]

        self.ingre_encoder = Encoder(
            n_layers=config["num_hidden_layers"], n_heads=config["num_attention_heads"], hidden_size=e,
            inner_size=config["inner_size"], hidden_dropout_prob=config["hidden_dropout_prob"],
            attn_dropout_prob=config["attention_probs_dropout_prob"], hidden_act=config["hidden_act"],
            layer_norm_eps=1e-12)
        for m in self.modules():                       # schgn.py:66,124-135: encoder linears only
            if isinstance(m, nn.Linear):
                truncated_normal_(m.weight, std=0.01)
                m.bias.data.zero_()

        self.g2i_edges, self.i2u_edges = self.load_graph(dataset)
        self.new_gcn = GraphConv(64, 64)
        for key in ("regs", "reg_image", "reg_w", "reg_g", "reg_health", "ssl"):
            setattr(self, key, config[key])

        def table(rows):
            return nn.Parameter(torch.empty(rows, e))
        self.user_embed, self.item_embed = table(self.n_users), table(self.n_items)
        self.ingre_embed_first = table(self.n_ingredients)
        self.ingre_embed_second = nn.Parameter(torch.zeros(1, e), requires_grad=False)   # padding ingredient
        self.ingre_embed_mask = table(1)                                                 # [MASK] ingredient
        self.health_embed = table(self.n_health)

        self.img_trans = nn.Linear(self.img_size, e)
        std = float(np.sqrt(2.0 / (self.img_size + e)))
        truncated_normal_(self.img_trans.weight, std=std)
        truncated_normal_(self.img_trans.bias, std=std)
        for name, fan_in, fan_out, bias, fan_std, init_bias in _HEADS:
            lin = nn.Linear(e * fan_in, e * fan_out if fan_out else 1, bias=bias)
            if fan_std:
                truncated_normal_(lin.weight, std=float(np.sqrt(2.0 / (e * fan_std))))
            else:
                nn.init.ones_(lin.weight)
            if init_bias:
                truncated_normal_(lin.bias, std=float(np.sqrt(2.0 / (e + e))))
            setattr(self, name, lin)
        self.mip_norm = nn.Linear(e, e)
        self.criterion = nn.BCELoss(reduction="none")
        for p in (self.user_embed, self.item_embed, self.ingre_embed_first, self.ingre_embed_mask, self.health_embed):
            truncated_normal_(p, std=0.01)
        self._edge_index = None
        self._eval_cache = None

    # ------------------------------------------------------------------ graph
    def load_graph(self, dataset):
        """Directed edges as `[E, 2]` rows (source, target): item -> user, ingredient -> item,
        calorie level -> item (schgn.py:139-151; the reference's two names are swapped, both lists are
        concatenated before use)."""
        U, I, G = self.n_users, self.n_items, self.n_ingredients
        ur = np.asarray(dataset.uRecipe_triples, dtype=np.int64)
        ri = np.asarray(dataset.rIngre_triples, dtype=np.int64)
        rc = np.asarray(dataset.rCalories_triples, dtype=np.int64)
        first = np.stack([ur[:, 1] + U, ur[:, 0]], 1)
        second = np.concatenate([np.stack([ri[:, 1] + U + I, ri[:, 0] + U], 1),
                                 np.stack([rc[:, 1] + U + I + G, rc[:, 0] + U], 1)], 0)
        dev = self.device
        return torch.from_numpy(first).to(dev), torch.from_numpy(second).to(dev)

    def _edges(self, g2i_edges, i2u_edges):
        if g2i_edges is self.g2i_edges and i2u_edges is self.i2u_edges:
            if self._edge_index is None or self._edge_index.device != self.user_embed.device:
                self._edge_index = torch.cat([g2i_edges, i2u_edges], 0).t().contiguous().to(self.user_embed.device)
            return self._edge_index
        return torch.cat([g2i_edges, i2u_edges], 0).t().contiguous()

    def gcn_tables(self, g2i_edges=None, i2u_edges=None):
        """(user, item, ingredient, health) rows of `tanh(GCNConv(cat(tables)))`."""
        edge_index = self._edges(self.g2i_edges if g2i_edges is None else g2i_edges,
                                 self.i2u_edges if i2u_edges is None else i2u_edges)
        x = torch.cat([self.user_embed, self.item_embed, self.ingre_embed_first, self.health_embed], 0)
        return torch.split(self.new_gcn(x, edge_index),
                           [self.n_users, self.n_items, self.n_ingredients, self.n_health], 0)

    # ------------------------------------------------------------------ batch-sized scorer (torch)
    def sequence_mask(self, lengths, max_len):
        return (torch.arange(max_len, device=lengths.device)[None, :] < lengths[:, None]).float()

    def attention_ingredient_level(self, ingre_emb, u_emb, img_emb, ingre_num):
        n = ingre_emb.shape[1]
        feats = torch.cat([ingre_emb, u_emb[:, None, :].expand(-1, n, -1), img_emb[:, None, :].expand(-1, n, -1)], 2)
        logit = self.h_att_ingre(torch.tanh(self.W_att_ingre(feats))).squeeze(-1)
        weight = F.softmax(logit + (1.0 - self.sequence_mask(ingre_num, n)) * -1e12, dim=1)
        return torch.sum(weight[:, :, None] * ingre_emb, dim=1)

    def attention_id_ingre_image(self, u_emb, i_emb, ingre_att_emb, img_emb, hl_emb):
        b = u_emb.shape[0]
        comps = torch.stack([i_emb, ingre_att_emb, img_emb, hl_emb], 0)                 # component-major
        pairs = torch.cat([u_emb[None].expand(4, -1, -1), comps], 2)
        logit = self.h_att_comp(torch.tanh(self.W_att_comp(pairs))).reshape(4 * b)
        weight = F.softmax(logit.view(b, 4), dim=1)                                     # as the reference reads it
        return torch.sum(weight[:, :, None] * comps.permute(1, 0, 2), dim=1)

    def compute_score(self, user, item, ingre, ingre_num, img, hl, is_training, g2i_edges, i2u_edges,
                      ingre_embedding, gcn=None):
        """schgn.py:233-268.  `gcn` lets a caller share one GCN evaluation between calls."""
        ug, ig, gg, hg = self.gcn_tables(g2i_edges, i2u_edges) if gcn is None else gcn
        ingre_embedding_gcn = torch.cat([gg, self.ingre_embed_second, self.ingre_embed_mask], 0)
        u_emb, i_emb = _rows(self.user_embed, user), _rows(self.item_embed, item)
        ingre_emb, hl_emb = _rows(ingre_embedding, ingre), _rows(self.health_embed, hl)
        img_emb = self.img_trans(img.to(torch.float32))
        u_final, i_final = u_emb + _rows(ug, user), i_emb + _rows(ig, item)
        ingre_final, hl_final = ingre_emb + _rows(ingre_embedding_gcn, ingre), hl_emb + _rows(hg, hl)
        ingre_att = self.attention_ingredient_level(ingre_final, u_final, img_emb, ingre_num)
        item_att = self.attention_id_ingre_image(u_final, i_final, ingre_att, img_emb, hl_final)
        hidden = self.W_concat(torch.cat([u_final, item_att, u_final * item_att], 1))
        score = self.output_mlp(F.relu(F.dropout(hidden, p=0.5, training=is_training))).squeeze()
        return score, u_emb, i_emb, ingre_emb, hl_emb, ingre_embedding_gcn, item_att

    def masked_ingre_prediction(self, ingre_emb, target_emb):
        e = self.mip_norm(ingre_emb.view(-1, self.emb_size))
        return torch.sigmoid(torch.sum(e * target_emb.view(-1, self.emb_size), -1))

    def compute_ssl_loss(self, ingre_embedding, ingre_embedding_gcn, masked_ingre_seq, pos_ingre, neg_ingre):
        pad = ((masked_ingre_seq == self.n_ingredients).float() * -1e8)[:, None, None, :]
        encoded = self.ingre_encoder(_rows(ingre_embedding_gcn, masked_ingre_seq), pad,
                                     output_all_encoded_layers=True)[-1]
        pos = self.masked_ingre_prediction(encoded, _rows(ingre_embedding, pos_ingre))
        neg = self.masked_ingre_prediction(encoded, _rows(ingre_embedding, neg_ingre))
        dist = torch.sigmoid(pos - neg)
        loss = self.criterion(dist, torch.ones_like(dist))
        return torch.sum(loss * (masked_ingre_seq == self.n_ingredients + 1).float().flatten())

    def calculate_loss(self, batch_data):
        b = batch_data
        ingre_embedding = torch.cat([self.ingre_embed_first, self.ingre_embed_second, self.ingre_embed_mask], 0)
        gcn = self.gcn_tables()
        pos = self.compute_score(b["u_id"], b["pos_i_id"], b["pos_ingre_code"], b["pos_ingre_num"], b["pos_img"],
                                 b["pos_cl"].long(), True, self.g2i_edges, self.i2u_edges, ingre_embedding, gcn)
        neg = self.compute_score(b["u_id"], b["neg_i_id"], b["neg_ingre_code"], b["neg_ingre_num"], b["neg_img"],
                                 b["neg_cl"].long(), True, self.g2i_edges, self.i2u_edges, ingre_embedding, gcn)
        ssl_loss = self.ssl * self.compute_ssl_loss(ingre_embedding, pos[5], b["masked_ingre_seq"],
                                                    b["pos_ingre_seq"], b["neg_ingre_seq"])
        bpr_loss = -torch.sum(torch.log(torch.sigmoid(pos[0] - neg[0])))
        reg_loss = self.regs * (_sq(pos[1]) + _sq(pos[2]) + _sq(neg[2]) + _sq(pos[3]) + _sq(neg[3]))
        reg_loss = reg_loss + self.reg_health * (_sq(pos[4]) + _sq(neg[4]))
        reg_loss = reg_loss + self.reg_image * _sq(self.img_trans.weight)
        reg_loss = reg_loss + self.reg_w * (_sq(self.W_concat.weight) + _sq(self.output_mlp.weight))
        reg_loss = reg_loss + self.reg_g * _sq(self.new_gcn.conv1.lin.weight)
        return bpr_loss, reg_loss, ssl_loss

    # ------------------------------------------------------------------ candidate scoring (torch)
    def _inference_table(self):
        return torch.cat([self.ingre_embed_first, self.ingre_embed_second], 0)

    def inference_by_user(self, batch_data):
        b = batch_data
        return self.compute_score(b["user_input"], b["item_input"], b["ingre_input"], b["ingre_num_input"],
                                  b["img_input"], b["cal_level_input"], False, self.g2i_edges, self.i2u_edges,
                                  self._inference_table(), self._cached_gcn())[0]

    def sample_sort_predict(self, batch_data):
        b = batch_data
        n, m = b["u_id"].size(0), self.config["neg_sample_num"] + 1
        items = torch.cat([b["neg_i_id"], b["pos_i_id"].unsqueeze(1)], 1).view(-1)
        rows = items.shape[0]
        ingres = torch.cat([b["neg_ingre_code"], b["pos_ingre_code"].unsqueeze(1)], 1).view(rows, -1)
        nums = torch.cat([b["neg_ingre_num"], b["pos_ingre_num"].unsqueeze(1)], 1).view(-1)
        img = torch.cat([b["neg_img"], b["pos_img"].unsqueeze(1)], 1).view(rows, -1)
        hl = torch.cat([b["neg_cl"].long(), b["pos_cl"].long().unsqueeze(1)], 1).view(-1)
        users = b["u_id"].view(n, 1).expand(n, m).reshape(-1)
        return self.compute_score(users, items, ingres, nums, img, hl, False, self.g2i_edges, self.i2u_edges,
                                  self._inference_table(), self._cached_gcn())[0].view(n, m)

    # ------------------------------------------------------------------ full sort (fused kernels)
    def _stamp(self):
        # `_param_generation` is bumped by the step drivers (`train.mark_parameters_updated`): a CUDA-graph
        # replay updates the parameters without changing `data_ptr` / `_version`
        return (getattr(self, "_param_generation", 0),) + tuple((p.data_ptr(), p._version) for p in self.parameters())

    def train(self, mode: bool = True):
        self._eval_cache = None          # a mode switch never keeps user-independent tables of older parameters
        return super().train(mode)

    def _cached_gcn(self):
        if torch.is_grad_enabled():
            return self.gcn_tables()
        return self._item_side()["gcn"]

    @torch.no_grad()
    def _item_side(self):
        """Everything in the scorer that does not depend on the user, computed once per parameter
        version: the GCN tables, the projected image features, the final item / ingredient / health
        rows and their images under the attention and concat weights (SURVEY.md 8f-2)."""
        cache = self._eval_cache
        stamp = self._stamp()
        if cache is not None and cache["stamp"] == stamp:
            return cache
        ds, dev, e = self.dataset, self.user_embed.device, self.emb_size
        gcn = self.gcn_tables()
        ug, ig, gg, hg = gcn
        img = torch.as_tensor(np.asarray(ds.embImage, dtype=np.float32), device=dev)
        codes = torch.as_tensor(np.asarray(ds.ingredientCodeDict), device=dev).to(torch.int32).contiguous()
        nums = torch.as_tensor(np.asarray(ds.ingredientNum), device=dev).to(torch.int32).contiguous()
        cal = torch.as_tensor(np.asarray(ds.cal_level), device=dev).long()
        if codes.shape[1] > 32:
            raise _lib.FoodRecError("the fused SCHGN scorer holds at most 32 ingredient slots per recipe")
        Wi, bi = self.W_att_ingre.weight, self.W_att_ingre.bias          # [e, 3e]: ingredient | user | image
        Wc, bc = self.W_att_comp.weight, self.W_att_comp.bias            # [e, 2e]: user | component
        # ingredient rows as the inference path sees them: table row + GCN row; the padding code maps
        # to the all-zero `ingre_embed_second` on both sides
        ingre_final = torch.cat([self.ingre_embed_first + gg, self.ingre_embed_second * 2], 0)
        img_emb = self.img_trans(img)
        item_final = self.item_embed + ig
        health_final = (self.health_embed + hg)[cal]
        cache = {
            "stamp": stamp, "gcn": gcn, "codes": codes, "nums": nums,
            "user_final": (self.user_embed + ug).contiguous(),
            "ingre_final": ingre_final.contiguous(),
            "ingre_key": (ingre_final @ Wi[:, :e].t()).contiguous(),          # W_att_ingre[:, ingredient] image
            "ingre_comp": (ingre_final @ Wc[:, e:].t()).contiguous(),         # W_att_comp[:, component] image
            "img_key": (img_emb @ Wi[:, 2 * e:].t() + bi).contiguous(),
            "comps": torch.stack([item_final, img_emb, health_final], 1).contiguous(),          # [I, 3, e]
            "comp_keys": torch.stack([item_final @ Wc[:, e:].t(), img_emb @ Wc[:, e:].t(),
                                      health_final @ Wc[:, e:].t()], 1).contiguous(),           # [I, 3, e]
            "Wi_user": Wi[:, e:2 * e].t().contiguous(), "Wc_user": Wc[:, :e].t().contiguous(), "bc": bc,
        }
        self._eval_cache = cache
        return cache

    def _scorer_tables(self, users: torch.Tensor):
        """The fused scorer's operands for `users`: their projected rows and the cached item-side tables."""
        c = self._item_side()
        e = self.emb_size
        u = c["user_final"][users]
        Wk, bk = self.W_concat.weight, self.W_concat.bias               # [e, 3e]: user | item | user * item
        return dict(
            user_final=u, user_key=u @ c["Wi_user"], user_comp=u @ c["Wc_user"] + c["bc"],
            user_hidden=u @ Wk[:, :e].t() + bk, W_item=Wk[:, e:2 * e].contiguous(), W_prod=Wk[:, 2 * e:].contiguous(),
            w_out=self.output_mlp.weight.reshape(-1).contiguous(), h_ingre=self.h_att_ingre.weight.reshape(-1),
            h_comp=self.h_att_comp.weight.reshape(-1), codes=c["codes"], nums=c["nums"], ingre_key=c["ingre_key"],
            ingre_final=c["ingre_final"], ingre_comp=c["ingre_comp"], img_key=c["img_key"], comps=c["comps"],
            comp_keys=c["comp_keys"])

    @torch.no_grad()
    def full_sort_scores(self, users: torch.Tensor, topk: int | None = None, hist=None):
        """Scores `[n_users_in_batch, n_items]` of the given users against every item; with `topk=k` the fused
        selection `(values [n, k], indices [n, k])` instead (the score block is never materialised)."""
        from .. import evaluation
        users = users.to(self._item_side()["user_final"].device).long().reshape(-1)
        return evaluation.schgn_pair_scores(topk=topk, user_ids=users, hist=hist, **self._scorer_tables(users))

    @torch.no_grad()
    def by_user_scores(self, users: torch.Tensor, cand_ptr, cand_items: torch.Tensor, block_pairs: int = 1 << 22):
        """By-user evaluation scores: user `users[r]` against its candidate list `cand_items[cand_ptr[r]:cand_ptr[r+1]]`
        (host `cand_ptr` from 0), each list scored as `inference_by_user` scores it in one batch -- including the
        reference's `.view(b, -1)` mixing of the list's component logits, so a score depends on the list's order and
        length.  Returns the flat fp32 device scores in list order.  Fused kernels `fr_schgn_attend_pairs` /
        `fr_schgn_score_pairs` over the cached item-side tables (`train.mark_parameters_updated` invalidates them)."""
        from .. import evaluation
        users = torch.as_tensor(users).to(self._item_side()["user_final"].device).long().reshape(-1)
        return evaluation.schgn_by_user_scores(cand_ptr, cand_items, block_pairs=block_pairs,
                                               **self._scorer_tables(users))

    def full_sort_predict(self, batch_data):
        """schgn.py:318-345: the batch user(s) against all items; `[n_items]` for one user (what
        `Trainer.evaluate` feeds `torch.topk`), `[n, n_items]` for several."""
        s = self.full_sort_scores(batch_data["u_id"].reshape(-1))
        return s[0] if s.shape[0] == 1 else s

    @torch.no_grad()
    def full_sort_topk(self, users: torch.Tensor, k: int, hist=None, block: int = 256):
        """Top-k items per user (values, int64 indices; score descending, ties to the lower item), 16 users per pass
        of the attention kernel, the selection fused into the scorer (`fr_schgn_score_topk`): `[users, items]` scores
        never reach HBM.  `hist` (`evaluation.HistoryCSR`) masks training interactions (the reference does not mask).
        `k` beyond the kernel's 64 falls back to dense scores + `torch.topk`."""
        users = users.reshape(-1)
        if k <= min(64, self.n_items):
            return self.full_sort_scores(users, topk=k, hist=hist)
        return self._full_sort_topk_dense(users, k, hist, block)

    @torch.no_grad()
    def _full_sort_topk_dense(self, users, k, hist, block):
        vals, idx = [], []
        for s in range(0, users.numel(), block):
            ub = users[s:s + block]
            sc = self.full_sort_scores(ub)
            if hist is not None:
                hist.mask_scores_(sc, ub)
            v, i = torch.topk(sc, k, dim=-1)
            vals.append(v)
            idx.append(i)
        return torch.cat(vals), torch.cat(idx)
