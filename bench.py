#!/usr/bin/env python
"""Benchmark of the graph-propagation + ranking hot path (contract: see DESIGN.md section "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--scale C2] [--dump-outputs DIR]

One "step" = one training batch (B = 512) of the CLUSSL model on the synthetic Allrecipes-scale
graph C2: full propagation over the four normalised graphs (forward), fused BPR / regulariser /
distance-correlation losses, backward through every propagation, Adam step -- the per-batch body of
the reference's `Trainer._train_epoch` (FoodRec/common/trainer.py:177-224).  The headline metric is
train epochs/s = 1 / (ceil(n_train / B) * seconds per step).  `value` is measured with the batch
indices already resident in HBM; `e2e` goes through the public model API with pinned HOST batches
(H2D inside the timed region) and reads every loss term back (D2H), like the reference trainer.

Beside the headline the same JSON line carries (each with its own roofline):
  parity                  loss terms + sampled gradient rows of the first batch vs the CPU oracle on this very graph
  eval / eval_c4          full-sort top-20 with history mask: C2 users, and the 1 M x 500 k sweep, user-sharded over the
                          ranks INCLUDING the final [U/P, k] gather
  partitioned_propagation row-partitioned 3-layer fwd+bwd propagation on a C5-shaped device-built graph (same total
                          problem at every N: strong scaling), NCCL all-gather path and peer-store (push) path
  knn                     cosine kNN (D = 4096 / 384) and centroid assignment shapes of the ranking kernel
  clussl_c3               the same CLUSSL step on the Foodcom-scale synthetic C3 (BASELINE.json configs[2]), 1 and N GPUs
  torch_cuda_baseline     the stock-PyTorch-on-the-same-GPU arm (uncoalesced COO `torch.sparse.mm`, stack/mean,
                          autograd, default Adam; `matmul` + `topk`): the bar SURVEY.md 2.1 names
  cpu_baseline            the oracle port on the host cores (context only)

`--impl reference` times the CPU restatement of the reference path (oracle/, torch-CPU ops -- the
same library ops the reference calls) on the host cores, same workload and metric.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from untouched (no __pycache__ in it)

import numpy as np  # noqa: E402
import torch  # noqa: E402

BATCH = 512
METRIC, UNIT = "train_epochs_per_s", "epochs/s"
PARAM_NAMES = ("user_embedding.weight", "item_embedding.weight", "ingre_embedding.weight",
               "image_prototype_embedding.weight", "text_prototype_embedding.weight")


class Cfg(dict):
    def __getitem__(self, k):
        return self.get(k)


def model_cfg(ds, device):
    # configs/model/PRICAI_ModelX.yaml (allrecipe block) + configs/overall.yaml
    return Cfg(device=device, embedding_size=64, train_batch_size=BATCH, is_multimodal_model=True, end2end=False,
               use_health_level_multi_hot=True, n_ri_layers=2, n_mm_layers=1, n_ui_layers=1, reg_weight=0.01,
               loss_cl=0.1, n_cluster=ds.cfg.n_cluster, knn_k=10, mm_image_weight=0.1, learning_rate=0.002)


def workload_name(scale, ds):
    return (f"{scale}: CLUSSL (PRICAI_ModelX) train step, B={BATCH}, {ds.n_users} users / {ds.n_items} items / "
            f"{ds.n_train} train interactions, {ds.cfg.n_cluster} clusters x2 (from {ds.cfg.dv}-d image / "
            f"{ds.cfg.dt}-d text features), {ds.num_ingredients} ingredients, d=64, "
            f"2 item-side layers x3 graphs + 1 user-item layer, fwd+bwd+Adam")


def config_of(scale, ds, world, steps_per_epoch):
    """Identical for both arms (the driver compares the two `config` objects)."""
    return {"workload": workload_name(scale, ds), "steps_per_epoch": steps_per_epoch,
            "multi_gpu": "single GPU" if world == 1 else
                         f"{world} ranks: replicated graph, per-rank batches of {BATCH}, NCCL all-reduce (AVG) of the dense "
                         f"gradients inside the captured step (weak scaling; see dp_control for the single-GPU control)"}


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm))
        return out


# ------------------------------------------------------------------------------- reference (oracle) arm
class OracleClussl:
    """Restatement of the reference's CLUSSL train step (oracle/, stock torch ops).  On the CPU it is the
    `cpu_baseline` leg and `--impl reference`; with `device='cuda'` the very same code is the stock-PyTorch-on-GPU
    arm (`torch_cuda_baseline`: uncoalesced COO `torch.sparse.mm`, stack/mean, autograd, default Adam)."""

    def __init__(self, ds, state_dict, lr, device="cpu", dtype=torch.float32):
        from oracle import adjacency
        self.ds = ds

        def adj(S):   # as the reference: an (uncoalesced-flagged) sparse COO moved to the device
            return S.to(device=device, dtype=dtype) if (device != "cpu" or dtype != torch.float32) else S
        self.S_ui = adj(adjacency.norm_adj_user_item(ds.train_coo_matrix, ds.n_users, ds.n_items))
        self.S_g = adj(adjacency.norm_adj_item_side(ds.rIngre_triples, ds.n_items, ds.num_ingredients))
        self.S_v = adj(adjacency.norm_adj_item_side(ds.image_cluster_triples, ds.n_items, ds.cfg.n_cluster))
        self.S_t = adj(adjacency.norm_adj_item_side(ds.text_cluster_triples, ds.n_items, ds.cfg.n_cluster))
        self.P = {k: state_dict[k].detach().to(device=device, dtype=dtype).clone().requires_grad_(True) for k in PARAM_NAMES}
        self.opt = torch.optim.Adam(list(self.P.values()), lr=lr)
        self.device = device

    def losses(self, batch):
        from oracle import losses, propagation
        ds, P = self.ds, self.P
        out = propagation.clussl_forward(
            self.S_ui, self.S_g, self.S_v, self.S_t, P["user_embedding.weight"], P["item_embedding.weight"],
            P["ingre_embedding.weight"], P["image_prototype_embedding.weight"], P["text_prototype_embedding.weight"],
            ds.n_users, ds.n_items, ds.num_ingredients, ds.cfg.n_cluster, 2, 1)
        u, p, n = (torch.as_tensor(batch[k]).to(self.device) for k in ("u_id", "pos_i_id", "neg_i_id"))
        return losses.clussl_loss(out, P["user_embedding.weight"], P["item_embedding.weight"], u, p, n, 0.01, 0.1)

    def loss_and_grads(self, batch):
        self.opt.zero_grad()
        terms = self.losses(batch)
        sum(terms).sum().backward()
        return [float(t) for t in terms], {k: v.grad.detach() for k, v in self.P.items()}

    def step(self, batch):
        self.opt.zero_grad()
        terms = self.losses(batch)
        sum(terms).sum().backward()
        self.opt.step()
        return terms


def time_cpu(oracle, batches, steps, warmup):
    for i in range(warmup):
        oracle.step(batches[i % len(batches)])
    t0 = time.perf_counter()
    for i in range(steps):
        oracle.step(batches[(warmup + i) % len(batches)])
    return (time.perf_counter() - t0) / steps


def ev_pair():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def timed_graph_ms(fn, reps):
    """Average device time of one `fn()` when `reps` of them run back to back: the calls are captured into a CUDA
    graph (no Python between the launches) and one replay is timed with events."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(3):
        a, b = ev_pair()
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best / reps


def timed_ms(fn, iters, warm=2):
    """Median-free simple device timing: `iters` calls between one CUDA-event pair on the current stream."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = ev_pair()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


# ------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", default="C2")
    ap.add_argument("--cpu-steps", type=int, default=3, help="steps of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-schgn", action="store_true", help="skip the SCHGN side measurement")
    ap.add_argument("--no-extras", action="store_true", help="headline + eval only (skip C4, partitioned propagation, kNN, baselines)")
    ap.add_argument("--eager", action="store_true", help="drop-in eager step (no CUDA graph)")
    ap.add_argument("--foreach-adam", action="store_true", help="torch's default foreach Adam instead of fused=True")
    ap.add_argument("--torch-adam", action="store_true", help="torch.optim.Adam(fused=True) instead of this library's fr_adam_step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss terms and the updated parameters to "
                         "DIR/<name>.npy (float32)")
    ap.add_argument("--c5-scale", type=float, default=0.2,
                    help="size of the partitioned-propagation graph relative to BASELINE configs[4] (1.0 = 10 M users / 2 M items "
                         "/ 200 M interactions; default 0.2 keeps the default run short)")
    ap.add_argument("--only", default="", help="comma list of side measurements to run (eval_c4, partitioned_propagation, "
                                               "dp_control, clussl_c3, knn, schgn, healthrec, torch_cuda_baseline); default all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 train step")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import foodrec_b200  # noqa: F401
    from foodrec_b200.synth import make_dataset, sample_train_batches

    if args.impl == "reference":
        if rank != 0:
            return 0
        torch.set_num_threads(os.cpu_count() or 1)
        ds = make_dataset(args.scale)
        steps_per_epoch = math.ceil(ds.n_train / BATCH)
        torch.manual_seed(999)
        sd = _init_state_dict(ds)
        oracle = OracleClussl(ds, sd, 0.002)
        batches = sample_train_batches(ds, BATCH, min(8, args.steps + args.warmup), seed=7)
        timed = args.steps
        s = time_cpu(oracle, batches, timed, min(args.warmup, 3))
        v = 1.0 / (steps_per_epoch * s)
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": s * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args.scale, ds, args.gpus, steps_per_epoch),
            "timed_steps": timed,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"{timed} train batches of {BATCH} (full-graph fwd+bwd+Adam each), "
                                       f"extrapolated to {steps_per_epoch} batches/epoch"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    # ------------------------------------------------------------------ B200 arm
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from foodrec_b200 import _lib, ops
    from foodrec_b200.models.pricai_modelx import PRICAI_ModelX

    ds = make_dataset(args.scale)
    steps_per_epoch = math.ceil(ds.n_train / BATCH)
    cfg = model_cfg(ds, str(dev))
    torch.manual_seed(999)
    model = PRICAI_ModelX(cfg, ds)
    sd0 = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.to(dev)
    model.train()
    # trainer.py:142-143 builds optim.Adam(params, lr, weight_decay).  Same optimizer, torch's fused
    # multi-tensor implementation (one launch instead of ~15), capturable so the step stays on the device.
    if args.torch_adam or args.foreach_adam:
        opt = torch.optim.Adam(model.parameters(), lr=cfg["learning_rate"], weight_decay=0.0,
                               capturable=not args.eager, fused=not args.foreach_adam)
    else:   # the same update as one multi-tensor launch of this library (train.FusedAdam, fr_adam_step)
        from foodrec_b200.train import FusedAdam
        opt = FusedAdam(model.parameters(), lr=cfg["learning_rate"])
    # weak scaling: every rank trains on its own batches of the replicated graph (see DESIGN.md, multi-GPU)
    host_batches = sample_train_batches(ds, BATCH, 64, seed=7 + rank)
    keys = ("u_id", "pos_i_id", "neg_i_id")
    pinned = [{k: torch.from_numpy(b[k]).pin_memory() for k in keys} for b in host_batches]
    resident = [{k: v.to(dev) for k, v in b.items()} for b in pinned]

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity at the benchmarked configuration: the first batch's loss terms and gradients (from the initial
    #      state) against the CPU oracle on this very graph, before anything has been trained
    parity = _parity_c2(model, ds, sd0, cfg, host_batches[0], resident[0]) if (world == 1 and not args.no_cpu_baseline) else None

    from foodrec_b200.train import GraphedTrainStep

    def eager(batch):
        opt.zero_grad()
        losses = model.calculate_loss(batch)
        loss = sum(losses)
        loss.backward()
        if world > 1 and hook is None:
            _allreduce_grads(model, world)
        elif world > 1:
            hook()
        opt.step()
        return losses

    hook = None
    step_mode = "eager"
    if args.eager:
        step = eager
    else:
        from foodrec_b200.train import OverlappedGradAllReduce
        try:   # N > 1: per-gradient NCCL all-reduces on a side stream, captured inside the graph
            hook = OverlappedGradAllReduce(model) if world > 1 else None
            step = GraphedTrainStep(model, opt, resident[0], keys=keys, grad_hook=hook)
            step_mode = "cuda_graph_replay"
        except Exception as e:  # noqa: BLE001  (capture of a collective refused: stay eager, say so)
            print(f"[bench] graph capture failed, running eager: {e}", file=sys.stderr)
            if world > 1 and hook is not None:
                hook.remove()
                hook = None
            step = eager

    # ---- value: inputs resident in HBM, --steps timed steps (each a different batch)
    sampler = ClockSampler(local_rank) if rank == 0 else None   # nvidia-smi needs ~0.3 s to start sampling
    for i in range(max(args.warmup, 3)):
        step(resident[i % len(resident)])
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = ev_pair()
    e0.record()
    for i in range(args.steps):
        last_losses = step(resident[(args.warmup + i) % len(resident)])
    e1.record()
    barrier()
    timed_steps = args.steps
    ms_dev = e0.elapsed_time(e1) / timed_steps
    launches = _lib.launch_count() - l0
    if args.dump_outputs and rank == 0:     # now: the steps below keep training the same model
        _dump_outputs(args.dump_outputs, last_losses, model)

    # ---- e2e: pinned host batches in, loss terms out, through the public model API
    h2d = sum(v.numel() * v.element_size() for v in pinned[0].values())
    graphed = step_mode == "cuda_graph_replay"

    def e2e_step(host_batch):
        if graphed:       # pinned host tensors -> the graph's static inputs (H2D), replay, all loss terms in one D2H
            step(host_batch)
            return step.loss_values()
        losses = step({k: v.to(dev, non_blocking=True) for k, v in host_batch.items()})
        return [float(x.item()) for x in losses]  # trainer.py:186: per-term .item()
    for i in range(2):
        e2e_step(pinned[i % len(pinned)])
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    n_e2e = args.steps
    for i in range(n_e2e):
        vals = e2e_step(pinned[(args.warmup + i) % len(pinned)])
        d2h = 4 * len(vals)
    barrier()
    ms_e2e = (time.perf_counter() - t0) * 1e3 / n_e2e
    clocks = sampler.stop() if sampler else None

    # ---- roofline of the dominant kernel (propagation SpMM), CUDA events around every launch
    prof = []
    model.fork_streams = False      # serialise the sub-graphs so each launch is timed alone on its stream
    ops.PROFILE = prof
    for i in range(3):
        eager(resident[i % len(resident)])  # same kernels as the graph replays; events need eager launches
    torch.cuda.synchronize()
    ops.PROFILE = None
    model.fork_streams = True
    l1 = _lib.launch_count()
    eager(resident[0])
    launches_per_step_eager = _lib.launch_count() - l1  # kernels of this library per step (graph replays the same)
    # Each of the step's propagation launches (3 eager steps recorded) is re-issued 20x back to back with the
    # same plan and operand shapes, bracketed by one CUDA-event pair on the launch stream: the stream stays
    # busy, so the figure is kernel time, not Python launch latency.  Operands stay L2-warm, as inside the step.
    tot_ms, tot_bytes, n_launch, REP = 0.0, 0.0, len(prof), 20
    probe_tot, gathered = 0.0, 0.0          # the same launches' row gathers alone (`fr_probe_gather`): the gather roofline
    probe_out = torch.empty(148 * 32 * 32, device=dev)
    bufs = {}
    def _buf(gr):
        key = (gr.n_rows, gr.n_cols)
        if key not in bufs:
            bufs[key] = (torch.randn(gr.n_cols, 64, device=dev), torch.randn(gr.n_rows, 64, device=dev),
                         torch.empty(gr.n_rows, 64, device=dev))
        return bufs[key]

    def _probe(gr, X):
        _lib.check(_lib.lib.fr_probe_gather(X.data_ptr(), 64, gr.col.data_ptr(), gr.nnz, 8, 148 * 32, probe_out.data_ptr(),
                                            _lib.stream_ptr()), "fr_probe_gather")
    n_grouped = 0
    for _, _, nb, g, has_z in prof:
        if isinstance(g, ops.PropGroup):      # one grouped launch over several graphs (CLUSSL's item-side layer)
            n_grouped += 1
            bs = [_buf(gr) for gr in g.graphs]
            Xs, Zs, Ys = [b[0] for b in bs], [b[1] if has_z else None for b in bs], [b[2] for b in bs]
            tot_ms += timed_graph_ms(lambda: ops.spmm_grouped(g, Xs, Zs, 0.5, 0.5, outs=Ys), REP)
            for gr, X in zip(g.graphs, Xs):
                probe_tot += timed_ms(lambda: _probe(gr, X), REP, warm=1)
                gathered += gr.nnz * 256.0
        else:
            X, Z, Y = _buf(g)
            tot_ms += timed_graph_ms(lambda: ops.spmm(g, X, Z=Z if has_z else None, alpha=0.5, beta=0.5, out=Y), REP)
            probe_tot += timed_ms(lambda: _probe(g, X), REP, warm=1)
            gathered += g.nnz * 256.0
        tot_bytes += nb
    del bufs
    peaks = _peaks()
    achieved = tot_bytes / (tot_ms * 1e-3) / 1e9 if tot_ms > 0 else 0.0
    tpeak = _tensor_peak()

    ev = _bench_eval(model, ds, dev, rank, world, barrier)
    extras = {}
    only = {x.strip() for x in args.only.split(",") if x.strip()}

    def side(name, fn, *a):
        """A side measurement must not cost the headline line: on one GPU a failure is recorded under its key (with
        several ranks it propagates -- the other ranks would wait in a collective)."""
        if only and name not in only:
            return
        if world > 1:
            extras[name] = fn(*a)
            return
        try:
            extras[name] = fn(*a)
        except Exception as e:  # noqa: BLE001
            extras[name] = {"error": f"{type(e).__name__}: {e}"}
            print(f"[bench] {name} failed: {e}", file=sys.stderr)
    if not args.no_extras:
        side("eval_c4", _bench_eval_c4, dev, rank, world, barrier, tpeak)
        side("partitioned_propagation", _bench_partitioned_propagation, dev, rank, world, barrier, peaks, args.c5_scale)
        if world > 1:
            side("dp_control", _bench_dp_control, model, ds, cfg, dev, world, steps_per_epoch)
        side("clussl_c3", _bench_c3, dev, rank, world, barrier)
    times = torch.tensor([ms_dev, ms_e2e, ev["ms_dev"], ev["ms_e2e"], ev["kernel_ms"]], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = float(times[0]), float(times[1])
    ev.update(ms_dev=float(times[2]), ms_e2e=float(times[3]), kernel_ms=float(times[4]))
    if rank != 0:
        return 0

    value = world / (steps_per_epoch * ms_dev * 1e-3)
    e2e = world / (steps_per_epoch * ms_e2e * 1e-3)
    ws_mb = _working_set_mb(model, opt)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": config_of(args.scale, ds, world, steps_per_epoch),
        "timed_steps": timed_steps,
        "l2": f"no explicit flush: step working set {ws_mb:.0f} MB (params+grads+Adam state+graphs+activations) exceeds the "
              f"126 MB L2",
        "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "timed_steps": n_e2e},
        "gpu_launches": int(launches) if step_mode == "eager" else int(launches_per_step_eager * timed_steps),
        "step_mode": step_mode,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "spmm_group_kernel<64,8,4> (user-item graph) + spmm_grouped_kernel<64> (the three "
                                               "item-side graphs of a layer in one grid)", "achieved": achieved, "peak": peaks[0],
                     "unit": "GB/s", "frac": achieved / peaks[0], "traffic": _spmm_traffic(), "peak_source": peaks[1],
                     "traffic_source": "profiles/: mean dram read+write bytes per launch, ncu --set full over the propagation "
                                       "launches of one step (below the algorithmic bytes: the step's tables stay in the 126 MB L2)",
                     "algorithmic_bytes_per_launch": tot_bytes / max(n_launch, 1),
                     "launches_per_step": n_launch / 3, "avg_launch_us": tot_ms * 1e3 / max(n_launch, 1),
                     "kernel_share_of_step": tot_ms / 3 / ms_dev,
                     "gather_bound": {
                         "note": "the tables are L2-resident at this scale, so the binding resource is the 256-byte row "
                                 "gather (L1/L2 -> SM), not HBM: `fr_probe_gather` issues only the gathers of the same "
                                 "launches (same column indices, nothing else) and is the ceiling for any gather-based SpMM; "
                                 "the HBM-regime figure is partitioned_propagation.single_gpu_roofline",
                         "gathered_GBs_in_kernel": gathered / (tot_ms * 1e-3) / 1e9,
                         "gather_only_probe_GBs": gathered / (probe_tot * 1e-3) / 1e9,
                         "kernel_time_over_gather_only_time": tot_ms / probe_tot, "frac_of_gather_roofline": probe_tot / tot_ms}},
    }
    if parity is not None:
        line["parity"] = parity
    n_eval = ev["n_users"]
    per_gpu_tfl = ev["flops_local"] / (ev["kernel_ms"] * 1e-3) / 1e12
    line["eval"] = {
        "metric": "full_sort_eval_users_per_s", "unit": "users/s",
        "workload": f"{n_eval} users x {ds.n_items} items, d=64, top-20, training-history mask, bf16 tcgen05 scores + fp32 "
                    f"re-score with per-row certificate, users sharded over {world} GPU(s), final [U/P, 20] gather included",
        "value": n_eval / (ev["ms_dev"] * 1e-3), "ms": ev["ms_dev"],
        "e2e": {"value": n_eval / (ev["ms_e2e"] * 1e-3), "ms": ev["ms_e2e"], "h2d_bytes": ev["h2d"],
                "d2h_bytes": ev["d2h"], "index_dtype": "int32"},
        "roofline": {"bound": "tensor", "kernel": "rank_topk_pair_kernel (cta_group::2; bounding + collection sweeps, FLOPs counted once)",
                     "achieved": per_gpu_tfl, "peak": tpeak[0], "unit": "TFLOP/s", "frac": per_gpu_tfl / tpeak[0],
                     "per": "GPU (this rank's users only)", "traffic": None, "peak_source": tpeak[1]},
        "exactness": ev.get("stats"),
        "metrics_vs_oracle": ev.get("metrics"),
    }
    if world == 1 and not args.no_extras:
        side("knn", _bench_knn, ds, dev, tpeak)
    if world == 1 and not args.no_schgn:
        torch.set_num_threads(os.cpu_count() or 1)
        side("schgn", _bench_schgn, ds, dev, steps_per_epoch, not args.no_cpu_baseline)
    if world == 1 and not args.no_extras:
        side("healthrec", _bench_healthrec, ds, dev, steps_per_epoch, peaks)
    if world == 1 and not args.no_extras:
        side("torch_cuda_baseline", _bench_torch_cuda, ds, sd0, cfg, host_batches, dev, steps_per_epoch, ms_dev, ev, model)
    line.update(extras)
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        oracle = OracleClussl(ds, sd0, cfg["learning_rate"])
        s = time_cpu(oracle, host_batches, args.cpu_steps, 1)
        line["cpu_baseline"] = {"value": 1.0 / (steps_per_epoch * s), "unit": UNIT, "cores": torch.get_num_threads(),
                                "kind": "port", "ms_per_step": s * 1e3,
                                "sample": f"{args.cpu_steps} train batches of {BATCH} on the same graph "
                                          f"(full fwd+bwd+Adam each), extrapolated to {steps_per_epoch} batches/epoch"}
    print(json.dumps(line))
    return 0


DUMP_LIMIT_BYTES = 64 << 20


def _dump_outputs(out_dir, losses, model):
    """What one train step hands its caller, the loss terms (mf, cl, reg), and what it leaves behind, every parameter
    after the optimizer step, as `out_dir/<name>.npy` in float32.  Model, batches and step count are seeded, so two
    builds run with the same arguments can be compared file by file.  The step sums gradients with float atomics and
    Adam turns gradients that are pure rounding noise into +-lr updates, so one build differs from run to run too: at
    C2 with --steps 300 (B200, 1000 W power limit) the loss terms agreed to 1e-6 and each parameter table to 5e-5 in
    relative L2 norm, single entries differing by up to 2e-3."""
    arrays = {"losses": torch.stack([t.detach().reshape(()).float() for t in losses]).cpu().numpy()}
    for name, p in model.named_parameters():
        arrays[name] = p.detach().float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------ parity at C2
def _parity_c2(model, ds, sd0, cfg, host_batch, dev_batch, n_rows=1024):
    """First batch from the initial state: every loss term and `n_rows` sampled gradient rows per table (the rows the
    batch touches first, then random ones) of the GPU step against the CPU oracle (fp32, the reference's own ops)
    following FoodRec/models/pricai_modelx.py:234-276.  The oracle is also run in fp64: `*_vs_f64` columns say how far
    the fp32 reference itself is from exact arithmetic -- the yardstick for the GPU's own distance."""
    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.perf_counter()
    model.zero_grad(set_to_none=True)
    terms = model.calculate_loss(dev_batch)
    sum(terms).backward()
    torch.cuda.synchronize()
    g_terms = [float(t) for t in terms]
    rng = np.random.default_rng(0)
    names = {"user_embedding.weight": model.user_embedding.weight, "item_embedding.weight": model.item_embedding.weight,
             "ingre_embedding.weight": model.ingre_embedding.weight,
             "image_prototype_embedding.weight": model.image_prototype_embedding.weight,
             "text_prototype_embedding.weight": model.text_prototype_embedding.weight}
    touched = {"user_embedding.weight": np.unique(host_batch["u_id"]),
               "item_embedding.weight": np.unique(np.concatenate([host_batch["pos_i_id"], host_batch["neg_i_id"]]))}
    rows = {}
    for k, p in names.items():
        n = p.shape[0]
        t = touched.get(k, np.empty(0, np.int64))[: n_rows // 2]
        rows[k] = np.unique(np.concatenate([t, rng.choice(n, size=min(n, n_rows - t.size), replace=False)]))
    g_grads = {k: p.grad[torch.from_numpy(rows[k]).to(p.device)].cpu() for k, p in names.items()}
    model.zero_grad(set_to_none=True)
    o32 = OracleClussl(ds, sd0, cfg["learning_rate"])
    r_terms, r_grads = o32.loss_and_grads(host_batch)
    o64 = OracleClussl(ds, sd0, cfg["learning_rate"], dtype=torch.float64)
    x_terms, x_grads = o64.loss_and_grads(host_batch)

    def rel(a, b):
        return abs(a - b) / max(abs(b), 1e-30)

    def grel(a, b):      # max-norm relative error over the sampled rows
        b = b.double()
        return float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-30))
    term_names = ("mf_loss", "cl_loss", "reg_loss")
    out = {"config": "C2, first batch from the initial state, fwd + bwd (no optimizer step)",
           "oracle": "oracle/ CLUSSL step on the host (torch-CPU fp32: the reference's own ops) and the same in fp64",
           "loss": {n: {"gpu": g, "oracle_f32": r, "rel_err_vs_oracle_f32": rel(g, r), "gpu_rel_err_vs_f64": rel(g, x),
                        "oracle_f32_rel_err_vs_f64": rel(r, x)}
                    for n, g, r, x in zip(term_names, g_terms, r_terms, x_terms)},
           "grad": {k: {"rows_compared": int(rows[k].size),
                        "rel_err_vs_oracle_f32": grel(g_grads[k], r_grads[k][rows[k]]),
                        "gpu_rel_err_vs_f64": grel(g_grads[k], x_grads[k][rows[k]]),
                        "oracle_f32_rel_err_vs_f64": grel(r_grads[k][rows[k]], x_grads[k][rows[k]])}
                    for k in names}}
    out["loss_rel_err"] = max(v["rel_err_vs_oracle_f32"] for v in out["loss"].values())
    out["grad_rel_err"] = max(v["rel_err_vs_oracle_f32"] for v in out["grad"].values())
    # The bar: losses 1e-5 relative (north star).  Gradients: 2e-5, except that no implementation can be asked to sit
    # closer to the fp32 reference than the fp32 reference sits to exact arithmetic (the distance-correlation term is
    # ill-conditioned: its diagonal 1/(2 D_ii) = 5000 factors cancel only numerically) -- so a table passes when the GPU
    # is within 2e-5 of the fp32 oracle OR at least as close to the fp64 result as the fp32 oracle is.
    out["tolerance"] = {"loss_rel": 1e-5, "grad_rel": 2e-5, "grad_alt": "gpu_rel_err_vs_f64 <= oracle_f32_rel_err_vs_f64 + 2e-5"}
    loss_ok = all(v["rel_err_vs_oracle_f32"] <= 1e-5 or v["gpu_rel_err_vs_f64"] <= v["oracle_f32_rel_err_vs_f64"] + 1e-5
                  for v in out["loss"].values())
    grad_ok = all(v["rel_err_vs_oracle_f32"] <= 2e-5 or v["gpu_rel_err_vs_f64"] <= v["oracle_f32_rel_err_vs_f64"] + 2e-5
                  for v in out["grad"].values())
    out["ok"] = bool(loss_ok and grad_ok)
    out["seconds"] = time.perf_counter() - t0
    return out


SCHGN_CFG = dict(embedding_size=64, train_batch_size=BATCH, is_multimodal_model=True, end2end=False,
                 num_attention_heads=2, num_hidden_layers=2, hidden_act="gelu", inner_size=256, hidden_dropout_prob=0.5,
                 attention_probs_dropout_prob=0.5, regs=0.01, reg_image=1, reg_w=0.05, reg_g=0.01, reg_health=0.01,
                 ssl=0.008, SCHGN_ssl=True, neg_sample_num=4, learning_rate=0.0005)  # configs/model/SCHGN.yaml


def _bench_schgn(ds, dev, steps_per_epoch, cpu_baseline):
    """BASELINE.json configs[1] names SCHGN on this graph: its train step (GCN on the propagation kernel,
    kernel gathers, batch-sized scorer in torch; one CUDA-graph replay per batch) and its full sort (fused pair
    scorer, 256 users) -- reported beside the headline, each with the CPU restatement timed on the host."""
    from foodrec_b200 import _lib
    from foodrec_b200.models.schgn import SCHGN
    from foodrec_b200.synth import sample_train_batches
    from foodrec_b200.train import GraphedTrainStep
    cfg = Cfg({**SCHGN_CFG, "device": str(dev)})
    torch.manual_seed(999)
    model = SCHGN(cfg, ds)
    sd0 = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.to(dev).train()
    host = sample_train_batches(ds, BATCH, 4, seed=21, schgn=True)
    batches = [{k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in b.items()} for b in host]
    opt = torch.optim.Adam(model.parameters(), lr=cfg["learning_rate"], fused=True, capturable=True)
    l0 = _lib.launch_count()
    step = GraphedTrainStep(model, opt, batches[0], keys=tuple(batches[0].keys()), warmup=3)
    launches_per_step = (_lib.launch_count() - l0) / 4          # 3 eager warm-up steps + the capture pass
    it = iter(range(10 ** 9))
    ms = timed_ms(lambda: step(batches[next(it) % 4]), 50, warm=5)
    n_nodes = ds.n_users + ds.n_items + ds.num_ingredients + ds.num_calories_level
    out = {"workload": f"SCHGN on the same graph: GCN over {n_nodes} nodes, B={BATCH}, {ds.image_size}-d image rows, "
                       f"masked-ingredient task, Adam; dropout on",
           "train_ms_per_step": ms, "train_epochs_per_s": 1.0 / (steps_per_epoch * ms * 1e-3),
           "library_launches_per_step": launches_per_step}
    model.eval()
    users = torch.arange(256, device=dev)
    with torch.no_grad():
        fs_ms = timed_ms(lambda: model.full_sort_topk(users, 20), 2, warm=1)
    out["full_sort"] = {"workload": f"256 users x {ds.n_items} items through the fused pair scorer + top-20",
                        "ms": fs_ms, "users_per_s": 256 / (fs_ms * 1e-3), "pairs_per_s": 256 * ds.n_items / (fs_ms * 1e-3)}
    if cpu_baseline:
        from oracle import schgn as O
        P = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and k != "ingre_embed_second")
             for k, v in sd0.items()}
        popt = torch.optim.Adam([v for v in P.values() if v.requires_grad], lr=cfg["learning_rate"])
        ei = O.schgn_edge_index(ds)
        sizes = (ds.n_users, ds.n_items, ds.num_ingredients, ds.num_calories_level)

        def cpu_step(hb):
            popt.zero_grad()
            sum(O.calculate_loss(P, {k: torch.from_numpy(np.asarray(v)) for k, v in hb.items()}, cfg, ei, sizes)).backward()
            popt.step()
        cpu_step(host[0])
        t0 = time.perf_counter()
        for hb in host[1:3]:
            cpu_step(hb)
        cpu_ms = (time.perf_counter() - t0) / 2 * 1e3
        with torch.no_grad():
            Pd = {k: v.detach() for k, v in P.items()}
            t0 = time.perf_counter()
            O.full_sort_scores(Pd, ds, 3, ei, sizes)
            cpu_fs = time.perf_counter() - t0
        out["cpu_baseline"] = {"kind": "port", "cores": torch.get_num_threads(), "train_ms_per_step": cpu_ms,
                               "full_sort_users_per_s": 1.0 / cpu_fs,
                               "sample": "2 train batches (dropout = identity); 1 user against all items"}
    return out


def _bench_eval(model, ds, dev, rank, world, barrier):
    """Full-sort evaluation of every C2 user (sharded by user over the ranks), k = 20, history mask, int32 indices;
    with world > 1 the timed region includes the final all-gather of the [U/P, 20] results."""
    from foodrec_b200 import evaluation as E
    model.eval()
    with torch.no_grad():
        user_all, item_all = model._tables()
        user_all, item_all = user_all.contiguous(), item_all.contiguous()
    hist = E.HistoryCSR(ds.train_coo_matrix, ds.n_users, dev)
    per = -(-ds.n_users // world)
    lo, hi = rank * per, min((rank + 1) * per, ds.n_users)
    users_host = torch.arange(lo, hi, dtype=torch.int64).pin_memory()
    users_dev = users_host.to(dev)
    stats = {}
    gathered = torch.empty((per * world, 20), dtype=torch.int32, device=dev) if world > 1 else None
    padded = torch.full((per, 20), -1, dtype=torch.int32, device=dev) if world > 1 else None

    def run(users):
        with torch.no_grad():
            item_bf16, bmax = E.to_bf16(item_all), E.max_row_norm(item_all)
            top = E.full_sort_topk(user_all, item_all, users, 20, hist=hist, B_bf16=item_bf16, b_max_norm=bmax,
                                   index_dtype=torch.int32, stats=stats)[1]
            if world > 1:
                import torch.distributed as dist
                padded[:top.shape[0]] = top
                dist.all_gather_into_tensor(gathered, padded)      # the only communication of the evaluation
            return top
    for _ in range(3):
        run(users_dev)
    barrier()
    ts = []
    for _ in range(5):
        a, b = ev_pair()
        a.record()
        run(users_dev)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        top = run(users_host.to(dev, non_blocking=True)).cpu()     # ids in from pinned host, top-K indices back out
    ms_e2e = (time.perf_counter() - t0) * 1e3 / 3
    prof = []
    E.PROFILE = prof
    run(users_dev)
    torch.cuda.synchronize()
    E.PROFILE = None
    out = {"ms_dev": sorted(ts)[len(ts) // 2], "ms_e2e": ms_e2e, "kernel_ms": prof[0][0].elapsed_time(prof[0][1]),
           "flops_local": prof[0][2], "n_users": ds.n_users, "h2d": users_host.numel() * 8,
           "d2h": top.numel() * top.element_size(), "stats": dict(stats)}
    if rank == 0 and world == 1:
        # Recall/NDCG of the fused path vs the fp32 oracle ranking on a 2048-user sample (4 d.p. equality)
        from foodrec_b200 import metrics as Mx
        sample = torch.arange(0, ds.n_users, max(1, ds.n_users // 2048))[:2048]
        S = (user_all[sample.to(dev)] @ item_all.t()).cpu()
        for r, u in enumerate(sample.tolist()):
            S[r, hist.idx_host[hist.ptr_host[u]:hist.ptr_host[u + 1]].astype(np.int64)] = -float("inf")
        ref = torch.topk(S, 20, dim=-1)[1].numpy()
        pos = [ds.testRatings[u] for u in sample.tolist()]
        got = top[sample - lo].numpy().astype(np.int64)
        a = Mx.topk_metrics(got, pos, metrics=("recall", "ndcg"), topk=(10, 20))
        b = Mx.topk_metrics(ref, pos, metrics=("recall", "ndcg"), topk=(10, 20))
        out["metrics"] = {"fused": a, "fp32_topk": b, "equal_4dp": a == b, "index_mismatches": int((got != ref).sum())}
    model.train()
    return out


def _spmm_traffic():
    for name in ("r2_spmm_step_traffic.json", "r1_spmm_step_traffic.json"):
        try:
            return float(json.load(open(os.path.join(ROOT, "profiles", name)))["dram_bytes_per_launch_mean"])
        except (OSError, KeyError, ValueError):
            continue
    return None


def _bench_eval_c4(dev, rank, world, barrier, tpeak):
    """BASELINE.json configs[3]: the full-sort sweep of 1 M users x 500 k items, d = 64, top-20, 20-item history mask
    per user, users sharded over the ranks (item table replicated), int32 results gathered once at the end
    (`dist.all_gather_into_tensor`, inside the timed region).  Replaces the per-user loop of `Trainer.evaluate`
    (FoodRec/common/trainer.py:476-503).  `roofline.frac` is PER GPU (this rank's FLOPs over this rank's kernel time)."""
    from foodrec_b200 import evaluation as E
    M_all, N, K, k = 1_000_000, 500_000, 64, 20
    per = -(-M_all // world)
    lo, hi = rank * per, min((rank + 1) * per, M_all)
    M = hi - lo
    g = torch.Generator(device=dev).manual_seed(4)
    I = torch.randn(N, K, device=dev, generator=g) * 0.1                    # replicated: same seed on every rank
    gu = torch.Generator(device=dev).manual_seed(1000 + rank)
    U = torch.randn(M, K, device=dev, generator=gu) * 0.1                   # this rank's users
    hist_idx = torch.sort(torch.randint(0, N, (M, 20), device=dev, generator=gu), dim=1)[0].to(torch.int32).reshape(-1)

    class _Hist:   # 20 training items per user (duplicates allowed: a sorted multiset masks the same columns)
        ptr = torch.arange(0, 20 * M + 1, 20, device=dev, dtype=torch.int64)
        idx = hist_idx
    Ib, bmax = E.to_bf16(I), E.max_row_norm(I)
    stats = {}
    gathered = torch.empty((per * world, k), dtype=torch.int32, device=dev) if world > 1 else None
    padded = torch.full((per, k), -1, dtype=torch.int32, device=dev) if world > 1 else None
    block = M                    # one launch per rank: the kernel is persistent over 256-row blocks and its workspace is per CTA

    def run():
        outs = []
        for s in range(0, M, block):
            e = min(M, s + block)
            rid = torch.arange(s, e, device=dev)
            outs.append(E.gemm_topk(U[s:e], I, k, row_ids=rid, hist=_Hist, B_bf16=Ib, b_max_norm=bmax,
                                    index_dtype=torch.int32, stats=stats))
        idx = torch.cat([o[1] for o in outs])
        if world > 1:
            import torch.distributed as dist
            padded[:M] = idx
            dist.all_gather_into_tensor(gathered, padded)
        return idx
    run()
    barrier()
    prof, ts = [], []
    E.PROFILE = prof
    for _ in range(2):
        a, b = ev_pair()
        a.record()
        idx = run()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    E.PROFILE = None
    barrier()
    n_l = len(prof) // 2
    kms = min(sum(x[0].elapsed_time(x[1]) for x in prof[:n_l]), sum(x[0].elapsed_time(x[1]) for x in prof[n_l:]))
    flops_local = sum(x[2] for x in prof[:n_l])
    t = torch.tensor([min(ts), kms], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, kms_max = float(t[0]), float(t[1])
    # exactness on 256 users of this rank's shard against the dense fp32 ranking
    sub = torch.arange(0, M, max(1, M // 256), device=dev)[:256]
    S = (U[sub].double() @ I.double().t()).float()
    hi2 = hist_idx.view(M, 20)[sub].long()
    S.scatter_(1, hi2, float("-inf"))
    ref = torch.topk(S, k, dim=-1)
    got = idx[sub].long()
    got_s = torch.gather(S, 1, got)
    tfl = flops_local / (kms * 1e-3) / 1e12
    return {"workload": f"{M_all} users x {N} items, d=64, top-20, 20-item history mask per user, users sharded over {world} "
                        f"GPU(s) ({M} per rank), int32 results all-gathered once (inside the timed region)",
            "users_per_s": M_all / (ms * 1e-3), "ms": ms, "kernel_ms_max_over_ranks": kms_max,
            "gather_bytes_per_rank": int(per * k * 4 * (world - 1)) if world > 1 else 0,
            "roofline": {"bound": "tensor", "achieved": tfl, "peak": tpeak[0], "unit": "TFLOP/s", "frac": tfl / tpeak[0],
                         "per": "GPU (rank 0's users over rank 0's kernel time)",
                         "note": "algorithmic FLOPs 2MNK counted once; the kernel runs a bounding sweep on every second column "
                                 "tile plus the collection sweep"},
            "exactness": dict(stats),
            "index_mismatches_vs_fp32_topk": int((got != ref[1]).sum()),
            "score_mismatches_beyond_fp32_noise": int(((got_s - ref[0]).abs() > 2e-6).sum())}


def _c5_shaped_graph(dev, n_users, n_items, n_inter, seed=5):
    """A C5-shaped user-item graph assembled ON THE DEVICE (SURVEY.md 8: 10 M users / 2 M items / 200 M interactions,
    scaled so one GPU holds the whole problem): log-normal user degrees, power-law item popularity, symmetrised and
    normalised with the reference's arithmetic (`graph.symmetric_normalised_device`)."""
    from foodrec_b200 import graph as G
    g = torch.Generator(device=dev).manual_seed(seed)
    deg = torch.exp(torch.randn(n_users, device=dev, generator=g))
    deg = torch.clamp((deg * (n_inter / n_users / deg.mean())).round(), min=1).long()
    users = torch.repeat_interleave(torch.arange(n_users, device=dev), deg)
    # popularity ~ rank^-0.7 through the inverse CDF of the continuous law, ranks scattered by a fixed permutation
    u01 = torch.rand(users.numel(), device=dev, generator=g)
    ranks = torch.clamp((u01.double().pow(1.0 / 0.3) * n_items).long(), max=n_items - 1)
    perm = torch.randperm(n_items, device=dev, generator=g)
    items = perm[ranks] + n_users
    return G.symmetric_normalised_device(users, items, n_users + n_items)


def _bench_partitioned_propagation(dev, rank, world, barrier, peaks, scale=0.2):
    """BASELINE.json configs[4], strong scaling: ONE propagation problem (3 layers, forward + backward, layer mean)
    on a C5-shaped graph -- the same graph at every N -- row-partitioned over the ranks.  Two exchange schemes:
    `all_gather` = one NCCL all-gather per layer (the north star's statement), `push` = the exchange fused into the
    SpMM epilogue (peer stores over NVLink, `fr_spmm_csr_f32_push`).  At N = 1 the same call is the single-GPU kernel in
    the HBM regime (table >> L2): its roofline is reported against the measured HBM peak."""
    from foodrec_b200 import dist as D, ops
    n_users, n_items, n_inter = int(10_000_000 * scale), int(2_000_000 * scale), int(200_000_000 * scale)
    layers, d = 3, 64
    g = _c5_shaped_graph(dev, n_users, n_items, n_inter)
    n = g.n_rows
    gen = torch.Generator(device=dev).manual_seed(11)
    ego = torch.randn(n, d, device=dev, generator=gen) * 0.1
    out = {"workload": f"C5-shaped graph built on the device: {n_users} users, {n_items} items, {g.nnz} stored entries "
                       f"(symmetrised), d=64 table {n * d * 4 / 1e6:.0f} MB, {layers} layers fwd + bwd, layer mean; "
                       f"same total problem at every N (strong scaling)",
           "world": world,
           "partition": "rows dealt round-robin to the ranks (rank p owns rows p, p + N, ...): equal stored entries per rank"}
    if world == 1:
        e1 = ego.clone().requires_grad_(True)

        def step1():
            e1.grad = None
            o = ops.propagate_mean(g, e1, layers)
            o.backward(o)                       # upstream gradient = the output itself (dense)
        ms = timed_ms(step1, 5, warm=2)
        X, Z, Y = ego, torch.randn_like(ego), torch.empty_like(ego)
        k_ms = timed_ms(lambda: ops.spmm(g, X, Z=Z, alpha=0.5, beta=0.5, out=Y), 10, warm=2)
        nb = g.spmm_bytes(d)
        ach = nb / (k_ms * 1e-3) / 1e9
        # parity at this size: 2 048 sampled rows (the 32 longest among them) of Y = 0.5 S X + 0.5 Z recomputed in fp64
        # from the CSR arrays with stock gathers, against the kernel's output (north star: 1e-5 relative)
        rp = torch.from_numpy(g.row_ptr_host.astype(np.int64)).to(dev)
        deg = rp[1:] - rp[:-1]
        rows_s = torch.unique(torch.cat([torch.topk(deg, 32)[1], torch.randint(0, n, (2016,), device=dev, generator=gen)]))
        worst = 0.0
        for r in rows_s.tolist():
            lo, hi = int(rp[r]), int(rp[r + 1])
            ref = 0.5 * (g.val[lo:hi].double()[:, None] * X[g.col[lo:hi].long()].double()).sum(0) + 0.5 * Z[r].double()
            worst = max(worst, float((Y[r].double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30)))
        out["parity_sampled_rows"] = {"rows": int(rows_s.numel()), "longest_row_entries": int(deg.max()),
                                      "max_rel_err_vs_fp64": worst, "tolerance": 1e-5, "ok": worst <= 1e-5}
        out.update(ms_fwd_bwd=ms, launches=2 * layers,
                   single_gpu_roofline={"bound": "hbm", "kernel": "spmm_group_kernel<64,8,4> (one layer, one direction)",
                                        "ms": k_ms, "algorithmic_bytes": nb, "achieved": ach, "peak": peaks[0], "unit": "GB/s",
                                        "frac": ach / peaks[0], "gathered_GBs": g.nnz * 264.0 / (k_ms * 1e-3) / 1e9,
                                        "traffic": _hbm_traffic() if abs(scale - 0.2) < 1e-9 else None})  # the ncu capture is of the default size
        return out
    import torch.distributed as dist
    pg = D.RowPartitionedGraph(g.row_ptr_host, g.col, g.val, n, rank, world, dev, balance="interleave")
    nnz_local = pg.local.nnz
    del g
    el = pg.local_rows(ego).requires_grad_(True)
    try:      # the exchange through this library's C ABI (fr_allgather_rows on its own NCCL communicator)
        comm, exchange_api = D.RowComm(device=dev), "fr_allgather_rows (C ABI, own NCCL communicator)"
    except Exception as e:  # noqa: BLE001  (NCCL could not be bound: the same collective through torch.distributed)
        comm, exchange_api = None, f"torch.distributed all_gather_into_tensor (fr_comm_init failed: {e})"

    def step_gather():
        el.grad = None
        o = D.propagate_mean_partitioned(pg, el, layers, group=comm)
        o.backward(o)
    for _ in range(2):
        step_gather()
    barrier()
    a, b = ev_pair()
    a.record()
    for _ in range(5):
        step_gather()
    b.record()
    barrier()
    t_gather = a.elapsed_time(b) / 5
    # local kernel time alone (no exchange): what the exchange is overlapped with / added to
    xf = torch.randn(pg.n_padded, d, device=dev)
    yl = torch.empty(pg.rows_per_rank, d, device=dev)
    k_ms = timed_ms(lambda: ops.spmm(pg.local, xf, Z=el.detach(), alpha=0.5, beta=0.5, out=yl), 10, warm=2)
    ag_ms = timed_ms(lambda: D._all_gather_rows(el.detach(), comm), 10, warm=2)
    t_push, push_err = None, None
    try:
        tables = D.PeerTables(pg.n_padded, d, dev)
        ep = pg.local_rows(ego).requires_grad_(True)

        def step_push():
            ep.grad = None
            o = D.propagate_mean_pushed(pg, ep, layers, tables)
            o.backward(o)
        for _ in range(2):
            step_push()
        barrier()
        a.record()
        for _ in range(5):
            step_push()
        b.record()
        barrier()
        t_push = a.elapsed_time(b) / 5
        same = torch.tensor([float(torch.equal(ep.grad, el.grad))], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        push_err = bool(same.item())
        tables.close()
    except Exception as e:  # noqa: BLE001  (peer mapping refused on this box: report the all-gather path alone)
        push_err = f"push path unavailable: {e}"
    t = torch.tensor([t_gather, k_ms, ag_ms, t_push if t_push is not None else 0.0], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if comm is not None:
        comm.close()
    recv = (world - 1) * pg.rows_per_rank * d * 4
    nb_local = 8 * nnz_local + 4 * (pg.rows_per_rank + 1) + 4 * d * pg.n_padded + 4 * d * pg.rows_per_rank
    out.update(
        all_gather={"ms_fwd_bwd_max_over_ranks": float(t[0]), "exchanges": 2 * layers, "api": exchange_api,
                    "one_all_gather_ms": float(t[2]), "bytes_received_per_rank_per_layer": recv,
                    "all_gather_GBs_per_rank": recv / (float(t[2]) * 1e-3) / 1e9,
                    "nvlink_frac_of_770GBs": recv / (float(t[2]) * 1e-3) / 1e9 / 770.0},
        push={"ms_fwd_bwd_max_over_ranks": float(t[3]) if t_push is not None else None,
              "bit_identical_to_all_gather_path": push_err,
              "bytes_stored_to_peers_per_rank_per_layer": recv},
        local_kernel={"ms_one_layer_max_over_ranks": float(t[1]), "stored_entries_this_rank": nnz_local,
                      "algorithmic_bytes_this_rank": nb_local, "achieved_GBs_per_gpu": nb_local / (float(t[1]) * 1e-3) / 1e9,
                      "frac_of_hbm_peak_per_gpu": nb_local / (float(t[1]) * 1e-3) / 1e9 / peaks[0]},
        limiter=("exchange" if float(t[2]) > float(t[1]) else "local kernel"),
        note="per layer every rank must receive the other ranks' rows of the table ((N-1)/N of it: the volume does not shrink "
             "with N) while its kernel time shrinks ~1/N; the exchange bounds the strong-scaling speed-up at "
             "t_kernel(1 GPU) / t_all_gather")
    return out


def _hbm_traffic():
    try:
        return float(json.load(open(os.path.join(ROOT, "profiles", "r2_spmm_hbm_regime.json")))["dram_bytes_per_launch"])
    except (OSError, KeyError, ValueError):
        return None


def _bench_dp_control(model, ds, cfg, dev, world, steps_per_epoch):
    """The replicated data-parallel step moves a global batch of 512 * N per step; ONE GPU can do that too.  This is
    the single-GPU step at B = 512 * N on the same graph (every rank measures it, rank 0 reports): the honest
    denominator for what N GPUs buy on a graph this small (VERDICT r1, weak 9)."""
    from foodrec_b200.models.pricai_modelx import PRICAI_ModelX
    from foodrec_b200.synth import sample_train_batches
    from foodrec_b200.train import GraphedTrainStep
    B = BATCH * world
    m2 = PRICAI_ModelX(cfg, ds).to(dev).train()
    opt2 = torch.optim.Adam(m2.parameters(), lr=cfg["learning_rate"], capturable=True, fused=True)
    hb = sample_train_batches(ds, B, 4, seed=99)
    bt = [{k: torch.from_numpy(b[k]).to(dev) for k in ("u_id", "pos_i_id", "neg_i_id")} for b in hb]
    step = GraphedTrainStep(m2, opt2, bt[0], keys=("u_id", "pos_i_id", "neg_i_id"))
    it = iter(range(10 ** 9))
    ms = timed_ms(lambda: step(bt[next(it) % 4]), 100, warm=5)
    return {"what": f"single-GPU CLUSSL step at B = {B} (= {world} x {BATCH}) on the same C2 graph, CUDA-graph replay",
            "ms_per_step": ms, "epochs_per_s_at_global_batch": (B / BATCH) / (steps_per_epoch * ms * 1e-3)}


def _bench_c3(dev, rank, world, barrier):
    """BASELINE.json configs[2]: CLUSSL with k-means item graphs + the contrastive term on the Foodcom-scale synthetic C3
    (7 600 users / 30 000 items / 192 000 interactions, 2 x 2 000 clusters), 1 and N GPUs.  Same step as the headline
    (CUDA-graph replay; N > 1: replicated graph, per-rank batches, gradient all-reduce inside the captured step)."""
    from foodrec_b200.models.pricai_modelx import PRICAI_ModelX
    from foodrec_b200.synth import make_dataset, sample_train_batches
    from foodrec_b200.train import FusedAdam, GraphedTrainStep, OverlappedGradAllReduce
    ds = make_dataset("C3")
    cfg = model_cfg(ds, str(dev))
    torch.manual_seed(999)
    m = PRICAI_ModelX(cfg, ds).to(dev).train()
    opt = FusedAdam(m.parameters(), lr=cfg["learning_rate"])
    keys = ("u_id", "pos_i_id", "neg_i_id")
    bt = [{k: torch.from_numpy(b[k]).to(dev) for k in keys} for b in sample_train_batches(ds, BATCH, 8, seed=31 + rank)]
    hook = OverlappedGradAllReduce(m) if world > 1 else None
    step = GraphedTrainStep(m, opt, bt[0], keys=keys, grad_hook=hook)
    for i in range(5):
        step(bt[i % 8])
    barrier()
    a, b = ev_pair()
    a.record()
    n = 300
    for i in range(n):
        step(bt[i % 8])
    b.record()
    barrier()
    t = torch.tensor([a.elapsed_time(b) / n], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    spe = math.ceil(ds.n_train / BATCH)
    if hook is not None:
        hook.remove()
    return {"workload": f"C3: CLUSSL train step, B={BATCH} per rank, {ds.n_users} users / {ds.n_items} items / {ds.n_train} train "
                        f"interactions, {ds.cfg.n_cluster} clusters x2, {ds.num_ingredients} ingredients; {world} GPU(s)",
            "ms_per_step_max_over_ranks": ms, "steps_per_epoch": spe, "timed_steps": n,
            "train_epochs_per_s": world / (spe * ms * 1e-3)}


def _bench_knn(ds, dev, tpeak):
    """The kNN / centroid shapes of the ranking kernel (FoodRec/utils/utils.py:118-183; dataset_process/*_kmeans.ipynb):
    cosine kNN of the C2 items over the 4096-d image and 384-d text features (k = 10), and the 6 nearest of 2000 centres."""
    from foodrec_b200 import evaluation as E
    out = {}
    for name, feat, k in (("image_knn_D4096", ds.embImage, 10), ("text_knn_D384", ds.embText, 10)):
        x = torch.from_numpy(feat).to(dev)
        xn = (x / torch.norm(x, p=2, dim=-1, keepdim=True)).contiguous()
        xb, bmax = E.to_bf16(xn), E.max_row_norm(xn)
        prof, st = [], {}
        E.PROFILE = prof
        ms = timed_ms(lambda: E.gemm_topk(xn, xn, k, A_bf16=xb, B_bf16=xb, b_max_norm=bmax, stats=st), 3, warm=1)
        E.PROFILE = None
        torch.cuda.synchronize()
        fl = 2.0 * x.shape[0] * x.shape[0] * x.shape[1]
        kms = min(p[0].elapsed_time(p[1]) for p in prof if p[2] >= 0.99 * fl)    # full launches only, not the re-runs of uncertified rows
        out[name] = {"workload": f"{x.shape[0]} x {x.shape[0]} cosine similarities, D = {x.shape[1]}, top-{k} (self kept)",
                     "ms_total": ms, "kernel_ms": kms, "exactness": dict(st),
                     "roofline": {"bound": "tensor", "achieved": fl / (kms * 1e-3) / 1e12, "peak": tpeak[0], "unit": "TFLOP/s",
                                  "frac": fl / (kms * 1e-3) / 1e12 / tpeak[0]}}
        del x, xn, xb
    x = torch.from_numpy(ds.embImage).to(dev)
    c = torch.from_numpy(ds.image_center).to(dev)
    ms = timed_ms(lambda: E.centroid_topk(x, c, 6), 3, warm=1)
    ref = ds.image_cluster_triples[:, 1].reshape(ds.n_items, 6)
    got = E.centroid_topk(x, c, 6).cpu().numpy()
    out["centroid_top6"] = {"workload": f"{x.shape[0]} items x {c.shape[0]} centres, D = {x.shape[1]}, 6 nearest (Euclidean)",
                            "ms_total": ms, "rows_identical_to_fp64_assignment": float((got == ref).all(axis=1).mean())}
    return out


def _bench_torch_cuda(ds, sd0, cfg, host_batches, dev, steps_per_epoch, ms_ours, ev, model):
    """SURVEY.md 2.1: 'the bar is the stock PyTorch ops on the same B200'.  The oracle's CLUSSL step with every tensor on
    the GPU (uncoalesced COO `torch.sparse.mm` at pricai_modelx.py:183,197,211,223, stack/mean, autograd, default
    Adam), and the reference's evaluation arithmetic (`matmul` + mask + `torch.topk`, trainer.py:495-497) batched over
    users -- timed with CUDA events on this box, beside this library's numbers."""
    from foodrec_b200 import evaluation as E
    out = {}
    o = OracleClussl(ds, sd0, cfg["learning_rate"], device=str(dev))
    bt = [{k: torch.from_numpy(b[k]).to(dev) for k in ("u_id", "pos_i_id", "neg_i_id")} for b in host_batches[:8]]
    it = iter(range(10 ** 9))
    ms = timed_ms(lambda: o.step(bt[next(it) % 8]), 20, warm=3)
    out["clussl_train_step"] = {"ms_per_step": ms, "epochs_per_s": 1.0 / (steps_per_epoch * ms * 1e-3),
                                "this_library_ms_per_step": ms_ours, "speedup": ms / ms_ours,
                                "what": "oracle CLUSSL step on cuda: COO torch.sparse.mm x7 fwd (+ autograd), stack/mean, "
                                        "index gathers, correlation_distance x3, torch.optim.Adam (default foreach)"}
    del o
    model.eval()
    with torch.no_grad():
        user_all, item_all = model._tables()
        user_all, item_all = user_all.contiguous(), item_all.contiguous()
        hist = E.HistoryCSR(ds.train_coo_matrix, ds.n_users, dev)

        def torch_eval():
            tops = []
            for s in range(0, ds.n_users, 8192):
                u = torch.arange(s, min(ds.n_users, s + 8192), device=dev)
                sc = user_all[u] @ item_all.t()
                hist.mask_scores_(sc, u)
                tops.append(torch.topk(sc, 20, dim=-1)[1])
            return torch.cat(tops)
        ms_e = timed_ms(torch_eval, 2, warm=1)
    model.train()
    out["full_sort_eval"] = {"ms": ms_e, "users_per_s": ds.n_users / (ms_e * 1e-3), "this_library_ms": ev["ms_dev"],
                             "speedup": ms_e / ev["ms_dev"],
                             "what": "fp32 matmul + history mask + torch.topk(20) in blocks of 8192 users"}
    return out


def _bench_healthrec(ds, dev, steps_per_epoch, peaks):
    """SURVEY.md 8f-1: HealthRec (`CIKM_Model`) on the same C2 data -- 2 + 1 propagation layers, BPR / KD / health terms,
    and dense Adam over ~200 M parameters, most of them the trainable raw-feature tables (cikm_model.py:83,87).  Two
    graph-replayed steps: this library's formulation (rows gathered before the feature projections, `fr_adam_step`)
    and the reference's (all-item projections at cikm_model.py:240-243, torch's fused Adam) on the same kernels otherwise."""
    from foodrec_b200.models.cikm_model import CIKM_Model
    from foodrec_b200.synth import sample_train_batches
    from foodrec_b200.train import FusedAdam, GraphedTrainStep
    cfg = Cfg(device=str(dev), embedding_size=64, train_batch_size=BATCH, is_multimodal_model=True, end2end=False,
              use_health_level_multi_hot=True, num_attention_heads=2, num_hidden_layers=2, attention_probs_dropout_prob=0.5,
              hidden_act="gelu", n_layers=2, ui_layers=1, reg_weight=0.5, loss_kd=0.05, loss_health=0.1, kd_threshold=0.4,
              learning_rate=0.001)          # configs/model/CIKM_Model.yaml
    bs = sample_train_batches(ds, BATCH, 4, seed=21)
    res = [{k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in b.items()} for b in bs]
    out = {}
    for name, all_items, own_adam in (("this_library", False, True), ("reference_formulation", True, False)):
        torch.manual_seed(999)
        m = CIKM_Model(cfg, ds).to(dev)
        m.train()
        m.project_all_items = all_items
        n_par = sum(p.numel() for p in m.parameters() if p.requires_grad)
        opt = (FusedAdam(m.parameters(), lr=cfg["learning_rate"]) if own_adam
               else torch.optim.Adam(m.parameters(), lr=cfg["learning_rate"], fused=True, capturable=True))
        step = GraphedTrainStep(m, opt, res[0])
        it = iter(range(10 ** 9))
        ms = timed_ms(lambda: step(res[next(it) % 4]), 30, warm=5)
        a_ms = timed_graph_ms(opt.step, 5)
        out[name] = {"ms_per_step": ms, "epochs_per_s": 1.0 / (steps_per_epoch * ms * 1e-3),
                     "adam": {"ms": a_ms, "parameters": n_par, "bytes": 28 * n_par,
                              "achieved_GBs": 28 * n_par / (a_ms * 1e-3) / 1e9, "frac_of_hbm_peak": 28 * n_par / (a_ms * 1e-3) / 1e9 / peaks[0],
                              "kernel": "adam_multi_kernel (fr_adam_step)" if own_adam else "torch.optim.Adam(fused=True)"},
                     "projection": "rows gathered first: [2B, Dv] x [Dv, 64]" if not all_items else "all items: [I, Dv] x [Dv, 64]"}
        del m, opt, step
        torch.cuda.empty_cache()
    out["workload"] = (f"HealthRec (CIKM_Model) train step on the C2 data, B={BATCH}: item-ingredient propagation x2 + user-item x1, "
                       f"transformer / attention / health head in torch, BPR + EmbLoss + KD fused, dense Adam")
    out["speedup_vs_reference_formulation"] = out["reference_formulation"]["ms_per_step"] / out["this_library"]["ms_per_step"]
    return out


def _tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["bf16_tflops"]), "MEASURED_PEAKS.json bf16_tflops burst (kernel timed alone; of measured)"
    return 1590.0, "B200_PROFILING.md fallback 1.59 PFLOP/s (of fallback)"


def _init_state_dict(ds):
    """Initial parameters exactly as the model constructor draws them (CPU, no library needed)."""
    import torch.nn as nn
    d, out = 64, {}
    for name, n in (("user_embedding", ds.n_users), ("item_embedding", ds.n_items),
                    ("ingre_embedding", ds.num_ingredients + 1), ("image_prototype_embedding", ds.cfg.n_cluster),
                    ("text_prototype_embedding", ds.cfg.n_cluster)):
        w = torch.empty(n, d)
        nn.init.xavier_uniform_(w)
        out[name + ".weight"] = w
    return out


def _allreduce_grads(model, world):
    import torch.distributed as dist
    grads = [p.grad for p in model.parameters() if p.grad is not None]
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat)
    flat.div_(world)
    o = 0
    for g in grads:
        g.copy_(flat[o:o + g.numel()].view_as(g))
        o += g.numel()


def _working_set_mb(model, opt):
    n = sum(p.numel() for p in model.parameters()) * 4 * 4  # param, grad, exp_avg, exp_avg_sq
    for g in (model.g_ui, model.g_image, model.g_text, model.g_ingre):
        n += g.nnz * 8 + g.n_seg * 16 + 3 * g.n_rows * 64 * 4
    return n / 1e6


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


if __name__ == "__main__":
    sys.exit(main())
