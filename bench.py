#!/usr/bin/env python
"""
bench.py -- molecular-graphs/sec of one GGNN training step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config C2|C4|C3|...]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

A "step" = one pass of the hot path over one batch of synthetic molecules: K0 (bond lists) -> forward ->
KL loss (Workflow.py:833-860) -> backward -> (N>1: one gradient all-reduce) -> Adam update.

Workload.  N = 1: BASELINE.json configs[1] ("C2"): GGNN hidden=message=128, 4 message passes, batch 1024 synthetic
13-atom molecules (gdb13 chemistry: F=8, Ef=3, APD=625), random-init weights.  N > 1: BASELINE.json configs[3] ("C4"):
GGNN defaults at ZINC scale (max_n_nodes=38), GLOBAL batch 4096 split contiguously over the ranks (2048 / 1024 / 512
molecules per rank) with ONE all-reduce of the flat gradient bucket per step -- strong scaling; `--scaling weak` gives
every rank its own full batch instead.  Before timing, the N>1 arm checks that the all-reduced gradient of a fixed
256-molecule batch equals the single-GPU gradient of the same batch (`dp_grad_rel_err`).

One JSON line on stdout (rank 0).  `value` = whole-job graphs/s with inputs resident in HBM, through
`graphinvent_b200.graphed.TrainStep` (the step as one CUDA-graph launch, capacity mode: no host synchronisation);
`e2e` = the same call driven from pinned HOST buffers (H2D of nodes/edges/targets + D2H of the loss inside the timed
region); `roofline` = dominant kernel class (the dense GEMMs) from CUDA-event pairs around every launch of the class in
an eager (un-captured) pass over the same step; `roofline_scatter` = the scatter-aggregate kernel (K2) alone at the C4
shape and inside a C4 step; `cpu_baseline` = the reference's CPU path on this host.  `--impl reference` times that CPU
path as its own arm (the unmodified reference modules when `baseline/_ref/graphinvent/gnn` is present, else the
oracle port).

`--dump-outputs DIR` writes what the last of the K timed steps computed (rank 0): `loss`, `logits` [B, APD],
`grads` (the flat gradient bucket) and `params` (the parameters after that step's Adam update, flattened in
`named_parameters()` order), as DIR/<name>.npy in float32.  Inputs and initial weights are seeded, so two builds
run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the tree may be read-only: no __pycache__ next to the sources

CONFIGS = {
    # name: (constants overrides, batch, atoms, atom types, charges, description)
    "C2": (dict(hidden_node_features=128, message_size=128, message_passes=4), 1024, 13, 5, 3,
           "GGNN hidden=128, 4 MP steps, batch=1024 synthetic 13-node graphs"),
    "C4": (dict(max_n_nodes=38, n_node_features=12, len_f_add_per_node=81), 4096, 38, 9, 3,
           "GGNN defaults ZINC-scale synthetic (max_n_nodes=38), batch=4096"),
    "C1": (dict(), 100, 13, 5, 3, "GGNN defaults gdb13 dims, batch=100 (reference plumbing size)"),
    "C3": (dict(model="AttGGNN", hidden_node_features=256, message_size=256, message_passes=6, max_n_nodes=40,
                n_node_features=12, len_f_add_per_node=81), 2048, 40, 9, 3,
           "AttentionGGNN hidden=256, 6 MP steps, batch=2048 synthetic 40-node graphs"),
    "C5T": (dict(model="EMN"), 1000, 13, 5, 3, "EMN defaults gdb13 dims, batch=1000 (training step of the C5 model)"),
}
UNIT = "graphs/s"
DUMP_LIMIT_BYTES = 64 << 20
CPU_MICRO_BATCH = 256     # the reference's O(V*E) prologue cannot run the large configurations whole (SURVEY.md 8d)
REF_DIR = os.path.join(ROOT, "baseline", "_ref", "graphinvent")


def config_model(cfg):
    return CONFIGS[cfg][0].get("model", "GGNN")


def metric_name(cfg):
    return f"molecular-graphs/sec (train fwd+bwd) {config_model(cfg)}"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), bf16_burst=float(d["bf16_tflops"]),
                    bf16_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


def make_constants_for(cfg):
    from graphinvent_b200.config import make_constants
    kw = {k: v for k, v in CONFIGS[cfg][0].items() if k != "model"}
    return make_constants(config_model(cfg), **kw)


def make_batch(cfg, seed, batch=None):
    """synthetic batch of the configuration (SURVEY.md 8d recipe), as int8 numpy arrays + float targets"""
    from graphinvent_b200 import synthetic as S
    _, B, n_atoms, n_types, n_charges, _ = CONFIGS[cfg]
    B = batch or B
    C = make_constants_for(cfg)
    nodes, edges = S.random_graphs(B, C.max_n_nodes, n_types, n_charges, seed=seed)
    apd = C.max_n_nodes * (C.len_f_add_per_node + C.len_f_conn_per_node) + 1
    target = S.random_targets(B, apd, seed=seed)
    return C, torch.from_numpy(nodes), torch.from_numpy(edges), torch.from_numpy(target), apd


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.rows = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def wait_first(self, timeout=3.0):
        """block until nvidia-smi delivered its first sample (it needs 0.1-1 s to start streaming)"""
        t_end = time.monotonic() + timeout
        while self.proc is not None and not self.rows and time.monotonic() < t_end:
            time.sleep(0.02)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), line.strip()))

    def stop(self, t0=None, t1=None):
        """t0, t1 (time.monotonic): the timed regions.  Samples inside [t0, t1] are used when there are any, else
        every sample taken under load since the start (and `window` says so)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows, window = [r for _, r in self.rows], "warm-up + timed regions"
        if t0 is not None and t1 is not None:
            inside = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15]
            if inside:
                rows, window = inside, "timed regions"
        sm, mx, pw, reasons = [], [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons),
                "window": window}


# ------------------------------------------------------------------------------------------
# CPU path of the reference: the unmodified reference modules when they travelled with the snapshot
# (baseline/_ref/graphinvent/gnn, placed there by __graft_entry__.build()), else the oracle port
# ------------------------------------------------------------------------------------------
def _reference_available():
    return os.path.isfile(os.path.join(REF_DIR, "gnn", "mpnn.py"))


class _CpuStep:
    """one CPU training step: forward + Workflow.loss + backward + Adam, on the reference modules or the port"""

    def __init__(self, cfg, seed=0):
        from oracle import mpnn_oracle as O
        self.O = O
        kw = {k: v for k, v in CONFIGS[cfg][0].items() if k != "model"}
        self.C = O.make_constants(config_model(cfg), **kw)
        sd = O.init_state_dict(self.C, seed=seed)
        self.kind = "reference" if _reference_available() else "port"
        if self.kind == "reference":
            if REF_DIR not in sys.path:
                sys.path.insert(0, REF_DIR)
            import gnn.mpnn as ref_mpnn                      # the reference's own modules, unmodified
            cls = {"GGNN": ref_mpnn.GGNN, "MNN": ref_mpnn.MNN, "AttGGNN": ref_mpnn.AttentionGGNN,
                   "EMN": ref_mpnn.EMN}[config_model(cfg)]
            self.net = cls(self.C)
            self.net.load_state_dict(sd)
            self.net.train()
            self.opt = torch.optim.Adam(self.net.parameters(), lr=1e-4)       # Workflow.py:191
        else:
            params = [v.clone().requires_grad_(True) for v in sd.values()]
            self.leaves = dict(zip(sd.keys(), params))
            self.opt = torch.optim.Adam(params, lr=1e-4)

    def __call__(self, nodes, edges, target):
        if self.kind == "reference":
            out = self.net(nodes, edges)                     # SummationMPNN.forward (summation_mpnn.py:80-149)
        else:
            out = self.O.forward(self.leaves, self.C, nodes, edges)
        loss = self.O.kl_loss(out, target)                   # Workflow.loss (Workflow.py:833-860), 3 lines
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        self.opt.step()
        return loss


def _pick_cpu_threads(cfg, nodes, edges, target):
    """The reference sets no thread count (PyTorch default = all cores); on a many-core host that default
    oversubscribes its small ATen ops badly, so give the CPU arm its best: time one step of a 128-molecule
    slice at a few thread counts and keep the fastest."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (ncpu, ncpu // 2, 64, 32, 16, 8) if 1 <= c <= ncpu}, reverse=True)
    n, e, t = nodes[:128], edges[:128], target[:128]
    best = (float("inf"), ncpu)
    for c in cands:
        torch.set_num_threads(c)
        step = _CpuStep(cfg)
        step(n, e, t)                                        # warm-up at this thread count
        t0 = time.perf_counter()
        step(n, e, t)
        dt = time.perf_counter() - t0
        if dt < best[0]:
            best = (dt, c)
    return best[1]


def cpu_train_steps(cfg, steps, warmup, budget_s=None, seed=1002):
    _, nodes, edges, target, _ = make_batch(cfg, seed)
    nodes, edges = nodes.float(), edges.float()              # BlockDatasetLoader.py:139-143
    if cfg not in ("C1", "C2"):      # micro-batch: the dense [V, E] prologue of the reference is quadratic in the batch
        nodes, edges, target = nodes[:CPU_MICRO_BATCH], edges[:CPU_MICRO_BATCH], target[:CPU_MICRO_BATCH]
    torch.set_num_threads(_pick_cpu_threads(cfg, nodes, edges, target))
    step = _CpuStep(cfg)
    B = nodes.shape[0]
    times = []
    t_begin = time.perf_counter()
    loss = None
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        loss = step(nodes, edges, target)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        if budget_s is not None and it >= warmup and time.perf_counter() - t_begin > budget_s:
            break
    return B, times, float(loss.detach()), step.kind


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None         # under torchrun only rank 0 measures the CPU path
    B, times, loss, kind = cpu_train_steps(args.config, args.steps, args.warmup)
    total = sum(times)
    value = B * len(times) / total
    cores = torch.get_num_threads()
    impl = ("unmodified reference modules (baseline/_ref/graphinvent/gnn: SummationMPNN.forward etc.) + Workflow.loss "
            "restated + torch.optim.Adam, CPU" if kind == "reference" else
            "oracle port of the reference CPU path (oracle/mpnn_oracle.py; baseline/_ref is not on this box)")
    line = {"impl": "reference", "metric": metric_name(args.config), "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": CONFIGS[args.config][5], "name": args.config, "step": "fwd+kl_loss+bwd+adam",
                       "impl": impl, "torch": torch.__version__,
                       "batch": B, "note": None if B == CONFIGS[args.config][1] else
                       f"micro-batch of {B}: the reference's dense [V,E] summation matrix does not fit the full batch"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": f"{len(times)} full steps of batch {B}", "os_cpu_count": os.cpu_count()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "final_loss": loss}
    return line


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def _time_scatter(S, E, ld, ent, iters=40):
    from graphinvent_b200._lib import check, lib
    g = torch.Generator(device="cpu").manual_seed(0)
    dst = torch.randint(0, S, (E,), generator=g).sort().values
    ptr = torch.zeros(S + 1, dtype=torch.int32)
    ptr[1:] = torch.bincount(dst, minlength=S).cumsum(0).int()
    msg = torch.randn(E, ld, device="cuda")
    out = torch.empty(S, ld, device="cuda")
    ptr, ent = ptr.cuda(), ent.cuda()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda t: ctypes.c_void_p(t.data_ptr() if t is not None else 0)
    for _ in range(5):
        check(lib.gib_scatter_sum(P(out), P(msg), ld, P(ptr), P(ent), None, S, st), "scatter")
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        check(lib.gib_scatter_sum(P(out), P(msg), ld, P(ptr), P(ent), None, S, st), "scatter")
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def scatter_roofline(pk):
    """K2 alone at the C4 single-GPU shape (V=155648 slots, E=352256 entries, msg=100 -> padded row 112 floats):
    working set 204 MB > 126 MB L2, so consecutive launches cannot hit in L2.  Bytes = SURVEY.md 8(d):
    E*msg*4 + V*msg*4 + (V+1)*4 (messages read once, aggregates written once, CSR row pointers)."""
    S, E, width = 155648, 352256, 100
    ld = (width + 15) // 16 * 16
    nbytes = E * width * 4 + S * width * 4 + (S + 1) * 4
    g = torch.Generator(device="cpu").manual_seed(1)
    ms_sorted = _time_scatter(S, E, ld, torch.arange(E, dtype=torch.int32))              # messages stored dst-sorted
    # the model's layout: rows grouped by bond type (84 / 14 / 2 %), so the entry index is a real indirection
    t = torch.multinomial(torch.tensor([0.84, 0.14, 0.02]), E, replacement=True, generator=g)
    order = torch.argsort(t, stable=True)
    ent_grouped = torch.empty(E, dtype=torch.int32)
    ent_grouped[order] = torch.arange(E, dtype=torch.int32)
    ms_grouped = _time_scatter(S, E, ld, ent_grouped)
    gbs = nbytes / ms_grouped / 1e6
    return {"kernel": "scatter_sum_kernel (K2)", "bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s",
            "frac": gbs / pk["hbm"], "traffic": 194499328,
            "traffic_source": "profiles/r02_ncu_tc3_stage5.md, r2k_scatter (ncu --set full: dram__bytes_read.sum 159.86 MB + dram__bytes_write.sum 34.64 MB, one launch of the streaming-hint variant; round 1, default caching: 208.56 MB)",
            "peak_source": pk["source"] + " (copy, burst)",
            "shape": {"slots": S, "entries": E, "width": width, "ld": ld},
            "layout": "bond-type-grouped message rows (the model's layout: entry index is an indirection)",
            "ms_per_launch": ms_grouped, "bytes_per_launch": nbytes, "bytes_definition": "SURVEY.md 8(d): E*msg*4 + V*msg*4 + (V+1)*4",
            "dst_sorted_layout": {"ms_per_launch": ms_sorted, "achieved": nbytes / ms_sorted / 1e6,
                                  "frac": nbytes / ms_sorted / 1e6 / pk["hbm"]},
            "l2": "working set 204 MB > 126 MB L2, no flush needed"}


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """arrays (name -> device tensor) as out_dir/<name>.npy in float32; if they hold more than `limit` bytes together,
    every array larger than its even share of the limit is replaced by a fixed seeded sample of its flattened elements
    (sorted indices, the same on every run)"""
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    share = limit // len(host)
    for i, (name, a) in enumerate(host.items()):
        if total > limit and a.nbytes > share:
            rng = np.random.default_rng(i)
            a = a.reshape(-1)[np.sort(rng.choice(a.size, share // 4, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def _flat_grads(net):
    return torch.cat([p.grad.detach().reshape(-1) for p in net.parameters()])


def dp_gradient_check(net, cfg, world, rank, dev):
    """all-reduced gradient of a fixed 256-molecule batch over the ranks == gradient of the whole batch on one GPU
    (SURVEY.md 8e).  Runs through the public module API; returns the relative L2 error on rank 0."""
    import torch.distributed as dist
    from graphinvent_b200 import functional as Fn
    from graphinvent_b200 import parallel
    G = 256
    _, nodes, edges, target, _ = make_batch(cfg, 4242, batch=G)
    nodes, edges, target = nodes.to(dev), edges.to(dev), target.to(dev)
    lo, hi = parallel.shard_bounds(G, rank, world)
    net.zero_grad(set_to_none=True)
    if hi > lo:
        out = net(nodes[lo:hi], edges[lo:hi])
        loss = Fn.kl_loss(out, target[lo:hi]) * ((hi - lo) / G)      # local batch mean -> share of the global mean
        loss.backward()
        flat = _flat_grads(net)
    else:
        flat = torch.zeros(sum(p.numel() for p in net.parameters()), device=dev)
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    err = None
    if rank == 0:
        net.zero_grad(set_to_none=True)
        loss = Fn.kl_loss(net(nodes, edges), target)
        loss.backward()
        full = _flat_grads(net)
        err = float((flat - full).norm() / full.norm())
    net.zero_grad(set_to_none=True)
    return err


def run_b200_arm(args):
    import torch.distributed as dist
    from graphinvent_b200 import functional as Fn
    from graphinvent_b200 import parallel
    from graphinvent_b200._lib import check, lib
    from graphinvent_b200.gnn import mpnn
    from graphinvent_b200.graphed import TrainStep
    from graphinvent_b200.optim import FlatAdam

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    cfg = args.config
    strong = args.scaling == "strong" and world > 1
    global_batch = CONFIGS[cfg][1] if (strong or world == 1) else CONFIGS[cfg][1] * world
    lo, hi = parallel.shard_bounds(global_batch, rank, world)
    B = hi - lo

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    C, nodes_h, edges_h, target_h, apd = make_batch(cfg, 1002 + rank, batch=B)     # int8 batch, as stored on disk
    torch.manual_seed(0)                      # identical random-init replicas on every rank
    net = mpnn.create(C).to(dev)
    dp_err = dp_gradient_check(net, cfg, world, rank, dev) if world > 1 else None
    dp_err_fp32 = None
    if world > 1:
        # the same check with the fp32 SIMT GEMMs: isolates the data-parallel plumbing (sharding, loss scaling,
        # all-reduce) from the tensor cores' 3xTF32 rounding, which differs between a shard and the whole batch
        from graphinvent_b200._lib import lib as _l
        _l.gib_set_tensor_cores(0)
        dp_err_fp32 = dp_gradient_check(net, cfg, world, rank, dev)
        _l.gib_set_tensor_cores(1)
    opt = FlatAdam(net.parameters(), lr=1e-4)
    entries = int((edges_h != 0).sum())
    cap = int(entries * 1.05) + 256           # static bond-entry capacity of the captured step
    in_dt = torch.int8 if args.input == "int8" else torch.float32
    nodes_in, edges_in = nodes_h.to(in_dt), edges_h.to(in_dt)
    step = TrainStep(net, opt, batch_size=B, entry_capacity=cap, input_dtype=in_dt, global_batch=global_batch)
    pin = [t.pin_memory() for t in (nodes_in, edges_in, target_h)]
    h2d = sum(t.numel() * t.element_size() for t in pin)
    step.load(*pin)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()               # before the warm-up: nvidia-smi takes a while to start streaming
        sampler.wait_first()
    W = max(args.warmup, 3)
    for _ in range(W):
        loss = step()
    barrier()

    # ---- timed region 1: exactly K steps, inputs resident in HBM -------------------------------------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_region0 = time.monotonic()
    ev0.record()
    for _ in range(args.steps):
        loss = step()
    ev1.record()
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    final_loss = float(loss)
    step.check()                              # capacity respected (one 64-byte read, outside the timed region)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": step.loss, "logits": step.out, "grads": step.gflat,
                                         "params": torch.cat([p.detach().reshape(-1) for p in step.params])})

    # ---- timed region 1b, only with --min-seconds: the same step for that long (a 20-step region is shorter than
    #      nvidia-smi's sampling period and than the power-cap time constant the sustained tensor peak is quoted under)
    long_run = None
    if args.min_seconds > 0:
        long_steps = max(args.steps, int(math.ceil(args.min_seconds * 1e3 / (ms_total / args.steps))))
        lv0, lv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        lv0.record()
        for _ in range(long_steps):
            loss = step()
        lv1.record()
        barrier()
        ms_long = max_over_ranks(lv0.elapsed_time(lv1))
        long_run = {"steps": long_steps, "ms_per_step": ms_long / long_steps,
                    "value": global_batch * long_steps / (ms_long / 1e3), "seconds": ms_long / 1e3}
    t_region1 = time.monotonic()
    clocks = sampler.stop(t_region0, t_region1) if rank == 0 else None

    # ---- timed region 2: end to end from pinned host buffers ---------------------------------------------
    # Every step: H2D of that step's inputs from pinned host memory into the step's static input buffers and D2H of
    # the step's loss into pinned memory; the host reads the value one step later so that it never stalls the launch
    # queue.  All copies and the final synchronisation are inside the timed region.
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    loss_events = [torch.cuda.Event(), torch.cuda.Event()]
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    host_losses = []
    for i in range(args.steps):
        loss_i = step(*pin)
        loss_host[i & 1].copy_(loss_i, non_blocking=True)               # D2H of this step's result
        loss_events[i & 1].record()
        if i > 0:                                                        # previous step's loss, read on the host
            loss_events[(i - 1) & 1].synchronize()
            host_losses.append(float(loss_host[(i - 1) & 1]))
    loss_events[(args.steps - 1) & 1].synchronize()
    host_losses.append(float(loss_host[(args.steps - 1) & 1]))
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    assert len(host_losses) == args.steps and all(np.isfinite(host_losses))

    # ---- kernel classes: an eager, exact-size pass over the same step through the module API with a CUDA-event pair
    #      around every GEMM / scatter launch (the captured step keeps the bond-type group sizes on the device, so
    #      its per-launch FLOP counts are not known on the host; the kernels and their order are the same) ----------
    launches0 = lib.gib_launch_count()
    step._enqueue_all()
    launches_per_step = int(lib.gib_launch_count() - launches0) + 1      # + the Adam launch
    torch.cuda.synchronize()
    dn, de, dt_ = nodes_in.to(dev), edges_in.to(dev), target_h.to(dev)
    net.entry_capacity = None

    def eager_fwd_bwd():
        net.zero_grad(set_to_none=True)
        Fn.kl_loss(net(dn, de), dt_).backward()
    prof_steps = max(3, min(args.steps, 20))
    for _ in range(2):
        eager_fwd_bwd()
    lib.gib_profile_enable(1)
    barrier()
    pv0, pv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pv0.record()
    for _ in range(prof_steps):
        eager_fwd_bwd()
    pv1.record()
    barrier()
    ms_instr = max_over_ranks(pv0.elapsed_time(pv1))
    if args.launch_table and rank == 0:
        cap_ = 1 << 16
        rms = (ctypes.c_double * cap_)(); rwork = (ctypes.c_double * cap_)(); rcls = (ctypes.c_int * cap_)()
        nrec = lib.gib_profile_records(rms, rwork, rcls, cap_)
        per = nrec // prof_steps if nrec > 0 and nrec % prof_steps == 0 and nrec <= cap_ else 0
        with open(args.launch_table, "w") as fh:
            fh.write(f"# {cfg}: timed launches of one eager forward + loss + backward (mean of {prof_steps} steps), "
                     "launch order; class 0 = tcgen05 forward/dX GEMM launch (a chain = several layers), 1 = tcgen05 dW "
                     "partials, 2 = K2, 3 / 4 = forward/dX and dW GEMMs on the fp32 SIMT kernels\n")
            fh.write("idx class  GFLOP_or_MB      us     TFLOP/s_or_GB/s\n")
            for i in range(per):
                t = sum(rms[i + k * per] for k in range(prof_steps)) / prof_steps
                wk = rwork[i]
                rate = wk / (t * 1e-3) / (1e12 if rcls[i] != 2 else 1e9) if t > 0 else 0.0
                fh.write(f"{i:3d} {rcls[i]:5d} {wk / (1e9 if rcls[i] != 2 else 1e6):12.3f} {t * 1e3:8.1f} {rate:10.1f}\n")
    pms = (ctypes.c_double * 5)(); pwork = (ctypes.c_double * 5)(); pcnt = (ctypes.c_longlong * 5)()
    check(lib.gib_profile_collect(pms, pwork, pcnt), "profile_collect")
    lib.gib_profile_enable(0)
    for p_, v_ in zip(step.params, step.views):          # the eager passes replaced .grad: hand the bucket views back
        p_.grad = v_

    # ---- the same step through the module API, eagerly (what Workflow.train_epoch would call; for comparison) ----
    module_api = None
    if world == 1 and not args.no_module_api:

        def eager():
            out = net(dn, de)
            l = Fn.kl_loss(out, dt_)
            opt.zero_grad(set_to_none=True)
            l.backward()
            opt.step()
            return l
        for _ in range(3):
            eager()
        torch.cuda.synchronize()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for _ in range(args.steps):
            eager()
        m1.record()
        torch.cuda.synchronize()
        module_api = {"value": B * args.steps / (m0.elapsed_time(m1) / 1e3), "unit": UNIT,
                      "ms_per_step": m0.elapsed_time(m1) / args.steps,
                      "how": "model(nodes, edges) -> kl_loss -> backward -> FlatAdam.step, eager launches, exact-size "
                             "mode (one 64-byte header read per forward)"}

    # ---- N > 1, strong scaling: the same global batch on ONE GPU (rank 0), for the scaling efficiency -----------
    single = None
    if strong and not args.no_single:
        del step
        torch.cuda.empty_cache()
        if rank == 0:
            Cg, ng, eg, tg, _ = make_batch(cfg, 1002, batch=global_batch)
            torch.manual_seed(0)
            net1 = mpnn.create(Cg).to(dev)
            opt1 = FlatAdam(net1.parameters(), lr=1e-4)
            st1 = TrainStep(net1, opt1, batch_size=global_batch, entry_capacity=int(int((eg != 0).sum()) * 1.05) + 256,
                            input_dtype=in_dt, global_batch=global_batch, group=False)
            st1.load(ng.to(in_dt), eg.to(in_dt), tg)
            for _ in range(3):
                st1()
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n1 = max(5, min(args.steps, 20))
            s0.record()
            for _ in range(n1):
                st1()
            s1.record()
            torch.cuda.synchronize()
            ms1 = s0.elapsed_time(s1) / n1
            single = {"n_gpus": 1, "global_batch": global_batch, "ms_per_step": ms1,
                      "value": global_batch / (ms1 / 1e3), "unit": UNIT, "steps": n1,
                      "how": "the same global batch and step on rank 0 alone, measured in this run after the N-GPU "
                             "regions (the other ranks idle)"}
            del st1, net1, opt1
        barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None

    pk = peaks()
    value = global_batch * args.steps / (ms_total / 1e3)
    e2e_value = global_batch * args.steps / (ms_e2e / 1e3)
    # dominant kernel class = forward/dX GEMMs (class 0) or dW GEMMs (class 1): report the larger one
    cls = 0 if pms[0] >= pms[1] else 1
    gemm_tflops = pwork[cls] / pms[cls] / 1e9 if pms[cls] > 0 else 0.0
    tensor_peak = pk["bf16_sustained"] / 2.0 / 3.0     # TF32 dense = bf16/2; fp32-accurate 3xTF32 = /3
    tf = lambda c: (pwork[c] / pms[c] / 1e9) if pms[c] else 0.0
    roofline = {"kernel": ["tc3_gemm_kernel<NT> (tcgen05 3xTF32, activation operand through tensor memory; forward + dX GEMMs)",
                           "tc3_gemm_kernel<TN> (weight-gradient GEMMs + fused bias partials)"][cls],
                "bound": "tensor", "achieved": gemm_tflops, "peak": tensor_peak, "unit": "TFLOP/s",
                "frac": gemm_tflops / tensor_peak, "traffic": None,
                "peak_source": pk["source"] + " bf16 sustained / 2 (TF32 rate) / 3 (fp32-accurate 3xTF32 issue)",
                "launches_timed": int(pcnt[cls]), "ms_in_class": pms[cls], "steps_timed": prof_steps,
                "how": "eager exact-size pass (module API forward + loss + backward) over the same kernels, CUDA-event pair per "
                       "launch; `achieved` = algorithmic FLOPs of the launches of THIS kernel / their summed durations "
                       "(the fp32 SIMT GEMM launches are listed separately under `classes`)",
                "share_of_step": pms[cls] / ms_instr, "ms_per_step_instrumented": ms_instr / prof_steps,
                "classes": {"gemm_nt": {"ms_per_step": pms[0] / prof_steps, "tflops": tf(0), "frac": tf(0) / tensor_peak,
                                        "launches_per_step": pcnt[0] / prof_steps},
                            "gemm_dw": {"ms_per_step": pms[1] / prof_steps, "tflops": tf(1), "frac": tf(1) / tensor_peak,
                                        "launches_per_step": pcnt[1] / prof_steps,
                                        "note": "main-stream part (partials); the reductions overlap on the side stream"},
                            "scatter": {"ms_per_step": pms[2] / prof_steps, "launches_per_step": pcnt[2] / prof_steps,
                                        "gbs_8d_bytes": (pwork[2] / pms[2] / 1e6) if pms[2] else None},
                            "gemm_nt_fp32_simt": {"ms_per_step": pms[3] / prof_steps, "tflops": tf(3),
                                                  "launches_per_step": pcnt[3] / prof_steps,
                                                  "note": "narrow / tiny forward + dX problems on sgemm_nt_kernel (APD "
                                                          "output layers, K < 32): a different kernel, not in `achieved`"},
                            "gemm_dw_fp32_simt": {"ms_per_step": pms[4] / prof_steps, "tflops": tf(4),
                                                  "launches_per_step": pcnt[4] / prof_steps},
                            "all_forward_dx_gemm_launches": {
                                "ms_per_step": (pms[0] + pms[3]) / prof_steps,
                                "tflops": ((pwork[0] + pwork[3]) / (pms[0] + pms[3]) / 1e9) if pms[0] + pms[3] else 0.0,
                                "frac": ((pwork[0] + pwork[3]) / (pms[0] + pms[3]) / 1e9 / tensor_peak) if pms[0] + pms[3] else 0.0,
                                "note": "tcgen05 and fp32 SIMT launches together (the round-1 / earlier round-2 definition "
                                        "of the class)"}}}
    line = {"metric": metric_name(cfg), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": CONFIGS[cfg][5], "name": cfg, "per_gpu_batch": B, "global_batch": global_batch,
                       "step": "k0+fwd+kl_loss+bwd" + ("+allreduce" if world > 1 else "") + "+adam",
                       "api": "graphinvent_b200.graphed.TrainStep (one CUDA-graph launch per step, capacity mode)",
                       "input_dtype": args.input, "entry_capacity": cap, "bond_entries_per_rank_batch": entries,
                       "optimizer": "graphinvent_b200.optim.FlatAdam (1 launch)",
                       "parallelism": f"dp{world}", "weights": "random init (reference initialisers: xavier-uniform MLPs, PyTorch-default GRU), torch.manual_seed(0)",
                       "l2": "per-step working set (saved activations + packed weights, "
                             f"{step.workspace_bytes / 1e6:.0f} MB) exceeds the 126 MB L2; no explicit flush"
                             if "step" in dir() else "working set exceeds L2"},
            "long_run": long_run,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps,
                    "how": "TrainStep(nodes, edges, target) with pinned host tensors: H2D into the static input buffers -> "
                           "graph launch -> Adam -> loss D2H to pinned memory, read on the host one step later"},
            "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
            "clocks": clocks, "roofline": roofline, "final_loss": final_loss}
    if dp_err is not None:
        line["dp_grad_rel_err"] = dp_err
        line["dp_grad_rel_err_fp32_gemms"] = dp_err_fp32
        line["dp_grad_check"] = ("||allreduce_r(grad of shard r of a fixed 256-molecule batch) - grad of the whole batch on "
                                 "rank 0||_2 / ||.||_2, module API, before the timed regions")
    if single is not None:
        line["single_gpu_same_workload"] = single
    if module_api is not None:
        line["module_api"] = module_api
    if world == 1:
        try:
            line["roofline_scatter"] = scatter_roofline(pk)
        except Exception as ex:  # keep the headline line even if the side measurement fails
            line["roofline_scatter"] = {"error": repr(ex)}
        if not args.no_k2_in_model:
            try:
                line["roofline_scatter"]["in_model_c4"] = k2_in_model(pk, dev)
            except Exception as ex:
                line["roofline_scatter"]["in_model_c4"] = {"error": repr(ex)}
    if world == 1 and not args.no_cpu_baseline:
        Bc, times, _, kind = cpu_train_steps(cfg, steps=8, warmup=1, budget_s=20.0)
        v = Bc * len(times) / sum(times)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                                "sample": f"{len(times)} full steps of batch {Bc} after 1 warm-up "
                                          f"({'unmodified reference modules' if kind == 'reference' else 'oracle port'}, "
                                          "fwd+kl_loss+bwd+adam)", "os_cpu_count": os.cpu_count()}
    if world > 1:
        dist.destroy_process_group()
    return line


def k2_in_model(pk, dev):
    """K2 timed where it runs: inside a C4 training step (B=4096, N=38: V=155648 slots), real bond-type-grouped
    layout, CUDA-event pairs around its launches; bytes per launch = SURVEY.md 8(d)."""
    from graphinvent_b200 import functional as Fn
    from graphinvent_b200._lib import check, lib
    from graphinvent_b200.gnn import mpnn
    C, nodes, edges, target, _ = make_batch("C4", 1004)
    torch.manual_seed(0)
    net = mpnn.create(C).to(dev)
    nodes, edges, target = nodes.to(dev), edges.to(dev), target.to(dev)

    def one():
        net.zero_grad(set_to_none=True)
        loss = Fn.kl_loss(net(nodes, edges), target)
        loss.backward()
    one()
    torch.cuda.synchronize()
    lib.gib_profile_enable(1)
    for _ in range(2):
        one()
    torch.cuda.synchronize()
    pms = (ctypes.c_double * 5)(); pwork = (ctypes.c_double * 5)(); pcnt = (ctypes.c_longlong * 5)()
    check(lib.gib_profile_collect(pms, pwork, pcnt), "profile_collect")
    lib.gib_profile_enable(0)
    gbs = pwork[2] / pms[2] / 1e6 if pms[2] else 0.0
    tensor_peak = pk["bf16_sustained"] / 6.0
    return {"launches": int(pcnt[2]), "ms_per_launch": pms[2] / max(1, pcnt[2]), "achieved": gbs, "unit": "GB/s",
            "frac": gbs / pk["hbm"], "entries": net.last_stats.get("entries"),
            "what": "forward K2 (width 100) and backward gather-reduce (width 100, accumulate) of 3 message passes",
            "c4_step_gemm_nt_tflops": pwork[0] / pms[0] / 1e9 if pms[0] else None,
            "c4_step_gemm_nt_frac": (pwork[0] / pms[0] / 1e9 / tensor_peak) if pms[0] else None,
            "c4_step_gemm_dw_tflops": pwork[1] / pms[1] / 1e9 if pms[1] else None}


class _StdoutToStderr:
    """NCCL (and anything else native) may print to fd 1 (e.g. "NCCL version ..."): the contract is ONE JSON line on
    stdout, so fd 1 is pointed at stderr while the benchmark runs and restored just before the line is printed."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS),
                    help="default: C2 at --gpus 1 (BASELINE configs[1]), C4 at --gpus > 1 (configs[3])")
    ap.add_argument("--scaling", default=None, choices=["strong", "weak"],
                    help="N > 1: strong (default) = the configuration's global batch split over the ranks; "
                         "weak = every rank its own full batch")
    ap.add_argument("--input", default="int8", choices=["int8", "float32"],
                    help="element type of the nodes / edges batches (int8 = the reference's on-disk type)")
    ap.add_argument("--min-seconds", type=float, default=0.0,
                    help="if > 0, an additional timed region of at least this many seconds (`long_run`)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-module-api", action="store_true")
    ap.add_argument("--no-single", action="store_true", help="N > 1: skip the single-GPU run of the same workload")
    ap.add_argument("--no-k2-in-model", action="store_true")
    ap.add_argument("--launch-table", default=None, help="write the per-launch timing table of the eager pass here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    if args.config is None:
        args.config = "C2" if max(world, args.gpus) == 1 else "C4"
    if args.scaling is None:
        args.scaling = "strong" if max(world, args.gpus) > 1 else "weak"
    if args.impl == "reference":
        args.steps = args.steps if args.steps is not None else 5
        args.warmup = args.warmup if args.warmup is not None else 1
        with _StdoutToStderr():
            line = run_reference_arm(args)
    else:
        args.steps = args.steps if args.steps is not None else 200
        args.warmup = args.warmup if args.warmup is not None else 5
        with _StdoutToStderr():
            line = run_b200_arm(args)
    if line is not None:
        print(json.dumps(line), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
