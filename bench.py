#!/usr/bin/env python
"""bench.py -- graph-snapshots/s for DCRNN on a METR-LA-shaped StaticGraphTemporalSignal
(BASELINE.json `metric`; workload = configs[1]: DCRNN K=2, 207 nodes, 1722 edges, 2 features,
12-step windows, hidden 32).

A "step" = one pass of the hot path over one batch of `--windows` windows per GPU (one launch of the
fused sm_100a kernel).  One graph-snapshot = one (207 x 2 x 12) window pushed through 12 chained DCRNN
cell steps, all 12 hidden states emitted (SURVEY.md section 8d).

  python bench.py [--gpus N --steps K --warmup W]      our arm (N>1 under torchrun, one rank per GPU)
  python bench.py --impl reference ...                 the reference's CPU path (oracle port) on the host cores
  python bench.py ... --dump-outputs DIR               also write what the last timed step returned (see `dump_outputs`)

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
_T0 = time.time()                                                   # process start: the secondary legs share one wall-clock budget
BUDGET_S = float(os.environ.get("STMP_BENCH_BUDGET_S", "210"))     # after this many seconds the line is printed with what is done
sys.path.insert(0, ROOT)

N_NODES, N_EDGES, F_IN, HORIZON, HIDDEN, K_HOPS = 207, 1722, 2, 12, 32, 2
# algorithmic (compulsory) HBM bytes per graph-snapshot: read the window once, write the 12 hidden states
BYTES_PER_SNAPSHOT = HORIZON * N_NODES * F_IN * 4 + HORIZON * N_NODES * HIDDEN * 4  # 337 824 B
# algorithmic FLOPs per snapshot (z/r share the diffusion): 9 GEMMs 207x34x32 + 2 dirs x (34+32) diffusion + gates
FLOPS_PER_SNAPSHOT = HORIZON * (9 * 2 * N_NODES * 34 * HIDDEN + 2 * 2 * N_EDGES * (34 + 32) + 10 * N_NODES * HIDDEN)
DUMP_WINDOWS = 128    # windows of the last step --dump-outputs writes: 128 x 318 KB of hidden states = 41 MB


def dump_rows(windows):
    """The fixed, seeded sample of a step's windows that --dump-outputs writes (all of them if there are at most DUMP_WINDOWS)."""
    return torch.randperm(windows, generator=torch.Generator().manual_seed(0))[:DUMP_WINDOWS].sort().values


def dump_outputs(out_dir, hidden, prediction):
    """hidden_states.npy: float32 (DUMP_WINDOWS, 12, 207, 32), BatchedDCRNN.forward's output for the sampled windows of the last
    timed device-resident step; prediction.npy: float32 (DUMP_WINDOWS, 207), the Linear head's output for the same windows in
    the last timed end-to-end step (absent if that leg failed).  The inputs depend only on the arguments, so two builds run
    with the same arguments can be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "hidden_states.npy"), hidden.numpy())
    if prediction is not None:
        np.save(os.path.join(out_dir, "prediction.npy"), prediction.numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_workload(seed=0, t_total=4096):
    from pytorch_geometric_temporal_b200.dataset import synthetic
    ei, ew, series = synthetic.metr_la_like(seed, t_total)
    return torch.from_numpy(ei), torch.from_numpy(ew), torch.from_numpy(series)


def make_model():
    from pytorch_geometric_temporal_b200.nn.recurrent import BatchedDCRNN
    torch.manual_seed(0)
    return BatchedDCRNN(F_IN, HIDDEN, K_HOPS)


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port of BatchedDCRNN.forward on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_reference(steps, warmup, windows=None, threads=None, budget_s=25.0):
    """Oracle port of BatchedDCRNN.forward on the host cores, EXACTLY `steps` timed steps.  The op sequence
    is many small ATen calls, so more threads is not faster: the thread count is calibrated (16 windows each)
    and the best is used; the per-step sample (windows per step) is then sized so that the whole run takes
    about `budget_s` seconds."""
    from oracle import recurrent as R
    ei, ew, series = make_workload()
    sd = {k: v.clone() for k, v in make_model().state_dict().items()}
    ncpu = os.cpu_count() or 1
    mk = lambda n: torch.stack([series[s:s + HORIZON] for s in (torch.arange(0, n) * 3).tolist()])
    cand = [threads] if threads else sorted({c for c in (4, 8, 16, 32, ncpu) if c <= ncpu})
    best, best_dt = cand[0], None
    Xc = mk(16)
    with torch.no_grad():
        ops16 = R.batched_dcrnn_operators(ei, ew, 16, N_NODES)   # the reference caches norms / reverse list (`cached_idx`, dcrnn.py:446-460)
        for c in cand:
            torch.set_num_threads(c)
            R.batched_dcrnn(sd, Xc[:4], ei, ew)
            t0 = time.perf_counter()
            R.batched_dcrnn(sd, Xc, ei, ew, ops=ops16)
            dt = time.perf_counter() - t0
            if best_dt is None or dt < best_dt:
                best, best_dt = c, dt
            if dt > 6.0:
                break
        torch.set_num_threads(best)
        if windows is None:
            windows = int(budget_s / max(1, steps + warmup) / (best_dt / 16))
            windows = max(4, min(64, windows))
        X = mk(windows)
        opsw = R.batched_dcrnn_operators(ei, ew, windows, N_NODES)
        for _ in range(warmup):
            R.batched_dcrnn(sd, X, ei, ew, ops=opsw)
        t0 = time.perf_counter()
        for _ in range(steps):
            out = R.batched_dcrnn(sd, X, ei, ew, ops=opsw)
        dt = time.perf_counter() - t0
    return {"value": windows * steps / dt, "ms_per_step": dt / steps * 1e3, "cores": best, "host_cores": ncpu, "steps_done": steps,
            "windows": windows, "out_checksum": float(out.abs().mean())}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference(args.steps, max(args.warmup, 1))
    windows = r["windows"]
    sample = (f"{windows} windows x {r['steps_done']} steps of BatchedDCRNN(2,32,K=2) fwd, oracle port (torch CPU ops = the reference's ATen "
              f"index_select/scatter_add_ path); {r['cores']} threads (best of calibration) on {r['host_cores']} host cores")
    line = {
        "impl": "reference", "metric": "graph-snapshots/sec", "value": r["value"], "unit": "snapshots/s", "n_gpus": args.gpus,
        "steps": r["steps_done"], "warmup": max(args.warmup, 1), "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "DCRNN K=2 METR-LA-shape (207 nodes, 1722 edges, 2 feats, 12-step window, hidden 32), forward",
                   "windows_per_step": windows},
        "cpu_baseline": {"value": r["value"], "unit": "snapshots/s", "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["value"], "unit": "snapshots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def spmm_probe(dev, pk):
    """SpMM GB/s vs HBM peak on the cfg5 shape (N=10^4, E=10^5 + N loops, F=128=[X|H], batch 32 > L2): the random graph of BASELINE
    configs[4] (headline of this leg) and, next to it, a sensor-network-like banded graph of the same size."""
    from pytorch_geometric_temporal_b200 import _lib, ops
    from pytorch_geometric_temporal_b200.dataset import synthetic
    from pytorch_geometric_temporal_b200.plan import GraphPlan
    B, N, F = 32, 10000, 128
    x = torch.randn(B, N, F, device=dev)
    y = torch.empty_like(x)

    def run(ei, ew):
        plan = GraphPlan(_lib.FLAVOR_CHEB, torch.from_numpy(ei).to(dev), torch.from_numpy(ew).to(dev), N, normalization="sym")
        nnz = plan.nnz(0)
        bytes_alg = B * (8 * N * F) + 8 * nnz + 4 * (N + 1)
        for _ in range(3):
            ops.spmm_raw(plan, 0, x, out=y)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        iters = 10
        e0.record()
        for _ in range(iters):
            ops.spmm_raw(plan, 0, x, out=y)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        return nnz, bytes_alg, ms, bytes_alg / (ms * 1e-3) / 1e9

    nnz, bytes_alg, ms, gbs = run(*synthetic.large_graph(N, 100000, 0))
    gather = 4 * nnz * F * B                       # source rows delivered L2 -> SM (every entry reads a 4F-byte row); not HBM traffic
    out = {"workload": "SpMM N=10000 nnz=%d F=128 batch=32 (in 164 MB + out 164 MB > L2)" % nnz, "ms": ms,
           "algorithmic_bytes": bytes_alg, "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
           "l2_gather_bytes": gather, "l2_to_sm_gbs": (gather + bytes_alg) / (ms * 1e-3) / 1e9,
           "note": "random graph: the gathered rows (5.5x the algorithmic bytes) leave L2 at its throughput cap (~6300 B/clk); l2_to_sm_gbs is that rate, see DESIGN.md section 3"}
    nnz2, bytes2, ms2, gbs2 = run(*synthetic.banded_graph(N, 100000, 64, 0))
    out["banded_graph"] = {"workload": "same sizes, every edge within 64 node ids (sensor-network-like ordering)",
                           "nnz": nnz2, "ms": ms2, "achieved": gbs2, "frac": gbs2 / pk["hbm_gbs"]}
    return out


class EpochFeeder(object):
    """Endless batches from an epoch-based loader: when an epoch is exhausted the next one is started with
    `set_epoch(epoch + 1)` (examples/indexBatching/DCRNN/pems_ddp.py:96,104).  With `drop_last=True` loaders every batch
    is full, so fixed-shape staging buffers (CUDA graphs) can be fed for any number of steps at any world size."""

    def __init__(self, loader):
        self.loader, self.epoch, self.it, self.batches = loader, 0, None, 0
        if len(loader) < 1:
            raise ValueError("loader yields no full batch per epoch (shard smaller than the batch size)")

    def next(self):
        for _ in range(2):
            if self.it is None:
                self.loader.set_epoch(self.epoch)
                self.it = iter(self.loader)
            try:
                b = next(self.it)
                self.batches += 1
                return b
            except StopIteration:
                self.it, self.epoch = None, self.epoch + 1
        raise RuntimeError("loader produced an empty epoch")


def train_probe(dev, world, rank, ei_d, ew_d, series, steps=5, windows=64):
    """Training step (fwd + bwd + ONE flat NCCL all-reduce + Adam): fused forward with stash + hand-written backward:
    BatchedDCRNN(2,32,K=2) + Linear(32,1) head, masked-MAE loss (examples/indexBatching/DCRNN/pems_ddp.py:104-121)."""
    import torch.distributed as dist
    from pytorch_geometric_temporal_b200 import distributed as D
    from pytorch_geometric_temporal_b200.signal import IndexBatchLoader, index_splits
    model = make_model().to(dev)
    head = torch.nn.Linear(HIDDEN, 1).to(dev)
    params = list(model.parameters()) + list(head.parameters())
    if world > 1:
        D.broadcast_parameters(model); D.broadcast_parameters(head)
    sync = D.FlatGradSync(params, average=False)       # the 1/world average is folded into the optimizer launch
    tr, _, _ = index_splits(series.size(0), HORIZON)
    loader = IndexBatchLoader(series.to(dev), tr, HORIZON, windows, shuffle=True, world_size=world, rank=rank, seed=0, drop_last=True)
    feeder = EpochFeeder(loader)
    opt = D.FlatAdam(sync, lr=1e-3)                    # torch.optim.Adam's update over the flat buffers: one launch (tests/test_gpu_train.py)
    sx = torch.empty((windows, HORIZON, N_NODES, F_IN), device=dev)
    sy = torch.empty((windows, HORIZON, N_NODES, F_IN), device=dev)
    loss_buf = torch.zeros((), device=dev)

    def body():
        h = model(sx, ei_d, ew_d)                      # (B,12,N,32)
        pred = head(h[:, -1]).squeeze(-1)              # (B,N)
        loss = D.masked_mae_loss(pred, sy[:, 0, :, 0])
        loss.backward()
        sync.all_reduce()
        opt.step(grad_scale=1.0 / world)               # also clears the gradient buffer
        loss_buf.copy_(loss.detach())

    def feed():
        x, y = feeder.next()
        sx.copy_(x); sy.copy_(y)

    # The step is a fixed sequence of ~45 launches (the recurrence kernels, the weight-gradient contraction, the head / loss and one Adam
    # launch): capture it ONCE in a CUDA graph (plans are cached, all
    # buffers static) and replay it -- graphs instead of a tracing compiler.  Falls back to eager if capture fails.
    mode = "cuda-graph"
    side = torch.cuda.Stream(device=dev)
    try:
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                feed(); body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body()
        run = graph.replay
    except Exception as e:  # noqa
        mode = f"eager (graph capture failed: {type(e).__name__})"
        torch.cuda.synchronize()
        run = body
    for _ in range(2):
        feed(); run()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        feed(); run()
    e1.record()
    torch.cuda.synchronize()
    loss = loss_buf
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    return {"value": world * windows / (ms * 1e-3), "unit": "snapshots/s", "ms_per_step": ms, "windows_per_step_per_gpu": windows,
            "path": "fused fwd (stmp_dcrnn_seq_fwd + stash) + persistent bwd (stmp_dcrnn_bwd_basis || stmp_dcrnn_bwd_seq) + stmp_dcrnn_bwd_wgrad + flat all-reduce + stmp_adam_flat", "launch": mode, "allreduce_bytes_per_step": sync.nbytes if world > 1 else 0,
            "loss": float(loss.detach())}


def run_ours(args):
    import torch.distributed as dist
    from pytorch_geometric_temporal_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    B = args.windows
    ei, ew, series = make_workload(seed=0)
    ei_d, ew_d = ei.to(dev), ew.to(dev)
    model = make_model().to(dev)

    # Rotating device-resident input batches: R x (B x 19 872 B); together with the 318 KB/window output
    # (B x 317 952 B written per step) each step's traffic exceeds the 126 MB L2.
    n_rot = 8
    g = torch.Generator().manual_seed(1234 + rank)
    starts = [torch.randint(0, series.size(0) - HORIZON, (B,), generator=g) for _ in range(n_rot)]
    host_batches = [torch.stack([series[s:s + HORIZON] for s in st.tolist()]).pin_memory() for st in starts]
    dev_batches = [hb.to(dev) for hb in host_batches]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident(i):
        with torch.no_grad():
            return model(dev_batches[i % n_rot], ei_d, ew_d)

    # ---- device-resident throughput (`value`) ----------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(max(args.warmup, 20)):     # >= 20 launches of warm-up: clocks are sampled under the same load
        out = step_resident(i)
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        out = step_resident(i)
    e1.record()
    barrier()
    launches = _lib.launch_count() - l0
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    dump = args.dump_outputs is not None and rank == 0
    if dump:
        rows = dump_rows(B)
        hidden = out[rows.to(dev)].cpu()
    t = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total * 1e-3)

    # ---- end to end through the public index-batching API --------------------------------------------------------
    # The reference's own large-scale data path (index-batching, signal/index_dataset.py:43-57 + dataset/metr_la.py:180-190)
    # keeps the normalised series resident on the GPU and ships only WHICH windows form a batch.  Every step here: the
    # host hands that step's window starts (pinned int64 [B]) to signal.DevicePrefetcher (H2D on a side stream while the
    # previous step computes) -> BatchedDCRNN.forward_indexed reads the windows in-kernel from the resident series ->
    # Linear(32,1) head on the last hidden state (the consumer of examples/indexBatching/DCRNN/pems_ddp.py:104-121) ->
    # the (B, N) prediction is copied to pinned host memory and read by the host, one step behind the launch front.
    from pytorch_geometric_temporal_b200.signal import DevicePrefetcher
    series_d = series.to(dev)
    torch.manual_seed(1)
    head = torch.nn.Linear(HIDDEN, 1).to(dev)
    head_w = head.weight.detach().t().unsqueeze(0).expand(B, HIDDEN, 1)
    head_b = head.bias.detach().view(1, 1, 1).expand(B, N_NODES, 1)
    host_starts = [st.to(torch.int64).pin_memory() for st in starts]
    pred_host = [torch.empty((B, N_NODES), pin_memory=True) for _ in range(2)]
    pred_done = [torch.cuda.Event() for _ in range(2)]
    head_done = [torch.cuda.Event() for _ in range(2)]
    d2h_stream = torch.cuda.Stream(device=dev)       # the result copy rides the copy engine next to the following step's kernel

    def run_e2e(n):
        last, prev, slot = 0.0, None, 0
        for st in DevicePrefetcher((host_starts[i % n_rot] for i in range(n)), dev):
            with torch.no_grad():
                h = model.forward_indexed(series_d, st, HORIZON, ei_d, ew_d)      # (B,12,N,32), windows read in-kernel
                # Linear(32,1) on the last step's rows of h, read in place (a strided batched product: no contiguous copy of the 31 MB slice)
                pred = torch.baddbmm(head_b, h[:, -1], head_w).squeeze(-1)                       # (B,N)
            head_done[slot].record()
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(head_done[slot])
                pred.record_stream(d2h_stream)
                pred_host[slot].copy_(pred, non_blocking=True)
                pred_done[slot].record()
            if prev is not None:
                pred_done[prev].synchronize()
                last = float(pred_host[prev][0, 0])
            prev, slot = slot, slot ^ 1
        if prev is not None:
            pred_done[prev].synchronize()
            last = float(pred_host[prev][0, 0]) + float(pred_host[prev][-1, -1])
        return last

    roofline = cpu_note = None
    e2e = {"value": None, "unit": "snapshots/s", "h2d_bytes_per_step": B * 8, "d2h_bytes_per_step": B * N_NODES * 4,
           "api": "IndexBatchLoader-style window starts (pinned host) -> signal.DevicePrefetcher -> BatchedDCRNN.forward_indexed(resident series) "
                  "-> Linear(32,1) head -> (B,N) prediction copied to pinned host memory (side stream) and read by the host every step, one step behind the launch front"}
    try:
        run_e2e(max(3, args.warmup // 2))
        barrier()
        e0.record()
        run_e2e(args.steps)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e["value"] = world * B * args.steps / (float(t.item()) * 1e-3)
    except Exception as e:  # noqa: the device-timed headline above must survive a failure here
        if world > 1:
            raise                                   # ranks must stay in lock step around collectives: fail loudly under torchrun
        e2e["error"] = f"{type(e).__name__}: {e}"
    if dump:
        # step i of run_e2e leaves its prediction in pred_host[i % 2]
        dump_outputs(args.dump_outputs, hidden, pred_host[(args.steps - 1) % 2][rows] if e2e["value"] is not None else None)

    # ---- roofline of the dominant kernel (k_dcrnn_seq_tc = the whole step) ---------------------------------------
    achieved_gbs = B * BYTES_PER_SNAPSHOT / (ms_step * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "dcrnn_seq_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"kernel": "k_dcrnn_seq_tc (tcgen05)", "bound": "hbm", "achieved": achieved_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": achieved_gbs / pk["hbm_gbs"], "traffic": traffic, "peak_source": pk["source"],
                "algorithmic_bytes_per_launch": B * BYTES_PER_SNAPSHOT,
                "note": "fused kernel is shared-memory-bandwidth bound (gather/scatter of the diffusion); contraction on tcgen05; HBM fraction reported as north_star asks",
                "fp32_tflops_achieved": B * FLOPS_PER_SNAPSHOT / (ms_step * 1e-3) / 1e12}
    line = {
        "metric": "graph-snapshots/sec", "value": value, "unit": "snapshots/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "DCRNN K=2 METR-LA-shape (207 nodes, 1722 edges, 2 feats, 12-step window, hidden 32), forward (BatchedDCRNN.forward), all 12 H_t written",
                   "windows_per_step_per_gpu": B, "parallelism": f"dp{world} (independent windows, no data-path collective)",
                   "l2_policy": "8 rotating input batches + 318 KB/window output: per-step traffic > 126 MB L2"},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "path_counters": {k: v for k, v in _lib.path_counters().items() if v},
        "spmm": None, "train": None, "cpu_baseline": None, "reference_gpu": None, "e2e_host_windows": None,
    }

    def host_windows_leg():
        """The round-1 e2e variant: the WINDOWS themselves (B x 19 872 B) come from pinned host memory every step."""
        metric_host = [torch.empty(1, pin_memory=True) for _ in range(2)]
        metric_done = [torch.cuda.Event() for _ in range(2)]

        def run(n):
            last, prev, slot = 0.0, None, 0
            for xb in DevicePrefetcher((host_batches[i % n_rot] for i in range(n)), dev):
                with torch.no_grad():
                    m = model(xb, ei_d, ew_d)[:, -1].abs().mean()
                metric_host[slot].copy_(m.reshape(1), non_blocking=True)
                metric_done[slot].record()
                if prev is not None:
                    metric_done[prev].synchronize()
                    last = float(metric_host[prev][0])
                prev, slot = slot, slot ^ 1
            metric_done[prev].synchronize()
            return last + float(metric_host[prev][0])

        run(3)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        run(args.steps)
        f1.record()
        barrier()
        tt = torch.tensor([f0.elapsed_time(f1)], device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return {"value": world * B * args.steps / (float(tt.item()) * 1e-3), "unit": "snapshots/s",
                "h2d_bytes_per_step": B * HORIZON * N_NODES * F_IN * 4, "d2h_bytes_per_step": 4,
                "api": "pinned host windows -> DevicePrefetcher -> BatchedDCRNN.forward -> scalar metric read every step"}

    # ---- secondary legs under a hard wall-clock budget ----------------------------------------------------------------
    # The headline numbers above are complete.  cpu_baseline / SpMM probe / reference-on-GPU / training probe run under a
    # deadline counted from process start, each inside its own try/except: a leg that fails is recorded as {"error": ...}
    # and a leg that does not return in time is listed in `legs_skipped` -- the line is printed either way.
    _secondary_legs(line, args, rank, world, dev, pk, ei_d, ew_d, series, host_windows_leg)
    if world > 1:
        dist.destroy_process_group()


def reference_gpu_probe(dev, ei_d, ew_d, series, windows, iters=5):
    """The "reference-on-B200" comparator (SURVEY 8d, GPU timing): the reference's op-for-op sequence -- index_select ->
    norm * x_j -> scatter_add_ -> matmul per gate per step, block-diagonal batch graph -- with every tensor on the GPU
    (oracle port, device-agnostic), eager and replayed from a CUDA graph.  Same windows per step as our arm."""
    from oracle import recurrent as R
    sd = {k: v.to(dev) for k, v in make_model().state_dict().items()}
    X = torch.stack([series[s:s + HORIZON] for s in (torch.arange(0, windows) * 3 % (series.size(0) - HORIZON)).tolist()]).to(dev)
    out = {}
    with torch.no_grad():
        ops = R.batched_dcrnn_operators(ei_d, ew_d, windows, N_NODES)
        for _ in range(2):
            y = R.batched_dcrnn(sd, X, ei_d, ew_d, ops=ops)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            y = R.batched_dcrnn(sd, X, ei_d, ew_d, ops=ops)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        out["eager"] = {"value": windows / (ms * 1e-3), "ms_per_step": ms}
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                y = R.batched_dcrnn(sd, X, ei_d, ew_d, ops=ops)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                y = R.batched_dcrnn(sd, X, ei_d, ew_d, ops=ops)
            g.replay()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(iters):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            out["cuda_graph"] = {"value": windows / (ms * 1e-3), "ms_per_step": ms}
        except Exception as e:  # noqa
            out["cuda_graph"] = {"error": f"{type(e).__name__}: {e}"}
    out.update({"unit": "snapshots/s", "windows_per_step": windows, "kind": "oracle op sequence (index_select/mul/scatter_add_/matmul) on cuda:0, fp32",
                "out_checksum": float(y.abs().mean())})
    return out


def _leg(fn):
    try:
        return fn()
    except Exception as e:  # noqa: a secondary leg never takes the headline down
        return {"error": f"{type(e).__name__}: {str(e)[:300]}"}


def _secondary_legs(line, args, rank, world, dev, pk, ei_d, ew_d, series, host_windows_leg=None):
    """cpu_baseline (rank 0, N=1), SpMM probe (rank 0), reference-on-GPU (rank 0, N=1), host-window e2e (all ranks), training
    probe (all ranks: it holds the all-reduce), each written into `line` as it finishes; the line is printed by rank 0
    when all are done or when the deadline expires.  Legs with collectives re-raise under torchrun (ranks must not diverge);
    everything else is recorded as {"error": ...}."""
    legs = _LegDeadline(line, ["cpu_baseline", "spmm", "reference_gpu", "e2e_host_windows", "train"], emit_line=(rank == 0),
                        seconds=max(20.0, BUDGET_S - (time.time() - _T0)))
    solo = (lambda fn: _leg(fn)) if world == 1 else (lambda fn: fn())

    def cpu_leg():
        r = cpu_reference(steps=10, warmup=1, budget_s=15.0)
        return {"value": r["value"], "unit": "snapshots/s", "cores": r["cores"], "kind": "port",
                "sample": f"{r['windows']} windows x {r['steps_done']} steps, oracle port of BatchedDCRNN.forward on torch CPU ops; "
                          f"{r['cores']} threads (best of calibration) on {r['host_cores']} host cores"}

    try:
        legs.done("cpu_baseline", _leg(cpu_leg) if (rank == 0 and world == 1 and not args.no_cpu) else None)
        legs.done("spmm", _leg(lambda: spmm_probe(dev, pk)) if (rank == 0 and not args.no_spmm) else None)
        legs.done("reference_gpu", _leg(lambda: reference_gpu_probe(dev, ei_d, ew_d, series, args.windows))
                  if (rank == 0 and world == 1 and not args.no_refgpu) else None)
        legs.done("e2e_host_windows", solo(host_windows_leg) if (host_windows_leg is not None and not args.no_hostwin) else None)
        legs.done("train", solo(lambda: train_probe(dev, world, rank, ei_d, ew_d, series)) if not args.no_train else None)
    except BaseException as e:  # noqa: print what is measured, then fail loudly
        line["leg_failure"] = f"{type(e).__name__}: {str(e)[:300]}"
        legs.finish()
        raise
    legs.finish()


class _LegDeadline(object):
    """Wall-clock deadline for the secondary legs of a bench line.  `done(key, value)` fills a leg in; `finish()` prints
    the line (once).  If the deadline expires first, the line is printed with the legs finished so far plus a
    `legs_skipped` note and the process exits 0 -- from a timer thread, so a leg stuck in native code cannot hold it up."""

    def __init__(self, line, legs, emit_line, seconds):
        self.line, self.pending, self.emit_line = line, list(legs), emit_line
        self.lock, self.closed = threading.Lock(), False
        self.timer = threading.Timer(seconds, self._expire)
        self.timer.daemon = True
        self.timer.start()

    def _expire(self):
        with self.lock:
            if self.closed:
                return
            self.closed = True
            if self.emit_line:
                self.line["legs_skipped"] = {"legs": list(self.pending), "why": f"wall-clock budget of {BUDGET_S:.0f} s reached"}
                emit(self.line)
            os._exit(0)

    def done(self, key, value):
        with self.lock:
            self.line[key] = value
            self.pending.remove(key)

    def finish(self):
        with self.lock:
            if self.closed:
                return
            self.closed = True
            self.timer.cancel()
            if self.emit_line:
                emit(self.line)


_REAL_STDOUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to
    stdout at communicator creation), so fd 1 is pointed at stderr for the whole run and the JSON line is written to
    the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--windows", type=int, default=1184, help="windows per step per GPU (8 per SM)")
    ap.add_argument("--no-spmm", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-refgpu", action="store_true")
    ap.add_argument("--no-hostwin", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's outputs for a fixed "
                    "sample of its windows as DIR/hidden_states.npy and DIR/prediction.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of our arm (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
