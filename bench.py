#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config, on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--skip-configs] [--dump-outputs DIR]

metric  : XSimGCL yelp2018 train steps/sec (+ full-catalog rank items/sec as `rank`)
workload: configs[2] of BASELINE.json -- XSimGCL, yelp2018 shape (31 668 x 38 048 x 1 237 259, synthetic power-law
          graph of that shape), 3 layers, d=64, B=2048, tau=0.2, lambda=0.2, eps=0.2, l*=1, lr=1e-3, reg=1e-4, fp32.
A step  = one pass of the hot path over one batch: propagate (3 SpMM) -> gather + BPR + L2 -> InfoNCE -> Horner
          backward (3 SpMM) -> Adam, on in-kernel Philox noise.
value   = steps/s with the batch indices already resident in HBM (a device pool of pre-sampled batches), CUDA-graph
          replay, CUDA-event timing, max over ranks.  N = 1: the fused single-GPU engine (srb_train_step).
          N > 1: the SAME job on bipartite-sharded tables (srb_shard_step; strong scaling), self-verified in the
          run against the single-GPU engine (`parity`).
e2e     = the same metric through the public API with HOST buffers, every step: one native sampler call (inside the
          timed region) -> pinned H2D copy of the batch -> the step -> D2H copy of the losses, read one step late.
          Same measurement at every N.
Other configs of BASELINE.json ride along as sub-records of the same JSON line: `config2` (LightGCN yelp2018),
`config4` (SGL edge-drop, amazon-kindle shape, view graphs rebuilt on the device), `config5` (SimGCL, synthetic
10 M x 2 M x 200 M, d = 128; single GPU at N = 1, bipartite-sharded at N > 1).
--impl reference times the reference's own CPU path on the host cores: the UNMODIFIED reference unpacked from
oracle/_ref/reference.zip (kind "reference") when build() made that archive, else the op-for-op port
oracle/torch_port.py (kind "port"); rank 0 only; best of a thread-count sweep.
--dump-outputs DIR (N = 1) writes what the last timed step left to its caller -- user_emb [U, d], item_emb [I, d] and
the four losses, float32 -- as DIR/<name>.npy (17.8 MB).  The inputs are seeded: the same arguments give the same
inputs on every run, so two builds can be compared output for output.  The step adds its gradient scatters with
atomics, so two runs of one build agree closely but not bit for bit (two pairs of runs, --steps 20 --warmup 5 on a B200
at 1000 W: tables within 5e-3 in relative Frobenius norm, losses within 1e-4 relative); compare with a tolerance.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(model="XSimGCL", shape="yelp2018", d=64, L=3, B=2048, tau=0.2, lam=0.2, eps=0.2, l_star=1, lr=1e-3, reg=1e-4)
METRIC = "XSimGCL yelp2018 train steps/sec"
WORKLOAD = "XSimGCL yelp2018-shape 31668x38048x1237259, L=3 d=64 B=2048 tau=0.2 lambda=0.2 eps=0.2 l*=1"
TRAFFIC_FILE = os.path.join("profiles", "r02_spmm_traffic.json")  # dram bytes per launch from this round's ncu capture

_JSON_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout: libraries that write banners to fd 1 (NCCL's version line) are
    pointed at stderr for the whole run, and the JSON line goes to the saved descriptor."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def log(msg):
    sys.stderr.write(f"[bench] {msg}\n")
    sys.stderr.flush()


def peaks():
    """Roofline denominators: the driver-measured copy bandwidth and cuBLAS bf16 rate of this pool's B200s."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d.get("bf16_tflops", 1702.0)), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1700.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as f:
            for line in f:
                parts = [x.strip() for x in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    mx.append(float(parts[2]))
                except ValueError:
                    continue
                for nm, val in zip(names, parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write {name: float32 / float64 array} as out_dir/<name>.npy; at most DUMP_LIMIT_BYTES in all."""
    arrays = {k: np.ascontiguousarray(v) for k, v in arrays.items()}
    for k, v in arrays.items():
        if v.dtype not in (np.float32, np.float64):
            raise ValueError(f"--dump-outputs: {k} is {v.dtype}, not float32 / float64")
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the limit of {DUMP_LIMIT_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v)


def spmm_bytes(n, nnz, d):
    """SURVEY 8(d): compulsory bytes of one SpMM = read CSR once + read X once + write Y once."""
    return 8 * nnz + 4 * (n + 1) + 8 * n * d


def step_bytes(model, n, nnz, d, L, view_nnz=None):
    """SURVEY 8(d): P * L * S + 28 * N * d with P = SpMM passes per layer per step."""
    S = spmm_bytes(n, nnz, d)
    if model in ("LightGCN", "XSimGCL"):
        prop = 2 * L * S
    elif model == "SimGCL":
        prop = 6 * L * S
    else:  # SGL: clean graph fwd + bwd, two view graphs fwd + bwd
        prop = 2 * L * S + 4 * L * spmm_bytes(n, view_nnz or nnz, d)
    return prop + 28 * n * d


def build_data(seed=0):
    from selfrec_b200 import synth
    return synth.make_interaction(CFG["shape"], seed=seed)


def xs_kwargs():
    return dict(eps=CFG["eps"], tau=CFG["tau"], cl_rate=CFG["lam"], layer_cl=CFG["l_star"])


def time_steps(step_fn, steps, warmup, torch, dist=None):
    """W warm-up steps, then K steps bracketed by a barrier + synchronize, CUDA events, max over ranks (ms total)."""
    for k in range(warmup):
        step_fn(k)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for k in range(steps):
        step_fn(k)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dist is not None:
        dist.barrier()
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def keep_load(step_fn, ms_per_step, torch, seconds=0.4):
    """The timed region of 20 steps lasts a few milliseconds -- shorter than nvidia-smi's sampling period -- so the clock
    sampler would see nothing.  After the timed region (its events are already recorded) the SAME step keeps running
    for `seconds`: the `clocks` entry is the median over the timed region and this continuation of the same load.
    The step count depends only on ms_per_step, which is identical on every rank."""
    n = int(min(20000, max(50, seconds * 1e3 / max(ms_per_step, 1e-3))))
    for k in range(n):
        step_fn(k)
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's CPU PyTorch path on the host cores
# ------------------------------------------------------------------------------------------
THREADS = (8, 16, 32, 64, 128)


class CpuPath:
    """The reference's CPU path for the bench workload: the unmodified reference when its archive travelled, else the
    port.  run(steps, warmup) -> seconds; rank() -> (seconds, users, items)."""

    def __init__(self, data):
        import torch
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import refarchive
        self.torch = torch
        self.kind = "port"
        self.scratch = tempfile.mkdtemp(prefix="srb_ref_")
        if refarchive.available():
            try:
                import ref_runner
                cwd = os.getcwd()
                root = refarchive.unpack(os.path.join(self.scratch, "reference"))
                self.ref = ref_runner.ReferenceXSimGCL(root, os.path.join(self.scratch, "run"), data.pair_users, data.pair_items, d=CFG["d"],
                                                       L=CFG["L"], B=CFG["B"], lr=CFG["lr"], reg=CFG["reg"], eps=CFG["eps"], tau=CFG["tau"],
                                                       lam=CFG["lam"], l_star=CFG["l_star"], test_users=1000)
                os.chdir(cwd)
                self.kind = "reference"
            except Exception as e:  # noqa: BLE001 -- the port is the documented fallback of the reference arm
                log(f"unmodified reference unusable ({type(e).__name__}: {e}); using the port")
        if self.kind == "port":
            import random
            import torch_port
            random.seed(0)
            self.tp = torch_port
            self.m = torch_port.XSimGCLCpu(data.norm_adj.tocsr(), data.user_num, data.item_num, CFG["d"], CFG["L"], CFG["eps"], CFG["tau"],
                                           CFG["lam"], CFG["l_star"], CFG["lr"], CFG["reg"])
            rp, ri = data.rated_csr()
            self.rp, self.ri = rp, ri
            self.rated = [set(ri[rp[u]:rp[u + 1]].tolist()) for u in range(data.user_num)]
            perm = np.random.default_rng(0).permutation(len(data.pair_users))
            self.pu, self.pi, self.ptr = data.pair_users[perm], data.pair_items[perm], 0
            self.data = data

    def run(self, steps, warmup):
        if self.kind == "reference":
            cwd = os.getcwd()
            os.chdir(os.path.join(self.scratch, "run"))
            try:
                return self.ref.time_steps(steps, max(warmup, 1))
            finally:
                os.chdir(cwd)
        def one():
            u, i, j, self.ptr = self.tp.sample_batch(self.pu, self.pi, self.ptr, CFG["B"], self.data.item_num, self.rated)
            if self.ptr >= len(self.pu):
                self.ptr = 0
            self.m.step(u, i, j)
        for _ in range(warmup):
            one()
        t0 = time.perf_counter()
        for _ in range(steps):
            one()
        return time.perf_counter() - t0

    def rank(self):
        if self.kind == "reference":
            cwd = os.getcwd()
            os.chdir(os.path.join(self.scratch, "run"))
            try:
                return self.ref.time_rank()
            finally:
                os.chdir(cwd)
        import oracle
        ue, ie = self.m.ue.detach().numpy(), self.m.ie.detach().numpy()
        sample = np.arange(0, self.data.user_num, max(1, self.data.user_num // 1000))[:1000]
        t0 = time.perf_counter()
        self.tp.rank_users(ue, ie, sample, self.rp, self.ri, 20, oracle.find_k_largest)
        return time.perf_counter() - t0, len(sample), self.data.item_num

    def sweep(self, budget_s=40.0):
        """Steps/s per thread count (1 warm-up + 2 timed steps each, within a time budget); returns (best_T, table)."""
        torch = self.torch
        cores = os.cpu_count() or 1
        table, t_start = {}, time.perf_counter()
        for T in [t for t in THREADS if t <= cores] or [cores]:
            torch.set_num_threads(T)
            table[T] = 2 / self.run(2, 1)
            if time.perf_counter() - t_start > budget_s:
                break
        best = max(table, key=table.get)
        torch.set_num_threads(best)
        return best, table


def run_reference(args, rank, world):
    if rank != 0:
        return
    data = build_data()
    cpu = CpuPath(data)
    best, table = cpu.sweep()
    steps = min(args.steps, 20)
    warm = min(max(args.warmup, 1), 5)
    # bounded: keep the whole arm within a few minutes whatever the host
    per_step = 1.0 / table[best]
    steps = max(2, min(steps, int(60.0 / per_step)))
    dt = cpu.run(steps, warm)
    val = steps / dt
    rdt, r_users, r_items = cpu.rank()
    note = ("UNMODIFIED reference (oracle/_ref/reference.zip): its own XSimGCL.train() loop, sampler, losses, torch.optim.Adam"
            if cpu.kind == "reference" else "op-for-op port of the reference's CPU path (oracle/torch_port.py) incl. Python sampler")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "steps/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak" if args.gpus == 1 else "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": note},
        "cpu_baseline": {"value": val, "unit": "steps/s", "cores": best, "kind": cpu.kind, "host_cores": os.cpu_count(),
                         "thread_sweep_steps_per_s": {str(k): v for k, v in table.items()},
                         "sample": f"{steps} full train steps after {warm} warm-up, torch threads = best of the sweep"},
        "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rank": {"value": r_users * r_items / rdt, "unit": "items/s", "sample": f"{r_users} of {data.user_num} users"},
    }
    emit(line)


def cpu_baseline(data, budget_s=45.0):
    """Bounded sample of the same workload on the host cores (reported beside, not the target)."""
    cpu = CpuPath(data)
    best, table = cpu.sweep(budget_s=budget_s * 0.6)
    per_step = 1.0 / table[best]
    steps = max(2, min(10, int(budget_s * 0.4 / per_step)))
    dt = cpu.run(steps, 1)
    return {"value": steps / dt, "unit": "steps/s", "cores": best, "kind": cpu.kind, "host_cores": os.cpu_count(),
            "thread_sweep_steps_per_s": {str(k): v for k, v in table.items()},
            "sample": f"{steps} full XSimGCL train steps ({'unmodified reference, its own train() loop' if cpu.kind == 'reference' else 'oracle/torch_port.py'}"
                      f", torch CPU, Python sampler) after 1 warm-up; thread count = best of the sweep"}


# ------------------------------------------------------------------------------------------
# sub-records: the other configs of BASELINE.json
# ------------------------------------------------------------------------------------------
def record_config2(args, dev, data):
    """configs[1]: LightGCN on yelp2018 shape, 3 layers, d=64, B=2048, one GPU."""
    import torch
    from selfrec_b200.engine import TrainEngine
    from selfrec_b200.shard_check import device_batches
    torch.manual_seed(2)
    eng = TrainEngine("LightGCN", data, 64, 3, 2048, 1e-3, 1e-4, l2_div=2048.0, device=dev)
    pool = device_batches(data, 2048, 32, seed=2, dev=dev)
    g = eng.capture()

    def step(k):
        eng.batch_dev.copy_(pool[k % 32], non_blocking=True)
        g.replay()

    ms = time_steps(step, args.steps, max(args.warmup, 3), torch)
    N, nnzA = eng.N, eng.adj.nnz
    sb = step_bytes("LightGCN", N, nnzA, 64, 3)
    pk = peaks()
    return {"workload": "LightGCN yelp2018-shape, L=3 d=64 B=2048 (SpMM + BPR fused step)", "value": args.steps / (ms * 1e-3), "unit": "steps/s",
            "ms_per_step": ms / args.steps, "step_algorithmic_bytes": sb, "step_frac_of_hbm": sb / (ms / args.steps * 1e-3) / 1e9 / pk["hbm_gbs"],
            "loss": eng.losses.cpu().tolist()}


def record_config4(args, dev):
    """configs[3]: SGL edge-drop on amazon-kindle shape (138 333 x 98 572 x 1 525 091 + 2 822 duplicate lines), 3 layers,
    d=64; the two view graphs are drawn (CPython-exact random.sample) and rebuilt on the device every epoch."""
    import random
    import torch
    from selfrec_b200 import synth
    from selfrec_b200.data.augmentor import sample_range
    from selfrec_b200.data.device_graph import DeviceBipartite
    from selfrec_b200.engine import TrainEngine
    from selfrec_b200.shard_check import device_batches
    U, I, nnz = synth.SHAPES["amazon-kindle"]
    pu, pi = synth.make_pairs(U, I, nnz, seed=4)
    dup = np.random.default_rng(4).choice(nnz, 2822, replace=False)  # kindle's duplicate lines -> 2.0 entries
    data = synth.ArrayInteraction(np.concatenate([pu, pu[dup]]), np.concatenate([pi, pi[dup]]), U, I)
    torch.manual_seed(4)
    random.seed(4)
    eng = TrainEngine("SGL", data, 64, 3, 2048, 1e-3, 1e-4, tau=0.2, cl_rate=0.1, device=dev)
    bip = DeviceBipartite.from_interaction_mat(data.interaction_mat, dev)

    def views():
        out = []
        for _ in range(2):
            keep = sample_range(bip.nnz, int(bip.nnz * (1 - 0.1)))
            out.append(bip.assemble(keep_idx=keep, reset_weights=True))
        return out

    v = views()  # warm-up of the assembly kernels
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    v = views()
    torch.cuda.synchronize()
    view_ms = 1e3 * (time.perf_counter() - t0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    keep_dev = torch.from_numpy(sample_range(bip.nnz, int(bip.nnz * 0.9))).to(dev)
    e0.record()
    bip.assemble(keep_idx=keep_dev, reset_weights=True)
    e1.record()
    torch.cuda.synchronize()
    eng.set_view_graphs(*v)
    pool = device_batches(data, 2048, 32, seed=4, dev=dev)
    g = eng.capture()

    def step(k):
        eng.batch_dev.copy_(pool[k % 32], non_blocking=True)
        g.replay()

    ms = time_steps(step, args.steps, max(args.warmup, 3), torch)
    sb = step_bytes("SGL", eng.N, eng.adj.nnz, 64, 3, view_nnz=v[0].nnz)
    pk = peaks()
    return {"workload": "SGL edge-drop amazon-kindle-shape 138333x98572x1525091 (+2822 duplicate lines), L=3 d=64 B=2048 rho=0.1 tau=0.2 lambda=0.1",
            "value": args.steps / (ms * 1e-3), "unit": "steps/s", "ms_per_step": ms / args.steps, "step_algorithmic_bytes": sb,
            "step_frac_of_hbm": sb / (ms / args.steps * 1e-3) / 1e9 / pk["hbm_gbs"],
            "views_per_epoch_ms": view_ms, "view_assemble_device_ms": e0.elapsed_time(e1),
            "view_note": "two views: random.sample keep-lists on the host (native, CPython-exact) + H2D + srb_graph_assemble on the device",
            "view_nnz": v[0].nnz, "loss": eng.losses.cpu().tolist()}


def record_config5(args, dev, world, rank, dist):
    """configs[4]: SimGCL on the synthetic 10 M x 2 M x 200 M bipartite graph (SURVEY 8d recipe: Zipf(1.1) on both
    sides, de-duplicated, first-appearance ids; generated, assembled and normalised on the GPU), d=128, L=3, B=2048,
    eps=0.1, lambda=0.5, tau=0.2.  N = 1: the single-GPU engine; N > 1: bipartite-sharded.  SRB_CONFIG5=<shape>
    selects another shape (e.g. synthetic-2M, the mid-size stand-in)."""
    import torch
    from selfrec_b200 import ops, synth
    from selfrec_b200.shard_check import device_batches, sharded_vs_single
    shape_name = os.environ.get("SRB_CONFIG5", "synthetic-10M")
    U, I, nnz = synth.SHAPES[shape_name]
    d, L, B = 128, 3, 2048
    kw = dict(eps=0.1, tau=0.2, cl_rate=0.5)
    rec = {"workload": f"SimGCL {shape_name} {U}x{I}x{nnz} Zipf(1.1) bipartite, L={L} d={d} B={B} eps=0.1 lambda=0.5 tau=0.2", "n_gpus": world}
    t0 = time.perf_counter()
    data = synth.make_device_interaction((U, I, nnz), seed=0, alpha=1.1, device=dev)
    torch.cuda.synchronize()
    rec["graph_build_s"] = time.perf_counter() - t0
    adj = data.norm_adj
    N, nnzA = adj.shape[0], adj.nnz
    rec.update(n=N, nnzA=nnzA, split_rows=adj.n_huge, split_row_chunks=adj.n_work)
    steps = max(3, min(args.steps, 10))
    pool = device_batches(data, B, 8, seed=5, dev=dev)
    pk = peaks()
    alg = spmm_bytes(N, nnzA, d)
    if world == 1:
        from selfrec_b200.engine import TrainEngine
        # the dominant kernel alone: full SpMM, live CUDA-event timing
        x = torch.randn(N, d, device=dev)
        y = torch.empty_like(x)
        ops._spmm_raw(adj, x, y)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(2):
            ops._spmm_raw(adj, x, y)
            ops._spmm_raw(adj, y, x)
        e1.record()
        torch.cuda.synchronize()
        sp_ms = e0.elapsed_time(e1) / 4
        del x, y
        torch.cuda.empty_cache()
        traffic = None
        tp = os.path.join(ROOT, TRAFFIC_FILE)
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f).get(shape_name)
        rec["spmm"] = {"kernel": "spmm_hub_kernel<128> + spmm_csr_kernel<128>", "ms_per_launch": sp_ms, "algorithmic_bytes": alg,
                       "achieved_gbs": alg / sp_ms / 1e6, "frac_of_hbm": alg / sp_ms / 1e6 / pk["hbm_gbs"],
                       "gather_bytes": 4 * nnzA * d, "gather_gbs": 4 * nnzA * d / sp_ms / 1e6, "dram_traffic": traffic,
                       "traffic_source": TRAFFIC_FILE if traffic else None,
                       # what the memory system actually moves: on a graph without community structure every non-zero whose
                       # column is not among the ~200 k rows L2 can hold costs a 512-byte DRAM read (DESIGN 4.1)
                       "dram_frac_of_hbm": (traffic / sp_ms / 1e6 / pk["hbm_gbs"]) if traffic else None}
        torch.manual_seed(5)
        eng = TrainEngine("SimGCL", data, d, L, B, 1e-3, 1e-4, device=dev, philox_seed=55, **kw)
        g = eng.capture()

        def step(k):
            eng.batch_dev.copy_(pool[k % 8], non_blocking=True)
            g.replay()

        ms = time_steps(step, steps, 3, torch)
        rec["engine"] = "single GPU (srb_train_step)"
        rec["loss"] = eng.losses.cpu().tolist()
        rec["mem_gb"] = torch.cuda.max_memory_allocated() / 1e9
        del eng, g
    else:
        from selfrec_b200.sharded import ShardedEngine
        sh = ShardedEngine("SimGCL", data, d, L, B, 1e-3, 1e-4, device=dev, philox_seed=55, **kw)
        sh.capture()

        def step(k):
            sh.batch_dev.copy_(pool[k % 8], non_blocking=True)
            sh.step_resident()

        ms = time_steps(step, steps, 3, torch, dist)
        sh.check_peers()
        layers = 4 * L  # 3 forward encoders + 1 merged backward chain
        rec["engine"] = f"bipartite-sharded x{world} (srb_shard_step), peer stores: {'NVSwitch multicast' if sh.use_multicast else 'P2P unicast'}"
        rec["nvlink_bytes_out_per_step_per_rank"] = int(sh.nvlink_bytes_per_layer() * layers)
        rec["loss"] = sh.losses.cpu().tolist()
        rec["mem_gb"] = torch.cuda.max_memory_allocated() / 1e9
        del sh
    torch.cuda.empty_cache()
    rec.update(steps=steps, ms_per_step=ms / steps, value=steps / (ms * 1e-3), unit="steps/s")
    sb = step_bytes("SimGCL", N, nnzA, d, L)
    rec["step_algorithmic_bytes"] = sb
    rec["step_frac_of_hbm"] = sb / (ms / steps * 1e-3) / 1e9 / (pk["hbm_gbs"] * world)
    del data, adj, pool
    torch.cuda.empty_cache()
    # self-verification on a graph of >= 1 M nodes (the full one does not leave room for a second engine):
    # sharded step vs single-GPU engine, same batches, same Philox noise
    try:
        mid = synth.make_device_interaction(synth.SHAPES["synthetic-2M"], seed=1, alpha=1.1, device=dev)
        mb = device_batches(mid, B, 3, seed=6, dev=dev)
        rec["parity_2p5M_nodes"] = {"strict_eps0": sharded_vs_single("SimGCL", mid, d, 2, B, mb, steps=2, dev=dev, **dict(kw, eps=0.0)),
                                    "configured": sharded_vs_single("SimGCL", mid, d, 2, B, mb, steps=2, dev=dev, **kw)}
    except Exception as e:  # noqa: BLE001
        rec["parity_2p5M_nodes"] = {"error": f"{type(e).__name__}: {e}"}
    return rec


# ------------------------------------------------------------------------------------------
# our arm, N = 1
# ------------------------------------------------------------------------------------------
def run_single(args, local_rank):
    import random
    import torch
    from selfrec_b200 import _lib, build, ops
    build.build()
    _lib.require_device()  # fails loudly without a GPU / without the library
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from selfrec_b200.engine import TrainEngine

    data = build_data()
    random.seed(1234)
    torch.manual_seed(1234)
    eng = TrainEngine("XSimGCL", data, CFG["d"], CFG["L"], CFG["B"], CFG["lr"], CFG["reg"], device=dev, philox_seed=2026, **xs_kwargs())
    P = 64

    def batch_stream():  # epochs back to back: a long --steps run must not end with the first epoch
        while True:
            yield from eng.batches()

    pool_host = np.stack([w.copy() for _, w in zip(range(P), eng.batches())])
    pool = torch.from_numpy(pool_host).to(dev)

    if args.profile:
        # ncu mode: eager launches only (every kernel individually visible), no baselines
        gen = batch_stream()
        for _ in range(args.warmup + args.steps):
            eng.step(next(gen))
        ue, ie = eng.forward_clean()
        rp, ri = data.rated_csr()
        ops.score_topk(ue, ie, torch.arange(eng.U, device=dev, dtype=torch.int32), torch.from_numpy(rp).to(dev),
                       torch.from_numpy(ri).to(dev), 20)
        torch.cuda.synchronize()
        emit({"profile_mode": True, "launches": _lib.launch_count()})
        return

    eng.batch_dev.copy_(pool[0])
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    eng.step_resident()
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - l0
    graph = eng.capture()

    def resident_step(k):
        eng.batch_dev.copy_(pool[k % P], non_blocking=True)  # D2D, 41 KB
        graph.replay()

    W = max(args.warmup, 3)
    clocks = ClockSampler(local_rank)
    for k in range(W):
        resident_step(k)
    clocks.start()
    ms = time_steps(resident_step, args.steps, 0, torch)
    outputs = None
    if args.dump_outputs:  # the last timed step's results, taken before keep_load steps on
        outputs = {"user_emb": eng.user_emb.cpu().numpy(), "item_emb": eng.item_emb.cpu().numpy(), "losses": eng.losses.cpu().numpy()}
    keep_load(resident_step, ms / args.steps, torch)  # nvidia-smi needs ~0.4 s of this same load to see it
    clk = clocks.stop()
    clk["window"] = "timed region + 0.4 s of the same graph-replay loop (keep_load)"
    value = args.steps / (ms * 1e-3)

    # same loop with an L2 flush between iterations, per-step events (extra evidence)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev, dtype=torch.float32)
    per = []
    for k in range(min(args.steps, 20)):
        flush.fill_(float(k))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        resident_step(k)
        e1.record()
        torch.cuda.synchronize()
        per.append(e0.elapsed_time(e1))
    ms_flushed = float(np.mean(per))
    del flush

    # ---- e2e: public API, host buffers, H2D + D2H every step ----
    gen = batch_stream()
    for _ in range(W):
        eng.step(next(gen), fetch_loss=True).get()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pending = None
    for _ in range(args.steps):
        h = eng.step(next(gen), fetch_loss=True)
        if pending is not None:
            loss_host = pending.get()  # D2H read of the previous step's result
        pending = h
    loss_host = pending.get()
    torch.cuda.synchronize()
    e2e_val = args.steps / (time.perf_counter() - t0)

    # ---- roofline of the dominant kernel (SpMM), live CUDA-event timing ----
    pk = peaks()
    N, nnzA = eng.N, eng.adj._nnz()
    x = torch.randn(N, CFG["d"], device=dev)
    y = torch.empty_like(x)
    for _ in range(3):
        ops._spmm_raw(eng.adj, x, y)
    R = 50
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(R):
        ops._spmm_raw(eng.adj, x, y)
        ops._spmm_raw(eng.adj, y, x)
    e1.record()
    torch.cuda.synchronize()
    spmm_ms = e0.elapsed_time(e1) / (2 * R)
    alg = spmm_bytes(N, nnzA, CFG["d"])
    achieved = alg / (spmm_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, TRAFFIC_FILE)
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f).get("yelp2018")
    sbytes = step_bytes("XSimGCL", N, nnzA, CFG["d"], CFG["L"])

    # ---- rank metric, on TRAINED tables (two epochs through the public API) ----
    n_train = 0
    for _ep in range(2):
        for w in eng.batches():
            eng.step(w)
            n_train += 1
    ue, ie = eng.forward_clean()
    rp, ri = data.rated_csr()
    users = torch.arange(eng.U, device=dev, dtype=torch.int32)
    rpd, rid = torch.from_numpy(rp).to(dev), torch.from_numpy(ri).to(dev)
    rank = {}
    fb_users = None
    for impl, tag in ((2, "tcgen05 tf32 candidates + exact fp32 rescoring"), (1, "cuda-core fp32")):
        ops.score_topk(ue, ie, users, rpd, rid, 20, impl=impl)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            ids_k, _sc = ops.score_topk(ue, ie, users, rpd, rid, 20, impl=impl)
        e1.record()
        torch.cuda.synchronize()
        rank[impl] = (e0.elapsed_time(e1) / 5, tag, ids_k)
        if impl == 2:
            st = {}
            ops.score_topk(ue, ie, users, rpd, rid, 20, impl=2, stats=st)
            fb_users = int(st["fallback_count"].item())
    assert torch.equal(rank[1][2], rank[2][2]), "tensor-core ranking differs from the exact kernel"
    rank_ms = rank[2][0]
    rank_val = eng.U * eng.I / (rank_ms * 1e-3)
    tf32_peak = pk["bf16_tflops"] / 2.0  # dense TF32 = half the measured bf16 rate of the same tensor pipe
    rank_tf = 2.0 * eng.U * eng.I * CFG["d"] / (rank_ms * 1e-3) / 1e12

    cpu = cpu_baseline(data) if not args.skip_cpu else None
    line = {
        "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": 1, "steps": args.steps, "warmup": W,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "parallelism": "single GPU (the N > 1 runs shard this same job: strong scaling)",
                   "l2": "no flush: per-step working set ~180 MB > 126 MB L2 (see value_l2_flushed)",
                   "inputs": f"{P} pre-sampled batches resident in HBM, CUDA-graph replay"},
        "clocks": clk,
        "e2e": {"value": e2e_val, "unit": "steps/s", "h2d_bytes_per_step": int(eng.words * 4), "d2h_bytes_per_step": 16,
                "note": "native sampler + pinned H2D + fused step + loss D2H each step"},
        "gpu_launches": int(launches_per_step * args.steps), "launches_per_step": int(launches_per_step),
        "value_l2_flushed": 1e3 / ms_flushed, "ms_per_step_l2_flushed": ms_flushed,
        "roofline": {"bound": "hbm", "kernel": "spmm_csr_kernel<64>", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "traffic_source": TRAFFIC_FILE if traffic else None,
                     "peak_source": pk["source"], "ms_per_launch": spmm_ms, "algorithmic_bytes_per_launch": alg,
                     # what actually bounds this kernel at yelp2018 size: X is L2-resident and every non-zero gathers one
                     # 256-byte row out of L2 (ceiling measured by tools/l2_microbench.cu, profiles/r01a_l2_gather_microbench.txt)
                     "l2_gather": {"bytes_per_launch": 4 * nnzA * CFG["d"], "achieved": 4 * nnzA * CFG["d"] / (spmm_ms * 1e-3) / 1e9,
                                   "peak": 18500.0, "unit": "GB/s", "frac": 4 * nnzA * CFG["d"] / (spmm_ms * 1e-3) / 1e9 / 18500.0,
                                   "peak_source": "measured random 256 B row gathers from an L2-resident table, 148 SMs"},
                     "step": {"algorithmic_bytes": sbytes, "achieved": sbytes / (ms / args.steps * 1e-3) / 1e9,
                              "frac": sbytes / (ms / args.steps * 1e-3) / 1e9 / pk["hbm_gbs"]}},
        "rank": {"metric": "full-catalog rank items/sec", "value": rank_val, "unit": "items/s", "ms": rank_ms,
                 "users": eng.U, "items": eng.I, "k": 20, "impl": rank[2][1], "ids_equal_to_exact_kernel": True,
                 "tables": f"trained: {n_train} steps (2 epochs) through the public API",
                 "users_rerun_by_exact_fallback": fb_users,
                 "cuda_core_ms": rank[1][0], "cuda_core_items_per_s": eng.U * eng.I / (rank[1][0] * 1e-3),
                 "roofline": {"bound": "tensor", "achieved": rank_tf, "peak": tf32_peak, "unit": "TFLOP/s", "frac": rank_tf / tf32_peak,
                              "peak_source": f"bf16_tflops / 2, {pk['source']}",
                              "note": "single-pass TF32 MMA; includes gather, rescoring and fallback launches"}},
        "cpu_baseline": cpu,
        "loss": [float(v) for v in loss_host.tolist()],
    }
    del eng, graph, pool
    torch.cuda.empty_cache()
    if not args.skip_configs:
        for name, fn in (("config2", lambda: record_config2(args, dev, data)), ("config4", lambda: record_config4(args, dev)),
                         ("config5", lambda: record_config5(args, dev, 1, 0, None))):
            t0 = time.perf_counter()
            try:
                line[name] = fn()
            except Exception as e:  # noqa: BLE001 -- a sub-record must not take the headline down with it
                line[name] = {"error": f"{type(e).__name__}: {e}"}
            line[name]["wall_s"] = time.perf_counter() - t0
            torch.cuda.empty_cache()
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    emit(line)


# ------------------------------------------------------------------------------------------
# our arm, N > 1: the same job, bipartite-sharded
# ------------------------------------------------------------------------------------------
def run_sharded(args, rank, world, local_rank):
    import random
    import torch
    import torch.distributed as dist
    from selfrec_b200 import _lib, build
    build.build()
    _lib.require_device()
    dev = torch.device("cuda", local_rank)
    from selfrec_b200.shard_check import sharded_vs_single
    from selfrec_b200.sharded import ShardedEngine
    from selfrec_b200.util.sampler import NativePairSampler
    data = build_data()
    B, d, L = CFG["B"], CFG["d"], CFG["L"]
    random.seed(1234)  # identical batches on every rank
    smp = NativePairSampler(data)
    smp.pull_state()
    smp.begin_epoch(want_perm=False)
    pool_host = smp.epoch(B, B)[:64].copy()
    smp.push_state()
    pool = torch.from_numpy(pool_host).to(dev)
    P = pool_host.shape[0]

    # ---- self-verification before anything is timed: sharded step == single-GPU engine, on both peer-store routes ----
    # "strict": eps = 0 -- every compared quantity (losses, Adam moments, clean forward) within 1e-4.
    # "configured": eps = 0.2 -- sign(y) * noise * eps is discontinuous at y = 0, so an element within fp32 rounding of
    # zero flips under the sharded summation order; the losses agree to 1e-4, `m_rows_off_frac` says how few rows differ.
    parity = {}
    for route, mc in (("unicast", False), ("multicast", True)):
        for tag, kw in (("strict_eps0", dict(xs_kwargs(), eps=0.0)), ("configured", xs_kwargs())):
            try:
                r = sharded_vs_single("XSimGCL", data, d, L, B, pool, steps=3, dev=dev, multicast=mc, **kw)
                keep = ("max_rel", "loss_rel", "m_user_rel", "m_item_rel", "final_user_rel", "final_item_rel", "m_rows_off_frac", "route", "steps")
                parity[f"{route}_{tag}"] = {k: r[k] for k in keep}
            except Exception as e:  # noqa: BLE001
                parity[f"{route}_{tag}"] = {"error": f"{type(e).__name__}: {e}"}
    parity_max = max([v.get("max_rel", float("inf")) for k, v in parity.items() if k.endswith("strict_eps0")])

    sh = ShardedEngine("XSimGCL", data, d, L, B, CFG["lr"], CFG["reg"], device=dev, philox_seed=2026, **xs_kwargs())
    l0 = _lib.launch_count()
    sh.step(words_dev=pool[0])
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - l0
    sh.capture()

    def resident_step(k):
        sh.batch_dev.copy_(pool[k % P], non_blocking=True)
        sh.step_resident()

    W = max(args.warmup, 3)
    for k in range(W):
        resident_step(k)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms = time_steps(resident_step, args.steps, 0, torch, dist)
    keep_load(resident_step, ms / args.steps, torch)  # (ms is the max over ranks: every rank runs the same number of steps)
    clk = clocks.stop() if rank == 0 else None
    if clk is not None:
        clk["window"] = "timed region + 0.4 s of the same graph-replay loop (keep_load)"
    value = args.steps / (ms * 1e-3)

    # ---- e2e: the N = 1 measurement -- native sampler inside the loop, pinned H2D, lagged pinned loss reads ----
    random.seed(4321)
    smp2 = NativePairSampler(data)
    pins = [torch.zeros(sh.words, dtype=torch.int32).pin_memory() for _ in range(8)]
    lpins = [torch.zeros(4).pin_memory() for _ in range(8)]
    evs, levs = [None] * 8, [None] * 8
    buf = np.empty(sh.words, dtype=np.int32)

    def stream():
        while True:
            smp2.pull_state()
            smp2.begin_epoch(want_perm=False)
            while smp2.next_batch(B, B, buf) > 0:
                yield buf
            smp2.push_state()

    gen = stream()

    def e2e_step(k):
        s = k % 8
        if evs[s] is not None:
            evs[s].synchronize()
        pins[s].numpy()[:] = next(gen)
        sh.batch_dev.copy_(pins[s], non_blocking=True)
        evs[s] = torch.cuda.Event()
        evs[s].record()
        sh.step_resident()
        lpins[s].copy_(sh.losses, non_blocking=True)
        levs[s] = torch.cuda.Event()
        levs[s].record()
        if k > 0:  # read the previous step's losses while this one runs
            levs[(k - 1) % 8].synchronize()
            return lpins[(k - 1) % 8].numpy().copy()
        return None

    for k in range(W):
        e2e_step(k)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        loss_host = e2e_step(W + k)
    torch.cuda.synchronize()
    te = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = args.steps / float(te.item())
    sh.check_peers()
    loss_now = sh.losses.cpu().tolist()
    nv_layer = sh.nvlink_bytes_per_layer()
    route = "one NVSwitch-multicast store per finished row" if sh.use_multicast else "one P2P store per finished row and peer"
    N, nnzA = sh.N, sh.nnzA
    del sh
    torch.cuda.empty_cache()
    c5 = None
    if not args.skip_configs:
        t0 = time.perf_counter()
        try:
            c5 = record_config5(args, dev, world, rank, dist)
        except Exception as e:  # noqa: BLE001
            c5 = {"error": f"{type(e).__name__}: {e}"}
        c5["wall_s"] = time.perf_counter() - t0
    if rank != 0:
        return
    pk = peaks()
    sbytes = step_bytes("XSimGCL", N, nnzA, d, L)
    line = {
        "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": W,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "parallelism": f"bipartite-sharded x{world}: users dealt cyclically (u % world; their rows never leave the GPU), item tables replicated; per layer the "
                                  f"item-side SpMM epilogue stores partial rows into the slice owner's staging area (P2P, reduce-scatter), the owner sums, "
                                  f"applies the epilogue and stores the finished rows to every rank ({route}), beside the user-side product; 2 synchronisations per "
                                  "layer folded into the kernels; last forward layer on the batch rows only; batch losses replicated on a compact [5B, d] "
                                  "table; one srb_shard_step call per step, captured in a CUDA graph",
                   "l2": "no flush: per-step working set > 126 MB L2",
                   "inputs": f"{P} pre-sampled batches resident in HBM on every rank; CUDA-graph replay"},
        "clocks": clk,
        "parity": parity, "parity_max_rel": parity_max, "parity_note": "parity_max_rel = the strict (eps = 0) runs; see bench.py run_sharded",
        "e2e": {"value": e2e_val, "unit": "steps/s", "h2d_bytes_per_step": int(pool_host.shape[1] * 4), "d2h_bytes_per_step": 16,
                "note": "every rank: native sampler (same seed) + pinned H2D + sharded step + loss D2H, read one step late"},
        "gpu_launches": int(launches_per_step * args.steps), "launches_per_step": int(launches_per_step),
        "roofline": {"bound": "hbm", "kernel": "spmm_csr_kernel<64> (sharded blocks)", "achieved": None, "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": None, "traffic": None, "peak_source": pk["source"],
                     "step": {"algorithmic_bytes": sbytes, "achieved": sbytes / (ms / args.steps * 1e-3) / 1e9,
                              "frac": sbytes / (ms / args.steps * 1e-3) / 1e9 / (pk["hbm_gbs"] * world)},
                     "nvlink_bytes_out_per_step_per_rank": int(nv_layer * 2 * L)},
        "cpu_baseline": None,
        "config5": c5,
        "loss": loss_now,
    }
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--profile", action="store_true", help="eager steps only, for ncu (never a bench value)")
    ap.add_argument("--skip-configs", action="store_true", help="headline metric only (no config2/4/5 sub-records)")
    ap.add_argument("--skip-cpu", action="store_true", help="no cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's parameters and losses as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "ours" or args.profile or world > 1):
        ap.error("--dump-outputs covers the single-process timed path (--impl ours, one GPU, no --profile)")
    claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        try:
            run_sharded(args, rank, world, local_rank)
        finally:
            dist.destroy_process_group()
    else:
        run_single(args, local_rank)


if __name__ == "__main__":
    main()
