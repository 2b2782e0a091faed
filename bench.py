#!/usr/bin/env python
"""Benchmark of the FIRA hot path: commits/s of one TRAINING step (forward + backward + Adam) on
synthetic commits that follow the DataSet's node/edge distribution (BASELINE.json metric, config
"run_model.py train, 1xB200, batch 64"; N GPUs -> global batch 64*N, weak scaling).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --steps K --warmup W    # reference algorithm on the host CPU cores

Prints ONE JSON line (rank 0).  `value` is device-timed with inputs resident in HBM; `e2e` is the
same step through the public TransModel.forward API with pinned HOST buffers (H2D of the batch and a
D2H read of the loss inside the timed region).  `roofline` is the GNN scatter kernel
(fira_gcn_aggregate) timed live with CUDA events against the measured HBM peak; `cpu_baseline` is
the CPU oracle port (oracle/fira_oracle.py, the reference algorithm as the reference executes it)
timed on this box's host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PER_GPU_BATCH = 64
VOCAB, AST_VOCAB = 24650, 71
N_POOL = 4                      # distinct synthetic batches rotated through the timed region
WORKLOAD = ("run_model.py train, 1xB200 per-GPU batch 64 (BASELINE.json configs[1]), "
            "synthetic commits with the DataSet node/edge distribution")


class DotDict(dict):
    def __getattr__(self, k):
        return self[k]


def model_args():
    return DotDict(sou_len=210, tar_len=30, att_len=25, ast_change_len=280, sub_token_len=160, lr=1e-4,
                   dropout_rate=0.1, num_head=8, embedding_dim=256, vocab_size=VOCAB,
                   ast_change_vocab_size=AST_VOCAB)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 2 + j and r[2 + j].startswith("Active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ data
def host_batch(first_index, batch_size, pin, trim=False):
    """One collated synthetic batch on the host: int64 id tensors + packed CSR (what a loader delivers).
    trim=True: the loader also drops the padding the whole batch shares (data.trim_batch_host)."""
    import torch
    from fira_icse_b200.data import trim_batch_host
    from fira_icse_b200.graph import PackedEdges
    from fira_icse_b200.synth import N_NODES, synth_batch
    ids, coo = synth_batch(first_index, batch_size, VOCAB, AST_VOCAB)
    t = {k: torch.from_numpy(v) for k, v in ids.items()}
    t["attr"] = torch.zeros(batch_size, 1, dtype=torch.int64)    # accepted and ignored by the model (Model.py:38)
    rowptr, col, val = PackedEdges.pack_host(coo, N_NODES, pin=False)
    if trim:
        lst = trim_batch_host([t["sou"], t["tar"], t["attr"], t["mark"], t["ast_change"], (rowptr, col, val),
                               t["tar_label"], t["sub_token"]], VOCAB)
        t = dict(zip(("sou", "tar", "attr", "mark", "ast_change", "_", "tar_label", "sub_token"), lst))
        rowptr, col, val = t.pop("_")
    if pin:
        t = {k: v.pin_memory() for k, v in t.items()}
        rowptr, col, val = rowptr.pin_memory(), col.pin_memory(), val.pin_memory()
    return t, (rowptr, col, val), coo


def device_batch(hb, dev, B):
    import torch
    from fira_icse_b200.graph import PackedEdges
    from fira_icse_b200.synth import N_NODES
    t, (rowptr, col, val), _ = hb
    d = {k: v.to(dev, non_blocking=True) for k, v in t.items()}
    n_nodes = t["sou"].shape[1] + t["sub_token"].shape[1] + t["ast_change"].shape[1]
    edges = PackedEdges.from_host(rowptr, col, val, B, n_nodes, dev)
    return [d["sou"], d["tar"], d["attr"], d["mark"], d["ast_change"], edges, d["tar_label"], d["sub_token"]]


def h2d_bytes(hb):
    t, csr, _ = hb
    return sum(v.numel() * v.element_size() for v in t.values()) + sum(v.numel() * v.element_size() for v in csr)


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_threads():
    """Host threads this process may really use: affinity mask, capped by a cgroup CPU quota if any."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def ref_worker(*argv, timeout=1500):
    """oracle/ref_cpu_bench.py in a subprocess with CUDA_VISIBLE_DEVICES="" (the reference branches on
    torch.cuda.is_available() globally, BASELINE.md section 2): the UNMODIFIED reference TransModel + Adam
    (oracle/_ref, staged by oracle/make_ref.sh) on this box's host cores.  -> parsed JSON line."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_cpu_bench.py"), *map(str, argv)],
                       env=env, capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError("reference CPU worker failed: " + r.stderr[-2000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def best_cpu_threads(limit):
    """torch CPU ops on a 100+ core host run SLOWER with every core (thread wake-up cost on 256-wide tensors):
    time one reference forward at a few thread counts and keep the fastest, so the CPU arm is the best the box's
    cores can do, not a strawman."""
    cands = sorted({c for c in (4, 8, 16, 32, 64, limit) if c <= limit})
    out = ref_worker("--calibrate", ",".join(map(str, cands)))
    return int(out["best_threads"]), out["calibration_s"]


REF_IMPL_TEXT = {
    "reference": "UNMODIFIED reference TransModel (oracle/_ref/{Model,gnn_transformer,combination_layer}.py, staged by "
                 "oracle/make_ref.sh) + torch.optim.Adam, fp32, dense float64 [64,650,650] adjacency, dropout on, "
                 "run_model.py:101-109 loop body, CUDA_VISIBLE_DEVICES='' subprocess",
    "port": "oracle port (oracle/fira_oracle.py; oracle/_ref was not staged on this box)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    avail = cpu_threads()
    threads, calib = best_cpu_threads(avail)
    out = ref_worker("--batch", PER_GPU_BATCH, "--steps", args.steps, "--warmup", args.warmup, "--threads", threads,
                     timeout=3000)
    dt = out["total_s"]
    value = PER_GPU_BATCH * args.steps / dt
    line = {"impl": "reference", "metric": "train_commits_per_sec", "value": value, "unit": "commits/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "per_gpu_batch": PER_GPU_BATCH, "global_batch": PER_GPU_BATCH,
                       "parallelism": "cpu",
                       "implementation": REF_IMPL_TEXT[out["impl"]],
                       "sample": f"each timed step = one full {PER_GPU_BATCH}-commit batch of the same synthetic stream"},
            "cpu_baseline": {"value": value, "unit": "commits/s", "cores": threads, "kind": out["impl"],
                             "cores_available": avail, "thread_calibration_s": calib,
                             "sample": f"{args.steps} training steps of {PER_GPU_BATCH} commits after {args.warmup} warm-up"},
            "e2e": {"value": value, "unit": "commits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "last_loss": out.get("last_loss")}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ roofline
def time_launches(launch, n_rot, reps=None, iters=12):
    """Average device time of ONE launch of a kernel, measured live: `reps` launches over `n_rot` rotating buffer sets
    (total > L2, so every launch finds its operands in HBM) are captured into one CUDA graph -- the way the training step
    issues them -- and the graph is replayed `iters` times between CUDA events recorded on the replay stream.  Launching
    one kernel at a time from Python would time the host's launch latency instead (the kernels here run 5-40 us)."""
    import torch
    reps = reps or max(8, n_rot)
    reps = (reps + n_rot - 1) // n_rot * n_rot
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(n_rot):
            launch(i)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(reps):
            launch(i)
    g.replay()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    torch.cuda.synchronize()
    for a, b in ev:
        a.record()
        g.replay()
        b.record()
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) / reps for a, b in ev)
    return sum(ms) / len(ms), ms[len(ms) // 2], reps * iters


def _cur():
    import torch
    return torch.cuda.current_stream().cuda_stream


TIMING_NOTE = "launches replayed from one CUDA graph over rotating buffer sets, CUDA events around the replay"


def spmm_roofline(dev, hb, B, bf16=False, label=None):
    """fira_gcn_aggregate (the stand-alone GNN scatter) on the padded 650-row graphs of `hb` (B commits), cold L2."""
    import torch
    from fira_icse_b200 import _lib
    from fira_icse_b200.graph import PackedEdges
    from fira_icse_b200.synth import N_CODE, N_SUB, N_AST, N_NODES
    _, (rowptr, col, val), _ = hb
    pe = PackedEdges.from_host(rowptr, col, val, B, N_NODES, dev)
    R = B * N_NODES
    tdt, esz, code = (torch.bfloat16, 2, 1) if bf16 else (torch.float32, 4, 0)
    n_pairs = max(3, int(400e6 // (2 * R * 256 * esz)) + 1)
    xs = [torch.randn(R, 256, device=dev).to(tdt) for _ in range(n_pairs)]
    ys = [torch.empty(R, 256, device=dev, dtype=tdt) for _ in range(n_pairs)]

    def launch(i):
        _lib.call("fira_gcn_aggregate", pe.rowptr.data_ptr(), pe.col.data_ptr(), pe.val.data_ptr(),
                  xs[i % n_pairs].data_ptr(), None, ys[i % n_pairs].data_ptr(), B, N_CODE, N_SUB, N_AST, 256, code, _cur())
    avg_ms, med_ms, n = time_launches(launch, n_pairs)
    alg_bytes = 2 * R * 256 * esz + (R + 1) * 4 + pe.nnz * 8        # SURVEY.md section 8d formula
    peak, how = measured_peaks()
    achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath) and B == PER_GPU_BATCH:   # dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu)
        traffic = json.load(open(tpath)).get("fira_gcn_aggregate_bf16_dram_bytes_per_launch" if bf16 else
                                             "fira_gcn_aggregate_dram_bytes_per_launch")
    kname = "csr_spmm_part_kernel<bf16,16>" if bf16 else "csr_spmm_kernel<float>"
    del xs, ys
    return {"bound": "hbm", "kernel": kname + " (fira_gcn_aggregate, the GNN scatter)", "achieved": achieved,
            "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_ms, "median_launch_ms": med_ms,
            "launches_timed": n, "rows": R, "nnz": pe.nnz, "commits": B, "peak_source": how,
            "dtype": "bf16" if bf16 else "f32", "shape": label or f"{B} commits x 650 padded node rows",
            "timing": TIMING_NOTE,
            "l2": f"cold: {n_pairs} rotating buffer pairs ({n_pairs * 2 * R * 256 * esz / 1e6:.0f} MB > 126 MB L2)"}


def spmm_packed_roofline(dev, pb):
    """The same kernel on the rows the TIMED STEP launches it on: the per-commit packed node rows of one bench batch
    (B = 1 ragged graph).  ~11 k rows = 12 MB: far too small for the HBM roofline to be the bound (launch + latency)."""
    import torch
    from fira_icse_b200 import _lib
    R = pb.rows
    n_pairs = max(3, int(400e6 // (2 * R * 256 * 2)) + 1)
    xs = [torch.randn(R, 256, device=dev).to(torch.bfloat16) for _ in range(n_pairs)]
    ys = [torch.empty(R, 256, device=dev, dtype=torch.bfloat16) for _ in range(n_pairs)]

    def launch(i):
        _lib.call("fira_gcn_aggregate", pb.rowptr.data_ptr(), pb.col.data_ptr(), pb.val.data_ptr(),
                  xs[i % n_pairs].data_ptr(), None, ys[i % n_pairs].data_ptr(), 1, pb.Rc, pb.Rs, pb.Ra, 256, 1, _cur())
    avg_ms, med_ms, n = time_launches(launch, n_pairs, reps=2 * n_pairs)
    nnz = int(pb.nnz)
    alg_bytes = 2 * R * 256 * 2 + (R + 1) * 4 + nnz * 8
    peak, how = measured_peaks()
    achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "csr_spmm_part_kernel<bf16,16> (fira_gcn_aggregate) on the packed rows of the timed step",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
            "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_ms, "median_launch_ms": med_ms,
            "launches_timed": n, "rows": R, "nnz": nnz, "peak_source": how, "dtype": "bf16", "timing": TIMING_NOTE,
            "note": "12 MB per launch: a same-size device copy does not reach the HBM roofline either; latency-bound"}


# ------------------------------------------------------------------------------------------------ fused GCN roofline
def gcn_fused_roofline(dev, pb):
    """The fused GCN layer kernel (fira_gcn_layer_fwd: gather -> tcgen05 -> bias/rowsum/dropout/residual/LayerNorm out of
    TMEM, ONE launch) on the node rows / adjacency of a packed bench batch `pb` (device), cold L2.  Algorithmic bytes =
    SURVEY.md 8d's fused formula: read H once + write the layer output once + rowptr + (col, val) + the weight once per
    launch; the kernel also writes Z (the pre-LayerNorm rows the backward needs) -- reported separately."""
    import torch
    from fira_icse_b200 import _lib
    R, Mc = pb.rows, pb.Rc
    n_sets = max(3, int(400e6 // (3 * R * 256 * 2)) + 1)
    bf = torch.bfloat16
    hs = [torch.randn(R, 256, device=dev).to(bf) for _ in range(n_sets)]
    zs = [torch.empty(R, 256, device=dev, dtype=bf) for _ in range(n_sets)]
    oa = [torch.empty(Mc, 256, device=dev, dtype=bf) for _ in range(n_sets)]
    ob = [torch.empty(R, 256, device=dev, dtype=bf) for _ in range(n_sets)]
    W = (torch.randn(256, 256, device=dev) / 16).to(bf)
    b2, c1 = torch.randn(256, device=dev) * 0.1, torch.randn(256, device=dev) * 0.1
    gamma, beta = torch.ones(256, device=dev), torch.zeros(256, device=dev)
    stats = torch.empty(2, R, device=dev)

    def launch(i):
        k = i % n_sets
        _lib.call("fira_gcn_layer_fwd", pb.rowptr.data_ptr(), pb.col.data_ptr(), pb.val.data_ptr(), hs[k].data_ptr(),
                  W.data_ptr(), b2.data_ptr(), c1.data_ptr(), gamma.data_ptr(), beta.data_ptr(), zs[k].data_ptr(),
                  oa[k].data_ptr(), ob[k].data_ptr(), Mc, stats.data_ptr(), stats.data_ptr() + 4 * R, R, 256, 0.2, 1234, None,
                  2, _cur())
    avg_ms, med_ms, n = time_launches(launch, n_sets, reps=2 * n_sets)
    nnz = int(pb.nnz)
    alg_bytes = 2 * R * 256 * 2 + (R + 1) * 4 + nnz * 8 + 256 * 256 * 2
    peak, how = measured_peaks()
    achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("fira_gcn_layer_fwd_dram_bytes_per_launch")
    return {"bound": "hbm", "kernel": "gcn_fused_kernel<0> (fira_gcn_layer_fwd: gather -> tcgen05.mma -> LayerNorm epilogue)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "algorithmic_bytes_per_launch": alg_bytes, "bytes_incl_saved_z": alg_bytes + R * 256 * 2,
            "avg_launch_ms": avg_ms, "median_launch_ms": med_ms, "launches_timed": n, "rows": R, "nnz": nnz,
            "peak_source": how, "dtype": "bf16", "timing": TIMING_NOTE,
            "shape": "node rows / adjacency of one packed bench batch (per-commit packed layout)",
            "l2": f"cold: {n_sets} rotating buffer sets ({n_sets * 4 * R * 256 * 2 / 1e6:.0f} MB > 126 MB L2)"}


# ------------------------------------------------------------------------------------------------ GEMM roofline
def gemm_roofline(dev, M, N=256, K=256, what="GCN layer product of a padded batch"):
    """The kernel family with the largest share of the bf16 step is the tcgen05 GEMM: time one shape live (bf16 in /
    out, bias) on rotating buffers (> L2) and report it against BOTH measured peaks (N = K = 256: HBM-bound by
    arithmetic intensity)."""
    import torch
    from fira_icse_b200 import ops
    n_buf = max(3, int(400e6 // ((M * K + M * N) * 2)) + 1)
    xs = [torch.randn(M, K, device=dev).to(torch.bfloat16) for _ in range(n_buf)]
    ys = [torch.empty(M, N, device=dev, dtype=torch.bfloat16) for _ in range(n_buf)]
    W = torch.randn(N, K, device=dev).to(torch.bfloat16)
    bias = torch.randn(N, device=dev)

    def launch(i):
        ops.gemm_tc(xs[i % n_buf], K, 1, W, K, 1, ys[i % n_buf], N, M, N, K, bias=bias)
    avg, med, n = time_launches(launch, n_buf, reps=2 * n_buf)
    alg_bytes = (M * K + N * K + M * N) * 2 + N * 4
    flops = 2.0 * M * N * K
    hbm, how = measured_peaks()
    tf_peak = 1645.8
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        tf_peak = float(json.load(open(path)).get("bf16_tflops", tf_peak))
    gbs = alg_bytes / (avg * 1e-3) / 1e9
    tfs = flops / (avg * 1e-3) / 1e12
    del xs, ys
    return {"kernel": "gemm_tc_kernel (fira_gemm_bf16_tc): " + what, "shape": [M, N, K],
            "bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
            "achieved_tflops": tfs, "peak_tflops": tf_peak, "frac_tensor": tfs / tf_peak,
            "algorithmic_bytes_per_launch": alg_bytes, "flops_per_launch": flops, "avg_launch_ms": avg,
            "median_launch_ms": med, "launches_timed": n, "peak_source": how, "timing": TIMING_NOTE,
            "note": "arithmetic intensity 2*256/(2+2+~0) ~ 128 FLOP/B < ridge ~250: the HBM roofline applies"}


# ------------------------------------------------------------------------------------------------ outputs
DUMP_SAMPLE = 1 << 23           # parameter entries written by --dump-outputs (32 MB in float32)


def dump_outputs(out_dir, model, loss_sum, n_tokens):
    """What the timed step hands its caller, read after the last timed step: the loss sum and token count it returns
    (loss_sum.npy, n_tokens.npy, float64) and the parameters Adam left (parameters.npy, float32).  Written by rank 0.
    Through the CUDA-graph engine (the default) the loss sum and token count are rank 0's own, over its shard of the
    global batch; through the eager --no-graph step they are global: the step's mean loss times its global token
    count, and that count.  Compare dumps taken with the same flags and world size.  The parameters are
    concatenated in model.parameters() order and sampled at DUMP_SAMPLE sorted positions drawn by numpy's generator
    with seed 0 (torch's generator is left alone: it seeds the dropout of the legs that follow).  Atomic gradient
    reductions make two runs of one build differ in the last bits, and Adam's normalised update magnifies that on
    entries whose gradient is near zero: compare dumps with a tolerance."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    n = flat.numel()
    idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_SAMPLE), replace=False)))
    arrays = {"loss_sum": loss_sum.double(), "n_tokens": n_tokens.double(),
              "parameters": flat[idx.to(flat.device)].float()}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------------ GPU arm
def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this framework has no CPU path "
                         "(use --impl reference for the CPU reference arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    import fira_icse_b200 as F
    from fira_icse_b200 import _lib
    from fira_icse_b200.engine import GraphedTrainStep
    from fira_icse_b200.parallel import DataParallelStep

    B = PER_GPU_BATCH

    def adam_factory(m):
        # Adam lr 1e-4 (run_model.py:60,101-109): the library's flat Adam (optim.FlatAdam, one launch per step) unless
        # FIRA_TORCH_ADAM=1 asks for torch.optim.Adam(fused=True) as the A/B
        if os.environ.get("FIRA_TORCH_ADAM", "0") != "0":
            return lambda ps: torch.optim.Adam(ps, lr=1e-4, fused=True, capturable=True)
        return lambda ps: F.FlatAdam(ps, lr=1e-4, groups=m.flat_groups())
    torch.manual_seed(0)
    model = F.TransModel(model_args()).to(dev)
    model.train()
    model.set_precision(args.precision)

    # every rank gets its own shard of the synthetic stream (graphs shard by commit, no data collective)
    packed = args.layout == "packed"
    full_host = host_batch(rank * N_POOL * B, B, pin=True, trim=False)
    if packed:
        # per-commit packed batches (fira_icse_b200/packed.py): node rows = the real nodes of every commit
        from fira_icse_b200.packed import PackedTables, pack_from_dataset
        from fira_icse_b200.synth import SynthDataset
        synth_ds = SynthDataset(rank * N_POOL * B, N_POOL * B, VOCAB, AST_VOCAB)
        synth_tables = PackedTables(synth_ds)
        import numpy as np
        pool_host = [pack_from_dataset(synth_tables, np.arange(i * B, (i + 1) * B), VOCAB, pin=True) for i in range(N_POOL)]
        pool_dev = [pb.to(dev) for pb in pool_host]
    else:
        pool_host = [host_batch((rank * N_POOL + i) * B, B, pin=True, trim=args.trim) for i in range(N_POOL)]
        pool_dev = [device_batch(hb, dev, B) for hb in pool_host]

    def host_list(hb):
        if packed:
            return hb
        t, csr, _ = hb
        return [t["sou"], t["tar"], None, t["mark"], t["ast_change"], csr, t["tar_label"], t["sub_token"]]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    last_loss = [0.0]
    last_step = [None]                  # what the last timed step returned, for --dump-outputs
    if args.graph:
        # whole step captured in a CUDA graph (fira_icse_b200/engine.py): one cudaGraphLaunch per step
        eng = GraphedTrainStep(model, B, adam_factory(model),
                               edge_capacity=(max(pb.nnz for pb in pool_host) + 4095) // 4096 * 4096 * 2 if packed else None)
        eng.load(pool_dev[0])
        eng.capture()                                                # one eager step + capture of this shape
        for hb in pool_dev[1:]:                                      # trimmed batches come in a few shapes:
            eng.step(hb)                                             # capture each shape's graph before timing
        eng.load(pool_dev[0])
        c0 = _lib.LAUNCH_COUNT
        eng._forward_backward(eng.cur)                               # count the C-ABI calls of one step (eager)
        launches_per_step = _lib.LAUNCH_COUNT - c0
        optimizer, bucket = eng.optimizer, eng.bucket

        def resident_step(i):
            last_step[0] = eng.step(pool_dev[i % N_POOL])            # (loss sum, token count)

        def e2e_step(i):
            eng.step(host_list(pool_host[i % N_POOL]))               # pinned host -> static device buffers -> replay
            last_loss[0] = (eng.loss_sum / eng.n_local).item()       # D2H read of the step's result
    else:
        if packed:
            raise SystemExit("bench.py: --layout packed runs through the graph engine (drop --no-graph)")
        dp = DataParallelStep(model, lambda ps: torch.optim.Adam(ps, lr=1e-4, fused=True))
        optimizer, bucket = dp.optimizer, dp.bucket
        launches_per_step = None

        def resident_step(i):
            last_step[0] = dp.step(pool_dev[i % N_POOL])             # (mean loss, token count)

        def e2e_step(i):
            loss, _ = dp.step(device_batch(pool_host[i % N_POOL], dev, B))
            last_loss[0] = loss.item()

    # ---- device-resident arm ("value")
    for i in range(args.warmup):
        resident_step(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.LAUNCH_COUNT
    ms = timed(resident_step, args.steps)
    launches = (_lib.LAUNCH_COUNT - launches0) if launches_per_step is None else launches_per_step * args.steps
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        loss, n_tok = last_step[0]
        dump_outputs(args.dump_outputs, model, loss if args.graph else loss * n_tok, n_tok)

    if args.timeline:
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(3):
                resident_step(i)
                torch.cuda.synchronize()
        if rank == 0:
            prof.export_chrome_trace(args.timeline)
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import timeline_summary as TS
            steps = TS.split_steps(TS.load(args.timeline), 3)
            with open(args.timeline + ".summary.txt", "w") as f:
                print(json.dumps({"value": value, "ms_per_step": ms / args.steps}), file=f)
                TS.summarize(steps[1], out=f)
            print(json.dumps({"timeline": args.timeline, "value": value, "ms_per_step": ms / args.steps}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    if args.profile_step:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        resident_step(0)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        if rank == 0:
            print(json.dumps({"profile_step": True, "value": value, "ms_per_step": ms / args.steps,
                              "launches_per_step": launches_per_step}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- end-to-end arm: pinned host batch -> H2D -> TransModel.forward -> backward -> Adam -> loss D2H
    for i in range(min(3, args.warmup)):
        e2e_step(i)
    ms_e2e = timed(e2e_step, args.steps)
    e2e_value = world * B * args.steps / (ms_e2e * 1e-3)

    # ---- the same, fed by the native loader: packed split arrays -> C++ gather/trim/CSR pack into pinned staging
    #      buffers on a background thread (data.PackedBatchLoader) -> H2D -> graph replay -> loss D2H
    loader_info = None
    if args.graph and (args.trim or packed):
        from fira_icse_b200.data import PackedBatchLoader
        from fira_icse_b200.synth import SynthDataset
        ds = SynthDataset(rank * N_POOL * B, N_POOL * B, VOCAB, AST_VOCAB)      # the commits of pool_host, in order
        import numpy as np
        laps = (args.steps + N_POOL) // N_POOL + 2                   # one long epoch cycling through the same batches
        ld = PackedBatchLoader(ds, B, VOCAB, shuffle=False, multiples=(8, 8, 8), prefetch=2, packed=packed,
                               indices=np.tile(np.arange(N_POOL * B), laps))
        stream_of_batches = iter(ld)

        def loader_step(i):
            eng.step(next(stream_of_batches))
            last_loss[0] = (eng.loss_sum / eng.n_local).item()
        for i in range(N_POOL):                                       # every shape the loader emits is captured
            loader_step(i)
        ms_ld = timed(loader_step, args.steps)
        loader_info = {"value": world * B * args.steps / (ms_ld * 1e-3), "unit": "commits/s",
                       "ms_per_step": ms_ld / args.steps,
                       "api": ("PackedBatchLoader(packed=True) (fira_host_gather_packed" if packed else
                               "PackedBatchLoader (fira_host_gather_batch") + ", pinned staging ring) -> GraphedTrainStep.step"}

    # ---- the reference-facing call with the reference's own input format: dense fp64 adjacency on the host
    dense_info = None
    if rank == 0 and world == 1:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import fira_oracle as O
        t, _, coo = full_host
        dense = torch.stack([O.dense_adjacency(r, c, v) for r, c, v in coo]).pin_memory()    # builds the INPUT only

        def dense_step(i):
            d = {k: v.to(dev, non_blocking=True) for k, v in t.items()}
            bucket.zero()
            loss_sum, n_tok = model(d["sou"], d["tar"], None, d["mark"], d["ast_change"],
                                    dense.to(dev, non_blocking=True), d["tar_label"], d["sub_token"], "train")
            loss = loss_sum / n_tok
            loss.backward()
            optimizer.step()
            last_loss[0] = loss.item()
        dense_step(0)
        k = min(args.steps, 5)
        ms_d = timed(dense_step, k)
        dense_info = {"value": B * k / (ms_d * 1e-3), "unit": "commits/s",
                      "h2d_bytes_per_step": int(dense.numel() * 8 + sum(v.numel() * 8 for v in t.values())),
                      "note": "eager (no CUDA graph); edge passed as the reference's dense float64 [B,650,650] host "
                              "tensor (Dataset.py:340)"}

    # ---- the fp32 parity mode (logits within 1e-4 of the reference) on the same batches: an extra key of the bf16 line
    parity_info = None
    if args.precision == "bf16" and args.graph and world == 1 and not args.skip_parity_mode:
        m32 = F.TransModel(model_args()).to(dev)
        m32.load_state_dict(model.state_dict())
        m32.train()
        m32.set_precision("fp32")
        eng32 = GraphedTrainStep(m32, B, adam_factory(m32),
                                 edge_capacity=eng.cap)
        for hb in pool_dev:
            eng32.step(hb)
        for hb in pool_dev:
            eng32.step(hb)
        k32 = max(4, min(10, args.steps))
        ms32 = timed(lambda i: eng32.step(pool_dev[i % N_POOL]), k32)
        parity_info = {"value": B * k32 / (ms32 * 1e-3), "unit": "commits/s", "ms_per_step": ms32 / k32, "steps": k32,
                       "precision_mode": "fp32 parity (fp32 storage, fp32 FFMA GEMMs): loss / logits within 1e-4 of the reference"}
        del eng32, m32
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rooflines (CUDA events, launches replayed from a graph over rotating > L2 buffers).  `roofline` = the GNN scatter
    # (the kernel BASELINE.json's metric names) on the 650-row padded graphs of one 64-commit batch; the same kernel on
    # the packed rows the timed step really launches it on, and on a batch large enough for HBM to be the bound (512
    # commits), sit next to it, with the fused GCN layer kernel, the fp32 scatter and the dominant GEMM shapes.
    roof = spmm_roofline(dev, full_host, B, bf16=args.precision == "bf16")
    extra = {}
    if args.precision == "bf16":
        torch.cuda.empty_cache()
        big = 8 * B
        extra["roofline_scatter_512_commits"] = spmm_roofline(dev, host_batch(0, big, pin=False, trim=False), big, bf16=True)
        torch.cuda.empty_cache()
        extra["roofline_scatter_fp32"] = spmm_roofline(dev, full_host, B, bf16=False)
        pb0 = pool_dev[0] if packed else None
        if pb0 is None:
            from fira_icse_b200.packed import PackedTables, pack_from_dataset
            from fira_icse_b200.synth import SynthDataset
            import numpy as np
            pb0 = pack_from_dataset(PackedTables(SynthDataset(rank * N_POOL * B, B, VOCAB, AST_VOCAB)), np.arange(B), VOCAB).to(dev)
        extra["roofline_scatter_step_shape"] = spmm_packed_roofline(dev, pb0)
        extra["roofline_gcn_fused"] = gcn_fused_roofline(dev, pb0)
        extra["roofline_gemm"] = gemm_roofline(dev, B * 650)
        extra["roofline_gemm_decoder"] = gemm_roofline(dev, B * 30, 256, 256, what="decoder projection of the timed step")
        torch.cuda.empty_cache()
        if os.environ.get("FIRA_GCN_FUSED", "0") != "0":
            # the GNN message passing of the timed step IS the fused kernel: it is the headline roofline then
            roof, extra["roofline_scatter_bf16"] = extra["roofline_gcn_fused"], roof

    # ---- CPU baseline on this box's host cores: the unmodified reference, same batch (bounded sample)
    cpu_info = None
    if not args.skip_cpu_baseline and world == 1:          # reported at N = 1 only (rank 0 is the only rank left here)
        avail = cpu_threads()
        threads, calib = best_cpu_threads(avail)
        out = ref_worker("--batch", B, "--steps", 3, "--warmup", 1, "--threads", threads)
        cpu_info = {"value": B * len(out["step_s"]) / out["total_s"], "unit": "commits/s", "cores": threads,
                    "kind": out["impl"], "cores_available": avail, "thread_calibration_s": calib,
                    "sample": f"{len(out['step_s'])} training steps of {B} commits after 1 warm-up: "
                              + REF_IMPL_TEXT[out["impl"]]}

    line = {"metric": "train_commits_per_sec", "value": value, "unit": "commits/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
                       "precision_mode": ("bf16 throughput (bf16 activations, tcgen05 GEMMs with fp32 TMEM accumulators, "
                                          "fp32 parameters/statistics/gradients)" if args.precision == "bf16" else
                                          "fp32 parity (fp32 storage, fp32 FFMA accumulate)"),
                       "optimizer": ("Adam lr 1e-4 (torch.optim.Adam fused)" if os.environ.get("FIRA_TORCH_ADAM", "0") != "0" else "Adam lr 1e-4 (fira_adam_flat: one launch over the flat parameter buffer)") + ", dropout on (0.1 / GCN 0.2)",
                       "launch": "whole step replayed as one CUDA graph" if args.graph else "eager launches",
                       "padding": ("per-commit packed batches: node rows = the real nodes of every commit (segments padded to "
                                   "1024/512/512-row buckets); loss and gradients equal the padded batch" if packed else
                                   "loader trims the padding the batch shares (code/sub-token/AST segments cut to the "
                                   "batch maximum, multiple of 8); real rows, loss and gradients unchanged"
                                   if args.trim else "full 210/160/280 padding"),
                       "batch_shapes": (sorted({pb.shape_key for pb in pool_host}) if packed else
                                        sorted({(hb[0]["sou"].shape[1], hb[0]["sub_token"].shape[1],
                                                 hb[0]["ast_change"].shape[1]) for hb in pool_host})),
                       "l2": f"{N_POOL} distinct batches rotated; one step touches >1 GB of activations (> 126 MB L2)"},
            "e2e": {"value": e2e_value, "unit": "commits/s",
                    "h2d_bytes_per_step": int(pool_host[0].h2d_bytes() if packed else h2d_bytes(pool_host[0])),
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                    "api": ("GraphedTrainStep.step(pinned host batch): H2D into the static buffers -> replay of the captured "
                            "TransModel." + ("forward_packed" if packed else "forward") + " + backward + Adam graph -> loss D2H"
                            if args.graph else "DataParallelStep.step: TransModel.forward eager + backward + Adam")},
            "e2e_loader": loader_info,
            "e2e_dense_edge": dense_info,
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, **extra,
            "fp32_parity_mode": parity_info,
            "cpu_baseline": cpu_info, "last_loss": last_loss[0]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("FIRA_PRECISION", "bf16"), choices=["bf16", "fp32"],
                    help="bf16 = BASELINE.json config (default); fp32 = parity mode")
    ap.add_argument("--layout", default=os.environ.get("FIRA_LAYOUT", "packed"), choices=["trimmed", "packed"],
                    help="trimmed = padded batches cut to the batch maximum; packed = per-commit packed node rows")
    ap.add_argument("--no-trim", dest="trim", action="store_false",
                    help="feed fully padded 210/160/280 batches instead of loader-trimmed ones")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="eager launches instead of the captured CUDA graph")
    ap.add_argument("--skip-parity-mode", action="store_true", help="leave out the fp32 parity-mode extra key")
    ap.add_argument("--skip-cpu-baseline", action="store_true",
                    help="profiling runs only (ncu): leave out the host-CPU leg")
    ap.add_argument("--timeline", default=None,
                    help="profiling runs only: after the timed region, 3 more steps under torch.profiler (CUPTI kernel "
                         "activity); writes the chrome trace to this path and its summary (tools/timeline_summary.py) "
                         "next to it, then exits")
    ap.add_argument("--profile-step", action="store_true",
                    help="profiling runs only (ncu --profile-from-start off): after the timed region, ONE more step "
                         "between cudaProfilerStart/Stop, then exit without the extra legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs) "
                         "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs writes what the last timed step computed: it needs --steps 1 or more")
    if not args.graph and args.layout == "packed":
        args.layout = "trimmed"                      # eager launches (profiling runs): the padded layout
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
