#!/usr/bin/env python
"""bench.py -- decode tokens/s for Llama-3.1-8B at P=98K, K=10, L=150 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W]                 # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W] # the reference's CPU path
    torchrun --nproc-per-node N ... bench.py --gpus N ...               # one rank per GPU
    python bench.py ... --dump-outputs DIR                              # + DIR/logits.npy of the last timed step

One "step" = one decode token for the whole batch through all 32 layers of a random-init
Llama-3.1-8B (library GEMMs for the projections/MLP; the 30 sparse layers run this repo's three
sm_100a kernels; the 2 dense layers run the same gather-attention kernel over the full context).
The context is synthetic (seeded random K/V pushed through the server's own fill()/build_table()).

The JSON line carries, besides the base contract:
  roofline     the dominant kernel (attend_kernel, the fused gather attention): algorithmic bytes
               per launch / CUDA-event duration per launch, against the measured HBM peak;
  cpu_baseline the reference's own CPU operators (oracle/_ref: lsh.batch_retrieve +
               sparse_attention_cpu.attention_wrapper, unmodified) timed on this box's host cores
               on a bounded sample (one sparse layer of the same shape), scaled to tokens/s;
  e2e          the same decode measured with host buffers: the token ids come from pinned host
               memory every step and the logits are read back to the host every step;
  hot_path     the sparse-attention path alone (30 layers x [SimHash | probe | attend]).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "decode tokens/sec Llama-3.1-8B @ P=98K, K10L150"
UNIT = "tokens/s"
PUBLISHED_B1 = 19.0  # BASELINE.md: reference end-to-end, B=1, 96K ctx, K10L150 on L20 + Xeon 8563C (read off a plot)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)   # examples/bench.py:14 (G=128)
    ap.add_argument("--warmup", type=int, default=32)   # examples/bench.py:28 (WARM_UP=32)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--B", type=int, default=1)
    ap.add_argument("--P", type=int, default=98000)
    ap.add_argument("--M", type=int, default=98304)
    ap.add_argument("--K", type=int, default=10)
    ap.add_argument("--L", type=int, default=150)
    ap.add_argument("--layers", type=int, default=0, help="debug: run fewer layers (result is then NOT the metric)")
    ap.add_argument("--parallel", default="dp", choices=["dp", "tp"],
                    help="dp: one independent replica per GPU (weak scaling, no data-path collective); "
                         "tp: KV-head tensor parallel cache + one all-gather of head outputs per layer (strong)")
    ap.add_argument("--model", default="8b", choices=["8b", "70b"], help="70b needs --parallel tp (weights + KV outgrow one GPU)")
    ap.add_argument("--tp-mode", default="megatron", choices=["ag", "megatron"],
                    help="ag: all-gather of head outputs, wo/MLP replicated (north-star); megatron: llama_dist.py:49-70 split, two all-reduces/layer")
    ap.add_argument("--tp-transport", default="peer", choices=["nccl", "peer"],
                    help="nccl collectives, or this repo's NVLink peer-memory exchange (csrc/peer.cu)")
    ap.add_argument("--no-tp-record", action="store_true", help="N > 1: skip the tensor-parallel variants measured after the replica run")
    ap.add_argument("--decode-impl", type=int, default=1, choices=[0, 1], help="1 = fused single-launch sparse layers (default), 0 = three launches (A/B measurements)")
    ap.add_argument("--dist", default="gauss", choices=["gauss", "clustered"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-worker", action="store_true", help="internal: time the reference in THIS process and print one JSON line")
    ap.add_argument("--ref-min-reps", type=int, default=3)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--profile-step", action="store_true",
                    help="bracket ONE extra decode step with cudaProfilerStart/Stop (for `ncu --profile-from-start off`)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the logits of the last timed decode step to DIR/logits.npy (float32, (B, vocab)), so that two builds "
                         "can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the decode step's logits: --impl ours only")
    return args


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])), mx.append(float(r[1]))
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def profiled_traffic(kernel_substr: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed
    `ncu --set full` capture (profiles/r2_dram_traffic_per_launch.json, written by scripts/summarize_ncu.py)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_dram_traffic_per_launch.json")) as f:
            for k, v in json.load(f).items():
                if kernel_substr in k:
                    return float(v)
    except Exception:
        pass
    return None


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# reference CPU path (oracle/_ref = the reference's own operators; else the C restatement)
# ------------------------------------------------------------------------------------------------
def host_info():
    """What decides how fast an OpenMP CPU path runs on this box: logical CPUs, physical cores, the affinity mask and cgroup
    CPU quota this process actually has, load."""
    info = {"logical_cpus": os.cpu_count(), "affinity_cpus": None, "physical_cores": None, "sockets": None, "cpu_model": None,
            "cgroup_cpu_max": None, "loadavg_1m": None}
    try:
        info["affinity_cpus"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    try:
        cores, model, phys, core = set(), None, None, None
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name") and model is None:
                    model = line.split(":", 1)[1].strip()
                elif line.startswith("physical id"):
                    phys = line.split(":", 1)[1].strip()
                elif line.startswith("core id"):
                    core = line.split(":", 1)[1].strip()
                elif not line.strip():
                    if phys is not None and core is not None:
                        cores.add((phys, core))
                    phys = core = None
        info["cpu_model"] = model
        if cores:
            info["physical_cores"] = len(cores)
            info["sockets"] = len({p for p, _ in cores})
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                info["cgroup_cpu_max"] = f.read().strip()
            break
        except Exception:
            pass
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except Exception:
        pass
    return info


def usable_cores(info) -> int:
    """Physical cores this process may actually use: min(physical cores, affinity mask, cgroup quota)."""
    n = info.get("physical_cores") or info.get("logical_cpus") or 1
    if info.get("affinity_cpus"):
        n = min(n, info["affinity_cpus"])
    q = info.get("cgroup_cpu_max")
    if q:
        parts = q.split()
        try:
            if parts[0] != "max" and int(parts[0]) > 0:
                period = int(parts[1]) if len(parts) > 1 else 100000
                n = min(n, max(1, int(parts[0]) // period))
        except Exception:
            pass
    return max(1, n)


def cpu_reference_layer(args, budget_s: float, min_reps: int = 3):
    """Times lsh.batch_retrieve + sparse_attention_cpu.attention_wrapper (unmodified reference,
    library/lsh/lsh.cc:210-241 + library/sparse_attention/sparse_attention.cc:629-745) on ONE sparse layer of
    the benchmark shape, on this host's cores, IN THIS PROCESS (whatever OpenMP environment it was started with).
    Returns dict(ms_layer, kind, cores, sample, nnz_frac)."""
    import torch
    from magicpig_b200 import synth
    from oracle import ref_loader
    import oracle

    B, Hq, Hkv, d, K, L = args.B, 32, 8, 128, args.K, args.L
    n, M = args.P - 68, args.M
    G = Hq // Hkv
    torch.manual_seed(0)
    hf = synth.make_hash_func(d, K, L, seed=0)
    q = synth.make_query(B, Hq, d, seed=1)
    key, value, kn, _ = synth.make_kv(B, Hkv, n, d, seed=2, dist=args.dist)
    # set-up only (not timed): key codes and their per-table sort; on the GPU when there is one (a 150-GFLOP GEMM and
    # 1200 sorts take ~40 s on the host)
    sdev = "cuda" if (torch.cuda.is_available() and os.environ.get("MPIG_REF_SETUP_CPU", "0") != "1") else "cpu"
    kcodes = synth.hash_keys(key.to(sdev), hf.to(sdev), K, L)
    qcodes = synth.hash_queries_ref(q, hf, K, L)
    q2 = q.reshape(B * Hq, d).contiguous()
    qn = q2.float().norm(p=2, dim=-1)
    cores = os.cpu_count() or 1
    if ref_loader.available():
        lsh_m, sa_m, flavour = ref_loader.load()
        R = lsh_m.LSH()
        R.alloc(K, L, 1, Hq, Hkv, B, M)
        S = sa_m.SparseAttentionServer()
        S.alloc(1, Hq, Hkv, d, B, M)
        for b in range(B):
            sc, si = kcodes[b].sort()
            R.fill(0, b, sc.cpu().contiguous(), si.int().cpu().contiguous())
            S.fill(0, b, key[b].contiguous(), value[b].contiguous(), kn[b].contiguous())
        del kcodes
        results = torch.zeros((B * Hq, M), dtype=torch.int32)
        nnz = torch.zeros((B * Hq,), dtype=torch.int32)
        out = torch.zeros((B * Hq, d), dtype=torch.bfloat16)
        mve = torch.zeros((2, B * Hq), dtype=torch.float32)

        def one():
            R.batch_retrieve(0, qcodes, results, nnz)
            S.attention_wrapper(0, K, L, out, mve, q2, qn, results, nnz)

        kind = "reference"
        host_cores = cores
        limit = int(os.environ.get("OMP_THREAD_LIMIT", "0") or 0)
        cores = min(64, limit) if limit > 0 else 64   # LSH_THREADS / ATTENTION_THREADS are #defined to 64 (lsh.h:12, sparse_attention.h:10)
        how = (f"unmodified reference operators (oracle/_ref, {flavour} build; its hard-coded 64 OpenMP threads"
               f"{f' capped at {limit} by OMP_THREAD_LIMIT' if limit > 0 else ''}, "
               f"OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND', 'unset')}, {host_cores} logical host CPUs)")
    else:
        kcodes = kcodes.cpu()
        Ts = []
        for b in range(B):
            sc, si = kcodes[b].sort()
            T = oracle.Tables(Hkv, L, K, M)
            T.fill(sc.contiguous(), si.int().contiguous())
            Ts.append(T)
        kp = torch.zeros((B * Hkv, M, d), dtype=torch.bfloat16); vp = torch.zeros((B * Hkv, M, d), dtype=torch.bfloat16)
        knp = torch.zeros((B * Hkv, M))
        kp[:, :n], vp[:, :n], knp[:, :n] = key.reshape(-1, n, d), value.reshape(-1, n, d), kn.reshape(-1, n)
        nnz = None

        def one():
            nonlocal nnz
            rs, nz = [], []
            for b in range(B):
                r, z, _ = oracle.batch_retrieve(Ts[b], qcodes[b * Hq:(b + 1) * Hq].contiguous(), G)
                rs.append(r), nz.append(z)
            nnz = torch.cat(nz)
            oracle.attention_wrapper(kp, vp, knp, K, L, q2, qn, torch.cat(rs), nnz)

        kind, cores = "port", 1
        how = "oracle/mpig_oracle.c restatement, single thread (oracle/_ref unavailable on this host)"
    for _ in range(3):
        one()
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < min_reps or (time.perf_counter() < t_end and len(times) < 2000):
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
    ms = 1e3 * statistics.mean(times)
    return dict(ms_layer=ms, ms_layer_min=1e3 * min(times), ms_layer_median=1e3 * statistics.median(times), kind=kind, cores=cores,
                reps=len(times), nnz_frac=float(nnz.float().mean()) / n,
                sample=f"1 of the 30 sparse layers (B={B}, Hq=32, Hkv=8, n={n}, K={K}, L={L}, {args.dist} keys), "
                       f"{len(times)} reps of batch_retrieve+attention_wrapper, x30 layers per token; {how}")


def reference_configs(info):
    """The protocols the reference arm is timed under (BASELINE.md 3.2, README.md:122-128, examples/bench.sh:1):
      stock         the build as shipped: 64 OpenMP threads, no binding (what round 1 measured; box-dependent)
      stock_pinned  the same 64 threads bound to cores (OMP_PROC_BIND=close OMP_PLACES=cores: the README's numactl -C line)
      tuned_pinned  team capped at the physical cores this process may use when that differs from 64
                    (README: "set the threads to the number of physical cores"; OMP_THREAD_LIMIT caps the hard-coded
                    num_threads(64) clauses -- every parallel region of the path is a `parallel for`, so the work is unchanged)
    """
    cfgs = [("stock", {}),
            ("stock_pinned", {"OMP_PROC_BIND": "close", "OMP_PLACES": "cores"})]
    nphys = usable_cores(info)
    if nphys != 64:
        cfgs.append(("tuned_pinned", {"OMP_PROC_BIND": "close", "OMP_PLACES": "cores", "OMP_THREAD_LIMIT": str(min(nphys, 64))}))
    if nphys < 64:   # oversubscribed hosts: spinning barriers are what made the stock run 5x slower on one box in round 1
        cfgs.append(("stock_passive", {"OMP_WAIT_POLICY": "passive"}))
    return cfgs


def run_reference_protocols(args, budget_s: float, min_reps: int = 3):
    """Each protocol in its own process (OpenMP reads its environment once, at start-up).  Returns (best, all, host_info)."""
    info = host_info()
    results = {}
    for name, env_add in reference_configs(info):
        env = dict(os.environ)
        env.update(env_add)
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-worker", "--B", str(args.B), "--P", str(args.P),
               "--M", str(args.M), "--K", str(args.K), "--L", str(args.L), "--dist", args.dist, "--cpu-seconds", str(budget_s),
               "--ref-min-reps", str(min_reps)]
        try:
            r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=max(300.0, 20 * budget_s))
            line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
            results[name] = json.loads(line)
            results[name]["env"] = env_add
        except Exception as e:
            results[name] = {"error": repr(e)[:300], "env": env_add}
    ok = {k: v for k, v in results.items() if "ms_layer" in v}
    if not ok:   # last resort: time it in this process
        r = cpu_reference_layer(args, budget_s, min_reps)
        r["protocol"] = "in_process"
        return r, results, info
    best_name = min(ok, key=lambda k: ok[k]["ms_layer"])
    best = dict(ok[best_name])
    best["protocol"] = best_name
    return best, results, info


def protocols_summary(all_results):
    return {k: ({"ms_per_layer": v["ms_layer"], "ms_per_layer_min": v.get("ms_layer_min"), "threads": v.get("cores"), "env": v.get("env")}
                if "ms_layer" in v else {"error": v.get("error"), "env": v.get("env")}) for k, v in all_results.items()}


def run_reference_arm(args, rank: int):
    """`--impl reference`: the reference's CPU implementation of the hot path, rank 0 only."""
    if rank != 0:
        return
    if args.ref_worker:
        r = cpu_reference_layer(args, budget_s=args.cpu_seconds, min_reps=args.ref_min_reps)
        print(json.dumps(r), flush=True)
        return
    n_sparse = 30
    budget = max(8.0, min(40.0, 0.15 * (args.steps + args.warmup)))
    best, all_results, info = run_reference_protocols(args, budget_s=budget, min_reps=max(3, min(args.steps, 64)))
    ms_token = best["ms_layer"] * n_sparse
    val = args.B * 1e3 / ms_token
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_token, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args),
        "where": "cpu",
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": best["cores"], "kind": best["kind"], "sample": best["sample"],
                         "protocol": best["protocol"], "ms_per_layer": best["ms_layer"], "threads": best["cores"],
                         "physical_cores_usable": usable_cores(info), "protocols": protocols_summary(all_results), "host": info},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "hot path only (30 sparse layers x [batch_retrieve + attention_wrapper] on host cores), the FASTEST of the protocols in "
                "cpu_baseline.protocols; excludes the reference's GPU-side GEMMs/window attention and its 60 PCIe hops per token, so it "
                "is an UPPER bound on the reference's tokens/s on this box (compare with this repo's hot_path.tokens_per_s, not with value)",
        "sample_fraction": best["nnz_frac"],
    }
    print(json.dumps(line))


def workload_config(args):
    model = "Llama-3.1-8B-Instruct" if args.model == "8b" else "Llama-3.1-70B-Instruct"
    layers = "32 layers: 30 LSH-sparse + 2 dense [0,16]" if args.model == "8b" else "80 layers: 75 LSH-sparse + 5 dense [0,16,32,48,64]"
    return {"workload": f"{model} decode B={args.B} P={args.P} M={args.M} K={args.K} L={args.L} "
                        f"({layers}; random-init weights; synthetic {args.dist} KV context)",
            "global_batch": args.B * (args.gpus if args.parallel == "dp" else 1), "seq_len": args.P,
            "parallelism": (f"dp{args.gpus}" if args.parallel == "dp" else f"kv-head-tp{args.gpus}") if args.gpus > 1 else "single",
            "l2_policy": "working set per step (16 GB weights + 30 distinct layers of tables/KV) >> 126 MB L2; no explicit flush"}


# ------------------------------------------------------------------------------------------------
# pieces of the measurement
# ------------------------------------------------------------------------------------------------
def model_shape(name: str):
    from magicpig_b200.llama_runner import LLAMA31_8B, LLAMA31_70B
    return {"8b": LLAMA31_8B, "70b": LLAMA31_70B}[name]


def needed_window(args, extra: int = 0) -> int:
    staged_tokens = 3
    need = (2 + staged_tokens + 3 + 3) + 4 + 2 * args.warmup + 2 * args.steps + 12 + extra
    return max(256, need)


def build_runner(args, shape, dev, rank, world, tp, tp_mode="ag", tp_transport="nccl", gen_buf=None):
    import torch.distributed as dist
    from magicpig_b200.llama_runner import LlamaDecodeRunner
    runner = LlamaDecodeRunner(shape, args.K, args.L, args.B, args.M, device=dev, seed=0, generation_buffer=gen_buf or needed_window(args),
                               num_layers=(args.layers or None), tp_rank=rank if tp else 0, tp_world=world if tp else 1,
                               tp_group=dist.group.WORLD if tp else None, tp_mode=tp_mode, tp_transport=tp_transport)
    runner.server.ctx.set_option("decode_impl", args.decode_impl)
    for key, env in (("pdl_first", "MPIG_PDL_FIRST"), ("fused_kreg", "MPIG_FUSED_KREG")):   # A/B switches for measurement scripts
        if os.environ.get(env) is not None:
            runner.server.ctx.set_option(key, int(os.environ[env]))
    t0 = time.time()
    runner.synthetic_prefill(args.P, seed=100 + (0 if tp else rank), dist=args.dist)
    return runner, time.time() - t0


def make_timed(world, dev):
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn_step, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn_step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms

    return timed


def graph_us_per_call(fn, calls_per_replay: int, reps: int = 5):
    """fn() enqueues `calls_per_replay` launches; captured in one CUDA graph, replayed `reps` times between CUDA events."""
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay()
    torch.cuda.synchronize()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(reps):
        g.replay()
    a1.record()
    torch.cuda.synchronize()
    us = a0.elapsed_time(a1) * 1e3 / (reps * calls_per_replay)
    del g
    return us, reps * calls_per_replay


def measure_hot_path(args, runner, dev, default_workload):
    """The sparse-attention path alone on this rank's heads: fused single-launch decode (the product path), the three-launch
    variant with per-stage CUDA events, the host-buffer entry point, and the roofline of the dominant kernel."""
    import ctypes
    import torch
    from magicpig_b200 import _native as N_
    srv, ctx = runner.server, runner.server.ctx
    sparse_layers = [l for l in range(runner.n_layers) if l not in srv.dense_layers]
    nS = len(sparse_layers)
    n = args.P - 68
    Hq, Hkv, d = runner.Hq_loc, runner.Hkv_loc, runner.d
    H_loc = args.B * Hq
    g = torch.Generator(device=dev).manual_seed(5)
    staged_tokens = 3
    out_tmp = torch.empty((args.B, Hq * d), dtype=torch.bfloat16, device=dev)
    qs = torch.randn((staged_tokens, nS, args.B, Hq, 1, d), generator=g, device=dev).to(torch.bfloat16)
    ks = torch.randn((staged_tokens, nS, args.B, Hkv, 1, d), generator=g, device=dev).to(torch.bfloat16)
    vs = torch.randn((staged_tokens, nS, args.B, Hkv, 1, d), generator=g, device=dev).to(torch.bfloat16)
    nnz_log = torch.zeros((staged_tokens, nS, H_loc), dtype=torch.int32, device=dev)
    fused = bool(ctx.get_info("fused_applicable"))
    for _ in range(2):  # clock / cache warm-up of the path itself
        ctx.plan()
        for li, l in enumerate(sparse_layers):
            ctx.decode(l, qs[0, li], ks[0, li], vs[0, li], out_tmp)
    torch.cuda.synchronize()
    # three-launch variant, CUDA events between the launches (no PDL overlap in this mode)
    for tok in range(staged_tokens):
        ctx.plan()
        for li, l in enumerate(sparse_layers):
            ctx.decode_timed(l, qs[tok, li], ks[tok, li], vs[tok, li], out_tmp)
            N_.check(ctx.lib.mpig_last_probe(ctx._h, ctypes.c_void_p(nnz_log[tok, li].data_ptr()), None,
                                             ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    times = ctx.timing_collect()
    stage_ms = [[t[i] for t in times] for i in range(3)]
    # the product path: nS layers back to back (fused: ONE launch per layer), CUDA events around whole tokens
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    hot_tokens = 3
    ev0.record()
    for tok in range(hot_tokens):
        ctx.plan()
        for li, l in enumerate(sparse_layers):
            ctx.decode(l, qs[tok, li], ks[tok, li], vs[tok, li], out_tmp)
    ev1.record()
    torch.cuda.synchronize()
    hot_ms_token = ev0.elapsed_time(ev1) / hot_tokens
    # ... the same layers captured in ONE CUDA graph like the decode step (no host launch cost): us per layer = the dominant kernel's
    # average launch duration as it runs in the step (30 distinct layers => cold L2 for tables / records)
    ctx.plan()
    us_graph, launches_timed = graph_us_per_call(
        lambda: [ctx.decode(l, qs[0, li], ks[0, li], vs[0, li], out_tmp) for li, l in enumerate(sparse_layers)], nS) if nS else (float("nan"), 0)
    # ... and through the HOST-buffer entry point (mpig_decode_host), synchronous per layer -- the boundary the reference's CPU
    # operators sit behind (attnserver.py:272,302-306)
    qh = qs[0].reshape(nS, args.B, Hq, d).cpu().pin_memory()
    kh = ks[0].reshape(nS, args.B, Hkv, d).cpu().pin_memory()
    vh = vs[0].reshape(nS, args.B, Hkv, d).cpu().pin_memory()
    oh = torch.empty((args.B, Hq * d), dtype=torch.bfloat16).pin_memory()
    host_ms = []
    host_args = [(l, qh[li], kh[li], vh[li]) for li, l in enumerate(sparse_layers)]   # the caller's per-layer host tensors
    for tok in range(4):
        ctx.plan()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for l, qa, ka, va in host_args:
            ctx.decode_host(l, qa, ka, va, oh)
        host_ms.append((time.perf_counter() - t0) * 1e3)
    hot_host_ms_token = min(host_ms[1:])
    # the gather phase on its own (BASELINE metric: "HBM GB/s on KV gather"): the fused kernel's debug instantiation stamps clock64 at
    # its phase boundaries; per CTA: first row requested -> all tiles consumed and merged.  One untimed pass, outside every timed region.
    gather_us = None
    if fused and ctx.get_info("fused_applicable"):
        try:
            ctx.set_option("fused_debug", 1)
            try:
                mhz = float(subprocess.check_output(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits", "-i",
                                                     str(torch.cuda.current_device())]).decode().split()[0])
            except Exception:
                mhz = 1965.0
            recs = []
            ctx.plan()
            for li, l in enumerate(sparse_layers):
                ctx.decode(l, qs[0, li], ks[0, li], vs[0, li], out_tmp)
                recs += [r for r in ctx.fused_debug_read(min(H_loc * 8, 8 * 148)) if r[0] and r[6] and r[8]]
            if recs:
                gather_us = statistics.median((r[8] - r[6]) / mhz for r in recs)
        except Exception:
            gather_us = None
        finally:
            ctx.set_option("fused_debug", 0)
    nnz_tot = nnz_log.reshape(-1, H_loc).sum(dim=1).cpu().tolist()
    attend_bytes, probe_bytes, nnz_fracs = [], [], []
    for c, tot in enumerate(nnz_tot):
        wlen = 68 + 2 + (c // max(nS, 1)) + 1
        # algorithmic bytes (SURVEY 8(d)): S3 = 520 B per sampled (q-head, key) pair [256 K + 256 V + 4 norm + 4 index], window rows
        # once per kv-head, q/out/LSE per q-head; S2 = L * (8 + 4*n/NB) per q-head + 4 per selected index (the reference's int32
        # format); S1 = hash_func once
        attend_bytes.append(tot * 520 + args.B * Hkv * wlen * 512 + H_loc * (d * 2 * 2 + 8))
        probe_bytes.append(H_loc * args.L * (8 + 4 * n / (1 << args.K)) + 4 * tot)
        nnz_fracs.append(tot / (H_loc * n))
    s1_bytes = args.K * args.L * d * 2
    layer_bytes = (statistics.mean(attend_bytes) + statistics.mean(probe_bytes) + s1_bytes) if attend_bytes else float("nan")
    peak, peak_src = measured_peak_gbs()
    gbs = (layer_bytes / 1e9) / (us_graph / 1e6) if nS else float("nan")
    three = {"simhash": 1e3 * statistics.mean(stage_ms[0]), "probe": 1e3 * statistics.mean(stage_ms[1]),
             "attend": 1e3 * statistics.mean(stage_ms[2])} if stage_ms[2] else None
    kname = ("fused_decode_kernel (one launch per sparse layer: SimHash -> probe -> gather attention + window, LSE merge folded in)"
             if fused else "three launches: simhash_kernel | probe_kernel | attend_mma_kernel")
    roofline = {"kernel": kname, "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "peak_source": peak_src,
                "traffic": profiled_traffic("fused_decode_kernel") if (default_workload and fused) else None,
                "traffic_source": ("profiles/r2_dram_traffic_per_launch.json (ncu --set full, same workload)" if (default_workload and fused) else None),
                "bytes_per_launch": layer_bytes,
                "bytes_breakdown": {"S1_hash_func": s1_bytes, "S2_probe": statistics.mean(probe_bytes) if probe_bytes else None,
                                    "S3_gather": statistics.mean(attend_bytes) if attend_bytes else None},
                "gather_phase": ({"us_median_per_cta": gather_us, "achieved": statistics.mean(attend_bytes) / (gather_us * 1e-6) / 1e9,
                                  "frac": statistics.mean(attend_bytes) / (gather_us * 1e-6) / 1e9 / peak, "unit": "GB/s",
                                  "note": "S3 bytes of a launch / median over CTAs of (first row requested -> all tiles consumed and merged), clock64 "
                                          "stamps of the kernel's debug instantiation in a separate untimed pass; the same fetch with nothing else "
                                          "in the kernel: profiles/r2_gather_microbench.txt"} if (gather_us and attend_bytes) else None),
                "us_per_launch": us_graph, "launches_timed": launches_timed,
                "timing": "one launch per sparse layer (30 distinct layers => cold L2), all captured in ONE CUDA graph like the step, CUDA "
                          "events around the replays; achieved = algorithmic (S1+S2+S3) bytes / that duration",
                "three_launch_us_per_layer": three}
    hot = {"ms_per_token": hot_ms_token, "tokens_per_s": args.B * 1e3 / hot_ms_token if hot_ms_token else None,
           "ms_per_token_graph": us_graph * nS / 1e3, "us_per_layer_graph": us_graph, "fused_single_launch": fused,
           "host_buffers_ms_per_token": hot_host_ms_token, "three_launch_us_per_layer": three,
           "sample_fraction": statistics.mean(nnz_fracs) if nnz_fracs else None,
           "note": "ms_per_token: the sparse layers enqueued back to back from the host, CUDA events around whole tokens; "
                   "ms_per_token_graph: the same launches replayed from one CUDA graph; three_launch_us_per_layer: the three-kernel "
                   "variant with an event between kernels; every layer has its own tables / records => cold L2"}
    return hot, roofline, 2 + staged_tokens + hot_tokens + 1 + 4


def measure_step(args, runner, dev, rank, world, local_rank, replicas, sample_clocks=True):
    """Capture the decode step, warm up, time `steps` steps (value: ids resident in HBM) and again with host buffers (e2e)."""
    import torch
    ctx = runner.server.ctx
    vocab = runner.shape.vocab_size
    timed = make_timed(world, dev)
    launches_before = ctx.launch_count
    if args.no_graph:
        used, launches_per_step = 0, None
    else:
        used = runner.capture(warm=3)
        launches_per_step = (ctx.launch_count - launches_before) // used
    step_fn = runner.step if args.no_graph else runner.replay
    ids_host = torch.randint(0, vocab, (args.steps + args.warmup + 8, args.B, 1), generator=torch.Generator().manual_seed(0),
                             dtype=torch.long).pin_memory()
    logits_host = torch.empty((args.B, vocab), dtype=torch.float32).pin_memory()
    runner.ids.copy_(ids_host[0])
    for _ in range(args.warmup):
        step_fn()
    if args.profile_step:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_fn()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    sampler = ClockSampler(local_rank)
    if rank == 0 and sample_clocks:
        sampler.start()
    ms_total = timed(step_fn, args.steps)
    clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
    logits = runner.logits.cpu() if args.dump_outputs else None   # what the last timed step returned (the e2e steps below advance it)
    tokens = args.B * args.steps * replicas
    value = tokens / (ms_total / 1e3)
    it = {"i": 0}

    def e2e_step():
        runner.ids.copy_(ids_host[it["i"] % ids_host.shape[0]], non_blocking=True)   # H2D from pinned memory
        it["i"] += 1
        lg = step_fn()
        logits_host.copy_(lg, non_blocking=True)                                         # D2H of the step's result
        torch.cuda.current_stream().synchronize()

    for _ in range(3):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    return dict(value=value, ms_per_step=ms_total / args.steps, e2e_value=tokens / (ms_e2e / 1e3), e2e_ms_per_step=ms_e2e / args.steps,
                clocks=clocks, launches_per_step=launches_per_step, h2d=args.B * 8, d2h=args.B * vocab * 4, logits=logits)


def dump_outputs(out_dir: str, logits):
    """`--dump-outputs`: the last timed step's logits as <out_dir>/logits.npy (float32).  Above 64 MB (B > 130) only a fixed,
    seeded sample of the batch rows is kept, in ascending row order."""
    import numpy as np
    a = logits.float().numpy()
    keep = (64 << 20) // a[0].nbytes
    if a.shape[0] > keep:
        a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), a)


def release_runner(runner):
    """Drop the captured graph FIRST (it may hold NCCL kernels), then the exchange object, then the context."""
    import gc
    import torch
    runner.graph = None
    gc.collect()
    torch.cuda.synchronize()
    if getattr(runner, "peer", None) is not None:
        runner.peer.close()
        runner.peer = None
    runner.server.ctx.close()
    gc.collect()
    torch.cuda.empty_cache()


def collective_us(runner, dev, mode, transport, B, reps=200):
    """The exchange step alone, `reps` back to back in one CUDA graph: us per collective of this layout / transport."""
    import torch
    from magicpig_b200 import tp as tpmod
    hs, Hq, d, W = runner.shape.hidden_size, runner.Hq_loc, runner.d, runner.tp_world
    if mode == "ag":
        a = torch.zeros((B, Hq * d), dtype=torch.bfloat16, device=dev)
        buf = torch.empty((W, B, Hq * d), dtype=torch.bfloat16, device=dev)
        one = (lambda: runner.peer.all_gather(a)) if transport == "peer" else (lambda: tpmod.gather_head_outputs(a, W, runner.tp_group, buf))
        payload = B * Hq * d * 2
    else:
        t = torch.zeros((B, hs), dtype=torch.bfloat16, device=dev)
        one = (lambda: runner.peer.all_reduce(t)) if transport == "peer" else (lambda: tpmod.all_reduce_sum(t, runner.tp_group))
        payload = B * hs * 2
    us, _ = graph_us_per_call(lambda: [one() for _ in range(reps)], reps, reps=3)
    return us, payload


def measure_tp_variants(args, dev, rank, world, local_rank, dp_value_per_gpu):
    """KV-head tensor parallelism of the SAME workload over the `world` GPUs (strong scaling), measured after the replica run:
    layouts "ag" (north-star: all-gather of head outputs, rest replicated) and "megatron" (llama_dist.py:49-70: wo/MLP sharded, two
    all-reduces per layer), each with NCCL collectives and with this repo's peer-memory exchange (csrc/peer.cu; for "ag" the stores
    come from the attention kernel's epilogue).  At world == 8 also C5: Llama-3.1-70B, Hq 8 / Hkv 1 per GPU."""
    import torch
    out = {"scaling": "strong", "world": world, "variants": {}, "single_gpu_tokens_per_s": dp_value_per_gpu}
    jobs = [("8b", m, t) for m in ("ag", "megatron") for t in ("nccl", "peer")]
    if world >= 4 and not args.layers:
        jobs += [("70b", "megatron", "nccl"), ("70b", "megatron", "peer")]
    for model, mode, transport in jobs:
        key = f"{model}/{mode}/{transport}"
        try:
            shape = model_shape(model)
            runner, prefill_s = build_runner(args, shape, dev, rank, world, True, mode, transport, gen_buf=2 * needed_window(args))   # two timed runs
            r = measure_step(args, runner, dev, rank, world, local_rank, 1, sample_clocks=False)
            cu, payload = collective_us(runner, dev, mode, transport, args.B)
            ncoll = runner.n_collectives
            # the same step with every exchange left out (wrong logits, per-rank compute only): the exchange's cost inside the
            # step -- latency plus the waiting for the slower rank -- is the measured difference
            runner.skip_exchange = True
            r0 = measure_step(args, runner, dev, rank, world, local_rank, 1, sample_clocks=False)
            runner.skip_exchange = False
            rec = {"tokens_per_s": r["value"], "ms_per_step": r["ms_per_step"], "e2e_tokens_per_s": r["e2e_value"],
                   "collectives_per_step": ncoll, "us_per_collective": cu, "payload_bytes": payload,
                   "collective_share_of_step": ncoll * cu / (r["ms_per_step"] * 1e3),
                   "ms_per_step_without_exchange": r0["ms_per_step"],
                   "exchange_ms_in_step": r["ms_per_step"] - r0["ms_per_step"],
                   "fused_single_launch": bool(runner.server.ctx.get_info("fused_applicable")),
                   "per_gpu_heads": {"Hq": runner.Hq_loc, "Hkv": runner.Hkv_loc}}
            if model == "8b" and dp_value_per_gpu:
                rec["speedup_vs_1gpu"] = r["value"] / dp_value_per_gpu
                rec["strong_scaling_efficiency"] = r["value"] / dp_value_per_gpu / world
            out["variants"][key] = rec
            release_runner(runner)
            del runner
        except Exception as e:   # a variant that cannot run is reported, it never blocks the line
            out["variants"][key] = {"error": repr(e)[:400]}
    ok = {k: v for k, v in out["variants"].items() if "tokens_per_s" in v and k.startswith("8b/")}
    if ok:
        best = max(ok, key=lambda k: ok[k]["tokens_per_s"])
        out["best_8b"] = best
        b = ok[best]
        share = b["exchange_ms_in_step"] / b["ms_per_step"]
        lim = "exchange latency" if share > 0.3 else "per-GPU weight/KV streaming + launch latency of the small per-rank kernels"
        out["limiter"] = (f"{best}: {b['collectives_per_step']} collectives/step cost {b['exchange_ms_in_step']:.2f} ms of the "
                          f"{b['ms_per_step']:.2f} ms step ({100 * share:.0f}%; stand-alone {b['us_per_collective']:.1f} us each); per-rank compute "
                          f"alone {b['ms_per_step_without_exchange']:.2f} ms vs {1e3 / dp_value_per_gpu if dp_value_per_gpu else 0:.2f} ms on one GPU -> {lim}")
    return out


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    tp = args.parallel == "tp" and world > 1
    shape = model_shape(args.model)
    default_workload = (args.B, args.P, args.M, args.K, args.L, args.layers, args.dist, args.model) == (1, 98000, 98304, 10, 150, 0, "gauss", "8b") and not tp
    runner, prefill_s = build_runner(args, shape, dev, rank, world, tp, args.tp_mode, args.tp_transport)
    ctx = runner.server.ctx
    n_layers = runner.n_layers
    n_sparse = len([l for l in range(n_layers) if l not in runner.server.dense_layers])
    hot, roofline, _ = measure_hot_path(args, runner, dev, default_workload)
    replicas = world if (world > 1 and not tp) else 1
    r = measure_step(args, runner, dev, rank, world, local_rank, replicas)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, r["logits"])

    line = None
    if rank == 0:
        n_dense = n_layers - n_sparse
        per_layer = 1 if hot["fused_single_launch"] else 3
        per_step_launches = r["launches_per_step"] if r["launches_per_step"] is not None else (per_layer * n_sparse + 2 * n_dense + 1)
        per_step_launches += runner.aux_launches_per_step   # harness kernels of this repo (GEMVs with fused norm / RoPE / SwiGLU)
        line = {
            "metric": METRIC if args.model == "8b" else METRIC.replace("8B", "70B"), "value": r["value"], "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong" if tp else "weak",
            "vs_baseline": (r["value"] / replicas / PUBLISHED_B1) if (args.B == 1 and not args.layers and args.model == "8b") else None,
            "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args),
            "where": "gpu",
            "clocks": r["clocks"],
            "e2e": {"value": r["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "ms_per_step": r["e2e_ms_per_step"]},
            "gpu_launches": int(per_step_launches) * args.steps,
            "roofline": roofline,
            "hot_path": hot,
            "setup": {"synthetic_prefill_s": prefill_s, "hbm_bytes_context": ctx.device_bytes, "generation_buffer": needed_window(args),
                      "cuda_graph": not args.no_graph, "sparse_layer_launches": per_layer,
                      "linear_layers": "mpig_aux_gemv (weight-streaming GEMV, SwiGLU fused) + cuBLAS lm_head" if (runner.use_gemv and args.B <= runner.GEMV_MAX_ROWS)
                      else "torch.nn.functional.linear (cuBLAS)"},
        }
        if tp:
            line["tp"] = {"mode": args.tp_mode, "transport": args.tp_transport, "collectives_per_step": runner.n_collectives}
        if args.layers:
            line["INVALID"] = f"debug run with {args.layers} layers: not the named config"
    # ---- N > 1: the same workload under KV-head tensor parallelism (strong scaling), reported inside the replica line ----------
    if world > 1 and not tp and not args.no_tp_record:
        dp_per_gpu = r["value"] / world
        release_runner(runner)
        del runner
        tp_rec = measure_tp_variants(args, dev, rank, world, local_rank, dp_per_gpu)
        if rank == 0:
            line["tp"] = tp_rec
        runner = None
    # ---- cpu_baseline: rank 0, N=1 only -------------------------------------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        release_runner(runner)
        runner = None
        try:
            rr, all_results, info = run_reference_protocols(args, budget_s=args.cpu_seconds)
            line["cpu_baseline"] = {"value": args.B * 1e3 / (rr["ms_layer"] * n_sparse), "unit": UNIT, "cores": rr["cores"], "kind": rr["kind"],
                                    "sample": rr["sample"], "ms_per_layer": rr["ms_layer"], "sample_fraction": rr["nnz_frac"],
                                    "protocol": rr["protocol"], "threads": rr["cores"], "physical_cores_usable": usable_cores(info),
                                    "protocols": protocols_summary(all_results), "host": info}
            # like for like: the sparse layers alone, this repo's kernels vs the reference's operators on this box
            ref_ms_token = rr["ms_layer"] * n_sparse
            line["hot_path_vs_reference"] = {
                "reference_ms_per_token": ref_ms_token,
                "device_buffers": ref_ms_token / line["hot_path"]["ms_per_token"],
                "host_buffers": ref_ms_token / line["hot_path"]["host_buffers_ms_per_token"],
                "note": "the sparse layers alone on both sides; host_buffers = through mpig_decode_host (q/k/v/out in host memory, "
                        "synchronous per layer), the boundary the reference's CPU operators sit behind"}
        except Exception as e:  # the baseline is a report, never a dependency of the product number
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(e)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # tear-down order: captured graphs (they may hold NCCL kernels) and exchange objects first, then the communicator
        if runner is not None:
            release_runner(runner)
            runner = None
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
