#!/usr/bin/env python
"""bench.py — MBAR self-consistent iteration throughput on B200 (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json metric / configs[2] shape): synthetic harmonic-oscillator u_kn, K = 256
states, N = 1e7 samples PER GPU (20.48 GB of fp64 in HBM, far larger than the 126 MB L2), equal N_k,
Philox-keyed generation on device.  A step = one full self-consistent iteration (Eq. C3):
one fused streaming pass over u_kn + (N>1) one NCCL all-reduce of the K+2 partials + the K-vector
update, device resident, no host round trip between steps.  Samples shard over ranks (weak
scaling: each rank owns 1e7 samples of a 1e7*N-sample problem), no other data-path collective.

Reported: value = K*N_total*iterations / second (entries/s, whole job), `iter_per_s`, achieved HBM
GB/s, `roofline` for the fused pass kernel (algorithmic bytes 8*K*N_local per launch over its
CUDA-event launch duration, against MEASURED_PEAKS.json), `e2e` through the reference-facing call
`pymbar_b200.mbar_solvers.self_consistent_update(u_kn_host, N_k, f_k)` with the u_kn upload inside
every timed step, and `cpu_baseline` = the numpy oracle port of the reference timed on this host.

`--config c2|c4|c5` runs one of the other BASELINE.json configs in detail (C2: K=64, N=1e6 adaptive solve; C4:
K=32, N=1e7 strong-scaled over the GPUs with the per-iteration exchange cost; C5: K=512, N=1.25e7 per GPU); the
default line carries their summaries under `configs`, multi-rank parity under `parity_multi_rank` (N > 1), the
Hessian kernel's fp64 roofline under `roofline_hessian` and the MBAR.__init__-shaped end-to-end leg under
`e2e_solve`.

`--impl reference`: the reference's own CPU algorithm (oracle numpy port — the reference is pure
Python and /root/reference does not exist on the GPU box) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K_STATES = 256
N_PER_GPU = 10_000_000
METRIC = "MBAR self-consistent iteration throughput at K=256, N=1e7 samples per GPU (u_kn entries/s; iter/s and HBM GB/s alongside)"
UNIT = "entries/s"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def workload_params(K):
    O_k = np.linspace(1.0, 5.0, K)      # utils_for_testing.py:64-66 spacing (SURVEY 8d)
    k_k = np.linspace(1.0, 3.0, K)
    return O_k, k_k


def global_N_k(K, N_total):
    N_k = np.full(K, N_total // K, dtype=np.float64)
    N_k[-1] += N_total - N_k.sum()
    return N_k


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(K, N_local):
    """(dram read+write bytes per launch, source) of the fused kernel.  DRAM counters cannot be read inside a
    timed run (they need ncu's replay), so this is the committed `ncu --set full` capture of the same kernel and
    shape (newest round first), scaled to this launch's N when the capture used a smaller N of the same K."""
    for name in ("fused_pass_c3_r2.json", "fused_pass_c3_r1.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            break
    try:
        t = json.load(open(path))
        if t["K"] == K:
            return (float(t["dram_bytes_per_launch"]) * (N_local / t["N"]),
                    f"profiles/{name} ({t.get('source', 'ncu --set full')}), K={t['K']} N={t['N']}")
    except Exception:
        pass
    return None


# ---------------------------------------------------------------------------------------------
# CPU legs (oracle = numpy port of the reference; test infrastructure used here only as the baseline)
# ---------------------------------------------------------------------------------------------
def cpu_sample(K, n_sample, seed=0):
    from oracle import testsystems as ots  # noqa: F401  (same functional form, numpy RNG on the host)

    O_k, k_k = workload_params(K)
    rng = np.random.default_rng(seed)
    per = max(1, n_sample // K)
    x = np.concatenate([rng.normal(O_k[k], k_k[k] ** -0.5, per) for k in range(K)])
    u_kn = 0.5 * k_k[:, None] * (x[None, :] - O_k[:, None]) ** 2
    return u_kn, np.full(K, float(per))


def time_cpu_reference(K, budget_s, steps, warmup):
    """Oracle self_consistent_update on a bounded sample sized to `budget_s` seconds in total."""
    from oracle import mbar_oracle as orc

    u, N_k = cpu_sample(K, 20 * K)
    f = np.zeros(K)
    t0 = time.perf_counter()
    orc.self_consistent_update(u, N_k, f)
    rate = u.size / max(time.perf_counter() - t0, 1e-6)              # entries/s, rough
    entries = rate * budget_s / max(1, steps + warmup)
    n_sample = int(min(max(entries / K, 40 * K), 2_000_000))
    u, N_k = cpu_sample(K, n_sample)
    for _ in range(warmup):
        f = orc.self_consistent_update(u, N_k, f)
        f -= f[0]
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        f = orc.self_consistent_update(u, N_k, f)
        f -= f[0]
        times.append(time.perf_counter() - t0)
    per_step = float(np.mean(times))
    return u.size / per_step, per_step, u.shape[1]


def time_c_port(K, n_sample=400_000):
    """The C/pthreads restatement of the same two sweeps with every host thread: context beside the
    single-threaded numpy port (which is what the reference's own implementation is)."""
    try:
        from oracle import c_oracle

        c_oracle.load(build=False)           # built by build(); the benchmark compiles nothing into the tree
        u, N_k = cpu_sample(K, n_sample)
        f = np.zeros(K)
        c_oracle.self_consistent_update(u, N_k, f)
        t0 = time.perf_counter()
        for _ in range(3):
            c_oracle.self_consistent_update(u, N_k, f)
        dt = (time.perf_counter() - t0) / 3
        return {"value": u.size / dt, "unit": UNIT, "threads": c_oracle.threads(),
                "what": "oracle/mbar_oracle.c (pthreads), same arithmetic, all host threads"}
    except Exception as exc:  # pragma: no cover
        return {"unavailable": str(exc)[:200]}


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    K = K_STATES
    value, per_step, n_sample = time_cpu_reference(K, budget_s=90.0, steps=args.steps, warmup=args.warmup)
    try:
        from threadpoolctl import threadpool_info
        blas = max([t.get("num_threads", 1) for t in threadpool_info()] or [1])
    except Exception:
        blas = None
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "iter_per_s_at_full_size": value / (K * N_PER_GPU),
        "config": {"workload": "MBAR self-consistent iteration, K=256, N=1e7 per GPU (reference timed on a bounded sample)",
                   "K": K, "N_sample": n_sample, "flush": "n/a (CPU)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port",
                         "host_cpus": os.cpu_count(), "blas_threads": blas,
                         "c_port_all_threads": time_c_port(K),
                         "sample": f"self_consistent_update (numpy oracle port of mbar_solvers.py:231-242, "
                                   f"scipy.special.logsumexp x2, single-threaded like the reference) on K={K}, "
                                   f"N={n_sample} of the same harmonic family; throughput is flat in N (BASELINE.md §2)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def alchemical_params(K):
    """C4 (BASELINE.json configs[3]): K lambda-windows, O(l) = 4 l, k(l) = 1 + 15 l (SURVEY.md 8d; the
    reference ships no alchemical code, examples/alchemical-free-energy/README.md:1-3 — synthetic)."""
    lam = np.linspace(0.0, 1.0, K)
    return 4.0 * lam, 1.0 + 15.0 * lam


class Rig:
    """Process-level plumbing shared by the config runners."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = env_int("WORLD_SIZE", 1)
        self.rank = env_int("RANK", 0)
        self.local = env_int("LOCAL_RANK", 0)
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: pymbar_b200 has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.distributed = self.world > 1
        if self.distributed:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))

    def barrier(self):
        if self.distributed:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        if self.distributed:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def attach(self, prob, peer=True):
        """NCCL communicator (+ peer-memory inboxes for the in-kernel exchange)."""
        from pymbar_b200 import DeviceProblem

        if not self.distributed:
            return
        uid = [DeviceProblem.comm_unique_id() if self.rank == 0 else None]
        self.dist.broadcast_object_list(uid, src=0)
        prob.comm_init(self.world, self.rank, uid[0])
        if peer:
            handles = [None] * self.world
            self.dist.all_gather_object(handles, prob.peer_export())
            prob.peer_attach(self.world, self.rank, handles)

    def close(self):
        if self.distributed:
            self.dist.barrier()
            self.dist.destroy_process_group()


def make_problem(rig, K, N_local, O_k, k_k, seed, sharded=True, peer=True):
    from pymbar_b200 import DeviceProblem

    world = rig.world if sharded else 1
    rank = rig.rank if sharded else 0
    N_total = N_local * world
    N_k = global_N_k(K, N_total)
    prob = DeviceProblem(None, N_k, device=rig.local, N_local=N_local)
    prob.synthesize(O_k, k_k, seed=seed, n_offset=rank * N_local, N_global=N_total)
    if sharded:
        rig.attach(prob, peer=peer)
    return prob, N_k


def timed_sci(rig, prob, K, steps, warmup, f0=None):
    """`steps` device-resident self-consistent iterations; CUDA events on the launching stream, max over ranks."""
    f = np.zeros(K) if f0 is None else f0
    f = prob.sci_iterate(f, warmup)
    rig.barrier()
    t0 = time.perf_counter()
    f = prob.sci_iterate(f, steps)
    rig.torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    loop = prob.last_loop_ms()
    total_ms, kernel_ms = rig.max_over_ranks([loop["total_ms"], loop["kernel_ms_sum"]])
    rig.barrier()
    return f, total_ms / steps, kernel_ms / steps, wall


def multi_rank_parity(rig, big_prob, f_big, K, iters=3, n_per_rank=4096):
    """Driver-visible multi-rank parity (VERDICT r1 'what's weak' 1).  Every rank downloads a slice of ITS shard,
    the slices form a small sample-sharded problem that runs `iters` device-resident self-consistent iterations
    through the same exchange path as the timed loop (in-kernel peer exchange, or NCCL when peers are off); rank 0
    compares with the CPU oracle on the concatenated slices and checks that all ranks hold bit-identical f —
    for the small problem AND for the timed full-size state."""
    from oracle import mbar_oracle as orc
    from pymbar_b200 import DeviceProblem

    dist, world, rank = rig.dist, rig.world, rig.rank
    sl = big_prob.download(0, n_per_rank)
    N_k = np.full(K, float(n_per_rank * world) / K)
    small = DeviceProblem(sl, N_k, device=rig.local)
    rig.attach(small, peer=not os.environ.get("MBAR_B200_NO_PEER"))
    f_dev = small.sci_iterate(np.zeros(K), iters)
    S_dev, sumL_dev, _ = small.streaming_pass(f_dev)                 # NCCL all-reduce path at the same point
    f_ad, r_ad = small.solve_adaptive(np.zeros(K), tol=1e-12, min_sc_iter=0)
    gathered = [None] * world
    dist.all_gather_object(gathered, sl.tobytes())
    ident = [None] * world
    dist.all_gather_object(ident, (f_dev.tobytes(), f_ad.tobytes(), np.asarray(f_big).tobytes()))
    out = None
    if rank == 0:
        u_cat = np.concatenate([np.frombuffer(b, dtype=np.float64).reshape(K, n_per_rank) for b in gathered], axis=1)
        f_ref = np.zeros(K)
        for _ in range(iters):
            nxt = orc.self_consistent_update(u_cat, N_k, f_ref)
            f_ref = nxt - nxt[0]
        S_ref, L_ref = orc.single_pass_sums(u_cat, N_k, f_dev)
        ad_ref = orc.adaptive(u_cat, N_k, np.zeros(K), tol=1e-12, options=dict(min_sc_iter=0))["x"]
        out = {
            "world": world, "samples_per_rank": n_per_rank, "sci_iterations": iters,
            "exchange": "nccl" if os.environ.get("MBAR_B200_NO_PEER") else "in-kernel peer memory",
            "max_abs_err_f_vs_oracle": float(np.max(np.abs(f_dev - f_ref))),
            "max_rel_err_S_vs_oracle": float(np.max(np.abs(S_dev - S_ref) / S_ref)),
            "rel_err_sumL_vs_oracle": float(abs(sumL_dev - L_ref.sum()) / abs(L_ref.sum())),
            "adaptive_max_abs_err_f_vs_oracle": float(np.max(np.abs(f_ad - ad_ref))),
            "adaptive_success": bool(r_ad["success"]),
            "bit_identical_f_across_ranks": all(x[0] == ident[0][0] for x in ident),
            "bit_identical_adaptive_f_across_ranks": all(x[1] == ident[0][1] for x in ident),
            "bit_identical_timed_f_across_ranks": all(x[2] == ident[0][2] for x in ident),
        }
        out["ok"] = bool(out["max_abs_err_f_vs_oracle"] < 1e-8 and out["adaptive_max_abs_err_f_vs_oracle"] < 1e-8
                         and out["max_rel_err_S_vs_oracle"] < 1e-10 and out["bit_identical_f_across_ranks"]
                         and out["bit_identical_adaptive_f_across_ranks"] and out["bit_identical_timed_f_across_ranks"])
    small.close()
    return out


def adaptive_report(prob, K, label, maxiter=100):
    """Adaptive solve (mbar_solvers.py:510-667) from f = 0 to tol 1e-12, device-resident vs host-stepped, plus the
    kernel-time budget it should be compared with (calibrated launches of the same kernels)."""
    rep = {}
    f0 = np.zeros(K)
    # calibration: one pass, one Hessian, on the resident data (CUDA events inside the library)
    prob.sci_iterate(f0, 3)
    prob.sci_iterate(f0, 10)
    pass_ms = prob.last_loop_ms()["kernel_ms_sum"] / 10
    prob.hessian(f0)
    prob.hessian(f0)
    hm = prob.last_hessian_ms()
    rep["pass_kernel_ms"] = pass_ms
    rep["hessian_ms"] = hm
    rep["pass_with_weights_ms"] = prob.last_pass_ms()       # the pass that fed the Hessian above (stores the weights)
    rep["kernels"] = prob.last_kernels()
    prob.pass_multi(np.stack([f0, f0]))
    prob.pass_multi(np.stack([f0, f0]))
    rep["pass_multi"] = {"last_launch_ms": prob.last_pass_ms(), "kernel": prob.last_kernels()["pass_kernel"],
                         "note": "M=2 in the kernel name: both candidates in ONE launch of this duration; otherwise "
                                 "two launches of this duration each"}
    for mode in ("device", "stepped"):
        prob.set_loop_mode(mode)
        polls0 = prob.loop_stats()["polls"]
        t0 = time.perf_counter()
        f, info = prob.solve_adaptive(np.zeros(K), tol=1e-12, maxiter=maxiter, min_sc_iter=0)
        wall = time.perf_counter() - t0
        d = {k: info[k] for k in ("success", "iterations", "nr_iterations", "sci_iterations", "passes",
                                  "hessian_passes", "gnorm", "device_ms")}
        d["wall_s"] = wall
        d["host_polls"] = prob.loop_stats()["polls"] - polls0
        m2 = "M=2" in rep["pass_multi"]["kernel"]
        cand_ms = rep["pass_multi"]["last_launch_ms"] * (1 if m2 else 2)
        budget = info["iterations"] * (rep["pass_with_weights_ms"] + cand_ms + hm["weights_ms"] + hm["hessian_ms"])
        # pass(+weights) + candidate pass(es) + Hessian kernels per iteration: no launch gaps, no Newton solve
        d["kernel_budget_ms"] = budget
        d["device_ms_over_budget"] = info["device_ms"] / budget if budget > 0 else None
        d["passes_per_s"] = info["passes"] / (info["device_ms"] * 1e-3) if info["device_ms"] > 0 else None
        rep[mode] = d
    prob.set_loop_mode("device")
    rep["label"] = label
    return rep, f


def hessian_roofline(prob, K, N_local, fp64_peak, plain_pass_ms=None):
    """roofline of the Hessian evaluation: useful symmetric flops K(K+1)N (one MAC = 2 flop on K(K+1)/2 entries)
    over the CUDA-event time of the DMMA kernel (+ the separate weights sweep when one runs), against the DMMA peak
    measured in this process.  The weights normally come out of the fused pass at the same f (WST variant), whose
    extra cost over a plain pass is reported as `weights_in_pass_ms` and included in `frac_all_in`."""
    f0 = np.zeros(K)
    prob.hessian(f0)
    ms, wst = [], []
    for _ in range(3):
        prob.hessian(f0)
        hm = prob.last_hessian_ms()
        ms.append(hm["weights_ms"] + hm["hessian_ms"])
        wst.append(prob.last_pass_ms())                      # the pass that fed this Hessian (stores the weights)
    t = float(np.median(ms))
    wst_ms = float(np.median(wst))
    if plain_pass_ms is None:
        prob.sci_iterate(f0, 3)
        prob.sci_iterate(f0, 10)
        plain_pass_ms = prob.last_loop_ms()["kernel_ms_sum"] / 10
    extra = max(0.0, wst_ms - plain_pass_ms)
    flops = float(K) * (K + 1) * N_local
    ach = flops / (t * 1e-3) / 1e12
    return {"bound": "fp64 tensor (DMMA.8x8x4; tcgen05 has no fp64 MMA)", "achieved": ach, "peak": fp64_peak[0],
            "unit": "TFLOP/s", "frac": ach / fp64_peak[0] if fp64_peak[0] else None,
            "useful_flops_per_launch": flops, "full_matrix_equivalent_tflops": 2.0 * K * K * N_local / (t * 1e-3) / 1e12,
            "launch_ms": t, "weights_ms": hm["weights_ms"], "dmma_kernel_ms": hm["hessian_ms"],
            "pass_with_weights_ms": wst_ms, "plain_pass_ms": plain_pass_ms, "weights_in_pass_ms": extra,
            "achieved_all_in": flops / ((t + extra) * 1e-3) / 1e12,
            "frac_all_in": flops / ((t + extra) * 1e-3) / 1e12 / fp64_peak[0] if fp64_peak[0] else None,
            "kernel": prob.last_kernels()["hessian_kernel"],
            "peak_source": "mbar_b200_measure_fp64_peak in this process: DMMA %.1f TFLOP/s, DFMA %.1f TFLOP/s "
                           "(shared fp64 datapath); MEASURED_PEAKS.json has no fp64 figure" % fp64_peak,
            "how": "CUDA events inside the library around weights_kernel and hessian kernel + reduction, median of 3"}


def run_c1(rig, args):
    """C1 (BASELINE.json configs[0]): testsystems.HarmonicOscillatorsTestCase defaults, K=5, N=5000 — the
    reference's own CPU-runnable case.  CPU leg: the numpy oracle port of the reference solve (this is the
    cpu_baseline of that config); GPU leg: the mirror's solve_mbar_for_all_states on the same host array, upload
    included, and |delta f| between the two."""
    from oracle import mbar_oracle as orc
    from oracle import testsystems as ots
    from pymbar_b200 import mbar_solvers as ms

    O, Kk, Nk = [0.0, 1.0, 2.0, 3.0, 4.0], [1.0, 2.0, 4.0, 8.0, 16.0], [1000] * 5
    _, u_kn, N_k = ots.harmonic_u_kn(O, Kk, Nk, seed=0)
    t0 = time.perf_counter()
    f_cpu = orc.mbar_f_k(u_kn, N_k)
    t_cpu = time.perf_counter() - t0
    sws = np.arange(5)
    ms._DEVICE = rig.local
    times = []
    for _ in range(4):
        proto = tuple({k: (dict(v) if isinstance(v, dict) else v) for k, v in st.items()}
                      for st in ms.DEFAULT_SOLVER_PROTOCOL)
        t0 = time.perf_counter()
        f_gpu = ms.solve_mbar_for_all_states(u_kn, np.asarray(N_k), np.zeros(5), sws, proto)
        times.append(time.perf_counter() - t0)
    ms.clear_cache()
    return {"workload": "C1: HarmonicOscillatorsTestCase defaults, K=5, N=5000, default solver protocol", "K": 5,
            "N": 5000, "reference_cpu_solve_s": t_cpu, "gpu_solve_s_first": times[0], "gpu_solve_s": float(np.median(times[1:])),
            "max_abs_df_vs_cpu": float(np.max(np.abs(f_gpu - f_cpu))),
            "note": "plumbing config: both legs are dominated by Python/scipy overhead (hybr with device closures)"}


def run_c2(rig, args):
    """C2: synthetic u_kn N=1e6, K=64, adaptive solver fp64 on one B200 (every rank runs its own copy)."""
    K, N = 64, 1_000_000
    O_k, k_k = workload_params(K)
    prob, N_k = make_problem(rig, K, N, O_k, k_k, args.seed, sharded=False)
    f, ms_step, kern_ms, _ = timed_sci(rig, prob, K, 200, 5)
    rep, f_sol = adaptive_report(prob, K, "C2 K=64 N=1e6")
    S, _, _ = prob.streaming_pass(f_sol)
    out = {"workload": "C2: K=64, N=1e6, adaptive solve + self-consistent passes, 1 GPU", "K": K, "N": N,
           "sci_ms_per_iteration": ms_step, "pass_kernel_ms": kern_ms,
           "sci_passes_per_s": 1e3 / ms_step, "hbm_gbs": 8.0 * K * N / (kern_ms * 1e-3) / 1e9,
           "entries_per_s": K * N / (ms_step * 1e-3),
           "adaptive": rep, "max_abs_S_minus_1_at_solution": float(np.max(np.abs(S - 1.0)))}
    prob.close()
    return out


def run_c4(rig, args):
    """C4: K=32 lambda-windows, N=1e7 TOTAL, sample-sharded over the ranks (strong scaling): per-iteration time
    with the in-kernel peer exchange, with NCCL, and with no exchange at all (same shard, no communicator)."""
    K, N_total = 32, 10_000_000
    world = rig.world
    N_local = N_total // world
    O_k, k_k = alchemical_params(K)
    steps = 400
    out = {"workload": f"C4: K=32 lambda-windows, N=1e7 total, sample-sharded x{world} (strong scaling)", "K": K,
           "N_total": N_local * world, "N_per_gpu": N_local, "n_gpus": world}
    solo, _ = make_problem(rig, K, N_local, O_k, k_k, args.seed, sharded=False)
    _, ms0, k0, _ = timed_sci(rig, solo, K, steps, 10)
    out["no_exchange_ms_per_iteration"] = ms0
    out["pass_kernel_ms"] = k0
    out["hbm_gbs_per_gpu_kernel"] = 8.0 * K * N_local / (k0 * 1e-3) / 1e9
    solo.close()
    prob, N_k = make_problem(rig, K, N_local, O_k, k_k, args.seed, sharded=True, peer=True)
    f, ms_peer, _, _ = timed_sci(rig, prob, K, steps, 10)
    out["peer_ms_per_iteration"] = ms_peer if world > 1 else None
    out["ms_per_iteration"] = ms_peer
    out["entries_per_s"] = K * N_local * world / (ms_peer * 1e-3)
    if world > 1:
        os.environ["MBAR_B200_NO_FUSED_EPILOGUE"] = "1"
        _, ms_nccl, _, _ = timed_sci(rig, prob, K, steps, 10)
        del os.environ["MBAR_B200_NO_FUSED_EPILOGUE"]
        out["nccl_ms_per_iteration"] = ms_nccl
        out["exchange_us_peer"] = (ms_peer - ms0) * 1e3
        out["exchange_us_nccl"] = (ms_nccl - ms0) * 1e3
    t0 = time.perf_counter()
    f_sol, info = prob.solve_adaptive(np.zeros(K), tol=1e-12, maxiter=100, min_sc_iter=0)
    out["adaptive"] = {k: info[k] for k in ("success", "iterations", "nr_iterations", "sci_iterations", "passes",
                                            "device_ms", "gnorm")}
    out["adaptive"]["wall_s"] = time.perf_counter() - t0
    ana = -0.5 * np.log(2 * np.pi / k_k)
    out["max_abs_err_vs_analytic_f"] = float(np.max(np.abs((f_sol - f_sol[0]) - (ana - ana[0]))))
    prob.close()
    return out


def run_c5(rig, args):
    """C5: K=512, N=1.25e7 per GPU (1e8 over 8 GPUs), sample-sharded, per-iteration exchange of the partials."""
    K, N_local = 512, 12_500_000
    O_k, k_k = workload_params(K)
    prob, N_k = make_problem(rig, K, N_local, O_k, k_k, args.seed, sharded=True, peer=True)
    f, ms_step, kern_ms, _ = timed_sci(rig, prob, K, 40, 4)
    out = {"workload": f"C5: K=512, N=1.25e7 per GPU, sample-sharded x{rig.world} (weak scaling)", "K": K,
           "N_per_gpu": N_local, "n_gpus": rig.world, "ms_per_iteration": ms_step, "pass_kernel_ms": kern_ms,
           "entries_per_s": K * N_local * rig.world / (ms_step * 1e-3),
           "hbm_gbs_per_gpu": 8.0 * K * N_local / (ms_step * 1e-3) / 1e9,
           "hbm_gbs_per_gpu_kernel": 8.0 * K * N_local / (kern_ms * 1e-3) / 1e9,
           "kernel": prob.last_kernels()["pass_kernel"]}
    if rig.world == 1 and args.c5_hessian:
        from pymbar_b200.problem import measure_fp64_peak

        out["roofline_hessian"] = hessian_roofline(prob, K, N_local, measure_fp64_peak(rig.local))
    prob.close()
    return out


def e2e_legs(rig, args, prob, K, N_local, N_k):
    """End to end through the reference-facing API with HOST buffers.
    (1) `e2e`: mbar_solvers.self_consistent_update(u_kn_host) — create + upload + pass + destroy per call — on a
        pinned array (the contract's 'pinned host memory') and on a pageable numpy array (what pymbar.MBAR holds,
        mbar.py:243).
    (2) `e2e_solve`: what MBAR.__init__ calls (mbar.py:413, :455): solve_mbar_for_all_states(pageable u_kn) and
        mbar_log_W_nk, with upload / solve / logW download itemised."""
    from pymbar_b200 import PinnedArray
    from pymbar_b200 import mbar_solvers as ms

    os.environ["PYMBAR_B200_CACHE"] = "0"              # every call uploads u_kn (no residency)
    os.environ["PYMBAR_B200_DEVICE"] = str(rig.local)
    ms._DEVICE = rig.local
    pin = PinnedArray((K, N_local))
    prob.download(0, N_local, out=pin.array)           # setup: host copy of this rank's shard
    if not rig.distributed:
        prob.close()                                   # never two 20 GB problems + staging at once
    h2d0 = 8 * K * N_local + 8 * K
    res = {}
    for kind in ("pinned", "pageable"):
        if kind == "pageable":
            # (one pageable + one pinned copy of the shard per rank: bounded to 4 ranks' worth of host memory)
            if args.e2e_pageable_steps <= 0 or rig.world > 4:
                continue
            src = np.empty((K, N_local))
            src[:] = pin.array
            nsteps = args.e2e_pageable_steps
        else:
            src = pin.array
            nsteps = args.e2e_steps
        fh = np.zeros(K)
        times = []
        for i in range(1 + nsteps):
            rig.barrier()
            t0 = time.perf_counter()
            if rig.distributed:
                # ONE sample-sharded call: every rank re-uploads its host shard into the attached problem, the
                # pass runs on all GPUs and the partial sums are all-reduced (NCCL) before f comes back
                prob.upload(src)
                out = prob.self_consistent_update(fh)
            else:
                out = ms.self_consistent_update(src, N_k, fh)
            dt = time.perf_counter() - t0
            if i > 0:
                times.append(dt)
            fh = out - out[0]
        e2e_s = rig.max_over_ranks([float(np.mean(times))])[0]
        res[kind] = {"value": K * N_local * rig.world / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d0,
                     "d2h_bytes_per_step": 8 * (2 * K + 2), "s_per_step": e2e_s, "steps": nsteps,
                     "h2d_gbs": h2d0 / e2e_s / 1e9, "pcie_fraction_of_gen5_x16": h2d0 / e2e_s / 63.0e9}
        if kind == "pageable":
            del src
    if rig.distributed:
        # every rank must hold the same f after the sharded call
        same = [None] * rig.world
        rig.dist.all_gather_object(same, fh.tobytes())
        res["pinned"]["bit_identical_f_across_ranks"] = all(b == same[0] for b in same)
        prob.close()
    e2e = dict(res["pinned"])
    if rig.distributed:
        e2e["call"] = ("DeviceProblem.upload(u_kn_host_shard[pinned]) + DeviceProblem.self_consistent_update(f_k) on "
                       "the sample-sharded problem of all ranks (upload of every shard + pass + NCCL all-reduce of "
                       "the partial sums inside every step)")
        e2e["note"] = "one multi-GPU call per step; time = max over ranks"
    else:
        e2e["call"] = ("pymbar_b200.mbar_solvers.self_consistent_update(u_kn_host[pinned], N_k, f_k), "
                       "PYMBAR_B200_CACHE=0 (create + upload + pass + destroy per call)")
        e2e["note"] = "single GPU"
    e2e["pageable_source"] = res.get("pageable")
    e2e["pcie_note"] = "fraction of 63 GB/s (PCIe Gen5 x16 payload ceiling); the step is the 20.48 GB upload"
    try:
        from pymbar_b200.problem import gpu_numa_node

        e2e["gpu_numa_node"] = gpu_numa_node(rig.local)      # pinned staging is allocated with this node preferred
    except Exception:  # pragma: no cover
        pass
    # ---- e2e_solve: the two calls of MBAR.__init__ on a pageable array, itemised ---------------------
    e2e_solve = None
    if args.e2e_solve and not rig.distributed:
        from pymbar_b200 import DeviceProblem

        src = np.empty((K, N_local))
        src[:] = pin.array
        pin.free()
        pin = None
        sws = np.arange(K)
        proto = tuple(dict(s) for s in ms.BOOTSTRAP_SOLVER_PROTOCOL)      # adaptive, min_sc_iter = 0
        t0 = time.perf_counter()
        f_sol = ms.solve_mbar_for_all_states(src, N_k.astype(np.int64), np.zeros(K), sws, proto)
        t_solve_call = time.perf_counter() - t0
        # itemised on an explicit problem (same code path the call above takes)
        t0 = time.perf_counter()
        p2 = DeviceProblem(src, N_k, device=rig.local)
        t_upload = time.perf_counter() - t0
        t0 = time.perf_counter()
        f2, info = p2.solve_adaptive(np.zeros(K), tol=1e-12, min_sc_iter=0)
        f2 = p2.self_consistent_update(f2)
        t_solve = time.perf_counter() - t0
        logw_rows = min(N_local, args.logw_rows)
        t0 = time.perf_counter()
        lw = p2.log_W_nk(f2, rows=logw_rows) if logw_rows < N_local else p2.log_W_nk(f2)
        t_logw = time.perf_counter() - t0
        e2e_solve = {
            "call": "mbar_solvers.solve_mbar_for_all_states(u_kn[pageable numpy], N_k, 0, sws, adaptive) "
                    "(mbar.py:413) and mbar_log_W_nk (mbar.py:455)",
            "solve_call_s": t_solve_call, "upload_s": t_upload, "upload_gbs": 8 * K * N_local / t_upload / 1e9,
            "solve_s": t_solve, "adaptive_iterations": info["iterations"], "solve_device_ms": info["device_ms"],
            "logW_rows": logw_rows, "logW_s": t_logw, "logW_d2h_gbs": 8 * K * logw_rows / t_logw / 1e9,
            "h2d_bytes": 8 * K * N_local, "d2h_bytes_logW": 8 * K * logw_rows,
            "normalisation_check": float(np.max(np.abs(np.exp(lw[:4096]) @ N_k - 1.0))),
        }
        p2.close()
        del src, lw
    if pin is not None:
        pin.free()
    return e2e, e2e_solve


class Watchdog:
    """Safety net for the driver's unattended runs: the line's core (value, roofline, cpu_baseline) is complete a
    few seconds after the timed loop; everything after it is supporting evidence.  If those sections have not
    finished by the deadline (a hung collective on one box must not cost the whole measurement), rank 0 prints what
    it has and every rank exits 0.  Never fires in a healthy run (N=1: ~70 s, N=8: ~200 s)."""

    def __init__(self, rank, deadline_s):
        self.rank, self.line, self.stage = rank, None, "setup"
        self.timer = threading.Timer(deadline_s, self.fire)
        self.timer.daemon = True
        self.timer.start()
        self.deadline_s = deadline_s

    def fire(self):
        if self.rank == 0 and self.line is not None:
            self.line["watchdog"] = (f"sections after the timed measurement did not finish within {self.deadline_s:.0f} s "
                                     f"(stopped in: {self.stage}); core fields are complete")
            print(json.dumps(self.line), flush=True)
        os._exit(0 if (self.line is not None or self.rank != 0) else 3)

    def cancel(self):
        self.timer.cancel()


def run_ours(args):
    rig = Rig()
    world, rank, local = rig.world, rig.rank, rig.local
    distributed = rig.distributed
    dog = Watchdog(rank, float(os.environ.get("BENCH_DEADLINE_S", "480")))

    if args.config != "c3":
        out = {"c1": run_c1, "c2": run_c2, "c4": run_c4, "c5": run_c5}[args.config](rig, args)
        if rank == 0:
            print(json.dumps({"metric": METRIC, "config_line": args.config, "n_gpus": world, "dtype": "f64",
                              "data": "synthetic", "config": out}), flush=True)
        rig.close()
        return

    from pymbar_b200.problem import measure_fp64_peak

    K, N_local = K_STATES, args.n_per_gpu
    N_total = N_local * world
    O_k, k_k = workload_params(K)
    prob, N_k = make_problem(rig, K, N_local, O_k, k_k, args.seed, sharded=True,
                             peer=not os.environ.get("MBAR_B200_NO_PEER"))

    f = np.zeros(K)
    f = prob.sci_iterate(f, args.warmup)                   # W untimed steps (also warms NCCL)
    rig.barrier()
    c0 = prob.counters()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    rig.barrier()
    t0 = time.perf_counter()
    f = prob.sci_iterate(f, args.steps)                    # exactly K timed steps, device resident
    rig.torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    loop = prob.last_loop_ms()                             # CUDA events on the launching stream
    rig.barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives: f_k after the last step (identical on every rank)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "f_k.npy"), np.asarray(f, dtype=np.float64))
    c1 = prob.counters()
    kernel_desc = prob.last_kernels()["pass_kernel"]      # the variant that actually ran in the timed loop

    total_ms, kernel_ms = rig.max_over_ranks([loop["total_ms"], loop["kernel_ms_sum"]])
    ms_per_step = total_ms / args.steps
    value = K * N_total * args.steps / (total_ms * 1e-3)
    kern_ms_per_launch = kernel_ms / args.steps
    peak, peak_src = measured_peak()
    achieved = 8.0 * K * N_local / (kern_ms_per_launch * 1e-3) / 1e9

    # read-only streaming ceiling of the same kernel's memory pipeline (arithmetic skipped), SURVEY 8d
    os.environ["MBAR_B200_FUSED_SKIP"] = "1"
    prob.sci_iterate(np.zeros(K), 3)
    prob.sci_iterate(np.zeros(K), 20)
    del os.environ["MBAR_B200_FUSED_SKIP"]
    ceil_ms = rig.max_over_ranks([prob.last_loop_ms()["kernel_ms_sum"] / 20])[0]
    stream_ceiling = 8.0 * K * N_local / (ceil_ms * 1e-3) / 1e9

    line = None
    if rank == 0:
        cpu_val, cpu_step, n_sample = time_cpu_reference(K, budget_s=args.cpu_budget, steps=2, warmup=1)
        traffic = ncu_traffic(K, N_local)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "iter_per_s": 1e3 / ms_per_step,
            "hbm_gbs_per_gpu": 8.0 * K * N_local / (ms_per_step * 1e-3) / 1e9,
            "config": {"workload": "MBAR self-consistent iteration (Eq. C3), synthetic harmonic u_kn, "
                                   "K=256, N=1e7 per GPU, fp64, device-resident, samples sharded over GPUs",
                       "K": K, "N_per_gpu": N_local, "N_total": N_total, "seed": args.seed,
                       "parallelism": f"sample-sharded x{world}; per iteration the {K + 2} partial sums are exchanged "
                                      + ("inside the pass kernel over NVLink peer memory (rank-ordered sum)"
                                         if (distributed and not os.environ.get("MBAR_B200_NO_PEER")) else
                                         "by one NCCL all-reduce" if distributed else "n/a (1 GPU)"),
                       "l2": "inputs (20.48 GB per GPU) far larger than the 126 MB L2; no flush needed",
                       "timing": "CUDA events on the launching stream around the K-step loop, max over ranks",
                       "wall_s_rank0": wall},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic[0] if traffic else None,
                         "traffic_source": traffic[1] if traffic else None,
                         "kernel": kernel_desc,
                         "algorithmic_bytes_per_launch": 8 * K * N_local,
                         "launch_ms": kern_ms_per_launch, "peak_source": peak_src,
                         "stream_ceiling_gbs": stream_ceiling,
                         "frac_of_stream_ceiling": achieved / stream_ceiling,
                         "stream_ceiling_how": "same kernel with the arithmetic skipped (MBAR_B200_FUSED_SKIP=1): "
                                               "cp.async.bulk ring + mbarriers only, 20 launches, CUDA events",
                         "how": "per-launch cudaEvent pairs recorded around the kernel inside the timed loop"},
            "cpu_baseline": {"value": cpu_val, "unit": UNIT, "cores": 1, "kind": "port",
                             "host_cpus": os.cpu_count(),
                             "c_port_all_threads": time_c_port(K),
                             "sample": f"numpy oracle self_consistent_update on K={K}, N={n_sample} of the same "
                                       f"family ({cpu_step:.2f} s/step); reference is single-threaded numpy"},
            "gpu_launches": c1["launches"] - c0["launches"],
            "clocks": clocks,
        }
    dog.line = line
    dog.stage = "parity_multi_rank"
    # multi-rank parity, visible to the driver (N > 1)
    parity_mr = multi_rank_parity(rig, prob, f, K) if distributed else None
    if line is not None:
        line["parity_multi_rank"] = parity_mr
    dog.stage = "roofline_hessian / adaptive_solve"

    # the Newton half of C3: Hessian roofline + adaptive solve (device-resident vs host-stepped), not timed above
    fp64_peak = measure_fp64_peak(local)
    roof_h = hessian_roofline(prob, K, N_local, fp64_peak, kern_ms_per_launch) if not distributed else None
    rig.barrier()
    if not distributed:
        adaptive_c3, f_solved = adaptive_report(prob, K, "C3 K=256 N=1e7", maxiter=100)
        adaptive_solve = dict(adaptive_c3["device"])
        adaptive_solve["stepped_device_ms"] = adaptive_c3["stepped"]["device_ms"]
        adaptive_solve["kernels"] = adaptive_c3["kernels"]
        adaptive_solve["hessian_ms"] = adaptive_c3["hessian_ms"]
    else:
        t0 = time.perf_counter()
        f_solved, info = prob.solve_adaptive(np.zeros(K), tol=1e-12, maxiter=100, min_sc_iter=0)
        adaptive_solve = {k: info[k] for k in ("success", "iterations", "nr_iterations", "sci_iterations", "passes",
                                               "hessian_passes", "gnorm", "device_ms")}
        adaptive_solve["wall_s"] = time.perf_counter() - t0

    if line is not None:
        line["roofline_hessian"] = roof_h
        line["adaptive_solve"] = adaptive_solve
    dog.stage = "parity spot check / e2e"
    # parity spot check of the timed state against the CPU oracle on a slice (not timed)
    parity = None
    if rank == 0:
        from oracle import mbar_oracle as orc
        from pymbar_b200 import DeviceProblem

        sl = prob.download(0, 4096)
        try:
            p2 = DeviceProblem(sl, N_k, device=local)
            Sdev, _, _ = p2.streaming_pass(f)
            S_ref, _ = orc.single_pass_sums(sl, N_k, f)
            parity = float(np.max(np.abs(Sdev - S_ref) / S_ref))
            p2.close()
        except Exception as exc:  # pragma: no cover
            parity = f"failed: {exc}"

    # ---- e2e legs (close the resident problem first) ---------------------------------------------------
    if line is not None:
        line["parity_S_rel_err_vs_oracle_slice"] = parity
    dog.stage = "e2e"
    e2e, e2e_solve = (None, None)
    if args.e2e_steps > 0:
        e2e, e2e_solve = e2e_legs(rig, args, prob, K, N_local, N_k)
    else:
        prob.close()
    if line is not None:
        line["e2e"] = e2e
        line["e2e_solve"] = e2e_solve
    import pymbar_b200

    pymbar_b200.trim()

    # ---- the other BASELINE configs, briefly (full detail: --config c1|c2|c4|c5) ------------------------
    configs = {}
    if line is not None:
        line["configs"] = configs
    if args.extra_configs:
        for name, fn in (("c1", run_c1), ("c2", run_c2), ("c4", run_c4), ("c5", run_c5)):
            dog.stage = f"configs.{name}"
            try:
                configs[name] = fn(rig, args)
            except Exception as exc:  # pragma: no cover
                configs[name] = {"failed": repr(exc)[:300]}
            pymbar_b200.trim()

    dog.stage = "done"
    dog.cancel()
    if rank == 0:
        # key order of the driver contract first, supporting evidence after
        order = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                 "vs_baseline", "dtype", "data", "iter_per_s", "hbm_gbs_per_gpu", "config", "roofline",
                 "roofline_hessian", "cpu_baseline", "e2e", "e2e_solve", "adaptive_solve", "gpu_launches", "clocks",
                 "parity_S_rel_err_vs_oracle_slice", "parity_multi_rank", "configs"]
        print(json.dumps({k: line.get(k) for k in order}), flush=True)
    rig.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=["c1", "c2", "c3", "c4", "c5"],
                    help="c3 (default) = BASELINE metric line with the other configs summarised under `configs`; "
                         "c2 / c4 / c5 = that BASELINE.json config alone, in detail")
    ap.add_argument("--n-per-gpu", type=int, default=N_PER_GPU)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-pageable-steps", type=int, default=2)
    ap.add_argument("--no-e2e-solve", dest="e2e_solve", action="store_false")
    ap.add_argument("--logw-rows", type=int, default=2_000_000,
                    help="rows of Log_W_nk downloaded in the e2e_solve leg (host memory: 8*K bytes each)")
    ap.add_argument("--no-extra-configs", dest="extra_configs", action="store_false")
    ap.add_argument("--no-c5-hessian", dest="c5_hessian", action="store_false")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write f_k after the last timed step as DIR/f_k.npy (float64; c3 workload of --impl ours); "
                         "the seeded inputs make it comparable between builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "c3"):
        ap.error("--dump-outputs applies to the default workload (--impl ours --config c3)")
    args.warmup = max(args.warmup, 3)
    world = env_int("WORLD_SIZE", 1)
    if args.gpus > 1 and world == 1 and args.impl == "ours":
        # convenience: relaunch under torchrun when called directly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), __file__] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
