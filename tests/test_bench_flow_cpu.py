"""Control-flow test of bench.py's repo arm without a GPU: the process plumbing (Rig), the device problem and the
mirror are replaced by shape-correct stand-ins, so every section of the default line and of `--config c1..c5` runs
end to end on CPU and the emitted JSON can be checked for the keys the driver parses.  Numbers are meaningless here;
what is tested is that no section raises and that the watchdog / key bookkeeping is consistent."""
import io
import json
import os
import sys
import types
from contextlib import redirect_stdout

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


class FakeProblem:
    def __init__(self, u_kn, N_k, device=0, N_local=None):
        self.N_k = np.asarray(N_k, float)
        self.K = len(self.N_k)
        self.N = int(u_kn.shape[1] if u_kn is not None else N_local)
        self._polls = 0
        self._mode = "device"

    def close(self): pass
    def __enter__(self): return self
    def __exit__(self, *a): pass
    def synthesize(self, *a, **k): pass
    def upload(self, u): pass
    def comm_init(self, *a): pass
    def peer_export(self): return b"x" * 64
    def peer_attach(self, *a): pass
    @staticmethod
    def comm_unique_id(): return b"i" * 128
    def sci_iterate(self, f, iters): return np.array(f, float)
    def last_loop_ms(self): return dict(total_ms=1.0, kernel_ms_sum=0.9, iters=1)
    def counters(self): return dict(launches=10, passes=10, h2d_bytes=0, d2h_bytes=0)
    def last_kernels(self): return dict(pass_kernel="pass_fused_kernel<fake, M=2>", hessian_kernel="hessian_fake")
    def last_pass_ms(self): return 0.5
    def last_hessian_ms(self): return dict(weights_ms=0.0, hessian_ms=2.0)
    def hessian(self, f): return np.eye(self.K)
    def pass_multi(self, f2): return np.ones_like(f2), np.zeros(len(f2))
    def streaming_pass(self, f, want_G=False): return np.ones(self.K), -1.0, None
    def self_consistent_update(self, f): return np.array(f, float)
    def set_loop_mode(self, mode="device", batch=0): self._mode = mode
    def loop_stats(self): return dict(polls=self._polls, mode=self._mode, batch=4, graph_captures=1, graph_launches=4)
    def solve_adaptive(self, f, tol=1e-12, maxiter=100, min_sc_iter=0, gamma=1.0):
        self._polls += 2
        return np.array(f, float), dict(success=1, iterations=5, nr_iterations=4, sci_iterations=1, passes=10,
                                        hessian_passes=5, max_delta=1e-13, gnorm=1e-9, device_ms=3.0)
    def download(self, n0=0, n=None, out=None):
        n = self.N - n0 if n is None else n
        if out is not None:
            out[:] = 1.0
            return out
        rng = np.random.RandomState(0)
        return rng.rand(self.K, n) * 3
    def log_W_nk(self, f, rows=None, **k):
        n = self.N if rows is None else rows
        return np.full((n, self.K), -np.log(self.N_k.sum()))


class FakePinned:
    def __init__(self, shape):
        assert shape[0] * shape[1] <= 1 << 22, "the flow test runs with a tiny --n-per-gpu"
        self.array = np.zeros(shape)
    def free(self): pass


class FakeDist:
    def __init__(self, world): self.world = world
    def all_gather_object(self, out, obj, group=None):
        for i in range(len(out)): out[i] = obj
    def broadcast_object_list(self, box, src=0, group=None): pass
    def barrier(self): pass


class FakeTorch:
    class cuda:
        @staticmethod
        def synchronize(): pass


def _run(monkeypatch, argv, world):
    import bench
    import pymbar_b200
    from pymbar_b200 import mbar_solvers as ms
    from pymbar_b200 import problem as prob_mod

    class FakeRig:
        def __init__(self):
            self.torch, self.dist = FakeTorch, FakeDist(world)
            self.world, self.rank, self.local = world, 0, 0
            self.distributed = world > 1
        def barrier(self): pass
        def max_over_ranks(self, v): return list(v)
        def attach(self, p, peer=True): pass
        def close(self): pass

    monkeypatch.setattr(bench, "Rig", FakeRig)
    monkeypatch.setattr(pymbar_b200, "DeviceProblem", FakeProblem)
    monkeypatch.setattr(pymbar_b200, "PinnedArray", FakePinned)
    monkeypatch.setattr(pymbar_b200, "trim", lambda: None)
    monkeypatch.setattr(prob_mod, "measure_fp64_peak", lambda dev=0: (37.0, 33.0))
    monkeypatch.setattr(prob_mod, "gpu_numa_node", lambda dev=0: 0)
    monkeypatch.setattr(ms, "self_consistent_update", lambda u, N, f, *a: np.zeros(len(N)))
    monkeypatch.setattr(ms, "solve_mbar_for_all_states", lambda u, N, f, sws, proto: np.zeros(len(N)))
    monkeypatch.setattr(ms, "clear_cache", lambda: None)
    monkeypatch.setattr(bench, "time_cpu_reference", lambda K, budget_s, steps, warmup: (1.0e7, 1.0, 1000))
    monkeypatch.setattr(bench, "time_c_port", lambda K, n_sample=0: {"value": 1.0e8})
    monkeypatch.setattr(bench, "ClockSampler", lambda idx: types.SimpleNamespace(start=lambda: None, stop=lambda: {"sm_mhz": 1.0}))
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    monkeypatch.setenv("WORLD_SIZE", str(world))
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    lines = [ln for ln in buf.getvalue().splitlines() if ln.startswith("{")]
    assert len(lines) == 1, buf.getvalue()[-2000:]
    return json.loads(lines[0])


@pytest.mark.parametrize("world", [1, 2])
def test_default_line_has_every_key_the_driver_reads(monkeypatch, world):
    d = _run(monkeypatch, ["--gpus", str(world), "--steps", "3", "--warmup", "3", "--n-per-gpu", "2048"], world)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks",
                "adaptive_solve", "configs"):
        assert key in d and (d[key] is not None or key == "vs_baseline"), key
    assert d["n_gpus"] == world and d["steps"] == 3 and d["dtype"] == "f64" and d["config"]["workload"]
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic", "kernel"}
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert set(d["configs"]) == {"c1", "c2", "c4", "c5"}
    assert not any("failed" in v for v in d["configs"].values()), d["configs"]
    if world > 1:
        assert d["parity_multi_rank"] is not None and "bit_identical_f_across_ranks" in d["parity_multi_rank"]
    else:
        assert d["roofline_hessian"]["frac"] > 0 and d["e2e_solve"] is not None
    assert "watchdog" not in d


def test_dump_outputs_writes_f_after_the_timed_steps(monkeypatch, tmp_path):
    # each stand-in iteration adds 1 to f: the dumped f_k counts warm-up + timed iterations of the main problem
    monkeypatch.setattr(FakeProblem, "sci_iterate", lambda self, f, iters: np.asarray(f, float) + iters)
    out = tmp_path / "dump"
    d = _run(monkeypatch, ["--steps", "7", "--warmup", "3", "--n-per-gpu", "2048", "--dump-outputs", str(out)], 1)
    assert d["steps"] == 7
    f = np.load(out / "f_k.npy")
    assert f.dtype == np.float64 and f.shape == (256,)
    np.testing.assert_array_equal(f, 10.0)
    assert sorted(os.listdir(out)) == ["f_k.npy"]


@pytest.mark.parametrize("cfg", ["c1", "c2", "c4", "c5"])
def test_single_config_lines(monkeypatch, cfg):
    d = _run(monkeypatch, ["--config", cfg], 1)
    assert d["config_line"] == cfg and d["config"]["workload"].startswith(cfg.upper())


def test_watchdog_prints_the_core_line_and_exits_zero():
    """A supporting section that never returns must not cost the measurement: after the deadline rank 0 prints the
    core line (with a `watchdog` note) and the process exits 0; ranks without a line exit 0 silently."""
    import subprocess

    code = ("import sys, time; sys.path.insert(0, %r); import bench; "
            "d = bench.Watchdog(int(sys.argv[1]), 0.4); "
            "d.line = {'metric': 'm', 'value': 1.0} if sys.argv[2] == 'line' else None; d.stage = 'e2e'; time.sleep(30)" % ROOT)
    out = subprocess.run([sys.executable, "-c", code, "0", "line"], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["value"] == 1.0 and "e2e" in d["watchdog"]
    out = subprocess.run([sys.executable, "-c", code, "3", "noline"], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and out.stdout.strip() == ""
    out = subprocess.run([sys.executable, "-c", code, "0", "noline"], capture_output=True, text=True, timeout=60)
    assert out.returncode == 3          # rank 0 with nothing measured: a failure, not a silent success
