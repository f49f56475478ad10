"""bench.py host logic without a GPU: run_ours() is driven with stand-ins for torch / torch.distributed and an engine
double built on the CPU oracle, so that a Python-level mistake (wrong name, wrong keyword, a rank-dependent code path,
a broken parity check) in the measurement script shows up on the CPU instead of costing a GPU run.  Nothing here
measures anything; the JSON line's shape and the in-bench parity check are what is checked."""
import ctypes
import importlib
import io
import json
import os
import sys
import types
from contextlib import redirect_stdout

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REC = 144


def mem(ptr, nbytes):
    return np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(ptr))


class FakeTensor:
    """A numpy-backed stand-in for the few torch.Tensor methods bench.py touches."""
    def __init__(self, arr):
        self.a = arr
        self.device = types.SimpleNamespace(index=0)
    def pin_memory(self): return self
    def reshape(self, *a): return FakeTensor(self.a.reshape(*a))
    def data_ptr(self): return self.a.ctypes.data
    def numel(self): return self.a.size
    def element_size(self): return self.a.itemsize
    def is_contiguous(self): return True
    def copy_(self, other): self.a[...] = other.a; return self
    def item(self): return self.a.reshape(-1)[0].item()
    def cpu(self): return self
    def numpy(self): return self.a
    def __getitem__(self, k): return FakeTensor(self.a[k])
    def __setitem__(self, k, v): self.a[k] = v.a if isinstance(v, FakeTensor) else v


class FakeEvent:
    def __init__(self, enable_timing=False): pass
    def record(self): pass
    def elapsed_time(self, other): return 1.0


NP = {"u8": np.uint8, "i32": np.int32, "i64": np.int64, "f64": np.float64, None: np.float32}


def fake_torch(world):
    t = types.ModuleType("torch")
    t.uint8, t.int32, t.int64, t.float64 = "u8", "i32", "i64", "f64"
    t.device = lambda kind, idx=0: types.SimpleNamespace(type=kind, index=idx)
    t.empty = lambda n, dtype=None, device=None: FakeTensor(np.zeros(n, dtype=NP[dtype]))
    t.zeros = t.empty
    t.zeros_like = lambda x: FakeTensor(np.zeros_like(x.a))
    t.empty_like = t.zeros_like
    t.tensor = lambda v, device=None, dtype=None: FakeTensor(np.array(v, dtype=NP[dtype]))
    cuda = types.ModuleType("torch.cuda")
    cuda.is_available = lambda: True
    cuda.set_device = lambda i: None
    cuda.synchronize = lambda: None
    cuda.Event = FakeEvent
    cuda.Stream = lambda device=None: types.SimpleNamespace(cuda_stream=0x1234, synchronize=lambda: None)
    cuda.set_stream = lambda s: None
    cuda.current_stream = lambda: types.SimpleNamespace(cuda_stream=0x1234, synchronize=lambda: None)
    t.cuda = cuda
    dist = types.ModuleType("torch.distributed")
    dist.calls = []
    dist.ReduceOp = types.SimpleNamespace(MAX="max", MIN="min")
    dist.init_process_group = lambda backend, device_id=None: dist.calls.append("init")
    dist.all_reduce = lambda tensor, op=None: dist.calls.append(("all_reduce", op))
    dist.barrier = lambda: dist.calls.append("barrier")
    dist.destroy_process_group = lambda: dist.calls.append("destroy")
    dist.get_world_size = lambda: world
    dist.get_rank = lambda: 0

    def all_gather(outs, x):                       # every "rank" contributed what rank 0 did
        for o in outs:
            o.a[...] = x.a
    def gather(x, outs, dst=0):                    # rank 0 holds everything, the other ranks nothing
        for i, o in enumerate(outs):
            o.a[...] = x.a if i == 0 else 0
    dist.all_gather, dist.gather = all_gather, gather
    t.distributed = dist
    return t, cuda, dist


class FakeEngine:
    """The engine's Python surface on top of the CPU oracle (generator twin + Accounter)."""
    def __init__(self, max_entries, device=0, max_batch=0, cuda_stream=None, flags=0, **kw):
        assert cuda_stream, "bench must hand the engine an explicit stream"
        self.launches, self.acc, self.gens = 0, O.ShardedAccounter(2), {}
    def gen_records(self, gp, first, n, dst):
        key = (gp.seed, gp.n_keys, gp.dist)
        if key not in self.gens:
            self.gens[key] = O.Gen(gp.seed, gp.n_keys, dist=gp.dist, zipf_s_milli=gp.zipf_s_milli, t0_ns=gp.t0_ns)
        self.gens[key].records(first, n, out=dst.a[: n * REC])
    def sync(self): pass
    def ingest(self, ptr, n):
        self.launches += 3
        self.acc.account(mem(ptr if isinstance(ptr, int) else ptr.data_ptr(), n * REC))
        return 0, n
    def ingest_events(self, ptr, n):
        ev = mem(ptr, n * 64).reshape(-1, 64)
        r = np.zeros((n, REC), dtype=np.uint8)
        r[:, 0:40], r[:, 40:48], r[:, 48:56], r[:, 56:60] = ev[:, 0:40], ev[:, 40:48], ev[:, 40:48], ev[:, 48:52]
        r[:, 64] = 1
        self.acc.account(r)
        self.launches += 4
        return 0, n
    def live_flows(self): return len(self.acc)
    def evict_into(self, out, cap):
        r = self.acc.evict()
        assert len(r) <= cap
        mem(out if isinstance(out, int) else out.data_ptr(), r.size)[...] = r.reshape(-1)
        return len(r)
    def stats(self): return {"kernel_launches": self.launches, "order_fixups": 0, "spills": 0}
    def close(self): pass


class FakeAgg:
    """N ranks folded into one: everything goes to the owner engine (the key sets would be disjoint)."""
    def __init__(self, eng, max_batch, dev, **kw):
        self.eng, self.local, self.exchanged_records = eng, FakeEngine(1, cuda_stream=1), 0
        self.locals = [self.local]
    def ingest(self, records, n):
        self.eng.ingest(records if isinstance(records, int) else records.data_ptr(), n); return 0
    def flush(self): return 0
    def reset_local(self): pass
    def exchange_stats(self): return {"nvlink_bytes_per_step_rank0": 0}
    def close(self): pass


def run_bench(monkeypatch, world, argv):
    torch, cuda, dist = fake_torch(world)
    monkeypatch.setitem(sys.modules, "torch", torch)
    monkeypatch.setitem(sys.modules, "torch.cuda", cuda)
    monkeypatch.setitem(sys.modules, "torch.distributed", dist)
    import netobserv_ebpf_agent_b200 as fa
    monkeypatch.setattr(fa, "FlowAggEngine", FakeEngine)
    sharded = types.ModuleType("netobserv_ebpf_agent_b200.sharded")
    sharded.PeerShardedAggregator = FakeAgg
    sharded.ShardedAggregator = FakeAgg
    monkeypatch.setitem(sys.modules, "netobserv_ebpf_agent_b200.sharded", sharded)
    monkeypatch.setenv("WORLD_SIZE", str(world)); monkeypatch.setenv("RANK", "0"); monkeypatch.setenv("LOCAL_RANK", "0")
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    sys.path.insert(0, ROOT)
    bench = importlib.import_module("bench")
    bench = importlib.reload(bench)
    monkeypatch.setattr(bench.ClockSampler, "start", lambda self: None)
    monkeypatch.setattr(bench.ClockSampler, "stop", lambda self: {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "samples": 9, "reasons": []})
    monkeypatch.setattr(bench.time, "sleep", lambda s: None)
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    lines = [ln for ln in buf.getvalue().splitlines() if ln.startswith("{")]
    assert len(lines) == 1, buf.getvalue()
    return json.loads(lines[0]), dist


CONTRACT_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                 "vs_baseline", "dtype", "data", "config", "roofline", "gpu_launches", "clocks", "e2e")
SMALL = ["--steps", "3", "--warmup", "3", "--e2e-steps", "2", "--batch", "8192", "--max-batch", "4096", "--mgpu-round", "4096",
         "--e2e-batch", "2048", "--verify-records", "30000", "--cpu-sample", "20000", "--workload", "zipf1m"]


def test_single_gpu_line_has_every_contract_key_and_the_parity_check_runs(monkeypatch):
    line, _ = run_bench(monkeypatch, 1, SMALL)
    for k in CONTRACT_KEYS + ("cpu_baseline", "parity_checked"):
        assert k in line, k
    assert line["n_gpus"] == 1 and "1M Zipf" in line["config"]["workload"]
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(line["roofline"])
    assert line["e2e"]["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["e2e"]["events_row"]["value"] > 0 and line["e2e"]["events_row"]["h2d_bytes_per_step"] * 9 == line["e2e"]["h2d_bytes_per_step"] * 4
    assert line["gpu_launches"] > 0
    assert line["parity_ok"] and line["parity_checked"] == line["flows_oracle"] > 1000
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] > 0


def test_default_workload_is_the_10m_flow_headline(monkeypatch):
    argv = [a for a in SMALL if a not in ("--workload", "zipf1m")] + ["--no-cpu"]
    line, _ = run_bench(monkeypatch, 1, argv)
    assert line["config"]["workload_key"] == "zipf10m" and line["config"]["flows"] == 10_000_000
    assert line["config"]["table_slots"] == 1 << 25 and line["config"]["full_cut"].startswith("on")
    assert line["parity_ok"]


def test_dump_outputs_holds_what_the_timed_steps_folded(monkeypatch, tmp_path):
    """--dump-outputs: the flows of warmup + --steps batches (all of them: they fit the sample), as float32 records;
    the same arguments write the same files."""
    argv = SMALL + ["--no-cpu", "--no-verify", "--no-e2e", "--steps", "2", "--warmup", "1"]
    line, _ = run_bench(monkeypatch, 1, argv + ["--dump-outputs", str(tmp_path / "a")])
    run_bench(monkeypatch, 1, argv + ["--dump-outputs", str(tmp_path / "b")])
    flows = np.load(tmp_path / "a" / "flows.npy")
    assert flows.dtype == np.float32 and flows.shape == (line["config"]["live_flows"], REC)
    assert np.load(tmp_path / "a" / "live_flows.npy").tolist() == [line["config"]["live_flows"]]
    assert np.array_equal(flows, np.load(tmp_path / "b" / "flows.npy"))
    recs = np.ascontiguousarray(flows.astype(np.uint8)).view(O.REC_DTYPE).reshape(-1)
    assert int(recs["packets"].sum()) == (1 + 2) * 8192


@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_multi_gpu_line_and_matched_collectives(monkeypatch, exchange):
    line, dist = run_bench(monkeypatch, 2, SMALL + ["--gpus", "2", "--exchange", exchange])
    for k in CONTRACT_KEYS[:-1]:
        assert k in line, k
    assert line["n_gpus"] == 2 and "cpu_baseline" not in line          # CPU baseline only at N=1
    if exchange == "peer":
        assert line["e2e"]["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 2 * line["e2e"]["records_per_step"] // 2 * 144
        assert ("all_reduce", "min") in dist.calls                     # go/no-go agreed by all ranks before the e2e loop
    else:
        assert "e2e" not in line
    assert dist.calls[0] == "init" and dist.calls[-1] == "destroy"


def test_reference_arm_prints_the_same_config_and_never_loads_the_product(monkeypatch):
    """--impl reference in a fresh interpreter: same `config` as the GPU arm, product library not loaded."""
    import subprocess
    code = ("import sys, json; sys.argv=['bench.py','--impl','reference','--steps','2','--warmup','1','--ref-sample','20000',"
            "'--workload','zipf1m','--batch','8192']; sys.path.insert(0, %r); import bench; bench.main(); "
            "print('LOADED', any('libflowagg' in l for l in open('/proc/self/maps')), 'netobserv_ebpf_agent_b200' in sys.modules)" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.strip().splitlines()
    ref = json.loads(lines[0])
    assert lines[-1] == "LOADED False False"
    assert ref["impl"] == "reference" and ref["cpu_baseline"]["kind"] == "port" and ref["value"] > 0
    assert ref["e2e"]["h2d_bytes_per_step"] == 0
    ours, _ = run_bench(monkeypatch, 1, SMALL + ["--no-cpu", "--no-verify"])
    ours_cfg = {k: v for k, v in ours["config"].items() if k in ref["config"]}
    assert ours_cfg == ref["config"]
