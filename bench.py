#!/usr/bin/env python
"""bench.py — flow-aggregation throughput on B200 (contract: the task prompt; measurement notes: DESIGN.md §7).

A "step" is one pass of the hot path (K1 flow_aggregate, reached through fa_ingest of the C ABI) over one batch of
synthetic 144-byte flow records that is already resident in HBM.  Workloads (BASELINE.json):
  zipf10m    the configuration the metric is quoted on ("@10M 5-tuples"): 10 M Zipf-1.1 5-tuples (default)
  uniform10m worst case for table locality: 10 M uniform 5-tuples
  zipf1m     configs[1]: 1 M Zipf-1.1 5-tuples
One JSON line on stdout (rank 0).  After the timed loop the engine's output is checked against the CPU oracle on a
fresh prefix of the same stream (`parity_checked` = flows compared bit for bit; --no-verify skips it).
--dump-outputs DIR writes what the timed steps computed (see dump_outputs()); the inputs depend on the arguments only,
so two builds run with the same arguments can be compared output for output.
--impl reference times the CPU restatement of pkg/flow.Accounter (the Go reference cannot be built in this image) on
a bounded sample of the same workload; that arm never loads the product library.
"""
import argparse
import datetime
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

REC = 144
# flow cache sizing per workload: max_entries = 0.75 x 2^k gets exactly 2^k table slots (SURVEY.md §8d: 2^25 slots for
# the 10 M-flow configurations = load 0.30, 2^21 for 1 M flows = load 0.48)
WORKLOADS = {
    "zipf10m": dict(n_keys=10_000_000, dist=1, seed=2, max_entries=3 << 23, no_full_cut=False,
                    label="synthetic record stream, 10M Zipf-1.1 5-tuples (BASELINE metric: '@10M 5-tuples')"),
    "uniform10m": dict(n_keys=10_000_000, dist=0, seed=2, max_entries=3 << 23, no_full_cut=False,
                       label="synthetic record stream, 10M uniform 5-tuples (worst-case table locality)"),
    # 1 M flows in 2^21 slots leave room for 0.57 M new flows only: every 2^22-record launch "could" overflow the cache,
    # so this workload runs the table as a plain map (FA_F_NO_FULL_CUT: max_entries only sizes it)
    "zipf1m": dict(n_keys=1_000_000, dist=1, seed=2, max_entries=3 << 19, no_full_cut=True,
                   label="synthetic record stream, 1M Zipf-1.1 5-tuples (BASELINE configs[1])"),
    # BASELINE configs[2]: the fused count-min (w = 2^20, d = 4) + HyperLogLog (p = 14) update inside K1, 100 M-key universe
    # (a 2^27-record step touches ~7 M of them; the exact table stays on as a plain map so that the same run checks flows,
    # sketch tables bit for bit against the CPU restatement, and the (eps, delta) / 3-sigma bounds against exact counts)
    "sketch100m": dict(n_keys=100_000_000, dist=1, seed=3, max_entries=3 << 25, no_full_cut=True,
                       sketch=dict(cms_log2_width=20, cms_depth=4, hll_precision=14, sketch_seed=0x5EED),
                       label="synthetic record stream, 100M Zipf-1.1 5-tuples, K1 with the fused count-min (w=2^20, d=4) + "
                             "HLL (p=14) update (BASELINE configs[2])"),
}
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_dram_traffic.json")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload):
    """DRAM bytes per record of K1 from the committed ncu --set full capture of this workload (profiles/), or None."""
    try:
        return json.load(open(TRAFFIC_FILE)).get(workload)
    except Exception:
        return None


def make_config(args, wl, world):
    """The workload description both arms print (identical keys and values for the same command line)."""
    return {"workload": wl["label"], "workload_key": args.workload, "flows": wl["n_keys"], "record_bytes": REC,
            "records_per_step_per_gpu": args.batch, "max_entries": wl["max_entries"],
            "table_slots": 1 << (4 * wl["max_entries"] // 3 - 1).bit_length(),
            "full_cut": "off (FA_F_NO_FULL_CUT)" if (wl["no_full_cut"] or world > 1) else "on (Accounter maxEntries rule)",
            "l2_policy": f"inputs larger than L2 ({args.batch * REC / 1e6:.0f} MB per step)", "n_gpus": world}


class ClockSampler:
    """nvidia-smi samples with timestamps; only samples inside the timed window are kept."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.p, self.t0, self.t1 = index, None, None, None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def window_begin(self):
        self.t0 = datetime.datetime.now()

    def window_end(self):
        self.t1 = datetime.datetime.now()

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, near, reasons = [], [], [], set()
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f")
                s, m = float(f[1]), float(f[2])
            except ValueError:
                continue
            inside = self.t0 is None or (self.t0 <= ts <= self.t1)
            if not inside:
                if self.t0 is not None and abs((ts - self.t0).total_seconds()) < 0.5:
                    near.append(s)
                continue
            sm.append(s); mx.append(m)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm and near:                              # window shorter than the sampling period
            sm = near
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window_ms": None if self.t0 is None else (self.t1 - self.t0).total_seconds() * 1e3,
                "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- CPU legs (oracle = checker / baseline)
def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def oracle_gen(wl):
    import oracle_lib as O
    return O.Gen(wl["seed"], wl["n_keys"], dist=wl["dist"], zipf_s_milli=1100, t0_ns=1_000_000, varying_desc=0)


def cpu_baseline_port(wl, sample_records, passes=4):
    """Single-thread CPU restatement of pkg/flow.Accounter (one goroutine in the reference)."""
    import oracle_lib as O
    g = oracle_gen(wl)
    sample = g.records(0, sample_records, threads=min(16, host_threads()))
    acc = O.Accounter(1 << 26)
    t0 = time.perf_counter()
    for _ in range(passes):                          # ~10-20 s of CPU work: the same slice folded `passes` times
        acc.account(sample)
    flows = len(acc)
    acc.evict()
    dt = time.perf_counter() - t0
    acc.close(); g.close()
    return {"value": passes * sample_records / dt / 1e6, "unit": "Mpkts/s", "cores": 1, "kind": "port",
            "sample": f"{passes} x {sample_records} records of the same stream, {flows} flows, incl. the final evict "
                      f"(CPU restatement of pkg/flow.Accounter; Go toolchain unavailable)", "seconds": dt}


def run_reference(args, wl):
    """--impl reference: the reference's CPU path for this step (Accounter restatement), all host threads.  Loads
    only oracle/ — never the product library."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:                                    # under torchrun only rank 0 runs the CPU arm
        return
    import oracle_lib as O
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    avail = host_threads()
    n = args.ref_sample
    g = oracle_gen(wl)
    ring = [g.records(i * n, n, threads=avail) for i in range(2)]          # inputs resident in host memory, like HBM for the GPU arm

    # "all the host threads it can use": containers often expose more CPUs than they may run on, so pick the thread
    # count that is actually fastest on this box (tried once each, outside the timed region)
    best, cores = None, avail
    for tcount in sorted({avail, max(1, avail // 2), max(1, avail // 4), min(avail, 16), min(avail, 8)}, reverse=True):
        acc = O.ShardedAccounter(tcount)
        acc.account(ring[0])                                               # builds the maps
        t0 = time.perf_counter(); acc.account(ring[1]); dt = time.perf_counter() - t0
        acc.close()
        if best is None or dt < best:
            best, cores = dt, tcount
    acc = O.ShardedAccounter(cores)                                        # persistent maps: steady state like the GPU arm
    for i in range(max(args.warmup, 1)):
        acc.account(ring[i % 2])
    t0 = time.perf_counter()
    for i in range(args.steps):
        acc.account(ring[i % 2])
    dt = time.perf_counter() - t0
    flows = len(acc)
    acc.close(); g.close()
    v = n * args.steps / dt / 1e6
    line = {"impl": "reference", "metric": "Mpkts/s aggregated", "value": v, "unit": "Mpkts/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64/u32 integer (add/or/min/max); no floating point",
            "data": "synthetic", "config": make_config(args, wl, world),
            "cpu_baseline": {"value": v, "unit": "Mpkts/s", "cores": cores, "kind": "port",
                             "sample": f"{n} records per step of the same stream ({flows} flows live), key-sharded over "
                                       f"{cores} threads, each a private persistent Accounter map (CPU restatement of "
                                       "pkg/flow.Accounter; Go toolchain unavailable)"},
            "e2e": {"value": v, "unit": "Mpkts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def record_order(r):
    """Permutation that sorts (n,144) records by two independent 64-bit hashes of their 40-byte keys."""
    k = np.ascontiguousarray(r[:, :40]).view("<u8")
    c = np.array([0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F, 0x165667B19E3779F9, 0xD6E8FEB86659FD93, 0xFF51AFD7ED558CCD], dtype=np.uint64)
    with np.errstate(over="ignore"):
        h1 = (k * c).sum(axis=1, dtype=np.uint64)
        h2 = ((k ^ (k >> np.uint64(29))) * c[::-1]).sum(axis=1, dtype=np.uint64)
    return np.lexsort((h2, h1))


DUMP_FLOWS = 1 << 15           # --dump-outputs: 32768 flows x 144 bytes as float32 = 18.9 MB (+ 32 MB of count-min)


def dump_outputs(out_dir, recs, sketch=None):
    """--dump-outputs: the flow table the timed steps left, as a caller of fa_evict receives it ((n,144) records; float32
    holds every byte exactly).  A larger table is sampled by key hash: the DUMP_FLOWS flows that come first in
    record_order(), so the sample depends on the flows alone, not on the slots the table keeps them in.  With the
    sketches on, also the count-min table and the HyperLogLog registers (fa_sketch_export)."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"flows": recs[record_order(recs)[:DUMP_FLOWS]].astype(np.float32),
           "live_flows": np.array([len(recs)], dtype=np.float64)}
    if sketch is not None:
        out["cms"], out["hll"] = sketch[0].astype(np.float64), sketch[1].astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def oracle_flows(wl, first, n, chunk=1 << 22, sketch=None):
    """The oracle's flows for records [first, first+n) of the workload stream, sorted like record_order(); with `sketch`
    (the workload's sketch parameters) also the CPU restatement's count-min table and HLL registers over the same records."""
    import ctypes as C
    import oracle_lib as O
    threads = min(host_threads(), 32)
    g = oracle_gen(wl)
    acc = O.ShardedAccounter(threads)
    buf = np.empty(chunk * REC, dtype=np.uint8)
    cms = hll = None
    if sketch:
        cms = np.zeros(sketch["cms_depth"] << sketch["cms_log2_width"], dtype=np.uint64)
        hll = np.zeros(1 << sketch["hll_precision"], dtype=np.uint8)
    done = 0
    while done < n:
        c = min(chunk, n - done)
        r = g.records(first + done, c, threads=threads, out=buf[: c * REC])
        acc.account(r)
        if sketch:
            b = O.as_bytes(r)
            O.lib().oracle_cms_update(cms.ctypes.data_as(C.POINTER(C.c_uint64)), sketch["cms_log2_width"], sketch["cms_depth"],
                                      sketch["sketch_seed"], O._p(b), c)
            O.lib().oracle_hll_update(O._p(hll), sketch["hll_precision"], sketch["sketch_seed"], O._p(b), c)
        done += c
    out = acc.evict()
    acc.close(); g.close()
    out = out[record_order(out)]
    return (out, cms, hll) if sketch else out


# --------------------------------------------------------------------------- GPU arm
def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    import netobserv_ebpf_agent_b200 as fa

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU fallback)")
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs needs a single-GPU run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch                                   # records per step per GPU
    ring = max(1, min(args.ring, args.steps + args.warmup))
    # Everything (engine kernels, NCCL, timing events) runs on ONE explicit torch stream: the legacy default
    # stream has handle 0, which the engine would take as "create your own".
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    if args.max_batch is None:
        args.max_batch = (1 << 24) if wl["no_full_cut"] else (1 << 23)
    max_batch = args.max_batch if world == 1 else args.mgpu_round
    no_cut = wl["no_full_cut"] or world > 1          # N>1: the owner table is a plain map behind the exchange
    eng = fa.FlowAggEngine(wl["max_entries"], device=local, max_batch=max_batch, cuda_stream=stream.cuda_stream,
                           flags=(fa.FA_F_NO_FULL_CUT if no_cut else 0) | (fa.FA_F_ENABLE_SKETCH if wl.get("sketch") else 0),
                           **(wl.get("sketch") or {}))
    # one key universe for the whole job; every rank generates its own slice of the record stream
    gp = fa.GenParams(seed=wl["seed"], n_keys=wl["n_keys"], dist=wl["dist"], zipf_s_milli=1100,
                      t0_ns=1_000_000, varying_desc=0)
    batches = []
    for i in range(ring):
        t = torch.empty(B * REC, dtype=torch.uint8, device=dev)
        for off in range(0, B, 1 << 24):                                   # generator launches of <= 2^24 records
            c = min(1 << 24, B - off)
            eng.gen_records(gp, (i * world + rank) * B + off, c, t[off * REC:])
        batches.append(t)
    eng.sync()

    agg = None
    if world > 1:
        from netobserv_ebpf_agent_b200.sharded import PeerShardedAggregator, ShardedAggregator
        if args.exchange == "peer":
            # local combine (K1+K2) -> K3 fused with the exchange (peer stores over NVLink) -> K1 on the owner
            # the combiner's scratch table holds one round's distinct flows: sized like the single-GPU table of the workload
            # (same load factor, so the local K1 probes like the N=1 run), never more than a round can fill
            agg = PeerShardedAggregator(eng, max_batch, dev, local_entries=min(2 * max_batch, wl["max_entries"]), profile=True)
        else:
            # local combine (K1+K2) -> K3 route -> NCCL all-to-all -> K1 on the owner
            agg = ShardedAggregator(eng, max_batch, dev, combine=not args.no_combine)

    def ingest_dev(ptr, n):
        if world == 1:
            rc, took = eng.ingest(ptr, n)
            assert rc == 0 and took == n, (rc, took)
        else:
            agg.ingest(ptr, n)

    def evict_dev():
        """Lookup-and-delete everything into device memory -> (tensor, flows); re-uses the first input batch when it fits."""
        nfl = eng.live_flows()
        buf = batches[0] if nfl <= B else torch.empty(nfl * REC, dtype=torch.uint8, device=dev)
        got = eng.evict_into(buf.data_ptr(), max(nfl, 1)) if nfl else 0
        assert got == nfl, (got, nfl)
        if agg is not None:
            agg.reset_local()                        # the combiners' cached keys go with the owners' flows
        return buf, nfl

    def finish():                                    # N>1: drain + exchange the batch still in a scratch table
        if world > 1:
            agg.flush()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        ingest_dev(batches[i % ring].data_ptr(), B)
    finish()
    barrier()

    def all_stats():                                 # owner engine + the combiner's scratch engine(s)
        s = eng.stats()
        if world > 1:
            for loc in ([agg.local] if hasattr(agg, "local") else agg.locals):
                ls = loc.stats()
                for k in ("kernel_launches", "order_fixups", "spills"):
                    s[k] += ls[k]
        return s
    st0 = all_stats()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)                              # nvidia-smi needs a moment before its first sample
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    sampler.window_begin()
    ev[0].record()
    for i in range(args.steps):
        ingest_dev(batches[(args.warmup + i) % ring].data_ptr(), B)
        if i == args.steps - 1:
            finish()
        ev[i + 1].record()
    barrier()
    sampler.window_end()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = ev[0].elapsed_time(ev[-1])
    step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    st1 = all_stats()
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = world * B * args.steps / (total_ms / 1e3) / 1e6
    launches = st1["kernel_launches"] - st0["kernel_launches"]
    flows = eng.live_flows()
    if args.dump_outputs:                            # the parity check below starts from an emptied table anyway
        sk = None
        if wl.get("sketch"):
            sp = wl["sketch"]
            sk = eng.sketch_export(sp["cms_log2_width"], sp["cms_depth"], sp["hll_precision"])
        out_dev, nfl = evict_dev()
        dump_outputs(args.dump_outputs, out_dev[: nfl * REC].cpu().numpy().reshape(-1, REC), sk)
    nvlink = agg.exchange_stats() if (world > 1 and hasattr(agg, "exchange_stats")) else None
    if nvlink is not None and getattr(agg, "profile", False):
        rounds_timed = args.steps * ((B + max_batch - 1) // max_batch)
        nvlink["phase_ms_per_round_rank0"] = {k_: round(v, 4) for k_, v in agg.phase_ms(rounds_timed).items()}
        # SURVEY.md 8d config 4: bytes crossing NVLink against the measured 770 GB/s per direction and GPU
        rounds_per_step = max(1, (B + max_batch - 1) // max_batch)
        per_step = nvlink["nvlink_bytes_per_round_rank0"] * rounds_per_step
        nvlink["nvlink_frac_of_770gbs_over_the_step"] = round(per_step / (total_ms / args.steps / 1e3) / 770e9, 4)
        rt = nvlink["phase_ms_per_round_rank0"].get("route", 0.0)
        if rt > 0:
            nvlink["nvlink_frac_of_770gbs_during_route"] = round(nvlink["nvlink_bytes_per_round_rank0"] / (rt / 1e3) / 770e9, 4)

    # ---------------------------------------------------------------- parity: the engine against the CPU oracle
    # Fresh state, then records [V0, V0+V) of the same stream through the same engine / aggregator, evict, compare
    # all flows bit for bit with the oracle's fold of the same records (rank 0; N>1: the ranks' evictions concatenated).
    parity = None
    if not args.no_verify:
        V = args.verify_records - args.verify_records % world
        V0 = 1 << 40                                 # far beyond anything the timed loop consumed
        finish()
        evict_dev()                                  # discard the timed loop's flows
        if wl.get("sketch"):
            eng.sketch_reset()
        mine = V // world
        done = 0
        while done < mine:                           # regenerate into the (now free) input ring, chunk by chunk
            c = min(mine - done, 1 << 24, B)
            eng.gen_records(gp, V0 + rank * mine + done, c, batches[-1])
            ingest_dev(batches[-1].data_ptr(), c)
            finish()
            torch.cuda.synchronize()
            done += c
        sk_ours = None
        if wl.get("sketch"):                          # before the eviction: the table's exact counts are the yardstick
            sp = wl["sketch"]
            sk_ours = eng.sketch_export(sp["cms_log2_width"], sp["cms_depth"], sp["hll_precision"]) + (eng.hll_estimate(),)
        out_dev, nfl = evict_dev()
        if world > 1:                                # concatenate on rank 0 (padded all_gather of byte tensors)
            cnt = torch.tensor([nfl], device=dev, dtype=torch.int64)
            cnts = [torch.zeros_like(cnt) for _ in range(world)]
            dist.all_gather(cnts, cnt)
            cnts = [int(c.item()) for c in cnts]
            pad = torch.zeros(max(cnts) * REC, dtype=torch.uint8, device=dev)
            pad[: nfl * REC] = out_dev[: nfl * REC]
            parts = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
            dist.gather(pad, parts, dst=0)
            if rank == 0:
                ours = np.concatenate([p[: c * REC].cpu().numpy().reshape(-1, REC) for p, c in zip(parts, cnts)])
        else:
            ours = out_dev[: nfl * REC].cpu().numpy().reshape(-1, REC)
        if rank == 0:
            t0 = time.perf_counter()
            want = oracle_flows(wl, V0, V, sketch=wl.get("sketch"))
            sk_want = None
            if wl.get("sketch"):
                want, *sk_want = want
            ours = ours[record_order(ours)]
            same = ours.shape == want.shape and bool(np.array_equal(ours, want))
            parity = {"parity_checked": int(len(want)) if same else 0, "parity_ok": same, "records": V,
                      "flows_engine": int(len(ours)), "flows_oracle": int(len(want)),
                      "seconds": round(time.perf_counter() - t0, 2),
                      "how": "fresh cache, records [2^40, 2^40+V) of the workload stream through the same engine"
                             + ("" if world == 1 else f" (sharded over {world} GPUs, evictions concatenated)") +
                             "; every flow record compared bit for bit with the CPU oracle's fold of the same records"}
            if sk_ours is not None:
                import math
                import oracle_lib as O
                sp = wl["sketch"]
                cms, hll, est = sk_ours
                parity["sketch_bit_exact"] = bool(np.array_equal(cms.reshape(-1), sk_want[0]) and np.array_equal(hll, sk_want[1]))
                f = np.ascontiguousarray(want).view(O.REC_DTYPE).reshape(-1)
                parity["hll_estimate"], parity["distinct_exact"] = est, int(len(f))
                parity["hll_rel_err"] = abs(est - len(f)) / max(len(f), 1)
                parity["hll_3sigma"] = 3 * 1.04 / math.sqrt(1 << sp["hll_precision"])
                samp = want[:: max(1, len(want) // 200_000)]            # point queries on a sample of the flows
                q = eng.cms_query(samp[:, :40]).astype(np.int64)
                exact = np.ascontiguousarray(samp).view(O.REC_DTYPE).reshape(-1)["packets"].astype(np.int64)
                eps_n = math.e / (1 << sp["cms_log2_width"]) * V
                parity["cms_never_under"] = bool((q >= exact).all())
                parity["cms_within_eps_frac"] = float(((q - exact) <= eps_n).mean())
                parity["cms_bound_frac"] = 1 - math.exp(-sp["cms_depth"])
                parity["parity_ok"] = bool(same and parity["sketch_bit_exact"] and parity["cms_never_under"]
                                           and parity["hll_rel_err"] <= parity["hll_3sigma"]
                                           and parity["cms_within_eps_frac"] >= parity["cms_bound_frac"] - 0.005)
            if not same:
                nbad = -1
                if ours.shape == want.shape:
                    nbad = int((ours != want).any(axis=1).sum())
                parity["mismatching_flows"] = nbad
        barrier()

    # ---------------------------------------------------------------- end-to-end through the C ABI, host buffers
    # Every rank feeds its own slice from pinned host memory over its own PCIe link (N > 1: through the sharded
    # aggregator, whose local engine does the H2D copy); the timed region has the copies, a per-step read-back and
    # the final lookup-and-delete to host memory.  Preparation failures are agreed on by all ranks before the
    # loop starts, so a rank can never be left alone inside a collective.
    e2e = None
    host_ok = world == 1 or args.exchange == "peer"       # the NCCL variant's scratch streams are device-input only
    if not args.no_e2e and host_ok:
        Be = min(args.e2e_batch, max_batch, B)
        prep_err = None
        hring, out_host = [], None
        try:
            finish()
            evict_dev()                                    # reset the cache
            for i in range(4):
                h = torch.empty(Be * REC, dtype=torch.uint8).pin_memory()
                d = batches[-1][: Be * REC]
                eng.gen_records(gp, (1 << 41) + (i * world + rank) * Be, Be, d)
                eng.sync()
                h.copy_(d)
                hring.append(h)
            out_host = torch.empty(min(wl["max_entries"], wl["n_keys"], 1 << 25) * REC, dtype=torch.uint8).pin_memory()
        except Exception as ex:                                # noqa: BLE001 - reported in the JSON line
            prep_err = repr(ex)
        ok = torch.tensor([0 if prep_err else 1], device=dev, dtype=torch.int32)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 1:
            def e2e_step(i):
                h = hring[i % len(hring)]
                if world == 1:
                    rc, took = eng.ingest(h.data_ptr(), Be)   # H2D inside
                    assert rc == 0 and took == Be
                else:
                    agg.ingest(h, Be)                          # H2D inside the local combiner's fa_ingest
            for i in range(2):
                e2e_step(i)
            eng.live_flows()
            barrier()
            t0 = time.perf_counter()
            d2h = 0
            for i in range(args.e2e_steps):
                e2e_step(i)
                eng.live_flows()                               # per-step result read-back (64 B)
                d2h += 64
            finish()
            nfl = eng.evict_into(out_host.data_ptr(), out_host.numel() // REC)   # final lookup-and-delete to host
            d2h += nfl * REC
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if world > 1:
                tt = torch.tensor([dt], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt = float(tt.item())
            e2e = {"value": world * Be * args.e2e_steps / dt / 1e6, "unit": "Mpkts/s",
                   "h2d_bytes_per_step": world * Be * REC, "d2h_bytes_per_step": d2h // args.e2e_steps,
                   "records_per_step": world * Be, "steps": args.e2e_steps, "flows_evicted_rank0": int(nfl),
                   "note": ("fa_ingest(pinned host records) + fa_live_flows per step, final fa_evict to host inside the "
                            "timed region; wall clock, max over ranks; every rank feeds its slice over its own PCIe link"
                            + ("" if world == 1 else "; d2h bytes are rank 0's"))}
        elif rank == 0:
            e2e = {"value": None, "unit": "Mpkts/s", "error": prep_err or "preparation failed on another rank"}
        # separate row (SURVEY.md 8d): the same packets as 64-byte events (fa_ingest_events) — 2.25 x fewer PCIe bytes
        if world == 1 and e2e and e2e.get("value") and not args.no_events:
            evring = []
            for h in hring:
                r = h.numpy().reshape(-1, REC)
                ev = torch.empty(Be * 64, dtype=torch.uint8).pin_memory()
                v = ev.numpy().reshape(-1, 64)
                v[:, 0:40] = r[:, 0:40]            # flow_id
                v[:, 40:48] = r[:, 40:48]          # ts = start
                v[:, 48:52] = r[:, 56:60]          # len = bytes (low 32 bits)
                v[:, 52:54] = r[:, 70:72]          # flags
                v[:, 54] = r[:, 98]                # dscp
                v[:, 55] = r[:, 96]                # direction
                v[:, 56:60] = r[:, 84:88]          # if_index
                v[:, 60:64] = r[:, 92:96]          # sampling
                evring.append(ev)
            evict_dev()
            for i in range(2):
                eng.ingest_events(evring[i % len(evring)].data_ptr(), Be)
            eng.live_flows()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(args.e2e_steps):
                rc, took = eng.ingest_events(evring[i % len(evring)].data_ptr(), Be)
                assert rc == 0 and took == Be
                eng.live_flows()
            nfl = eng.evict_into(out_host.data_ptr(), out_host.numel() // REC)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            e2e["events_row"] = {"value": Be * args.e2e_steps / dt / 1e6, "unit": "Mpkts/s", "h2d_bytes_per_step": Be * 64,
                                 "d2h_bytes_per_step": (64 * args.e2e_steps + nfl * REC) // args.e2e_steps,
                                 "note": "same packets as 64-byte fa_packet_event (no MACs / TLS fields): fa_ingest_events + "
                                         "fa_live_flows per step, final fa_evict to host; parity with the 144-byte path: tests/test_events.py"}

    if rank == 0:
        peak, peak_src = peaks()
        kern_ms = statistics.mean(step_ms)
        launches_per_step = max(1, (B + max_batch - 1) // max_batch)
        per_launch = min(B, max_batch)
        achieved = B * REC / (kern_ms / 1e3) / 1e9
        tr = ncu_traffic(args.workload) if world == 1 else None
        cfg = make_config(args, wl, world)
        cfg.update({"records_per_launch": per_launch, "live_flows": int(flows), "input_ring_batches": ring,
                    "timed_region_ms": total_ms,
                    "parallelism": "1 GPU" if world == 1 else
                    f"hash-sharded x{world}: " + ("" if args.no_combine else "per-round local combine (K1+K2) -> ") +
                    ("K3 fused with the exchange (peer stores over NVLink, device-side counts)" if args.exchange == "peer"
                     else "K3 route -> NCCL all-to-all") + " -> K1 on the owner"})
        if nvlink:
            cfg["nvlink"] = nvlink
        line = {"metric": "Mpkts/s aggregated", "value": value, "unit": "Mpkts/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u64/u32 integer (add/or/min/max); no floating point", "data": "synthetic",
                "config": cfg,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": (tr["dram_bytes_per_record"] * per_launch) if tr else None,
                             "traffic_source": tr["source"] if tr else None,
                             "algorithmic_bytes_per_launch": REC * per_launch, "peak_source": peak_src,
                             "kernel": "fa::aggregate (K1); 144 algorithmic bytes per record; duration = CUDA-event time of "
                                       "one step / %d K1 launches (each followed by 2 early-exit re-fold kernels); traffic = "
                                       "ncu dram bytes per record x records per launch" % launches_per_step},
                "gpu_launches": int(launches), "clocks": clocks,
                "order_fixups": st1["order_fixups"] - st0["order_fixups"], "spills": st1["spills"]}
        if parity:
            line.update(parity)
        if e2e:
            line["e2e"] = e2e
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline_port(wl, args.cpu_sample)
        print(json.dumps(line), flush=True)
    if agg is not None and hasattr(agg, "close"):
        agg.close()
    eng.close()
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------- BASELINE config 5: RTT + DNS tracker path
def feature_samples(wl, n_dns, n_rtt, seed=5):
    """Host-built feature samples over the workload's key universe: (n_dns,104) DNS responses and (n_rtt,72) RTT samples."""
    import oracle_lib as O
    g = oracle_gen(wl)
    rng = np.random.default_rng(seed)
    kd = g.records(1 << 42, n_dns, threads=min(16, host_threads()))[:, :40]
    kr = g.records((1 << 42) + n_dns, n_rtt, threads=min(16, host_threads()))[:, :40]
    g.close()
    dns = np.zeros(n_dns, dtype=O.DNSREC_DTYPE)
    dns["id"] = kd
    d = dns["dns"]
    ts = 1_000_000 + np.arange(n_dns, dtype=np.uint64)
    d["start"], d["end"] = ts, ts
    d["latency"] = rng.integers(50_000, 40_000_000, n_dns)
    d["id"], d["flags"], d["eth"] = rng.integers(1, 1 << 16, n_dns), 0x8180, 0x0800
    d["errno"] = np.where(rng.random(n_dns) < 0.02, 3, 0)
    d["name"][:, :13] = np.frombuffer(b"\x03www\x07example\x00", dtype=np.uint8)
    dns["dns"] = d
    add = np.zeros(n_rtt, dtype=O.ADDREC_DTYPE)
    add["id"] = kr
    a = add["add"]
    tr = 1_000_000 + np.arange(n_rtt, dtype=np.uint64)
    a["start"], a["end"], a["eth"] = tr, tr, 0x0800
    a["rtt"] = rng.integers(20_000, 80_000_000, n_rtt)
    add["add"] = a
    return dns, add


def run_rttdns(args):
    """configs[4]: 70 % flow records, 30 % DNS responses (flow_id + dns_metrics, 104 B), one RTT sample (72 B) per 10
    packets of the TCP flows (80 % of the flows): K1 + the K6 feature folds + merged eviction, 1 GPU."""
    import torch
    import netobserv_ebpf_agent_b200 as fa
    import oracle_lib as O
    wl = WORKLOADS["zipf10m"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    B = min(args.batch, 1 << 25)
    Bf = B * 7 // 10; Bd = B - Bf; Br = Bf * 8 // 100
    mb = 1 << 22
    eng = fa.FlowAggEngine(wl["max_entries"], device=0, max_batch=mb, cuda_stream=stream.cuda_stream,
                           flags=fa.FA_F_ENABLE_RTT | fa.FA_F_ENABLE_DNS | fa.FA_F_NO_FULL_CUT)
    gp = fa.GenParams(seed=wl["seed"], n_keys=wl["n_keys"], dist=wl["dist"], zipf_s_milli=1100, t0_ns=1_000_000, varying_desc=0)
    base = [torch.empty(Bf * REC, dtype=torch.uint8, device=dev) for _ in range(2)]
    for i, t in enumerate(base):
        eng.gen_records(gp, i * Bf, Bf, t)
    nd, nr = min(Bd, 1 << 22), min(Br, 1 << 21)                       # sample arrays are cycled within a step
    dns_h, add_h = feature_samples(wl, nd, nr)
    dns_d = torch.from_numpy(dns_h.view(np.uint8).reshape(-1).copy()).to(dev)
    add_d = torch.from_numpy(add_h.view(np.uint8).reshape(-1).copy()).to(dev)
    eng.sync()

    def feed(ptr, n_have, n_want, width, call):
        done = 0
        while done < n_want:
            c = min(n_have, n_want - done, mb)
            call(C.c_void_p(ptr), c)
            done += c

    import ctypes as C
    L = fa.lib()

    def step(i):
        rc, took = eng.ingest(base[i % 2].data_ptr(), Bf)
        assert rc == 0 and took == Bf
        feed(dns_d.data_ptr(), nd, Bd, 104, lambda p, c: fa._lib.check(L.fa_ingest_dns(eng._h, p, c)))
        feed(add_d.data_ptr(), nr, Br, 72, lambda p, c: fa._lib.check(L.fa_ingest_additional(eng._h, p, c)))
    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    st0 = eng.stats()
    sampler = ClockSampler(0); sampler.start(); time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.window_begin(); e0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    e1.record(); torch.cuda.synchronize(); sampler.window_end()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    st1 = eng.stats()
    # parity on a fresh prefix: engine vs the oracle's LookupAndDeleteMap view
    out = eng.evict(features=True)
    del out
    V = 1 << 21
    vb = fa.gen_records_host(gp, 1 << 40, V)
    eng.ingest(vb); eng.ingest_dns(dns_h[: V // 4]); eng.ingest_additional(add_h[: V // 8])
    g_recs, g_dns, g_add, g_pres = eng.evict(features=True)
    om = O.FlowMap(); om.account(vb); om.fold_dns(dns_h[: V // 4]); om.fold_additional(add_h[: V // 8])
    o_recs, o_dns, o_add, o_pres = om.evict()
    gp_, op_ = O.sort_perm(g_recs), O.sort_perm(o_recs)
    same = len(gp_) == len(op_) and all(np.array_equal(g[gp_], o[op_]) for g, o in ((g_recs, o_recs), (g_dns, o_dns), (g_add, o_add), (g_pres, o_pres)))
    peak, peak_src = peaks()
    bytes_step = Bf * REC + Bd * 104 + Br * 72
    achieved = bytes_step * args.steps / (ms / 1e3) / 1e9
    line = {"metric": "Mpkts/s aggregated", "value": (Bf + Bd + Br) * args.steps / (ms / 1e3) / 1e6, "unit": "Mpkts/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64/u32 integer (add/or/min/max); no floating point", "data": "synthetic",
            "config": {"workload": "RTT+DNS tracker path (BASELINE configs[4]): 70% flow records, 30% DNS responses, 1 RTT sample per 10 "
                                   "packets of the TCP flows; 10M Zipf-1.1 5-tuples", "workload_key": "rttdns",
                       "flow_records_per_step": Bf, "dns_samples_per_step": Bd, "rtt_samples_per_step": Br,
                       "l2_policy": f"inputs larger than L2 ({bytes_step / 1e6:.0f} MB per step)", "n_gpus": 1},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "peak_source": peak_src, "kernel": "K1 + K6 feature folds (dns_fold / additional_fold); blended algorithmic bytes = "
                                                            "144 B per flow record + 104 B per DNS sample + 72 B per RTT sample"},
            "gpu_launches": int(st1["kernel_launches"] - st0["kernel_launches"]), "clocks": clocks,
            "parity_checked": int(len(op_)) if same else 0, "parity_ok": bool(same)}
    print(json.dumps(line), flush=True)
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="zipf10m", choices=sorted(WORKLOADS) + ["rttdns"])
    ap.add_argument("--batch", type=int, default=None,
                    help="records per step per GPU; default 3 x 2^26 at N = 1 (29 GB: at 16-17 Gpkt/s the driver's 20 steps are a "
                         "timed region of >= 200 ms), 2^27 = one exchange round per step at N > 1 (10-11 ms per step)")
    ap.add_argument("--max-batch", type=int, default=None,
                    help="records per K1 launch (N = 1); default 2^23 with the Accounter's maxEntries rule on (the largest size "
                         "that keeps its fast-path test true on every workload), 2^24 for the plain-map workload zipf1m")
    ap.add_argument("--mgpu-round", type=int, default=1 << 27, help="N>1: records per combine -> exchange -> fold round")
    ap.add_argument("--ring", type=int, default=2, help="distinct pre-generated input batches cycled through")
    ap.add_argument("--e2e-batch", type=int, default=1 << 22)
    ap.add_argument("--e2e-steps", type=int, default=32)
    ap.add_argument("--cpu-sample", type=int, default=1 << 25)
    ap.add_argument("--ref-sample", type=int, default=1 << 24)
    ap.add_argument("--verify-records", type=int, default=1 << 25)
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-combine", action="store_true", help="N>1: route raw records instead of per-batch partial flows")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N>1: 'peer' = K3 stores into the owners' buffers over NVLink (no host sync); 'nccl' = all_to_all_single")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-events", action="store_true", help="skip the 64-byte packet-event row of e2e")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the flows they left in the table (a key-hash sample of at most "
                         f"{DUMP_FLOWS}) and, with sketches on, the sketch tables as DIR/<name>.npy (1 GPU, flow workloads)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload == "rttdns"):
        ap.error("--dump-outputs covers the GPU arm of the flow workloads")
    if args.batch is None:
        args.batch = (3 << 26) if args.gpus == 1 else (1 << 27)
    if args.workload == "rttdns":
        return run_rttdns(args)
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
