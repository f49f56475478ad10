"""(f3) packet-drop fold and the RTT-minimum extension: fa_ingest_pkt_drops / fa_evict_ex against the oracle.

Pinned by the reference's own test of AccumulateDrops, pkg/model/flow_content_test.go:55-104 (transcribed below).  The
RTT minimum has no reference analogue (PARITY UNPINNED): it is checked against the oracle's definition — the smallest
non-zero flow_rtt among a flow's samples.  CPU tests run the kernels on the engine emulation, gpu ones on the device."""
import numpy as np
import pytest

import oracle_lib as O
from common import gen_host
from test_gpu_features import keys_of, make_add, make_dns


def make_drops(rng, keys, n):
    r = np.zeros(n, dtype=O.DROPREC_DTYPE)
    r["id"] = keys[rng.integers(0, len(keys), n)]
    d = r["drop"]
    d["start"] = np.where(rng.random(n) < 0.1, 0, rng.integers(1, 1 << 40, n))
    d["end"] = np.where(rng.random(n) < 0.1, 0, rng.integers(1, 1 << 40, n))
    d["bytes"] = np.where(rng.random(n) < 0.1, 60_000, rng.integers(0, 3_000, n))          # some flows saturate
    d["packets"] = np.where(rng.random(n) < 0.05, 65_535, rng.integers(0, 4, n))
    d["cause"] = np.where(rng.random(n) < 0.4, 0, rng.integers(1, 1 << 32, n))
    d["flags"] = rng.integers(0, 1 << 16, n)
    d["eth"] = np.where(rng.random(n) < 0.4, 0, rng.choice([0x0800, 0x86DD], n))
    d["state"] = np.where(rng.random(n) < 0.4, 0, rng.integers(1, 256, n))
    d["pad"] = rng.integers(0, 256, (n, 3))                                                  # ignored on input, zero on output
    r["drop"] = d
    return r


def test_oracle_reproduces_the_reference_test_of_accumulate_drops():
    """flow_content_test.go:55-104."""
    base = np.zeros(1, dtype=O.REC_DTYPE)
    base["start"], base["end"], base["packets"] = 10, 20, 3
    met = base.view(np.uint8).reshape(-1)[40:].copy()
    drops, has = np.zeros(32, dtype=np.uint8), np.zeros(1, dtype=np.uint8)
    o1 = np.zeros(1, dtype=O.DROP_DTYPE); o1["start"] = o1["end"] = 25; o1["bytes"], o1["packets"], o1["cause"], o1["flags"], o1["state"] = 5, 1, 100, 0b11, 200
    o2 = np.zeros(1, dtype=O.DROP_DTYPE); o2["start"] = o2["end"] = 30; o2["bytes"], o2["packets"], o2["cause"], o2["flags"], o2["state"] = 10, 2, 101, 0b1001, 201
    L = O.lib()
    L.oracle_accumulate_drops(O._p(met), O._p(drops), O._p(has), O._p(o1.view(np.uint8).reshape(-1)))
    # met = raw 104-byte metrics: start@0, end@8
    assert int(met[:8].view("<u8")[0]) == 10 and int(met[8:16].view("<u8")[0]) == 25 and has[0] == 1
    d = drops.view(O.DROP_DTYPE)[0]
    assert (d["start"], d["end"], d["bytes"], d["packets"], d["cause"], d["flags"], d["state"]) == (25, 25, 5, 1, 100, 0b11, 200)
    L.oracle_accumulate_drops(O._p(met), O._p(drops), O._p(has), O._p(o2.view(np.uint8).reshape(-1)))
    assert int(met[:8].view("<u8")[0]) == 10 and int(met[8:16].view("<u8")[0]) == 30
    d = drops.view(O.DROP_DTYPE)[0]
    assert (d["start"], d["end"], d["bytes"], d["packets"], d["cause"], d["flags"], d["state"]) == (25, 25, 15, 3, 101, 0b1011, 201)


def compare_ex(eng, om):
    got = eng.evict_ex()
    want = om.evict_ex()
    gp, op = O.sort_perm(got[0]), O.sort_perm(want[0])
    assert len(gp) == len(op)
    for name, g, o in zip(("records", "dns", "additional", "pkt_drops", "rtt_min", "present"), got, want):
        gs, os_ = g.reshape(len(g), -1)[gp], o.reshape(len(o), -1)[op]
        if not np.array_equal(gs, os_):
            bad = np.nonzero((gs != os_).any(axis=1))[0]
            raise AssertionError(f"{name}: {len(bad)} of {len(gs)} differ; first {bad[0]}:\n engine {gs[bad[0]].tolist()}\n oracle {os_[bad[0]].tolist()}")
    return len(gp)


def check_golden():
    """The reference's test through the engine: base record, then the two drop samples."""
    import netobserv_ebpf_agent_b200 as fa
    base = np.zeros(1, dtype=O.REC_DTYPE); base["start"], base["end"], base["packets"] = 10, 20, 3
    base["src_port"] = 7
    s = np.zeros(2, dtype=O.DROPREC_DTYPE)
    s["id"] = base.view(np.uint8).reshape(-1, 144)[:, :40]
    s["drop"]["start"] = s["drop"]["end"] = [25, 30]
    s["drop"]["bytes"], s["drop"]["packets"], s["drop"]["cause"], s["drop"]["flags"], s["drop"]["state"] = [5, 10], [1, 2], [100, 101], [0b11, 0b1001], [200, 201]
    with fa.FlowAggEngine(64, flags=fa.FA_F_ENABLE_PKT_DROP, max_batch=1024) as eng:
        eng.ingest(base.view(np.uint8).reshape(-1, 144))
        eng.ingest_pkt_drops(s[:1]); eng.ingest_pkt_drops(s[1:])
        recs, _, _, drops, rmin, pres = eng.evict_ex()
    r, d = recs.view(O.REC_DTYPE).reshape(-1)[0], drops.view(O.DROP_DTYPE).reshape(-1)[0]
    assert (r["start"], r["end"], r["packets"]) == (10, 30, 3) and pres[0] == 4 and rmin[0] == 0
    assert (d["start"], d["end"], d["bytes"], d["packets"], d["cause"], d["flags"], d["state"]) == (25, 25, 15, 3, 101, 0b1011, 201)


def check_random(n_keys, n_base, n_feat, max_entries, max_batch):
    import netobserv_ebpf_agent_b200 as fa
    rng = np.random.default_rng(17)
    base = gen_host(seed=33, n=n_base, n_keys=n_keys, dist=1)
    keys = np.concatenate([np.unique(base[:, :40], axis=0), keys_of(34, max(n_keys // 10, 3))])   # some flows exist through features only
    drops, add, dns = make_drops(rng, keys, n_feat), make_add(rng, keys, n_feat), make_dns(rng, keys, n_feat)
    om = O.FlowMap()
    flags = fa.FA_F_ENABLE_PKT_DROP | fa.FA_F_ENABLE_RTT | fa.FA_F_ENABLE_DNS
    with fa.FlowAggEngine(max_entries, flags=flags, max_batch=max_batch) as eng:
        h = n_feat // 2
        eng.ingest_pkt_drops(drops[:h]); eng.ingest(base[: n_base // 2]); eng.ingest_additional(add); eng.ingest_dns(dns)
        eng.ingest_pkt_drops(drops[h:]); eng.ingest(base[n_base // 2:])
        om.fold_drops(drops); om.account(base); om.fold_additional(add); om.fold_dns(dns)
        assert eng.stats()["pkt_drops_ingested"] == n_feat
        n1 = compare_ex(eng, om)
        # a second eviction period starts from scratch
        eng.ingest_pkt_drops(drops[:100]); om.fold_drops(drops[:100])
        eng.ingest_additional(add[:100]); om.fold_additional(add[:100])
        n2 = compare_ex(eng, om)
    assert n1 >= n_keys // 2 and 0 < n2 <= 200


def test_golden_on_the_emulation(engine_emul):
    check_golden()


def test_random_streams_on_the_emulation(engine_emul):
    check_random(n_keys=120, n_base=1_500, n_feat=1_200, max_entries=1 << 10, max_batch=1_024)


def test_drops_need_the_flag(engine_emul):
    import netobserv_ebpf_agent_b200 as fa
    with fa.FlowAggEngine(64, max_batch=256) as eng:
        with pytest.raises(fa.FlowAggError) as ei:
            eng.ingest_pkt_drops(np.zeros(1, dtype=O.DROPREC_DTYPE))
        assert ei.value.code == -22 and "FA_F_ENABLE_PKT_DROP" in str(ei.value)


@pytest.mark.gpu
def test_golden_gpu():
    check_golden()


@pytest.mark.gpu
def test_random_streams_gpu():
    check_random(n_keys=5_000, n_base=80_000, n_feat=60_000, max_entries=1 << 17, max_batch=1 << 15)


EVICT_OUT_BYTES = {"dns": 64, "additional": 32, "pkt_drops": 32, "rtt_min": 8, "present": 1}


def evict_outputs(flags, where):
    """Build one feature-laden state and evict it with each feature output placed as where[name]: "host", "device"
    (fa_device_alloc: plain memory on the emulation) or None.  -> {name: bytes per flow, records sorted by key}."""
    import ctypes as C
    import netobserv_ebpf_agent_b200 as fa
    from netobserv_ebpf_agent_b200._lib import EvictOut, check, lib
    rng = np.random.default_rng(5)
    base = gen_host(seed=41, n=500, n_keys=60, dist=1)
    keys = np.concatenate([np.unique(base[:, :40], axis=0), keys_of(42, 8)])
    with fa.FlowAggEngine(1 << 10, flags=flags, max_batch=512) as eng:
        eng.ingest(base)
        if flags:
            eng.ingest_pkt_drops(make_drops(rng, keys, 300)); eng.ingest_additional(make_add(rng, keys, 300))
            eng.ingest_dns(make_dns(rng, keys, 300))
        n = eng.live_flows()
        records, host, ptrs = np.zeros((n, 144), np.uint8), {}, {}
        for name, width in EVICT_OUT_BYTES.items():
            if where[name] == "host":
                host[name] = np.full((n, width), 0xAB, np.uint8)             # stale bytes: must be overwritten
                ptrs[name] = host[name].ctypes.data
            elif where[name] == "device":
                p = C.c_void_p()
                check(lib().fa_device_alloc(eng._h, n * width, C.byref(p)))
                ptrs[name] = p.value
            else:
                ptrs[name] = None
        got = C.c_size_t(0)
        check(lib().fa_evict_ex(eng._h, C.byref(EvictOut(records=records.ctypes.data, **ptrs)), n, C.byref(got)))
        assert got.value == n
        perm = O.sort_perm(records)
        out = {"records": records[perm]}
        for name, width in EVICT_OUT_BYTES.items():
            if where[name] == "host":
                out[name] = host[name][perm]
            elif where[name] == "device":
                out[name] = np.frombuffer(C.string_at(ptrs[name], n * width), np.uint8).reshape(n, width)[perm]
                check(lib().fa_device_free(eng._h, ptrs[name]))
    return out


def test_evict_outputs_on_the_emulation(engine_emul):
    """fa_evict_ex's five feature outputs stage through the device or are written in place: every mix of host, device
    and absent outputs gives the same bytes, and without feature folds the host outputs come back zeroed."""
    import netobserv_ebpf_agent_b200 as fa
    flags = fa.FA_F_ENABLE_PKT_DROP | fa.FA_F_ENABLE_RTT | fa.FA_F_ENABLE_DNS
    names = list(EVICT_OUT_BYTES)
    want = evict_outputs(flags, dict.fromkeys(names, "host"))
    assert want["present"].any() and want["rtt_min"].any()
    mixes = [dict.fromkeys(names, "device"), dict.fromkeys(names, None),
             dict(zip(names, ["host", "device", None, "device", "host"])), dict(zip(names, ["device", None, "host", "host", "device"]))]
    for where in mixes:
        got = evict_outputs(flags, where)
        assert sorted(got) == sorted(["records"] + [k for k in names if where[k]])
        for name, a in got.items():
            assert np.array_equal(a, want[name]), (where, name)
    plain = evict_outputs(0, dict.fromkeys(names, "host"))
    assert all(not plain[name].any() for name in names)
    assert len(plain["records"]) < len(want["records"])          # the feature samples created flows of their own


def test_hot_keys_and_crowded_tiles_on_the_emulation(engine_emul):
    """K6 folds a tile's samples of one flow in shared memory before touching the table: a handful of keys (every tile is
    almost all duplicates) and a key set larger than the tile's election set both have to stay exact."""
    check_random(n_keys=6, n_base=400, n_feat=1_500, max_entries=1 << 12, max_batch=1_024)
    check_random(n_keys=700, n_base=6_000, n_feat=2_000, max_entries=1 << 13, max_batch=2_048)
