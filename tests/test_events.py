"""fa_ingest_events: 64-byte packet events fold exactly like the single-packet records flow_monitor would build for
them (bpf/flows.c:228-245).  The checker expands the events on the host (numpy) and runs the oracle's Accounter."""
import numpy as np
import pytest

import oracle_lib as O
from common import gen_host

EVENT_DTYPE = np.dtype([("id", "u1", 40), ("ts", "<u8"), ("len", "<u4"), ("flags", "<u2"), ("dscp", "u1"), ("dir", "u1"),
                        ("if_index", "<u4"), ("sampling", "<u4")])
assert EVENT_DTYPE.itemsize == 64


def events_of(recs):
    """The packet events behind single-packet records (what the generator's records describe)."""
    r = np.ascontiguousarray(recs).view(O.REC_DTYPE).reshape(-1)
    ev = np.zeros(len(r), dtype=EVENT_DTYPE)
    ev["id"] = np.ascontiguousarray(recs)[:, :40]
    ev["ts"], ev["len"], ev["flags"], ev["dscp"], ev["dir"] = r["start"], r["bytes"], r["flags"], r["dscp"], r["direction"]
    ev["if_index"], ev["sampling"] = r["if_index"], r["sampling"]
    return ev


def expand(ev):
    """Host restatement of the expansion: new_flow of flows.c:228-245 without MACs / TLS."""
    out = np.zeros(len(ev), dtype=O.REC_DTYPE)
    ids = ev["id"].copy(); ids[:, 39] = 0
    raw = out.view(np.uint8).reshape(-1, 144)
    raw[:, :40] = ids
    out["start"] = out["end"] = ev["ts"]
    out["bytes"], out["packets"], out["flags"] = ev["len"], 1, ev["flags"]
    v4 = (ids[:, :10] == 0).all(axis=1) & (ids[:, 10] == 0xFF) & (ids[:, 11] == 0xFF)
    out["eth"] = np.where(v4, 0x0800, 0x86DD)
    out["if_index"], out["sampling"], out["direction"], out["dscp"] = ev["if_index"], ev["sampling"], ev["dir"], ev["dscp"]
    return raw


def check(n=30_000, n_keys=2_000, max_entries=1 << 12, max_batch=8_192, varying=1):
    import netobserv_ebpf_agent_b200 as fa
    recs = gen_host(seed=61, n=n, n_keys=n_keys, dist=1, varying=varying)
    ev = events_of(recs)
    ev["id"][::3, 39] = 0x5A                                       # padding byte of the key: ignored on input
    acc = O.Accounter(max_entries)
    acc.account(expand(ev))
    want = O.sort_records(acc.evict())
    with fa.FlowAggEngine(max_entries, max_batch=max_batch) as eng:
        raw = ev.view(np.uint8).reshape(-1)
        rc, took = eng.ingest_events(raw[: (n // 2) * 64])
        assert rc == 0 and took == n // 2
        rc, took = eng.ingest_events(raw[(n // 2) * 64:])
        assert rc == 0 and took == n - n // 2
        st = eng.stats()
        assert st["h2d_bytes"] == n * 64 and st["records_ingested"] == n
        got = O.sort_records(eng.evict())
    assert np.array_equal(got, want)
    acc.close()


def test_events_on_the_emulation(engine_emul):
    check(n=6_000, n_keys=300, max_entries=1 << 10, max_batch=2_048)


def test_full_cut_with_events_on_the_emulation(engine_emul):
    """The Accounter's maxEntries rule cuts an event chunk at the same packet as a record chunk."""
    import netobserv_ebpf_agent_b200 as fa
    recs = gen_host(seed=62, n=3_000, n_keys=900, dist=0)
    ev = events_of(recs).view(np.uint8).reshape(-1)
    with fa.FlowAggEngine(200, max_batch=1_024) as a, fa.FlowAggEngine(200, max_batch=1_024) as b:
        rc_a, took_a = a.ingest_events(ev)
        rc_b, took_b = b.ingest(expand(events_of(recs)))
        assert (rc_a, took_a) == (rc_b, took_b) and rc_a == fa.FA_FULL and 200 <= took_a < 3_000
        assert np.array_equal(O.sort_records(a.evict()), O.sort_records(b.evict()))


def test_the_gpu_tests_below_get_the_real_library():
    """The emulation the tests above swapped in ends with them: the gpu tests of this module run on libflowagg.so."""
    import netobserv_ebpf_agent_b200._lib as L
    assert L.lib()._name == L.lib_path()


@pytest.mark.gpu
def test_events_gpu():
    check(n=400_000, n_keys=60_000, max_entries=1 << 17, max_batch=1 << 16)


@pytest.mark.gpu
def test_events_from_device_memory_gpu():
    import torch
    import netobserv_ebpf_agent_b200 as fa
    recs = gen_host(seed=63, n=100_000, n_keys=5_000, dist=1)
    ev = events_of(recs)
    acc = O.Accounter(1 << 14); acc.account(expand(ev)); want = O.sort_records(acc.evict()); acc.close()
    with fa.FlowAggEngine(1 << 14, max_batch=1 << 15) as eng:
        d = torch.from_numpy(ev.view(np.uint8).reshape(-1).copy()).cuda()
        rc, took = eng.ingest_events(d)
        assert rc == 0 and took == len(ev) and eng.stats()["h2d_bytes"] == 0
        assert np.array_equal(O.sort_records(eng.evict()), want)
