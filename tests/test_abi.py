"""CPU-only checks of the drop-in boundary: the library loads, exports every symbol the header
declares, and the header's struct layouts match the agent's ABI (offsets from SURVEY.md §8a, and the
layout of the reference's own bpf/types.h stored under tests/golden/)."""
import json
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "flowagg.h")


def test_library_loads_and_exports_every_declared_symbol():
    import netobserv_ebpf_agent_b200 as fa
    from netobserv_ebpf_agent_b200._lib import SIGNATURES
    L = fa.lib()
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    declared = set(re.findall(r"\b(fa_[a-z0-9_]+)\s*\(", text))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(L, name), f"libflowagg.so does not export {name}"
    assert declared == set(SIGNATURES), declared ^ set(SIGNATURES)
    assert L.fa_abi_version() == 1


def test_no_cpu_fallback():
    """Without a CUDA device the product path must fail loudly, never compute on the CPU."""
    import torch
    import netobserv_ebpf_agent_b200 as fa
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(fa.FlowAggError) as ei:
        fa.FlowAggEngine(1000)
    assert ei.value.code == -19


def test_product_does_not_touch_oracle():
    """Only tests/, smoke() and bench.py's CPU legs may use oracle/."""
    pkg = os.path.join(ROOT, "netobserv_ebpf_agent_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")) or f == "Makefile":
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert "liboracle" not in txt and "oracle_lib" not in txt and "oracle/" not in txt, (dp, f)


C_PROBE = r'''
#include <stdio.h>
#include <stddef.h>
#include "flowagg.h"
#define P(t, f) printf(#t "." #f " %zu\n", offsetof(t, f))
int main(void) {
  printf("sizeof.fa_flow_id %zu\n", sizeof(fa_flow_id));
  printf("sizeof.fa_flow_metrics %zu\n", sizeof(fa_flow_metrics));
  printf("sizeof.fa_flow_record %zu\n", sizeof(fa_flow_record));
  printf("sizeof.fa_dns_metrics %zu\n", sizeof(fa_dns_metrics));
  printf("sizeof.fa_additional_metrics %zu\n", sizeof(fa_additional_metrics));
  printf("sizeof.fa_dns_record %zu\n", sizeof(fa_dns_record));
  printf("sizeof.fa_additional_record %zu\n", sizeof(fa_additional_record));
  P(fa_flow_id, src_ip); P(fa_flow_id, dst_ip); P(fa_flow_id, src_port); P(fa_flow_id, dst_port);
  P(fa_flow_id, transport_protocol); P(fa_flow_id, icmp_type); P(fa_flow_id, icmp_code);
  P(fa_flow_metrics, start_mono_time_ts); P(fa_flow_metrics, end_mono_time_ts); P(fa_flow_metrics, bytes);
  P(fa_flow_metrics, packets); P(fa_flow_metrics, eth_protocol); P(fa_flow_metrics, flags);
  P(fa_flow_metrics, src_mac); P(fa_flow_metrics, dst_mac); P(fa_flow_metrics, if_index_first_seen);
  P(fa_flow_metrics, lock); P(fa_flow_metrics, sampling); P(fa_flow_metrics, direction_first_seen);
  P(fa_flow_metrics, errno_); P(fa_flow_metrics, dscp); P(fa_flow_metrics, nb_observed_intf);
  P(fa_flow_metrics, observed_direction); P(fa_flow_metrics, observed_intf); P(fa_flow_metrics, ssl_version);
  P(fa_flow_metrics, tls_cipher_suite); P(fa_flow_metrics, tls_key_share); P(fa_flow_metrics, tls_types);
  P(fa_flow_metrics, misc_flags);
  P(fa_dns_metrics, latency); P(fa_dns_metrics, id); P(fa_dns_metrics, flags); P(fa_dns_metrics, eth_protocol);
  P(fa_dns_metrics, errno_); P(fa_dns_metrics, name);
  P(fa_additional_metrics, flow_rtt); P(fa_additional_metrics, ipsec_encrypted_ret);
  P(fa_additional_metrics, eth_protocol); P(fa_additional_metrics, ipsec_encrypted);
  P(fa_flow_record, metrics); P(fa_dns_record, dns); P(fa_additional_record, additional);
  return 0;
}
'''

EXPECT = {  # SURVEY.md §8a (verified there against bpf/types.h compiled with gcc and the Go mirrors)
    "sizeof.fa_flow_id": 40, "sizeof.fa_flow_metrics": 104, "sizeof.fa_flow_record": 144,
    "sizeof.fa_dns_metrics": 64, "sizeof.fa_additional_metrics": 32, "sizeof.fa_dns_record": 104,
    "sizeof.fa_additional_record": 72,
    "fa_flow_id.src_ip": 0, "fa_flow_id.dst_ip": 16, "fa_flow_id.src_port": 32, "fa_flow_id.dst_port": 34,
    "fa_flow_id.transport_protocol": 36, "fa_flow_id.icmp_type": 37, "fa_flow_id.icmp_code": 38,
    "fa_flow_metrics.start_mono_time_ts": 0, "fa_flow_metrics.end_mono_time_ts": 8, "fa_flow_metrics.bytes": 16,
    "fa_flow_metrics.packets": 24, "fa_flow_metrics.eth_protocol": 28, "fa_flow_metrics.flags": 30,
    "fa_flow_metrics.src_mac": 32, "fa_flow_metrics.dst_mac": 38, "fa_flow_metrics.if_index_first_seen": 44,
    "fa_flow_metrics.lock": 48, "fa_flow_metrics.sampling": 52, "fa_flow_metrics.direction_first_seen": 56,
    "fa_flow_metrics.errno_": 57, "fa_flow_metrics.dscp": 58, "fa_flow_metrics.nb_observed_intf": 59,
    "fa_flow_metrics.observed_direction": 60, "fa_flow_metrics.observed_intf": 68,
    "fa_flow_metrics.ssl_version": 92, "fa_flow_metrics.tls_cipher_suite": 94, "fa_flow_metrics.tls_key_share": 96,
    "fa_flow_metrics.tls_types": 98, "fa_flow_metrics.misc_flags": 99,
    "fa_dns_metrics.latency": 16, "fa_dns_metrics.id": 24, "fa_dns_metrics.flags": 26,
    "fa_dns_metrics.eth_protocol": 28, "fa_dns_metrics.errno_": 30, "fa_dns_metrics.name": 31,
    "fa_additional_metrics.flow_rtt": 16, "fa_additional_metrics.ipsec_encrypted_ret": 24,
    "fa_additional_metrics.eth_protocol": 28, "fa_additional_metrics.ipsec_encrypted": 30,
    "fa_flow_record.metrics": 40, "fa_dns_record.dns": 40, "fa_additional_record.additional": 40,
}


def _run_c(src, includes):
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "p.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "p")
        subprocess.run(["/usr/bin/gcc", "-std=gnu11", "-o", exe, c] + [f"-I{i}" for i in includes], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    return {k: int(v) for k, v in (ln.split() for ln in out.strip().splitlines())}


def test_header_layout_matches_agent_abi():
    got = _run_c(C_PROBE, [os.path.join(ROOT, "include")])
    assert got == EXPECT


REF_PROBE = r'''
#include <stdio.h>
#include <stddef.h>
#include <stdint.h>
#include <stdbool.h>
typedef uint8_t __u8; typedef uint16_t __u16; typedef uint32_t __u32; typedef uint64_t __u64;
typedef int32_t s32; typedef int64_t s64; typedef int16_t s16; typedef int8_t s8;
struct bpf_spin_lock { __u32 val; };
#include "types.h"
#define P(n, t, f) printf(n " %zu\n", offsetof(t, f))
int main(void) {
  printf("sizeof.fa_flow_id %zu\n", sizeof(flow_id));
  printf("sizeof.fa_flow_metrics %zu\n", sizeof(flow_metrics));
  printf("sizeof.fa_flow_record %zu\n", sizeof(flow_record));
  printf("sizeof.fa_dns_metrics %zu\n", sizeof(dns_metrics));
  printf("sizeof.fa_additional_metrics %zu\n", sizeof(additional_metrics));
  P("fa_flow_id.src_port", flow_id, src_port); P("fa_flow_id.transport_protocol", flow_id, transport_protocol);
  P("fa_flow_id.icmp_code", flow_id, icmp_code);
  P("fa_flow_metrics.packets", flow_metrics, packets); P("fa_flow_metrics.eth_protocol", flow_metrics, eth_protocol);
  P("fa_flow_metrics.flags", flow_metrics, flags); P("fa_flow_metrics.src_mac", flow_metrics, src_mac);
  P("fa_flow_metrics.dst_mac", flow_metrics, dst_mac);
  P("fa_flow_metrics.if_index_first_seen", flow_metrics, if_index_first_seen); P("fa_flow_metrics.lock", flow_metrics, lock);
  P("fa_flow_metrics.sampling", flow_metrics, sampling); P("fa_flow_metrics.direction_first_seen", flow_metrics, direction_first_seen);
  P("fa_flow_metrics.errno_", flow_metrics, errno); P("fa_flow_metrics.dscp", flow_metrics, dscp);
  P("fa_flow_metrics.nb_observed_intf", flow_metrics, nb_observed_intf);
  P("fa_flow_metrics.observed_direction", flow_metrics, observed_direction);
  P("fa_flow_metrics.observed_intf", flow_metrics, observed_intf); P("fa_flow_metrics.ssl_version", flow_metrics, ssl_version);
  P("fa_flow_metrics.tls_cipher_suite", flow_metrics, tls_cipher_suite); P("fa_flow_metrics.tls_key_share", flow_metrics, tls_key_share);
  P("fa_flow_metrics.tls_types", flow_metrics, tls_types); P("fa_flow_metrics.misc_flags", flow_metrics, misc_flags);
  P("fa_dns_metrics.latency", dns_metrics, latency); P("fa_dns_metrics.id", dns_metrics, id);
  P("fa_dns_metrics.flags", dns_metrics, flags); P("fa_dns_metrics.eth_protocol", dns_metrics, eth_protocol);
  P("fa_dns_metrics.errno_", dns_metrics, errno); P("fa_dns_metrics.name", dns_metrics, name);
  P("fa_additional_metrics.flow_rtt", additional_metrics, flow_rtt);
  P("fa_additional_metrics.ipsec_encrypted_ret", additional_metrics, ipsec_encrypted_ret);
  P("fa_additional_metrics.eth_protocol", additional_metrics, eth_protocol);
  P("fa_additional_metrics.ipsec_encrypted", additional_metrics, ipsec_encrypted);
  P("fa_flow_record.metrics", flow_record, metrics);
  return 0;
}
'''


REF_LAYOUT = os.path.join(ROOT, "tests", "golden", "reference_types_h_layout.json")


def test_header_layout_matches_reference_types_h():
    """Cross-check against the reference's own header: REF_PROBE's output on its bpf/types.h, stored by
    tests/golden/make_reference_layout.py (the header itself is never copied into the repo)."""
    ref = json.load(open(REF_LAYOUT))["layout"]
    got = _run_c(C_PROBE, [os.path.join(ROOT, "include")])
    assert len(ref) == 38                                    # every line REF_PROBE prints
    for k, v in ref.items():
        assert got[k] == v == EXPECT[k], (k, v, got[k], EXPECT[k])


def test_oracle_dtype_matches_expected_offsets():
    f = O.REC_DTYPE.fields
    assert f["start"][1] == 40 and f["packets"][1] == 64 and f["eth"][1] == 68 and f["flags"][1] == 70
    assert f["src_mac"][1] == 72 and f["if_index"][1] == 84 and f["sampling"][1] == 92 and f["dscp"][1] == 98
    assert f["obs_intf"][1] == 108 and f["ssl_version"][1] == 132 and f["misc"][1] == 139
