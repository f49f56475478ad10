#!/usr/bin/env python
"""Regenerates tests/golden/reference_types_h_layout.json from a checkout of netobserv-ebpf-agent.

  python tests/golden/make_reference_layout.py <netobserv-ebpf-agent>/bpf [commit]

Compiles REF_PROBE (tests/test_abi.py) against the reference's own bpf/types.h with gcc and stores the struct sizes
and field offsets it prints, so that test_abi.py can hold include/flowagg.h to the reference's layout without the
reference tree at hand.  Only the numbers are stored; the header is not copied.
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from test_abi import REF_LAYOUT, REF_PROBE, _run_c  # noqa: E402


def main(bpf_dir, commit=None):
    types_h = os.path.join(bpf_dir, "types.h")
    layout = _run_c(REF_PROBE, [bpf_dir])
    doc = {"source": "netobserv-ebpf-agent bpf/types.h, compiled with gcc by REF_PROBE in tests/test_abi.py",
           "commit": commit, "types_h_sha256": hashlib.sha256(open(types_h, "rb").read()).hexdigest(), "layout": layout}
    with open(REF_LAYOUT, "w") as f:
        json.dump(doc, f, indent=1)
        f.write("\n")
    print(REF_LAYOUT, len(layout), "entries")


if __name__ == "__main__":
    main(*sys.argv[1:3])
