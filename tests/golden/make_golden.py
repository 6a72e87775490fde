"""Regenerates the committed fixtures under tests/golden/ from the oracle (run from the repo root:
`python tests/golden/make_golden.py`).

The reference is Java and cannot be imported or run in this image, so these are NOT outputs of the reference: they are
regression pins of the oracle (and, through the gpu tests, of the CUDA path), plus the exact values java/PinRingHash.java
prints with the reference's own hash library wherever a JVM + zero-allocation-hashing 0.8 exist."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle_py as orc  # noqa: E402
from rapid_b200 import workloads as W  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
K = 10


def ring_keys():
    n = 16
    hb, off, ports = W.packed_endpoints(0, n)
    u = orc.Universe()
    tags = u.add_bulk(hb, off, ports)
    hi, lo = W.node_ids(0, n)
    v = orc.MembershipView(u, K, tags, hi, lo)
    out = {
        "endpoints": [{"hostname": "10.0.0.0", "port": int(p)} for p in ports],
        "node_ids": [[int(a), int(b)] for a, b in zip(hi, lo)],
        "keys": [[v.key(k, i) for i in range(n)] for k in range(K)],
        "rings": [v.getRing(k) for k in range(K)],
        "configuration_id": v.getCurrentConfigurationId(),
        "xxh64": {"empty_seed0": orc.xxh64(b"", 0), "hashInt_1000_seed3": orc.xx_hash_int(1000, 3),
                  "hashLong_minus1_seed0": orc.xx_hash_long(-1, 0)},
    }
    with open(os.path.join(HERE, "ring_keys.json"), "w") as f:
        json.dump(out, f, indent=1)


def cut_scenarios():
    """small end-to-end scenarios: view -> alert batch -> per-receiver proposals (oracle) -> decision"""
    cases = []
    for name, n, nj, H, L in (("c1", 50, 0, 9, 4), ("c2", 400, 0, 9, 4), ("c3", 400, 0, 9, 4), ("c5", 600, 3, 9, 4)):
        hb, off, ports = W.packed_endpoints(0, n + nj)
        u = orc.Universe()
        tags = u.add_bulk(hb, off, ports)
        hi, lo = W.node_ids(0, n)
        v = orc.MembershipView(u, K, tags[:n], hi, lo)
        obs = lambda ids: v.tables(ids)[0]
        if name == "c1":
            b = W.c1_single_crash(obs, n)
        elif name == "c2":
            b = W.c2_simultaneous_crash(obs, n, 0.01)
        elif name == "c3":
            b = W.c3_correlated_partition(obs, np.asarray(v.getRing(0)), n, 0.05)
        else:
            jo = np.asarray([v.getExpectedObserversOf(n + j) for j in range(nj)], np.int32)
            b = W.c5_churn(obs, jo, n, 3, nj)
        ring0 = np.asarray(v.getRing(0), np.int32)
        blocked = W.blocked_by_receiver(b.blocked, ring0, 0, n)
        sim = orc.ClusterSim(v, K, H, L, n)
        cfg = v.getCurrentConfigurationId()
        o_len, o_ann, o_ids, o_off = sim.apply_batch(b.src, b.dst, b.ring, b.status, np.full(len(b), cfg, np.int64), blocked=blocked)
        r0 = int(np.nonzero(o_len)[0][0])
        cases.append({
            "name": name, "n": n, "n_joiners": nj, "K": K, "H": H, "L": L, "configuration_id": cfg,
            "cells": {"src": b.src.tolist(), "dst": b.dst.tolist(), "ring": b.ring.tolist(), "status": b.status.tolist()},
            "blocked_receivers": np.nonzero(blocked)[0].tolist(),
            "proposal_len": sorted(set(o_len.tolist())),
            "proposal_canonical": o_ids[o_off[r0]: o_off[r0 + 1]].tolist(),
            "announced_count": int(o_ann.sum()),
            "expected_cut": b.expected_cut.tolist(),
        })
    with open(os.path.join(HERE, "cut_scenarios.json"), "w") as f:
        json.dump(cases, f)


def paxos_rule_cases():
    """selectProposalUsingCoordinatorRule (Paxos.java:271-328) on seeded message lists: values are small ints (0 = empty list),
    the answer is the INDEX of the message whose vval is chosen (-1 = empty)."""
    import random
    rng = random.Random(20260922)
    u = orc.Universe()
    vals = {0: []}
    for i in range(1, 6):
        vals[i] = [u.add("v", 10 * i + j) for j in range(1 + i % 3)]
    cases = []
    for _ in range(40):
        N = rng.choice([4, 5, 6, 9, 16, 33, 100])
        m = rng.randint(1, 2 * N)
        ranks = [(rng.randint(0, 2), rng.choice([-3, 0, 1, 7, 2**31 - 1])) for _ in range(rng.randint(1, 3))]
        msgs = [{"vrnd": rng.choice(ranks), "value": rng.randint(0, rng.randint(1, 5))} for _ in range(m)]
        px = orc.ClassicPaxos(u, u.add("me", 1), 7, 1, N)
        chosen = px.selectProposalUsingCoordinatorRule([{"vrnd": x["vrnd"], "vval": vals[x["value"]]} for x in msgs])
        # the rule returns a value; the fixtures pin the first message carrying it among those the rule could have taken it from
        cases.append({"N": N, "vrnd": [list(x["vrnd"]) for x in msgs], "value": [x["value"] for x in msgs],
                      "chosen_value": next((k for k, v in vals.items() if v == chosen), None)})
    with open(os.path.join(HERE, "paxos_rule_cases.json"), "w") as f:
        json.dump(cases, f)


def failure_detector_stream():
    """alerts of 14 failure-detector intervals (PingPongFailureDetector.java:75-85) of a 60-node view under a fixed scenario"""
    n = 60
    hb, off, ports = W.packed_endpoints(0, n)
    u = orc.Universe()
    tags = u.add_bulk(hb, off, ports)
    hi, lo = W.node_ids(0, n)
    v = orc.MembershipView(u, K, tags, hi, lo)
    sim = orc.FdSim(v, K, np.arange(n))
    flags = np.zeros(n, np.uint8)
    flags[[4, 17]] = orc.FD_CRASHED
    flags[30] = orc.FD_INGRESS_BLOCKED
    flags[41] = orc.FD_EGRESS_BLOCKED
    out = {"n": n, "K": K, "flags": flags.tolist(), "cfg": 99, "intervals": [sim.tick(flags, 99) for _ in range(14)]}
    with open(os.path.join(HERE, "failure_detector_stream.json"), "w") as f:
        json.dump(out, f)


def xxh64_vectors():
    """XXH64 digests from two implementations independent of the oracle: python-xxhash (bytes, and hashInt / hashLong as
    little-endian bytes) and the system libxxhash.  Not oracle pins: tests/test_oracle_xxh64.py holds the oracle to them."""
    import ctypes
    import random
    import struct
    import xxhash
    lx = ctypes.CDLL("libxxhash.so.0")
    lx.XXH64.restype = ctypes.c_uint64
    lx.XXH64.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint64]
    rng = random.Random(7)
    out = {"python_xxhash": {"version": xxhash.VERSION, "bytes": [], "int": [], "long": []}, "libxxhash": []}
    for n in list(range(0, 80)) + [127, 128, 129, 1000]:
        data = bytes(rng.getrandbits(8) for _ in range(n))
        out["python_xxhash"]["bytes"].append([data.hex(), [[seed, xxhash.xxh64(data, seed=seed).intdigest()]
                                                           for seed in (0, 1, 2, 9, 0xDEADBEEF, 2**63 + 5)]])
    for seed in range(10):
        for v in (0, 1, -1, 1234, 65535, 2**31 - 1, -(2**31)):
            out["python_xxhash"]["int"].append([v, seed, xxhash.xxh64(struct.pack("<i", v), seed=seed).intdigest()])
        for v in (0, 1, -1, 2**63 - 1, -(2**63), 0x0123456789ABCDEF):
            out["python_xxhash"]["long"].append([v, seed, xxhash.xxh64(struct.pack("<q", v), seed=seed).intdigest()])
    rng = random.Random(11)
    for n in (0, 1, 3, 4, 7, 8, 9, 15, 31, 32, 33, 63, 64, 100):
        data = bytes(rng.getrandbits(8) for _ in range(n))
        out["libxxhash"].append([data.hex(), [[seed, lx.XXH64(data, n, seed)] for seed in (0, 3, 9)]])
    with open(os.path.join(HERE, "xxh64_vectors.json"), "w") as f:
        json.dump(out, f)


if __name__ == "__main__":
    orc.build()
    ring_keys()
    cut_scenarios()
    paxos_rule_cases()
    failure_detector_stream()
    xxh64_vectors()
    print("wrote", os.listdir(HERE))
