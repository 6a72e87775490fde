#!/usr/bin/env python
"""bench.py — alert cells / second to a converged, quorum-decided cut (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c5|c4|c3|c2] [--nodes n]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic alert stream, from an empty detector to the decision:
    [per batch] filter -> per-receiver cut detection (subject-bucketed kernels) -> implicit invalidation -> per-node proposal
    fingerprints -> fast-round vote tally [-> NCCL histogram all-reduce when sharded] -> decision on the host.
Workloads (SURVEY.md §8d):
    c5 (default)  BASELINE config 5: 1,000,000 virtual nodes, K=10 H=9 L=4, ONE 1 % churn batch (5,000 crashes + 5,000 joins,
                  ~10^5 alert cells), every receiver gets the batch in array order
    c4            BASELINE config 4: 100,000 nodes, 1 % flip-flop stream over T = 8 batches with 1/4 duplicate re-sends, every
                  receiver applies each batch in ITS OWN permuted order, detector state carried from batch to batch; the step
                  ends with the batch in which the cut is decided (duplicates count as applied cells).  --stream sequence
                  (default): the 8 batches are handed over in ONE rapid_cd_apply_batches call — handleMessage once per batch
                  with the announcedProposal gating between them, computed in one pass over the state; --stream batches: 8 calls
    c3 / c2       BASELINE configs 3 / 2 (10,000-node correlated partition / 2,000-node simultaneous crash), one batch
Receivers are sharded over the GPUs by ring-0 range; the cluster size stays fixed ("scaling": "strong").

`value`  : cells of one step / device time of one step, with the cell arrays resident in HBM when the timed region starts.
           The timed region is ONE device-side stopwatch over all K steps (a CUDA event on the detector's stream before the
           first step, one on the tally's stream after the last): kernels, the epoch resets between steps, the one host
           synchronisation per batch (the decision) and every idle gap in between are inside it.  Max over ranks.
`e2e`    : the same through the host-facing C ABI: host arrays in, H2D copies, kernels, decision read back — wall clock.
--impl reference : the reference's own CPU path.  The reference is Java and cannot be built or run in this image (no JDK), so
           this times oracle/'s literal C++ restatement of it (kind "port") on all host cores on a FIXED sample of the same
           workload (8 virtual nodes per thread x the full stream, one FastPaxos instance per thread x 4096 votes); `value` is
           the measured rate of that sample, the whole-cluster extrapolation is a labelled side field.
"""
import argparse
import atexit
import ctypes as C
import json
import os
import signal
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K, H, L = 10, 9, 4          # Cluster.java:72-74
METRIC = "alert_cells_per_sec_to_converged_cut"
UNIT = "cells/s"
DEFAULT_NODES = {"c5": 1_000_000, "c4": 100_000, "c3": 10_000, "c2": 2_000}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--nodes", type=int, default=0, help="cluster size (default: the BASELINE size of the workload)")
    p.add_argument("--workload", default="c5", choices=["c5", "c4", "c3", "c2"])
    p.add_argument("--kernel", default="auto", choices=["auto", "bucketed", "sweep"])
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-carried", action="store_true", help="skip the extra carried-state (read-modify-write) measurement of c5")
    p.add_argument("--stream", default="sequence", choices=["sequence", "batches"],
                   help="c4 only: deliver the 8-batch stream as ONE rapid_cd_apply_batches call (one pass over the detector state, "
                        "checked on the device, batch-by-batch replay if refused) or as 8 separate calls")
    p.add_argument("--emulate-shard", type=int, default=0,
                   help="tuning aid: run rank 0's shard of a G-way run on ONE GPU without NCCL (no decision is reached)")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write what the last timed step computed as DIR/<name>.npy (float32 / float64), to compare two builds "
                        "output for output")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    if a.nodes <= 0:
        a.nodes = DEFAULT_NODES[a.workload]
    return a


def n_joiners(args):
    return args.nodes // 200 if args.workload == "c5" else 0


class Stream:
    """The workload: a list of alert batches applied in order to detectors that start empty."""

    def __init__(self, args, W, obs, joiner_obs, ring0):
        n = args.nodes
        self.perm = [None]
        if args.workload == "c5":
            self.batches = [W.c5_churn(obs, joiner_obs, n, n // 200, n // 200)]
        elif args.workload == "c2":
            self.batches = [W.c2_simultaneous_crash(obs, n, 0.01)]
        elif args.workload == "c3":
            self.batches = [W.c3_correlated_partition(obs, ring0, n, 0.05)]
        else:
            self.batches = W.c4_flip_flop_stream(obs, n, 0.01, T=8)
            self.perm = [b.meta["perm_seed"] for b in self.batches]
        self.blocked = self.batches[0].blocked
        self.expected_cut = self.batches[-1].expected_cut
        self.cells = [len(b) for b in self.batches]
        # subjects first seen in batch t ("fresh": their rows are written, never read) / seen before ("carried": 2 B read + 2 B written)
        seen = np.zeros(n + n_joiners(args) + 1, bool)
        self.fresh, self.carried = [], []
        for b in self.batches:
            u = np.unique(b.dst)
            self.fresh.append(int((~seen[u]).sum()))
            self.carried.append(int(seen[u].sum()))
            seen[u] = True
        self.subjects = int(seen.sum())

    def name(self, args, upto):
        n, A = args.nodes, sum(self.cells[: upto + 1])
        if args.workload == "c5":
            return "C5 %d-node K=10 H=9 L=4, 1%% churn batch (%d DOWN + %d UP subjects, %d cells)" % (n, n // 200, n // 200, A)
        if args.workload == "c2":
            return "C2 %d-node K=10 H=9 L=4, 1%% simultaneous crash (%d subjects, %d cells)" % (n, self.subjects, A)
        if args.workload == "c3":
            return "C3 %d-node K=10 H=9 L=4, 5%% correlated one-way partition (%d subjects, %d cells)" % (n, self.subjects, A)
        return ("C4 %d-node K=10 H=9 L=4, 1%% flip-flop stream: %d subjects, %d batches with 1/4 duplicate re-sends, per-receiver "
                "permuted order, state carried; decided in batch %d after %d cells" % (n, self.subjects, len(self.batches), upto, A))


# --------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# --------------------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.rows, self.proc, self.dev, self.t_begin = [], None, device_index, 0.0
        self.first = threading.Event()

    def start(self):
        """Start ONE polling nvidia-smi and wait until it delivers its first row: its start-up (NVML init over every GPU of
        the box) must not overlap the timed region, or it slows the rank that shares the GPU with it."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self._reap)        # a run that fails while the poller is stopped must not leave it behind
            threading.Thread(target=self._pump, daemon=True).start()
            self.first.wait(10.0)
        except OSError:
            self.proc = None

    def _reap(self):
        if self.proc.poll() is None:
            self.proc.kill()
        self.proc.wait()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))
            self.first.set()

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def pause(self):
        """One poll stalls the GPU it queries for ~1 ms (measured: 1 step in 50 of a 2-GPU run takes +0.85 ms with the poller,
        none without) — more than a whole 8-GPU step.  The poller is therefore stopped across the K device-timed steps (a sample
        is taken right before) and resumed right after: its samples bracket that loop within one period and run through the
        end-to-end timed loop, which executes the same kernels."""
        if self.proc is None:
            return
        n = len(self.rows)
        t0 = time.perf_counter()
        while len(self.rows) == n and time.perf_counter() - t0 < 0.3:      # a fresh sample under the warm-up load
            time.sleep(0.005)
        try:
            self.proc.send_signal(signal.SIGSTOP)
            self.paused = True
        except OSError:
            pass

    def resume(self):
        if self.proc is not None and getattr(self, "paused", False):
            try:
                self.proc.send_signal(signal.SIGCONT)
            except OSError:
                pass
            self.paused = False

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.resume()
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        timed = [r for t, r in self.rows if t >= self.t_begin]
        for r in (timed if timed else [r for _, r in self.rows]):
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "poll": "nvidia-smi -lms 100 from before the timed region to the end of the run (through the end-to-end timed loop); "
                        "stopped across the K device-timed steps, with a sample right before and after them, because one poll stalls "
                        "the polled GPU for ~1 ms (more than an 8-GPU step)"}


def ncu_traffic(args, gpus, suffix=""):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the committed ncu --set full
    capture of this very configuration (profiles/traffic.json); None if that configuration was not captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get("%s:%d:%d%s" % (args.workload, args.nodes, gpus, suffix))
    except Exception:
        return None


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------------------------
# CPU legs (oracle): cpu_baseline at N=1 and --impl reference
# --------------------------------------------------------------------------------------------------------------
class CpuProblem:
    """The workload inside the oracle (built once; construction is outside every timed region)."""

    NODES_PER_THREAD = 8        # sampled virtual nodes per host thread
    VOTES = 4096                # votes handed to every sampled FastPaxos instance

    def __init__(self, args):
        from oracle import oracle_py as orc
        from rapid_b200 import workloads as W
        self.orc, self.args = orc, args
        n, nj = args.nodes, n_joiners(args)
        t0 = time.time()
        hb, off, ports = W.packed_endpoints(0, n + nj)
        self.u = orc.Universe()
        tags = self.u.add_bulk(hb, off, ports)
        hi, lo = W.node_ids(0, n)
        self.view = orc.MembershipView(self.u, K, tags[:n], hi, lo)
        self.cfg = self.view.getCurrentConfigurationId()
        obs = lambda ids: self.view.tables(ids)[0]
        joiner_obs = np.asarray([self.view.getExpectedObserversOf(n + j) for j in range(nj)], np.int32).reshape(nj, K)
        ring0 = np.asarray(self.view.getRing(0), np.int32)
        self.ring0 = ring0
        self.st = Stream(args, W, obs, joiner_obs, ring0)
        self.live = int(n - int(self.st.blocked.sum()))
        self.setup_s = time.time() - t0

    def measure(self, threads):
        """Time the literal C++ restatement on a FIXED sample: `8 x threads` live virtual nodes apply the whole stream (all
        threads busy), then `threads` FastPaxos instances count 4096 of the votes each.  Everything reported is measured on
        that sample; the whole-cluster figure is a labelled extrapolation."""
        orc, st, n = self.orc, self.st, self.args.nodes
        W = __import__("rapid_b200.workloads", fromlist=["x"])
        blocked_r = W.blocked_by_receiver(st.blocked, self.ring0, 0, n)
        live_pos = np.nonzero(blocked_r == 0)[0]
        Rs = int(min(self.NODES_PER_THREAD * threads, len(live_pos)))
        # the sampled receivers are the first Rs LIVE ring-0 positions; the oracle simulates positions [0, hi) and we block the rest
        hi = int(live_pos[Rs - 1]) + 1
        sim = orc.ClusterSim(self.view, K, H, L, hi)
        t_apply, cells, decided_batch, prop = 0.0, 0, None, None
        for bi, b in enumerate(st.batches):
            out = sim.apply_batch(b.src, b.dst, b.ring, b.status, np.full(len(b), self.cfg, np.int64), blocked=blocked_r[:hi],
                                  perm_seed=st.perm[bi], threads=threads)
            t_apply += sim.last_seconds
            cells += len(b)
            o_len, o_ann, o_ids, o_off = out
            if o_len.max() > 0:
                r = int(np.nonzero(o_len)[0][0])
                prop = o_ids[o_off[r]: o_off[r + 1]]
                if len(prop) == len(st.expected_cut) and (np.sort(prop) == st.expected_cut).all():
                    decided_batch = bi
                    break
        assert decided_batch is not None, "oracle did not converge to the expected cut"
        Vs = int(min(self.VOTES, self.live))
        senders = np.arange(Vs, dtype=np.int32)
        t_tally = orc.sim_tally(self.u, self.cfg, n, threads, senders, np.full(Vs, self.cfg, np.int64), np.zeros(Vs, np.int32),
                                np.array([0, len(prop)], np.int32), prop, threads=threads)[3]
        apply_whole = t_apply * self.live / Rs
        tally_whole = t_tally * (self.live / threads) * (self.live / Vs)
        return {
            "value": cells / (t_apply + t_tally), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": ("literal C++ restatement of MultiNodeCutDetector / MembershipService batch handler / FastPaxos tally "
                       "(oracle/, g++ -O2; the Java reference cannot run here: no JDK).  MEASURED: %d of the %d live virtual nodes "
                       "apply the whole %d-cell stream (%d batch(es)) on %d threads in %.3f s, then %d FastPaxos instances count "
                       "%d votes each (every vote re-hashes the %d-endpoint proposal like List.hashCode) in %.3f s; value = cells "
                       "/ (%.3f + %.3f s)" % (Rs, self.live, cells, decided_batch + 1, threads, t_apply, threads, Vs, len(prop),
                                              t_tally, t_apply, t_tally)),
            "sampled_nodes": Rs, "sampled_votes_per_instance": Vs, "apply_s": t_apply, "tally_s": t_tally,
            "apply_node_cells_per_s": Rs * cells / t_apply, "tally_votes_per_s": threads * Vs / max(t_tally, 1e-9),
            "extrapolated_whole_cluster": {
                "value": cells / (apply_whole + tally_whole), "apply_only_value": cells / apply_whole, "unit": UNIT,
                "how": "NOT measured: apply time x (%d live nodes / %d sampled) + tally time x (%d nodes / %d instances) x (%d "
                       "votes / %d) — every one of the reference's N processes runs its own detector AND its own tally of N "
                       "votes, while the GPU arm runs N detectors and ONE cluster-wide tally" % (
                           self.live, Rs, self.live, threads, self.live, Vs)},
            "setup_s": round(self.setup_s, 1),
        }, cells, decided_batch


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle_py as orc
    threads = max(1, orc.hardware_threads())
    prob = CpuProblem(args)
    log("[reference] setup %.1fs (n=%d), %d threads" % (prob.setup_s, args.nodes, threads))
    vals = []
    for i in range(args.warmup + args.steps):
        d, cells, upto = prob.measure(threads)
        if i >= args.warmup:
            vals.append(d)
    v = float(np.mean([x["value"] for x in vals]))
    d = dict(vals[-1])
    d["value"] = v
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
        "warmup": args.warmup, "ms_per_step": 1e3 * cells / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u16", "data": "synthetic",
        "config": {"workload": prob.st.name(args, upto), "nodes": args.nodes, "cells": cells, "subjects": prob.st.subjects,
                   "K": K, "H": H, "L": L,
                   "note": "CPU arm: a bounded sample of the workload (see cpu_baseline.sample); value is the sample's measured rate"},
        "cpu_baseline": d,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# --------------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import rapid_b200 as rb
    from rapid_b200 import _native as N
    from rapid_b200 import workloads as W

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log("note: WORLD_SIZE=%d but --gpus %d; using WORLD_SIZE" % (world, args.gpus))
    G = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (librapid_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    if G > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    n, nj = args.nodes, n_joiners(args)
    t0 = time.time()
    hb, off, ports = W.packed_endpoints(0, n + nj)
    view = rb.MembershipView.from_packed(K, hb[: off[n]], off[: n + 1], ports[:n], device=local)
    if nj:
        jh = hb[off[n]: off[n + nj]]
        first = C.c_int32(0)
        N.check(N.lib().rapid_view_register_joiners(view._h, nj, N.ptr(np.ascontiguousarray(jh)),
                                                    N.ptr(np.ascontiguousarray(off[n:] - off[n])),
                                                    N.ptr(np.ascontiguousarray(ports[n:])), C.byref(first)))
        assert first.value == n
    obs, _ = view.tables()
    ring0 = view.getRing(0)
    joiner_obs = view.joinerTables() if nj else np.zeros((0, K), np.int32)
    st = Stream(args, W, obs, joiner_obs, ring0)
    T = len(st.batches)
    hi, lo = W.node_ids(0, n)
    cfg = view.getCurrentConfigurationId(hi, lo)
    Gs = args.emulate_shard if (args.emulate_shard > 1 and G == 1) else G      # sharding arithmetic only
    begin = rank * n // Gs
    R = (rank + 1) * n // Gs - begin
    emulated = Gs != G
    blocked = W.blocked_by_receiver(st.blocked, ring0, begin, R)
    cl = rb.VirtualCluster(view, H, L, n_receivers=R, receiver_begin=begin, kernel=args.kernel, max_subjects=st.subjects + 64)
    fp = rb.FastPaxos(cfg, n, sender_capacity=n, device=local)
    comm = None
    if G > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.from_numpy(rb.NcclComm.unique_id()))
        dist.broadcast(uid, 0)
        comm = rb.NcclComm(rank, G, uid.cpu().numpy(), local)
    want = rb.proposal_fingerprint(st.expected_cut)
    log("[rank %d] setup %.1fs: n=%d receivers=[%d,%d) batches=%d cells=%d subjects=%d" % (
        rank, time.time() - t0, n, begin, begin + R, T, sum(st.cells), st.subjects))

    # device-resident inputs (torch only holds the memory)
    dev = [(torch.from_numpy(b.dst).cuda(), torch.from_numpy(b.ring).cuda(), torch.from_numpy(b.status).cuda()) for b in st.batches]
    d_blocked = torch.from_numpy(blocked).cuda()
    asynchronous = args.kernel != "sweep"
    sequence = args.workload == "c4" and args.stream == "sequence" and args.kernel != "sweep"
    if sequence:
        cat = (torch.from_numpy(np.concatenate([b.dst for b in st.batches])).cuda(),
               torch.from_numpy(np.concatenate([b.ring for b in st.batches])).cuda(),
               torch.from_numpy(np.concatenate([b.status for b in st.batches])).cuda())
        seq_off = np.concatenate([[0], np.cumsum(st.cells)]).astype(np.int64)
        assert all(st.perm[t] == st.perm[0] + t for t in range(T))        # batch b is permuted with perm_seed + b
        host_cat = (np.concatenate([b.dst for b in st.batches]), np.concatenate([b.ring for b in st.batches]),
                    np.concatenate([b.status for b in st.batches]))

    acc = {"apply": 0.0, "main": 0.0, "tally": 0.0, "launches": 0, "main_by_batch": [0.0] * T, "calls": [0] * T}

    def step_device():
        """clear -> every batch of the stream ENQUEUED (batch, then its tally, ordered on the device) -> ONE host synchronisation:
        the decision and the index of the batch that produced it.  Votes after the decision are ignored on the device."""
        if T == 1 and asynchronous:
            # the whole epoch (resets, the batch, its tally) enqueued by one C call; the decision is the step's one host synchronisation
            d_dst, d_ring, d_status = dev[0]
            fp.epochAsync(cl, cfg, st.cells[0], d_dst.data_ptr(), d_ring.data_ptr(), d_status.data_ptr(), comm=comm,
                          blocked_dev=d_blocked.data_ptr(), perm_seed=st.perm[0])
            res = fp.result()
            return res, (res.decided_in if res.decided_in is not None and res.decided_in >= 0 else None)
        cl.clear()
        fp.reset(cfg)
        if sequence:
            # the whole stream in one call (one host synchronisation inside it: the outcome of the device-side check), then the tally
            cl.handleBatchesDevice(cfg, int(seq_off[-1]), cat[0].data_ptr(), cat[1].data_ptr(), cat[2].data_ptr(), seq_off,
                                   blocked_dev=d_blocked.data_ptr(), perm_seed=st.perm[0])
            fp.tallyClusterAsync(cl, comm)
            res = fp.result()
            return res, (T - 1 if res.decided else None)
        for bi in range(T):
            d_dst, d_ring, d_status = dev[bi]
            cl.handleBatchDevice(cfg, st.cells[bi], d_dst.data_ptr(), d_ring.data_ptr(), d_status.data_ptr(),
                                 blocked_dev=d_blocked.data_ptr(), perm_seed=st.perm[bi], wait=not asynchronous)
            fp.tallyClusterAsync(cl, comm)
        res = fp.result()
        return res, (res.decided_in if res.decided_in is not None and res.decided_in >= 0 else None)

    def step_profile():
        """the same stream with a host synchronisation after every call, to read the per-call device times (NOT the timed loop)"""
        cl.clear()
        fp.reset(cfg)
        res = None
        if sequence:
            cl.handleBatchesDevice(cfg, int(seq_off[-1]), cat[0].data_ptr(), cat[1].data_ptr(), cat[2].data_ptr(), seq_off,
                                   blocked_dev=d_blocked.data_ptr(), perm_seed=st.perm[0])
            res = fp.tallyCluster(cl, comm)
            tot, main = cl.lastDeviceMs()
            acc["apply"] += tot; acc["main"] += main; acc["tally"] += fp.lastDeviceMs()
            acc["main_by_batch"][0] += main; acc["calls"][0] += 1
            acc["launches"] += cl.lastPath()[1] + 3 + fp.lastLaunches() + 2     # + announced_in kernels, clear(), reset()
            return res
        for bi in range(T):
            d_dst, d_ring, d_status = dev[bi]
            cl.handleBatchDevice(cfg, st.cells[bi], d_dst.data_ptr(), d_ring.data_ptr(), d_status.data_ptr(),
                                 blocked_dev=d_blocked.data_ptr(), perm_seed=st.perm[bi], wait=True)
            res = fp.tallyCluster(cl, comm)
            tot, main = cl.lastDeviceMs()
            acc["apply"] += tot; acc["main"] += main; acc["tally"] += fp.lastDeviceMs()
            acc["main_by_batch"][bi] += main; acc["calls"][bi] += 1
            acc["launches"] += cl.lastPath()[1] + fp.lastLaunches() + (2 if bi == 0 else 0)     # + clear(), reset()
        return res

    def step_host():
        cl.clear()
        fp.reset(cfg)
        res = None
        if sequence:
            cl.handleBatches(cfg, None, host_cat[0], host_cat[1], host_cat[2], seq_off, blocked=blocked, perm_seed=st.perm[0],
                             read_outputs=False)
            return fp.tallyCluster(cl, comm)
        for bi, b in enumerate(st.batches):
            cl.handleBatch(cfg, None, b.dst, b.ring, b.status, blocked=blocked, perm_seed=st.perm[bi], read_outputs=False)
            res = fp.tallyCluster(cl, comm)
            if res.decided:
                break
        return res

    def barrier():
        torch.cuda.synchronize()
        if G > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def check(res):
        assert emulated or (res.decided and (res.hash, res.hash2, res.length) == (want[0], want[1], len(st.expected_cut))), \
            "decision differs from the expected cut: %r" % (res,)

    clocks = Clocks(local)
    if rank == 0 and not os.environ.get("RAPID_B200_NO_CLOCKS"):
        clocks.start()             # polls from here on; samples taken from the start of the timed region are reported
    upto = T - 1
    for _ in range(max(3, args.warmup)):
        res, upto_w = step_device()
        check(res)
        upto = upto_w if upto_w is not None else T - 1
    cells_step = sum(st.cells[: upto + 1])        # cells delivered up to and including the deciding batch

    import gc
    gc.collect()
    gc.disable()                   # no collector pauses inside the timed loops (one late rank stalls the whole all-reduce)
    clocks.mark_begin()
    if rank == 0:
        clocks.pause()
    barrier()                      # nothing rank-specific between the barrier and the first timed step
    per_step = []
    w0 = time.perf_counter()
    cl.timerStart()                # device-side stopwatch over ALL the steps: kernels, resets, host syncs, idle gaps
    for _ in range(args.steps):
        t_step = time.perf_counter()
        res, _ = step_device()
        per_step.append((time.perf_counter() - t_step) * 1e3)
    dev_ms = fp.timerStop(cl)
    if rank == 0:
        clocks.resume()
    barrier()
    wall_ms = (time.perf_counter() - w0) * 1e3
    if os.environ.get("RAPID_B200_STEP_TIMES"):
        log("[rank %d] per-step host wall ms: %s" % (rank, " ".join("%.3f" % x for x in per_step)))
    check(res)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cl, res, begin, "rank%d_" % rank if G > 1 else "", G)
    prof_steps = max(2, min(args.steps, 5))
    for _ in range(prof_steps):
        check(step_profile())
    for k in ("apply", "main", "tally"):
        acc[k] *= args.steps / prof_steps          # per-call device times are reported per step of the timed loop
    acc["main_by_batch"] = [x * args.steps / prof_steps for x in acc["main_by_batch"]]
    acc["calls"] = [c * args.steps // prof_steps for c in acc["calls"]]
    acc["launches"] = acc["launches"] * args.steps // prof_steps
    log("[rank %d] per step: device stopwatch %.3f ms (host wall median %.3f max %.3f ms); per-call device times from %d profiled "
        "steps: apply %.3f ms (dominant kernel %.3f ms), tally %.3f ms" % (
            rank, dev_ms / args.steps, float(np.median(per_step)), max(per_step), prof_steps, acc["apply"] / args.steps,
            acc["main"] / args.steps, acc["tally"] / args.steps))
    # end-to-end through the host-facing ABI (host arrays, H2D, reset, kernels, decision back)
    for _ in range(2):
        step_host()
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        res = step_host()
    barrier()
    e2e_ms = (time.perf_counter() - e0) * 1e3 / args.steps
    check(res)

    # the carried path of C5 (read-modify-write rows): the same batch delivered as two halves, no clear() in between
    carried = None
    if args.workload == "c5" and not args.no_carried and asynchronous:
        b = st.batches[0]
        A, half = len(b), len(b) // 2
        u1 = np.unique(b.dst[:half]); u2 = np.unique(b.dst[half:])
        S_carried = int(np.isin(u2, u1).sum()); S_fresh2 = len(u2) - S_carried
        d_dst, d_ring, d_status = dev[0]
        ms2, reps = 0.0, max(3, min(args.steps, 10))
        for i in range(reps + 1):
            cl.clear(); fp.reset(cfg)
            cl.handleBatchDevice(cfg, half, d_dst.data_ptr(), d_ring.data_ptr(), d_status.data_ptr(), blocked_dev=d_blocked.data_ptr())
            cl.handleBatchDevice(cfg, A - half, d_dst.data_ptr() + 4 * half, d_ring.data_ptr() + half, d_status.data_ptr() + half,
                                 blocked_dev=d_blocked.data_ptr())
            res = fp.tallyCluster(cl, comm)
            if i:
                ms2 += cl.lastDeviceMs()[1]
        check(res)
        alg2 = (4 * S_carried + 2 * S_fresh2) * R + 5 * R
        carried = {"kernel": "k_apply_uniform (second half of the batch: %d carried subjects read-modify-write 4 B per (subject, "
                             "receiver), %d fresh ones write 2 B)" % (S_carried, S_fresh2),
                   "kernel_ms": ms2 / reps, "algorithmic_bytes_per_launch": int(alg2)}
    gc.enable()
    clk = clocks.stop() if rank == 0 else None

    # per-rank breakdown (diagnosis of a late rank: every other rank's wait for it shows up in their tally time)
    mine = torch.tensor([float(np.median(per_step)), max(per_step), acc["apply"] / args.steps, acc["tally"] / args.steps,
                         acc["main"] / args.steps], dtype=torch.float64, device="cuda")
    if G > 1:
        allr = [torch.zeros_like(mine) for _ in range(G)]
        dist.all_gather(allr, mine)
    else:
        allr = [mine]
    per_rank = [[round(float(x), 4) for x in r.cpu()] for r in allr]
    t = torch.tensor([dev_ms, acc["main"], e2e_ms, wall_ms], dtype=torch.float64, device="cuda")
    if G > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, main_ms, e2e_ms, wall_ms = [float(x) for x in t.cpu()]
    ms_per_step = dev_ms / args.steps
    main_per = main_ms / args.steps

    line = None
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        # algorithmic bytes of the dominant kernel over one step: per batch, 2 B written per (fresh subject, receiver), 4 B (2 read
        # + 2 written) per (carried subject, receiver), + flags / blocked read once per receiver
        alg = sum((2 * st.fresh[bi] + 4 * st.carried[bi]) * R + 5 * R for bi in range(upto + 1))
        n_kernel_launches = upto + 1
        seq_stats = None
        if sequence:
            # ONE pass over the state for the whole stream: every subject of the stream is first seen in this call (the step starts
            # from clear()), so its row is written once and never read: 2 B per (subject, receiver)
            alg = 2 * st.subjects * R + 5 * R
            n_kernel_launches = 1
            seq_stats = cl.sequenceStats()
        achieved = alg / (main_per * 1e-3) / 1e9 if main_per > 0 else 0.0
        path = cl.lastPath()[0]
        kname = {1: "k_sweep", 2: "k_apply_uniform<false>", 3: "k_apply_generic", 4: "k_apply_uniform<true> (permuted delivery)"}.get(path)
        if sequence:
            kname += " [sequence of batches, one pass]"
        line = {
            "metric": METRIC, "value": cells_step / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": G, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u16", "data": "synthetic",
            "config": {"workload": st.name(args, upto), "nodes": n, "cells": cells_step, "batches": upto + 1,
                       "alert_messages": sum(b.n_messages() for b in st.batches[: upto + 1]),
                       "subjects": st.subjects, "K": K, "H": H, "L": L, "receivers_per_gpu": R,
                       "parallelism": "virtual nodes sharded by ring-0 range x%d; one NCCL histogram all-reduce per batch" % G,
                       "l2": ("per-step mask state %.2f GB per GPU vs 126 MB L2: %s" % (
                           2 * st.subjects * R / 1e9, "inputs larger than L2, no flush" if 2 * st.subjects * R > 4 * 126e6 else
                           "fits in L2 — every step starts from clear() and rewrites it; reported as is")),
                       "timing": "one device-side stopwatch over all steps (CUDA event on the detector's stream before the first "
                                 "step, on the tally's stream after the last): kernels, epoch resets, the one host sync per step "
                                 "(the decision; every batch and its tally are enqueued, all %d batches of the stream are "
                                 "applied) and idle gaps included; max over ranks.  Per-kernel times come from extra profiled "
                                 "steps with a host sync per call" % T,
                       "kernel_path": {1: "sweep", 2: "bucketed-uniform", 3: "bucketed-generic", 4: "bucketed-permuted"}.get(path)},
            "wall_ms_per_step": wall_ms / args.steps,
            "device_ms_in_calls_per_step": {"apply": acc["apply"] / args.steps, "tally": acc["tally"] / args.steps},
            "per_rank_ms": {"host_wall_per_step_median": [r[0] for r in per_rank], "host_wall_per_step_max": [r[1] for r in per_rank],
                            "apply_device": [r[2] for r in per_rank], "tally_device_incl_allreduce_wait": [r[3] for r in per_rank],
                            "dominant_kernel": [r[4] for r in per_rank]},
            "clocks": clk,
            "e2e": {"value": cells_step / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(sum(st.cells[bi] * 6 + R for bi in range(upto + 1))),
                    "d2h_bytes_per_step": (64 + 36) * (upto + 1)},
            "gpu_launches": int(acc["launches"]),
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(args, G), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(alg / n_kernel_launches), "launches_per_step": n_kernel_launches,
                         "kernel_ms": main_per / n_kernel_launches, "kernel_ms_per_step": main_per,
                         "kernel_share_of_step": main_per / ms_per_step if ms_per_step else None,
                         "per_batch": [{"fresh_subjects": st.fresh[bi], "carried_subjects": st.carried[bi],
                                        "kernel_ms": acc["main_by_batch"][bi] / max(1, acc["calls"][bi])} for bi in range(upto + 1)]},
        }
        if sequence:
            line["config"]["stream"] = ("the %d batches handed over in ONE rapid_cd_apply_batches call: handleMessage once per batch with the "
                                        "announcedProposal gating between them, computed in one pass over the detector state after a "
                                        "device-side check per receiver (sequences served in one pass / replayed batch by batch so far: "
                                        "%d / %d)" % (T, seq_stats[0], seq_stats[1]))
            line["roofline"]["per_batch"] = None
            line["roofline"]["note"] = "one launch for the whole stream; all %d subjects are first seen in it: 2 B written per (subject, receiver)" % st.subjects
        if carried is not None:
            ach2 = carried["algorithmic_bytes_per_launch"] / (carried["kernel_ms"] * 1e-3) / 1e9
            carried.update({"bound": "hbm", "achieved": ach2, "peak": peak, "unit": "GB/s", "frac": ach2 / peak,
                            "traffic": ncu_traffic(args, G, ":carried")})
            line["roofline_carried"] = carried
    if G > 1:
        dist.barrier()
    if rank == 0:
        if not args.no_cpu_baseline and G == 1:
            try:
                from oracle import oracle_py as orc
                line["cpu_baseline"] = CpuProblem(args).measure(max(1, orc.hardware_threads()))[0]
            except Exception as e:       # the baseline is a reported extra; never lose the GPU line over it
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
        emit(line)
    if G > 1:
        dist.destroy_process_group()


DUMP_MAX_RECEIVERS = 1 << 20


def dump_outputs(d, cl, res, begin, prefix, G):
    """What the last timed step handed its caller, as DIR/<prefix><name>.npy:
        decision.npy              FastPaxos.result(): decided, hash (hi, lo), hash2 (hi, lo), length, count, votes_received,
                                  decided_in (-1: none)
        cut.npy                   the decided proposal (node ids, as getProposal lists them) of the first receiver holding it
        receivers.npy             ring-0 positions of the receivers the next three arrays describe
        proposal_fingerprint.npy  VirtualCluster.readOutputs(): per receiver hash (hi, lo), hash2 (hi, lo)
        proposal_len.npy, announced.npy
    uint64 fingerprints are split into 32-bit halves so that float64 holds them exactly.  Above DUMP_MAX_RECEIVERS receivers
    (over all ranks) a fixed seeded sample of them is written, which keeps the files under 64 MB."""
    os.makedirs(d, exist_ok=True)
    out = cl.readOutputs()
    R, cap = len(out.proposal_len), DUMP_MAX_RECEIVERS // G
    idx = np.arange(R) if R <= cap else np.sort(np.random.default_rng(0).choice(R, cap, replace=False))

    def halves(h):
        h = np.asarray(h, np.uint64)
        return np.stack([h >> np.uint64(32), h & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64)

    holders = np.nonzero((out.proposal_hash == res.hash) & (out.proposal_hash2 == res.hash2) & (out.proposal_len == res.length))[0]
    cut = cl.getProposal(int(holders[0])) if res.decided and len(holders) else []
    arrays = {
        "decision": np.concatenate([[float(res.decided)], halves([res.hash, res.hash2]).ravel(),
                                    [res.length, res.count, res.votes_received, -1 if res.decided_in is None else res.decided_in]]),
        "cut": np.asarray(cut, np.float64),
        "receivers": (begin + idx).astype(np.float64),
        "proposal_fingerprint": np.concatenate([halves(out.proposal_hash[idx]), halves(out.proposal_hash2[idx])], axis=1),
        "proposal_len": out.proposal_len[idx].astype(np.float32),
        "announced": out.announced[idx].astype(np.float32),
    }
    for name, a in arrays.items():
        np.save(os.path.join(d, prefix + name + ".npy"), a)
    log("outputs of the last timed step: %s (%d of %d receivers)" % (", ".join(prefix + k + ".npy" for k in arrays), len(idx), R))


_JSON_OUT = None


def emit(line):
    """the ONE JSON line, on the real stdout"""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _JSON_OUT
    args = parse()
    # Libraries print to stdout behind our back (NCCL's "NCCL version ..." banner): keep the real stdout for the JSON
    # line only and point fd 1 at stderr for everything else.
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
