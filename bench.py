#!/usr/bin/env python
"""bench.py — raft ticks/sec at 1,048,576 groups x 5 replicas (BASELINE.json configs[2]/[3]).

A *step* is one raft tick over every group of the job: the fused sm_100a tick kernel Step()s that tick's
append-acks / votes, applies proposals, runs the matchIndex -> commitIndex quorum (q-th largest of the
replica columns, term-gated) and the election timers, for all groups at once (SURVEY §8a rows a3-a16).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by the driver under torch.distributed.run (one rank per GPU); the groups are sharded
contiguously (strong scaling: the job stays 1,048,576 groups) and every tick ends with one all-gather of
the committed indices over NVLink (SURVEY §8e).

Timing rules followed: W >= 3 warm-up steps; every timed step reads a different pre-generated inbox slot and
the per-step footprint (state + inbox, ~260 MB at N=1) is larger than L2; for the standalone quorum kernel
every timed launch reads a never-touched column set after an explicit L2 flush; device time by CUDA events on
the engine's stream; max over ranks; clocks sampled during the timed region.
"""
from __future__ import annotations

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

G_TOTAL = 1 << 20
R = 5
SEED = 0x5EED0003
L2_BYTES = 126 * 1024 * 1024
MAX_SLOTS = 48


# ---------------------------------------------------------------------------------------------------
def steady_state(G: int, Rr: int, group_base: int, seed: int) -> dict:
    """BASELINE configs[2] initial state (SURVEY §8d): every group has a leader — this node, at replica slot
    g % R — term 1..8, last_index in [2^20, 2^40), follower match = last_index - geometric lag (mean ~4),
    99% of groups already past term_start."""
    from raftsql_b200 import empty_state

    rng = np.random.default_rng(seed + group_base)
    st = empty_state(G, Rr)
    g = np.arange(group_base, group_base + G, dtype=np.uint64)
    st["self_id"][:] = (g % np.uint64(Rr) + np.uint64(1)).astype(np.uint8)
    st["role"][:] = 2
    st["lead"][:] = st["self_id"]
    st["term"][:] = rng.integers(1, 9, size=G, dtype=np.uint64)
    st["vote"][:] = st["self_id"]
    st["last_index"][:] = rng.integers(2 ** 20, 2 ** 40, size=G, dtype=np.uint64)
    st["last_term"][:] = st["term"]
    lag = rng.geometric(0.2, size=(Rr, G)).astype(np.uint64)
    st["match"][:] = st["last_index"][None, :] - lag
    st["match"][st["self_id"] - 1, np.arange(G)] = st["last_index"]
    st["committed"][:] = st["last_index"] - np.uint64(40)
    gate_open = rng.random(G) < 0.99
    st["term_start"][:] = np.where(gate_open, st["committed"] - np.uint64(5), st["last_index"] - np.uint64(1))
    st["randomized_timeout"][:] = 10
    return st


def tick_bytes_per_group(Rr: int, inbox: str = "compact", ticks_per_launch: int = 1, write_through: bool = True) -> dict:
    """Algorithmic HBM bytes of one tick per group on the steady-state trace (DESIGN.md §4): every follower acks,
    proposals arrive on 3 of 4 ticks.
      "wide":    tick mode 0 — 64-bit state columns + the wide inbox columns;
      "bytes":   tick mode 3 — the byte inbox (R-1 sender bytes + 1 proposal byte + two base words) on 64-bit state;
      "compact": tick mode 4 — the byte inbox on compact state (32-bit offsets).  With ticks_per_launch = K > 1 the state
                 is read once per K ticks (registers carry it from tick to tick) and, unless write_through, also written
                 once per K ticks; every tick still reads its frame and writes its out word + commit-advance byte."""
    if inbox == "wide":
        read = 8 * 5 + 8 * Rr + Rr + 4 + 16 * (Rr - 1)  # meta,term,last_index,committed,term_start + match + types + prop + ack term/index
        write = 8 + 4 + 8 * (Rr - 1) + 8 + 12           # meta, out, acked match, committed, (last_index + self match) x 3/4
        return {"read": read, "write": write, "total": read + write}
    if inbox == "bytes":
        read = 8 * 5 + 8 * Rr + (Rr - 1) + 1 + 16
        write = 8 + 4 + 8 * (Rr - 1) + 8 + 12 + 8
        return {"read": read, "write": write, "total": read + write}
    K = max(1, ticks_per_launch)
    state_read = 1 + 8 + 4 + 4 + 4 * Rr            # flag, meta, commit, window, match[R] (last row = lastIndex)
    state_write = 8 + 4 + 4 + 4 * (Rr - 1) + 3     # meta, commit, window, acked match rows, lastIndex row x 3/4
    frame = (Rr - 1) + 1                           # sender bytes + proposal byte
    outputs = 4 + 1                                # out word + commit-advance byte
    read = frame + state_read / K
    write = outputs + (state_write if (write_through or K == 1) else state_write / K)
    return {"read": round(read, 2), "write": round(write, 2), "total": round(read + write, 2)}


def quorum_bytes_per_group(Rr: int) -> int:
    return 8 * Rr + 16  # SURVEY §8d: match[R] + committed + term_start, all u64 (reads)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        super().__init__(daemon=True)
        self.device, self.rows, self._halt = device, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.device)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._halt.wait(0.1)

    def finish(self) -> dict:
        self._halt.set()
        self.join(timeout=6)
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def sass_instruction_count(kernel_substr: str):
    """Static SASS instruction count of a kernel in the loaded libmrq.so (None if cuobjdump is unavailable)."""
    try:
        lib = os.path.join(ROOT, "raftsql_b200", "libmrq.so")
        txt = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, timeout=120).stdout
        for part in txt.split("Function : ")[1:]:
            name = part.split("\n", 1)[0].strip()
            if kernel_substr in name:
                import re

                return len(re.findall(r"/\*[0-9a-f]{4}\*/\s+[^;]*;", part))
    except Exception:
        pass
    return None


def ncu_field(kernel: str, field: str):
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[kernel][field]
    except Exception:
        return None


def ncu_traffic(kernel: str, mangled_substr: str | None = None):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu summary (bench.py never runs
    under a profiler itself).  The figure is REFUSED (None) when the summary was captured from a binary whose SASS
    instruction count for this kernel differs from the library loaded now: a capture of another kernel version is
    not a measurement of this one."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[kernel]
        if mangled_substr and t.get("sass_instructions") is not None:
            now = sass_instruction_count(mangled_substr)
            if now is not None and int(t["sass_instructions"]) != now:
                return None
        return int(t["dram_read_bytes"]) + int(t["dram_write_bytes"])
    except Exception:
        return None


def cpu_quota_cores():
    """CPUs' worth of time the container's cgroup allows (cpu.max), or None when unlimited / unknown: the host may show
    128 hardware threads and still give this process 16 CPUs of time, which is what bounds every host-side leg."""
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if quota == "max" else round(int(quota) / int(period), 2)
    except Exception:
        return None


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------
def cpu_reference_ticks(G: int, Rr: int, state: dict, inboxes: list, budget_s: float, warmup: int = 1,
                        steps: int | None = None, nthreads: int | None = None):
    """Time the CPU restatement of the reference path (oracle/, 'port') on all host threads (or `nthreads`)."""
    import oracle

    nt = nthreads or oracle.hw_threads()
    orc = oracle.Oracle(G, Rr, seed=SEED)
    orc.import_state(state)
    k = 0
    for _ in range(warmup):
        orc.tick(inboxes[k % len(inboxes)], nthreads=nt)
        k += 1
    t0 = time.perf_counter()
    n = 0
    while True:
        orc.tick(inboxes[k % len(inboxes)], nthreads=nt)
        k += 1
        n += 1
        el = time.perf_counter() - t0
        if (steps is not None and n >= steps) or (steps is None and (el >= budget_s or n >= 400)):
            break
    return n / el, nt, n, el, orc


def host_inboxes_from_oracle(G: int, Rr: int, state: dict, n: int, group_base: int = 0):
    """Generate the trace on the host (same generator as the device: include/mrq_trace.h)."""
    import oracle
    from raftsql_b200 import _ffi, preset_trace

    p = preset_trace(3)
    po = oracle.TraceParams()
    for name, _ in _ffi.TraceParams._fields_:
        setattr(po, name, getattr(p, name))
    nt = oracle.hw_threads()
    orc = oracle.Oracle(G, Rr, seed=SEED, group_base=group_base)
    orc.import_state(state)
    out = []
    for t in range(n):
        ib = orc.gen_trace(po, t, nthreads=nt)
        out.append(ib)
        orc.tick(ib, nthreads=nt)
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU path.  The Go reference cannot be built here (no Go toolchain;
    its raft arithmetic is an un-vendored dependency), so this is the oracle port, multi-threaded."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle

    G = G_TOTAL
    st = steady_state(G, R, 0, SEED)
    nslots = min(args.steps + args.warmup, 6)
    inboxes = host_inboxes_from_oracle(G, R, st, nslots)
    tps, nt, n, el, _ = cpu_reference_ticks(G, R, st, inboxes, 1e9, warmup=max(1, args.warmup), steps=args.steps)
    line = {
        "impl": "reference", "metric": "raft_ticks_per_sec_1Mx5", "value": tps, "unit": "ticks/s",
        "n_gpus": args.gpus, "steps": n, "warmup": max(1, args.warmup), "ms_per_step": 1e3 * el / n,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "1,048,576 groups x 5 replicas, steady-state append/ack trace (BASELINE configs[2]/[3])",
                   "groups_total": G, "replicas": R},
        "cpu_baseline": {"value": tps, "unit": "ticks/s", "cores": nt, "kind": "port", "cpu_quota_cores": cpu_quota_cores(),
                         "sample": f"{n} full ticks over all {G} groups on {nt} threads"},
        "e2e": {"value": tps, "unit": "ticks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "C restatement of etcd-raft v2.x per-message semantics (oracle/raft_oracle.c); the Go reference "
                "is not buildable in this environment",
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch

    from raftsql_b200 import Engine, _ffi, preset_trace
    from raftsql_b200.packed import Pack8

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist = None
        torch.cuda.set_device(local)
    dev = local
    assert G_TOTAL % world == 0
    weak = bool(getattr(args, "weak", False)) and world > 1  # --weak: every GPU keeps 1,048,576 groups (job = N x that)
    G = G_TOTAL if weak else G_TOTAL // world
    groups_job = G * world
    base = rank * G
    K, W = args.steps, max(3, args.warmup)
    nslots = min(K + W, MAX_SLOTS)
    reps = max(1, int(os.environ.get("MRQ_BENCH_REPS", "5")))
    inbox = args.inbox
    mode = {"compact": 4, "bytes": 3, "wide": 0}[inbox]
    fast = os.environ.get("MRQ_BENCH_FAST") == "1"  # profiling runs (ncu): kernels only, no CPU legs

    eng = Engine(G, R, seed=SEED, group_base=base, device=dev, inbox_slots=nslots + 1)  # + one slot for the post-roll's empty inbox
    if args.l2 is not None:
        eng.set_l2_policy(args.l2)
    st0 = steady_state(G, R, base, SEED)
    eng.import_state(st0)
    p = preset_trace(3)

    if world > 1 and args.gather != "none":  # the per-tick all-gather of committed[]: fused peer stores (default) or ncclAllGather
        from raftsql_b200 import multi

        multi.attach(eng, dist, args.gather)

    # dry run (tick mode 0): generate the trace tick by tick on the device (each tick's acks depend on that tick's
    # state), one inbox slot per tick; then rewind the state so the timed runs replay exactly these inputs.
    e2e_steps = min(K, nslots)
    commits_after = None
    for t in range(nslots):
        eng.gen_trace(p, t, slot=t)
        eng.tick(t)
        if t == e2e_steps - 1:
            commits_after = eng.sync_commits().copy()  # what the first e2e_steps ticks commit (checks the e2e leg)
    eng.synchronize()
    want_e2e = not fast
    host_ib = [eng.read_inbox(s) for s in range(e2e_steps if want_e2e else 0)]  # every rank runs the e2e leg on its own shard

    def rewind(tick_mode, graph, write_through=1):
        eng.set_tick_mode(0)
        eng.import_state(st0)
        eng.tick_count = 0
        eng.set_tick_mode(tick_mode)
        eng.set_graph_mode(graph)
        eng.set_write_through(write_through)
        if tick_mode >= 3:
            eng.set_packed_base(base0, st0["term"])
        if world > 1 and args.gather == "fused":
            eng.comm_set_mode(1)  # the rewind changed committed[] behind the peers' backs: republish the high words

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run_ticks(n, first_slot):
        # n ticks in one C call: mode 4 runs them in one launch pair; modes 0-3 replay a CUDA graph (small shards) or
        # issue the per-tick launches
        eng.tick_many([(first_slot + k) % nslots for k in range(n)])

    def post_roll(med_ms):
        """~2 s of tick launches on EMPTY inboxes after the timed repetitions, so that the clock sampler sees the GPU under
        the tick kernels (every rank runs the same number of chunks: the stop decision is rank 0's, all-reduced)."""
        if eng_mode() >= 3:
            zero = np.zeros((max(R - 1, 0), G), np.uint8)
            eng.post_inbox_packed(zero, np.zeros(G, np.uint8), (), slot=nslots, keep=True)
        else:
            eng.clear_inbox(nslots)
        t_start = time.perf_counter()
        while True:
            for _ in range(100):
                eng.tick_many([nslots] * 64)
            eng.synchronize()
            done = time.perf_counter() - t_start >= 2.0
            if dist is not None:
                flag_t = torch.tensor([1 if done else 0], dtype=torch.int32, device="cuda")
                dist.broadcast(flag_t, 0)
                done = bool(flag_t.item())
            if done:
                break

    cur_mode = [0]

    def eng_mode():
        return cur_mode[0]

    def last_step_outputs(tick_mode):
        """What a caller of the timed path reads after its last tick: every group's commit index, that tick's out words
        (and in tick mode 4 its commit advances), and the term / role / last index columns.  float64 holds the u64 indices
        exactly (they stay below 2^53); 40 B per group, 40 MB at 1,048,576 groups."""
        st = eng.export_state(("term", "role", "last_index"))
        got = {"committed": eng.sync_commits().astype(np.float64), "out": eng.sync_out().astype(np.float64),
               "term": st["term"].astype(np.float64), "role": st["role"].astype(np.float32),
               "last_index": st["last_index"].astype(np.float64)}
        if tick_mode == 4:
            got["commit_advance"] = eng.sync_tick_deltas().astype(np.float32)
        return got

    dumped = {}

    def timed_leg(tick_mode, graph, write_through=1, nreps=reps, sample_clocks=False, dump=False):
        """`nreps` repetitions of: rewind, W warm-up ticks, then EXACTLY K ticks between barrier + synchronize, CUDA
        events on the engine's stream, max over ranks.  Returns (median ms for K ticks, all reps, launches, clocks).
        With `dump`, the outputs of the last rep's last tick go to `dumped` (every rep replays the same inputs)."""
        out_ms, launches, clocks = [], 0, None
        cur_mode[0] = tick_mode
        rewind(tick_mode, graph, write_through)  # rehearsal (untimed): graphs captured, descriptor tables built
        run_ticks(W, 0)
        run_ticks(K, W)
        eng.synchronize()
        sampler = None
        if sample_clocks:
            sampler = ClockSampler(dev)
            sampler.start()
        for _ in range(nreps):
            rewind(tick_mode, graph, write_through)
            barrier()
            run_ticks(W, 0)
            eng.synchronize()
            c0 = eng.counters()
            barrier()
            eng.timer_start()
            run_ticks(K, W)
            ms = eng.timer_stop()
            barrier()
            launches = eng.counters()["kernel_launches"] - c0["kernel_launches"]
            if dist is not None:
                t = torch.tensor([ms], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            out_ms.append(ms)
        if dump:
            dumped.update(last_step_outputs(tick_mode))
        med = float(np.median(out_ms))
        if sampler is not None:
            # keep the GPU under the tick kernels ~2 s more so that the sampler sees it at the clocks of the timed region
            # (the region itself lasts a fraction of a millisecond).  Replaying the trace's slots without a rewind would
            # feed stale acks to a state that has moved on, so the post-roll ticks EMPTY inboxes (timers only) instead.
            post_roll(med)
            clocks = sampler.finish()
        if dist is not None:
            lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
            dist.all_reduce(lt)
            launches = int(lt.item())
        return med, out_ms, launches, clocks

    graph = {"off": 0, "on": 1, "auto": 2}[args.graph]
    wt = 0 if args.write_back == "end" else 1
    legs = {}

    def leg_record(name, tm, gr, w_):
        m_, r_, l_, _ = timed_leg(tm, gr, w_, nreps=3)
        ib_name = {4: "compact", 3: "bytes", 0: "wide"}[tm]
        tbl = tick_bytes_per_group(R, ib_name, K if (tm == 4 and gr != 0) else 1, bool(w_))
        gbs = tbl["total"] * G / (m_ / K * 1e-3) / 1e9
        peak_ = measured_peak_gbs()[0]
        legs[name] = {"ticks_per_s": K / (m_ / 1e3), "us_per_tick": m_ / K * 1e3, "launches": l_,
                      "bytes_per_group_tick": tbl["total"], "achieved_GBps": gbs, "frac": gbs / peak_,
                      "us_per_tick_reps": [round(x / K * 1e3, 2) for x in r_]}

    want_variants = rank == 0 and world == 1 and not fast and mode == 4
    if want_variants:
        # round 1's path — wide inbox, 64-bit state, a launch pair per tick — timed FIRST, on an L2 no later mode has
        # marked (its evict-last lines would otherwise squat there: measured 91 us instead of 37 us per tick)
        leg_record("wide_inbox_mode0", 0, graph, 1)
    # byte frames (include/mrq_packed8.h) of the same trace, one per slot, resident in HBM: tick modes 3 / 4 read the
    # bytes themselves (no wide inbox, no unpack pass)
    base0 = (st0["last_index"] - np.uint64(40)).astype(np.uint64)
    n_escapes = 0
    if mode >= 3:
        pk = Pack8(st0["self_id"], base0, st0["term"], R)
        eng.set_tick_mode(mode)
        for t in range(nslots):  # in tick order: the window only moves forward
            ib = host_ib[t] if t < len(host_ib) else eng.read_inbox(t)
            w8, p8, wide8 = pk.frame(ib)
            n_escapes += len(wide8)
            eng.post_inbox_packed(w8, p8, wide8, slot=t, keep=True)

    dump_dir = getattr(args, "dump_outputs", None) if rank == 0 else None  # N > 1: rank 0's shard
    ms, ms_reps, launches_timed, clocks = timed_leg(mode, graph, wt, sample_clocks=True, dump=bool(dump_dir))
    ticks_per_s = K / (ms / 1e3)
    peak, peak_src = measured_peak_gbs()
    batched = mode == 4 and graph != 0 and not (world > 1 and args.gather == "nccl")  # (a per-tick ncclAllGather forces per-tick launches)

    # ---- roofline of the dominant kernel ---------------------------------------------------------------
    tb = tick_bytes_per_group(R, inbox, K if batched else 1, bool(wt))
    tick_kernel_ms = ms / K  # back-to-back on one stream: event time / K is the per-tick share of the launch
    tick_gbs = tb["total"] * G / (tick_kernel_ms * 1e-3) / 1e9
    kernel_name = {4: "tick_fast4_kernel<5> (+ tick_slow4_kernel<5> over the groups that left the fast path)",
                   3: "tick_fast8_kernel<5> (+ tick_slow8_kernel<5>)",
                   0: "tick_fast_kernel<5> (+ tick_slow_kernel<5> over the slow list, empty on this trace)"}[mode]
    frames_mb = nslots * G * R / 1e6
    line = {
        "metric": "raft_ticks_per_sec_1Mx5", "value": ticks_per_s, "unit": "ticks/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak" if weak else "strong", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": "1,048,576 groups x 5 replicas, steady-state append/ack trace (BASELINE configs[2]/[3])",
                   "groups_total": groups_job, "groups_per_gpu": G, "replicas": R, "parallelism": f"groups sharded x{world}",
                   "collective": ("none" if world == 1 else
                                  "all-gather of committed[] per tick, fused into the tick kernel as peer stores over NVLink"
                                  if args.gather == "fused" else "ncclAllGather(committed) per tick" if args.gather == "nccl"
                                  else "none in the timed region (--gather none: shards tick independently; SURVEY 8d config 4)"),
                   "tick_mode": mode,
                   "inbox": ({4: f"byte frames resident in HBM, one per slot, {n_escapes} escaped messages; compact state (tick mode 4)",
                              3: f"byte frames resident in HBM, one per slot, {n_escapes} escaped messages; wide state (tick mode 3)",
                              0: "wide columns resident in HBM, one inbox slot per tick (tick mode 0)"}[mode]),
                   "launches": (f"one launch pair per {K} ticks (mrq_tick_many; state carried in registers, "
                                f"{'written through every tick' if wt else 'written back after the last tick'})" if batched
                                else "one launch pair per tick"),
                   "timing": f"median of {reps} repetitions of [rewind, {W} warm-up ticks, {K} timed ticks]",
                   "l2": ((f"inputs larger than L2: {nslots} rotating byte frames + per-slot out/advance buffers "
                           f"({frames_mb + nslots * G * 5 / 1e6:.0f} MB) vs 126 MB L2; ") if mode >= 3 else
                          (f"inputs larger than L2: {nslots} rotating inbox slots, per-step footprint "
                           f"{(tb['total'] * G) / 1e6:.0f} MB vs 126 MB L2; ")) +
                         "the engine state is re-used every tick by design and may stay L2-resident"},
        "ms_per_step_reps": [round(x / K, 6) for x in ms_reps],
        "group_ticks_per_sec": ticks_per_s * groups_job,
        "roofline": {"bound": "hbm", "kernel": kernel_name,
                     "achieved": tick_gbs, "peak": peak, "unit": "GB/s",
                     "frac": tick_gbs / peak,
                     "traffic": (None if world != 1 or mode != 4 else
                                 ncu_traffic("tick_fast4_kernel<5>", "tick_fast4_kernelILi5") if not batched else
                                 ncu_traffic("tick_fast4_kernel<5> (20 ticks per launch)", "tick_fast4_kernelILi5") if K == 20 else None),
                     "traffic_source": "profiles/r02_traffic.json (ncu --set full, cold cache, one isolated launch" +
                                       (f" of {K} ticks: stores still dirty in L2 at its end are not in it)" if batched else ")"),
                     "peak_source": peak_src, "algorithmic_bytes_per_group": tb,
                     "algorithmic_bytes_per_launch": tb["total"] * G * (K if batched else 1)},
        "gpu_launches": launches_timed,
        "clocks": clocks,
    }
    if world == 1 and mode == 4 and batched and K == 20 and line["roofline"]["traffic"]:
        # what the HBM fraction does not say: the launch is instruction-issue bound, and the L2 absorbs most of the write-through
        winst = ncu_field("tick_fast4_kernel<5> (20 ticks per launch)", "warp_instructions")
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        line["roofline"]["note"] = ("algorithmic bytes include the per-tick write-through of the state (40 B per group-tick); the 126 MB L2 "
                                    "absorbs most of it (DRAM traffic of the launch = `traffic`), and the kernel is bound by instruction issue")
        if winst:
            line["roofline"]["issue"] = {"warp_instructions_per_launch": winst, "schedulers": 148 * 4,
                                         "ipc_per_scheduler": winst / (148 * 4 * mhz * 1e6 * (ms * 1e-3)),
                                         "source": "profiles/r02_traffic.json (smsp__inst_executed.sum of the same launch shape) / measured time"}

    if rank == 0 and world == 1:
        # the other ways to run the same K ticks, each [rewind, W, K] x 3 (median): what the batching and the layout buy
        if want_variants:
            for name, (tm, gr, w_) in {"compact_per_tick_launches": (4, 0, 1), "compact_batched_write_through": (4, 2, 1),
                                        "compact_batched_write_back_at_end": (4, 2, 0), "bytes_on_wide_state_mode3": (3, 0, 1)}.items():
                leg_record(name, tm, gr, w_)
            rewind(mode, graph, wt)
        line["variants"] = legs
        line["roofline_quorum_kernel"] = bench_quorum_kernel(torch, eng, peak, K, W)
        with Engine(262144, 7, seed=0x5EED0005, device=dev) as e7:  # BASELINE configs[4]'s shape: R = 7, 72 B per group
            line["roofline_quorum_kernel_262144x7"] = bench_quorum_kernel(torch, e7, peak, K, W, G=262144, Rr=7)
    if rank == 0 and world == 1 and fast:
        line["e2e"] = None
    elif world == 1:
        line["e2e"] = bench_e2e(eng, st0, base0, host_ib, commits_after, e2e_steps)
        # CPU baseline: the oracle port on this box's host cores, bounded sample
        try:
            tps, nt, n, el, _ = cpu_reference_ticks(G_TOTAL, R, st0, host_ib[:4], budget_s=12.0)
            line["cpu_baseline"] = {"value": tps, "unit": "ticks/s", "cores": nt, "kind": "port", "cpu_quota_cores": cpu_quota_cores(),
                                    "sample": f"{n} full ticks over all {G_TOTAL} groups x {R} replicas in {el:.1f} s on {nt} threads"}
            tps1, _, n1, el1, _ = cpu_reference_ticks(G_TOTAL, R, st0, host_ib[:4], budget_s=3.0, nthreads=1)
            line["cpu_baseline"]["single_thread"] = {"value": tps1, "cores": 1, "sample": f"{n1} full ticks in {el1:.1f} s"}
        except Exception as ex:  # the baseline must never take the GPU numbers down with it
            line["cpu_baseline"] = {"value": None, "unit": "ticks/s", "cores": 0, "kind": "port", "sample": f"failed: {ex}"}
    if world > 1:
        if args.gather != "none":
            # correctness of the gather on every rank: it must equal the concatenation of all shards' commits
            mine = torch.from_numpy(eng.sync_commits().view(np.int64)).cuda()
            allc = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allc, mine)
            g = eng.sync_gathered().view(np.int64)
            ok = torch.tensor([int(np.array_equal(g, torch.cat(allc).cpu().numpy()))], device="cuda")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            line["gather_check"] = bool(ok.item())
        else:
            line["gather_check"] = None
        # end to end at N GPUs: every rank encodes and ships its shard's byte frames over its own PCIe link each tick
        e2e = None if fast else bench_e2e(eng, st0, base0, host_ib, commits_after, e2e_steps, dist=dist, torch=torch)
        if rank == 0:
            line["e2e"] = e2e
    eng.close()
    if dump_dir:
        os.makedirs(dump_dir, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(dump_dir, f"{name}.npy"), a)
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def bench_quorum_kernel(torch, eng, peak, K, W, G=None, Rr=None):
    """The standalone quorum kernel (K3) on never-touched column sets: achieved = (8R+16) * G / launch time.
    (G, Rr) default to the headline shape; bench.py also runs BASELINE configs[4]'s shape, 262,144 x 7, on an engine of 7 replicas.)"""
    G = G_TOTAL if G is None else G
    R = globals()["R"] if Rr is None else Rr  # noqa: N806 — shadows the module constant on purpose inside this function
    stride = G
    nsets = min(K + W, 40)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1234)
    sets = []
    for _ in range(nsets):
        li = torch.randint(2 ** 20, 2 ** 40, (G,), generator=gen, device="cuda", dtype=torch.int64)
        lag = torch.randint(0, 12, (R, G), generator=gen, device="cuda", dtype=torch.int64)
        match = (li.unsqueeze(0) - lag).contiguous()
        committed = (li - 40).contiguous()
        gate = (committed - 5).contiguous()
        sets.append((match, committed, gate))
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    out = {}
    for variant, name in ((0, "ldg256"), (1, "tma_bulk"), (2, "ldg128")):
        for m, c, g in sets[:W]:  # warm-up launches (these sets are not reused in the timed loop of this variant)
            eng.quorum_commit_ext(m.data_ptr(), c.data_ptr(), g.data_ptr(), G, stride, variant)
        eng.synchronize()
        timed = sets[W:] if len(sets) > W else sets
        reps = []
        for rep in range(3):  # three independent repetitions; the median is reported (not the best)
            # restore committed so that commits advance again, then flush L2 so every timed launch reads HBM
            for (m, c, g) in sets:
                c.copy_(g + 5)
            flush.fill_(rep + 1)
            torch.cuda.synchronize()
            eng.timer_start()
            for m, c, g in timed:
                eng.quorum_commit_ext(m.data_ptr(), c.data_ptr(), g.data_ptr(), G, stride, variant)
            reps.append(eng.timer_stop() / len(timed))
        per = sorted(reps)[1]
        gbs = quorum_bytes_per_group(R) * G / (per * 1e-3) / 1e9
        out[name] = {"us_per_launch": per * 1e3, "achieved": gbs, "frac": gbs / peak, "launches": len(timed),
                     "us_per_launch_reps": [round(x * 1e3, 2) for x in reps]}
    best = max(out, key=lambda k: out[k]["achieved"])
    return {"bound": "hbm", "kernel": f"quorum_kernel ({best})", "achieved": out[best]["achieved"], "peak": peak,
            "unit": "GB/s", "frac": out[best]["frac"],
            "traffic": (ncu_traffic(*{"ldg256": ("quorum_kernel_ldg256<5>", "quorum_kernel_ldg256ILi5"),
                                      "tma_bulk": ("quorum_kernel_tma<5>", "quorum_kernel_tmaILi5"),
                                      "ldg128": ("quorum_kernel_ldg<5>", "quorum_kernel_ldgILi5")}[best]) if (R == 5 and G == G_TOTAL) else None),
            "algorithmic_bytes_per_group": quorum_bytes_per_group(R), "variants": out,
            "cold": f"{len(sets)} distinct column sets ({quorum_bytes_per_group(R) * G / 1e6:.1f} MB each), L2 flushed before timing"}


def bench_e2e(eng, st0, base0, host_ib, commits_ref, steps, dist=None, torch=None):
    """The same ticks through the C-ABI with HOST buffers, everything on the clock: per step the host ENCODES that tick's
    inbox into a byte frame (mrq_pack8, on the library's host thread pool — frame k+1 is built while tick k runs), the
    frame goes H2D from pinned memory (copy stream), mrq_tick (tick mode 4), and the tick's commit advances come back
    D2H (1 B per group) and are waited for before the step counts.  Every step ships a DIFFERENT tick of the trace.
    With `dist`, every rank runs its shard and the elapsed time is the max over ranks (barrier on both sides).
    The result is accepted only if the commit indices rebuilt from the drained advances equal `commits_ref` — what the
    same ticks commit from the device-generated wide inbox in tick mode 0."""
    import ctypes as C
    import queue

    from raftsql_b200 import _ffi as F
    from raftsql_b200.packed import Pack8, PinnedArray

    G, Rr = eng.G, eng.R
    S = min(steps, len(host_ib))
    L, h = eng.L, eng.h
    NB = 4  # pinned frame buffers in flight: built / copying / ticking / draining

    def sync_all():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def rewind(tick_mode):
        eng.set_tick_mode(0)
        eng.import_state(st0)
        eng.tick_count = 0
        eng.set_tick_mode(tick_mode)
        if tick_mode >= 3:
            eng.set_packed_base(base0, st0["term"])
        return eng.sync_commits().copy()

    # -- wide form (33 B per slot, pageable numpy arrays): the straightforward host path, for scale -------------
    rewind(0)
    sync_all()
    nw = min(4, S)
    t0 = time.perf_counter()
    for k in range(nw):
        eng.post_inbox_dense(host_ib[k], slot=k % 2)
        eng.tick(k % 2)
        eng.sync_commits()
    el_w = max_over_ranks(time.perf_counter() - t0)
    wide = {"value": nw / el_w, "h2d_bytes_per_step": sum(a.nbytes for a in host_ib[0].values()),
            "d2h_bytes_per_step": G * 8, "api": "mrq_post_inbox_dense + mrq_tick + mrq_sync_commits"}

    class Frame:  # one pinned buffer per frame: R-1 sender rows, then the proposal bytes (a single H2D copy)
        def __init__(self):
            self.buf = PinnedArray((max(Rr - 1, 0) + 1, G), np.uint8)
            self.word, self.prop = self.buf.array[: max(Rr - 1, 0)], self.buf.array[max(Rr - 1, 0)]
            self.word_ptr, self.prop_ptr = self.buf.ptr, self.buf.ptr + max(Rr - 1, 0) * G

        def free(self):
            self.buf.free()

    bufs = [Frame() for _ in range(NB)]
    delta = PinnedArray((G,), np.uint8)
    dptr = C.cast(delta.ptr, F.u8p)

    def view_of(b, wide_msgs):
        arr = (F.Msg * max(1, len(wide_msgs)))()
        for i, (g, frm, ty, term, index, logterm, commit) in enumerate(wide_msgs):
            arr[i].group, arr[i].from_, arr[i].type = g, frm, ty
            arr[i].term, arr[i].index, arr[i].logterm, arr[i].commit = term, index, logterm, commit
        v = F.InboxPacked()
        v.word, v.prop_count8 = bufs[b].word_ptr, C.cast(bufs[b].prop_ptr, F.u8p)
        v.wide, v.n_wide, v.word_bits, v.reserved = arr, len(wide_msgs), 8, 0
        return v, arr

    def run(nsteps, accumulate, encode_on_clock=True, frames=None):
        base = rewind(4)
        acc = np.zeros(G, np.uint64)
        pk = Pack8(st0["self_id"], base0, st0["term"], Rr)
        ready: queue.Queue = queue.Queue()
        free = threading.Semaphore(NB)
        pack_s = [0.0]
        n_esc = [0]

        def packer():  # the host's frame builder: one frame per tick, in posting order (the window only moves forward)
            for k in range(nsteps):
                free.acquire()
                b = k % NB
                t1 = time.perf_counter()
                _, _, wide_msgs = pk.frame(host_ib[k % S], word_out=bufs[b].word, prop8_out=bufs[b].prop)
                pack_s[0] += time.perf_counter() - t1
                n_esc[0] += len(wide_msgs)
                ready.put(view_of(b, wide_msgs))

        sync_all()
        t0 = time.perf_counter()
        th = threading.Thread(target=packer, daemon=True)
        th.start()
        cur = ready.get()
        rc = L.mrq_post_inbox_packed(h, 0, C.byref(cur[0]))
        for k in range(nsteps):
            rc |= L.mrq_tick(h, k % 2)
            rc |= L.mrq_drain_tick_deltas(h, dptr)
            nxt = None
            if k + 1 < nsteps:  # the next tick's frame: encoded underneath this tick, copied underneath it too
                nxt = ready.get()
                rc |= L.mrq_post_inbox_packed(h, (k + 1) % 2, C.byref(nxt[0]))
            rc |= L.mrq_drain_wait(h)  # this step's result is on the host
            if rc != 0:
                raise RuntimeError("C-ABI call failed: " + (L.mrq_last_error(h) or b"?").decode())
            free.release()  # tick k is done, so frame k's copy is too: its pinned buffer may be rebuilt
            if accumulate:
                assert delta.array.max() < 255
                acc += delta.array
            cur = nxt
        el = max_over_ranks(time.perf_counter() - t0)
        th.join()
        eng.synchronize()
        return el, base + acc, pack_s[0] / nsteps, n_esc[0]

    run(3, False)
    _, commits, _, _ = run(S, True)
    same = bool(np.array_equal(commits, commits_ref)) and bool(np.array_equal(commits, eng.sync_commits()))
    el, _, pack_avg, n_esc = run(S, False)
    ws = 1 if dist is None else dist.get_world_size()  # bytes are whole-job figures (all ranks)
    h2d = (max(Rr - 1, 0) + 1) * G
    res = {"value": S / el, "unit": "ticks/s", "h2d_bytes_per_step": h2d * ws, "d2h_bytes_per_step": G * ws, "steps": S,
           "api": "mrq_pack8 (host encode, in the timed region) + mrq_post_inbox_packed (pinned, 8-bit form, copy stream) + "
                  "mrq_tick (tick mode 4) + mrq_drain_tick_deltas/mrq_drain_wait (1 B/group)",
           "encode_in_timed_region": True, "pack_us_per_tick": pack_avg * 1e6, "us_per_tick": el / S * 1e6,
           "host_cpu_quota_cores": cpu_quota_cores(),
           "equals_wide_form": same, "escapes": n_esc, "h2d_GBps_per_gpu": h2d * S / el / 1e9,
           "inputs": f"{S} distinct consecutive ticks of the trace, one per step (host wide inbox -> byte frame -> device)",
           "wide_form": wide}
    # the same loop with the frames already encoded (a transport that delivers byte frames): what the link + device do alone
    pre = [Frame() for _ in range(S)]
    pk = Pack8(st0["self_id"], base0, st0["term"], Rr)
    views = []
    for k in range(S):
        _, _, wm = pk.frame(host_ib[k], word_out=pre[k].word, prop8_out=pre[k].prop)
        v = F.InboxPacked()
        v.word, v.prop_count8 = pre[k].word_ptr, C.cast(pre[k].prop_ptr, F.u8p)
        arr = (F.Msg * max(1, len(wm)))()
        for i, (g, frm, ty, term, index, logterm, commit) in enumerate(wm):
            arr[i].group, arr[i].from_, arr[i].type = g, frm, ty
            arr[i].term, arr[i].index, arr[i].logterm, arr[i].commit = term, index, logterm, commit
        v.wide, v.n_wide, v.word_bits, v.reserved = arr, len(wm), 8, 0
        views.append((v, arr))

    def run_pre(nsteps):
        rewind(4)
        sync_all()
        t0 = time.perf_counter()
        rc = L.mrq_post_inbox_packed(h, 0, C.byref(views[0][0]))
        for k in range(nsteps):
            rc |= L.mrq_tick(h, k % 2)
            rc |= L.mrq_drain_tick_deltas(h, dptr)
            if k + 1 < nsteps:
                rc |= L.mrq_post_inbox_packed(h, (k + 1) % 2, C.byref(views[k + 1][0]))
            rc |= L.mrq_drain_wait(h)
            assert rc == 0
        el_ = max_over_ranks(time.perf_counter() - t0)
        eng.synchronize()
        return el_

    run_pre(3)
    el_p = run_pre(S)
    res["preencoded"] = {"value": S / el_p, "us_per_tick": el_p / S * 1e6, "h2d_GBps_per_gpu": h2d * S / el_p / 1e9,
                         "encode_in_timed_region": False,
                         "note": "frames encoded before the clock starts (a transport delivering byte frames): link + device only"}
    for fr in bufs + pre:
        fr.free()
    delta.free()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gather", default="fused", choices=["fused", "nccl", "none"],
                    help="N>1: how committed[] is all-gathered each tick (none: not at all — the scaling leg "
                         "without the collective in the timed region)")
    ap.add_argument("--write-back", default="every-tick", choices=["every-tick", "end"],
                    help="tick mode 4, one launch per K ticks: state columns written after every tick (default) or the last")
    ap.add_argument("--l2", type=int, default=None, choices=[0, 1],
                    help="L2 residency hints of the tick kernel (default: the engine's, on)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="how mrq_tick_many runs K ticks: auto/on = tick mode 4 in ONE launch pair, modes 0-3 as a CUDA graph "
                         "(auto: small shards only); off = per-tick launches in every mode")
    ap.add_argument("--inbox", default="compact", choices=["compact", "bytes", "wide"],
                    help="the timed ticks: compact = byte frames on compact state (tick mode 4, default); bytes = byte frames on "
                         "wide state (tick mode 3); wide = wide inbox columns (tick mode 0, round 1's path)")
    ap.add_argument("--weak", action="store_true",
                    help="N>1: weak scaling — every GPU keeps 1,048,576 groups, the job is N times that (default: the job "
                         "stays 1,048,576 groups, BASELINE configs[3]); compare group_ticks_per_sec across N")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl ours: after the timed ticks, write what the last one computed as DIR/<name>.npy (float32 / "
                         "float64): commit indices, out words, commit advances, term, role, last index; the inputs are "
                         "seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
