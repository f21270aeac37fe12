#!/usr/bin/env python
"""bench.py -- rendered messages/s of the NUTS message path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of synthetic input per rank:
BASELINE config 3 (1M say() messages x 10k users in 100 rooms of 100, 64-word swear
list, ban_swearing on: contains_swearing -> gated write_user / write_room_except ->
colour render + fan-out) plus config 4's ban verdicts (100k sites + 100k names vs
10k-entry lists).  Ranks own disjoint rooms (weak scaling, no data-path collective).

value = deliveries/s ("rendered messages/s") with inputs resident in HBM, timed with
CUDA events on the stream the kernels run on, max over ranks.  e2e = the same through
the host-buffer C-ABI (nutsb_*_batch with pinned host inputs, per-user streams copied
back to pinned host memory).  roofline = the render+fan-out kernel's algorithmic bytes
over its own CUDA-event time vs the measured HBM copy bandwidth.  cpu_baseline = the
reference's own C routines (oracle/_ref, built from nuts333.c) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

METRIC = "rendered messages/sec (colour+swear+ban)"
UNIT = "deliveries/s"

# per-rank shard of the workload
N_MSGS = 1_000_000
N_USERS = 10_000
USERS_PER_ROOM = 100
N_SWEAR = 64
KERNEL_TIMING_STEPS = 3
IN_FLIGHT = 1
N_BAN_QUERIES = 100_000
N_BAN_ENTRIES = 10_000
SEED = 0x333


def workload_name():
    return ("C3+C4 per rank: %d say() msgs x %d users (%d rooms of %d), %d-word swear list, ban_swearing; "
            "%d sites + %d names vs %d-entry ban lists" % (N_MSGS, N_USERS, N_USERS // USERS_PER_ROOM, USERS_PER_ROOM,
                                                           N_SWEAR, N_BAN_QUERIES, N_BAN_QUERIES, N_BAN_ENTRIES))


def make_inputs(rank: int, n_msgs: int):
    """The rank's shard (its own rooms, users and messages: nuts333_b200/shard.py), generated
    on the host once; the same generator feeds every leg."""
    from nuts333_b200 import shard, synth
    seed = SEED + 0x1000 * rank
    words = synth.swear_words(N_SWEAR)
    sh = shard.shard_inputs(rank, n_msgs, N_USERS, USERS_PER_ROOM, words, gated=True)
    st, so = synth.sites(N_BAN_QUERIES, seed=seed)
    nt, no = synth.names(N_BAN_QUERIES)
    sfile = synth.ban_file(0, N_BAN_ENTRIES, N_BAN_QUERIES, N_BAN_QUERIES, True, seed=seed)
    ufile = synth.ban_file(1, N_BAN_ENTRIES, N_BAN_QUERIES, N_BAN_QUERIES, True, seed=seed)
    return dict(words=words, users=sh["users"], n_rooms=sh["n_rooms"], bodies=sh["bodies"], ops=sh["ops"],
                speaker=sh["speaker"], sites=(st, so), names=(nt, no), sfile=sfile, ufile=ufile)


DUMP_SEED = 0x333D
DUMP_STREAM_CAP = 1 << 20           # bytes of a user's stream the sample looks at
DUMP_HEAD_USERS = 8
DUMP_POINTS = 2 << 20


def dump_outputs(out_dir: str, lane: dict, dev) -> None:
    """--dump-outputs: what one lane's last step handed its caller, as .npy files of float32 (bytes, 0/1 verdicts)
    or float64 (offsets, counts), about 47 MB in all, so that two builds can be compared output for output.  The
    three verdict arrays and the per-user stream offsets are written whole.  Of the ~5 GB of stream bytes, a sample
    fixed by DUMP_SEED and the user count alone, so that it lines up element for element across builds whatever
    stream lengths they produce: the first 1 MiB of the streams of 8 users (stream_heads, one row per user of
    stream_head_users), and the bytes at 2M (user, offset < 1 MiB) pairs (stream_points).  -1 marks an offset at or
    past the end of the user's stream."""
    import torch

    class DevBuf:                       # a buffer the library owns in HBM, seen by torch without a copy
        def __init__(self, ptr, n, typestr):
            self.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(int(ptr), False), version=2)

    s = lane["streams"]
    n_users, total = int(s.n_users), int(s.total_bytes)
    off = torch.as_tensor(DevBuf(s.off, n_users + 1, "<i8"), device=dev).cpu().numpy()
    data = torch.as_tensor(DevBuf(s.bytes, total, "|u1"), device=dev) if total else torch.zeros(0, dtype=torch.uint8, device=dev)
    lens = np.diff(off)
    rng = np.random.default_rng(DUMP_SEED)
    head_users = np.sort(rng.choice(n_users, min(DUMP_HEAD_USERS, n_users), replace=False))
    heads = np.full((len(head_users), DUMP_STREAM_CAP), -1, np.float32)
    for row, u in enumerate(head_users):
        n = int(min(lens[u], DUMP_STREAM_CAP))
        heads[row, :n] = data[int(off[u]):int(off[u]) + n].cpu().numpy()
    pu = rng.integers(0, n_users, DUMP_POINTS)
    pj = rng.integers(0, DUMP_STREAM_CAP, DUMP_POINTS)
    inside = pj < lens[pu]
    points = np.full(DUMP_POINTS, -1, np.float32)
    points[inside] = data[torch.from_numpy(off[pu[inside]] + pj[inside]).to(dev)].cpu().numpy()
    out = dict(contains_swearing=lane["verdict"].cpu().numpy().astype(np.float32),
               site_banned=lane["vs"].cpu().numpy().astype(np.float32),
               user_banned=lane["vu"].cpu().numpy().astype(np.float32),
               stream_off=off.astype(np.float64),
               n_deliveries=np.array([int(s.n_deliveries)], np.float64),
               stream_head_users=head_users.astype(np.float64),
               stream_heads=heads,
               stream_points=points)
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(d / f"{name}.npy", a)


# ---------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.samples, self.proc, self.th = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        """Keep the samples taken inside [t0, t1] (the timed region); if the region was
        shorter than the sampling period, keep the nearest ones taken under the same load."""
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        if not inside:
            inside = sorted(self.samples, key=lambda s: min(abs(s[0] - t0), abs(s[0] - t1)))[:5]
        self.samples = inside

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for _, s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, val in zip(names, f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own C routines on host cores
# ---------------------------------------------------------------------------------------
def _ref_worker(args):
    """One process = one single-threaded reference instance (its state is global) on one
    room-shard of the sample.  Returns (deliveries, bytes, seconds, kind)."""
    rank, shard, n_shards, n_msgs, n_ban = args[:5]
    both_sinks = len(args) > 5 and args[5]
    if len(args) > 6 and args[6] is not None:             # the one-core leg: pinned (BASELINE.md section 3: taskset)
        try:
            os.sched_setaffinity(0, {args[6]})
        except OSError:
            pass
    import tempfile
    import oracle_lib as O
    inp = make_inputs(rank, n_msgs)
    words, users, ops = inp["words"], inp["users"], inp["ops"]
    R = O.ref()
    if R is not None:
        R._tmp = tempfile.mkdtemp(prefix="nutsref_cwd_")     # per process: the reference reads ./datafiles/
    kind = "reference" if R is not None else "port"
    P = O.port()
    bt, bo = inp["bodies"]
    # this worker's share: messages whose room % n_shards == shard
    room_of_op = ops["target"].copy()
    k1 = ops["kind"] == 1
    msg_room = room_of_op[k1]
    mine_msg = (msg_room % n_shards) == shard
    mine_op = np.repeat(mine_msg, 3)
    sel = np.nonzero(mine_op)[0]
    lens = np.diff(ops["off"].astype(np.int64))
    sub_texts = [ops["text"][int(ops["off"][i]):int(ops["off"][i + 1])].tobytes() for i in sel]
    text, off = O.pack(sub_texts)
    msg_idx = np.nonzero(mine_msg)[0]
    remap = -np.ones(len(mine_msg), np.int64)
    remap[msg_idx] = np.arange(len(msg_idx))
    sub = dict(text=text, off=off, kind=ops["kind"][sel], target=ops["target"][sel], except_user=ops["except_user"][sel],
               flags=ops["flags"][sel], gate=remap[ops["gate"][sel]].astype(np.int32))
    bsel = [bt[int(bo[i]):int(bo[i + 1])].tobytes() for i in msg_idx]
    b2, bo2 = O.pack(bsel)
    st, so = inp["sites"]
    nt, no = inp["names"]
    qs = [st[int(so[i]):int(so[i + 1])].tobytes() for i in range(shard, n_ban, n_shards)]
    qn = [nt[int(no[i]):int(no[i + 1])].tobytes() for i in range(shard, n_ban, n_shards)]
    qst, qso = O.pack(qs)
    qnt, qno = O.pack(qn)
    comp = dict(n_msgs=len(msg_idx), n_ban=len(qs) + len(qn))
    t0 = time.perf_counter()
    if R is not None:
        R.set_swear_words(words[:-1])
        R.set_ban_file(0, inp["sfile"]); R.set_ban_file(1, inp["ufile"])
        ta = time.perf_counter()
        v = R.contains_swearing_batch(b2, bo2)
        tb = time.perf_counter()
        R.ban_batch(0, qst, qso); R.ban_batch(1, qnt, qno)
        tc = time.perf_counter()
        R.write_batch(sub, inp["n_rooms"], users, verdict=v, sink_mode=1)
        td = time.perf_counter()
        deliveries = None
        nbytes = int(R.lib.ref_total_write_bytes())
        dt = td - t0
        comp.update(swear_s=tb - ta, bans_s=tc - tb, write_s=td - tc)
        deliveries, _ = P.write_batch_count(sub, users, verdict=v)      # counted outside the timed region
        if both_sinks:                                                  # the faithful sink: write(2) to /dev/null (c:1318 ...)
            te = time.perf_counter()
            R.write_batch(sub, inp["n_rooms"], users, verdict=v, sink_mode=2)
            comp.update(write_devnull_s=time.perf_counter() - te, write_calls=int(R.lib.ref_total_write_calls()))
    else:
        ta = time.perf_counter()
        v = P.contains_swearing_batch(b2, bo2, words)
        tb = time.perf_counter()
        P.ban_batch(0, inp["sfile"], qst, qso); P.ban_batch(1, inp["ufile"], qnt, qno)
        tc = time.perf_counter()
        deliveries, nbytes = P.write_batch_count(sub, users, verdict=v)
        td = time.perf_counter()
        dt = td - t0
        comp.update(swear_s=tb - ta, bans_s=tc - tb, write_s=td - tc)
    comp["deliveries"] = int(deliveries)
    return deliveries, nbytes, dt, kind, comp


def reference_step(rank: int, n_msgs: int, n_ban: int, procs: int, both_sinks: bool = False, components: dict | None = None):
    """Runs the reference's CPU path over a bounded sample with `procs` host processes (one process: pinned to one
    core, in a child so that the caller's affinity is left alone).  components: filled with the slowest worker's
    time per component (swear, bans, render + fan-out) and the sample's sizes."""
    import multiprocessing as mp
    import oracle_lib as O
    O.port(); O.ref()                       # build / load the checkers once, before forking
    pin = None
    if procs == 1:
        try:
            pin = sorted(os.sched_getaffinity(0))[-1]
        except (AttributeError, OSError):
            pin = None
    args = [(rank, s, procs, n_msgs, n_ban, both_sinks, pin) for s in range(procs)]
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_ref_worker, args)
    wall = time.perf_counter() - t0
    d = sum(r[0] for r in res)
    busy = max(r[2] for r in res)
    if components is not None:
        for k in ("swear_s", "bans_s", "write_s", "write_devnull_s"):
            vals = [r[4][k] for r in res if k in r[4]]
            if vals:
                components[k] = max(vals)
        for k in ("n_msgs", "n_ban", "deliveries", "write_calls"):
            vals = [r[4][k] for r in res if k in r[4]]
            if vals:
                components[k] = sum(vals)
        components["pinned_core"] = pin
    return d, sum(r[1] for r in res), busy, wall, res[0][3]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    procs = max(1, os.cpu_count() or 1)
    procs = min(procs, 64)
    n_msgs = min(20_000 * max(1, procs // 4), N_MSGS)
    n_ban = max(procs, n_msgs * N_BAN_QUERIES // N_MSGS)        # the sample keeps the step's msgs : ban-queries ratio
    times, deliv = [], 0
    comp = {}
    for i in range(args.warmup + args.steps):
        d, nbytes, busy, wall, kind = reference_step(0, n_msgs, n_ban, procs, components=comp)
        if i >= args.warmup:
            times.append(busy); deliv += d
    total = sum(times)
    value = deliv / total
    sample = ("%d of %d msgs (all %d users, same generator) + %d of %d ban queries per list, per step; "
              "%d single-threaded reference processes sharded by room; write(2) hooked to a byte counter"
              % (n_msgs, N_MSGS, N_USERS, n_ban, N_BAN_QUERIES, procs))
    line = dict(impl="reference", metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * total / max(1, args.steps), higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="u8", data="synthetic",
                config=dict(workload=workload_name(), note="reference CPU path on a bounded sample of the workload: the rate "
                            "of a proportional %.0f %% sample (msgs and ban queries in the step's ratio), not a full step" % (100.0 * n_msgs / N_MSGS),
                            components=dict(comp, note="slowest worker's seconds per component in the last step (the ban checks re-open "
                                            "and re-parse the 10k-entry file per query, nuts333.c:330-364: about half of the time)")),
                cpu_baseline=dict(value=value, unit=UNIT, cores=procs, kind=kind, sample=sample),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from nuts333_b200 import api, build

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    build.build()
    dev = torch.device("cuda", local)

    inp = make_inputs(rank, N_MSGS)
    ops, users = inp["ops"], inp["users"]
    ctx = api.Context(local)
    stream = torch.cuda.Stream(device=dev, priority=-1)         # (the library's side stream is created at the lowest priority)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_profiling(True)
    ctx.set_swear_words(inp["words"])
    ctx.set_ban_files(inp["sfile"], inp["ufile"])
    ctx.set_users(users["room"], users["flags"], users["level"], inp["n_rooms"])

    def to_dev(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    def pad16(a):                      # packed text buffers are read in 16-byte vectors
        return np.concatenate([a, np.zeros(32, np.uint8)])

    bt, bo = inp["bodies"]
    st_, so_ = inp["sites"]
    nt_, no_ = inp["names"]
    d = dict(bt=to_dev(pad16(bt)), bo=to_dev(bo.view(np.int64)), text=to_dev(pad16(ops["text"])),
             off=to_dev(ops["off"].view(np.int64)), kind=to_dev(ops["kind"]), target=to_dev(ops["target"]),
             exc=to_dev(ops["except_user"]), flags=to_dev(ops["flags"]), gate=to_dev(ops["gate"]),
             st=to_dev(pad16(st_)), so=to_dev(so_.view(np.int64)), nt=to_dev(pad16(nt_)), no=to_dev(no_.view(np.int64)),
             verdict=torch.zeros(N_MSGS, dtype=torch.uint8, device=dev),
             vs=torch.zeros(N_BAN_QUERIES, dtype=torch.uint8, device=dev),
             vu=torch.zeros(N_BAN_QUERIES, dtype=torch.uint8, device=dev))
    n_ops = len(ops["kind"])
    input_bytes = sum(int(v.numel() * v.element_size()) for k, v in d.items() if k not in ("verdict", "vs", "vu"))
    torch.cuda.synchronize()

    state = dict(deliv=0, bytes=0, launches=0, fan_ms=0.0, fan_in=0, fan_out=0, plan_ms=0.0, direct_ms=0.0, render_ms=0.0, ksteps=0)
    state_lock = threading.Lock()

    # Batches in flight on this GPU: every lane is a context of its own (own stream, own scratch and stream
    # buffers) fed by its own host thread; the inputs in HBM are shared, the verdict outputs are per lane.
    # With two lanes one batch's planning / rendering (issue-bound) runs beside the other's fan-out (HBM-bound).
    lanes = [dict(ctx=ctx, stream=stream, verdict=d["verdict"], vs=d["vs"], vu=d["vu"])]

    def add_lane():
        c2 = api.Context(local)
        s2 = torch.cuda.Stream(device=dev, priority=-1)
        c2.set_stream(s2.cuda_stream); c2.set_profiling(True)
        c2.set_swear_words(inp["words"]); c2.set_ban_files(inp["sfile"], inp["ufile"])
        c2.set_users(users["room"], users["flags"], users["level"], inp["n_rooms"])
        lanes.append(dict(ctx=c2, stream=s2, verdict=torch.zeros_like(d["verdict"]), vs=torch.zeros_like(d["vs"]),
                          vu=torch.zeros_like(d["vu"])))

    for _ in range(1, max(1, args.in_flight)):
        add_lane()

    def step_device(L=None):
        L = L or lanes[0]
        c = L["ctx"]
        c.verdicts_dev("contains_swearing", N_MSGS, d["bt"].data_ptr(), d["bo"].data_ptr(), L["verdict"].data_ptr())
        c.verdicts_dev("site_banned", N_BAN_QUERIES, d["st"].data_ptr(), d["so"].data_ptr(), L["vs"].data_ptr())
        c.verdicts_dev("user_banned", N_BAN_QUERIES, d["nt"].data_ptr(), d["no"].data_ptr(), L["vu"].data_ptr())
        s = c.write_batch_dev(n_ops, d["text"].data_ptr(), d["off"].data_ptr(), d["kind"].data_ptr(),
                              d["target"].data_ptr(), d["exc"].data_ptr(), d["flags"].data_ptr(),
                              d["gate"].data_ptr(), L["verdict"].data_ptr())
        L["streams"] = s
        t = c.timing()
        with state_lock:
            state["deliv"] += int(s.n_deliveries); state["bytes"] += int(s.total_bytes)
            state["launches"] += int(t.launches) + 3
            state["fan_ms"] += float(t.fanout_ms); state["fan_in"] += int(t.fanout_bytes_in); state["fan_out"] += int(t.fanout_bytes_out)
            state["plan_ms"] += float(t.plan_ms); state["direct_ms"] += float(t.direct_ms); state["render_ms"] += float(t.render_ms)
            state["ksteps"] += 1
        return s

    def run_steps(k):
        """exactly k steps, dealt to the lanes"""
        if len(lanes) == 1:
            for _ in range(k):
                step_device()
            return
        share = [k // len(lanes) + (1 if i < k % len(lanes) else 0) for i in range(len(lanes))]
        th = [threading.Thread(target=lambda L=L, m=m: [step_device(L) for _ in range(m)]) for L, m in zip(lanes, share)]
        for t in th:
            t.start()
        for t in th:
            t.join()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local)
    if os.environ.get("BENCH_CLOCKS", "rank0") == "all" or rank == 0:    # rank 0 prints the line; nvidia-smi loops on every
        clocks.start()                      # nvidia-smi needs ~0.1 s to start: launched before the warm-up
    run_steps(args.warmup * len(lanes))
    for k in state:
        state[k] = 0 if not isinstance(state[k], float) else 0.0
    barrier()
    marker = torch.cuda.Stream(device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record(marker)                   # the device is idle here (barrier above): the lanes' first kernels come after
    run_steps(args.steps)
    for L in lanes:
        marker.wait_stream(L["stream"])
    e1.record(marker)
    barrier()
    tw1 = time.perf_counter()
    clocks.window(tw0, tw1)
    clk = clocks.stop()
    ms = e0.elapsed_time(e1)
    dev_state = dict(state)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, lanes[0], dev)
    # ---- per-kernel durations: the same step with every kernel on one stream (no k_render / k_direct beside
    #      the plan / the fan-out), so that each kernel is timed alone with CUDA events on its own stream
    ctx.set_overlap(False)
    step_device()                       # warm-up of the serial schedule
    for k in state:
        state[k] = 0 if not isinstance(state[k], float) else 0.0
    for _ in range(KERNEL_TIMING_STEPS):
        step_device()
    torch.cuda.synchronize()
    kstate = dict(state)
    # the three verdict kernels by themselves (CUDA events on the stream they run on)
    comp_ms = {}
    L0 = lanes[0]
    for nme, n_q, a, b, out in (("swear", N_MSGS, d["bt"], d["bo"], L0["verdict"]), ("site", N_BAN_QUERIES, d["st"], d["so"], L0["vs"]),
                                ("user", N_BAN_QUERIES, d["nt"], d["no"], L0["vu"])):
        fn = {"swear": "contains_swearing", "site": "site_banned", "user": "user_banned"}[nme]
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KERNEL_TIMING_STEPS)]
        for a0, a1 in evs:
            a0.record(stream)
            ctx.verdicts_dev(fn, n_q, a.data_ptr(), b.data_ptr(), out.data_ptr())
            a1.record(stream)
        torch.cuda.synchronize()
        comp_ms[nme] = min(a0.elapsed_time(a1) for a0, a1 in evs)
    ctx.set_overlap(os.environ.get('NUTSB_OVERLAP', '1') != '0')

    # ---- beside the headline (one batch at a time): the same K steps with two batches in flight on the GPU
    #      (a second context and host thread), one batch's planning under the other's fan-out
    two_ms = 0.0
    if len(lanes) == 1 and not args.no_e2e:
        add_lane()
        run_steps(2 * args.warmup)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(marker)
        run_steps(args.steps)
        for L in lanes:
            marker.wait_stream(L["stream"])
        f1.record(marker)
        barrier()
        two_ms = f0.elapsed_time(f1)
        lanes.pop().get("ctx").close()

    # ---- e2e: host buffers through the C-ABI, H2D and D2H inside the timed region.  The step's inputs sit in
    #      pinned host memory (the library copies straight from the caller's buffers); the result lands in the
    #      library's own pinned buffers.
    pinned = []

    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        pinned.append(t)
        return t.numpy()

    bt, bo, st_, so_, nt_, no_ = (pin(a) for a in (bt, bo, st_, so_, nt_, no_))
    hops = {k: (pin(v) if isinstance(v, np.ndarray) else v) for k, v in ops.items()}
    # the speech tier takes the input lines themselves (verb, speaker, body): say() composed on the device
    from nuts333_b200 import synth
    un, uo = synth.names(N_USERS)
    ctx.set_user_names([un[int(uo[u]):int(uo[u + 1])].tobytes() for u in range(N_USERS)], np.zeros(N_USERS, np.uint8))
    ctx.set_ban_swearing(True)
    sp_verb, sp_spk = pin(np.zeros(N_MSGS, np.uint8)), pin(inp["speaker"].astype(np.int32))

    def e2e_leg(mode):
        """One leg through the host-buffer entry points: verdict batches, then nutsb_write_batch (mode "streams":
        streams in pinned host memory), nutsb_write_batch_iov ("iov": gather lists into the pool of renderings) or
        nutsb_speech_batch_iov ("speech_iov": the 1M input lines of say() in -- swear verdicts, composition and
        rendering on the device -- gather lists out)."""
        iov = mode != "streams"
        r = dict(h2d_ms=0.0, d2h_ms=0.0, ms=0.0, deliv=0, h2d=0, d2h=0, extra={})
        for i in range(1 + e2e_steps):                     # first pass allocates the pinned result buffers
            barrier()
            t0 = time.perf_counter()
            vs = ctx.site_banned_batch(st_, so_)
            vu = ctx.user_banned_batch(nt_, no_)
            keep = []
            if mode == "speech_iov":
                v = np.zeros(0, np.uint8)                  # the verdicts stay on the device
                s = api._IovStreams()
                ctx._ck(ctx.lib.nutsb_speech_batch_iov(ctx._h, N_MSGS, api._addr(sp_verb), api._addr(sp_spk), api._addr(bt),
                                                       api._addr(bo), s))
            else:
                v = ctx.contains_swearing_batch(bt, bo)
                o = ctx._ops_struct(dict(hops, verdict=v), keep)
            if mode == "iov":
                s = api._IovStreams()
                ctx._ck(ctx.lib.nutsb_write_batch_iov(ctx._h, o, s))
            if iov:
                touch = int(np.ctypeslib.as_array(api.C.cast(s.pool, api.u8p), shape=(16,))[0])      # touch the result
                touch += int(np.ctypeslib.as_array(api.C.cast(s.iov, api.u64p), shape=(2,))[1])
                out_bytes = int(s.pool_bytes) + int(s.pool2_bytes) + 16 * int(s.n_iov) + 12 * N_USERS
            else:
                s = api._Streams()
                ctx._ck(ctx.lib.nutsb_write_batch(ctx._h, o, s))
                touch = int(np.ctypeslib.as_array(api.C.cast(s.bytes, api.u8p), shape=(16,))[0])
                out_bytes = int(s.total_bytes)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if i == 0:
                # outside the timed passes: the BYTES of sampled users' streams, so that the three legs can be told
                # to deliver the same streams and not just the same counts
                import hashlib
                sample = range(0, N_USERS, max(1, N_USERS // 64))
                offs = np.ctypeslib.as_array(api.C.cast(s.off, api.u64p), shape=(N_USERS + 1,))
                h = hashlib.sha256()
                if iov:
                    first = np.ctypeslib.as_array(api.C.cast(s.first, api.u64p), shape=(N_USERS,))
                    cnt = np.ctypeslib.as_array(api.C.cast(s.count, api.C.POINTER(api.C.c_uint32)), shape=(N_USERS,))
                    pieces = np.ctypeslib.as_array(api.C.cast(s.iov, api.u64p), shape=(int(s.n_iov), 2))
                    for u in sample:
                        for k in range(int(first[u]), int(first[u]) + int(cnt[u])):
                            if pieces[k, 1]:
                                h.update(api.C.string_at(int(pieces[k, 0]), int(pieces[k, 1])))
                else:
                    for u in sample:
                        h.update(api.C.string_at(s.bytes + int(offs[u]), int(offs[u + 1] - offs[u])))
                r["sample_sha"] = h.hexdigest()
            if i == 0 and iov:
                # the lists describe every byte of every stream
                lens = np.ctypeslib.as_array(api.C.cast(s.iov, api.u64p), shape=(int(s.n_iov), 2))[:, 1]
                assert int(lens.sum()) == int(s.total_bytes), "gather lists do not add up to the streams"
                r["extra"] = dict(pool_bytes=int(s.pool_bytes) + int(s.pool2_bytes), n_iov=int(s.n_iov), stream_bytes=int(s.total_bytes))
            if i > 0:
                tt = ctx.timing()
                r["h2d_ms"] += float(tt.h2d_ms); r["d2h_ms"] += float(tt.d2h_ms)
                r["ms"] += dt * 1e3; r["deliv"] += int(s.n_deliveries)
                r["h2d"] = int(bt.nbytes + bo.nbytes + st_.nbytes + so_.nbytes + nt_.nbytes + no_.nbytes)
                r["h2d"] += (5 * N_MSGS if mode == "speech_iov" else
                             int(ops["text"].nbytes + ops["off"].nbytes + 2 * n_ops + 12 * n_ops + v.nbytes))
                r["d2h"] = out_bytes + 8 * (N_USERS + 1) + v.nbytes + vs.nbytes + vu.nbytes
        return r

    e2e_steps = max(1, min(args.steps, 3))
    zero = dict(h2d_ms=0.0, d2h_ms=0.0, ms=0.0, deliv=0, h2d=0, d2h=0, extra={}, sample_sha="")
    leg_s = zero if args.no_e2e else e2e_leg("streams")
    leg_v = zero if args.no_e2e else e2e_leg("iov")
    leg_p = zero if args.no_e2e else e2e_leg("speech_iov")
    if not args.no_e2e:                                    # the three legs deliver the same streams
        assert leg_v["deliv"] == leg_s["deliv"] == leg_p["deliv"], (leg_s["deliv"], leg_v["deliv"], leg_p["deliv"])
        assert leg_v["extra"]["stream_bytes"] == leg_p["extra"]["stream_bytes"]
        assert leg_s["sample_sha"] == leg_v["sample_sha"] == leg_p["sample_sha"], "the e2e legs deliver different bytes"
    e2e_h2d_ms, e2e_d2h_ms, e2e_ms, e2e_deliv, h2d, d2h = (leg_s[k] for k in ("h2d_ms", "d2h_ms", "ms", "deliv", "h2d", "d2h"))

    # ---- the last leg again with two calls in flight (two contexts, two host threads): one call's H2D and
    #      kernels run under the other's D2H (PCIe is full duplex: scripts/probes/pcie_probe.py)
    pipe_ms, pipe_deliv, lib_pipe_ms, lib_pipe3_ms = 0.0, 0, 0.0, 0.0
    if not args.no_e2e:
        c2 = api.Context(local)
        c2.set_swear_words(inp["words"]); c2.set_ban_files(inp["sfile"], inp["ufile"])
        c2.set_users(users["room"], users["flags"], users["level"], inp["n_rooms"])
        c2.set_user_names([un[int(uo[u]):int(uo[u + 1])].tobytes() for u in range(N_USERS)], np.zeros(N_USERS, np.uint8))
        c2.set_ban_swearing(True)
        got = [0, 0]

        def pipe_worker(k, cx, reps):
            for _ in range(reps):
                cx.site_banned_batch(st_, so_); cx.user_banned_batch(nt_, no_)
                s = api._IovStreams()
                cx._ck(cx.lib.nutsb_speech_batch_iov(cx._h, N_MSGS, api._addr(sp_verb), api._addr(sp_spk), api._addr(bt), api._addr(bo), s))
                got[k] += int(s.n_deliveries)

        for reps in (1, e2e_steps):                        # first round allocates the second context's buffers
            got[0] = got[1] = 0
            barrier()
            t0 = time.perf_counter()
            th = [threading.Thread(target=pipe_worker, args=(k, cx, reps)) for k, cx in enumerate((ctx, c2))]
            for t in th:
                t.start()
            for t in th:
                t.join()
            torch.cuda.synchronize()
            pipe_ms = (time.perf_counter() - t0) * 1e3
        pipe_deliv = got[0] + got[1]
        c2.close()
        # the same through the library's own pipe (nutsb_pipe: two contexts and their worker threads inside the
        # library, one caller thread that submits call k+1 before it waits for call k)
        lib_pipe = {}
        for depth in (2, 3):
            pp = api.Pipe(local, depth)
            pp.set_swear_words(inp["words"]); pp.set_users(users["room"], users["flags"], users["level"], inp["n_rooms"])
            pp.set_user_names([un[int(uo[u]):int(uo[u + 1])].tobytes() for u in range(N_USERS)], np.zeros(N_USERS, np.uint8))
            pp.set_ban_swearing(True)
            sub = lambda: pp.submit_speech_iov(sp_verb, sp_spk, bt, bo)
            raw_wait = lambda t: pp.lib.nutsb_pipe_wait(pp._h, t, api.C.byref(api._IovStreams()))
            for reps in (depth, 3 * e2e_steps):             # first round allocates the contexts' buffers
                barrier()
                t0 = time.perf_counter()
                tk = [sub() for _ in range(min(depth, reps))]      # `depth` calls in flight, then one in for one out
                for k in range(reps):
                    assert raw_wait(tk[k]) == 0
                    if len(tk) < reps:
                        tk.append(sub())
                torch.cuda.synchronize()
                lib_pipe[depth] = (time.perf_counter() - t0) * 1e3 / reps
            pp.close()
        lib_pipe_ms, lib_pipe3_ms = lib_pipe[2], lib_pipe[3]
    # ---- reduce over ranks
    vals = torch.tensor([ms, e2e_ms, leg_v["ms"], leg_p["ms"], two_ms, pipe_ms, lib_pipe_ms, lib_pipe3_ms], dtype=torch.float64, device=dev)
    sums = torch.tensor([dev_state["deliv"], e2e_deliv, dev_state["launches"], leg_v["deliv"], pipe_deliv], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    ms_max, e2e_ms_max, iov_ms_max, sp_ms_max, two_ms_max, pipe_ms_max, lib_pipe_ms_max, lib_pipe3_ms_max = (float(vals[i]) for i in range(8))
    total_deliv, total_e2e_deliv, total_launch, total_iov_deliv = float(sums[0]), float(sums[1]), int(sums[2]), float(sums[3])

    if rank == 0:
        peaks = {}
        pk = ROOT / "MEASURED_PEAKS.json"
        if pk.exists():
            peaks = json.loads(pk.read_text())
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
        ks = max(1, kstate["ksteps"])
        fan_bytes = (kstate["fan_in"] + kstate["fan_out"]) / ks
        fan_ms = kstate["fan_ms"] / ks
        achieved = fan_bytes / (fan_ms * 1e-3) / 1e9 if fan_ms > 0 else 0.0
        traffic, traffic_src = None, None
        tp = ROOT / "profiles" / "fanout_traffic.json"
        if tp.exists():             # an ncu figure (dram__bytes_read.sum + dram__bytes_write.sum of one k_fanout launch), NOT measured by this run
            try:
                tj = json.loads(tp.read_text())
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
            except Exception:
                traffic = None
        line = dict(metric=METRIC, value=total_deliv / (ms_max * 1e-3), unit=UNIT, n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms_max / max(1, args.steps), higher_is_better=True, scaling="weak",
                    vs_baseline=None, dtype="u8", data="synthetic",
                    config=dict(workload=workload_name(), sharding="rooms per rank, no collective",
                                l2="inputs (%.0f MB) and outputs (%.1f GB) per step exceed the 126 MB L2; no flush needed"
                                   % (input_bytes / 1e6, dev_state["bytes"] / max(1, args.steps) / 1e9),
                                batches_in_flight=len(lanes),
                                two_batches_in_flight=(None if two_ms_max <= 0 else dict(
                                    value=total_deliv / (two_ms_max * 1e-3),
                                    ms_per_step=two_ms_max / max(1, args.steps),
                                    note="same K steps dealt to two contexts / host threads on the GPU; not the headline")),
                                source_msgs_per_s=world * N_MSGS * args.steps / (ms_max * 1e-3),
                                ban_queries_per_step=2 * N_BAN_QUERIES,
                                kernel_ms_alone=dict(plan=kstate["plan_ms"] / ks, render=kstate["render_ms"] / ks, fanout=fan_ms,
                                                     direct=kstate["direct_ms"] / ks, steps=ks,
                                                     how="extra steps after the timed region with nutsb_set_overlap(0): "
                                                         "every kernel on one stream, CUDA events around each"),
                                timed_region_ms=dict(plan_until_fanout=dev_state["plan_ms"] / max(1, dev_state["ksteps"]),
                                                     render_span=dev_state["render_ms"] / max(1, dev_state["ksteps"]),
                                                     fanout_and_direct=dev_state["fan_ms"] / max(1, dev_state["ksteps"]),
                                                     how="CUDA events of the timed steps themselves (side stream on)"),
                                plan_ms=kstate["plan_ms"] / ks, render_ms=kstate["render_ms"] / ks, fanout_ms=fan_ms,
                                direct_ms=kstate["direct_ms"] / ks),
                    roofline=dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak,
                                  traffic=traffic, traffic_source=traffic_src, kernel="k_fanout", peak_source=peak_src,
                                  algorithmic_bytes_per_launch=fan_bytes,
                                  frac_of_spec_8000=achieved / 8000.0,          # SURVEY 8d: both percentages
                                  whole_step=dict(achieved=(dev_state["bytes"] / max(1, args.steps) + input_bytes) / (ms_max / max(1, args.steps) * 1e-3) / 1e9,
                                                  unit="GB/s", note="stream bytes written + input bytes read per step / ms_per_step (rank 0): "
                                                                    "what the planning, rendering and verdict kernels cost on top of the fan-out")),
                    e2e=(None if args.no_e2e else
                         dict(value=total_e2e_deliv / (e2e_ms_max * 1e-3), unit=UNIT, h2d_bytes_per_step=h2d,
                              d2h_bytes_per_step=d2h, steps=e2e_steps, ms_per_step=e2e_ms_max / e2e_steps,
                              write_batch_h2d_ms=e2e_h2d_ms / e2e_steps, write_batch_d2h_ms=e2e_d2h_ms / e2e_steps,
                              host_memory="pinned (inputs: caller's pinned buffers; streams: the library's pinned buffer)")),
                    gpu_launches=total_launch, clocks=clk)
        if not args.no_e2e:
            # the same step with gather lists as the result (nutsb_write_batch_iov): what a host that writev()s needs.
            # Reported beside `e2e`, which stays the full per-recipient streams.
            line["e2e_iov"] = dict(value=total_iov_deliv / (iov_ms_max * 1e-3), unit=UNIT, h2d_bytes_per_step=leg_v["h2d"],
                                   d2h_bytes_per_step=leg_v["d2h"], steps=e2e_steps, ms_per_step=iov_ms_max / e2e_steps,
                                   write_batch_h2d_ms=leg_v["h2d_ms"] / e2e_steps, write_batch_d2h_ms=leg_v["d2h_ms"] / e2e_steps,
                                   result="per-user struct iovec lists into one pinned pool: every room op rendered once per "
                                          "colour setting + every write_user op rendered once; byte-identical to `e2e`'s streams "
                                          "when gathered (tests/test_iov.py)", **leg_v["extra"])
            # ... and from the input lines themselves: say(user, inpstr) x 1M through nutsb_speech_batch_iov
            line["e2e_speech_iov"] = dict(value=total_iov_deliv / (sp_ms_max * 1e-3), unit=UNIT, h2d_bytes_per_step=leg_p["h2d"],
                                          d2h_bytes_per_step=leg_p["d2h"], steps=e2e_steps, ms_per_step=sp_ms_max / e2e_steps,
                                          input="verb, speaker and body of every line (nutsb_speech_batch_iov): swear verdicts, "
                                                "say()'s composition and the rendering all on the device", **leg_p["extra"])
            line["e2e_speech_iov"]["two_calls_in_flight"] = dict(
                value=float(sums[4]) / (pipe_ms_max * 1e-3), ms_per_step=pipe_ms_max / (2 * e2e_steps),
                note="two contexts / host threads per GPU, %d calls each: one call's H2D and kernels under the other's D2H" % e2e_steps)
            line["e2e_speech_iov"]["library_pipe"] = dict(
                value=total_iov_deliv / e2e_steps / (lib_pipe_ms_max * 1e-3), ms_per_call=lib_pipe_ms_max,
                depth3=dict(value=total_iov_deliv / e2e_steps / (lib_pipe3_ms_max * 1e-3), ms_per_call=lib_pipe3_ms_max),
                note="nutsb_pipe (depth 2; depth3: three contexts): ONE caller thread keeps `depth` calls in flight; the speech lines only "
                     "(the step's two ban batches, 0.2 ms, are not part of these calls); the D2H floor of a call is 3.5 ms")
        line["roofline"]["whole_step"]["frac"] = line["roofline"]["whole_step"]["achieved"] / peak
        line["config"]["verdict_kernel_ms"] = dict(comp_ms, how="each verdict kernel alone, CUDA events, best of %d" % KERNEL_TIMING_STEPS)
        if world == 1 and not args.no_cpu_baseline:
            procs = 1
            comp = {}
            dcpu, nbytes, busy, wall, kind = reference_step(0, 40_000, 4_000, procs, both_sinks=True, components=comp)
            line["cpu_baseline"] = dict(value=dcpu / busy, unit=UNIT, cores=procs, kind=kind,
                                        sample="40000 of 1000000 msgs (all 10000 users) + 4000 of 100000 ban queries per "
                                               "list, one single-threaded reference process pinned to core %s, write(2) hooked "
                                               "to a byte counter" % comp.get("pinned_core"))
            # what the one number above hides: per component, the reference on one pinned core against this GPU.
            # The reference's ban checks re-open and re-parse the 10k-entry file per query (nuts333.c:330-364): they
            # are ~90 % of its time on this workload, so the whole-step ratio is mostly a ban-file ratio.
            write_ms = ms_max / max(1, args.steps) - sum(comp_ms.values())
            gpu_d = total_deliv / max(1, args.steps)
            vc = dict(
                render_fanout=dict(gpu=gpu_d / (write_ms * 1e-3), cpu_1core=comp["deliveries"] / comp["write_s"], unit="deliveries/s",
                                   cpu_sink="write(2) hooked to a byte counter (no syscalls)",
                                   gpu_note="step time minus the verdict kernels, inputs resident in HBM, streams left in HBM"),
                swear=dict(gpu=N_MSGS / (comp_ms["swear"] * 1e-3), cpu_1core=comp["n_msgs"] / comp["swear_s"], unit="msgs/s", words=N_SWEAR),
                bans=dict(gpu=2 * N_BAN_QUERIES / ((comp_ms["site"] + comp_ms["user"]) * 1e-3), cpu_1core=comp["n_ban"] / comp["bans_s"],
                          unit="queries/s", entries=N_BAN_ENTRIES),
                cpu_time_share=dict(swear=comp["swear_s"] / busy, bans=comp["bans_s"] / busy, render_fanout=comp["write_s"] / busy),
                pinned_core=comp.get("pinned_core"))
            if "write_devnull_s" in comp:
                vc["render_fanout"]["cpu_1core_devnull"] = comp["deliveries"] / comp["write_devnull_s"]
                vc["render_fanout"]["cpu_devnull_sink"] = "the faithful sink: real write(2) to /dev/null, %.2f calls per delivery" % (comp.get("write_calls", 0) / max(1, comp["deliveries"]))
            for k in ("render_fanout", "swear", "bans"):
                vc[k]["ratio"] = vc[k]["gpu"] / vc[k]["cpu_1core"]
            if not args.no_e2e:
                vc["render_fanout"]["gpu_e2e_streams"] = line["e2e"]["value"]
                vc["render_fanout"]["gpu_e2e_gather_lists"] = line["e2e_iov"]["value"]
            line["vs_cpu_components"] = vc
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    for L in lanes:
        L["ctx"].close()
    return 0


# ---------------------------------------------------------------------------------------
# the other BASELINE configs (BASELINE.md section 3: "reported per config and GPU count")
# ---------------------------------------------------------------------------------------
def run_config(args):
    """--config c2 | c4 | c5: one JSON line each, same timing rules as the default line (CUDA events on the stream the
    kernels run on, >= 3 warm-up steps, max over ranks).  c2 = BASELINE config 2 (100k msgs x 1k users in one room,
    colour only), c4 = config 4 alone (100k sites + 100k names vs 10k-entry lists), c5 = config 5 (10M msgs x 100k users,
    admission -> swear -> say, rooms sharded over the GPUs by the library's sharder: STRONG scaling, total work fixed)."""
    import torch
    import torch.distributed as dist
    from nuts333_b200 import api, build, synth

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    build.build()
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    stream = torch.cuda.Stream(device=dev, priority=-1)         # (the library's side stream is created at the lowest priority)
    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    pad16 = lambda a: np.concatenate([a, np.zeros(32, np.uint8)])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    words = synth.swear_words(N_SWEAR)
    cfg = args.config
    line = None
    if cfg == "c2":
        M, U = 100_000, 1_000
        users, n_rooms = synth.users(U, U)                       # one room
        bt, bo = synth.bodies(M, None)
        ops, spk, rm = synth.say_ops(M, U, U, bt, bo, gated=False)
        ctx = api.Context(local); ctx.set_stream(stream.cuda_stream); ctx.set_profiling(True)
        ctx.set_users(users["room"], users["flags"], users["level"], n_rooms)
        dd = dict(text=to_dev(pad16(ops["text"])), off=to_dev(ops["off"].view(np.int64)), kind=to_dev(ops["kind"]), target=to_dev(ops["target"]),
                  exc=to_dev(ops["except_user"]), flags=to_dev(ops["flags"]))
        acc = dict(deliv=0, bytes=0, fan_ms=0.0, fan_b=0, n=0, launches=0)

        def step():
            st = ctx.write_batch_dev(len(ops["kind"]), dd["text"].data_ptr(), dd["off"].data_ptr(), dd["kind"].data_ptr(), dd["target"].data_ptr(),
                                     dd["exc"].data_ptr(), dd["flags"].data_ptr())
            t = ctx.timing()
            acc["deliv"] += int(st.n_deliveries); acc["bytes"] += int(st.total_bytes); acc["fan_ms"] += float(t.fanout_ms)
            acc["fan_b"] += int(t.fanout_bytes_in) + int(t.fanout_bytes_out); acc["n"] += 1; acc["launches"] += int(t.launches)
        for _ in range(args.warmup):
            step()
        for k in acc:
            acc[k] = 0 if not isinstance(acc[k], float) else 0.0
        tw0 = time.perf_counter()
        ms = timed(step, args.steps, 0)
        tw1 = time.perf_counter()
        in_bytes = int(ops["text"].nbytes + ops["off"].nbytes + 10 * len(ops["kind"]))
        # host buffers: streams (the full per-recipient bytes) and gather lists
        hops = {k: v for k, v in ops.items()}
        e2e = {}
        for mode in ("streams", "iov"):
            fn = ctx.write_batch if mode == "streams" else ctx.write_batch_iov
            fn(hops); barrier()
            t0 = time.perf_counter()
            for _ in range(2):
                r = fn(hops)
            torch.cuda.synchronize()
            e2e[mode] = (time.perf_counter() - t0) / 2
        d_per = acc["deliv"] / acc["n"]
        ach = acc["fan_b"] / acc["n"] / (acc["fan_ms"] / acc["n"] * 1e-3) / 1e9
        line = dict(metric=METRIC, value=acc["deliv"] / (ms * 1e-3), unit=UNIT, n_gpus=1, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="u8", data="synthetic",
                    config=dict(workload="C2: %d say() lines x %d users in ONE room, colour expand/strip only (no swear gate), 1 B200" % (M, U),
                                l2="outputs (%.1f GB) per step exceed the 126 MB L2" % (acc["bytes"] / acc["n"] / 1e9), source_msgs_per_s=M * args.steps / (ms * 1e-3)),
                    roofline=dict(bound="hbm", kernel="k_fanout", achieved=ach, peak=peak, unit="GB/s", frac=ach / peak, traffic=None, peak_source=peak_src,
                                  whole_step=dict(achieved=(acc["bytes"] / acc["n"] + in_bytes) / (ms / args.steps * 1e-3) / 1e9, unit="GB/s",
                                                  frac=(acc["bytes"] / acc["n"] + in_bytes) / (ms / args.steps * 1e-3) / 1e9 / peak)),
                    e2e=dict(value=d_per / e2e["streams"], unit=UNIT, h2d_bytes_per_step=in_bytes, d2h_bytes_per_step=int(acc["bytes"] / acc["n"]), ms_per_step=1e3 * e2e["streams"]),
                    e2e_iov=dict(value=d_per / e2e["iov"], unit=UNIT, ms_per_step=1e3 * e2e["iov"]),
                    gpu_launches=acc["launches"])
        ctx.close()
    elif cfg == "c4":
        NQ, NE = 100_000, 10_000
        st_, so_ = synth.sites(NQ); nt_, no_ = synth.names(NQ)
        ctx = api.Context(local); ctx.set_stream(stream.cuda_stream)
        dd = dict(st=to_dev(pad16(st_)), so=to_dev(so_.view(np.int64)), nt=to_dev(pad16(nt_)), no=to_dev(no_.view(np.int64)),
                  vs=torch.zeros(NQ, dtype=torch.uint8, device=dev), vu=torch.zeros(NQ, dtype=torch.uint8, device=dev))
        res = {}
        for nl in (True, False):                                 # the file with and without its last newline (the feof quirk)
            sf, uf = synth.ban_file(0, NE, NQ, NQ, nl), synth.ban_file(1, NE, NQ, NQ, nl)
            ctx.set_ban_files(sf, uf)

            def step():
                ctx.verdicts_dev("site_banned", NQ, dd["st"].data_ptr(), dd["so"].data_ptr(), dd["vs"].data_ptr())
                ctx.verdicts_dev("user_banned", NQ, dd["nt"].data_ptr(), dd["no"].data_ptr(), dd["vu"].data_ptr())
            tw0 = time.perf_counter()
            res[nl] = timed(step, args.steps, args.warmup)
            tw1 = time.perf_counter()
            t0 = time.perf_counter()
            for _ in range(3):
                ctx.site_banned_batch(st_, so_); ctx.user_banned_batch(nt_, no_)
            res[(nl, "e2e")] = (time.perf_counter() - t0) / 3
        ms = res[True]
        algo = int(st_.nbytes + nt_.nbytes + 2 * NQ + len(sf) + len(uf))
        line = dict(metric="ban verdicts/sec (site_banned + user_banned)", value=2 * NQ * args.steps / (ms * 1e-3), unit="queries/s", n_gpus=1, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="u8", data="synthetic",
                    config=dict(workload="C4: %d sites + %d names vs %d-entry siteban / userban files" % (NQ, NQ, NE),
                                without_trailing_newline_ms_per_step=res[False] / args.steps,
                                l2="queries (3 MB) and tables live in L2 / shared memory: latency-bound, not HBM-bound (SURVEY 8d)"),
                    roofline=dict(bound="hbm", kernel="k_ac_match<0> + k_set_match", achieved=algo / (ms / args.steps * 1e-3) / 1e9, peak=peak, unit="GB/s",
                                  frac=algo / (ms / args.steps * 1e-3) / 1e9 / peak, traffic=None, peak_source=peak_src,
                                  note="working set in L2: the HBM floor is microseconds; reported for completeness"),
                    e2e=dict(value=2 * NQ / res[(True, "e2e")], unit="queries/s", h2d_bytes_per_step=int(st_.nbytes + so_.nbytes + nt_.nbytes + no_.nbytes),
                             d2h_bytes_per_step=2 * NQ, ms_per_step=1e3 * res[(True, "e2e")]),
                    gpu_launches=2 * args.steps)
        ctx.close()
    else:                                                        # c5
        UT, UPR, MT = args.c5_users, 100, args.c5_msgs
        CH = min(args.c5_chunk * world, MT)                      # a chunk = --c5-chunk messages per GPU
        n_chunks = (MT + CH - 1) // CH
        users, n_rooms = synth.users(UT, UPR)
        m = api.MultiContext(rank=(world, rank, local))
        m.set_profiling(True)
        m.set_swear_words(words)
        sfile, ufile = synth.ban_file(0, N_BAN_ENTRIES, UT, UT, True), synth.ban_file(1, N_BAN_ENTRIES, UT, UT, True)
        m.set_ban_files(sfile, ufile)
        ctx = m.ctx(rank)
        ctx.set_stream(stream.cuda_stream)
        # stage A, admission (site_banned or user_banned => never a recipient, never a speaker): split by rank, gathered
        st_, so_ = synth.sites(UT); nt_, no_ = synth.names(UT)
        lo, hi = rank * UT // world, (rank + 1) * UT // world
        dA = dict(st=to_dev(pad16(st_)), so=to_dev(so_.view(np.int64)), nt=to_dev(pad16(nt_)), no=to_dev(no_.view(np.int64)),
                  vs=torch.zeros(UT, dtype=torch.uint8, device=dev), vu=torch.zeros(UT, dtype=torch.uint8, device=dev))

        def admission():
            ctx.verdicts_dev("site_banned", hi - lo, dA["st"].data_ptr(), dA["so"].data_ptr() + 8 * lo, dA["vs"].data_ptr() + lo)
            ctx.verdicts_dev("user_banned", hi - lo, dA["nt"].data_ptr(), dA["no"].data_ptr() + 8 * lo, dA["vu"].data_ptr() + lo)
        admission(); torch.cuda.synchronize()
        banned = (dA["vs"] | dA["vu"])
        if world > 1:
            parts = [torch.zeros_like(banned) for _ in range(world)]
            dist.all_gather(parts, banned)                         # (gathering outputs: the only cross-rank traffic)
            banned = torch.zeros_like(banned)
            for r in range(world):
                a, b = r * UT // world, (r + 1) * UT // world
                banned[a:b] = parts[r][a:b]
        banned = banned.cpu().numpy().astype(bool)
        uf2, ur2 = users["flags"].copy(), users["room"].copy()
        uf2[banned] |= api.UF_LOGIN; ur2[banned] = -1
        m.set_users(ur2, uf2, users["level"], n_rooms)
        _, ush, _ = m.plan()
        # stage B + C inputs, chunk by chunk: every rank generates the same global chunk, the library routes it, the
        # rank's share goes to its HBM (resident before anything is timed)
        chunks = []
        for c in range(n_chunks):
            m0, n = c * CH, min(CH, MT - c * CH)
            bt, bo = synth.bodies(n, words, m0=m0)
            ops, spk, rm = synth.say_ops(n, UT, UPR, bt, bo, gated=True, m0=m0)
            dead = np.repeat(banned[spk], 3)
            ops["kind"] = np.where(dead, np.uint8(3), ops["kind"]).astype(np.uint8)      # a banned speaker says nothing (NUTSB_OP_NONE)
            r = m.route(dict(ops, verdict=np.zeros(n, np.uint8)), rank)
            b_lo, b_hi = rank * n // world, (rank + 1) * n // world
            chunks.append(dict(n=n, n_ops=len(r["kind"]), bt=to_dev(pad16(bt)), bo=to_dev(bo.view(np.int64)), b_lo=b_lo, b_hi=b_hi,
                               text=to_dev(pad16(r["text"])), off=to_dev(r["off"].view(np.int64)), kind=to_dev(r["kind"]), target=to_dev(r["target"]),
                               exc=to_dev(r["except_user"]), flags=to_dev(r["flags"]), gate=to_dev(r["gate"]),
                               verdict=torch.zeros(n, dtype=torch.uint8, device=dev),
                               parts=[torch.zeros(n, dtype=torch.uint8, device=dev) for _ in range(world)] if world > 1 else None))
        acc = dict(deliv=0, bytes=0, launches=0, fan_ms=0.0, fan_b=0, n=0)
        digests = [None]

        def job(with_digests=False):
            admission()
            dg = None
            for ck in chunks:
                # swear verdicts: this rank's index range, then gathered (1 byte per message)
                ctx.verdicts_dev("contains_swearing", ck["b_hi"] - ck["b_lo"], ck["bt"].data_ptr(), ck["bo"].data_ptr() + 8 * ck["b_lo"],
                                 ck["verdict"].data_ptr() + ck["b_lo"])
                if world > 1:
                    with torch.cuda.stream(stream):
                        dist.all_gather(ck["parts"], ck["verdict"])
                        for r in range(world):
                            a, b = r * ck["n"] // world, (r + 1) * ck["n"] // world
                            ck["verdict"][a:b] = ck["parts"][r][a:b]
                st = ctx.write_batch_dev(ck["n_ops"], ck["text"].data_ptr(), ck["off"].data_ptr(), ck["kind"].data_ptr(), ck["target"].data_ptr(),
                                         ck["exc"].data_ptr(), ck["flags"].data_ptr(), ck["gate"].data_ptr(), ck["verdict"].data_ptr())
                t = ctx.timing()
                acc["deliv"] += int(st.n_deliveries); acc["bytes"] += int(st.total_bytes); acc["launches"] += int(t.launches) + 1
                acc["fan_ms"] += float(t.fanout_ms); acc["fan_b"] += int(t.fanout_bytes_in) + int(t.fanout_bytes_out); acc["n"] += 1
                if with_digests:
                    dg = m.stream_digests(dg)
            if with_digests:
                digests[0] = dg
        job(with_digests=True)                                   # warm-up no. 1, with the per-user digests of the whole job
        for _ in range(max(0, args.warmup - 1)):
            job()
        for k in acc:
            acc[k] = 0 if not isinstance(acc[k], float) else 0.0
        tw0 = time.perf_counter()
        ms = timed(job, args.steps, 0)
        tw1 = time.perf_counter()
        mine = ush == rank
        # a checksum of the per-user digests: the same number whatever the GPU count means the same streams
        chk = np.bitwise_xor.reduce(digests[0][mine]) if mine.any() else np.uint64(0)
        sm = torch.tensor([float(acc["deliv"]), float(acc["bytes"]), float(acc["launches"])], dtype=torch.float64, device=dev)
        cx = torch.tensor([np.int64(np.uint64(chk).astype(np.int64))], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            cxs = [torch.zeros_like(cx) for _ in range(world)]
            dist.all_gather(cxs, cx)
            allx = np.bitwise_xor.reduce(np.array([int(t[0]) for t in cxs], np.int64).astype(np.uint64))
        else:
            allx = np.uint64(chk)
        ach = acc["fan_b"] / max(1, acc["n"]) / (acc["fan_ms"] / max(1, acc["n"]) * 1e-3) / 1e9 if acc["fan_ms"] > 0 else 0.0
        in_bytes = sum(int(v.numel() * v.element_size()) for ck in chunks for k, v in ck.items() if isinstance(v, torch.Tensor) and k != "verdict")
        line = dict(metric=METRIC, value=float(sm[0]) / (ms * 1e-3), unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="u8", data="synthetic",
                    config=dict(workload="C5: full pipeline, %d msgs x %d users (%d rooms of %d): admission (site_banned | user_banned, %d-entry lists) -> "
                                         "contains_swearing (%d words) -> say() render + fan-out, in %d message-ordered chunks (%d messages per GPU each); one step = the whole job"
                                         % (MT, UT, n_rooms, UPR, N_BAN_ENTRIES, N_SWEAR, n_chunks, args.c5_chunk),
                                sharding="rooms dealt to the GPUs by nutsb_multi (the library's sharder), streams stay in HBM; swear / ban batches split by "
                                         "index range and their verdict bytes gathered (NCCL all_gather: the only cross-rank traffic)",
                                l2="per chunk and GPU: inputs and outputs far beyond the 126 MB L2",
                                banned_users=int(banned.sum()), deliveries_per_job=float(sm[0]) / args.steps, stream_bytes_per_job=float(sm[1]) / args.steps,
                                digest_checksum="%016x" % int(allx), source_msgs_per_s=MT * args.steps / (ms * 1e-3)),
                    roofline=dict(bound="hbm", kernel="k_fanout", achieved=ach, peak=peak, unit="GB/s", frac=ach / peak, traffic=None, peak_source=peak_src,
                                  whole_step=dict(achieved=(float(sm[1]) / args.steps / world + in_bytes) / (ms / args.steps * 1e-3) / 1e9, unit="GB/s per GPU",
                                                  frac=(float(sm[1]) / args.steps / world + in_bytes) / (ms / args.steps * 1e-3) / 1e9 / peak)),
                    e2e=None, gpu_launches=int(sm[2]))
        m.close()
    clocks.window(tw0, tw1)
    clk = clocks.stop()
    if rank == 0:
        line["clocks"] = clk
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--in-flight", type=int, default=IN_FLIGHT, help="batches in flight per GPU (one context + host thread each)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--config", default="c3c4", choices=["c3c4", "c2", "c4", "c5"],
                    help="c3c4 (default): the headline workload; c2 / c4 / c5: the other BASELINE configs, one line each")
    ap.add_argument("--c5-msgs", type=int, default=10_000_000)
    ap.add_argument("--c5-chunk", type=int, default=10_000_000,
                    help="config 5: messages per GPU in one chunk = one write batch (default: the whole job in one; 1000000 = the same HBM per GPU at every N)")
    ap.add_argument("--c5-users", type=int, default=100_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != "c3c4"):
        ap.error("--dump-outputs is implemented for the default workload (--impl ours --config c3c4) only")
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs writes the last timed step's results: it needs --steps 1 or more")
    if args.impl == "reference":
        return run_reference(args)
    if args.config != "c3c4":
        return run_config(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
