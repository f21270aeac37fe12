"""What recording costs a speech batch (nutsb_set_speech_record): bench.py's C3 lines (1M say() lines over 10k users in
100 rooms, 64-word swear list, ban_swearing) through nutsb_speech_batch_iov with recording off and on.

Reports
  * wall ms per call, off and on (host clock around the call, which returns with the gather lists on the host and, with
    recording on, the records applied; pinned inputs; warm-up calls first, then off / on alternating for `--reps` rounds);
  * nutsb_timing of one more call each way with profiling on;
  * the recording step's own device time: in a torch.profiler run of one call, the kernels on the context's stream from
    k_speech_rec_mark to k_speech_rec_pack (the step's scans and sort included), summed, and their span;
  * the bytes the step brings to the host, read from the same traces: the copy right after k_speech_rec_pack (the packed
    size, 8 bytes) and the call's last device-to-host copy (the packed records: per room that recorded anything, a
    24-byte header and the bytes strncpy keeps of its last 15 records), checked against the restatement of the packing;
  * the card name and power limit.
Checks every room's buffer (rows and head) against a numpy restatement of record() over the lines: the last 15 say()
lines of each room that the swear list (the oracle's verdicts) does not refuse, from an empty start.

    python scripts/probes/speech_record_probe.py --out profiles/speech_record_probe.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

N_MSGS, N_USERS, USERS_PER_ROOM, N_SWEAR = 1_000_000, 10_000, 100, 64


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [line.strip() for line in q.stdout.splitlines() if line.strip()]


def restate(spk, bt, bo, room, names, refused, n_rooms, review_lines, review_len):
    """record()'s rows and head of every room, and the packed bytes the device step copies"""
    row_len = review_len + 2
    kept = ~refused & (room[spk] >= 0)
    idx = np.nonzero(kept)[0]
    rooms_of = room[spk[idx]]
    out, packed = [], 8
    for r in range(n_rooms):
        lines = idx[rooms_of == r]
        c = len(lines)
        rows = [b"\0" * row_len] * review_lines
        if c:
            packed += 24
        for i, m in enumerate(lines[-review_lines:]):
            body = bt[int(bo[m]):int(bo[m + 1])].tobytes()
            t = {b"?": b" asks: ", b"!": b" exclaims: "}.get(body[-1:], b" says: ")
            text = (names[int(spk[m])] + t + body + b"\n")[:review_len].split(b"\0")[0]
            packed += len(text)
            rows[(c - min(c, review_lines) + i) % review_lines] = text.ljust(review_len, b"\0") + b"\n\0"
        out.append((rows, c % review_lines))
    return out, packed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--msgs", type=int, default=N_MSGS)
    args = ap.parse_args()

    import torch
    import oracle_lib as O
    from nuts333_b200 import api, build, shard, synth
    build.build()
    if torch.cuda.device_count() < 1:
        raise SystemExit("no CUDA device")

    words = synth.swear_words(N_SWEAR)
    sh = shard.shard_inputs(0, args.msgs, N_USERS, USERS_PER_ROOM, words, gated=True)
    us, n_rooms = sh["users"], sh["n_rooms"]
    bt, bo = sh["bodies"]
    verb = np.zeros(args.msgs, np.uint8)                      # say()
    spk = sh["speaker"].astype(np.int32)
    un, uo = synth.names(N_USERS)
    names = [un[int(uo[u]):int(uo[u + 1])].tobytes() for u in range(N_USERS)]
    sflags = np.zeros(N_USERS, np.uint8)
    pinned = []

    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        pinned.append(t)
        return t.numpy()

    lines = tuple(pin(a) for a in (verb, spk, bt, bo))

    ctx = api.Context(0)
    ctx.set_swear_words(words)
    ctx.set_users(us["room"], us["flags"], us["level"], n_rooms)
    ctx.set_user_names(names, sflags)
    ctx.set_ban_swearing(True)

    def call(on):
        ctx.set_speech_record(on)
        t0 = time.perf_counter()
        ctx.speech_batch_iov(*lines)
        return (time.perf_counter() - t0) * 1e3

    # one recorded call from empty buffers, checked against the restatement
    call(True)
    refused = O.port().contains_swearing_batch(bt, bo, words) != 0
    want, packed_bytes = restate(spk, bt, bo, np.asarray(us["room"]), names, refused, n_rooms, api.REVIEW_LINES, api.REVIEW_LEN)
    got = [ctx.review_buffer(r) for r in range(n_rooms)]
    check = dict(rooms=n_rooms, rooms_equal=sum(g == w for g, w in zip(got, want)), recorded_lines=int((~refused).sum()))
    assert check["rooms_equal"] == n_rooms, check

    for _ in range(args.warmup):
        call(False); call(True)
    wall = {"off": [], "on": []}
    for _ in range(args.reps):
        wall["off"].append(call(False))
        wall["on"].append(call(True))

    timing = {}
    ctx.set_profiling(True)
    for name, on in (("off", False), ("on", True)):
        call(on)
        t = ctx.timing()
        timing[name] = dict(h2d_ms=round(t.h2d_ms, 3), d2h_ms=round(t.d2h_ms, 3), total_ms=round(t.total_ms, 3),
                            plan_ms=round(t.plan_ms, 3), render_ms=round(t.render_ms, 3), launches=int(t.launches))
    ctx.set_profiling(False)

    from torch.profiler import ProfilerActivity, profile
    steps = []
    for _ in range(3):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(True)
            torch.cuda.synchronize()
        ev = sorted([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                     and "Memcpy" not in e.name and "Memset" not in e.name],
                    key=lambda e: e.time_range.start)
        first = next(i for i, e in enumerate(ev) if "k_speech_rec_mark" in e.name)
        last = next(i for i, e in enumerate(ev) if "k_speech_rec_pack" in e.name)
        step = ev[first:last + 1]
        with tempfile.TemporaryDirectory() as td:
            prof.export_chrome_trace(str(Path(td) / "trace.json"))
            trace = json.loads((Path(td) / "trace.json").read_text())["traceEvents"]
        pack_end = max(e["ts"] + e.get("dur", 0) for e in trace if "k_speech_rec_pack" in e.get("name", ""))
        d2h = sorted((e for e in trace if "Memcpy DtoH" in e.get("name", "")), key=lambda e: e["ts"])
        size_copy = next(e for e in d2h if e["ts"] >= pack_end)
        steps.append(dict(kernels=[e.name.replace("void ", "").split("(")[0] for e in step],
                          kernel_us=round(sum(e.time_range.elapsed_us() for e in step), 2),
                          span_us=round(step[-1].time_range.end - step[0].time_range.start, 2),
                          size_copy_bytes=int(size_copy["args"]["bytes"]), records_copy_bytes=int(d2h[-1]["args"]["bytes"])))
    copied = steps[-1]["size_copy_bytes"] + steps[-1]["records_copy_bytes"]
    check["bytes_to_host_equal_restatement"] = copied == packed_bytes

    out = dict(
        probe="speech_record_probe",
        cards=card_info(),
        workload=dict(lines=args.msgs, verb="say", users=N_USERS, rooms=n_rooms, swear_words=N_SWEAR, ban_swearing=True,
                      call="nutsb_speech_batch_iov"),
        wall_ms={k: dict(median=round(float(np.median(v)), 3), min=round(float(np.min(v)), 3), max=round(float(np.max(v)), 3),
                         all=[round(x, 3) for x in v]) for k, v in wall.items()},
        timing=timing,
        record_step=dict(device=steps, bytes_to_host=copied),
        check=check,
        note="wall: host clock around one call, off / on alternating; record_step.device: torch.profiler, kernels from "
             "k_speech_rec_mark to k_speech_rec_pack (kernel_us: their summed durations, span_us: first start to last end); "
             "size_copy_bytes / records_copy_bytes: the two device-to-host copies of the step in the same trace; bytes_to_host: "
             "their sum (equal to the restatement of the packing: check)")
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(json.dumps(dict(cards=out["cards"], wall_ms={k: v["median"] for k, v in out["wall_ms"].items()},
                          record_step=out["record_step"]["device"][-1], bytes=copied, check=check)))
    ctx.close()
    assert check["bytes_to_host_equal_restatement"], (copied, packed_bytes)


if __name__ == "__main__":
    main()
