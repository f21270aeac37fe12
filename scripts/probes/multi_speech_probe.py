"""Speech batches over several GPUs: nutsb_multi_speech_batch_iov at 1 / 2 / 4 / 8 GPUs against nutsb_speech_batch_iov
on one context, on bench.py's C3 lines (1M say() lines over 10k users in 100 rooms, 64-word swear list, ban_swearing)
with a share of them turned into shouts.  Every shard is given the whole batch (73 MB of input per shard) and takes
the swear verdicts of every line, so the probe shows what the replicated input costs against the per-shard work.

Reports wall ms per call (host clock around the call, which ends with its results on the host; warm-up calls first,
then the configurations in turn, `--reps` rounds), each shard's nutsb_timing (h2d / d2h / total, taken in one more call
with profiling on), the shout share, and the card name and power limit.  Checks, for every configuration, the
per-user stream lengths and the bytes of 64 sampled users against the one-context run.

    python scripts/probes/multi_speech_probe.py --out profiles/multi_speech_probe.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

N_MSGS, N_USERS, USERS_PER_ROOM, N_SWEAR = 1_000_000, 10_000, 100, 64


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [line.strip() for line in q.stdout.splitlines() if line.strip()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shout-share", type=float, default=0.001)
    ap.add_argument("--msgs", type=int, default=N_MSGS)
    args = ap.parse_args()

    import torch
    from nuts333_b200 import api, build, shard, synth
    build.build()
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        raise SystemExit("no CUDA device")

    words = synth.swear_words(N_SWEAR)
    sh = shard.shard_inputs(0, args.msgs, N_USERS, USERS_PER_ROOM, words, gated=True)
    us, n_rooms = sh["users"], sh["n_rooms"]
    bt, bo = sh["bodies"]
    rng = np.random.default_rng(0x333)
    verb = np.zeros(args.msgs, np.uint8)
    verb[rng.random(args.msgs) < args.shout_share] = api.SPEECH_SHOUT
    spk = sh["speaker"].astype(np.int32)
    un, uo = synth.names(N_USERS)
    names = [un[int(uo[u]):int(uo[u + 1])].tobytes() for u in range(N_USERS)]
    sflags = np.zeros(N_USERS, np.uint8)

    pinned = []

    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        pinned.append(t)
        return t.numpy()

    verb, spk, bt, bo = pin(verb), pin(spk), pin(bt), pin(bo)
    lines = (verb, spk, bt, bo)
    h2d_bytes = int(verb.nbytes + spk.nbytes + bt.nbytes + bo.nbytes)

    one = api.Context(0)
    one.set_swear_words(words)
    one.set_users(us["room"], us["flags"], us["level"], n_rooms)
    one.set_user_names(names, sflags)
    one.set_ban_swearing(True)

    configs = {"one_context": one}
    for g in (1, 2, 4, 8):
        if g <= n_dev:
            m = api.MultiContext(list(range(g)))
            m.set_swear_words(words)
            m.set_user_names(names, sflags)
            m.set_users(us["room"], us["flags"], us["level"], n_rooms)
            m.set_ban_swearing(True)
            configs["multi_%dgpu" % g] = m

    def call(name):
        c = configs[name]
        t0 = time.perf_counter()
        iv = c.speech_batch_iov(*lines)
        return (time.perf_counter() - t0) * 1e3, iv

    # correctness against the one-context run, and warm-up
    _, ref = call("one_context")
    ref_len, ref_deliv = np.diff(ref.off), ref.n_deliveries
    sample = list(range(0, N_USERS, N_USERS // 64))[:64]
    ref_bytes = {u: ref.user(u) for u in sample}
    checks = {}
    for name in configs:
        for _ in range(args.warmup):
            call(name)
        if name != "one_context":
            _, iv = call(name)
            checks[name] = dict(lengths_equal=bool((iv.len == ref_len).all()),
                                sampled_users_equal=all(iv.user(u) == ref_bytes[u] for u in sample),
                                total_bytes=iv.total_bytes, n_deliveries=iv.n_deliveries)
            assert checks[name]["lengths_equal"] and checks[name]["sampled_users_equal"], name
            assert iv.total_bytes == ref.total_bytes and iv.n_deliveries == ref.n_deliveries, name
    del ref

    wall = {name: [] for name in configs}
    for _ in range(args.reps):                       # the configurations in turn, round after round
        for name in configs:
            wall[name].append(call(name)[0])

    timing = {}
    for name, c in configs.items():
        c.set_profiling(True)
        call(name)
        if name == "one_context":
            tms = [c.timing()]
        else:
            tms = [c.timing(s) for s in range(c.n_shards)]
        timing[name] = [dict(h2d_ms=round(t.h2d_ms, 3), d2h_ms=round(t.d2h_ms, 3), total_ms=round(t.total_ms, 3),
                             plan_ms=round(t.plan_ms, 3), render_ms=round(t.render_ms, 3)) for t in tms]
        c.set_profiling(False)

    out = dict(
        probe="multi_speech_probe",
        cards=card_info(), n_devices=n_dev,
        workload=dict(lines=args.msgs, users=N_USERS, rooms=n_rooms, swear_words=N_SWEAR, ban_swearing=True,
                      shouts=int((verb == api.SPEECH_SHOUT).sum()), shout_share=float((verb == api.SPEECH_SHOUT).mean()),
                      h2d_bytes_per_shard=h2d_bytes, stream_bytes=int(ref_len.sum()), deliveries=int(ref_deliv)),
        wall_ms={k: dict(median=round(float(np.median(v)), 3), min=round(float(np.min(v)), 3), max=round(float(np.max(v)), 3),
                         all=[round(x, 3) for x in v]) for k, v in wall.items()},
        timing=timing, checks=checks,
        note="wall: host clock around one call (results on the host when it returns), pinned inputs; timing: nutsb_timing "
             "of each shard in one more call with profiling on (total_ms: the write pipeline's kernels, from the end of "
             "the composition to the last kernel)")
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(json.dumps(dict(cards=out["cards"], workload=out["workload"], wall_ms={k: v["median"] for k, v in out["wall_ms"].items()})))
    for c in configs.values():
        c.close()


if __name__ == "__main__":
    main()
