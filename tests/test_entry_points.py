"""The write entry points side by side.

  * one seeded batch through every host-buffer entry point (nutsb_write_batch, _iov, _keep, the queue's
    flush / flush_iov, nutsb_speech_batch, _iov): the same bytes per user whatever the result form, the
    nutsb_timing counters bench.py reads, and h2d_ms / d2h_ms written by every call that copies;
  * the device-composed calls refuse a population with clones or remote users (their relays are made only
    by the queue's host-side expansion) instead of delivering streams without them.
On the SIMT emulator here, on the GPU with `-m gpu`.
"""
import ctypes as C
import random

import numpy as np
import pytest

import oracle_lib as O
from nuts333_b200 import api

U, NR = 40, 4
COUNTERS = ("launches", "fanout_launches", "slab_bytes", "fanout_bytes_in", "fanout_bytes_out", "render_bytes_in")

# (launches, fanout_launches, slab_bytes, fanout_bytes_in, fanout_bytes_out, render_bytes_in) of each call, minted
# by running this file's generator on the emulator at commit 9bfcc87, before the write entry points shared one path.
# "plain": colour on / off listeners only (gather lists skip the fan-out); "filtered": ignall users and a write_level op.
MINTED = {
    "plain": {
        "write_batch": (25, 1, 19130, 19130, 86557, 8585), "write_batch_iov": (24, 0, 19130, 0, 0, 8585),
        "write_batch_keep": (25, 1, 19130, 19130, 86557, 8585),
        "flush": (25, 1, 19130, 19130, 86557, 8585), "flush_iov": (24, 0, 19130, 0, 0, 8585),
        "speech_batch": (25, 1, 62577, 62577, 308212, 28982), "speech_batch_iov": (24, 0, 62577, 0, 0, 28982),
    },
    "filtered": {
        "write_batch": (36, 1, 17831, 17831, 73405, 7943), "write_batch_iov": (36, 1, 17831, 17831, 73405, 7943),
        "write_batch_keep": (36, 1, 17831, 17831, 73405, 7943),
        "flush": (36, 1, 17831, 17831, 73405, 7943), "flush_iov": (36, 1, 17831, 17831, 73405, 7943),
        "speech_batch": (36, 1, 59449, 59449, 263241, 27085), "speech_batch_iov": (36, 1, 59449, 59449, 263241, 27085),
    },
}


def population(seed, filtered):
    rng = random.Random(seed)
    room = np.array([rng.randint(0, NR - 1) for _ in range(U)], np.int32)
    flags = np.array([rng.choice([0, api.UF_COLOUR]) for _ in range(U)], np.uint8)
    if filtered:
        for u in rng.sample(range(U), 6):
            flags[u] |= api.UF_IGNALL
    level = np.array([rng.randint(0, 4) for _ in range(U)], np.uint8)
    names = [("U" + "".join(rng.choice("abcdefgh") for _ in range(rng.randint(2, 8)))).encode() for _ in range(U)]
    return dict(room=room, flags=flags, level=level, names=names)


def write_ops(seed, filtered, n=300):
    rng = random.Random(seed)
    words = ["hello", "~FRred", "~OLbold~RS", "what", "ok", "a/~b", "line", "~", "x" * 30]
    texts, kind, target, exc = [], [], [], []
    for i in range(n):
        texts.append((" ".join(rng.choice(words) for _ in range(rng.randint(1, 6))) + "\n").encode())
        k = 2 if filtered and i == n // 2 else rng.choice([0, 1, 1, 1])
        kind.append(k)
        if k == 0:
            target.append(rng.randint(0, U - 1)); exc.append(-1)
        elif k == 1:
            target.append(rng.choice([-1] + list(range(NR)) * 4)); exc.append(rng.randint(-1, U - 1))
        else:
            target.append(2); exc.append(-1)
    text, off = O.pack(texts)
    return dict(text=text, off=off, kind=np.array(kind, np.uint8), target=np.array(target, np.int32),
                except_user=np.array(exc, np.int32), flags=np.zeros(n, np.uint8)), texts


def speech_lines(seed, filtered, n=200):
    rng = random.Random(seed)
    verbs = [0, 1, 2, 3, 4, 5] if filtered else [0, 1, 2, 3, 5]        # echo makes a write_level op
    words = ["hello", "there", "~FRred", "~OLbold~RS", "what", "ok", "x" * 20, "/~FG"]
    bodies = [(rng.choice(["", ";", "#"]) + " ".join(rng.choice(words) for _ in range(rng.randint(1, 6)))
               + rng.choice(["", "?", "!"])).encode() for _ in range(n)]
    verb = np.array([rng.choice(verbs) for _ in range(n)], np.uint8)
    speaker = np.array([rng.randint(0, U - 1) for _ in range(n)], np.int32)
    bt, bo = O.pack(bodies)
    return verb, speaker, bt, bo, bodies


def _setup(ctx, pop):
    ctx.set_swear_words(["fuck", "shit", "cunt", "*"])
    ctx.set_users(pop["room"], pop["flags"], pop["level"], NR)
    ctx.set_user_names(pop["names"], np.zeros(U, np.uint8))


def _queue(t, ops, texts):
    for i, s in enumerate(texts):
        k, tg, ex = int(ops["kind"][i]), int(ops["target"][i]), int(ops["except_user"][i])
        if k == 0:
            t.write_user(tg, s)
        elif k == 1:
            t.write_room_except(None if tg < 0 else tg, s, None if ex < 0 else ex)
        else:
            t.write_level(tg, False, s, None if ex < 0 else ex)


def _keep(ctx, ops):
    keep = []
    o = ctx._ops_struct(ops, keep)
    st = api._Streams()
    ctx._ck(ctx.lib.nutsb_write_batch_keep(ctx._h, C.byref(o), C.byref(st)))
    return st


def run_forms(ctx, seed, filtered):
    """-> {call: (counters, h2d_ms, d2h_ms)}; asserts that every result form gives the same bytes per user"""
    pop = population(seed, filtered)
    _setup(ctx, pop)
    ctx.set_profiling(True)
    ops, texts = write_ops(seed + 1, filtered)
    verb, speaker, bt, bo, bodies = speech_lines(seed + 2, filtered)
    t = api.Talker(ctx)
    res = {}

    def call(name, fn):
        ctx.write_batch_dev(0, 0, 0, 0, 0, 0, 0)          # a device-tier call first: no copies of its own
        r = fn()
        tm = ctx.timing()
        res[name] = (tuple(int(getattr(tm, f)) for f in COUNTERS), float(tm.h2d_ms), float(tm.d2h_ms))
        if name == "write_batch_keep":
            return r
        # the bytes now: gather lists point into the context's pinned buffers, which the next call reuses
        return r.off.copy(), int(r.n_deliveries), [r.user(u) for u in range(U)]

    st = call("write_batch", lambda: ctx.write_batch(ops))
    dg = ctx.stream_digests()
    forms = [call("write_batch_iov", lambda: ctx.write_batch_iov(ops))]
    kp = call("write_batch_keep", lambda: _keep(ctx, ops))
    assert kp.on_device == 1 and kp.total_bytes == sum(map(len, st[2])) and kp.n_deliveries == st[1]
    assert (ctx.stream_digests() == dg).all()
    _queue(t, ops, texts)
    forms.append(call("flush", t.flush))
    _queue(t, ops, texts)
    forms.append(call("flush_iov", t.flush_iov))
    for off, nd, users in forms:
        assert (off == st[0]).all() and nd == st[1] and users == st[2]

    sp = call("speech_batch", lambda: ctx.speech_batch(verb, speaker, bt, bo))
    si = call("speech_batch_iov", lambda: ctx.speech_batch_iov(verb, speaker, bt, bo))
    fn = [t.say, t.shout, t.emote, t.semote, t.echo, t.bcast]
    for v, s, b in zip(verb, speaker, bodies):
        fn[int(v)](int(s), b)
    sq = t.flush()
    assert sp[0][-1] > 0
    for off, nd, users in (si, (sq.off, sq.n_deliveries, [sq.user(u) for u in range(U)])):
        assert (off == sp[0]).all() and nd == sp[1] and users == sp[2]
    ctx.set_profiling(False)
    return res


def _check_forms(ctx, overlap=False):
    """overlap=False: one stream, the path the literals were minted on (the emulator has no side stream).
    overlap=True (a device with the side stream): k_direct shares the fan-out's launch (k_fanout_direct), one
    launch less wherever there is a fan-out; every other counter is the same."""
    ctx.set_overlap(overlap)
    try:
        for seed, case in ((71, "plain"), (72, "filtered")):
            res = run_forms(ctx, seed, case == "filtered")
            want = {k: ((v[0] - v[1],) + v[1:] if overlap else v) for k, v in MINTED[case].items()}
            assert {k: v[0] for k, v in res.items()} == want, (case, overlap)
            for name, (_, h2d, d2h) in res.items():
                assert h2d > 0, (case, name)
                assert (d2h == 0) if name == "write_batch_keep" else (d2h > 0), (case, name)
    finally:
        ctx.set_overlap(True)


def _clone_population(ctx):
    ctx.set_users(np.zeros(3, np.int32), np.array([0, 0, api.UF_CLONE], np.uint8), np.ones(3, np.uint8), 1)
    ctx.set_user_names([b"alice", b"bob", b"bob"], np.zeros(3, np.uint8))
    ctx.set_clones(np.array([-1, -1, 1], np.int32), np.array([0, 0, 2], np.uint8))


def _remote_population(ctx):
    # user 2 lives on another talker, reached through the link pseudo-user 3 (in no room)
    ctx.set_users(np.array([0, 0, 0, -1], np.int32), np.array([0, 0, api.UF_REMOTE, 0], np.uint8), np.ones(4, np.uint8), 1)
    ctx.set_user_names([b"alice", b"bob", b"carol", b"link"], np.zeros(4, np.uint8))
    ctx.set_remotes(np.array([-1, -1, 3, -1], np.int32), np.zeros(4, np.uint8))


def _check_refusal(ctx):
    ctx.set_swear_words(["fuck", "shit", "cunt", "*"])
    bt, bo = O.pack([b"hello"])
    verb, spk = np.zeros(1, np.uint8), np.zeros(1, np.int32)
    for make in (_clone_population, _remote_population):
        make(ctx)
        calls = (lambda: ctx.speech_batch(verb, spk, bt, bo),
                 lambda: ctx.speech_batch_iov(verb, spk, bt, bo),
                 lambda: ctx._ck(ctx.lib.nutsb_speech_batch_dev(ctx._h, 0, None, None, None, None, C.byref(api._Streams()))))
        for fn in calls:
            with pytest.raises(api.NutsbError) as e:
                fn()
            assert e.value.code == api.E_UNSUPPORTED, make.__name__
    # the context goes on with a plain population
    ctx.set_users(np.zeros(3, np.int32), np.zeros(3, np.uint8), np.ones(3, np.uint8), 1)
    ctx.set_user_names([b"alice", b"bob", b"carol"], np.zeros(3, np.uint8))
    st = ctx.speech_batch(verb, spk, bt, bo)
    assert st.user(0) == b"You say: hello\n\r" and st.user(1) == st.user(2) == b"alice says: hello\n\r"
    assert ctx.speech_batch_iov(verb, spk, bt, bo).user(1) == st.user(1)


def test_result_forms_on_emulator(sim_lib):
    ctx = api.Context(0, sim_lib)
    _check_forms(ctx)
    ctx.close()


def test_speech_refuses_relays_on_emulator(sim_lib):
    ctx = api.Context(0, sim_lib)
    _check_refusal(ctx)
    ctx.close()


@pytest.mark.gpu
def test_result_forms_on_gpu(gpu_ctx):
    _check_forms(gpu_ctx, overlap=False)
    _check_forms(gpu_ctx, overlap=True)


@pytest.mark.gpu
def test_speech_refuses_relays_on_gpu(gpu_ctx):
    _check_refusal(gpu_ctx)
