"""Speech batches that record (nutsb_set_speech_record): say / emote / echo lines sent through nutsb_speech_batch,
nutsb_speech_batch_iov and nutsb_speech_batch_dev go into the rooms' review buffers as record() (c:2062) would put
them, in batch order.

  * parity through review: the batch's streams followed by what a review of every room queues == the oracle port's
    streams for the same lines followed by those reviews (the port's record / review are pinned to the reference's
    own functions by test_review.py);
  * ring state: every room's rows and head == those of a context fed the same lines through the queue tier, also
    from a non-zero starting head;
  * recording off, validation errors and record() calls pending in the queue leave the buffers alone;
  * nutsb_multi: 1 / 2 / 3 shards (2 and 4 on one GPU, every device on a box with several), buffers that follow
    their rooms across a re-plan, rank mode refused;
  * a large batch on the GPU against a numpy restatement of "the last 15 per room".
The emulator runs everything but the device-pointer call and the large case; `-m gpu` runs them on the B200.
"""
import ctypes as C
import random

import numpy as np
import pytest

import oracle_lib as O
from nuts333_b200 import api

STOCK = ["fuck", "shit", "cunt", "*"]
REVIEW = 6
ROW = api.REVIEW_LEN + 2
# records per room the script aims at: none, one, one short of the ring, the ring, one over, three rings and more
TARGET = [0, 1, 14, 15, 16, 50]


def make_script(seed, per_room=2):
    """Users in len(TARGET) rooms (and some in none; invisible and muzzled ones among them), lines of all six verbs:
    room r gets about TARGET[r] recorded lines from its own speakers; the other lines record nothing (shout, semote,
    bcast, muzzled or roomless speakers) or swear, which records only with ban_swearing off."""
    rng = random.Random(seed)
    NR = len(TARGET)
    room, sflags = [], []
    for r in range(NR):
        for i in range(per_room + 2):
            room.append(r)
            sflags.append(0 if i == 0 else rng.choice([0, 0, 1, 2]))       # (user 0 of a room speaks freely)
    for _ in range(4):
        room.append(-1); sflags.append(rng.choice([0, 1]))
    U = len(room)
    room = np.array(room, np.int32)
    sflags = np.array(sflags, np.uint8)
    users = dict(room=room, flags=np.array([rng.choice([0, 1]) for _ in range(U)], np.uint8),
                 level=np.array([rng.randint(0, 4) for _ in range(U)], np.uint8))
    names = [("U%d" % u + "".join(rng.choice("abcdefghij") for _ in range(rng.randint(0, 8)))).encode() for u in range(U)]
    words = ["hello", "there", "~FRred", "~OLbold~RS", "what", "ok", "x" * 60, "~", "/~FG", "y" * 97]

    def body():
        b = " ".join(rng.choice(words) for _ in range(rng.randint(1, 7)))
        if rng.random() < 0.15: b = ";" + b
        if rng.random() < 0.3: b += rng.choice("?!")
        return b.encode()

    speakers_of = {r: [u for u in range(U) if room[u] == r and not (sflags[u] & 2)] for r in range(NR)}
    lines = []
    for r, t in enumerate(TARGET):
        for _ in range(t):
            lines.append((rng.choice([0, 2, 4]), rng.choice(speakers_of[r]), body()))
    for _ in range(40):
        k = rng.random()
        if k < 0.4:
            lines.append((rng.choice([1, 3, 5]), rng.randrange(U), body()))
        elif k < 0.7:                        # muzzled or roomless speakers: nothing to record
            u = rng.choice([u for u in range(U) if room[u] < 0 or sflags[u] & 2])
            lines.append((rng.randrange(6), u, body()))
        else:                                # swearing in a room that already speaks (room 0 stays silent)
            r = rng.randrange(1, NR)
            lines.append((rng.choice([0, 2, 4]), rng.choice(speakers_of[r]), b"oh shit " + body()))
    lines.append((0, speakers_of[5][0], b"z" * 250))          # cut at REVIEW_LEN
    lines.append((2, speakers_of[5][0], b";" + b"w" * 230))
    rng.shuffle(lines)
    verb = np.array([l[0] for l in lines], np.uint8)
    spk = np.array([l[1] for l in lines], np.int32)
    bodies = [l[2] for l in lines]
    bt, bo = O.pack(bodies)
    reviewers = [speakers_of[r][0] for r in range(NR)]
    return dict(users=users, n_rooms=NR, names=names, sflags=sflags, verb=verb, speaker=spk, bodies=bodies, bt=bt, bo=bo,
                reviewers=reviewers)


def setup(ctx, c, ban, record=True):
    ctx.set_swear_words(STOCK)
    ctx.set_users(c["users"]["room"], c["users"]["flags"], c["users"]["level"], c["n_rooms"])
    ctx.set_user_names(c["names"], c["sflags"])
    ctx.set_ban_swearing(ban)
    ctx.set_speech_record(record)


def fresh(lib, c, ban, record=True):
    ctx = api.Context(0, lib)
    setup(ctx, c, ban, record)
    return ctx


def port_with_reviews(port, c, ban):
    """the port's streams for the script followed by one review of every room"""
    NR = c["n_rooms"]
    verb = np.concatenate([c["verb"], np.full(NR, REVIEW, np.uint8)])
    spk = np.concatenate([c["speaker"], np.array(c["reviewers"], np.int32)])
    bt, bo = O.pack(list(c["bodies"]) + [b""] * NR)
    nt, no = O.pack(c["names"])
    ops = port.speech_ops(verb, spk, bt, bo, nt, no, c["sflags"], c["users"]["room"], ban, STOCK)
    off, data, _ = port.write_batch(ops, c["users"])
    return [data[int(off[u]):int(off[u + 1])].tobytes() for u in range(len(off) - 1)]


def review_all(ctx, c):
    t = api.Talker(ctx)
    for r, u in enumerate(c["reviewers"]):
        t.review(u, r)
    return t.flush()


def queue_fed(lib, c, ban, seed_records=()):
    """a context fed the script through the queue tier (records applied at the flush)"""
    q = fresh(lib, c, ban, record=False)
    t = api.Talker(q)
    for r, s in seed_records:
        t.record(r, s)
    t.flush()
    fn = [t.say, t.shout, t.emote, t.semote, t.echo, t.bcast]
    for v, s, b in zip(c["verb"], c["speaker"], c["bodies"]):
        fn[int(v)](int(s), b)
    t.flush()
    return q


def buffers(ctx, n_rooms):
    return [ctx.review_buffer(r) for r in range(n_rooms)]


def record_row(text):
    """record(): strncpy(REVIEW_LEN) -- cut at an embedded NUL, NUL-padded -- then '\\n' and NUL"""
    return text[:api.REVIEW_LEN].split(b"\0")[0].ljust(api.REVIEW_LEN, b"\0") + b"\n\0"


def _check_parity(lib, port, seed, forms):
    for ban in (True, False):
        c = make_script(seed)
        want = port_with_reviews(port, c, ban)
        q = queue_fed(lib, c, ban)
        for form in forms:
            ctx = fresh(lib, c, ban)
            args = (c["verb"], c["speaker"], c["bt"], c["bo"])
            st = ctx.speech_batch(*args) if form == "host" else ctx.speech_batch_iov(*args).streams()
            assert buffers(ctx, c["n_rooms"]) == buffers(q, c["n_rooms"]), (form, ban)
            rv = review_all(ctx, c)
            for u in range(len(want)):
                assert st.user(u) + rv.user(u) == want[u], (form, ban, u)
            ctx.close()
        q.close()


def _check_start_head(lib, seed):
    """earlier record() calls, flushed: the batch's records go in after them"""
    c = make_script(seed)
    seeds = [(r, b"seed %d-%d" % (r, i)) for r in range(c["n_rooms"]) for i in range(r * 3)] + [(5, b"q" * 230)]
    q = queue_fed(lib, c, True, seeds)
    ctx = fresh(lib, c, True)
    t = api.Talker(ctx)
    for r, s in seeds:
        t.record(r, s)
    t.flush()
    heads = [ctx.review_buffer(r)[1] for r in range(c["n_rooms"])]
    assert any(h != 0 for h in heads)
    ctx.speech_batch_iov(c["verb"], c["speaker"], c["bt"], c["bo"])
    assert buffers(ctx, c["n_rooms"]) == buffers(q, c["n_rooms"])
    ctx.close(); q.close()


def _check_left_alone(lib, port):
    c = make_script(31)
    NR = c["n_rooms"]
    args = (c["verb"], c["speaker"], c["bt"], c["bo"])
    ctx = fresh(lib, c, True, record=False)
    t = api.Talker(ctx)
    t.record(2, b"before")
    t.flush()
    before = buffers(ctx, NR)
    # recording off (the default)
    ctx.speech_batch(*args)
    ctx.speech_batch_iov(*args)
    assert buffers(ctx, NR) == before
    ctx.set_speech_record(True)
    # a device status error: offsets that are not monotone inside the batch, a speaker out of range
    bad = c["bo"].copy(); bad[3], bad[4] = bad[4], bad[3]
    with pytest.raises(api.NutsbError) as e:
        ctx.speech_batch(c["verb"], c["speaker"], c["bt"], bad)
    assert e.value.code == api.E_INVAL
    spk = c["speaker"].copy(); spk[-1] = len(c["names"])
    with pytest.raises(api.NutsbError) as e:
        ctx.speech_batch_iov(c["verb"], spk, c["bt"], c["bo"])
    assert e.value.code == api.E_RANGE
    assert buffers(ctx, NR) == before
    # record() pending in the queue: flush first
    t.record(1, b"pending")
    with pytest.raises(api.NutsbError) as e:
        ctx.speech_batch(*args)
    assert e.value.code == api.E_STATE
    assert buffers(ctx, NR) == before
    t.flush()
    ctx.speech_batch(*args)
    q = queue_fed(lib, c, True, [(2, b"before"), (1, b"pending")])
    assert buffers(ctx, NR) == buffers(q, NR)
    ctx.close(); q.close()


def _check_nul_and_order(lib):
    """strncpy stops at an embedded NUL; the ring keeps the last 15 in batch order"""
    users = dict(room=np.zeros(2, np.int32), flags=np.zeros(2, np.uint8), level=np.ones(2, np.uint8))
    bodies = [b"ab\0cd", b"x" * 199, b"y" * 200] + [b"line %d" % i for i in range(20)]
    verb = np.array([4] + [0] * (len(bodies) - 1), np.uint8)
    c = dict(users=users, n_rooms=1, names=[b"Ann", b"Bo"], sflags=np.zeros(2, np.uint8))
    bt, bo = O.pack(bodies)
    ctx = fresh(lib, c, False)
    ctx.speech_batch(verb[:3], np.zeros(3, np.int32), bt, bo[:4])
    rows, line = ctx.review_buffer(0)
    assert line == 3
    assert rows[0] == record_row(b"- ab") and rows[1] == record_row(b"Ann says: " + b"x" * 199 + b"\n")
    assert rows[2] == record_row(b"Ann says: " + b"y" * 200) and rows[3] == b"\0" * ROW
    spk = np.array([i % 2 for i in range(len(bodies))], np.int32)
    ctx.speech_batch_iov(verb, spk, bt, bo)
    rows, line = ctx.review_buffer(0)
    assert line == (3 + len(bodies)) % 15
    texts = [b"- ab\0cd\n"] + [[b"Ann", b"Bo"][i % 2] + b" says: " + b + b"\n" for i, b in enumerate(bodies) if i]
    for i, tx in enumerate(texts[-15:]):
        assert rows[(line + i) % 15] == record_row(tx), i
    with pytest.raises(api.NutsbError) as e:
        ctx.review_buffer(1)
    assert e.value.code == api.E_RANGE
    ctx.close()


def _check_multi(lib, devices):
    for ban in (True, False):
        c = make_script(41 + len(devices))
        NR = c["n_rooms"]
        args = (c["verb"], c["speaker"], c["bt"], c["bo"])
        one = fresh(lib, c, ban)
        one.speech_batch(*args)
        m = api.MultiContext(devices, lib)
        m.set_swear_words(STOCK)
        m.set_user_names(c["names"], c["sflags"])
        m.set_users(c["users"]["room"], c["users"]["flags"], c["users"]["level"], NR)
        m.set_ban_swearing(ban)
        m.set_speech_record(True)
        m.speech_batch(*args)
        assert [m.review_buffer(r) for r in range(NR)] == buffers(one, NR), (devices, ban)
        # a re-plan that moves rooms: every buffer follows its room
        rs0 = m.plan()[0].copy()
        m.set_users(c["users"]["room"], c["users"]["flags"], c["users"]["level"], NR, room_weight=np.arange(1, NR + 1, dtype=np.uint64) ** 3)
        one.set_users(c["users"]["room"], c["users"]["flags"], c["users"]["level"], NR)
        if len(devices) > 1:
            assert (m.plan()[0] != rs0).any()
        assert [m.review_buffer(r) for r in range(NR)] == buffers(one, NR), (devices, ban)
        m.speech_batch_iov(*args)
        one.speech_batch_iov(*args)
        assert [m.review_buffer(r) for r in range(NR)] == buffers(one, NR), (devices, ban)
        # a shard's refusal (record() pending on its queue) leaves every shard's buffers alone
        before = buffers(one, NR)
        api.Talker(m.ctx(0)).record(0, b"pending")
        with pytest.raises(api.NutsbError) as e:
            m.speech_batch(*args)
        assert e.value.code == api.E_STATE
        assert [m.review_buffer(r) for r in range(NR)] == before
        m.close(); one.close()


def _check_refused_replan(lib, devices):
    """a re-plan refused for a record() pending on a shard changes nothing; after the flush, the retry carries every
    room's buffer (the pending record included) to its new place"""
    c = make_script(51)
    NR = c["n_rooms"]
    users = c["users"]
    args = (c["verb"], c["speaker"], c["bt"], c["bo"])
    one = fresh(lib, c, True)
    one.speech_batch(*args)
    m = api.MultiContext(devices, lib)
    m.set_swear_words(STOCK)
    m.set_user_names(c["names"], c["sflags"])
    m.set_users(users["room"], users["flags"], users["level"], NR)
    m.set_ban_swearing(True)
    m.set_speech_record(True)
    m.speech_batch(*args)
    rs = m.plan()[0].copy()
    g = int(np.nonzero(rs == 1)[0][0])                       # shard 1's local room 0 (local rooms keep the global order)
    t = api.Talker(m.ctx(1))
    t.record(0, b"pending on shard 1")
    weights = np.arange(1, NR + 1, dtype=np.uint64) ** 3
    with pytest.raises(api.NutsbError) as e:
        m.set_users(users["room"], users["flags"], users["level"], NR, room_weight=weights)
    assert e.value.code == api.E_STATE
    assert (m.plan()[0] == rs).all()
    t.flush()
    t1 = api.Talker(one)
    t1.record(g, b"pending on shard 1")
    t1.flush()
    assert [m.review_buffer(r) for r in range(NR)] == buffers(one, NR)
    m.set_users(users["room"], users["flags"], users["level"], NR, room_weight=weights)
    assert (m.plan()[0] != rs).any()
    assert [m.review_buffer(r) for r in range(NR)] == buffers(one, NR)
    m.close(); one.close()


def test_refused_replan_keeps_the_buffers_on_emulator(sim_lib):
    _check_refused_replan(sim_lib, [0, 0])


def test_parity_through_review_on_emulator(sim_lib, port):
    _check_parity(sim_lib, port, 21, ("host", "iov"))


def test_ring_state_from_a_later_head_on_emulator(sim_lib):
    _check_start_head(sim_lib, 22)


def test_off_and_failures_leave_the_buffers_alone_on_emulator(sim_lib, port):
    _check_left_alone(sim_lib, port)


def test_embedded_nul_and_batch_order_on_emulator(sim_lib):
    _check_nul_and_order(sim_lib)


@pytest.mark.parametrize("devices", [[0], [0, 0], [0, 0, 0]])
def test_multi_on_emulator(sim_lib, devices):
    _check_multi(sim_lib, devices)


def test_rank_mode_refuses(sim_lib):
    m = api.MultiContext(lib=sim_lib, rank=(2, 0, 0))
    with pytest.raises(api.NutsbError) as e:
        m.set_speech_record(True)
    assert e.value.code == api.E_UNSUPPORTED
    m.set_speech_record(False)
    m.close()


# ---- on the GPU -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu_lib():
    from nuts333_b200 import build
    build.build()
    return api.load_library()


@pytest.mark.gpu
def test_parity_through_review_on_gpu(gpu_lib, port):
    _check_parity(gpu_lib, port, 23, ("host", "iov"))
    _check_start_head(gpu_lib, 24)
    _check_left_alone(gpu_lib, port)
    _check_nul_and_order(gpu_lib)


@pytest.mark.gpu
def test_device_pointer_call_on_gpu(gpu_lib, port):
    """nutsb_speech_batch_dev: the same streams (digests) as the host call, and the records applied on return"""
    import torch
    for ban in (True, False):
        c = make_script(25)
        want = port_with_reviews(port, c, ban)
        q = queue_fed(gpu_lib, c, ban)
        ctx = fresh(gpu_lib, c, ban, record=False)
        st = ctx.speech_batch(c["verb"], c["speaker"], c["bt"], c["bo"])
        dg = ctx.stream_digests()
        ctx.set_speech_record(True)
        d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (c["verb"], c["speaker"], c["bt"], c["bo"].view(np.int64))]
        out = api._Streams()
        ctx._ck(ctx.lib.nutsb_speech_batch_dev(ctx._h, len(c["verb"]), *[t.data_ptr() for t in d], C.byref(out)))
        assert out.on_device == 1
        assert buffers(ctx, c["n_rooms"]) == buffers(q, c["n_rooms"])
        assert (ctx.stream_digests() == dg).all()
        rv = review_all(ctx, c)
        for u in range(len(want)):
            assert st.user(u) + rv.user(u) == want[u], (ban, u)
        ctx.close(); q.close()


@pytest.mark.gpu
def test_multi_on_gpu(gpu_lib):
    import torch
    for devices in ([0, 0], [0, 0, 0, 0]) + ((list(range(torch.cuda.device_count())),) if torch.cuda.device_count() > 1 else ()):
        _check_multi(gpu_lib, devices)
    _check_refused_replan(gpu_lib, [0, 0])
    m = api.MultiContext(lib=gpu_lib, rank=(2, 1, 0))
    with pytest.raises(api.NutsbError) as e:
        m.set_speech_record(True)
    assert e.value.code == api.E_UNSUPPORTED
    m.close()


def restate_last15(verb, spk, bodies, room, names, sflags, n_rooms, refused):
    """record()'s rows and heads of every room after the lines, from an empty start: the composed room line of
    say / emote / echo (speaker in a room, not muzzled, not refused), the last 15 of each room in batch order"""
    per = [[] for _ in range(n_rooms)]
    for m in range(len(verb)):
        v, u = int(verb[m]), int(spk[m])
        if v not in (0, 2, 4) or room[u] < 0 or sflags[u] & 2 or refused[m]:
            continue
        b = bodies[m]
        nm = b"A presence" if sflags[u] & 1 else names[u]
        if v == 0:
            t = {b"?": b" asks: ", b"!": b" exclaims: "}.get(b[-1:], b" says: ")
            text = nm + t + b + b"\n"
        elif v == 2:
            text = nm + (b[1:] if b[:1] == b";" else b" " + b) + b"\n"
        else:
            text = b"- " + b + b"\n"
        per[int(room[u])].append(text)
    out = []
    for r in range(n_rooms):
        rows = [b"\0" * ROW] * 15
        for i, text in enumerate(per[r][-15:]):
            rows[(len(per[r]) - min(len(per[r]), 15) + i) % 15] = record_row(text)
        out.append((rows, len(per[r]) % 15))
    return out


@pytest.mark.gpu
def test_large_batch_on_gpu(gpu_lib, port):
    """200k lines over 5k users in 50 rooms, ban_swearing on, against the numpy restatement"""
    rng = np.random.default_rng(7)
    U, NR, N = 5000, 50, 200_000
    room = rng.integers(-1, NR, U).astype(np.int32)
    room[:NR] = np.arange(NR)
    sflags = rng.choice(np.array([0, 0, 0, 1, 2], np.uint8), U)
    names = [b"user%d" % u for u in range(U)]
    words = [b"hello", b"there", b"shit", b"~FRred", b"ok?", b"x" * 90, b"yes!"]
    verb = rng.choice(np.array([0, 0, 0, 1, 2, 3, 4, 5], np.uint8), N)
    spk = rng.integers(0, U, N).astype(np.int32)
    bodies = [b" ".join(words[i] for i in rng.integers(0, len(words), rng.integers(1, 6))) for _ in range(N)]
    for m in rng.integers(0, N, N // 20):
        bodies[m] = b";" + bodies[m]
    bt, bo = O.pack(bodies)
    users = dict(room=room, flags=np.zeros(U, np.uint8), level=np.ones(U, np.uint8))
    c = dict(users=users, n_rooms=NR, names=names, sflags=sflags)
    ctx = fresh(gpu_lib, c, True)
    ctx.speech_batch_iov(verb, spk, bt, bo)
    refused = port.contains_swearing_batch(bt, bo, STOCK) != 0
    refused &= (verb == 0) | (verb == 2)                        # echo never asks
    want = restate_last15(verb, spk, bodies, room, names, sflags, NR, refused)
    assert buffers(ctx, NR) == want
    ctx.close()
