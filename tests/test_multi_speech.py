"""nutsb_multi speech batches: say / shout / emote / semote / echo / bcast lines composed on every shard (each shard is
given the whole batch and picks its lines on the device) == the oracle == the one-context speech batch, with streams
and with gather lists; and nutsb_multi_write_batch_iov == nutsb_multi_write_batch.  The populations hold what the
shard mode has to get right: speakers in no room (echo yields nothing anywhere), muzzled speakers (their refusal only
on their own shard), invisible speakers, shouts / semotes / broadcasts and echo's write_level from speakers who live on
another shard (gated on a swear verdict taken there too), recipients behind filters.  Shards on one device exercise
the same host logic as shards on several (the emulator here; with `-m gpu` 2 and 4 shards on cuda:0, and every device
when the box has two or more)."""
import random

import numpy as np
import pytest

import oracle_lib as O
from nuts333_b200 import api
from test_multi import make_case as make_write_case
from test_speech import STOCK, make_case as make_speech_case


def make_case(seed, U, NR, N, plain=False):
    """test_speech's population and lines, with some bodies emptied and a few swearing lines put in.  plain: every
    recipient a plain listener and no echo (no write_level): the gather lists point into the renderings' pools"""
    c = make_speech_case(seed, U, NR, N)
    if plain:
        c["users"]["flags"] &= 1
        c["verb"][c["verb"] == 4] = 1
    rng = random.Random(seed + 1000)
    bodies = list(c["bodies"])
    for m in range(N):
        r = rng.random()
        if r < 0.06:
            bodies[m] = b""
        elif r < 0.12:
            bodies[m] = rng.choice([b"oh shit", b"FUCK!", b";cunt?", b"#shit"])
    c["bodies"] = bodies
    c["bt"], c["bo"] = O.pack(bodies)
    return c


def _port(port, c, ban):
    nt, no = O.pack(c["names"])
    ops = port.speech_ops(c["verb"], c["speaker"], c["bt"], c["bo"], nt, no, c["sflags"], c["users"]["room"], ban, STOCK)
    return port.write_batch(ops, c["users"])


def _multi(lib, devices, c, ban, rank=None):
    m = api.MultiContext(devices, lib, rank=rank)
    m.set_swear_words(STOCK)
    m.set_user_names(c["names"], c["sflags"])                 # before the population: given to the shards with the plan
    m.set_users(c["users"]["room"], c["users"]["flags"], c["users"]["level"], c["n_rooms"])
    m.set_ban_swearing(ban)
    return m


def _one(ctx, c, ban):
    ctx.set_swear_words(STOCK)
    ctx.set_users(c["users"]["room"], c["users"]["flags"], c["users"]["level"], c["n_rooms"])
    ctx.set_user_names(c["names"], c["sflags"])
    ctx.set_ban_swearing(ban)


def _check_pieces_in_pools(m, iv, devices):
    _, ush, _ = m.plan()
    pools = {s: [(a, a + n) for a, n in m.shard_iov(s).pools if n] for s in range(len(devices))}
    for u in range(len(ush)):
        for a, n in iv.pieces(u):
            if n:
                assert any(lo <= int(a) and int(a) + int(n) <= hi for lo, hi in pools[int(ush[u])]), u


def _check_speech(lib, one, port, devices, seed, U, NR, N, plain=False):
    for ban in (True, False):
        c = make_case(seed, U, NR, N, plain)
        args = (c["verb"], c["speaker"], c["bt"], c["bo"])
        _one(one, c, ban)
        st = one.speech_batch(*args)
        want = [st.user(u) for u in range(U)]
        off, data, nd = _port(port, c, ban)
        assert all(want[u] == data[int(off[u]):int(off[u + 1])].tobytes() for u in range(U))
        assert st.n_deliveries == int(nd.sum())
        one_dg = one.stream_digests()
        m = _multi(lib, devices, c, ban)
        got, total, deliv = m.speech_batch(*args)
        for u in range(U):
            assert got[u] == want[u], (devices, ban, u)
        assert total == st.total_bytes and deliv == st.n_deliveries
        iv = m.speech_batch_iov(*args)
        assert iv.total_bytes == total and iv.n_deliveries == deliv
        assert (iv.len == np.diff(st.off)).all()
        for u in range(U):
            assert iv.user(u) == want[u], (devices, ban, u)
        _check_pieces_in_pools(m, iv, devices)
        _, total2, deliv2 = m.speech_batch(*args, keep=True)
        assert total2 == total and deliv2 == deliv
        assert (m.stream_digests() == one_dg).all()
        m.close()


def _check_write_iov(lib, devices, seed, U, NR, N):
    c = make_write_case(seed, U, NR, N)
    o, us = c["ops"], c["users"]
    m = api.MultiContext(devices, lib)
    m.set_users(us["room"], us["flags"], us["level"], NR)
    got, total, deliv = m.write_batch(o)
    iv = m.write_batch_iov(o)
    assert iv.total_bytes == total and iv.n_deliveries == deliv
    for u in range(U):
        assert iv.user(u) == got[u] and int(iv.len[u]) == len(got[u]), (devices, u)
    _check_pieces_in_pools(m, iv, devices)
    m.close()


def _check_errors(lib, devices):
    c = make_case(81, 20, 3, 40)
    args = (c["verb"], c["speaker"], c["bt"], c["bo"])
    m = api.MultiContext(devices, lib)
    m.set_users(c["users"]["room"], c["users"]["flags"], c["users"]["level"], c["n_rooms"])
    with pytest.raises(api.NutsbError) as e:                   # names not set
        m.speech_batch(*args)
    assert e.value.code == api.E_STATE
    m.set_user_names(c["names"], c["sflags"])
    want, total, deliv = m.speech_batch(*args)
    assert total > 0
    bad_spk = c["speaker"].copy(); bad_spk[7] = 20
    bad_verb = c["verb"].copy(); bad_verb[3] = 6
    for call in (m.speech_batch, m.speech_batch_iov):
        with pytest.raises(api.NutsbError) as e:
            call(c["verb"], bad_spk, c["bt"], c["bo"])
        assert e.value.code == api.E_RANGE
        assert m.speech_batch(*args) == (want, total, deliv)  # the handle runs the next batch correctly
        with pytest.raises(api.NutsbError) as e:
            call(bad_verb, c["speaker"], c["bt"], c["bo"])
        assert e.value.code == api.E_INVAL
        assert m.speech_batch(*args) == (want, total, deliv)
    # a new population the names do not match
    m.set_users(np.zeros(21, np.int32), np.zeros(21, np.uint8), np.ones(21, np.uint8), 1)
    with pytest.raises(api.NutsbError) as e:
        m.speech_batch(*args)
    assert e.value.code == api.E_STATE
    m.set_users(c["users"]["room"], c["users"]["flags"], c["users"]["level"], c["n_rooms"])
    assert m.speech_batch(*args) == (want, total, deliv)
    m.close()


def test_multi_speech_on_emulator(sim_lib, port):
    one = api.Context(0, sim_lib)
    _check_speech(sim_lib, one, port, [0], 71, 24, 3, 90)
    _check_speech(sim_lib, one, port, [0, 0], 72, 30, 4, 120)
    _check_speech(sim_lib, one, port, [0, 0, 0], 73, 36, 5, 150)
    _check_speech(sim_lib, one, port, [0, 0, 0], 82, 36, 5, 150, plain=True)
    one.close()


def test_multi_write_iov_on_emulator(sim_lib):
    _check_write_iov(sim_lib, [0, 0, 0], 74, 30, 5, 140)
    _check_write_iov(sim_lib, [0], 75, 12, 2, 60)


def test_multi_speech_errors_on_emulator(sim_lib):
    _check_errors(sim_lib, [0, 0])


def test_multi_speech_rank_view_on_emulator(sim_lib, port):
    """one process per GPU: each rank returns exactly its own users' streams; together the ranks cover the population once"""
    c = make_case(76, 30, 4, 120)
    off, data, nd = _port(port, c, True)
    args = (c["verb"], c["speaker"], c["bt"], c["bo"])
    seen, deliv_sum = np.zeros(30, np.int32), 0
    for rank in range(2):
        m = _multi(sim_lib, None, c, True, rank=(2, rank, 0))
        _, ush, _ = m.plan()
        got, _, deliv = m.speech_batch(*args)
        iv = m.speech_batch_iov(*args)
        deliv_sum += deliv
        for u in range(30):
            if ush[u] == rank:
                seen[u] += 1
                assert got[u] == iv.user(u) == data[int(off[u]):int(off[u + 1])].tobytes()
            else:
                assert got[u] == b"" and iv.count[u] == 0 and iv.len[u] == 0
        m.close()
    assert (seen == 1).all() and deliv_sum == int(nd.sum())


def _big_case(seed, U, NR, N):
    """N lines over U users in NR rooms: mostly say / emote, some shouts and echoes"""
    rng = np.random.default_rng(seed)
    room = rng.integers(0, NR, U).astype(np.int32)
    room[rng.random(U) < 0.02] = -1
    flags = rng.choice(np.array([0, 1, 1, 0, 4, 8, 5, 9, 2], np.uint8), U)
    level = rng.integers(0, 5, U).astype(np.uint8)
    names = [b"U%d" % u for u in range(U)]
    sflags = rng.choice(np.array([0, 0, 0, 0, 0, 0, 1, 2], np.uint8), U)
    verb = rng.choice(np.array([0] * 80 + [2] * 15 + [4] * 4 + [1], np.uint8), N)
    words = [b"hi", b"ok", b"shit", b"what?", b"fine!", b";wave", b"#x"]
    bodies = [words[i] for i in rng.integers(0, len(words), N)]
    bt, bo = O.pack(bodies)
    return dict(users=dict(room=room, flags=flags, level=level), n_rooms=NR, names=names, sflags=sflags,
                verb=verb, speaker=rng.integers(0, U, N).astype(np.int32), bt=bt, bo=bo)


def _check_big(lib, one, devices):
    """a batch whose route scan spans many blocks: per-user lengths, digests and 64 users' bytes against one context"""
    c = _big_case(91, 5000, 50, 200_000)
    args = (c["verb"], c["speaker"], c["bt"], c["bo"])
    _one(one, c, True)
    st = one.speech_batch(*args)
    one_dg = one.stream_digests()
    m = _multi(lib, devices, c, True)
    iv = m.speech_batch_iov(*args)
    assert iv.total_bytes == st.total_bytes and iv.n_deliveries == st.n_deliveries
    assert (iv.len == np.diff(st.off)).all()
    for u in range(0, 5000, 5000 // 64):
        assert iv.user(u) == st.user(u), u
    _, total, deliv = m.speech_batch(*args, keep=True)
    assert total == st.total_bytes and deliv == st.n_deliveries
    assert (m.stream_digests() == one_dg).all()
    m.close()


@pytest.mark.gpu
def test_multi_speech_on_gpu(gpu_ctx, port):
    lib = gpu_ctx.lib
    _check_speech(lib, gpu_ctx, port, [0, 0], 77, 400, 7, 3000)
    _check_speech(lib, gpu_ctx, port, [0, 0, 0, 0], 78, 1500, 40, 6000)
    _check_speech(lib, gpu_ctx, port, [0, 0], 83, 1500, 40, 6000, plain=True)
    _check_write_iov(lib, [0, 0, 0, 0], 79, 1500, 40, 6000)
    _check_errors(lib, [0, 0])
    _check_big(lib, gpu_ctx, [0, 0, 0, 0])
    import torch
    n = torch.cuda.device_count()
    if n >= 2:
        devs = list(range(min(n, 8)))
        _check_speech(lib, gpu_ctx, port, devs, 80, 3000, 64, 20000)
        _check_write_iov(lib, devs, 81, 3000, 64, 20000)
        _check_big(lib, gpu_ctx, devs)
