"""The host side's own bookkeeping, on the emulator:

  * closing a context gives back every buffer it allocated -- a bare one, one that has installed tables and run a
    write batch and a recording speech batch, the shards of a nutsb_multi and the lanes of a nutsb_pipe that did the
    same.  The emulator's device and pinned buffers are malloc'd, so a buffer left behind shows as heap growth;
  * the emulator library is rebuilt when any source of the product library changes.
"""
import ctypes as C
import gc
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from nuts333_b200 import api, synth

ROOT = Path(__file__).resolve().parent.parent
N_USERS, PER_ROOM, N_LINES = 24, 6, 40
# A bare context is cheap to make.  A busy one takes about a second on the emulator (its batches), so it gets fewer
# cycles: a buffer left behind costs at least the 512 bytes of slack every allocation carries, which a few show.
CYCLES = dict(bare=(20, 300), busy=(2, 8), multi=(2, 8), pipe=(2, 8))      # (warm-up, measured)


class _Mallinfo2(C.Structure):
    _fields_ = [(f, C.c_size_t) for f in ("arena", "ordblks", "smblks", "hblks", "hblkhd", "usmblks", "fsmblks",
                                          "uordblks", "fordblks", "keepcost")]


def _work():
    """A small population and batch that reach every kind of buffer a context keeps: a 64-word swear list, both ban
    files, user names, a gated write batch and a speech batch of all six verbs."""
    rng = np.random.default_rng(5)
    words = synth.swear_words(64)
    us, n_rooms = synth.users(N_USERS, PER_ROOM)
    un, uo = synth.names(N_USERS)
    names = [un[int(uo[u]):int(uo[u + 1])].tobytes() for u in range(N_USERS)]
    bt, bo = synth.bodies(N_LINES, words)
    ops, _, _ = synth.say_ops(N_LINES, N_USERS, PER_ROOM, bt, bo, gated=True)
    ops["verdict"] = rng.integers(0, 2, N_LINES).astype(np.uint8)
    speech = (rng.integers(0, 6, N_LINES).astype(np.uint8), rng.integers(0, N_USERS, N_LINES).astype(np.int32), bt, bo)
    return dict(words=words, users=us, n_rooms=n_rooms, names=names, sflags=np.zeros(N_USERS, np.uint8),
                siteban=synth.ban_file(0, 50, 300, 300, False), userban=synth.ban_file(1, 50, 300, 300, True),
                ops=ops, speech=speech)


def _setup(h, w):
    """tables, names and population, through whichever handle (Context / MultiContext)"""
    us = w["users"]
    h.set_swear_words(w["words"])
    h.set_ban_files(w["siteban"], w["userban"])
    h.set_user_names(w["names"], w["sflags"])
    h.set_users(us["room"], us["flags"], us["level"], w["n_rooms"])
    h.set_speech_record(True)


def _cycle(lib, variant, w):
    """one create / use / close of the variant's handle"""
    if variant == "bare":
        api.Context(0, lib).close()
    elif variant == "busy":
        ctx = api.Context(0, lib)
        _setup(ctx, w)
        ctx.write_batch_iov(w["ops"])
        ctx.speech_batch(*w["speech"])
        ctx.close()
    elif variant == "multi":
        m = api.MultiContext([0, 0], lib)
        _setup(m, w)
        m.write_batch_iov(w["ops"])
        m.speech_batch(*w["speech"])
        m.close()
    else:
        us = w["users"]
        p = api.Pipe(0, 2, lib)
        p.set_swear_words(w["words"])
        p.set_user_names(w["names"], w["sflags"])
        p.set_users(us["room"], us["flags"], us["level"], w["n_rooms"])
        for lane in range(2):
            ctx = p.ctx(lane)
            ctx.set_ban_files(w["siteban"], w["userban"])
            ctx.set_speech_record(True)
        for submit, args in ((p.submit_write_iov, (w["ops"],)), (p.submit_speech_iov, w["speech"])):
            tickets = [submit(*args) for _ in range(2)]                 # one call on each lane
            for t in tickets:
                p.wait(t)
        p.close()


def measure(variant):
    """Run in the child process: prints the heap's growth per cycle, in bytes.  The heap in use is what glibc's
    malloc has handed out and not had back, all arenas and mmap'd blocks included."""
    from cpusim.build_sim import build_sim
    libc = C.CDLL(None)
    libc.mallinfo2.restype = _Mallinfo2

    def heap_in_use():
        gc.collect()
        m = libc.mallinfo2()
        return m.uordblks + m.hblkhd
    lib = api.bind(C.CDLL(str(build_sim())))
    w = _work()
    warmup, cycles = CYCLES[variant]
    for _ in range(warmup):
        _cycle(lib, variant, w)
    before = heap_in_use()
    for _ in range(cycles):
        _cycle(lib, variant, w)
    print((heap_in_use() - before) / cycles)


@pytest.fixture
def growth_per_cycle(sim_lib):
    """-> f(variant): the heap's growth per cycle, measured in a child process with glibc's per-thread cache off.
    mallinfo2 counts the chunks that cache holds as in use, and it fills over the first few dozen cycles: with it
    on, a few cycles cannot tell a leak from the cache filling.  (sim_lib: the library is built before the child
    needs it.)"""
    libc = C.CDLL(None)
    if not hasattr(libc, "mallinfo2"):
        pytest.skip("no mallinfo2 (glibc < 2.33)")

    def run(variant):
        tun = "glibc.malloc.tcache_count=0"
        env = dict(os.environ, GLIBC_TUNABLES=":".join(filter(None, (os.environ.get("GLIBC_TUNABLES"), tun))))
        code = (f"import sys; sys.path[:0] = {[str(ROOT), str(ROOT / 'tests')]!r}; "
                f"import test_host_lifetime as t; t.measure({variant!r})")
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-4000:]
        return float(r.stdout.split()[-1])
    return run


@pytest.mark.parametrize("variant", list(CYCLES))
def test_closing_frees_every_buffer(growth_per_cycle, variant):
    assert growth_per_cycle(variant) < 64


def test_emulator_rebuilds_on_every_product_source():
    from cpusim.build_sim import DEPS
    deps = {d.resolve() for d in DEPS}
    sources = sorted(p.resolve() for p in (ROOT / "nuts333_b200" / "csrc").iterdir() if p.suffix in (".cu", ".cuh"))
    assert sources and [p.name for p in sources if p not in deps] == []
