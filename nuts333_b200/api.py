"""Host-side mirror of the reference's write surface over the C-ABI (include/nutsb200.h).

`Context` is a thin ctypes binding of libnutsb200.so; `Talker` keeps the reference's
own names and ambient globals (nuts333.c:1291-1429, 2540, 330, 349; nuts333.h:201,293):

    t = Talker(ctx)
    t.force_listen = 1                      # h:293
    t.com_num = SHOUT                       # h:201
    t.write_room_except(room, text, user)   # c:1401
    streams = t.flush()                     # per-user socket bytes

Everything here is plumbing: the work happens in the CUDA kernels behind the C-ABI.
There is no CPU fallback -- constructing a Context without a usable GPU raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

OP_USER, OP_ROOM, OP_LEVEL = 0, 1, 2
OF_FORCE_LISTEN, OF_SHOUT, OF_ABOVE, OF_GATE_IF_SET, OF_PAGER, OF_PLAIN, OF_RAW = 1, 2, 4, 8, 16, 32, 64
UF_COLOUR, UF_LOGIN, UF_IGNALL, UF_IGNSHOUT, UF_CLONE, UF_REMOTE = 1, 2, 4, 8, 16, 32
MAX_TEXT = 2000

# com_num values that matter on the path (enum comvals, nuts333.h:181-183)
SAY, SHOUT, SEMOTE = 3, 4, 7
# speech verbs of the composer (nutsb200.h) and per-user speech flags
SPEECH_SAY, SPEECH_SHOUT, SPEECH_EMOTE, SPEECH_SEMOTE, SPEECH_ECHO, SPEECH_BCAST = range(6)
SF_INVIS, SF_MUZZLED = 1, 2
# user levels (nuts333.h: level_name[])
NEW, USER, WIZ, ARCH, GOD = 0, 1, 2, 3, 4

E_INVAL, E_NOMEM, E_CUDA, E_UNSUPPORTED, E_RANGE, E_STATE = -1, -2, -3, -4, -5, -6
REVIEW_LINES, REVIEW_LEN = 15, 200            # nuts333.h:37, :39 (NUTSB_REVIEW_LINES / NUTSB_REVIEW_LEN)

u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)
i32p = C.POINTER(C.c_int32)


class NutsbError(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        super().__init__(f"nutsb error {code}: {detail}")


class _Ops(C.Structure):
    _fields_ = [("n_ops", C.c_int64), ("text", C.c_void_p), ("text_off", C.c_void_p), ("kind", C.c_void_p),
                ("target", C.c_void_p), ("except_user", C.c_void_p), ("flags", C.c_void_p),
                ("gate", C.c_void_p), ("verdict", C.c_void_p)]


class _Streams(C.Structure):
    _fields_ = [("n_users", C.c_int64), ("total_bytes", C.c_uint64), ("n_deliveries", C.c_uint64),
                ("off", C.c_void_p), ("bytes", C.c_void_p), ("on_device", C.c_int32)]


class _IovStreams(C.Structure):
    _fields_ = [("n_users", C.c_int64), ("total_bytes", C.c_uint64), ("n_deliveries", C.c_uint64),
                ("off", C.c_void_p), ("first", C.c_void_p), ("count", C.c_void_p), ("iov", C.c_void_p),
                ("n_iov", C.c_uint64), ("pool", C.c_void_p), ("pool_bytes", C.c_uint64),
                ("pool2", C.c_void_p), ("pool2_bytes", C.c_uint64)]


class _MStreams(C.Structure):
    _fields_ = [("n_users", C.c_int64), ("total_bytes", C.c_uint64), ("n_deliveries", C.c_uint64),
                ("len", C.c_void_p), ("ptr", C.c_void_p), ("on_device", C.c_int32)]


class _MIovStreams(C.Structure):
    _fields_ = [("n_users", C.c_int64), ("total_bytes", C.c_uint64), ("n_deliveries", C.c_uint64),
                ("len", C.c_void_p), ("iov", C.c_void_p), ("count", C.c_void_p)]


class Timing(C.Structure):
    _fields_ = [("plan_ms", C.c_float), ("render_ms", C.c_float), ("fanout_ms", C.c_float), ("direct_ms", C.c_float),
                ("total_ms", C.c_float), ("h2d_ms", C.c_float), ("d2h_ms", C.c_float),
                ("fanout_bytes_in", C.c_uint64), ("fanout_bytes_out", C.c_uint64),
                ("render_bytes_in", C.c_uint64), ("slab_bytes", C.c_uint64),
                ("launches", C.c_uint32), ("fanout_launches", C.c_uint32)]


EXPORTS = [
    "nutsb_version", "nutsb_strerror", "nutsb_last_error", "nutsb_create", "nutsb_destroy",
    "nutsb_set_profiling", "nutsb_get_timing", "nutsb_set_overlap", "nutsb_set_stream", "nutsb_set_swear_words",
    "nutsb_set_ban_files", "nutsb_ban_edit", "nutsb_get_ban_file", "nutsb_set_users", "nutsb_set_users_remap", "nutsb_set_clones", "nutsb_set_remotes", "nutsb_set_room_names", "nutsb_write_batch", "nutsb_write_batch_dev", "nutsb_write_batch_iov",
    "nutsb_contains_swearing_batch", "nutsb_contains_swearing_batch_dev", "nutsb_site_banned_batch",
    "nutsb_site_banned_batch_dev", "nutsb_user_banned_batch", "nutsb_user_banned_batch_dev",
    "nutsb_set_user_names", "nutsb_set_ban_swearing", "nutsb_speech_batch", "nutsb_speech_batch_dev", "nutsb_speech_batch_iov", "nutsb_q_speech",
    "nutsb_q_record", "nutsb_q_review", "nutsb_q_review_clear", "nutsb_set_speech_record", "nutsb_get_review_buffer",
    "nutsb_q_tell", "nutsb_q_pemote", "nutsb_q_wizshout", "nutsb_q_revtell",
    "nutsb_colour_com_count_batch", "nutsb_colour_com_strip_batch", "nutsb_stream_digests", "nutsb_q_write_user", "nutsb_q_write_room", "nutsb_q_write_room_except",
    "nutsb_q_write_level", "nutsb_q_write_sock", "nutsb_q_page_line", "nutsb_q_more", "nutsb_q_pending", "nutsb_flush", "nutsb_flush_iov", "nutsb_contains_swearing",
    "nutsb_site_banned", "nutsb_user_banned",
    "nutsb_write_batch_keep", "nutsb_stream_digests_continue", "nutsb_delivery_digests",
    "nutsb_multi_create", "nutsb_multi_create_rank", "nutsb_multi_destroy", "nutsb_multi_last_error", "nutsb_multi_n_shards", "nutsb_multi_ctx",
    "nutsb_multi_set_swear_words", "nutsb_multi_set_ban_files", "nutsb_multi_set_profiling", "nutsb_multi_set_users", "nutsb_multi_plan",
    "nutsb_multi_route", "nutsb_multi_write_batch", "nutsb_multi_stream_digests", "nutsb_multi_contains_swearing_batch",
    "nutsb_multi_site_banned_batch", "nutsb_multi_user_banned_batch", "nutsb_multi_get_timing",
    "nutsb_multi_write_batch_iov", "nutsb_multi_shard_iov", "nutsb_multi_set_user_names", "nutsb_multi_set_ban_swearing",
    "nutsb_multi_speech_batch", "nutsb_multi_speech_batch_iov", "nutsb_multi_set_speech_record", "nutsb_multi_get_review_buffer",
    "nutsb_pipe_create", "nutsb_pipe_destroy", "nutsb_pipe_depth", "nutsb_pipe_ctx", "nutsb_pipe_set_swear_words", "nutsb_pipe_set_users",
    "nutsb_pipe_set_user_names", "nutsb_pipe_set_ban_swearing", "nutsb_pipe_submit_speech_iov", "nutsb_pipe_submit_write_iov", "nutsb_pipe_wait",
]


def library_path() -> Path:
    return Path(__file__).resolve().parent / "_lib" / "libnutsb200.so"


def bind(lib: C.CDLL) -> C.CDLL:
    """Declares the C-ABI's signatures on a loaded library."""
    vp = C.c_void_p
    lib.nutsb_version.restype = C.c_int
    lib.nutsb_strerror.restype = C.c_char_p
    lib.nutsb_strerror.argtypes = [C.c_int]
    lib.nutsb_last_error.restype = C.c_char_p
    lib.nutsb_last_error.argtypes = [vp]
    lib.nutsb_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.nutsb_destroy.argtypes = [vp]
    lib.nutsb_destroy.restype = None
    lib.nutsb_set_profiling.argtypes = [vp, C.c_int]
    lib.nutsb_get_timing.argtypes = [vp, C.POINTER(Timing)]
    lib.nutsb_set_stream.argtypes = [vp, vp]
    lib.nutsb_set_overlap.argtypes = [vp, C.c_int]
    lib.nutsb_set_swear_words.argtypes = [vp, C.POINTER(C.c_char_p)]
    lib.nutsb_set_ban_files.argtypes = [vp, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]
    lib.nutsb_set_users.argtypes = [vp, C.c_int32, C.c_int32, i32p, u8p, u8p]
    lib.nutsb_set_users_remap.argtypes = [vp, C.c_int32, C.c_int32, i32p, u8p, u8p, i32p]
    lib.nutsb_q_write_sock.argtypes = [vp, C.c_int32, C.c_char_p]
    lib.nutsb_write_batch.argtypes = [vp, C.POINTER(_Ops), C.POINTER(_Streams)]
    lib.nutsb_write_batch_dev.argtypes = [vp, C.POINTER(_Ops), C.POINTER(_Streams)]
    lib.nutsb_write_batch_iov.argtypes = [vp, C.POINTER(_Ops), C.POINTER(_IovStreams)]
    for name in ("contains_swearing", "site_banned", "user_banned"):
        getattr(lib, f"nutsb_{name}_batch").argtypes = [vp, C.c_int64, vp, vp, vp]
        getattr(lib, f"nutsb_{name}_batch_dev").argtypes = [vp, C.c_int64, vp, vp, vp]
        getattr(lib, f"nutsb_{name}").argtypes = [vp, C.c_char_p]
    lib.nutsb_set_user_names.argtypes = [vp, C.c_int32, vp, vp, vp]
    lib.nutsb_set_ban_swearing.argtypes = [vp, C.c_int]
    lib.nutsb_speech_batch.argtypes = [vp, C.c_int64, vp, vp, vp, vp, C.POINTER(_Streams)]
    lib.nutsb_speech_batch_dev.argtypes = [vp, C.c_int64, vp, vp, vp, vp, C.POINTER(_Streams)]
    lib.nutsb_speech_batch_iov.argtypes = [vp, C.c_int64, vp, vp, vp, vp, C.POINTER(_IovStreams)]
    lib.nutsb_q_speech.argtypes = [vp, C.c_int, C.c_int32, C.c_char_p]
    lib.nutsb_set_speech_record.argtypes = [vp, C.c_int]
    lib.nutsb_get_review_buffer.argtypes = [vp, C.c_int32, vp, C.POINTER(C.c_int32)]
    lib.nutsb_set_clones.argtypes = [vp, C.c_int32, vp, vp]
    lib.nutsb_set_room_names.argtypes = [vp, C.c_int32, vp, vp]
    lib.nutsb_set_remotes.argtypes = [vp, C.c_int32, vp, vp]
    lib.nutsb_ban_edit.argtypes = [vp, C.c_int, C.c_int, C.c_char_p, C.POINTER(C.c_int)]
    lib.nutsb_get_ban_file.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
    lib.nutsb_q_record.argtypes = [vp, C.c_int32, C.c_char_p]
    lib.nutsb_q_review.argtypes = [vp, C.c_int32, C.c_int32, C.c_char_p]
    lib.nutsb_q_review_clear.argtypes = [vp, C.c_int32]
    lib.nutsb_q_tell.argtypes = [vp, C.c_int32, C.c_int32, C.c_char_p]
    lib.nutsb_q_pemote.argtypes = [vp, C.c_int32, C.c_int32, C.c_char_p]
    lib.nutsb_q_wizshout.argtypes = [vp, C.c_int32, C.c_int, C.c_char_p, C.c_char_p]
    lib.nutsb_q_revtell.argtypes = [vp, C.c_int32]
    lib.nutsb_colour_com_count_batch.argtypes = [vp, C.c_int64, vp, vp, vp]
    lib.nutsb_colour_com_strip_batch.argtypes = [vp, C.c_int64, vp, vp, C.POINTER(vp), C.POINTER(vp)]
    lib.nutsb_stream_digests.argtypes = [vp, u64p]
    lib.nutsb_q_write_user.argtypes = [vp, C.c_int32, C.c_char_p]
    lib.nutsb_q_write_room.argtypes = [vp, C.c_int32, C.c_char_p, C.c_int, C.c_int]
    lib.nutsb_q_write_room_except.argtypes = [vp, C.c_int32, C.c_char_p, C.c_int32, C.c_int, C.c_int]
    lib.nutsb_q_write_level.argtypes = [vp, C.c_int, C.c_int, C.c_char_p, C.c_int32]
    lib.nutsb_q_page_line.argtypes = [vp, C.c_int32, C.c_char_p, C.c_int]
    lib.nutsb_q_more.argtypes = [vp, C.c_int32, C.c_int32, C.c_char_p, C.c_size_t, C.POINTER(C.c_int64), C.POINTER(C.c_int)]
    lib.nutsb_q_pending.restype = C.c_int64
    lib.nutsb_q_pending.argtypes = [vp]
    lib.nutsb_flush.argtypes = [vp, C.POINTER(_Streams)]
    lib.nutsb_flush_iov.argtypes = [vp, C.POINTER(_IovStreams)]
    lib.nutsb_write_batch_keep.argtypes = [vp, C.POINTER(_Ops), C.POINTER(_Streams)]
    lib.nutsb_stream_digests_continue.argtypes = [vp, u64p]
    lib.nutsb_delivery_digests.argtypes = [vp, u64p, u64p]
    lib.nutsb_multi_create.argtypes = [C.POINTER(vp), i32p, C.c_int]
    lib.nutsb_multi_create_rank.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int]
    lib.nutsb_multi_destroy.argtypes = [vp]
    lib.nutsb_multi_destroy.restype = None
    lib.nutsb_multi_last_error.argtypes = [vp]
    lib.nutsb_multi_last_error.restype = C.c_char_p
    lib.nutsb_multi_n_shards.argtypes = [vp]
    lib.nutsb_multi_ctx.argtypes = [vp, C.c_int]
    lib.nutsb_multi_ctx.restype = vp
    lib.nutsb_multi_set_swear_words.argtypes = [vp, C.POINTER(C.c_char_p)]
    lib.nutsb_multi_set_ban_files.argtypes = [vp, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]
    lib.nutsb_multi_set_profiling.argtypes = [vp, C.c_int]
    lib.nutsb_multi_set_users.argtypes = [vp, C.c_int32, C.c_int32, i32p, u8p, u8p, u64p]
    lib.nutsb_multi_plan.argtypes = [vp, i32p, i32p, i32p]
    lib.nutsb_multi_route.argtypes = [vp, C.POINTER(_Ops), C.c_int, C.POINTER(_Ops)]
    lib.nutsb_multi_write_batch.argtypes = [vp, C.POINTER(_Ops), C.POINTER(_MStreams), C.c_int]
    lib.nutsb_multi_stream_digests.argtypes = [vp, u64p, C.c_int]
    for name in ("contains_swearing", "site_banned", "user_banned"):
        getattr(lib, f"nutsb_multi_{name}_batch").argtypes = [vp, C.c_int64, vp, vp, vp]
    lib.nutsb_multi_get_timing.argtypes = [vp, C.c_int, C.POINTER(Timing)]
    lib.nutsb_multi_write_batch_iov.argtypes = [vp, C.POINTER(_Ops), C.POINTER(_MIovStreams)]
    lib.nutsb_multi_shard_iov.argtypes = [vp, C.c_int, C.POINTER(_IovStreams)]
    lib.nutsb_multi_set_user_names.argtypes = [vp, C.c_int32, vp, vp, vp]
    lib.nutsb_multi_set_ban_swearing.argtypes = [vp, C.c_int]
    lib.nutsb_multi_speech_batch.argtypes = [vp, C.c_int64, vp, vp, vp, vp, C.POINTER(_MStreams), C.c_int]
    lib.nutsb_multi_speech_batch_iov.argtypes = [vp, C.c_int64, vp, vp, vp, vp, C.POINTER(_MIovStreams)]
    lib.nutsb_multi_set_speech_record.argtypes = [vp, C.c_int]
    lib.nutsb_multi_get_review_buffer.argtypes = [vp, C.c_int32, vp, C.POINTER(C.c_int32)]
    lib.nutsb_pipe_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int]
    lib.nutsb_pipe_destroy.argtypes = [vp]
    lib.nutsb_pipe_destroy.restype = None
    lib.nutsb_pipe_depth.argtypes = [vp]
    lib.nutsb_pipe_ctx.argtypes = [vp, C.c_int]
    lib.nutsb_pipe_ctx.restype = vp
    lib.nutsb_pipe_set_swear_words.argtypes = [vp, C.POINTER(C.c_char_p)]
    lib.nutsb_pipe_set_users.argtypes = [vp, C.c_int32, C.c_int32, i32p, u8p, u8p]
    lib.nutsb_pipe_set_user_names.argtypes = [vp, C.c_int32, vp, vp, vp]
    lib.nutsb_pipe_set_ban_swearing.argtypes = [vp, C.c_int]
    lib.nutsb_pipe_submit_speech_iov.argtypes = [vp, C.c_int64, vp, vp, vp, vp, u64p]
    lib.nutsb_pipe_submit_write_iov.argtypes = [vp, C.POINTER(_Ops), u64p]
    lib.nutsb_pipe_wait.argtypes = [vp, C.c_uint64, C.POINTER(_IovStreams)]
    return lib


_LIB = None


def load_library() -> C.CDLL:
    """Loads nuts333_b200/_lib/libnutsb200.so (built by nuts333_b200.build).  Fails
    loudly when it is missing: there is nothing to fall back to."""
    global _LIB
    if _LIB is None:
        p = library_path()
        if not p.exists():
            raise FileNotFoundError(f"{p} is missing: run `python -m nuts333_b200.build` (needs nvcc)")
        _LIB = bind(C.CDLL(str(p)))
    return _LIB


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _addr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def pack(strings):
    """list[bytes] -> (u8 array, u64 offsets[n+1])"""
    off = np.zeros(len(strings) + 1, dtype=np.uint64)
    if len(strings):
        off[1:] = np.cumsum([len(s) for s in strings], dtype=np.uint64)
    data = np.frombuffer(b"".join(strings), dtype=np.uint8)
    return (data.copy() if data.size else np.zeros(0, np.uint8)), off


class Streams:
    """Per-user socket streams returned by a write batch (host copy)."""

    def __init__(self, off, data, n_deliveries):
        self.off, self.data, self.n_deliveries = off, data, int(n_deliveries)

    @property
    def n_users(self):
        return len(self.off) - 1

    @property
    def total_bytes(self):
        return int(self.off[-1]) if len(self.off) else 0

    def user(self, u) -> bytes:
        return self.data[int(self.off[u]):int(self.off[u + 1])].tobytes()


class IovStreams:
    """Per-user gather lists returned by nutsb_write_batch_iov: what a host hands to writev(2).  The pieces
    point into the context's pinned pool, so this object is valid until the next batch on the context;
    user(u) / streams() gather the bytes a socket would receive."""

    def __init__(self, off, first, count, iov, pools, n_deliveries, raw=None):
        self.off, self.first, self.count, self.iov = off, first, count, iov      # iov: u64[n_iov, 2] = (address, length)
        self.pools = [(int(a), int(n)) for a, n in pools]                       # (address, bytes) of the host pools
        self.n_deliveries = int(n_deliveries)
        self.raw = raw

    @property
    def pool_bytes(self):
        return sum(n for _, n in self.pools)

    @property
    def n_users(self):
        return len(self.first)

    @property
    def n_iov(self):
        return len(self.iov)

    @property
    def total_bytes(self):
        return int(self.off[-1]) if len(self.off) else 0

    def pieces(self, u):
        f, c = int(self.first[u]), int(self.count[u])
        return self.iov[f:f + c]

    def user(self, u) -> bytes:
        return b"".join(C.string_at(int(a), int(n)) for a, n in self.pieces(u) if n)

    def streams(self) -> "Streams":
        """The same result as nutsb_write_batch would return (gathered on the host)."""
        parts = [self.user(u) for u in range(self.n_users)]
        data = np.frombuffer(b"".join(parts), np.uint8)
        return Streams(self.off.copy(), data, self.n_deliveries)


def _review_buffer(fn, h, room, ck):
    buf = (C.c_uint8 * (REVIEW_LINES * (REVIEW_LEN + 2)))()
    line = C.c_int32(0)
    ck(fn(h, room, buf, C.byref(line)))
    raw = bytes(buf)
    return [raw[i * (REVIEW_LEN + 2):(i + 1) * (REVIEW_LEN + 2)] for i in range(REVIEW_LINES)], line.value


class Context:
    """One context per GPU (nutsb_create / nutsb_destroy)."""

    def __init__(self, device: int = 0, lib: C.CDLL | None = None):
        self.lib = lib if lib is not None else load_library()
        self._h = C.c_void_p()
        rc = self.lib.nutsb_create(C.byref(self._h), device)
        if rc != 0:
            raise NutsbError(rc, "nutsb_create failed (no usable CUDA device?)")
        self.n_users = 0

    def close(self):
        if self._h:
            self.lib.nutsb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc < 0:
            raise NutsbError(rc, (self.lib.nutsb_last_error(self._h) or b"").decode(errors="replace"))
        return rc

    # -- tables / population -------------------------------------------------------------
    def set_swear_words(self, words):
        """words: the reference's swear_words[] content; the list ends at the first
        entry starting with '*' (nuts333.h:275-277) or at the end of the sequence."""
        ws = [w if isinstance(w, bytes) else w.encode() for w in words]
        arr = (C.c_char_p * (len(ws) + 1))(*ws, None)
        self._ck(self.lib.nutsb_set_swear_words(self._h, arr))

    def set_ban_files(self, siteban: bytes | None, userban: bytes | None):
        """Raw bytes of datafiles/siteban and datafiles/userban; None = file missing."""
        self._ck(self.lib.nutsb_set_ban_files(self._h, siteban, len(siteban or b""), userban, len(userban or b"")))

    def set_users(self, room, flags, level, n_rooms: int, prev_index=None):
        """prev_index[u]: the index user u had in the population before (-1: new), when users joined or left"""
        room, flags, level = _np(room, np.int32), _np(flags, np.uint8), _np(level, np.uint8)
        if prev_index is None:
            self._ck(self.lib.nutsb_set_users(self._h, len(room), n_rooms, room.ctypes.data_as(i32p),
                                              flags.ctypes.data_as(u8p), level.ctypes.data_as(u8p)))
        else:
            prev = _np(prev_index, np.int32)
            self._ck(self.lib.nutsb_set_users_remap(self._h, len(room), n_rooms, room.ctypes.data_as(i32p),
                                                    flags.ctypes.data_as(u8p), level.ctypes.data_as(u8p), prev.ctypes.data_as(i32p)))
        self.n_users = len(room)

    def set_user_names(self, names, speech_flags):
        """names: list[bytes] (user->name); speech_flags: SF_INVIS | SF_MUZZLED per user"""
        data, off = pack([n if isinstance(n, bytes) else n.encode() for n in names])
        fl = _np(speech_flags, np.uint8)
        self._ck(self.lib.nutsb_set_user_names(self._h, len(names), _addr(data) if data.size else None, _addr(off), _addr(fl)))

    def set_ban_swearing(self, on: bool):
        self._ck(self.lib.nutsb_set_ban_swearing(self._h, 1 if on else 0))

    def speech_batch(self, verb, speaker, bodies, body_off) -> "Streams":
        """say/shout/emote/semote/echo/bcast lines composed and rendered on the device."""
        verb, speaker = _np(verb, np.uint8), _np(speaker, np.int32)
        bodies, body_off = _np(bodies, np.uint8), _np(body_off, np.uint64)
        st = _Streams()
        self._ck(self.lib.nutsb_speech_batch(self._h, len(verb), _addr(verb), _addr(speaker),
                                             _addr(bodies) if bodies.size else None, _addr(body_off), C.byref(st)))
        return self._host_streams(st)

    def speech_batch_iov(self, verb, speaker, bodies, body_off) -> "IovStreams":
        """speech_batch with gather lists as the result (nutsb_speech_batch_iov)."""
        verb, speaker = _np(verb, np.uint8), _np(speaker, np.int32)
        bodies, body_off = _np(bodies, np.uint8), _np(body_off, np.uint64)
        st = _IovStreams()
        self._ck(self.lib.nutsb_speech_batch_iov(self._h, len(verb), _addr(verb), _addr(speaker),
                                                 _addr(bodies) if bodies.size else None, _addr(body_off), C.byref(st)))
        return self._host_iov(st)

    def set_speech_record(self, on: bool):
        """on: speech batches record what say / emote / echo send to the room in its review buffer, as the queue
        tier does (nutsb_set_speech_record)"""
        self._ck(self.lib.nutsb_set_speech_record(self._h, 1 if on else 0))

    def review_buffer(self, room):
        """-> (rows, line): the room's REVIEW_LINES rows of REVIEW_LEN + 2 bytes each and the ring position"""
        return _review_buffer(self.lib.nutsb_get_review_buffer, self._h, room, self._ck)

    def set_clones(self, owner, hear):
        owner, hear = _np(owner, np.int32), _np(hear, np.uint8)
        self._ck(self.lib.nutsb_set_clones(self._h, len(owner), _addr(owner), _addr(hear)))

    def set_remotes(self, link, old_peer):
        link, old_peer = _np(link, np.int32), _np(old_peer, np.uint8)
        self._ck(self.lib.nutsb_set_remotes(self._h, len(link), _addr(link), _addr(old_peer)))

    def set_room_names(self, names):
        data = np.frombuffer(b"".join(names) or b"\0", np.uint8)
        off = np.zeros(len(names) + 1, np.uint64)
        off[1:] = np.cumsum([len(n) for n in names])
        self._ck(self.lib.nutsb_set_room_names(self._h, len(names), _addr(data), _addr(off)))

    def ban_edit(self, which: int, add: bool, token) -> int:
        """ban_site/ban_user (add) or unban_site/unban_user on the context's lists -> 0 done, 1 nothing to do"""
        r = C.c_int(0)
        self._ck(self.lib.nutsb_ban_edit(self._h, which, 1 if add else 0, token if isinstance(token, bytes) else token.encode("latin-1"), C.byref(r)))
        return r.value

    def ban_file(self, which: int):
        """the list as it stands -> bytes, or None when there is no file"""
        p, n, pr = C.c_void_p(), C.c_size_t(0), C.c_int(0)
        self._ck(self.lib.nutsb_get_ban_file(self._h, which, C.byref(p), C.byref(n), C.byref(pr)))
        if not pr.value:
            return None
        return C.string_at(p, n.value) if n.value else b""

    def set_profiling(self, on=True):
        self._ck(self.lib.nutsb_set_profiling(self._h, 1 if on else 0))

    def set_overlap(self, on: bool = True):
        self._ck(self.lib.nutsb_set_overlap(self._h, 1 if on else 0))

    def set_stream(self, cuda_stream: int):
        self._ck(self.lib.nutsb_set_stream(self._h, C.c_void_p(cuda_stream)))

    def timing(self) -> Timing:
        t = Timing()
        self._ck(self.lib.nutsb_get_timing(self._h, C.byref(t)))
        return t

    # -- write batches -------------------------------------------------------------------
    @staticmethod
    def _ops_struct(ops, keep):
        n = len(ops["kind"])
        arrs = dict(text=_np(ops["text"], np.uint8), off=_np(ops["off"], np.uint64), kind=_np(ops["kind"], np.uint8),
                    target=_np(ops["target"], np.int32), except_user=_np(ops["except_user"], np.int32),
                    flags=_np(ops["flags"], np.uint8))
        gate = ops.get("gate")
        verdict = ops.get("verdict")
        if gate is not None and verdict is not None:
            arrs["gate"], arrs["verdict"] = _np(gate, np.int32), _np(verdict, np.uint8)
        keep.append(arrs)
        o = _Ops(n, _addr(arrs["text"]) if arrs["text"].size else None, _addr(arrs["off"]), _addr(arrs["kind"]),
                 _addr(arrs["target"]), _addr(arrs["except_user"]), _addr(arrs["flags"]),
                 _addr(arrs.get("gate")), _addr(arrs.get("verdict")))
        return o

    def write_batch(self, ops) -> Streams:
        """ops: dict(text u8[], off u64[n+1], kind u8[n], target i32[n], except_user i32[n],
        flags u8[n][, gate i32[n], verdict u8[]]) in host memory."""
        keep = []
        o = self._ops_struct(ops, keep)
        st = _Streams()
        self._ck(self.lib.nutsb_write_batch(self._h, C.byref(o), C.byref(st)))
        return self._host_streams(st)

    def write_batch_iov(self, ops) -> IovStreams:
        """write_batch with gather lists as the result (nutsb_write_batch_iov)."""
        keep = []
        o = self._ops_struct(ops, keep)
        st = _IovStreams()
        self._ck(self.lib.nutsb_write_batch_iov(self._h, C.byref(o), C.byref(st)))
        return self._host_iov(st)

    def _host_iov(self, st) -> IovStreams:
        U, n = int(st.n_users), int(st.n_iov)
        off = np.ctypeslib.as_array(C.cast(st.off, u64p), shape=(U + 1,)).copy()
        first = np.ctypeslib.as_array(C.cast(st.first, u64p), shape=(max(U, 1),))[:U].copy()
        count = np.ctypeslib.as_array(C.cast(st.count, C.POINTER(C.c_uint32)), shape=(max(U, 1),))[:U].copy()
        iov = (np.ctypeslib.as_array(C.cast(st.iov, u64p), shape=(n, 2)).copy() if n else np.zeros((0, 2), np.uint64))
        return IovStreams(off, first, count, iov, [(st.pool or 0, st.pool_bytes), (st.pool2 or 0, st.pool2_bytes)],
                          st.n_deliveries, raw=st)

    def _host_streams(self, st) -> Streams:
        U = int(st.n_users)
        off = np.ctypeslib.as_array(C.cast(st.off, u64p), shape=(U + 1,)).copy()
        total = int(st.total_bytes)
        data = (np.ctypeslib.as_array(C.cast(st.bytes, u8p), shape=(total,)).copy() if total
                else np.zeros(0, np.uint8))
        return Streams(off, data, st.n_deliveries)

    def write_batch_dev(self, n_ops, text, off, kind, target, except_user, flags, gate=0, verdict=0):
        """All arguments are device addresses (ints).  Returns the raw nutsb_streams
        (device pointers, owned by the context)."""
        o = _Ops(n_ops, text, off, kind, target, except_user, flags, gate or None, verdict or None)
        st = _Streams()
        self._ck(self.lib.nutsb_write_batch_dev(self._h, C.byref(o), C.byref(st)))
        return st

    def stream_digests(self):
        d = np.zeros(max(self.n_users, 1), np.uint64)
        self._ck(self.lib.nutsb_stream_digests(self._h, d.ctypes.data_as(u64p)))
        return d[:self.n_users]

    def delivery_digests(self, n_ops):
        """SURVEY.md 8(d) parity digests of the last write batch -> (per_user u64[U], per_op u64[n_ops])"""
        pu, po = np.zeros(max(self.n_users, 1), np.uint64), np.zeros(max(n_ops, 1), np.uint64)
        self._ck(self.lib.nutsb_delivery_digests(self._h, pu.ctypes.data_as(u64p), po.ctypes.data_as(u64p)))
        return pu[:self.n_users], po[:n_ops]

    # -- verdict batches -----------------------------------------------------------------
    def _verdicts(self, name, text, off):
        text, off = _np(text, np.uint8), _np(off, np.uint64)
        n = len(off) - 1
        v = np.zeros(max(n, 1), np.uint8)
        self._ck(getattr(self.lib, f"nutsb_{name}_batch")(self._h, n, _addr(text) if text.size else None,
                                                          _addr(off), _addr(v)))
        return v[:n]

    def contains_swearing_batch(self, text, off):
        return self._verdicts("contains_swearing", text, off)

    def site_banned_batch(self, text, off):
        return self._verdicts("site_banned", text, off)

    def user_banned_batch(self, text, off):
        return self._verdicts("user_banned", text, off)

    def colour_com_count_batch(self, text, off):                      # c:2563
        text, off = _np(text, np.uint8), _np(off, np.uint64)
        n = len(off) - 1
        cnt = np.zeros(max(n, 1), np.int32)
        self._ck(self.lib.nutsb_colour_com_count_batch(self._h, n, _addr(text) if text.size else None, _addr(off), _addr(cnt)))
        return cnt[:n]

    def colour_com_strip_batch(self, text, off):                      # c:2588
        """-> (bytes u8[], off u64[n+1]) of the stripped strings"""
        text, off = _np(text, np.uint8), _np(off, np.uint64)
        n = len(off) - 1
        ob, oo = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.nutsb_colour_com_strip_batch(self._h, n, _addr(text) if text.size else None, _addr(off),
                                                       C.byref(ob), C.byref(oo)))
        o = np.ctypeslib.as_array(C.cast(oo, u64p), shape=(n + 1,)).copy()
        total = int(o[n])
        d = np.ctypeslib.as_array(C.cast(ob, u8p), shape=(total,)).copy() if total else np.zeros(0, np.uint8)
        return d, o

    def verdicts_dev(self, name, n, text, off, verdict):
        self._ck(getattr(self.lib, f"nutsb_{name}_batch_dev")(self._h, n, text, off, verdict))


class Talker:
    """The reference's call surface, same names and argument meaning.  Users and rooms
    are passed as their index in the reference's lists (None = NULL)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.force_listen = 0      # nuts333.h:293
        self.com_num = -1          # nuts333.h:201
        self.filepos = {}          # user->filepos (nuts333.h:75), per user index

    @staticmethod
    def _s(s):
        return s if isinstance(s, bytes) else s.encode("latin-1")

    def _shout(self):
        return 1 if self.com_num in (SHOUT, SEMOTE) else 0

    def write_user(self, user, s):                                   # c:1291
        c = self.ctx
        c._ck(c.lib.nutsb_q_write_user(c._h, -1 if user is None else user, self._s(s)))

    def write_room(self, rm, s):                                     # c:1390
        self.write_room_except(rm, s, None)

    def write_room_except(self, rm, s, user):                        # c:1401
        c = self.ctx
        c._ck(c.lib.nutsb_q_write_room_except(c._h, -1 if rm is None else rm, self._s(s),
                                              -1 if user is None else user,
                                              1 if self.force_listen else 0, self._shout()))

    def write_level(self, level, above, s, user):                    # c:1372
        c = self.ctx
        c._ck(c.lib.nutsb_q_write_level(c._h, level, 1 if above else 0, self._s(s), -1 if user is None else user))

    def write_sock(self, sock_user, s):                              # c:1281, a user's own socket
        c = self.ctx
        c._ck(c.lib.nutsb_q_write_sock(c._h, sock_user, self._s(s)))

    def _speech(self, verb, user, inpstr):
        c = self.ctx
        c._ck(c.lib.nutsb_q_speech(c._h, verb, user, self._s(inpstr)))

    def record(self, rm, s):                                         # c:2062
        c = self.ctx
        c._ck(c.lib.nutsb_q_record(c._h, rm, self._s(s)))

    def review(self, user, rm, room_name=None):                      # c:5192 (rm resolved by the caller)
        c = self.ctx
        c._ck(c.lib.nutsb_q_review(c._h, user, rm, self._s(room_name if room_name is not None else "room%d" % rm)))

    def clear_revbuff(self, rm):                                     # c:2626
        c = self.ctx
        c._ck(c.lib.nutsb_q_review_clear(c._h, rm))

    def tell(self, user, target, inpstr):                            # c:4128 (target resolved by the caller)
        c = self.ctx
        c._ck(c.lib.nutsb_q_tell(c._h, user, target, self._s(inpstr)))

    def pemote(self, user, target, inpstr):                          # c:4234
        c = self.ctx
        c._ck(c.lib.nutsb_q_pemote(c._h, user, target, self._s(inpstr)))

    def wizshout(self, user, inpstr, lev=-1, level_name=None):       # c:6527
        c = self.ctx
        c._ck(c.lib.nutsb_q_wizshout(c._h, user, lev, None if level_name is None else self._s(level_name), self._s(inpstr)))

    def revtell(self, user):                                         # c:7699
        c = self.ctx
        c._ck(c.lib.nutsb_q_revtell(c._h, user))

    def say(self, user, inpstr):                                     # c:4062
        self._speech(SPEECH_SAY, user, inpstr)

    def shout(self, user, inpstr):                                   # c:4105
        self._speech(SPEECH_SHOUT, user, inpstr)

    def emote(self, user, inpstr):                                   # c:4188
        self._speech(SPEECH_EMOTE, user, inpstr)

    def semote(self, user, inpstr):                                  # c:4213
        self._speech(SPEECH_SEMOTE, user, inpstr)

    def echo(self, user, inpstr):                                    # c:4289
        self._speech(SPEECH_ECHO, user, inpstr)

    def bcast(self, user, inpstr):                                   # c:4772
        self._speech(SPEECH_BCAST, user, inpstr)

    def more(self, user, sock, filename) -> int:                    # c:2205
        """The pager: queues one page of `filename` for the user on socket `sock` (a user
        index; user None = the login-stage call more(NULL,sock,file)).  The file position
        is kept per user like user->filepos.  Returns more()'s return value (0, 1 or 2)."""
        c = self.ctx
        try:
            with open(filename, "rb") as fh:
                data = fh.read()
        except OSError:
            data = None
        key = -1 if user is None else user
        pos = C.c_int64(self.filepos.get(key, 0))
        rv = C.c_int(0)
        c._ck(c.lib.nutsb_q_more(c._h, key, sock, data, 0 if data is None else len(data), C.byref(pos), C.byref(rv)))
        if user is not None:
            self.filepos[key] = pos.value
        return rv.value

    def pending(self) -> int:
        return int(self.ctx.lib.nutsb_q_pending(self.ctx._h))

    def flush(self) -> Streams:
        """Runs everything queued; the host then write()s each user's stream."""
        c = self.ctx
        st = _Streams()
        c._ck(c.lib.nutsb_flush(c._h, C.byref(st)))
        return c._host_streams(st)

    def flush_iov(self) -> IovStreams:
        """Runs everything queued; the host then writev()s each user's gather list."""
        c = self.ctx
        st = _IovStreams()
        c._ck(c.lib.nutsb_flush_iov(c._h, C.byref(st)))
        return c._host_iov(st)

    def contains_swearing(self, s) -> int:                            # c:2540
        return self.ctx._ck(self.ctx.lib.nutsb_contains_swearing(self.ctx._h, self._s(s)))

    def site_banned(self, site) -> int:                               # c:330
        return self.ctx._ck(self.ctx.lib.nutsb_site_banned(self.ctx._h, self._s(site)))

    def user_banned(self, name) -> int:                               # c:349
        return self.ctx._ck(self.ctx.lib.nutsb_user_banned(self.ctx._h, self._s(name)))


class MIovStreams:
    """Per-user gather lists of a nutsb_multi batch in GLOBAL user order (nutsb_miov_streams): user u's pieces lie in
    the gather list of u's shard.  Valid until the next batch on the MultiContext."""

    def __init__(self, st):
        U = int(st.n_users)
        arr = lambda p, t: np.ctypeslib.as_array(C.cast(p, C.POINTER(t)), shape=(max(U, 1),))[:U].copy()
        self.len, self.iov_addr, self.count = arr(st.len, C.c_uint64), arr(st.iov, C.c_uint64), arr(st.count, C.c_uint32)
        self.total_bytes, self.n_deliveries = int(st.total_bytes), int(st.n_deliveries)

    @property
    def n_users(self):
        return len(self.len)

    def pieces(self, u):
        """u64[count[u], 2] = (address, length) of u's pieces"""
        n = int(self.count[u])
        if not n:
            return np.zeros((0, 2), np.uint64)
        return np.ctypeslib.as_array(C.cast(int(self.iov_addr[u]), u64p), shape=(n, 2)).copy()

    def user(self, u) -> bytes:
        return b"".join(C.string_at(int(a), int(n)) for a, n in self.pieces(u) if n)


class MultiContext:
    """nutsb_multi: one population and one batch over several GPUs (include/nutsb200.h).  `devices`: one context per
    entry (the same device may be named twice); or rank=(n_shards, shard, device) for one process per GPU."""

    def __init__(self, devices=None, lib=None, rank=None):
        self.lib = lib or load_library()
        self._h = C.c_void_p()
        if rank is not None:
            rc = self.lib.nutsb_multi_create_rank(C.byref(self._h), int(rank[0]), int(rank[1]), int(rank[2]))
        else:
            d = _np(devices, np.int32)
            rc = self.lib.nutsb_multi_create(C.byref(self._h), d.ctypes.data_as(i32p), len(d))
        if rc != 0:
            raise NutsbError(rc, "nutsb_multi_create failed: there is no CPU fallback")
        self.n_users = 0
        self._ctxs = {}

    def _ck(self, rc):
        if rc < 0:
            raise NutsbError(rc, (self.lib.nutsb_multi_last_error(self._h) or b"").decode(errors="replace"))

    def close(self):
        if self._h:
            self.lib.nutsb_multi_destroy(self._h)
            self._h = C.c_void_p()

    @property
    def n_shards(self):
        return int(self.lib.nutsb_multi_n_shards(self._h))

    def ctx(self, shard) -> "Context":
        """The shard's own context (None when this process does not run it); owned by the MultiContext."""
        if shard not in self._ctxs:
            h = self.lib.nutsb_multi_ctx(self._h, shard)
            if not h:
                return None
            c = Context.__new__(Context)
            c.lib, c._h, c.n_users = self.lib, C.c_void_p(h), 0
            c.close = lambda: None
            self._ctxs[shard] = c
        return self._ctxs[shard]

    def set_swear_words(self, words):
        ws = [w if isinstance(w, bytes) else w.encode() for w in words]
        arr = (C.c_char_p * (len(ws) + 1))(*ws, None)
        self._ck(self.lib.nutsb_multi_set_swear_words(self._h, arr))

    def set_ban_files(self, siteban, userban):
        self._ck(self.lib.nutsb_multi_set_ban_files(self._h, siteban, 0 if siteban is None else len(siteban),
                                                    userban, 0 if userban is None else len(userban)))

    def set_profiling(self, on=True):
        self._ck(self.lib.nutsb_multi_set_profiling(self._h, 1 if on else 0))

    def set_users(self, room, flags, level, n_rooms, room_weight=None):
        room, flags, level = _np(room, np.int32), _np(flags, np.uint8), _np(level, np.uint8)
        w = None if room_weight is None else _np(room_weight, np.uint64)
        self._ck(self.lib.nutsb_multi_set_users(self._h, len(room), n_rooms, room.ctypes.data_as(i32p), flags.ctypes.data_as(u8p),
                                                level.ctypes.data_as(u8p), None if w is None else w.ctypes.data_as(u64p)))
        self.n_users, self.n_rooms = len(room), n_rooms

    def plan(self):
        """-> room_shard[n_rooms], user_shard[n_users], user_local[n_users]"""
        rs, us, ul = np.zeros(max(self.n_rooms, 1), np.int32), np.zeros(max(self.n_users, 1), np.int32), np.zeros(max(self.n_users, 1), np.int32)
        self._ck(self.lib.nutsb_multi_plan(self._h, rs.ctypes.data_as(i32p), us.ctypes.data_as(i32p), ul.ctypes.data_as(i32p)))
        return rs[:self.n_rooms], us[:self.n_users], ul[:self.n_users]

    def _ops(self, ops, keep):
        return Context._ops_struct(ops, keep)

    def route(self, ops, shard):
        """The shard's routed ops as numpy copies (dict like `ops`, local indices)."""
        keep = []
        o = self._ops(ops, keep)
        r = _Ops()
        self._ck(self.lib.nutsb_multi_route(self._h, C.byref(o), shard, C.byref(r)))
        n = int(r.n_ops)
        arr = lambda p, t, k: (np.ctypeslib.as_array(C.cast(p, C.POINTER(t)), shape=(k,)).copy() if k else np.zeros(0, t))
        off = arr(r.text_off, C.c_uint64, n + 1)
        out = dict(text=arr(r.text, C.c_uint8, int(off[-1])), off=off, kind=arr(r.kind, C.c_uint8, n), target=arr(r.target, C.c_int32, n),
                   except_user=arr(r.except_user, C.c_int32, n), flags=arr(r.flags, C.c_uint8, n))
        if r.gate:
            out["gate"] = arr(r.gate, C.c_int32, n)
            out["verdict"] = np.ascontiguousarray(ops["verdict"], np.uint8)
        return out

    def write_batch(self, ops, keep=False):
        """-> list[bytes] per user in GLOBAL order (None per user when keep), total_bytes, n_deliveries"""
        k = []
        o = self._ops(ops, k)
        st = _MStreams()
        self._ck(self.lib.nutsb_multi_write_batch(self._h, C.byref(o), C.byref(st), 1 if keep else 0))
        if keep:
            return None, int(st.total_bytes), int(st.n_deliveries)
        U = int(st.n_users)
        ln = np.ctypeslib.as_array(C.cast(st.len, u64p), shape=(max(U, 1),))[:U]
        pt = np.ctypeslib.as_array(C.cast(st.ptr, u64p), shape=(max(U, 1),))[:U]
        return [C.string_at(int(pt[u]), int(ln[u])) if ln[u] else b"" for u in range(U)], int(st.total_bytes), int(st.n_deliveries)

    def write_batch_iov(self, ops) -> MIovStreams:
        """write_batch with gather lists as the result (nutsb_multi_write_batch_iov)."""
        k = []
        o = self._ops(ops, k)
        st = _MIovStreams()
        self._ck(self.lib.nutsb_multi_write_batch_iov(self._h, C.byref(o), C.byref(st)))
        return MIovStreams(st)

    def shard_iov(self, shard) -> IovStreams:
        """The shard's own result of the last gather-list batch (local user order; its pools hold the pieces)."""
        st = _IovStreams()
        self._ck(self.lib.nutsb_multi_shard_iov(self._h, shard, C.byref(st)))
        return Context._host_iov(None, st)

    def set_user_names(self, names, speech_flags):
        """names: list[bytes] in global user order; speech_flags: SF_INVIS | SF_MUZZLED per user"""
        data, off = pack([n if isinstance(n, bytes) else n.encode() for n in names])
        fl = _np(speech_flags, np.uint8)
        self._ck(self.lib.nutsb_multi_set_user_names(self._h, len(names), _addr(data) if data.size else None, _addr(off), _addr(fl)))

    def set_ban_swearing(self, on: bool):
        self._ck(self.lib.nutsb_multi_set_ban_swearing(self._h, 1 if on else 0))

    @staticmethod
    def _lines(verb, speaker, bodies, body_off):
        a = (_np(verb, np.uint8), _np(speaker, np.int32), _np(bodies, np.uint8), _np(body_off, np.uint64))
        return a, (len(a[0]), _addr(a[0]), _addr(a[1]), _addr(a[2]) if a[2].size else None, _addr(a[3]))

    def speech_batch(self, verb, speaker, bodies, body_off, keep=False):
        """say/shout/emote/semote/echo/bcast lines (global speaker indices) composed on every shard
        -> list[bytes] per user in GLOBAL order (None when keep), total_bytes, n_deliveries"""
        arrs, args = self._lines(verb, speaker, bodies, body_off)      # (arrs: the inputs stay alive through the call)
        st = _MStreams()
        self._ck(self.lib.nutsb_multi_speech_batch(self._h, *args, C.byref(st), 1 if keep else 0))
        if keep:
            return None, int(st.total_bytes), int(st.n_deliveries)
        U = int(st.n_users)
        ln = np.ctypeslib.as_array(C.cast(st.len, u64p), shape=(max(U, 1),))[:U]
        pt = np.ctypeslib.as_array(C.cast(st.ptr, u64p), shape=(max(U, 1),))[:U]
        return [C.string_at(int(pt[u]), int(ln[u])) if ln[u] else b"" for u in range(U)], int(st.total_bytes), int(st.n_deliveries)

    def speech_batch_iov(self, verb, speaker, bodies, body_off) -> MIovStreams:
        """speech_batch with gather lists as the result (nutsb_multi_speech_batch_iov)."""
        arrs, args = self._lines(verb, speaker, bodies, body_off)      # (arrs: the inputs stay alive through the call)
        st = _MIovStreams()
        self._ck(self.lib.nutsb_multi_speech_batch_iov(self._h, *args, C.byref(st)))
        return MIovStreams(st)

    def set_speech_record(self, on: bool):
        """Context.set_speech_record on every shard (refused in rank mode)"""
        self._ck(self.lib.nutsb_multi_set_speech_record(self._h, 1 if on else 0))

    def review_buffer(self, room):
        """-> (rows, line) of global room `room` (Context.review_buffer)"""
        return _review_buffer(self.lib.nutsb_multi_get_review_buffer, self._h, room, self._ck)

    def stream_digests(self, digest=None):
        """Per-user digests in global order; digest given: the fold continues from it (chunked jobs)."""
        cont = digest is not None
        d = np.zeros(max(self.n_users, 1), np.uint64) if digest is None else np.ascontiguousarray(digest, np.uint64)
        self._ck(self.lib.nutsb_multi_stream_digests(self._h, d.ctypes.data_as(u64p), 1 if cont else 0))
        return d[:self.n_users]

    def _verdicts(self, fn, data, off):
        data, off = _np(data, np.uint8), _np(off, np.uint64)
        n = len(off) - 1
        v = np.zeros(max(n, 1), np.uint8)
        self._ck(fn(self._h, n, _addr(data) if data.size else None, _addr(off), _addr(v)))
        return v[:n]

    def contains_swearing_batch(self, data, off):
        return self._verdicts(self.lib.nutsb_multi_contains_swearing_batch, data, off)

    def site_banned_batch(self, data, off):
        return self._verdicts(self.lib.nutsb_multi_site_banned_batch, data, off)

    def user_banned_batch(self, data, off):
        return self._verdicts(self.lib.nutsb_multi_user_banned_batch, data, off)

    def timing(self, shard) -> Timing:
        t = Timing()
        self._ck(self.lib.nutsb_multi_get_timing(self._h, shard, C.byref(t)))
        return t


class Pipe:
    """nutsb_pipe: `depth` host-buffer calls in flight on one device (include/nutsb200.h)."""

    def __init__(self, device=0, depth=2, lib=None):
        self.lib = lib or load_library()
        self._h = C.c_void_p()
        rc = self.lib.nutsb_pipe_create(C.byref(self._h), device, depth)
        if rc != 0:
            raise NutsbError(rc, "nutsb_pipe_create failed: there is no CPU fallback")
        self.depth, self._keep = depth, {}

    def _ck(self, rc):
        if rc < 0:
            raise NutsbError(rc, "nutsb_pipe")

    def close(self):
        if self._h:
            self.lib.nutsb_pipe_destroy(self._h)
            self._h = C.c_void_p()

    def ctx(self, lane) -> "Context":
        c = Context.__new__(Context)
        c.lib, c._h, c.n_users = self.lib, C.c_void_p(self.lib.nutsb_pipe_ctx(self._h, lane)), 0
        c.close = lambda: None
        return c

    def set_swear_words(self, words):
        ws = [w if isinstance(w, bytes) else w.encode() for w in words]
        self._ck(self.lib.nutsb_pipe_set_swear_words(self._h, (C.c_char_p * (len(ws) + 1))(*ws, None)))

    def set_users(self, room, flags, level, n_rooms):
        room, flags, level = _np(room, np.int32), _np(flags, np.uint8), _np(level, np.uint8)
        self._ck(self.lib.nutsb_pipe_set_users(self._h, len(room), n_rooms, room.ctypes.data_as(i32p), flags.ctypes.data_as(u8p), level.ctypes.data_as(u8p)))
        self.n_users = len(room)

    def set_user_names(self, names, speech_flags):
        data, off = pack([n if isinstance(n, bytes) else n.encode() for n in names])
        fl = _np(speech_flags, np.uint8)
        self._ck(self.lib.nutsb_pipe_set_user_names(self._h, len(names), _addr(data) if data.size else None, _addr(off), _addr(fl)))

    def set_ban_swearing(self, on):
        self._ck(self.lib.nutsb_pipe_set_ban_swearing(self._h, 1 if on else 0))

    def submit_speech_iov(self, verb, speaker, bodies, body_off) -> int:
        a = (_np(verb, np.uint8), _np(speaker, np.int32), _np(bodies, np.uint8), _np(body_off, np.uint64))
        t = C.c_uint64()
        self._ck(self.lib.nutsb_pipe_submit_speech_iov(self._h, len(a[0]), _addr(a[0]), _addr(a[1]), _addr(a[2]) if a[2].size else None, _addr(a[3]), C.byref(t)))
        self._keep[t.value % self.depth] = a               # the inputs stay alive until the lane is reused
        return t.value

    def submit_write_iov(self, ops) -> int:
        keep = []
        o = Context._ops_struct(ops, keep)
        t = C.c_uint64()
        self._ck(self.lib.nutsb_pipe_submit_write_iov(self._h, C.byref(o), C.byref(t)))
        self._keep[t.value % self.depth] = keep
        return t.value

    def wait(self, ticket) -> "IovStreams":
        st = _IovStreams()
        self._ck(self.lib.nutsb_pipe_wait(self._h, ticket, C.byref(st)))
        return Context._host_iov(None, st)
