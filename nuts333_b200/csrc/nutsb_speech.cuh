// nutsb_speech.cuh -- the callers' composition (SURVEY.md 8f rank 2): what say / shout /
// emote / semote / echo / bcast turn one input line into, as write ops.
//
//   say    nuts333.c:4062-4100     shout  c:4105-4126     emote  c:4188-4210
//   semote c:4213-4232             echo   c:4289-4305     bcast  c:4772-4788
//
// Every verb yields at most three ops ("slots"):
//   slot 0  the refusal to the speaker: "You are muzzled ..." or, gated on the swear
//           verdict of the body, noswearing (nuts333.h:151)
//   slot 1  the speaker's own copy ("You say: ...") or echo's write_level(WIZ,1,"(name) ")
//   slot 2  the line to the room / to every room
// and every op's text is  lit[a] + name? + lit[b] + body[skip..] + lit[c].
// The rules are one __host__ __device__ function so that the queue tier (host strings,
// nutsb_q_speech) and the batch tier (device composer, k_speech_*) cannot drift apart.
#pragma once
#include "nutsb_common.cuh"
#include "nutsb_kernels.cuh"          // nutsb_seg_bounds

#define NUTSB_SPEECH_SAY    0
#define NUTSB_SPEECH_SHOUT  1
#define NUTSB_SPEECH_EMOTE  2
#define NUTSB_SPEECH_SEMOTE 3
#define NUTSB_SPEECH_ECHO   4
#define NUTSB_SPEECH_BCAST  5
#define NUTSB_SPEECH_VERBS  6

// per-user speech flags (nutsb_set_user_names)
#define NUTSB_SF_INVIS   0x01u   // user->vis == 0: others see invisname
#define NUTSB_SF_MUZZLED 0x02u   // user->muzzled

#define NUTSB_NLIT 27
#define NUTSB_LIT_NL 13
#define NUTSB_LIT_INVISNAME 26

// The literals of the six callers, as they stand in the reference's sprintf formats.
// (id, text) -- the host builds the device table from this list.
#define NUTSB_SPEECH_LITERALS(X) \
    X(0, "") \
    X(1, "You are muzzled, you cannot speak.\n") \
    X(2, "You are muzzled, you cannot shout.\n") \
    X(3, "You are muzzled, you cannot emote.\n") \
    X(4, "You are muzzled, you cannot echo.\n") \
    X(5, "You are muzzled, you cannot broadcast anything.\n") \
    X(6, "Swearing is not allowed here.\n") \
    X(7, "You say: ") X(8, "You ask: ") X(9, "You exclaim: ") \
    X(10, " says: ") X(11, " asks: ") X(12, " exclaims: ") \
    X(13, "\n") \
    X(14, "~OLYou shout:~RS ") X(15, "~OL") X(16, " shouts:~RS ") \
    X(17, " ") X(18, "~OL!!~RS ") \
    X(19, "(") X(20, ") ") X(21, "- ") \
    X(22, "\07\n~BR*** Broadcast message from ") X(23, " ***\n") X(24, "\n\n") \
    X(25, "\07\n~BR*** Broadcast message ***\n") \
    X(26, "A presence")

struct SpeechSlot {
    u8  kind;        // NUTSB_OP_* (NUTSB_OP_NONE: the slot is unused)
    u8  flags;       // NUTSB_OF_*
    u8  gated;       // 0 unconditional, 1 live iff the body is clean, 2 live iff it swears
    u8  a, b, c;     // literal ids
    u8  name;        // 0 none, 1 name as others see it (invisname when invisible), 2 user->name
    u8  body;        // 0 no body, 1 whole body, 2 body without its first byte
    i32 target, except_user;
};

// verb, slot in 0..2, the speaker's index / room (-1 none) / speech flags, ban_swearing,
// first and last byte of the body (0 when empty).
__host__ __device__ __forceinline__ SpeechSlot nutsb_speech_slot(u32 verb, u32 slot, i32 spk, i32 room, u32 sflags,
                                                               bool ban_swearing, u8 first, u8 last)
{
    SpeechSlot s;
    s.kind = NUTSB_OP_NONE; s.flags = 0; s.gated = 0; s.a = s.b = s.c = 0; s.name = 0; s.body = 0;
    s.target = -1; s.except_user = -1;
    const bool muzzled = (sflags & NUTSB_SF_MUZZLED) != 0;
    // A speaker in no room is a user away on another talker: say() relays the line over the
    // netlink and writes nothing locally (c:4071-4076, out of scope); emote() and echo() are not
    // reached for such users (exec_com forwards their commands) and would dereference
    // user->room in record() (c:4209, c:4304).  Those three yield nothing here; the muzzle
    // check comes first (c:4068).
    if (room < 0 && !muzzled && (verb == NUTSB_SPEECH_SAY || verb == NUTSB_SPEECH_EMOTE || verb == NUTSB_SPEECH_ECHO)) return s;
    // only say / shout / emote ask contains_swearing (c:4091, c:4116, c:4198)
    const bool checks = ban_swearing && (verb == NUTSB_SPEECH_SAY || verb == NUTSB_SPEECH_SHOUT || verb == NUTSB_SPEECH_EMOTE);
    if (slot == 0) {
        if (muzzled) {
            s.kind = NUTSB_OP_USER; s.target = spk;
            s.a = verb == NUTSB_SPEECH_SAY ? 1 : verb == NUTSB_SPEECH_SHOUT ? 2 : verb == NUTSB_SPEECH_ECHO ? 4
                : verb == NUTSB_SPEECH_BCAST ? 5 : 3;
        } else if (checks) {
            s.kind = NUTSB_OP_USER; s.target = spk; s.a = 6; s.gated = 2; s.flags = NUTSB_OF_GATE_IF_SET;
        }
        return s;
    }
    if (muzzled) return s;
    const u8 g = checks ? 1 : 0;
    const u32 t = last == '?' ? 1u : last == '!' ? 2u : 0u;          // c:4080-4084
    switch (verb) {
    case NUTSB_SPEECH_SAY:
        if (slot == 1) { s.kind = NUTSB_OP_USER; s.target = spk; s.a = (u8)(7 + t); s.body = 1; s.c = NUTSB_LIT_NL; }
        else { s.kind = NUTSB_OP_ROOM; s.target = room; s.except_user = spk; s.name = 1; s.b = (u8)(10 + t); s.body = 1; s.c = NUTSB_LIT_NL; }
        s.gated = g; break;
    case NUTSB_SPEECH_SHOUT:
        if (slot == 1) { s.kind = NUTSB_OP_USER; s.target = spk; s.a = 14; s.body = 1; s.c = NUTSB_LIT_NL; }
        else { s.kind = NUTSB_OP_ROOM; s.target = -1; s.except_user = spk; s.flags = NUTSB_OF_SHOUT; s.a = 15; s.name = 1; s.b = 16; s.body = 1; s.c = NUTSB_LIT_NL; }
        s.gated = g; break;
    case NUTSB_SPEECH_EMOTE:
        if (slot == 2) { s.kind = NUTSB_OP_ROOM; s.target = room; s.name = 1;
                         if (first == ';') s.body = 2; else { s.b = 17; s.body = 1; }
                         s.c = NUTSB_LIT_NL; s.gated = g; }
        break;
    case NUTSB_SPEECH_SEMOTE:
        if (slot == 2) { s.kind = NUTSB_OP_ROOM; s.target = -1; s.flags = NUTSB_OF_SHOUT; s.a = 18; s.name = 1;
                         if (first == '#') s.body = 2; else { s.b = 17; s.body = 1; }
                         s.c = NUTSB_LIT_NL; }
        break;
    case NUTSB_SPEECH_ECHO:
        if (slot == 1) { s.kind = NUTSB_OP_LEVEL; s.target = 2 /* WIZ */; s.flags = NUTSB_OF_ABOVE; s.a = 19; s.name = 2; s.b = 20; }
        else { s.kind = NUTSB_OP_ROOM; s.target = room; s.a = 21; s.body = 1; s.c = NUTSB_LIT_NL; }
        break;
    case NUTSB_SPEECH_BCAST:
        if (slot == 2) { s.kind = NUTSB_OP_ROOM; s.target = -1; s.flags = NUTSB_OF_FORCE_LISTEN; s.body = 1; s.c = 24;
                         if (sflags & NUTSB_SF_INVIS) s.a = 25; else { s.a = 22; s.name = 2; s.b = 23; } }
        break;
    default: break;
    }
    if (s.kind != NUTSB_OP_NONE && s.gated == 0) s.flags &= (u8)~NUTSB_OF_GATE_IF_SET;
    return s;
}

// ---- device composer ---------------------------------------------------------------------
struct SpeechView {
    i64 n;
    const u8  *verb;         // [n]
    const i32 *speaker;      // [n]
    const u8  *body; const u64 *body_off;        // packed bodies
    const u8  *names; const u64 *name_off;       // packed user names, [U+1]
    const u8  *sflags;       // [U]
    const i32 *user_room;    // [U] room' (n_rooms = no room)
    const u8  *lit; const u32 *lit_off;          // the literal table, [NLIT+1]
    i32 n_users, n_rooms;
    u32 ban_swearing;
};

// Shard mode (nutsb_multi): every shard is given the whole batch and composes the lines that produce an op
// on it.  The speaker index of a line is GLOBAL; the SpeechView's names / name_off / sflags are the global
// tables, its user_room / n_rooms the shard's own.  Where a slot's op lands: write_user and the speaker's
// room -> the speaker's shard (a room's users live with it); all rooms (target -1: shout / semote / bcast)
// and write_level (echo) -> every shard.
struct SpeechShard {
    const i32 *sel;          // [k] the lines this shard composes, in batch order (k_speech_route + a scan)
    i64 k;
    const i32 *user_shard, *user_local;          // [n_users], global
    const u8  *has_room;     // [n_users], global: the user is in a room
    i32 shard;
};

// The rule's view of speaker `spk` (global) on this shard: on its own shard the local index and room, elsewhere
// the global index (it only names the speaker's name) and a room that only says whether it has one.
__device__ __forceinline__ bool nutsb_speech_home(const SpeechView &v, const SpeechShard &sh, i32 spk, i32 *who, i32 *room)
{
    const bool home = sh.user_shard[spk] == sh.shard;
    if (home) {
        *who = sh.user_local[spk];
        *room = v.user_room[*who] < v.n_rooms ? v.user_room[*who] : -1;
    } else {
        *who = spk; *room = sh.has_room[spk] ? 0 : -1;
    }
    return home;
}

// The slot as this shard delivers it: away from the speaker's shard only the all-room and level ops are left,
// and nobody is excluded (the speaker is in none of this shard's rooms).
__device__ __forceinline__ void nutsb_speech_away(SpeechSlot &s)
{
    if (s.kind == NUTSB_OP_USER || (s.kind == NUTSB_OP_ROOM && s.target >= 0)) s.kind = NUTSB_OP_NONE;
    s.except_user = -1;
}

// One thread per line of the whole batch: keep[m] = line m produces an op on this shard.  The line checks of
// k_speech_measure are made here, for every line, so that each shard reports what one context would.
__global__ void __launch_bounds__(256)
k_speech_route(SpeechView v, SpeechShard sh, u8 *keep, u32 *status)
{
    const i64 m = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= v.n) return;
    keep[m] = 0;
    const i32 spk = v.speaker[m];
    const u32 verb = v.verb[m];
    if (spk < 0 || spk >= v.n_users || verb >= NUTSB_SPEECH_VERBS) {
        atomicOr(status, spk < 0 || spk >= v.n_users ? NUTSB_ST_BAD_INDEX : NUTSB_ST_BAD_KIND);
        return;
    }
    const u64 b0 = v.body_off[m], b1 = v.body_off[m + 1];
    if (b1 < b0 || b0 < v.body_off[0] || b1 > v.body_off[v.n]) { atomicOr(status, NUTSB_ST_BAD_OFFSETS); return; }
    const u8 first = b1 > b0 ? v.body[b0] : 0, last = b1 > b0 ? v.body[b1 - 1] : 0;
    const bool home = sh.user_shard[spk] == sh.shard;
    const i32 room = sh.has_room[spk] ? 0 : -1;          // (the rule asks only whether there is one)
    bool any = false;
    for (u32 s = 0; s < 3; ++s) {
        const SpeechSlot sl = nutsb_speech_slot(verb, s, spk, room, v.sflags[spk], v.ban_swearing != 0, first, last);
        any |= sl.kind != NUTSB_OP_NONE && (home || sl.kind == NUTSB_OP_LEVEL || (sl.kind == NUTSB_OP_ROOM && sl.target < 0));
    }
    keep[m] = any ? 1 : 0;
}

__device__ __forceinline__ u32 nutsb_speech_len(const SpeechView &v, const SpeechSlot &s, i32 spk, u32 blen)
{
    if (s.kind == NUTSB_OP_NONE) return 0;
    u32 n = (v.lit_off[s.a + 1] - v.lit_off[s.a]) + (v.lit_off[s.b + 1] - v.lit_off[s.b]) + (v.lit_off[s.c + 1] - v.lit_off[s.c]);
    if (s.name == 2 || (s.name == 1 && !(v.sflags[spk] & NUTSB_SF_INVIS))) n += (u32)(v.name_off[spk + 1] - v.name_off[spk]);
    else if (s.name == 1) n += v.lit_off[NUTSB_LIT_INVISNAME + 1] - v.lit_off[NUTSB_LIT_INVISNAME];
    if (s.body == 1) n += blen; else if (s.body == 2) n += blen ? blen - 1 : 0;
    return n;
}

// One thread per message: the three slot lengths (0 for an unused slot).  SHARD: one thread per selected line
// j (line sel[j]); its slots are ops 3j..3j+2.
template <bool SHARD>
__global__ void __launch_bounds__(256)
k_speech_measure(SpeechView v, SpeechShard sh, u32 *slot_len, u32 *status)
{
    const i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (SHARD ? sh.k : v.n)) return;
    const i64 m = SHARD ? (i64)sh.sel[j] : j;
    const i32 spk = v.speaker[m];
    const u32 verb = v.verb[m];
    if (spk < 0 || spk >= v.n_users || verb >= NUTSB_SPEECH_VERBS) {
        atomicOr(status, spk < 0 || spk >= v.n_users ? NUTSB_ST_BAD_INDEX : NUTSB_ST_BAD_KIND);
        slot_len[3 * j] = slot_len[3 * j + 1] = slot_len[3 * j + 2] = 0;
        return;
    }
    const u64 b0 = v.body_off[m], b1 = v.body_off[m + 1];
    if (b1 < b0 || b0 < v.body_off[0] || b1 > v.body_off[v.n]) {       // not monotone: nothing is read through these offsets
        atomicOr(status, NUTSB_ST_BAD_OFFSETS);
        slot_len[3 * j] = slot_len[3 * j + 1] = slot_len[3 * j + 2] = 0;
        return;
    }
    const u32 blen = (u32)(b1 - b0);
    const u8 first = blen ? v.body[b0] : 0, last = blen ? v.body[b1 - 1] : 0;
    i32 who = spk, room;
    bool home = true;
    if (SHARD) home = nutsb_speech_home(v, sh, spk, &who, &room);
    else room = v.user_room[spk] < v.n_rooms ? v.user_room[spk] : -1;
    for (u32 s = 0; s < 3; ++s) {
        SpeechSlot sl = nutsb_speech_slot(verb, s, who, room, v.sflags[spk], v.ban_swearing != 0, first, last);
        if (SHARD && !home) nutsb_speech_away(sl);
        u32 len = nutsb_speech_len(v, sl, spk, blen);
        if (len > NUTSB_MAX_TEXT) { atomicOr(status, NUTSB_ST_TEXT_TOO_LONG); len = 0; }
        slot_len[3 * j + s] = len;
    }
}

// Half a warp per message.  A message's three ops are fifteen pieces (per op: literal a | name | literal b |
// body | literal c).  Lane p of the group works out piece p -- its op's slot rule, source and length -- and
// where it lands (text_off[3m + s] + the lengths of the op's earlier pieces); the lanes that hold an op's first
// piece write the op itself (kind, target, except, flags, gate).  Then the group copies the pieces one after
// the other, all lanes on one piece.  (One warp per message with the rules evaluated op after op was 809
// instructions per message, issue-bound at 0.92 ms for 1M lines.)
// SHARD: one group per selected line j (line sel[j], ops 3j..3j+2; the gate stays the line's index in the batch).
#define NUTSB_SPEECH_GROUP 16
template <bool SHARD>
__global__ void __launch_bounds__(256)
k_speech_compose(SpeechView v, SpeechShard sh, const u64 *text_off, u8 *text, u8 *kind, i32 *target, i32 *except_user, u8 *flags, i32 *gate)
{
    constexpr int G = NUTSB_SPEECH_GROUP;
    const int lane = threadIdx.x & 31, gl = lane % G, g0 = lane - gl;
    const i64 j = ((i64)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const bool have = j < (SHARD ? sh.k : v.n);
    // -- piece gl of message m (lane 15 has none)
    const u32 s = (u32)gl / 5u, part = (u32)gl % 5u;
    const u8 *src = nullptr; u32 len = 0; u8 *dst = nullptr;
    if (have && gl < 15) {
        const i64 m = SHARD ? (i64)sh.sel[j] : j;
        const i32 spk = v.speaker[m];
        const u32 verb = v.verb[m];
        const bool ok = spk >= 0 && spk < v.n_users && verb < NUTSB_SPEECH_VERBS;
        const u64 b0 = v.body_off[m], b1 = v.body_off[m + 1];
        const u32 blen = (u32)(b1 - b0);
        const u8 first = blen ? v.body[b0] : 0, last = blen ? v.body[b1 - 1] : 0;
        i32 who = spk, room = -1;
        bool home = true;
        if (SHARD) { if (ok) home = nutsb_speech_home(v, sh, spk, &who, &room); }   // (selected lines are valid)
        else room = ok ? (v.user_room[spk] < v.n_rooms ? v.user_room[spk] : -1) : -1;
        const u32 sf = ok ? v.sflags[spk] : 0u;
        const i64 q = 3 * j + s;
        SpeechSlot sl{};
        sl.kind = NUTSB_OP_NONE; sl.target = -1; sl.except_user = -1;
        if (ok) sl = nutsb_speech_slot(verb, s, who, room, sf, v.ban_swearing != 0, first, last);
        if (SHARD && !home) nutsb_speech_away(sl);
        const u64 o0 = text_off[q];
        const u32 slen = (u32)(text_off[q + 1] - o0);
        // (a composed line over NUTSB_MAX_TEXT was measured as 0 and flagged: dropped here)
        const bool dead = sl.kind == NUTSB_OP_NONE || (slen == 0 && nutsb_speech_len(v, sl, spk, blen) != 0);
        if (part == 0) {
            kind[q] = dead ? (u8)NUTSB_OP_NONE : sl.kind;
            target[q] = sl.target; except_user[q] = sl.except_user; flags[q] = sl.flags;
            gate[q] = (!dead && sl.gated) ? (i32)m : -1;
        }
        if (!dead && slen) {
            if (part == 1) {
                if (sl.name) {
                    const bool real = sl.name == 2 || !(sf & NUTSB_SF_INVIS);
                    src = real ? v.names + v.name_off[spk] : v.lit + v.lit_off[NUTSB_LIT_INVISNAME];
                    len = real ? (u32)(v.name_off[spk + 1] - v.name_off[spk])
                               : v.lit_off[NUTSB_LIT_INVISNAME + 1] - v.lit_off[NUTSB_LIT_INVISNAME];
                }
            } else if (part == 3) {
                if (sl.body) {
                    const u32 skip = sl.body == 2 && blen ? 1u : 0u;
                    src = v.body + b0 + skip; len = blen - skip;
                }
            } else {
                const u32 li = part == 0 ? sl.a : part == 2 ? sl.b : sl.c;
                const u32 l0 = v.lit_off[li];
                src = v.lit + l0; len = v.lit_off[li + 1] - l0;
            }
            dst = text + o0;
        }
    }
    // where the piece lands: after the op's earlier pieces (the lanes just below)
    u32 before = 0;
#pragma unroll
    for (int d = 1; d < 5; ++d) { const u32 t = __shfl_up_sync(NUTSB_FULL, len, d); if (part >= (u32)d) before += t; }
    dst += before;
    // -- the group copies piece after piece
    for (int i = 0; i < 15; ++i) {
        const u32 n = __shfl_sync(NUTSB_FULL, len, g0 + i);
        const u8 *ps = (const u8 *)(size_t)__shfl_sync(NUTSB_FULL, (u64)(size_t)src, g0 + i);
        u8 *pd = (u8 *)(size_t)__shfl_sync(NUTSB_FULL, (u64)(size_t)dst, g0 + i);
        for (u32 k = (u32)gl; k < n; k += G) pd[k] = ps[k];
    }
}

// ---- recording (nutsb_set_speech_record): record(user->room, text) of say / emote / echo ----------------------
// c:4099, c:4209, c:4304.  The lines a batch records in a room go into its ring in batch order, so only the last
// REVIEW_LINES of each room can survive the batch, and of each only what strncpy keeps: its first REVIEW_LEN bytes,
// up to an embedded NUL.  The steps, all on the context's main stream (the scans and the sort share its scan state):
//   k_speech_rec_mark    key[j] = the room composed line j records in, or NUTSB_REC_NONE
//   scan (compaction)    the marked lines' rooms and line indices, in batch order, and their number
//   radix sort by room   stable: batch order within a room
//   k_speech_rec_bounds  seg[r] .. seg[r+1]: room r's records in the sorted order
//   k_speech_rec_tail    per room: the bytes strncpy keeps of its last min(c, REVIEW_LINES) records
//   scan over the rooms  where each room's record lands in the packed buffer
//   k_speech_rec_pack    per room that recorded anything:  u32 room | u32 c | u8 len[16] | the kept bytes, line after line
// The host copies the packed buffer once and applies it to the rings after the batch has been delivered.
#define NUTSB_REC_NONE 0xffffffffu
#define NUTSB_REC_HEAD 24u

// One thread per composed line j (line sel[j] of the batch in shard mode; its ops are 3j..3j+2).  Recorded: say,
// emote and echo whose room op (slot 2) is live with a room -- not muzzled, in a room, on the speaker's own shard --
// and not refused for swearing.
template <bool SHARD>
__global__ void __launch_bounds__(256)
k_speech_rec_mark(const u8 *verb, SpeechShard sh, i64 k, const u8 *kind, const i32 *target, const i32 *gate, const u8 *verdict, u32 *key)
{
    const i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const i64 m = SHARD ? (i64)sh.sel[j] : j;
    const u32 v = verb[m];
    const i64 q = 3 * j + 2;
    const i32 g = gate[q];
    const bool rec = (v == NUTSB_SPEECH_SAY || v == NUTSB_SPEECH_EMOTE || v == NUTSB_SPEECH_ECHO)
                     && kind[q] == NUTSB_OP_ROOM && target[q] >= 0 && (g < 0 || !verdict[g]);
    key[j] = rec ? (u32)target[q] : NUTSB_REC_NONE;
}

// Thread i in [0, k]: the room bounds of the *n_rec sorted keys (seg[0..n_rooms]).
__global__ void __launch_bounds__(256)
k_speech_rec_bounds(const u32 *keys, const u32 *n_rec, i64 k, u32 n_rooms, u32 *seg)
{
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > k) return;
    nutsb_seg_bounds(keys, (i64)*n_rec, i, n_rooms, seg);
}

// One warp per room, lane i on the room's i-th kept record: how many bytes strncpy takes of it.  vals[] = the sorted
// records' positions in line[] (the composed line indices in batch order).  bytes[r] = room r's size in the packed
// buffer (0: nothing recorded there).
__global__ void __launch_bounds__(256)
k_speech_rec_tail(const u32 *seg, const u32 *vals, const u32 *line, const u64 *text_off, const u8 *text, u32 n_rooms,
                  u8 *lens, u32 *bytes)
{
    const i64 r = ((i64)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const u32 lane = threadIdx.x & 31;
    if (r >= n_rooms) return;                                   // (the whole warp)
    const u32 b = seg[r + 1], c = b - seg[r], t = c < NUTSB_REVIEW_LINES ? c : NUTSB_REVIEW_LINES;
    u32 len = 0;
    if (lane < t) {
        const u64 q = 3ull * line[vals[b - t + lane]] + 2;
        const u64 o0 = text_off[q], o1 = text_off[q + 1];
        const u32 lim = o1 - o0 < NUTSB_REVIEW_LEN ? (u32)(o1 - o0) : NUTSB_REVIEW_LEN;
        const u8 *p = text + o0;
        while (len < lim && p[len]) ++len;
        lens[16 * r + lane] = (u8)len;
    }
    for (int d = 16; d; d >>= 1) len += __shfl_xor_sync(NUTSB_FULL, len, d);
    if (lane == 0) bytes[r] = c ? NUTSB_REC_HEAD + len : 0;
}

// One warp per room that recorded anything: its header and kept bytes at out + off[r].
__global__ void __launch_bounds__(256)
k_speech_rec_pack(const u32 *seg, const u32 *vals, const u32 *line, const u64 *text_off, const u8 *text, u32 n_rooms,
                  const u8 *lens, const u64 *off, u8 *out)
{
    const i64 r = ((i64)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const u32 lane = threadIdx.x & 31;
    if (r >= n_rooms) return;
    const u32 b = seg[r + 1], c = b - seg[r], t = c < NUTSB_REVIEW_LINES ? c : NUTSB_REVIEW_LINES;
    if (c == 0) return;
    u8 *dst = out + off[r];
    if (lane < NUTSB_REC_HEAD) {
        const u32 w = lane < 4 ? (u32)r : c;
        dst[lane] = lane < 8 ? (u8)(w >> (8 * (lane & 3))) : (lane - 8 < t ? lens[16 * r + lane - 8] : (u8)0);
    }
    dst += NUTSB_REC_HEAD;
    for (u32 i = 0; i < t; ++i) {
        const u32 n = lens[16 * r + i];
        const u8 *src = text + text_off[3ull * line[vals[b - t + i]] + 2];
        for (u32 x = lane; x < n; x += 32) dst[x] = src[x];
        dst += n;
    }
}
