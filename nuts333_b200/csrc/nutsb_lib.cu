// nutsb_lib.cu -- host side of libnutsb200.so: context, tables, population,
// the write pipeline's orchestration and the C-ABI of include/nutsb200.h.
//
// There is no CPU implementation of any entry point in this file: every batch
// call launches the kernels of nutsb_kernels.cuh / nutsb_match.cuh and fails
// with NUTSB_E_CUDA when no device is usable.
#include "nutsb_kernels.cuh"
#include "nutsb_match.cuh"
#include "nutsb_speech.cuh"

#define NUTSB_API extern "C" __attribute__((visibility("default")))

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <new>
#include <numeric>
#include <string>
#include <vector>

// ---------------------------------------------------------------------------------------
// buffers
// ---------------------------------------------------------------------------------------
// Each owns its memory and frees it when destroyed: nutsb_destroy makes the context's device current first.
struct DBuf {                        // growable device buffer
    void *p = nullptr; size_t cap = 0;
    DBuf() = default;
    DBuf(const DBuf &) = delete; DBuf &operator=(const DBuf &) = delete;
    ~DBuf() { if (p) cudaFree(p); }
    template <class T> T *as() const { return (T *)p; }
};
struct HBuf {                        // growable pinned host buffer
    void *p = nullptr; size_t cap = 0;
    HBuf() = default;
    HBuf(const HBuf &) = delete; HBuf &operator=(const HBuf &) = delete;
    ~HBuf() { if (p) cudaFreeHost(p); }
    template <class T> T *as() const { return (T *)p; }
};

struct AcHost {
    std::vector<u32> trans; u8 clsmap[256]; u32 ncls = 1, nstates = 1, root_match = 0;
    std::vector<u16> tr16; u8 cls2[256]; u32 thresh = 0x10000u, maxpat = 0;     // the one-byte compact form (empty: does not fit)
    std::vector<u16> t2; u16 clsA[256]; u8 clsB[256]; u32 t2_rs = 0;            // k_ac_pair's form (empty: does not fit)
};
struct AcDev { DBuf trans, clsmap, tr16, cls2, t2, clsA, clsB; AcView view{}; bool present = false; };
struct SetDev { DBuf slot_off, slot_len, pool; SetView view{}; bool present = false; };

struct ClassSet {                    // one class granularity (with / without level)
    std::vector<i32> user_cls, room_cls_off; std::vector<u8> cls_flags, cls_level;
    DBuf d_user_cls, d_room_cls_off, d_cls_flags, d_cls_level;
    i32 n_cls = 0, max_per_room = 0;
};

// An op list in host vectors (the queue; one shard's share of a routed batch).  The per-op vectors always
// have one entry per op, so the op count and the text length mark a point to roll back to.
struct HostOps {
    std::vector<u8> text; std::vector<u64> off{0}; std::vector<u8> kind, flags;
    std::vector<i32> target, except, gate;
    struct Mark { size_t n, text; };

    size_t n() const { return kind.size(); }
    void push(u8 k, i32 t, const u8 *bytes, size_t len, i32 x, u8 f, i32 g)
    {
        text.insert(text.end(), bytes, bytes + len);
        off.push_back((u64)text.size());
        kind.push_back(k); target.push_back(t); except.push_back(x); flags.push_back(f); gate.push_back(g);
    }
    Mark mark() const { return { n(), text.size() }; }
    void rollback(const Mark &m)
    {
        text.resize(m.text); off.resize(m.n + 1);
        kind.resize(m.n); target.resize(m.n); except.resize(m.n); flags.resize(m.n); gate.resize(m.n);
    }
    void clear() { rollback({ 0, 0 }); }
    // the list as a batch; gated only when given the verdicts its gates index
    nutsb_ops view(const u8 *verdict) const
    {
        static const u8 z8 = 0; static const i32 z32 = 0;
        nutsb_ops o{};
        o.n_ops = (i64)n();
        o.text = text.empty() ? &z8 : text.data(); o.text_off = off.data();
        o.kind = kind.empty() ? &z8 : kind.data(); o.flags = flags.empty() ? &z8 : flags.data();
        o.target = target.empty() ? &z32 : target.data(); o.except_user = except.empty() ? &z32 : except.data();
        if (verdict) { o.gate = gate.empty() ? &z32 : gate.data(); o.verdict = verdict; }
        return o;
    }
};

// A review buffer as the reference keeps it (a room's, nuts333.h:95; a user's revtell, nuts333.h:73): N rows of
// REVIEW_LEN+2 bytes, `line` the next row to write.  nutsb_get_review_buffer hands `buf` out as it stands.
template <int N> struct ReviewRing {
    char buf[N][NUTSB_REVIEW_LEN + 2]; int line;
    // one row as record() (c:2062) / record_tell() (c:2074) write it, given the len <= REVIEW_LEN bytes their
    // strncpy keeps: those bytes, NUL padding up to REVIEW_LEN, '\n', NUL
    void put(const void *bytes, size_t len)
    {
        char *row = buf[line];
        memcpy(row, bytes, len);
        memset(row + len, 0, NUTSB_REVIEW_LEN - len);
        row[NUTSB_REVIEW_LEN] = '\n'; row[NUTSB_REVIEW_LEN + 1] = '\0';
        line = (line + 1) % N;
    }
};

// Profiling events (nutsb_set_profiling): the points a write batch records, one meaning each.
enum Ev {
    EV_START,                   // run_write begins
    EV_RENDER0, EV_RENDER1,     // k_render
    EV_DIRECT0, EV_DIRECT1,     // the direct ops: k_direct (nothing between the two when fused into the fan-out), k_direct_compact
    EV_FAN0, EV_FAN1,           // the renderings to their recipients: k_fanout / k_fanout_direct, k_iov for gather lists
    EV_END,                     // the batch's last kernel is done
    EV_H2D0, EV_H2D1,           // the host input's copies to HBM
    EV_D2H0, EV_D2H1,           // the result's copies to pinned host memory
    EV_COUNT
};

struct nutsb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr; bool own_stream = true;
    cudaStream_t side = nullptr; bool overlap = true;     // k_render / k_direct run beside the plan / the fan-out ...
    int side_render = 8;                                  // ... with this many k_render blocks per SM
    int fd_dir_per_sm = 0;                                // k_fanout_direct: direct blocks per SM (0: one per 256 events)
    cudaEvent_t dep[4] = {nullptr, nullptr, nullptr, nullptr};
    int sm_count = 148;
    std::string err;
    bool profiling = false; nutsb_timing tm{};
    cudaEvent_t ev[EV_COUNT] = {};

    // tables
    DBuf d_codetab;
    AcDev swear, site; SetDev userban;
    bool site_file = false, user_file = false;
    std::vector<u8> ban_bytes[2];   // the two lists as they stand on disk (nutsb_ban_edit edits them)

    // population
    bool have_users = false, all_simple = true, has_clones = false;   // has_clones: some user is a clone or a remote user
    i32 n_clone_flag = 0, n_remote_flag = 0;
    i32 U = 0, R = 0, Rt = 1;
    std::vector<i32> user_room, user_slot, slot_user, room_slot_off;
    std::vector<u8> uflags, ulevel;
    std::vector<i32> remote_link; std::vector<u8> remote_old;   // per user; link -1 = not a remote user
    std::vector<i32> remotes;                                   // the remote users, in user-list order
    std::vector<i32> clone_owner; std::vector<u8> clone_hear;   // per user; owner -1 = not a clone
    std::vector<std::vector<i32>> room_clones;                  // clones of every room, in user-list order
    std::vector<std::string> room_names;                        // default "room<index>"
    DBuf d_user_room, d_user_slot, d_slot_user, d_room_slot_off, d_slot_cf, d_slot_lv;
    ClassSet cls[2];                 // [0] keyed without level, [1] with level

    // per-batch scratch
    DBuf d_status, d_len_on, d_len_off, d_nrep, d_eoff, d_sums, d_scan_ticket;
    void *scan_state_seen = nullptr; size_t scan_state_cap = 0; u32 scan_epoch = 0;      // k_scan1's per-tile state: flags carry the scan's epoch
    DBuf d_ek[2], d_ev_[2];          // (room, op) entries, ping-pong
    DBuf d_hist, d_hoffs;
    DBuf d_room_ent_off, d_e_info, d_e_delta, d_e_slot, d_e_scan, d_counts, d_room_b_off;
    DBuf d_bl_op, d_bl_room, d_evk[2], d_evv[2], d_ev_ukey, d_ev_delta, d_ev_op;
    DBuf d_sv_ukey, d_sv_delta, d_sv_op, d_sv_pre, d_ev_off;
    DBuf d_vp_on, d_vp_off, d_cp;
    DBuf d_room_tile_off, d_room_cell_off, d_room_item_off, d_counters;
    DBuf d_runs, d_items, d_slab, d_bl_meta, d_slots;
    DBuf d_off, d_out, d_digest;
    DBuf d_dpre, d_dir, d_iov, d_iov_first, d_iov_cnt;           // gather-list mode (nutsb_write_batch_iov)
    HBuf h_small, h_off, h_out, h_dir, h_iov, h_iov_first, h_iov_cnt;
    u64 last_total = 0; bool have_streams = false;
    // what nutsb_delivery_digests needs of the last write batch (its arrays stay in the scratch buffers until the next one)
    struct LastBatch { bool valid = false; OpsView ops{}; ClassPrefix cpx{}; bool has_level = false; u64 off_base = 0; u32 *sv_slot = nullptr; } last;
    DBuf d_room_users, d_room_users_off, d_dg;

    // staging for the host-buffer entry points
    DBuf s_text, s_toff, s_kind, s_target, s_except, s_flags, s_gate, s_verdict, s_v8;

    // speech: user names / flags, the callers' literals
    bool have_names = false; bool ban_swearing = false;
    std::vector<u8> names, sflags; std::vector<u64> name_off;
    std::vector<std::string> lits;
    DBuf d_names, d_name_off, d_sflags, d_lit, d_lit_off;
    DBuf d_sp_len, d_sp_off, d_sp_text, d_sp_kind, d_sp_target, d_sp_except, d_sp_flags, d_sp_gate, d_sp_verdict;
    DBuf s_verb, s_speaker, s_body, s_boff;
    // the shard mode of the speech batch (nutsb_multi): this context is shard `shard`; the global population's tables
    // (nutsb_multi_set_users / nutsb_multi_set_user_names) and the lines it selects from a batch
    i32 shard = -1, g_U = 0; bool have_g_names = false;
    DBuf d_g_user_shard, d_g_user_local, d_g_has_room, d_g_names, d_g_name_off, d_g_sflags, d_sp_keep, d_sp_sel;

    // queue tier
    HostOps q;
    std::vector<u8> q_sw_text; std::vector<u64> q_sw_off{0};     // bodies whose swear verdict gates queued ops
    std::vector<u8> q_sw_verdict;                                // ... their verdicts, once taken (flush / review)

    // review buffers, host state of the queue tier
    struct PendingRec { i32 room, gate; std::string text; };
    std::vector<ReviewRing<NUTSB_REVTELL_LINES>> revtell;        // per user
    std::vector<ReviewRing<NUTSB_REVIEW_LINES>> rev;             // per room
    std::vector<PendingRec> q_rec;                               // record() calls whose line may still be refused (swearing)
    // the speech batch's records (nutsb_set_speech_record): k_speech_rec_* scratch, the packed records on the host
    bool speech_record = false, rec_ready = false; u64 rec_total = 0;
    DBuf d_rec_key, d_rec_line, d_rec_k[2], d_rec_v[2], d_rec_cnt, d_rec_seg, d_rec_lens, d_rec_bytes, d_rec_off, d_rec_out;
    HBuf h_rec;
};

static int fail(nutsb_ctx *c, int code, const char *fmt, const char *a = "")
{
    if (c) { char b[512]; snprintf(b, sizeof b, fmt, a); c->err = b; }
    return code;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) \
    return fail(c, e_ == cudaErrorMemoryAllocation ? NUTSB_E_NOMEM : NUTSB_E_CUDA, #call ": %s", cudaGetErrorString(e_)); } while (0)
#define CKL() CK(cudaGetLastError())
#define TRY(x) do { int r_ = (x); if (r_ != NUTSB_OK) return r_; } while (0)

static int ev_record(nutsb_ctx *c, Ev e, cudaStream_t s)        // a profiling event, when profiling is on
{
    if (c->profiling) CK(cudaEventRecord(c->ev[e], s));
    return NUTSB_OK;
}
static int ev_elapsed(nutsb_ctx *c, float *ms, Ev a, Ev b) { CK(cudaEventElapsedTime(ms, c->ev[a], c->ev[b])); return NUTSB_OK; }

static int ensure(nutsb_ctx *c, DBuf &b, size_t bytes)
{
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes + 256 <= b.cap) return NUTSB_OK;
    if (b.p) { CK(cudaStreamSynchronize(c->stream)); CK(cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 512;             // slack: fewer re-allocations, readable padding
    CK(cudaMalloc(&b.p, want));
    b.cap = want;
    return NUTSB_OK;
}
static int ensure_host(nutsb_ctx *c, HBuf &b, size_t bytes)
{
    if (bytes + 64 <= b.cap) return NUTSB_OK;
    if (b.p) { CK(cudaStreamSynchronize(c->stream)); CK(cudaFreeHost(b.p)); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 4096;
    CK(cudaHostAlloc(&b.p, want, cudaHostAllocDefault));
    b.cap = want;
    return NUTSB_OK;
}

static int upload(nutsb_ctx *c, DBuf &b, const void *src, size_t bytes)
{
    TRY(ensure(c, b, bytes ? bytes : 1));
    if (bytes) CK(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return NUTSB_OK;
}

static inline u32 cdiv(u64 a, u64 b) { return (u32)((a + b - 1) / b); }
static inline u32 bits_for(u64 n) { u32 b = 0; while (b < 32 && (1ull << b) < n) ++b; return b; }

// ---------------------------------------------------------------------------------------
// scan / sort drivers
// ---------------------------------------------------------------------------------------
struct InU32 { const u32 *p; __device__ u64 operator()(i64 i) const { return p[i]; } };
struct InU64 { const u64 *p; __device__ u64 operator()(i64 i) const { return p[i]; } };
struct InI32 { const i32 *p; __device__ u64 operator()(i64 i) const { return (u64)(i64)p[i]; } };
struct InU8 { const u8 *p; __device__ u64 operator()(i64 i) const { return p[i]; } };
// compaction: the indices i < n with keep[i] set, in order, into sel[]; their number into sel[n]
struct OutSel {
    const u8 *keep; i32 *sel; i64 n;
    __device__ void operator()(i64 i, u64 ex) const { if (i == n) sel[n] = (i32)ex; else if (keep[i]) sel[ex] = (i32)i; }
};
struct OutU64 { u64 *p; __device__ void operator()(i64 i, u64 ex) const { p[i] = ex; } };
// the speech batch's records (k_speech_rec_mark's keys): the marked lines' rooms and indices in order, their number
struct InRecKey { const u32 *key; __device__ u64 operator()(i64 i) const { return key[i] != NUTSB_REC_NONE; } };
struct OutRec {
    const u32 *key; u32 *room, *line, *count; i64 n;
    __device__ void operator()(i64 i, u64 ex) const { if (i == n) *count = (u32)ex; else if (key[i] != NUTSB_REC_NONE) { room[ex] = key[i]; line[ex] = (u32)i; } }
};
struct InEntryPacked {
    const u8 *info;
    __device__ u64 operator()(i64 i) const { const u32 f = info[i]; return (u64)(f & 1u) | ((u64)((f >> 1) != 0) << 32); }
};
struct InSlabLen { const u32 *len, *bl_op; __device__ u64 operator()(i64 g) const { return len[bl_op[g]]; } };
struct InSlabLen2 {                 // both settings in one scan: low word colour on, high word colour off
    const u32 *len_on, *len_off, *bl_op;
    __device__ u64 operator()(i64 g) const { const u32 op = bl_op[g]; return (u64)len_on[op] | ((u64)len_off[op] << 32); }
};
struct OutSplit { u64 *a, *b; __device__ void operator()(i64 i, u64 ex) const { a[i] = (u32)ex; b[i] = ex >> 32; } };
struct InClassLen {                 // bytes class column j receives from slab op g
    OpsView ops; const u32 *bl_op, *bl_room, *len_on, *len_off;
    const i32 *room_cls_off; const u8 *cls_flags, *cls_level; i32 j;
    __device__ u64 operator()(i64 g) const
    {
        const u32 room = bl_room[g], op = bl_op[g];
        const i32 k = room_cls_off[room] + j;
        if (k >= room_cls_off[room + 1]) return 0;
        const u32 cf = cls_flags[k];
        if (!nutsb_class_delivers(cf, cls_level[k], ops.kind[op], ops.flags[op], ops.target[op])) return 0;
        return (cf & NUTSB_UF_COLOUR) ? len_on[op] : len_off[op];
    }
};

// Exclusive scan of in(0..n) into out(0..n) (out(n) = total).  n = *n_dev when given.  One launch (k_scan1).
template <class In, class Out>
static int run_scan(nutsb_ctx *c, In in, Out out, i64 n_upper, const u32 *n_dev)
{
    const bool small = (u64)n_upper + 1 <= 16384u;                 // 64 tiles of 256: one look-back window
    const u32 nb = cdiv((u64)n_upper + 1, small ? NUTSB_SCAN_THREADS : NUTSB_SCAN_TILE);
    TRY(ensure(c, c->d_sums, ((size_t)nb + 1) * sizeof(ScanState)));
    if (!c->d_scan_ticket.p) { TRY(ensure(c, c->d_scan_ticket, 64)); CK(cudaMemsetAsync(c->d_scan_ticket.p, 0, 64, c->stream)); }
    if (c->d_sums.p != c->scan_state_seen || c->d_sums.cap != c->scan_state_cap) {     // a fresh (re)allocation: whatever it holds must not look like a flag
        CK(cudaMemsetAsync(c->d_sums.p, 0, c->d_sums.cap, c->stream));
        c->scan_state_seen = c->d_sums.p; c->scan_state_cap = c->d_sums.cap;
    }
    if (++c->scan_epoch >= 0x3fffffffu) { c->scan_epoch = 1; CK(cudaMemsetAsync(c->d_sums.p, 0, c->d_sums.cap, c->stream)); }
    if (small) {
        auto k1 = k_scan1<In, Out, 1>;
        NUTSB_LAUNCH(nb, NUTSB_SCAN_THREADS, c->stream, k1, in, out, n_upper, n_dev, c->d_sums.as<ScanState>(), c->d_scan_ticket.as<u32>(), c->scan_epoch, nb); CKL();
    } else {
        auto k1 = k_scan1<In, Out, NUTSB_SCAN_ITEMS>;
        NUTSB_LAUNCH(nb, NUTSB_SCAN_THREADS, c->stream, k1, in, out, n_upper, n_dev, c->d_sums.as<ScanState>(), c->d_scan_ticket.as<u32>(), c->scan_epoch, nb); CKL();
    }
    c->tm.launches += 1;
    return NUTSB_OK;
}

// Stable LSD radix sort of (key, val) pairs from kb[0] / vb[0].  On return *keys / *vals point at
// the sorted arrays (one of the two ping-pong buffers).  vals start as iota unless vals_given.
static int radix_sort(nutsb_ctx *c, DBuf kb[2], DBuf vb[2], i64 n_upper, const u32 *n_dev, u32 key_bits,
                      u32 **keys, u32 **vals, bool vals_given = false)
{
    const u32 passes = key_bits ? cdiv(key_bits, NUTSB_RS_BITS) : 1;
    const u32 bits = std::max(1u, cdiv(key_bits, passes));            // digit width: passes balanced, tables small
    const u32 nblk = cdiv((u64)(n_upper > 0 ? n_upper : 1), NUTSB_RS_CHUNK);
    const size_t hn = ((size_t)1 << bits) * nblk;
    TRY(ensure(c, c->d_hist, hn * sizeof(u32)));
    TRY(ensure(c, c->d_hoffs, (hn + 1) * sizeof(u64)));
    for (int q = 0; q < 2; ++q) { TRY(ensure(c, kb[q], (size_t)n_upper * 4 + 16)); TRY(ensure(c, vb[q], (size_t)n_upper * 4 + 16)); }
    int cur = 0;
    for (u32 p = 0; p < passes; ++p) {
        const int shift = (int)(p * bits);
        NUTSB_LAUNCH(nblk, NUTSB_RS_THREADS, c->stream, k_rs_hist, kb[cur].as<u32>(), n_upper, n_dev, shift, bits,
                     c->d_hist.as<u32>(), nblk); CKL();
        TRY(run_scan(c, InU32{c->d_hist.as<u32>()}, OutU64{c->d_hoffs.as<u64>()}, (i64)hn, nullptr));
        NUTSB_LAUNCH(nblk, NUTSB_RS_THREADS, c->stream, k_rs_scatter, kb[cur].as<u32>(),
                     p == 0 && !vals_given ? (const u32 *)nullptr : vb[cur].as<u32>(), n_upper, n_dev, shift, bits,
                     c->d_hoffs.as<u64>(), nblk, kb[cur ^ 1].as<u32>(), vb[cur ^ 1].as<u32>()); CKL();
        c->tm.launches += 2;
        cur ^= 1;
    }
    *keys = kb[cur].as<u32>(); *vals = vb[cur].as<u32>();
    return NUTSB_OK;
}

// ---------------------------------------------------------------------------------------
// tables
// ---------------------------------------------------------------------------------------
static void build_codetab(u8 *tab)
{
    // nuts333.h:248-254, in table order (the index selects the ANSI string)
    static const char *codes = "RSOLULLIRVFKFRFGFYFBFMFTFWBKBRBGBYBBBMBTBW";
    memset(tab, 0, NUTSB_CODETAB_BYTES);
    for (int k = 0; k < 21; ++k) tab[(codes[2 * k] - 'A') * 26 + (codes[2 * k + 1] - 'A')] = (u8)(k + 1);
}

// Aho-Corasick automaton with full transitions, byte classes, match bit in bit 31.
static void build_ac(const std::vector<std::string> &pats, bool fold_case, AcHost &ac)
{
    u8 word_cls[256]; memset(word_cls, 0, sizeof word_cls);
    ac.ncls = 1; ac.root_match = 0;
    size_t total = 1;
    for (auto &p : pats) {
        if (p.empty()) ac.root_match = 1;
        total += p.size();
        for (unsigned char b : p) if (!word_cls[b]) word_cls[b] = (u8)ac.ncls++;
    }
    for (int b = 0; b < 256; ++b) {
        int f = (fold_case && b >= 'A' && b <= 'Z') ? b + 32 : b;
        ac.clsmap[b] = word_cls[f];
    }
    const u32 nc = ac.ncls;
    std::vector<i32> go(total * nc, -1);
    std::vector<u8> match(total, 0);
    u32 ns = 1;
    for (auto &p : pats) {
        u32 s = 0;
        for (unsigned char b : p) {
            i32 &nx = go[(size_t)s * nc + word_cls[b]];
            if (nx < 0) nx = (i32)ns++;
            s = (u32)nx;
        }
        if (!p.empty()) match[s] = 1;
    }
    std::vector<u32> failv(ns, 0), queue; queue.reserve(ns);
    for (u32 ccls = 0; ccls < nc; ++ccls) {
        i32 &nx = go[ccls];
        if (nx < 0) nx = 0; else { failv[nx] = 0; queue.push_back((u32)nx); }
    }
    for (size_t qi = 0; qi < queue.size(); ++qi) {
        const u32 s = queue[qi];
        match[s] |= match[failv[s]];
        for (u32 ccls = 0; ccls < nc; ++ccls) {
            i32 &nx = go[(size_t)s * nc + ccls];
            const u32 via = (u32)go[(size_t)failv[s] * nc + ccls];
            if (nx < 0) nx = (i32)via; else { failv[nx] = via; queue.push_back((u32)nx); }
        }
    }
    ac.nstates = ns;
    ac.trans.resize((size_t)ns * nc);
    for (size_t i = 0; i < (size_t)ns * nc; ++i) {
        const u32 t = (u32)go[i];
        ac.trans[i] = t | (match[t] ? 0x80000000u : 0u);
    }
    // the one-byte compact form: states renumbered with the match states last (the root stays 0: it is a match state only for an
    // empty pattern, which root_match covers), entries = byte offset of the target's row, classes pre-doubled
    ac.tr16.clear(); ac.maxpat = 0; ac.thresh = 0x10000u;
    for (auto &p : pats) ac.maxpat = std::max<u32>(ac.maxpat, (u32)p.size());
    if ((size_t)ns * nc <= NUTSB_AC_SMEM_ENTRIES && nc <= 127 && (size_t)ns * nc * 2 <= 0xffffu) {
        std::vector<u32> newid(ns, 0); u32 k = 0;
        for (u32 st = 0; st < ns; ++st) if (!match[st] || st == 0) newid[st] = k++;
        ac.thresh = k == ns ? 0x10000u : k * nc * 2;              // (no match state at all: never reached)
        for (u32 st = 1; st < ns; ++st) if (match[st]) newid[st] = k++;
        ac.tr16.assign((size_t)ns * nc, 0);
        for (u32 st = 0; st < ns; ++st)
            for (u32 cc = 0; cc < nc; ++cc) ac.tr16[(size_t)newid[st] * nc + cc] = (u16)(newid[(u32)go[(size_t)st * nc + cc]] * nc * 2);
        for (int b = 0; b < 256; ++b) ac.cls2[b] = (u8)(2 * ac.clsmap[b]);
    }
    // k_ac_pair's form: the table squared (two bytes a step), rows padded to a power of two so that row | column is the
    // entry's byte offset; bits 14 / 15 of an entry flag a match state after the first / the second byte.  It leans on
    // the one-byte form for its second looks, and has to fit 16 KB (14 bits of row offset).
    ac.t2.clear(); ac.t2_rs = 0;
    if (!ac.tr16.empty()) {
        u32 rs = 4; while (rs < 2 * nc * nc) rs <<= 1;
        if ((u64)ns * rs <= 0x4000u) {
            ac.t2_rs = rs;
            ac.t2.assign((size_t)ns * (rs / 2), 0);
            for (u32 st = 0; st < ns; ++st)
                for (u32 a = 0; a < nc; ++a) {
                    const u32 mid = (u32)go[(size_t)st * nc + a];
                    for (u32 b = 0; b < nc; ++b) {
                        const u32 fin = (u32)go[(size_t)mid * nc + b];
                        ac.t2[(size_t)st * (rs / 2) + a * nc + b] = (u16)(fin * rs | (mid && match[mid] ? 0x4000u : 0u) | (fin && match[fin] ? 0x8000u : 0u));
                    }
                }
            for (int b = 0; b < 256; ++b) { ac.clsA[b] = (u16)(2 * nc * ac.clsmap[b]); ac.clsB[b] = (u8)(2 * ac.clsmap[b]); }
        }
    }
}

static int upload_ac(nutsb_ctx *c, const AcHost &h, AcDev &d)
{
    TRY(upload(c, d.trans, h.trans.data(), h.trans.size() * sizeof(u32)));
    TRY(upload(c, d.clsmap, h.clsmap, 256));
    d.view.trans = d.trans.as<u32>(); d.view.clsmap = d.clsmap.as<u8>();
    d.view.ncls = h.ncls; d.view.nstates = h.nstates; d.view.root_match = h.root_match;
    d.view.tr16 = nullptr; d.view.cls2 = nullptr; d.view.thresh = h.thresh; d.view.maxpat = h.maxpat;
    if (!h.tr16.empty()) {
        TRY(upload(c, d.tr16, h.tr16.data(), h.tr16.size() * sizeof(u16)));
        TRY(upload(c, d.cls2, h.cls2, 256));
        d.view.tr16 = d.tr16.as<u16>(); d.view.cls2 = d.cls2.as<u8>();
    }
    d.view.t2 = nullptr; d.view.clsA = nullptr; d.view.clsB = nullptr; d.view.t2_rs = h.t2_rs;
    if (!h.t2.empty()) {
        TRY(upload(c, d.t2, h.t2.data(), h.t2.size() * sizeof(u16)));
        TRY(upload(c, d.clsA, h.clsA, sizeof h.clsA));
        TRY(upload(c, d.clsB, h.clsB, 256));
        d.view.t2 = d.t2.as<u16>(); d.view.clsA = d.clsA.as<u16>(); d.view.clsB = d.clsB.as<u8>();
    }
    d.present = true;
    CK(cudaStreamSynchronize(c->stream));
    return NUTSB_OK;
}

// The fscanf("%s") / feof loop of nuts333.c:338-342 applied to file bytes: a
// token is tested only when the scan that read it stopped on a whitespace byte.
// Tokens reach strstr/strcmp as C strings, i.e. cut at an embedded NUL.
static int ban_tokens(nutsb_ctx *c, const u8 *f, size_t n, std::vector<std::string> &out)
{
    auto ws = [](u8 b) { return b == ' ' || (b >= 9 && b <= 13); };
    size_t p = 0;
    while (true) {
        while (p < n && ws(f[p])) ++p;
        if (p >= n) break;
        const size_t b = p;
        while (p < n && !ws(f[p])) ++p;
        if (p >= n) break;                          // ran into EOF: feof() already true, never tested
        if (p - b > NUTSB_MAX_BAN_TOKEN) return fail(c, NUTSB_E_RANGE, "ban token longer than 81 bytes%s");
        size_t m = 0; while (m < p - b && f[b + m]) ++m;
        out.emplace_back((const char *)f + b, m);
    }
    return NUTSB_OK;
}

// ---------------------------------------------------------------------------------------
// C-ABI: lifecycle
// ---------------------------------------------------------------------------------------
NUTSB_API int nutsb_version(void) { return NUTSB_VERSION; }

NUTSB_API const char *nutsb_strerror(int code)
{
    switch (code) {
    case NUTSB_OK: return "ok";
    case NUTSB_E_INVAL: return "invalid argument";
    case NUTSB_E_NOMEM: return "out of memory";
    case NUTSB_E_CUDA: return "CUDA error";
    case NUTSB_E_UNSUPPORTED: return "unsupported recipient type (remote)";
    case NUTSB_E_RANGE: return "value out of range";
    case NUTSB_E_STATE: return "call order";
    }
    return "unknown";
}
NUTSB_API const char *nutsb_last_error(const nutsb_ctx *c) { return c ? c->err.c_str() : ""; }

NUTSB_API void nutsb_destroy(nutsb_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (auto &e : c->ev) if (e) cudaEventDestroy(e);
    for (auto &e : c->dep) if (e) cudaEventDestroy(e);
    if (c->side) { cudaStreamSynchronize(c->side); cudaStreamDestroy(c->side); }
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;                                                   // (the buffers free themselves)
}

static int set_swear_impl(nutsb_ctx *c, const char *const *words)
{
    std::vector<std::string> pats;
    for (size_t i = 0; words && words[i] && words[i][0] != '*'; ++i) pats.emplace_back(words[i]);
    AcHost h; build_ac(pats, true, h);
    return upload_ac(c, h, c->swear);
}

NUTSB_API int nutsb_create(nutsb_ctx **out, int device)
{
    if (!out) return NUTSB_E_INVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return NUTSB_E_CUDA;
    nutsb_ctx *c = new (std::nothrow) nutsb_ctx;
    if (!c) return NUTSB_E_NOMEM;
    c->device = device;
    int rc = [&]() -> int {
        CK(cudaSetDevice(device));
        // the main stream at the highest priority, the side stream at the lowest: k_render runs BESIDE the planning
        // kernels (small grids, bound by their own latency) -- when both have blocks waiting the planner's go first,
        // the renderer fills what is left
        int prio_least = 0, prio_greatest = 0;
        CK(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
        CK(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_greatest));
        CK(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
        CK(cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, prio_least));
        if (const char *e = getenv("NUTSB_SIDE_RENDER")) c->side_render = std::max(1, atoi(e));     // tuning aids
        if (const char *e = getenv("NUTSB_OVERLAP")) c->overlap = atoi(e) != 0;
        if (const char *e = getenv("NUTSB_FD_DIR_PER_SM")) c->fd_dir_per_sm = std::max(0, atoi(e));
        for (auto &e : c->ev) CK(cudaEventCreate(&e));
        for (auto &e : c->dep) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CK(cudaFuncSetAttribute(k_fanout, cudaFuncAttributeMaxDynamicSharedMemorySize, NUTSB_FAN_SMEM));
        CK(cudaFuncSetAttribute(k_fanout_direct, cudaFuncAttributeMaxDynamicSharedMemorySize, NUTSB_FD_SMEM));
        CK(cudaFuncSetAttribute(k_direct, cudaFuncAttributeMaxDynamicSharedMemorySize, NUTSB_DIR_SMEM));
        CK(cudaFuncSetAttribute(k_ac_pair<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, NUTSB_ACP_SMEM(0x4000)));
        CK(cudaFuncSetAttribute(k_ac_pair<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, NUTSB_ACP_SMEM(2 * NUTSB_AC_SMEM_ENTRIES)));
        u8 tab[NUTSB_CODETAB_BYTES]; build_codetab(tab);
        TRY(upload(c, c->d_codetab, tab, sizeof tab));
        TRY(ensure(c, c->d_status, 64)); TRY(ensure(c, c->d_counts, 64));
        TRY(ensure(c, c->d_counters, 1024));
        TRY(ensure_host(c, c->h_small, 4096));
        {   // the callers' literals (nutsb_speech.cuh)
            c->lits.assign(NUTSB_NLIT, std::string());
#define NUTSB_LIT_X(id, text) c->lits[id] = std::string(text, sizeof(text) - 1);
            NUTSB_SPEECH_LITERALS(NUTSB_LIT_X)
#undef NUTSB_LIT_X
            std::vector<u8> bytes; std::vector<u32> off(NUTSB_NLIT + 1, 0);
            for (int i = 0; i < NUTSB_NLIT; ++i) { bytes.insert(bytes.end(), c->lits[i].begin(), c->lits[i].end()); off[i + 1] = (u32)bytes.size(); }
            TRY(upload(c, c->d_lit, bytes.data(), bytes.size()));
            TRY(upload(c, c->d_lit_off, off.data(), off.size() * 4));
            CK(cudaStreamSynchronize(c->stream));
        }
        static const char *stock[] = { "fuck", "shit", "cunt", "*" };      // nuts333.h:275-277
        TRY(set_swear_impl(c, stock));
        CK(cudaStreamSynchronize(c->stream));
        return NUTSB_OK;
    }();
    if (rc != NUTSB_OK) { nutsb_destroy(c); return rc; }
    *out = c;
    return NUTSB_OK;
}

NUTSB_API int nutsb_set_profiling(nutsb_ctx *c, int on) { if (!c) return NUTSB_E_INVAL; c->profiling = on != 0; return NUTSB_OK; }
NUTSB_API int nutsb_set_overlap(nutsb_ctx *c, int on) { if (!c) return NUTSB_E_INVAL; c->overlap = on != 0; return NUTSB_OK; }
NUTSB_API int nutsb_get_timing(const nutsb_ctx *c, nutsb_timing *out) { if (!c || !out) return NUTSB_E_INVAL; *out = c->tm; return NUTSB_OK; }
NUTSB_API int nutsb_set_stream(nutsb_ctx *c, void *s)
{
    if (!c) return NUTSB_E_INVAL;
    CK(cudaStreamSynchronize(c->stream));
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    c->stream = (cudaStream_t)s; c->own_stream = false;
    return NUTSB_OK;
}

// ---------------------------------------------------------------------------------------
// C-ABI: tables and population
// ---------------------------------------------------------------------------------------
NUTSB_API int nutsb_set_swear_words(nutsb_ctx *c, const char *const *words)
{
    if (!c) return NUTSB_E_INVAL;
    CK(cudaSetDevice(c->device));
    return set_swear_impl(c, words);
}

static int set_ban_files_impl(nutsb_ctx *c, const void *siteban, size_t sn, const void *userban, size_t un)
{
    CK(cudaSetDevice(c->device));
    std::vector<std::string> st, ut;
    if (siteban) TRY(ban_tokens(c, (const u8 *)siteban, sn, st));
    if (userban) TRY(ban_tokens(c, (const u8 *)userban, un, ut));
    c->site_file = siteban != nullptr; c->user_file = userban != nullptr;
    // (the vectors may be the very buffers passed in: nutsb_ban_edit)
    if ((const void *)c->ban_bytes[0].data() != siteban || !siteban) c->ban_bytes[0].assign((const u8 *)siteban, (const u8 *)siteban + (siteban ? sn : 0));
    if ((const void *)c->ban_bytes[1].data() != userban || !userban) c->ban_bytes[1].assign((const u8 *)userban, (const u8 *)userban + (userban ? un : 0));
    { AcHost h; build_ac(st, false, h); TRY(upload_ac(c, h, c->site)); }
    // exact-match set
    u32 nslots = 1; while (nslots < 2 * ut.size() + 1) nslots <<= 1;
    std::vector<u32> so(nslots, 0xffffffffu), sl(nslots, 0); std::vector<u8> pool;
    for (auto &t : ut) {
        u32 h = 0x811c9dc5u; for (unsigned char b : t) { h ^= b; h *= 0x01000193u; }
        h &= nslots - 1;
        while (so[h] != 0xffffffffu) h = (h + 1) & (nslots - 1);
        so[h] = (u32)pool.size(); sl[h] = (u32)t.size();
        pool.insert(pool.end(), t.begin(), t.end());
    }
    pool.push_back(0);
    TRY(upload(c, c->userban.slot_off, so.data(), so.size() * 4));
    TRY(upload(c, c->userban.slot_len, sl.data(), sl.size() * 4));
    TRY(upload(c, c->userban.pool, pool.data(), pool.size()));
    c->userban.view.slot_off = c->userban.slot_off.as<u32>(); c->userban.view.slot_len = c->userban.slot_len.as<u32>();
    c->userban.view.pool = c->userban.pool.as<u8>(); c->userban.view.mask = nslots - 1;
    c->userban.view.count = (u32)ut.size(); c->userban.present = true;
    CK(cudaStreamSynchronize(c->stream));
    return NUTSB_OK;
}

NUTSB_API int nutsb_set_ban_files(nutsb_ctx *c, const void *siteban, size_t sn, const void *userban, size_t un)
{
    if (!c) return NUTSB_E_INVAL;
    return set_ban_files_impl(c, siteban, sn, userban, un);
}

// Ban-list maintenance, nuts333.c:6216-6429, on the lists the context holds: ban_site / ban_user
// (add = 1) append "token\n" unless a TESTED token equals it; unban_site / unban_user (add = 0)
// rewrite the list without it -- every tested token as "token\n", the last token dropped when it ran
// into EOF (the same feof() loop as site_banned), an emptied list removed.  The matchers in HBM are
// rebuilt at once.  *result: 0 done, 1 nothing to do ("already banned" / "not currently banned").
NUTSB_API int nutsb_ban_edit(nutsb_ctx *c, int which, int add, const char *token, int *result)
{
    if (!c || !token || !result || which < 0 || which > 1) return NUTSB_E_INVAL;
    std::string tok(token);
    if (tok.empty() || tok.size() > (which ? 12u : 79u)) return fail(c, NUTSB_E_RANGE, "ban token length (site < 80, user <= 12: the reference's buffers)%s");
    for (unsigned char b : tok) if (b == ' ' || (b >= 9 && b <= 13)) return fail(c, NUTSB_E_INVAL, "ban token holds white space%s");
    if (which && tok[0] >= 'a' && tok[0] <= 'z') tok[0] = (char)(tok[0] - 32);      // c:6269, c:6402
    const bool present = which ? c->user_file : c->site_file;
    const std::vector<u8> &f = c->ban_bytes[which];
    *result = 1;
    if (!present && !add) return NUTSB_OK;                          // c:6349
    std::vector<std::string> tested;
    if (present) TRY(ban_tokens(c, f.data(), f.size(), tested));
    std::vector<u8> nf; bool npresent = true;
    if (add) {
        for (auto &t : tested) if (t == tok) return NUTSB_OK;       // c:6234: "already banned"
        nf = present ? f : std::vector<u8>();
        nf.insert(nf.end(), tok.begin(), tok.end()); nf.push_back('\n');              // c:6250, fopen("a")
    } else {
        bool found = false;
        for (auto &t : tested) {
            if (t == tok) { found = true; continue; }
            nf.insert(nf.end(), t.begin(), t.end()); nf.push_back('\n');               // c:6361
        }
        if (!found) return NUTSB_OK;                                // c:6369
        npresent = !nf.empty();                                     // c:6375: an emptied list is unlinked
    }
    *result = 0;
    std::vector<u8> other = c->ban_bytes[which ^ 1];
    const bool opresent = which ? c->site_file : c->user_file;
    const void *sp = which ? (opresent ? (const void *)other.data() : nullptr) : (npresent ? (const void *)nf.data() : nullptr);
    const void *up = which ? (npresent ? (const void *)nf.data() : nullptr) : (opresent ? (const void *)other.data() : nullptr);
    static const u8 none = 0;                                       // an existing but empty file is not NULL
    if (!which && npresent && nf.empty()) sp = &none;
    if (which && npresent && nf.empty()) up = &none;
    if (!which && opresent && other.empty()) up = &none;
    if (which && opresent && other.empty()) sp = &none;
    return set_ban_files_impl(c, sp, which ? other.size() : nf.size(), up, which ? nf.size() : other.size());
}

// The list as it stands (what the talker writes back to datafiles/siteban | userban).  *present = 0: no file.
NUTSB_API int nutsb_get_ban_file(nutsb_ctx *c, int which, const void **bytes, size_t *len, int *present)
{
    if (!c || !bytes || !len || !present || which < 0 || which > 1) return NUTSB_E_INVAL;
    *present = (which ? c->user_file : c->site_file) ? 1 : 0;
    *bytes = c->ban_bytes[which].data(); *len = *present ? c->ban_bytes[which].size() : 0;
    return NUTSB_OK;
}

static int build_classes(nutsb_ctx *c, ClassSet &cs, bool with_level, const std::vector<i32> &order,
                         const u8 *flags, const u8 *level)
{
    const i32 U = c->U, Rt = c->Rt;
    cs.user_cls.assign(U, 0); cs.room_cls_off.assign(Rt + 1, 0); cs.cls_flags.clear(); cs.cls_level.clear();
    i32 prev_room = -1; u32 prev_key = 0xffffffffu; i32 k = -1;
    std::vector<i32> per_room(Rt, 0);
    for (i32 s = 0; s < U; ++s) {
        const i32 u = order[s], r = c->user_room[u];
        const u32 key = (u32)(flags[u] & 0x3f) | (with_level ? (u32)level[u] << 8 : 0u);
        if (r != prev_room || key != prev_key) {
            ++k; cs.cls_flags.push_back((u8)(flags[u] & 0x3f)); cs.cls_level.push_back(with_level ? level[u] : 0);
            per_room[r]++; prev_room = r; prev_key = key;
        }
        cs.user_cls[u] = k;
    }
    cs.n_cls = k + 1; cs.max_per_room = 0;
    for (i32 r = 0; r < Rt; ++r) { cs.room_cls_off[r + 1] = cs.room_cls_off[r] + per_room[r]; cs.max_per_room = std::max(cs.max_per_room, per_room[r]); }
    TRY(upload(c, cs.d_user_cls, cs.user_cls.data(), (size_t)U * 4));
    TRY(upload(c, cs.d_room_cls_off, cs.room_cls_off.data(), (size_t)(Rt + 1) * 4));
    TRY(upload(c, cs.d_cls_flags, cs.cls_flags.data(), cs.cls_flags.size()));
    TRY(upload(c, cs.d_cls_level, cs.cls_level.data(), cs.cls_level.size()));
    return NUTSB_OK;
}

static int set_users_impl(nutsb_ctx *c, int32_t n_users, int32_t n_rooms, const int32_t *room,
                          const uint8_t *flags, const uint8_t *level, const int32_t *prev_index)
{
    if (!c || n_users < 0 || n_rooms < 0 || (n_users && (!room || !flags || !level))) return fail(c, NUTSB_E_INVAL, "nutsb_set_users: bad argument%s");
    CK(cudaSetDevice(c->device));
    for (i32 u = 0; u < n_users; ++u) {
        if (room[u] >= n_rooms || room[u] < -1) return fail(c, NUTSB_E_RANGE, "user room out of range%s");
    }
    // queued ops name users and rooms by their index in the population they were queued under: a new
    // population may only come in between two flushes
    if (c->q.n() || !c->q_rec.empty())
        return fail(c, NUTSB_E_STATE, "nutsb_set_users with ops still queued: flush first%s");
    c->have_users = false; c->have_streams = false;
    // review buffers live as long as their room / user does (the reference clears them in create_room c:2799,
    // create_user c:2747 and clear_revbuff c:2626 only): room r keeps buffer r; user u keeps the buffer of
    // prev_index[u] (nutsb_set_users_remap), index u itself without a map; new rooms / users start empty
    {
        std::vector<ReviewRing<NUTSB_REVIEW_LINES>> rev((size_t)n_rooms, ReviewRing<NUTSB_REVIEW_LINES>{});
        for (size_t r = 0; r < rev.size() && r < c->rev.size(); ++r) rev[r] = c->rev[r];
        c->rev.swap(rev);
        std::vector<ReviewRing<NUTSB_REVTELL_LINES>> rt((size_t)n_users, ReviewRing<NUTSB_REVTELL_LINES>{});
        for (i32 u = 0; u < n_users; ++u) {
            const i32 p = prev_index ? prev_index[u] : u;
            if (p >= 0 && (size_t)p < c->revtell.size()) rt[(size_t)u] = c->revtell[(size_t)p];
        }
        c->revtell.swap(rt);
    }
    c->U = n_users; c->R = n_rooms; c->Rt = n_rooms + 1;
    c->user_room.resize(n_users);
    for (i32 u = 0; u < n_users; ++u) c->user_room[u] = room[u] < 0 ? n_rooms : room[u];
    // slot order: (room, flags, level, index) -- compatible with both class granularities
    std::vector<i32> order(n_users); std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](i32 a, i32 b) {
        if (c->user_room[a] != c->user_room[b]) return c->user_room[a] < c->user_room[b];
        const u32 ka = (u32)(flags[a] & 0x3f), kb = (u32)(flags[b] & 0x3f);
        if (ka != kb) return ka < kb;
        return level[a] < level[b];
    });
    c->slot_user = order; c->user_slot.assign(n_users, 0); c->room_slot_off.assign(c->Rt + 1, 0);
    for (i32 s = 0; s < n_users; ++s) { c->user_slot[order[s]] = s; c->room_slot_off[c->user_room[order[s]] + 1]++; }
    for (i32 r = 0; r < c->Rt; ++r) c->room_slot_off[r + 1] += c->room_slot_off[r];
    c->all_simple = true;
    for (i32 u = 0; u < n_users; ++u) if (flags[u] & NUTSB_UF_FILTERED) c->all_simple = false;
    c->uflags.assign(flags, flags + n_users);
    c->n_clone_flag = c->n_remote_flag = 0;
    for (i32 u = 0; u < n_users; ++u) { c->n_clone_flag += (flags[u] & NUTSB_UF_CLONE) != 0; c->n_remote_flag += (flags[u] & NUTSB_UF_REMOTE) != 0; }
    c->has_clones = c->n_clone_flag + c->n_remote_flag > 0;
    c->ulevel.assign(level, level + n_users);
    if ((i32)c->sflags.size() != n_users) c->have_names = false;             // nutsb_set_user_names follows the population
    c->remote_link.clear(); c->remote_old.clear(); c->remotes.clear();
    c->clone_owner.clear(); c->clone_hear.clear(); c->room_clones.clear();       // nutsb_set_clones follows the population
    TRY(upload(c, c->d_user_room, c->user_room.data(), (size_t)n_users * 4));
    TRY(upload(c, c->d_user_slot, c->user_slot.data(), (size_t)n_users * 4));
    TRY(upload(c, c->d_slot_user, c->slot_user.data(), (size_t)n_users * 4));
    TRY(upload(c, c->d_room_slot_off, c->room_slot_off.data(), (size_t)(c->Rt + 1) * 4));
    {
        std::vector<u8> cf(n_users), lv(n_users);
        for (i32 s = 0; s < n_users; ++s) { cf[s] = (u8)(flags[order[s]] & 0x3f); lv[s] = level[order[s]]; }
        TRY(upload(c, c->d_slot_cf, cf.data(), (size_t)n_users));
        TRY(upload(c, c->d_slot_lv, lv.data(), (size_t)n_users));
        CK(cudaStreamSynchronize(c->stream));          // cf/lv go out of scope
    }
    {   // every room's users in user-list order (the order write_room_except reaches them, c:1409): for the per-op digests
        std::vector<i32> ro((size_t)c->Rt + 1, 0), ru((size_t)n_users);
        for (i32 u = 0; u < n_users; ++u) ro[(size_t)c->user_room[u] + 1]++;
        for (i32 r = 0; r < c->Rt; ++r) ro[(size_t)r + 1] += ro[(size_t)r];
        std::vector<i32> cur(ro.begin(), ro.end() - 1);
        for (i32 u = 0; u < n_users; ++u) ru[(size_t)cur[(size_t)c->user_room[u]]++] = u;
        TRY(upload(c, c->d_room_users, ru.data(), (size_t)n_users * 4));
        TRY(upload(c, c->d_room_users_off, ro.data(), ro.size() * 4));
        CK(cudaStreamSynchronize(c->stream));
    }
    c->last.valid = false;
    TRY(build_classes(c, c->cls[0], false, order, flags, level));
    TRY(build_classes(c, c->cls[1], true, order, flags, level));
    CK(cudaStreamSynchronize(c->stream));
    c->have_users = true;
    return NUTSB_OK;
}

NUTSB_API int nutsb_set_users(nutsb_ctx *c, int32_t n_users, int32_t n_rooms, const int32_t *room,
                               const uint8_t *flags, const uint8_t *level)
{ return set_users_impl(c, n_users, n_rooms, room, flags, level, nullptr); }

NUTSB_API int nutsb_set_users_remap(nutsb_ctx *c, int32_t n_users, int32_t n_rooms, const int32_t *room,
                                     const uint8_t *flags, const uint8_t *level, const int32_t *prev_index)
{ return set_users_impl(c, n_users, n_rooms, room, flags, level, prev_index); }

static PopView pop_view(const nutsb_ctx *c, int with_level)
{
    const ClassSet &cs = c->cls[with_level ? 1 : 0];
    PopView p{};
    p.n_users = c->U; p.n_rooms = c->R; p.n_rooms_tot = c->Rt;
    p.user_room = c->d_user_room.as<i32>(); p.user_cls = cs.d_user_cls.as<i32>();
    p.user_slot = c->d_user_slot.as<i32>(); p.slot_user = c->d_slot_user.as<i32>();
    p.slot_cf = c->d_slot_cf.as<u8>(); p.slot_lv = c->d_slot_lv.as<u8>();
    p.room_slot_off = c->d_room_slot_off.as<i32>(); p.room_cls_off = cs.d_room_cls_off.as<i32>();
    p.cls_flags = cs.d_cls_flags.as<u8>(); p.cls_level = cs.d_cls_level.as<u8>();
    p.codetab = c->d_codetab.as<u8>();
    p.has_clones = c->has_clones ? 1u : 0u;
    return p;
}

// ---------------------------------------------------------------------------------------
// the write pipeline (device pointers in, streams in HBM out)
// ---------------------------------------------------------------------------------------
static int status_to_error(nutsb_ctx *c, u32 st)
{
    if (st & NUTSB_ST_BAD_OFFSETS)   return fail(c, NUTSB_E_INVAL, "text_off is not monotone%s");
    if (st & NUTSB_ST_TEXT_TOO_LONG) return fail(c, NUTSB_E_RANGE, "string longer than NUTSB_MAX_TEXT (2000) bytes%s");
    if (st & NUTSB_ST_BAD_KIND)      return fail(c, NUTSB_E_INVAL, "unknown op kind%s");
    if (st & NUTSB_ST_BAD_INDEX)     return fail(c, NUTSB_E_RANGE, "user/room index out of range%s");
    if (st & NUTSB_ST_RENDER_MISMATCH) return fail(c, NUTSB_E_CUDA, "internal: rendered length mismatch%s");
    return NUTSB_OK;
}

// Gather-list request (nutsb_write_batch_iov): when every recipient is a plain listener the fan-out is
// skipped altogether: `compact` comes back true and the pool (slab + direct renderings) and the lists are
// left in HBM for the caller to bring over; otherwise the streams are made as usual (compact = false).
struct IovReq {
    bool compact = false;
    u64 slab_span = 0, direct_bytes = 0, n_iov = 0;      // h_out = the slab's two renderings, h_dir = the direct renderings
};

// What run_write's two tails take over from its steps A-E.
struct Planned {
    OpsView ops; PopView pop; ClassPrefix cpx; Sizes sz;
    u32 *sv_slot, *counts; u64 *counters;
    u64 off_base, slab_on, slab_off;
    bool has_level, alias, par; cudaStream_t sd;
};

// The end of every write batch: the result (bytes = NULL: gather lists, no streams in HBM) and the byte counters.
static void finish(nutsb_ctx *c, nutsb_streams *out, const u8 *bytes, u64 total, u64 deliveries,
                   u64 slab, u64 fan_in, u64 fan_out, u64 render_in)
{
    c->last_total = total; c->have_streams = bytes != nullptr;      // (nutsb_stream_digests needs the streams)
    c->tm.slab_bytes = slab; c->tm.fanout_bytes_in = fan_in; c->tm.fanout_bytes_out = fan_out; c->tm.render_bytes_in = render_in;
    out->n_users = c->U; out->total_bytes = total; out->n_deliveries = deliveries;
    out->off = c->d_off.as<u64>(); out->bytes = bytes; out->on_device = 1;
}

// Gather lists instead of streams: direct ops rendered one after the other (k_direct_compact), one list entry
// per stretch of slab bytes and per direct rendering (k_iov); no copy plan, no fan-out.
static int write_iov_tail(nutsb_ctx *c, const Planned &p, nutsb_streams *out, IovReq *iv)
{
    const i32 U = c->U; const Sizes &sz = p.sz;
    cudaStream_t st = c->stream;
    u32 *h32 = c->h_small.as<u32>(); u64 *h64 = c->h_small.as<u64>();
    *iv = IovReq{ true, p.off_base + p.slab_off, sz.direct_bytes, 2ull * sz.n_events + (u64)U };
    TRY(ensure(c, c->d_dir, sz.direct_bytes + 64));
    TRY(ensure(c, c->d_iov, (size_t)iv->n_iov * sizeof(IovEnt)));
    TRY(ensure(c, c->d_iov_first, (size_t)U * 8)); TRY(ensure(c, c->d_iov_cnt, (size_t)U * 4));
    TRY(ensure_host(c, c->h_dir, (size_t)sz.direct_bytes + 64));                        // the entries hold host addresses
    TRY(ensure_host(c, c->h_iov, (size_t)iv->n_iov * sizeof(IovEnt)));
    TRY(ensure_host(c, c->h_iov_first, ((size_t)U + 1) * 8)); TRY(ensure_host(c, c->h_iov_cnt, ((size_t)U + 1) * 4));
    TRY(ensure_host(c, c->h_off, ((size_t)U + 1) * 8));
    TRY(ev_record(c, EV_DIRECT0, st));
    if (sz.n_events > 0) {
        DirectArgs da{ p.ops, p.pop, p.cpx, c->d_room_b_off.as<u32>(), c->d_ev_off.as<u32>(), c->d_sv_ukey.as<u32>(), c->d_sv_op.as<u32>(),
                       c->d_sv_pre.as<u64>(), c->d_off.as<u64>(), p.sv_slot, c->d_sv_delta.as<i32>(), c->d_dir.as<u8>(), (i64)sz.n_events, p.counters,
                       c->d_status.as<u32>(), c->d_slab.as<u8>(), p.off_base, 0u, c->d_slots.as<SlotInfo>(), c->d_dpre.as<u64>() };
        NUTSB_LAUNCH_SMEM(cdiv(sz.n_events, NUTSB_DIRECT_THREADS), NUTSB_DIRECT_THREADS, NUTSB_DIR_SMEM, st, k_direct_compact, da); CKL();
        c->tm.launches++;
    }
    TRY(ev_record(c, EV_DIRECT1, st)); TRY(ev_record(c, EV_FAN0, st));
    IovArgs ia{ p.pop, c->d_slots.as<SlotInfo>(), c->d_vp_on.as<u64>(), c->d_vp_off.as<u64>(), c->d_sv_ukey.as<u32>(), p.sv_slot,
                c->d_dpre.as<u64>(), sz.n_events, (u64)(size_t)c->h_out.p, (u64)(size_t)c->h_dir.p, p.off_base,
                c->d_iov.as<IovEnt>(), c->d_iov_first.as<u64>(), c->d_iov_cnt.as<u32>(), p.counters };
    NUTSB_LAUNCH(cdiv(std::max<u64>(sz.n_events, (u64)U), 256), 256, st, k_iov, ia); CKL();
    c->tm.launches++;
    TRY(ev_record(c, EV_FAN1, st)); TRY(ev_record(c, EV_END, st));
    // the rest of the result, beside the slab's copy on the side stream
    if (sz.direct_bytes) CK(cudaMemcpyAsync(c->h_dir.p, c->d_dir.p, (size_t)sz.direct_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(c->h_iov.p, c->d_iov.p, (size_t)iv->n_iov * sizeof(IovEnt), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(c->h_iov_first.p, c->d_iov_first.p, (size_t)U * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(c->h_iov_cnt.p, c->d_iov_cnt.p, (size_t)U * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(c->h_off.p, c->d_off.p, ((size_t)U + 1) * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h64 + 8, p.counters, 24, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h32 + 4, c->d_status.p, 4, cudaMemcpyDeviceToHost, st));
    if (p.par) CK(cudaStreamWaitEvent(st, c->dep[1], 0));      // the slab is rendered and on the host
    TRY(ev_record(c, EV_D2H1, st));
    CK(cudaStreamSynchronize(st));
    TRY(status_to_error(c, h32[4]));
    if (c->profiling) {
        TRY(ev_elapsed(c, &c->tm.plan_ms, EV_START, EV_DIRECT0));
        TRY(ev_elapsed(c, &c->tm.render_ms, EV_RENDER0, EV_RENDER1));
        TRY(ev_elapsed(c, &c->tm.fanout_ms, EV_FAN0, EV_FAN1));
        TRY(ev_elapsed(c, &c->tm.direct_ms, EV_DIRECT0, EV_DIRECT1));
        TRY(ev_elapsed(c, &c->tm.total_ms, EV_START, EV_END));
        TRY(ev_elapsed(c, &c->tm.d2h_ms, EV_END, EV_D2H1));        // what of the copies is left after the last kernel
    }
    finish(c, out, nullptr, sz.total_bytes, h64[8], p.slab_on + p.slab_off, 0, 0, h64[10]);
    return NUTSB_OK;
}

static int write_streams_tail(nutsb_ctx *c, const Planned &p, nutsb_streams *out)
{
    const Sizes &sz = p.sz;
    cudaStream_t st = c->stream, sd = p.sd;
    u32 *h32 = c->h_small.as<u32>(); u64 *h64 = c->h_small.as<u64>();
    TRY(ensure(c, c->d_out, sz.total_bytes + 64));
    Geometry geo{ c->d_room_b_off.as<u32>(), c->d_room_tile_off.as<u32>(), c->d_room_cell_off.as<u64>(), c->d_room_item_off.as<u32>() };

    // -- I. direct ops + seams.  With the overlap on they share ONE launch with the fan-out (k_fanout_direct,
    //    below): blocks of both kinds on every SM.  Otherwise (or when there is nothing to fan out) k_direct
    //    runs by itself, here.
    const bool fan = sz.cells > 0 && sz.items > 0;
    const bool fused = p.par && fan && sz.n_events > 0;
    DirectArgs da{ p.ops, p.pop, p.cpx, c->d_room_b_off.as<u32>(), c->d_ev_off.as<u32>(), c->d_sv_ukey.as<u32>(), c->d_sv_op.as<u32>(),
                   c->d_sv_pre.as<u64>(), c->d_off.as<u64>(), p.sv_slot, c->d_sv_delta.as<i32>(), c->d_out.as<u8>(), (i64)sz.n_events, p.counters,
                   c->d_status.as<u32>(), c->d_slab.as<u8>(), p.off_base, p.has_level ? 1u : 0u, c->d_slots.as<SlotInfo>(), nullptr };
    u32 n_dir = cdiv(sz.n_events, NUTSB_DIRECT_THREADS);
    if (fused && c->fd_dir_per_sm > 0) n_dir = std::min(n_dir, (u32)(c->sm_count * c->fd_dir_per_sm));   // grid-strided direct blocks
    TRY(ev_record(c, EV_DIRECT0, sd));
    if (sz.n_events > 0 && !fused) {
        if (p.par) { CK(cudaEventRecord(c->dep[2], st)); CK(cudaStreamWaitEvent(sd, c->dep[2], 0)); }
        NUTSB_LAUNCH_SMEM(n_dir, NUTSB_DIRECT_THREADS, NUTSB_DIR_SMEM, sd, k_direct, da); CKL();
        c->tm.launches++;
    }
    TRY(ev_record(c, EV_DIRECT1, sd));
    if (p.par) CK(cudaEventRecord(c->dep[3], sd));

    // -- F. copy plan: the run list and the work-item descriptors
    if (fan) {
        TRY(ensure(c, c->d_items, (size_t)sz.items * sizeof(ItemDesc)));
        u32 *cursor = p.counts + 4;
        CK(cudaMemsetAsync(cursor, 0, 4, st));
        PlanArgs pa{ p.pop, geo, p.cpx, c->d_off.as<u64>(), c->d_ev_off.as<u32>(), c->d_sv_ukey.as<u32>(), c->d_sv_delta.as<i32>(),
                     c->d_sv_pre.as<u64>(), c->d_bl_meta.as<u32>(), (u64)sz.cells, p.off_base, p.has_level ? 1u : 0u,
                     c->d_slots.as<SlotInfo>(), cursor, nullptr, c->d_items.as<ItemDesc>(), p.counters, c->d_status.as<u32>() };
        // plain listeners: at most one run per cell plus one per event; behind a filter the count is taken first
        u64 n_runs = sz.cells + sz.n_events;
        if (!p.alias) {
            NUTSB_LAUNCH(sz.items, NUTSB_UCHUNK, st, k_plan<false>, pa); CKL();
            CK(cudaMemcpyAsync(h32 + 6, cursor, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemsetAsync(cursor, 0, 4, st));
            CK(cudaStreamSynchronize(st));
            n_runs = h32[6];
            c->tm.launches++;
        }
        if (n_runs >= 0xfffffff0ull) return fail(c, NUTSB_E_RANGE, "more than 2^32 copy runs in one batch%s");
        TRY(ensure(c, c->d_runs, (n_runs + 1) * sizeof(uint4)));
        pa.runs = c->d_runs.as<uint4>();
        NUTSB_LAUNCH(sz.items, NUTSB_UCHUNK, st, k_plan<true>, pa); CKL();
        c->tm.launches++;
    }

    // -- H. fan-out: after the slab is rendered
    if (p.par) CK(cudaStreamWaitEvent(st, c->dep[1], 0));
    TRY(ev_record(c, EV_FAN0, st));
    if (fan) {
        FanoutArgs fa{ c->d_items.as<ItemDesc>(), c->d_runs.as<uint4>(), c->d_slab.as<u8>(), p.off_base, c->d_out.as<u8>() };
        if (fused) {
            const u32 total = sz.items + n_dir;
            const u32 stride = std::max(1u, total / n_dir);        // a direct block every `stride` blocks
            NUTSB_LAUNCH_SMEM(total, NUTSB_FAN_THREADS, NUTSB_FD_SMEM, st, k_fanout_direct, fa, da, n_dir, stride); CKL();
        } else {
            NUTSB_LAUNCH_SMEM(sz.items, NUTSB_FAN_THREADS, NUTSB_FAN_SMEM, st, k_fanout, fa); CKL();
        }
        c->tm.launches++; c->tm.fanout_launches = 1;
    }
    TRY(ev_record(c, EV_FAN1, st));
    if (p.par) CK(cudaStreamWaitEvent(st, c->dep[3], 0));
    TRY(ev_record(c, EV_END, st));

    NUTSB_LAUNCH(1, 32, st, k_readback_end, p.counters, c->d_status.as<u32>(), h64 + 8, h32 + 4); CKL();
    c->tm.launches++;
    CK(cudaStreamSynchronize(st));
    TRY(status_to_error(c, h32[4]));
    c->last.valid = true; c->last.ops = p.ops; c->last.cpx = p.cpx; c->last.has_level = p.has_level; c->last.off_base = p.off_base; c->last.sv_slot = p.sv_slot;
    if (c->profiling) {
        // with the side stream on, render_ms / direct_ms are the side kernels' own spans and overlap plan_ms / fanout_ms
        CK(cudaEventSynchronize(c->ev[EV_DIRECT1]));
        TRY(ev_elapsed(c, &c->tm.plan_ms, EV_START, EV_FAN0));
        TRY(ev_elapsed(c, &c->tm.render_ms, EV_RENDER0, EV_RENDER1));
        TRY(ev_elapsed(c, &c->tm.fanout_ms, EV_FAN0, EV_FAN1));
        TRY(ev_elapsed(c, &c->tm.direct_ms, EV_DIRECT0, EV_DIRECT1));
        TRY(ev_elapsed(c, &c->tm.total_ms, EV_START, EV_END));
        if (!p.par) c->tm.plan_ms -= c->tm.render_ms + c->tm.direct_ms;
    }
    const u64 slab = p.slab_on + p.slab_off;                   // (fan-out input: each rendering of a tile is read once per work item)
    finish(c, out, c->d_out.as<u8>(), sz.total_bytes, h64[8], slab, slab, sz.total_bytes - h64[9], h64[10]);
    return NUTSB_OK;
}

static int run_write(nutsb_ctx *c, const nutsb_ops *o, nutsb_streams *out, IovReq *iv = nullptr)
{
    if (!c->have_users) return fail(c, NUTSB_E_STATE, "nutsb_set_users has not been called%s");
    const i64 n = o->n_ops;
    const i32 U = c->U, Rt = c->Rt;
    cudaStream_t st = c->stream;
    c->have_streams = false; c->last.valid = false;
    c->tm.launches = 0; c->tm.fanout_launches = 0;
    if (c->side) CK(cudaStreamSynchronize(c->side));           // idle unless an earlier batch failed half-way
    TRY(ev_record(c, EV_START, st));

    TRY(ensure(c, c->d_off, ((size_t)U + 1) * 8));
    u32 *h32 = c->h_small.as<u32>(); u64 *h64 = c->h_small.as<u64>();

    auto finish_empty = [&]() -> int {
        CK(cudaMemsetAsync(c->d_off.p, 0, ((size_t)U + 1) * 8, st));
        TRY(ensure(c, c->d_out, 16));
        CK(cudaStreamSynchronize(st));
        finish(c, out, c->d_out.as<u8>(), 0, 0, 0, 0, 0, 0);
        return NUTSB_OK;
    };
    if (n == 0) return finish_empty();

    OpsView ops{ n, o->text, o->text_off, o->kind, o->target, o->except_user, o->flags,
                 o->gate && o->verdict ? o->gate : nullptr, o->gate && o->verdict ? o->verdict : nullptr };
    PopView pop0 = pop_view(c, 0);

    // -- A. measure + expansion counts
    TRY(ensure(c, c->d_len_on, (size_t)n * 4)); TRY(ensure(c, c->d_len_off, (size_t)n * 4));
    TRY(ensure(c, c->d_nrep, (size_t)n * 4)); TRY(ensure(c, c->d_eoff, ((size_t)n + 1) * 8));
    CK(cudaMemsetAsync(c->d_status.p, 0, 64, st));
    CK(cudaMemsetAsync(c->d_counters.p, 0, 1024, st));
    u32 *len_on = c->d_len_on.as<u32>(), *len_off = c->d_len_off.as<u32>(), *nrep = c->d_nrep.as<u32>();
    NUTSB_LAUNCH(std::min<u32>(cdiv(n, NUTSB_MEASURE_THREADS), (u32)c->sm_count * 5u), NUTSB_MEASURE_THREADS, st, k_measure, ops, pop0, len_on, len_off, nrep,
                 c->d_status.as<u32>(), c->d_counters.as<u64>() + 8); CKL();
    c->tm.launches++;
    TRY(run_scan(c, InU32{nrep}, OutU64{c->d_eoff.as<u64>()}, n, nullptr));

    // -- read-back #1: number of (room, op) entries, validation status
    static_assert(2 * NUTSB_SLAB_TOT_WAYS <= 64, "k_readback1 copies the slab totals with one block of 64 threads");
    NUTSB_LAUNCH(1, 64, st, k_readback1, c->d_eoff.as<u64>() + n, c->d_status.as<u32>(), c->d_counters.as<u64>() + 8,
                 h64, h32 + 4, h64 + 64); CKL();
    c->tm.launches++;
    CK(cudaStreamSynchronize(st));
    const u64 E = h64[0]; const u32 status = h32[4];
    u64 slab_on = 0, slab_off = 0;
    for (int w = 0; w < NUTSB_SLAB_TOT_WAYS; ++w) { slab_on += h64[64 + 2 * w]; slab_off += h64[65 + 2 * w]; }
    const u64 off_base = (slab_on + 15) & ~(u64)15;            // the colour-off renderings follow the colour-on ones
    TRY(status_to_error(c, status));
    if (E == 0) return finish_empty();
    if (E >= 0xfffffff0ull) return fail(c, NUTSB_E_RANGE, "more than 2^32 (room, op) entries in one batch%s");
    const bool has_level = (status & NUTSB_ST_HAS_LEVEL) != 0;
    const bool alias = c->all_simple && !has_level;
    const bool compact = iv && alias && U > 0;                 // gather lists: plain listeners only
    const PopView pop = pop_view(c, has_level ? 1 : 0);
    const ClassSet &cs = c->cls[has_level ? 1 : 0];

    // -- B. expand + bucket by room
    for (int q = 0; q < 2; ++q) { TRY(ensure(c, c->d_ek[q], (size_t)E * 4 + 16)); TRY(ensure(c, c->d_ev_[q], (size_t)E * 4 + 16)); }
    NUTSB_LAUNCH(cdiv(n, 256), 256, st, k_expand, ops, pop, nrep, c->d_eoff.as<u64>(), c->d_ek[0].as<u32>(), c->d_ev_[0].as<u32>()); CKL();
    c->tm.launches++;
    // the op index rides as the key's payload: the first pass must not use iota
    u32 *e_room = nullptr, *e_op = nullptr;
    TRY(radix_sort(c, c->d_ek, c->d_ev_, (i64)E, nullptr, std::max(1u, bits_for((u64)Rt)), &e_room, &e_op, true));
    TRY(ensure(c, c->d_room_ent_off, ((size_t)Rt + 2) * 4));

    // -- C. classify entries, scatter the slab list and the event list
    TRY(ensure(c, c->d_e_info, E)); TRY(ensure(c, c->d_e_delta, E * 4)); TRY(ensure(c, c->d_e_slot, E * 4));
    TRY(ensure(c, c->d_e_scan, (E + 1) * 8));
    EntryArrays ea{ e_room, e_op, c->d_e_info.as<u8>(), c->d_e_delta.as<i32>(), c->d_e_slot.as<u32>() };
    NUTSB_LAUNCH(cdiv(E + 1, 256), 256, st, k_entry_info, ops, pop, ea, (i64)E, len_on, len_off, c->d_room_ent_off.as<u32>()); CKL();
    TRY(run_scan(c, InEntryPacked{c->d_e_info.as<u8>()}, OutU64{c->d_e_scan.as<u64>()}, (i64)E, nullptr));
    u32 *counts = c->d_counts.as<u32>();
    TRY(ensure(c, c->d_room_b_off, ((size_t)Rt + 2) * 4));
    NUTSB_LAUNCH(cdiv((u64)Rt + 1, 256), 256, st, k_room_b_off, c->d_room_ent_off.as<u32>(), c->d_e_scan.as<u64>(), (i64)E, (u32)Rt, c->d_room_b_off.as<u32>(), counts); CKL();
    TRY(ensure(c, c->d_bl_op, E * 4 + 16)); TRY(ensure(c, c->d_bl_room, E * 4 + 16)); TRY(ensure(c, c->d_bl_meta, E * 4 + 16));
    for (int q = 0; q < 2; ++q) { TRY(ensure(c, c->d_evk[q], E * 4 + 16)); TRY(ensure(c, c->d_evv[q], E * 4 + 16)); }
    TRY(ensure(c, c->d_ev_ukey, E * 4)); TRY(ensure(c, c->d_ev_delta, E * 4)); TRY(ensure(c, c->d_ev_op, E * 4));
    EntryScatter es{ e_room, e_op, c->d_e_info.as<u8>(), c->d_e_delta.as<i32>(), c->d_e_slot.as<u32>(),
                     c->d_room_ent_off.as<u32>(), c->d_e_scan.as<u64>(), c->d_bl_op.as<u32>(), c->d_bl_room.as<u32>(),
                     c->d_bl_meta.as<u32>(), ops, c->d_evk[0].as<u32>(), c->d_ev_ukey.as<u32>(), c->d_ev_op.as<u32>(), c->d_ev_delta.as<i32>() };
    NUTSB_LAUNCH(cdiv(E, 256), 256, st, k_entry_scatter, es, (i64)E); CKL();
    c->tm.launches += 3;

    // -- slab prefixes (per colour) and, when classes differ in what they take, per class column
    TRY(ensure(c, c->d_vp_on, (E + 2) * 8)); TRY(ensure(c, c->d_vp_off, (E + 2) * 8));
    if (slab_on < 0xffffffffull) {                             // (slab_off <= slab_on) both prefixes fit 32 bits: one scan
        TRY(run_scan(c, InSlabLen2{len_on, len_off, c->d_bl_op.as<u32>()}, OutSplit{c->d_vp_on.as<u64>(), c->d_vp_off.as<u64>()}, (i64)E, counts));
    } else {
        TRY(run_scan(c, InSlabLen{len_on, c->d_bl_op.as<u32>()}, OutU64{c->d_vp_on.as<u64>()}, (i64)E, counts));
        TRY(run_scan(c, InSlabLen{len_off, c->d_bl_op.as<u32>()}, OutU64{c->d_vp_off.as<u64>()}, (i64)E, counts));
    }
    ClassPrefix cpx{ c->d_vp_on.as<u64>(), c->d_vp_off.as<u64>(), nullptr, (u64)E + 1, pop.room_cls_off, pop.cls_flags };
    if (!alias) {
        const i32 J = std::max(1, cs.max_per_room);
        TRY(ensure(c, c->d_cp, (size_t)J * (E + 1) * 8));
        for (i32 j = 0; j < J; ++j) {
            InClassLen in{ ops, c->d_bl_op.as<u32>(), c->d_bl_room.as<u32>(), len_on, len_off, pop.room_cls_off, pop.cls_flags, pop.cls_level, j };
            TRY(run_scan(c, in, OutU64{c->d_cp.as<u64>() + (size_t)j * (E + 1)}, (i64)E, counts));
        }
        cpx.cp = c->d_cp.as<u64>();
    }

    // -- G. render the slab, once per colour setting: needs only the slab list and its prefixes, so it
    //    runs on the side stream while this one goes on planning
    const bool par = c->overlap && c->side != nullptr;
    cudaStream_t sd = par ? c->side : st;
    u64 *counters = c->d_counters.as<u64>();
    if (off_base + slab_off >= (1ull << 40)) return fail(c, NUTSB_E_RANGE, "more than 2^40 bytes of rendered slab in one batch%s");
    TRY(ensure(c, c->d_slab, off_base + slab_off + 256));
    if (compact) TRY(ensure_host(c, c->h_out, (size_t)(off_base + slab_off) + 64));      // before anything is queued on the side stream
    if (par) { CK(cudaEventRecord(c->dep[0], st)); CK(cudaStreamWaitEvent(sd, c->dep[0], 0)); }
    TRY(ev_record(c, EV_RENDER0, sd));
    {
        RenderArgs ra{ ops, c->d_codetab.as<u8>(), c->d_bl_op.as<u32>(), c->d_vp_on.as<u64>(), c->d_vp_off.as<u64>(), counts,
                       c->d_slab.as<u8>(), off_base, counters, c->d_status.as<u32>() };
        // grid from the host's bound on the slab ops (E entries); warps past the device's count leave at once
        u32 grid = cdiv(E, NUTSB_REN_OPS * (NUTSB_REN_THREADS / 32));
        if (par) grid = std::min(grid, (u32)(c->sm_count * c->side_render));
        NUTSB_LAUNCH(grid, NUTSB_REN_THREADS, sd, k_render, ra); CKL();
        c->tm.launches++;
    }
    TRY(ev_record(c, EV_RENDER1, sd));
    // gather lists: the slab is part of the result as it stands -- on its way to the host while the planning goes on
    if (compact && off_base + slab_off) CK(cudaMemcpyAsync(c->h_out.p, c->d_slab.p, (size_t)(off_base + slab_off), cudaMemcpyDeviceToHost, sd));
    if (par) CK(cudaEventRecord(c->dep[1], sd));

    // -- D. events: sort by recipient slot, prefix of byte deltas
    u32 *sv_slot = nullptr, *perm = nullptr;
    TRY(radix_sort(c, c->d_evk, c->d_evv, (i64)E, counts + 1, bits_for((u64)std::max(U, 1)), &sv_slot, &perm));
    TRY(ensure(c, c->d_sv_ukey, E * 4 + 16)); TRY(ensure(c, c->d_sv_delta, E * 4 + 16)); TRY(ensure(c, c->d_sv_op, E * 4 + 16));
    TRY(ensure(c, c->d_sv_pre, (E + 2) * 8)); TRY(ensure(c, c->d_ev_off, ((size_t)U + 2) * 4));
    NUTSB_LAUNCH(cdiv(E + 1, 256), 256, st, k_ev_gather, perm, counts + 1, c->d_ev_ukey.as<u32>(), c->d_ev_delta.as<i32>(),
                 c->d_ev_op.as<u32>(), c->d_sv_ukey.as<u32>(), c->d_sv_delta.as<i32>(), c->d_sv_op.as<u32>(), sv_slot, (u32)U, c->d_ev_off.as<u32>()); CKL();
    TRY(run_scan(c, InI32{c->d_sv_delta.as<i32>()}, OutU64{c->d_sv_pre.as<u64>()}, (i64)E, counts + 1));
    c->tm.launches += 1;

    // -- E. stream offsets (a scan over the users' stream lengths, each computed as it is read), geometry
    UserLenIn uli{ cpx, pop, c->d_room_b_off.as<u32>(), c->d_ev_off.as<u32>(), c->d_sv_pre.as<u64>() };
    TRY(run_scan(c, uli, OutU64{c->d_off.as<u64>()}, (i64)U, nullptr));
    TRY(ensure(c, c->d_slots, ((size_t)U + 1) * sizeof(SlotInfo)));
    if (U > 0) {
        SlotInfoArgs sa{ pop, cpx, c->d_room_b_off.as<u32>(), c->d_ev_off.as<u32>(), c->d_sv_pre.as<u64>(), c->d_off.as<u64>(), c->d_slots.as<SlotInfo>() };
        NUTSB_LAUNCH(cdiv((u64)U, 128), 128, st, k_slot_info, sa); CKL();
        c->tm.launches++;
    }
    if (compact) {                                             // where each direct rendering goes in its pool
        TRY(ensure(c, c->d_dpre, (E + 2) * 8));
        TRY(run_scan(c, InDirectLen{ c->d_sv_ukey.as<u32>(), sv_slot, c->d_sv_delta.as<i32>(), c->d_slots.as<SlotInfo>(),
                                     c->d_vp_on.as<u64>(), c->d_vp_off.as<u64>() }, OutU64{c->d_dpre.as<u64>()}, (i64)E, counts + 1));
    }
    TRY(ensure(c, c->d_room_tile_off, ((size_t)Rt + 2) * 4)); TRY(ensure(c, c->d_room_cell_off, ((size_t)Rt + 2) * 8));
    TRY(ensure(c, c->d_room_item_off, ((size_t)Rt + 2) * 4));
    // read-back #2 (sizes): k_geometry writes them straight into pinned host memory (zero-copy: the context's
    // h_small is device-accessible under unified addressing), so that nothing waits in a copy queue -- in
    // gather-list mode the slab's copy to the host is in flight on the side stream by now
    Sizes *hs = (Sizes *)(c->h_small.as<u8>() + 256);
    NUTSB_LAUNCH(1, NUTSB_SCAN_THREADS, st, k_geometry, pop, c->d_room_b_off.as<u32>(), c->d_off.as<u64>(), counts,
                 c->d_vp_on.as<u64>(), c->d_vp_off.as<u64>(),
                 c->d_room_tile_off.as<u32>(), c->d_room_cell_off.as<u64>(), c->d_room_item_off.as<u32>(), hs,
                 compact ? c->d_dpre.as<u64>() : (const u64 *)nullptr); CKL();
    c->tm.launches++;
    CK(cudaStreamSynchronize(st));
    const Planned p{ ops, pop, cpx, *hs, sv_slot, counts, counters, off_base, slab_on, slab_off, has_level, alias, par, sd };
    if (p.sz.slab_on != slab_on || p.sz.slab_off != slab_off) return fail(c, NUTSB_E_CUDA, "internal: slab size mismatch%s");
    return compact ? write_iov_tail(c, p, out, iv) : write_streams_tail(c, p, out);
}

static int check_ops(nutsb_ctx *c, const nutsb_ops *o)
{
    if (!c || !o || o->n_ops < 0) return fail(c, NUTSB_E_INVAL, "null argument or negative n_ops%s");
    if (o->n_ops >= 0xfffffff0ll) return fail(c, NUTSB_E_RANGE, "more than 2^32 ops in one batch%s");
    if (o->n_ops && (!o->text_off || !o->kind || !o->target || !o->except_user || !o->flags))
        return fail(c, NUTSB_E_INVAL, "ops array is NULL%s");
    return NUTSB_OK;
}

// The host-side check of op i, for the paths that expand or route ops on the host before the device sees
// them: NUTSB_OK, or the error code with *why set.
static int host_op_error(const nutsb_ops *o, i64 i, i32 U, i32 R, const char **why)
{
    if (o->text_off[i + 1] < o->text_off[i]) { *why = "text_off is not monotone"; return NUTSB_E_INVAL; }
    const u8 k = o->kind[i];
    if (k == NUTSB_OP_NONE) return NUTSB_OK;
    if (k > NUTSB_OP_LEVEL) { *why = "unknown op kind"; return NUTSB_E_INVAL; }
    const i32 t = o->target[i], x = o->except_user[i];
    if (x >= U || x < -1 || (k == NUTSB_OP_USER && t >= U) || (k == NUTSB_OP_ROOM && (t >= R || t < -1))) {
        *why = "user/room index out of range"; return NUTSB_E_RANGE;
    }
    return NUTSB_OK;
}

// Clones and remote users (nuts333.c:1416-1426, 1299-1307) are reached through relays / frames that are
// extra write_user calls, made on the host (q_push).  Ops that have not been through that expansion are
// refused with such users in the population, rather than delivered differently from the reference.
// Every write entry point starts here.
static int begin_write(nutsb_ctx *c, bool expanded)
{
    if (!expanded && c->has_clones)
        return fail(c, NUTSB_E_UNSUPPORTED, "population holds clones / remote users: use the host-buffer or the queue tier%s");
    CK(cudaSetDevice(c->device));
    return NUTSB_OK;
}

// ops in host memory -> the context's staging buffers in HBM (*d = the same batch with device pointers)
static int upload_ops(nutsb_ctx *c, const nutsb_ops *o, nutsb_ops *d)
{
    const i64 n = o->n_ops;
    cudaStream_t st = c->stream;
    TRY(ev_record(c, EV_H2D0, st));
    *d = *o;
    if (n <= 0) return ev_record(c, EV_H2D1, st);
    const u64 t0 = o->text_off[0], t1 = o->text_off[n];
    if (t1 < t0) return fail(c, NUTSB_E_INVAL, "text_off is not monotone%s");
    if (t1 > t0 && !o->text) return fail(c, NUTSB_E_INVAL, "text is NULL%s");
    // text is uploaded from t0 on; offsets are used as they are (base pointer shifted back)
    TRY(ensure(c, c->s_text, (size_t)(t1 - t0) + 64));
    if (t1 > t0) CK(cudaMemcpyAsync(c->s_text.p, o->text + t0, (size_t)(t1 - t0), cudaMemcpyHostToDevice, st));
    TRY(upload(c, c->s_toff, o->text_off, ((size_t)n + 1) * 8));
    TRY(upload(c, c->s_kind, o->kind, (size_t)n));
    TRY(upload(c, c->s_target, o->target, (size_t)n * 4));
    TRY(upload(c, c->s_except, o->except_user, (size_t)n * 4));
    TRY(upload(c, c->s_flags, o->flags, (size_t)n));
    d->text = c->s_text.as<u8>() - t0; d->text_off = c->s_toff.as<u64>(); d->kind = c->s_kind.as<u8>();
    d->target = c->s_target.as<i32>(); d->except_user = c->s_except.as<i32>(); d->flags = c->s_flags.as<u8>();
    d->gate = nullptr; d->verdict = nullptr;
    if (o->gate && o->verdict) {
        i32 mx = -1; for (i64 i = 0; i < n; ++i) mx = std::max(mx, o->gate[i]);
        TRY(upload(c, c->s_gate, o->gate, (size_t)n * 4));
        TRY(upload(c, c->s_verdict, o->verdict, (size_t)(mx + 1)));
        d->gate = c->s_gate.as<i32>(); d->verdict = c->s_verdict.as<u8>();
    }
    return ev_record(c, EV_H2D1, st);
}

// Streams HBM -> pinned host memory (h_off, h_out)
static int streams_to_host(nutsb_ctx *c, const nutsb_streams &ds)
{
    cudaStream_t st = c->stream;
    TRY(ev_record(c, EV_D2H0, st));
    TRY(ensure_host(c, c->h_off, ((size_t)c->U + 1) * 8));
    TRY(ensure_host(c, c->h_out, (size_t)ds.total_bytes + 16));
    CK(cudaMemcpyAsync(c->h_off.p, ds.off, ((size_t)c->U + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (ds.total_bytes) CK(cudaMemcpyAsync(c->h_out.p, ds.bytes, (size_t)ds.total_bytes, cudaMemcpyDeviceToHost, st));
    TRY(ev_record(c, EV_D2H1, st));
    CK(cudaStreamSynchronize(st));
    if (c->profiling) TRY(ev_elapsed(c, &c->tm.d2h_ms, EV_D2H0, EV_D2H1));
    return NUTSB_OK;
}

// Gather lists on the host after run_write(..., &iv): as run_write brought them over (plain listeners only),
// or, for recipients behind filters, one piece per user's stream.
static int fetch_iov(nutsb_ctx *c, const nutsb_streams &ds, const IovReq &iv, nutsb_iov_streams *out)
{
    const size_t U = (size_t)c->U;
    out->pool2 = nullptr; out->pool2_bytes = 0;
    if (iv.compact) {
        out->n_iov = iv.n_iov; out->pool_bytes = iv.slab_span;
        out->pool2 = c->h_dir.as<u8>(); out->pool2_bytes = iv.direct_bytes;
    } else {
        TRY(streams_to_host(c, ds));
        TRY(ensure_host(c, c->h_iov_first, (U + 1) * 8)); TRY(ensure_host(c, c->h_iov_cnt, (U + 1) * 4));
        TRY(ensure_host(c, c->h_iov, (U + 1) * sizeof(nutsb_iovec)));
        const u64 *off = c->h_off.as<u64>();
        nutsb_iovec *v = c->h_iov.as<nutsb_iovec>();
        for (size_t u = 0; u < U; ++u) {
            v[u].base = c->h_out.as<u8>() + off[u]; v[u].len = (size_t)(off[u + 1] - off[u]);
            c->h_iov_first.as<u64>()[u] = u; c->h_iov_cnt.as<u32>()[u] = 1;
        }
        out->n_iov = U; out->pool_bytes = ds.total_bytes;
    }
    out->n_users = (int64_t)U; out->total_bytes = ds.total_bytes; out->n_deliveries = ds.n_deliveries;
    out->off = c->h_off.as<u64>(); out->first = c->h_iov_first.as<u64>(); out->count = c->h_iov_cnt.as<u32>();
    out->iov = c->h_iov.as<nutsb_iovec>();
    out->pool = c->h_out.as<u8>();
    return NUTSB_OK;
}

// The form a write entry point hands its result over in: streams left in HBM, streams in pinned host memory, or
// gather lists (include/nutsb200.h: with plain listeners only, what crosses PCIe is the slab's two renderings,
// the direct ops' renderings and 16 bytes per piece -- not one copy of the bytes per recipient).
struct Result { enum Form { HBM, HOST, IOV } form; nutsb_streams *st; nutsb_iov_streams *iov; };

// The last step of every write entry point: run_write's result in the requested form, and the copy timings
// (0 for copies the call did not make).
static int deliver(nutsb_ctx *c, bool uploaded, const nutsb_streams &ds, const IovReq &iv, const Result &r)
{
    if (c->profiling) {
        c->tm.h2d_ms = 0;
        if (uploaded) TRY(ev_elapsed(c, &c->tm.h2d_ms, EV_H2D0, EV_H2D1));
    }
    if (r.form == Result::IOV) return fetch_iov(c, ds, iv, r.iov);
    if (r.form == Result::HBM) { if (c->profiling) c->tm.d2h_ms = 0; *r.st = ds; return NUTSB_OK; }
    TRY(streams_to_host(c, ds));
    *r.st = ds;
    r.st->off = c->h_off.as<u64>(); r.st->bytes = c->h_out.as<u8>(); r.st->on_device = 0;
    return NUTSB_OK;
}

// A write batch of ops, in HBM or (upload) in host memory.  expanded: the ops have been through the queue's
// clone / remote expansion.
static int write_ops(nutsb_ctx *c, const nutsb_ops *o, bool upload, bool expanded, const Result &r)
{
    if (!r.st && !r.iov) return fail(c, NUTSB_E_INVAL, "null argument%s");
    TRY(check_ops(c, o));
    TRY(begin_write(c, expanded));
    nutsb_ops d = *o;
    if (upload) TRY(upload_ops(c, o, &d));
    nutsb_streams ds{}; IovReq iv;
    TRY(run_write(c, &d, &ds, r.form == Result::IOV ? &iv : nullptr));
    return deliver(c, upload, ds, iv, r);
}

NUTSB_API int nutsb_write_batch_dev(nutsb_ctx *c, const nutsb_ops *o, nutsb_streams *out)
{ return write_ops(c, o, false, false, { Result::HBM, out, nullptr }); }

// ops in host memory, streams left in HBM (digests, or a later copy, are the caller's business)
NUTSB_API int nutsb_write_batch_keep(nutsb_ctx *c, const nutsb_ops *o, nutsb_streams *out)
{ return write_ops(c, o, true, false, { Result::HBM, out, nullptr }); }

static int stream_digests(nutsb_ctx *c, uint64_t *digest, bool cont)
{
    if (!c || !digest) return NUTSB_E_INVAL;
    if (!c->have_streams) return fail(c, NUTSB_E_STATE, "no write batch has run%s");
    CK(cudaSetDevice(c->device));
    if (c->U == 0) return NUTSB_OK;
    TRY(ensure(c, c->d_digest, (size_t)c->U * 16));
    u64 *d_out = c->d_digest.as<u64>(), *d_init = d_out + c->U;
    if (cont) CK(cudaMemcpyAsync(d_init, digest, (size_t)c->U * 8, cudaMemcpyHostToDevice, c->stream));
    const u32 grid = std::min<u32>((u32)c->U, (u32)c->sm_count * 16u);
    NUTSB_LAUNCH(grid, 256, c->stream, k_digest, c->d_out.as<u8>(), c->d_off.as<u64>(), c->U, cont ? (const u64 *)d_init : (const u64 *)nullptr, d_out); CKL();
    CK(cudaMemcpyAsync(digest, d_out, (size_t)c->U * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return NUTSB_OK;
}
NUTSB_API int nutsb_stream_digests(nutsb_ctx *c, uint64_t *digest) { return stream_digests(c, digest, false); }
NUTSB_API int nutsb_stream_digests_continue(nutsb_ctx *c, uint64_t *digest) { return stream_digests(c, digest, true); }

// The parity digests of SURVEY.md 8(d) for the last write batch (its streams and scratch arrays still in HBM):
// per_user[n_users] and per_op[n_ops], host arrays, either may be NULL.
NUTSB_API int nutsb_delivery_digests(nutsb_ctx *c, uint64_t *per_user, uint64_t *per_op)
{
    if (!c) return NUTSB_E_INVAL;
    if (!c->have_streams || !c->last.valid) return fail(c, NUTSB_E_STATE, "no write batch with streams in HBM has run (or it was empty)%s");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const i64 n = c->last.ops.n; const size_t U = (size_t)c->U;
    // upper bounds on the slab ops and the events: the entries of the batch (the counts themselves are on the device)
    u32 hcounts[2];
    CK(cudaMemcpyAsync(hcounts, c->d_counts.p, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const size_t nS = hcounts[0], nE = hcounts[1];
    const size_t bytes = (2 * (nS + 1) + (nE + 1) + U + 1 + (size_t)n + 1) * 8 + ((nE + 1) + 2 * ((size_t)n + 1)) * 4;
    TRY(ensure(c, c->d_dg, bytes));
    u64 *p64 = c->d_dg.as<u64>();
    DgArgs A{};
    A.ops = c->last.ops; A.pop = pop_view(c, c->last.has_level ? 1 : 0); A.cpx = c->last.cpx;
    A.bl_op = c->d_bl_op.as<u32>(); A.bl_meta = c->d_bl_meta.as<u32>(); A.ev_slot_sorted = c->last.sv_slot;
    A.sv_ukey = c->d_sv_ukey.as<u32>(); A.sv_op = c->d_sv_op.as<u32>(); A.sv_pre = c->d_sv_pre.as<u64>();
    A.slots = c->d_slots.as<SlotInfo>(); A.slab = c->d_slab.as<u8>(); A.out = c->d_out.as<u8>(); A.off_base = c->last.off_base;
    A.counts = c->d_counts.as<u32>(); A.has_level = c->last.has_level ? 1u : 0u;
    A.nrep = c->d_nrep.as<u32>(); A.room_users = c->d_room_users.as<i32>(); A.room_users_off = c->d_room_users_off.as<i32>();
    A.dg_on = p64; A.dg_off = A.dg_on + nS + 1; A.ev_d = A.dg_off + nS + 1; A.per_user = A.ev_d + nE + 1; A.per_op = A.per_user + U + 1;
    u32 *p32 = (u32 *)(A.per_op + n + 1);
    A.ev_len = p32; A.op_g = p32 + nE + 1; A.op_ev = A.op_g + n + 1;
    CK(cudaMemsetAsync(A.ev_len, 0, (nE + 1) * 4, st));
    CK(cudaMemsetAsync(A.op_g, 0xff, 2 * ((size_t)n + 1) * 4, st));
    if (nS) { NUTSB_LAUNCH(cdiv(nS, 256), 256, st, k_dg_slab, A); CKL(); }
    if (nE) { NUTSB_LAUNCH(cdiv(nE, 256), 256, st, k_dg_events, A); CKL(); }
    if (U && per_user) { NUTSB_LAUNCH(cdiv(U, 128), 128, st, k_dg_user, A); CKL(); }
    if (n && per_op) { NUTSB_LAUNCH(cdiv((u64)n, 128), 128, st, k_dg_op, A); CKL(); }
    if (per_user && U) CK(cudaMemcpyAsync(per_user, A.per_user, U * 8, cudaMemcpyDeviceToHost, st));
    if (per_op && n) CK(cudaMemcpyAsync(per_op, A.per_op, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return NUTSB_OK;
}

// ---------------------------------------------------------------------------------------
// verdict batches
// ---------------------------------------------------------------------------------------
static int run_ac(nutsb_ctx *c, const AcDev &ac, i64 n, const u8 *bytes, const u64 *off, u8 *verdict)
{
    if (n == 0) return NUTSB_OK;
    if (ac.view.tr16 && ac.view.maxpat <= 256) {                   // the warp-cooperative form
        // no string-start mask (k_ac_pair): two bytes a step when the squared table fits 16 KB, else one
        const bool pair = ac.view.t2 != nullptr;
        const u32 tb = ((pair ? ac.view.nstates * ac.view.t2_rs : ac.view.nstates * ac.view.ncls * 2u) + 15u) & ~15u;
        const u32 smem = NUTSB_ACP_SMEM(tb);
        const u32 per_sm = std::max(1u, std::min(8u, (227u * 1024u) / (smem + 1024u)));
        const u32 g = std::min<u32>(cdiv(n, NUTSB_ACW_THREADS), (u32)c->sm_count * per_sm);
        if (pair) { NUTSB_LAUNCH_SMEM(g, NUTSB_ACW_THREADS, smem, c->stream, k_ac_pair<true>, bytes, off, n, ac.view, tb, verdict); }
        else      { NUTSB_LAUNCH_SMEM(g, NUTSB_ACW_THREADS, smem, c->stream, k_ac_pair<false>, bytes, off, n, ac.view, tb, verdict); }
        CKL();
        return NUTSB_OK;
    }
    const u32 grid = std::min<u32>(cdiv(n, NUTSB_AC_THREADS), (u32)c->sm_count * 8u);
    const bool smem = ac.view.nstates <= 32768u && (u64)ac.view.nstates * ac.view.ncls <= NUTSB_AC_SMEM_ENTRIES;
    if (smem) { NUTSB_LAUNCH(grid, NUTSB_AC_THREADS, c->stream, k_ac_match<true>, bytes, off, n, ac.view, verdict); }
    else      { NUTSB_LAUNCH(grid, NUTSB_AC_THREADS, c->stream, k_ac_match<false>, bytes, off, n, ac.view, verdict); }
    CKL();
    return NUTSB_OK;
}

enum { V_SWEAR, V_SITE, V_USER };

static int verdict_dev(nutsb_ctx *c, int which, i64 n, const u8 *bytes, const u64 *off, u8 *verdict)
{
    if (!c || n < 0 || (n && (!off || !verdict))) return fail(c, NUTSB_E_INVAL, "bad argument%s");
    CK(cudaSetDevice(c->device));
    if (n == 0) return NUTSB_OK;
    if (which == V_SWEAR) return run_ac(c, c->swear, n, bytes, off, verdict);
    if (which == V_SITE) {
        if (!c->site_file || !c->site.present) { CK(cudaMemsetAsync(verdict, 0, (size_t)n, c->stream)); return NUTSB_OK; }   // c:337
        return run_ac(c, c->site, n, bytes, off, verdict);
    }
    if (!c->user_file || !c->userban.present) { CK(cudaMemsetAsync(verdict, 0, (size_t)n, c->stream)); return NUTSB_OK; }       // c:356
    NUTSB_LAUNCH(cdiv(n, 256), 256, c->stream, k_set_match, bytes, off, n, c->userban.view, verdict); CKL();
    return NUTSB_OK;
}

static int verdict_host(nutsb_ctx *c, int which, i64 n, const u8 *bytes, const u64 *off, u8 *verdict)
{
    if (!c || n < 0 || (n && (!off || !verdict))) return fail(c, NUTSB_E_INVAL, "bad argument%s");
    CK(cudaSetDevice(c->device));
    if (n == 0) return NUTSB_OK;
    const u64 t0 = off[0], t1 = off[n];
    if (t1 < t0 || (t1 > t0 && !bytes)) return fail(c, NUTSB_E_INVAL, "bad offsets%s");
    for (i64 i = 0; i < n; ++i) if (off[i + 1] < off[i]) return fail(c, NUTSB_E_INVAL, "offsets are not monotone%s");
    TRY(ensure(c, c->s_text, (size_t)(t1 - t0) + 64));
    if (t1 > t0) CK(cudaMemcpyAsync(c->s_text.p, bytes + t0, (size_t)(t1 - t0), cudaMemcpyHostToDevice, c->stream));
    TRY(upload(c, c->s_toff, off, ((size_t)n + 1) * 8));
    TRY(ensure(c, c->s_v8, (size_t)n));
    TRY(verdict_dev(c, which, n, c->s_text.as<u8>() - t0, c->s_toff.as<u64>(), c->s_v8.as<u8>()));
    CK(cudaMemcpyAsync(verdict, c->s_v8.p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return NUTSB_OK;
}

NUTSB_API int nutsb_contains_swearing_batch(nutsb_ctx *c, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return verdict_host(c, V_SWEAR, n, b, o, v); }
NUTSB_API int nutsb_contains_swearing_batch_dev(nutsb_ctx *c, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return verdict_dev(c, V_SWEAR, n, b, o, v); }
NUTSB_API int nutsb_site_banned_batch(nutsb_ctx *c, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return verdict_host(c, V_SITE, n, b, o, v); }
NUTSB_API int nutsb_site_banned_batch_dev(nutsb_ctx *c, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return verdict_dev(c, V_SITE, n, b, o, v); }
NUTSB_API int nutsb_user_banned_batch(nutsb_ctx *c, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return verdict_host(c, V_USER, n, b, o, v); }
NUTSB_API int nutsb_user_banned_batch_dev(nutsb_ctx *c, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return verdict_dev(c, V_USER, n, b, o, v); }

// colour_com_count / colour_com_strip over host strings
static int colour_com(nutsb_ctx *c, i64 n, const u8 *bytes, const u64 *off, i32 *count, const u8 **out_bytes, const u64 **out_off)
{
    if (!c || n < 0 || (n && !off) || (!count && (!out_bytes || !out_off))) return fail(c, NUTSB_E_INVAL, "bad argument%s");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    TRY(ensure_host(c, c->h_off, ((size_t)n + 1) * 8));
    if (n == 0) { if (out_off) { c->h_off.as<u64>()[0] = 0; *out_off = c->h_off.as<u64>(); *out_bytes = c->h_out.as<u8>(); } return NUTSB_OK; }
    const u64 t0 = off[0], t1 = off[n];
    if (t1 < t0 || (t1 > t0 && !bytes)) return fail(c, NUTSB_E_INVAL, "bad offsets%s");
    for (i64 i = 0; i < n; ++i) if (off[i + 1] < off[i]) return fail(c, NUTSB_E_INVAL, "offsets are not monotone%s");
    TRY(ensure(c, c->s_text, (size_t)(t1 - t0) + 64));
    if (t1 > t0) CK(cudaMemcpyAsync(c->s_text.p, bytes + t0, (size_t)(t1 - t0), cudaMemcpyHostToDevice, st));
    TRY(upload(c, c->s_toff, off, ((size_t)n + 1) * 8));
    TRY(ensure(c, c->s_gate, (size_t)n * 4)); TRY(ensure(c, c->d_sp_len, (size_t)n * 4));
    const u8 *dtext = c->s_text.as<u8>() - t0;
    NUTSB_LAUNCH(cdiv(n, 256), 256, st, k_colour_com_count, dtext, c->s_toff.as<u64>(), n, c->d_codetab.as<u8>(),
                 c->s_gate.as<i32>(), c->d_sp_len.as<u32>()); CKL();
    if (count) CK(cudaMemcpyAsync(count, c->s_gate.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    if (out_bytes) {
        TRY(ensure(c, c->d_sp_off, ((size_t)n + 1) * 8));
        TRY(run_scan(c, InU32{c->d_sp_len.as<u32>()}, OutU64{c->d_sp_off.as<u64>()}, n, nullptr));
        TRY(ensure(c, c->d_sp_text, (size_t)(t1 - t0) + 64));            // a stripped string is never longer
        NUTSB_LAUNCH(cdiv(n, 256), 256, st, k_colour_com_strip, dtext, c->s_toff.as<u64>(), n, c->d_codetab.as<u8>(),
                     c->d_sp_off.as<u64>(), c->d_sp_text.as<u8>()); CKL();
        TRY(ensure_host(c, c->h_out, (size_t)(t1 - t0) + 16));
        CK(cudaMemcpyAsync(c->h_off.p, c->d_sp_off.p, ((size_t)n + 1) * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(c->h_out.p, c->d_sp_text.p, (size_t)(t1 - t0), cudaMemcpyDeviceToHost, st));
        *out_bytes = c->h_out.as<u8>(); *out_off = c->h_off.as<u64>();
    }
    CK(cudaStreamSynchronize(st));
    c->have_streams = false;        // the pinned result buffers were reused
    return NUTSB_OK;
}
NUTSB_API int nutsb_colour_com_count_batch(nutsb_ctx *c, int64_t n, const uint8_t *b, const uint64_t *o, int32_t *count)
{ if (!count) return NUTSB_E_INVAL; return colour_com(c, n, b, o, count, nullptr, nullptr); }
NUTSB_API int nutsb_colour_com_strip_batch(nutsb_ctx *c, int64_t n, const uint8_t *b, const uint64_t *o, const uint8_t **ob, const uint64_t **oo)
{ if (!ob || !oo) return NUTSB_E_INVAL; return colour_com(c, n, b, o, nullptr, ob, oo); }

static int verdict_one(nutsb_ctx *c, int which, const char *s)
{
    if (!c || !s) return NUTSB_E_INVAL;
    const u64 off[2] = { 0, (u64)strlen(s) };
    u8 v = 0;
    const int rc = verdict_host(c, which, 1, (const u8 *)s, off, &v);
    return rc < 0 ? rc : (int)v;
}
NUTSB_API int nutsb_contains_swearing(nutsb_ctx *c, const char *s) { return verdict_one(c, V_SWEAR, s); }
NUTSB_API int nutsb_site_banned(nutsb_ctx *c, const char *s) { return verdict_one(c, V_SITE, s); }
NUTSB_API int nutsb_user_banned(nutsb_ctx *c, const char *s) { return verdict_one(c, V_USER, s); }

// ---------------------------------------------------------------------------------------
// queue tier
// ---------------------------------------------------------------------------------------
static int q_push_one(nutsb_ctx *c, u8 kind, i32 target, const char *str, size_t n, i32 except_user, u8 flags, i32 gate)
{
    if (n > NUTSB_MAX_TEXT) return fail(c, NUTSB_E_RANGE, "string longer than NUTSB_MAX_TEXT (2000) bytes%s");
    c->q.push(kind, target, (const u8 *)str, n, except_user, flags, gate);     // copied: callers reuse text[] at once
    return NUTSB_OK;
}

// colour_com_strip(), nuts333.c:2588-2610, on the host (what a peer older than 3.2 is sent, c:1300)
static std::string host_colour_com_strip(const char *s, size_t n)
{
    struct Tab { u8 t[NUTSB_CODETAB_BYTES]; Tab() { build_codetab(t); } };
    static const Tab T;                                  // C++11: initialised once, whatever the number of threads / contexts
    const u8 *tab = T.t;
    std::string o; o.reserve(n);
    for (size_t p = 0; p < n; ) {
        if (s[p] == '~' && p + 2 < n) {
            const u32 a = (u32)(u8)s[p + 1] - 'A', b = (u32)(u8)s[p + 2] - 'A';
            if (a < 26u && b < 26u && tab[a * 26u + b]) { p += 3; continue; }
        }
        o.push_back(s[p++]);
    }
    return o;
}

// write_user(u, str) as the queue sees it: a remote user's string is framed for its netlink
// (nuts333.c:1299-1306: "MSG <name>\n<str>[\n]EMSG\n", handed to write_sock unrendered), everybody else's is queued as it is.
static int q_push_user(nutsb_ctx *c, i32 u, const char *str, size_t n, u8 flags, i32 gate)
{
    if (u >= 0 && (size_t)u < c->remote_link.size() && c->remote_link[(size_t)u] >= 0) {
        if ((size_t)u + 1 >= c->name_off.size()) return fail(c, NUTSB_E_STATE, "nutsb_set_user_names does not match the population%s");
        std::string f = "MSG " + std::string((const char *)c->names.data() + c->name_off[(size_t)u], (size_t)(c->name_off[(size_t)u + 1] - c->name_off[(size_t)u])) + "\n";
        f += c->remote_old[(size_t)u] ? host_colour_com_strip(str, n) : std::string(str, n);
        if (f.back() != '\n' || f.size() == 5 + (size_t)(c->name_off[(size_t)u + 1] - c->name_off[(size_t)u])) f += "\n";
        f += "EMSG\n";
        return q_push_one(c, NUTSB_OP_USER, c->remote_link[(size_t)u], f.data(), f.size(), -1, (u8)((flags & NUTSB_OF_GATE_IF_SET) | NUTSB_OF_RAW), gate);
    }
    return q_push_one(c, NUTSB_OP_USER, u, str, n, -1, flags, gate);
}

// One call of the reference's write surface.  Besides the op itself:
//  * a room op that names a room with clones in it makes the relays of nuts333.c:1416-1426:
//    write_user(clone->owner, "~FT[ <room> ]:~RS <str>") for every clone that would have been a recipient;
//  * every remote user that would have been a recipient of a room / level op gets its frame (q_push_user).
// All of them at their place in the user list: before the op itself when a clone precedes its (local) owner
// there, after it otherwise, in list order -- and under the op's own gate.
// users flagged as clones / remote users need nutsb_set_clones / nutsb_set_remotes before anything is queued:
// without them their relays and frames would silently be missing
static int relays_ready(nutsb_ctx *c)
{
    if (c->n_clone_flag && (i32)c->clone_owner.size() != c->U) return fail(c, NUTSB_E_STATE, "users flagged NUTSB_UF_CLONE: nutsb_set_clones has not been called%s");
    if (c->n_remote_flag && (i32)c->remote_link.size() != c->U) return fail(c, NUTSB_E_STATE, "users flagged NUTSB_UF_REMOTE: nutsb_set_remotes has not been called%s");
    return NUTSB_OK;
}

static int q_push_impl(nutsb_ctx *c, u8 kind, i32 target, const char *str, size_t n, i32 except_user, u8 flags, i32 gate);

// all or nothing: a call that fails half-way (a relay or a frame longer than NUTSB_MAX_TEXT) leaves the queue as it was
static int q_push_n(nutsb_ctx *c, u8 kind, i32 target, const char *str, size_t n, i32 except_user, u8 flags, i32 gate = -1)
{
    if (!c || !str) return NUTSB_E_INVAL;
    if (c->has_clones) TRY(relays_ready(c));
    const HostOps::Mark m = c->q.mark();
    const int rc = q_push_impl(c, kind, target, str, n, except_user, flags, gate);
    if (rc != NUTSB_OK) c->q.rollback(m);
    return rc;
}
static int q_push(nutsb_ctx *c, u8 kind, i32 target, const char *str, i32 except_user, u8 flags, i32 gate = -1)
{
    if (!c || !str) return NUTSB_E_INVAL;
    return q_push_n(c, kind, target, str, strlen(str), except_user, flags, gate);
}

static int q_push_impl(nutsb_ctx *c, u8 kind, i32 target, const char *str, size_t n, i32 except_user, u8 flags, i32 gate)
{
    if (kind == NUTSB_OP_USER) return q_push_user(c, target, str, n, flags, gate);
    struct Extra { i32 pos, user; bool relay; };
    std::vector<Extra> before, after;
    if (kind == NUTSB_OP_ROOM && target >= 0 && (size_t)target < c->room_clones.size() && !c->room_clones[(size_t)target].empty()) {
        int swears = -1;
        for (i32 cl : c->room_clones[(size_t)target]) {
            const u32 uf = c->uflags[(size_t)cl];
            if (uf & NUTSB_UF_LOGIN) continue;                                              // c:1410
            if ((uf & NUTSB_UF_IGNALL) && !(flags & NUTSB_OF_FORCE_LISTEN)) continue;       // c:1413
            if ((uf & NUTSB_UF_IGNSHOUT) && (flags & NUTSB_OF_SHOUT)) continue;             // c:1414
            if (cl == except_user) continue;                                                // c:1415
            const i32 owner = c->clone_owner[(size_t)cl];
            const u8 hear = c->clone_hear[(size_t)cl];
            if (hear == 0 || (c->uflags[(size_t)owner] & NUTSB_UF_IGNALL)) continue;        // c:1417
            if (hear == 1) {                                                                // c:1421: CLONE_HEAR_SWEARS
                if (swears < 0) {
                    const u64 so[2] = { 0, (u64)n }; u8 v = 0; static const u8 zero = 0;
                    TRY(nutsb_contains_swearing_batch(c, 1, n ? (const u8 *)str : &zero, so, &v));
                    swears = v;
                }
                if (!swears) continue;
            }
            const bool local = !(c->uflags[(size_t)owner] & NUTSB_UF_REMOTE);
            (cl < owner && local ? before : after).push_back({ cl, owner, true });
        }
    }
    for (i32 u : c->remotes) {
        const u32 uf = c->uflags[(size_t)u];
        if (uf & NUTSB_UF_LOGIN) continue;
        if (kind == NUTSB_OP_ROOM) {                                                        // c:1410-1415
            const i32 ru = c->user_room[(size_t)u];
            if (ru >= c->R || (target >= 0 && ru != target)) continue;
            if ((uf & NUTSB_UF_IGNALL) && !(flags & NUTSB_OF_FORCE_LISTEN)) continue;
            if ((uf & NUTSB_UF_IGNSHOUT) && (flags & NUTSB_OF_SHOUT)) continue;
            if (u == except_user) continue;
        } else {                                                                            // c:1379-1383
            if (u == except_user) continue;
            if ((flags & NUTSB_OF_ABOVE) ? (i32)c->ulevel[(size_t)u] < target : (i32)c->ulevel[(size_t)u] > target) continue;
        }
        after.push_back({ u, u, false });
    }
    std::stable_sort(after.begin(), after.end(), [](const Extra &a, const Extra &b) { return a.pos < b.pos; });
    std::string relay;
    if (kind == NUTSB_OP_ROOM && target >= 0 && (!before.empty() || !after.empty())) {
        const std::string nm = (size_t)target < c->room_names.size() ? c->room_names[(size_t)target] : "room" + std::to_string(target);
        relay = "~FT[ " + nm + " ]:~RS " + std::string(str, n);                               // c:1424
    }
    const u8 rflags = (u8)(flags & NUTSB_OF_GATE_IF_SET);
    for (const Extra &e : before) TRY(q_push_user(c, e.user, relay.data(), relay.size(), rflags, gate));
    TRY(q_push_one(c, kind, target, str, n, except_user, flags, gate));
    for (const Extra &e : after) {
        if (e.relay) TRY(q_push_user(c, e.user, relay.data(), relay.size(), rflags, gate));
        else TRY(q_push_user(c, e.user, str, n, rflags, gate));
    }
    return NUTSB_OK;
}

// Clones (nuts333.h:58-62, 79): owner[u] = index of the clone's owner, -1 for everybody else (a clone is a
// user flagged NUTSB_UF_CLONE in nutsb_set_users); hear[u] = clone_hear (0 nothing, 1 swears, 2 all).
// Call after nutsb_set_users.  The relay is made by the queue tier's expansion, which the host-buffer batch
// calls use too; the other write calls refuse the population (begin_write).
NUTSB_API int nutsb_set_clones(nutsb_ctx *c, int32_t n_users, const int32_t *owner, const uint8_t *hear)
{
    if (!c || (n_users && (!owner || !hear))) return NUTSB_E_INVAL;
    if (!c->have_users || n_users != c->U) return fail(c, NUTSB_E_STATE, "nutsb_set_clones does not match the population%s");
    for (i32 u = 0; u < n_users; ++u) {
        const bool is_clone = (c->uflags[(size_t)u] & NUTSB_UF_CLONE) != 0;
        if (is_clone != (owner[u] >= 0)) return fail(c, NUTSB_E_INVAL, "owner[] and the NUTSB_UF_CLONE flags disagree%s");
        if (owner[u] >= n_users || (owner[u] >= 0 && (c->uflags[(size_t)owner[u]] & NUTSB_UF_CLONE)))
            return fail(c, NUTSB_E_RANGE, "clone owner out of range (or a clone itself)%s");
        if (hear[u] > 2) return fail(c, NUTSB_E_RANGE, "clone_hear is 0, 1 or 2%s");
    }
    c->clone_owner.assign(owner, owner + n_users); c->clone_hear.assign(hear, hear + n_users);
    c->room_clones.assign((size_t)c->R, std::vector<i32>());
    for (i32 u = 0; u < n_users; ++u)
        if (owner[u] >= 0 && c->user_room[(size_t)u] < c->R) c->room_clones[(size_t)c->user_room[(size_t)u]].push_back(u);
    return NUTSB_OK;
}

// Remote users: see include/nutsb200.h
NUTSB_API int nutsb_set_remotes(nutsb_ctx *c, int32_t n_users, const int32_t *link, const uint8_t *old_peer)
{
    if (!c || (n_users && (!link || !old_peer))) return NUTSB_E_INVAL;
    if (!c->have_users || n_users != c->U) return fail(c, NUTSB_E_STATE, "nutsb_set_remotes does not match the population%s");
    if (!c->have_names || (i32)c->sflags.size() != c->U) return fail(c, NUTSB_E_STATE, "nutsb_set_remotes needs nutsb_set_user_names%s");
    for (i32 u = 0; u < n_users; ++u) {
        const bool is_remote = (c->uflags[(size_t)u] & NUTSB_UF_REMOTE) != 0;
        if (is_remote != (link[u] >= 0)) return fail(c, NUTSB_E_INVAL, "link[] and the NUTSB_UF_REMOTE flags disagree%s");
        if (link[u] >= n_users) return fail(c, NUTSB_E_RANGE, "link pseudo-user out of range%s");
        if (link[u] >= 0 && ((c->uflags[(size_t)link[u]] & (NUTSB_UF_CLONE | NUTSB_UF_REMOTE)) || c->user_room[(size_t)link[u]] < c->R))
            return fail(c, NUTSB_E_INVAL, "a link pseudo-user is a plain user in no room%s");
    }
    c->remote_link.assign(link, link + n_users); c->remote_old.assign(old_peer, old_peer + n_users);
    c->remotes.clear();
    for (i32 u = 0; u < n_users; ++u) if (link[u] >= 0) c->remotes.push_back(u);
    return NUTSB_OK;
}

// rm->name of every room (the relay's prefix, review's header); rooms never named are "room<index>"
NUTSB_API int nutsb_set_room_names(nutsb_ctx *c, int32_t n_rooms, const uint8_t *names, const uint64_t *off)
{
    if (!c || n_rooms < 0 || (n_rooms && (!names || !off))) return NUTSB_E_INVAL;
    c->room_names.clear();
    for (i32 r = 0; r < n_rooms; ++r) {
        if (off[r + 1] < off[r] || off[r + 1] - off[r] > 20) return fail(c, NUTSB_E_RANGE, "room name longer than ROOM_NAME_LEN (20)%s");
        c->room_names.emplace_back((const char *)names + off[r], (size_t)(off[r + 1] - off[r]));
    }
    return NUTSB_OK;
}

NUTSB_API int nutsb_q_write_user(nutsb_ctx *c, int32_t user, const char *str) { return q_push(c, NUTSB_OP_USER, user, str, -1, 0); }
NUTSB_API int nutsb_q_write_room_except(nutsb_ctx *c, int32_t room, const char *str, int32_t except_user, int force_listen, int shout)
{ return q_push(c, NUTSB_OP_ROOM, room, str, except_user, (u8)((force_listen ? NUTSB_OF_FORCE_LISTEN : 0) | (shout ? NUTSB_OF_SHOUT : 0))); }
NUTSB_API int nutsb_q_write_room(nutsb_ctx *c, int32_t room, const char *str, int force_listen, int shout)
{ return nutsb_q_write_room_except(c, room, str, -1, force_listen, shout); }
NUTSB_API int nutsb_q_write_level(nutsb_ctx *c, int level, int above, const char *str, int32_t except_user)
{ return q_push(c, NUTSB_OP_LEVEL, level, str, except_user, above ? NUTSB_OF_ABOVE : 0); }
// write_sock(sock, str), nuts333.c:1281-1286, for a socket that is a user's (or a netlink's pseudo-user's): the
// bytes as they are, in order with everything else queued for that socket
NUTSB_API int nutsb_q_write_sock(nutsb_ctx *c, int32_t sock_user, const char *str)
{
    if (!c || !str) return NUTSB_E_INVAL;
    const HostOps::Mark m = c->q.mark();
    const int rc = q_push_one(c, NUTSB_OP_USER, sock_user, str, strlen(str), -1, NUTSB_OF_RAW, -1);
    if (rc != NUTSB_OK) c->q.rollback(m);
    return rc;
}
NUTSB_API int nutsb_q_page_line(nutsb_ctx *c, int32_t sock_user, const char *str, int plain)
{ return q_push(c, NUTSB_OP_USER, sock_user, str, -1, (u8)(NUTSB_OF_PAGER | (plain ? NUTSB_OF_PLAIN : 0))); }

// more(), nuts333.c:2205-2322, for a local user (the netlink branch, sock == -1, is out of scope).
NUTSB_API int nutsb_q_more(nutsb_ctx *c, int32_t user, int32_t sock_user, const void *file, size_t n,
                           int64_t *filepos, int *retval)
{
    if (!c || !filepos || !retval) return NUTSB_E_INVAL;
    if (!file) { if (user >= 0) *filepos = 0; *retval = 0; return NUTSB_OK; }        // c:2214-2217
    const u8 *f = (const u8 *)file;
    size_t pos = 0;
    if (user >= 0 && *filepos > 0) pos = (size_t)*filepos < n ? (size_t)*filepos : n;   // c:2219 fseek
    bool eof = false;
    std::string text;
    // fgets(text, sizeof(text)-1, fp): at most 1998 bytes, stops after '\n'; feof is raised only
    // when the read runs into the end of the file
    auto fgets_ = [&]() {
        size_t got = 0;
        std::string line;
        while (got < NUTSB_MAX_TEXT - 2) {
            if (pos >= n) { eof = true; break; }
            const u8 b = f[pos++]; line.push_back((char)b); ++got;
            if (b == '\n') break;
        }
        if (got) text = line;                          // NULL return leaves text untouched
    };
    int lines = 0; int64_t num_chars = 0;
    fgets_();
    while (!eof && (lines < 23 || user < 0)) {         // c:2237
        const size_t len = strlen(text.c_str());      // the chunk is used as a C string
        TRY(nutsb_q_page_line(c, sock_user, text.c_str(), user < 0));
        num_chars += (int64_t)len;
        lines += (int)(len / 80) + (len < 80);        // c:2303
        fgets_();
    }
    if (user < 0) { *retval = 2; return NUTSB_OK; }    // c:2309
    if (eof) { *filepos = 0; *retval = 2; return NUTSB_OK; }
    *filepos += num_chars;                             // c:2316
    TRY(nutsb_q_write_user(c, user, "           ~BB*** Press <return> to continue, 'e'<return> to exit ***"));
    *retval = 1;
    return NUTSB_OK;
}

NUTSB_API int64_t nutsb_q_pending(const nutsb_ctx *c) { return c ? (int64_t)c->q.n() : 0; }

// record(), nuts333.c:2062-2071
static void do_record(nutsb_ctx *c, i32 room, const char *str)
{
    if (room < 0 || room >= (i32)c->rev.size()) return;
    c->rev[(size_t)room].put(str, strnlen(str, NUTSB_REVIEW_LEN));
}

// The swear verdicts of the queued lines, taken in one device batch.
static int resolve_verdicts(nutsb_ctx *c)
{
    const i64 n_sw = (i64)c->q_sw_off.size() - 1;
    if ((i64)c->q_sw_verdict.size() < n_sw) {
        static const u8 zero = 0;
        std::vector<u8> v((size_t)n_sw, 0);
        TRY(nutsb_contains_swearing_batch(c, n_sw, c->q_sw_text.empty() ? &zero : c->q_sw_text.data(), c->q_sw_off.data(), v.data()));
        c->q_sw_verdict.swap(v);
    }
    return NUTSB_OK;
}

// ... and the record() calls that waited for them (a line refused for swearing is never recorded)
static int resolve_records(nutsb_ctx *c)
{
    TRY(resolve_verdicts(c));
    for (const auto &r : c->q_rec)
        if (r.gate < 0 || !c->q_sw_verdict[(size_t)r.gate]) do_record(c, r.room, r.text.c_str());
    c->q_rec.clear();
    return NUTSB_OK;
}

NUTSB_API int nutsb_q_record(nutsb_ctx *c, int32_t room, const char *str)
{
    if (!c || !str) return NUTSB_E_INVAL;
    if (room < 0 || room >= c->R) return fail(c, NUTSB_E_RANGE, "room index out of range%s");
    c->q_rec.push_back({ room, -1, std::string(str) });      // after the records still waiting for a verdict
    return NUTSB_OK;
}

NUTSB_API int nutsb_q_review_clear(nutsb_ctx *c, int32_t room)     // clear_revbuff(), c:2626
{
    if (!c) return NUTSB_E_INVAL;
    if (room < 0 || room >= c->R) return fail(c, NUTSB_E_RANGE, "room index out of range%s");
    TRY(resolve_records(c));
    for (auto &l : c->rev[(size_t)room].buf) l[0] = '\0';
    return NUTSB_OK;
}

// review(), nuts333.c:5192-5222, for a room the caller has resolved (get_room / has_room_access are the
// talker's): the buffered lines go through write_user again, oldest first.
NUTSB_API int nutsb_q_review(nutsb_ctx *c, int32_t user, int32_t room, const char *room_name)
{
    if (!c || !room_name) return NUTSB_E_INVAL;
    if (room < 0 || room >= c->R) return fail(c, NUTSB_E_RANGE, "room index out of range%s");
    TRY(resolve_records(c));
    const auto &rb = c->rev[(size_t)room];
    int cnt = 0;
    for (int i = 0; i < NUTSB_REVIEW_LINES; ++i) {
        const int line = (rb.line + i) % NUTSB_REVIEW_LINES;
        if (rb.buf[line][0]) {
            if (++cnt == 1) {
                const std::string head = std::string("\n~BB~FG*** Review buffer for the ") + room_name + " ***\n\n";
                TRY(nutsb_q_write_user(c, user, head.c_str()));
            }
            TRY(nutsb_q_write_user(c, user, rb.buf[line]));
        }
    }
    if (!cnt) return nutsb_q_write_user(c, user, "Review buffer is empty.\n");
    return nutsb_q_write_user(c, user, "\n~BB~FG*** End ***\n\n");
}

static void q_clear(nutsb_ctx *c)
{
    c->q.clear(); c->q_sw_text.clear(); c->q_sw_off.assign(1, 0); c->q_sw_verdict.clear(); c->q_rec.clear();
}

// Policy (include/nutsb200.h): the queue is emptied when the batch has run, or when it can never run (a
// validation error: the same ops would fail again).  After NUTSB_E_NOMEM / NUTSB_E_CUDA the queue -- ops,
// swear bodies, pending record() calls -- is kept as it was, so that the flush can be tried again; the review
// buffers take the pending lines only once the batch that delivers them has succeeded.
static int flush_impl(nutsb_ctx *c, const Result &r)
{
    if (!c || (!r.st && !r.iov)) return NUTSB_E_INVAL;
    // the swear verdicts the queued say/shout/emote lines branch on: one device batch (unless a review took them)
    int rc = resolve_verdicts(c);
    const i64 n_sw = (i64)c->q_sw_off.size() - 1;
    const nutsb_ops o = c->q.view(rc == NUTSB_OK && n_sw > 0 ? c->q_sw_verdict.data() : nullptr);
    if (rc == NUTSB_OK) rc = write_ops(c, &o, true, true, r);
    if (rc == NUTSB_OK) rc = resolve_records(c);
    if (rc != NUTSB_E_NOMEM && rc != NUTSB_E_CUDA) q_clear(c);
    return rc;
}
NUTSB_API int nutsb_flush(nutsb_ctx *c, nutsb_streams *out) { return flush_impl(c, { Result::HOST, out, nullptr }); }
NUTSB_API int nutsb_flush_iov(nutsb_ctx *c, nutsb_iov_streams *out) { return flush_impl(c, { Result::IOV, nullptr, out }); }

// The host-buffer batch tier.  With clones / remote users in the population every op goes through the
// queue tier's expansion (the relays of c:1416-1426, the frames of c:1299-1307, each under the op's own gate)
// before the batch runs, so that the streams are the reference's here too.
static int write_batch_public(nutsb_ctx *c, const nutsb_ops *o, const Result &r)
{
    if (!c || !c->has_clones) return write_ops(c, o, true, false, r);
    TRY(check_ops(c, o));
    if (!c->have_users) return fail(c, NUTSB_E_STATE, "nutsb_set_users has not been called%s");
    if (c->q.n() || !c->q_rec.empty()) return fail(c, NUTSB_E_STATE, "a batch over a population with clones / remote users needs an empty queue: flush first%s");
    const bool gated = o->gate && o->verdict;
    int rc = NUTSB_OK;
    for (i64 i = 0; i < o->n_ops && rc == NUTSB_OK; ++i) {
        const char *why = "";
        if ((rc = host_op_error(o, i, c->U, c->R, &why)) != NUTSB_OK) { rc = fail(c, rc, "%s", why); break; }
        if (o->kind[i] == NUTSB_OP_NONE) continue;
        static const char none = 0;
        const size_t n = (size_t)(o->text_off[i + 1] - o->text_off[i]);
        rc = q_push_n(c, o->kind[i], o->target[i], n ? (const char *)o->text + o->text_off[i] : &none, n, o->except_user[i], o->flags[i], gated ? o->gate[i] : -1);
    }
    if (rc == NUTSB_OK) {
        const nutsb_ops e = c->q.view(gated ? o->verdict : nullptr);
        rc = write_ops(c, &e, true, true, r);
    }
    q_clear(c);
    return rc;
}
NUTSB_API int nutsb_write_batch(nutsb_ctx *c, const nutsb_ops *o, nutsb_streams *out)
{ if (!out) return fail(c, NUTSB_E_INVAL, "null argument%s"); return write_batch_public(c, o, { Result::HOST, out, nullptr }); }
NUTSB_API int nutsb_write_batch_iov(nutsb_ctx *c, const nutsb_ops *o, nutsb_iov_streams *out)
{ if (!out) return fail(c, NUTSB_E_INVAL, "null argument%s"); return write_batch_public(c, o, { Result::IOV, nullptr, out }); }

// ---------------------------------------------------------------------------------------
// the callers' composition
// ---------------------------------------------------------------------------------------
NUTSB_API int nutsb_set_user_names(nutsb_ctx *c, int32_t n_users, const uint8_t *names, const uint64_t *off, const uint8_t *sflags)
{
    if (!c || n_users < 0 || (n_users && (!off || !sflags))) return fail(c, NUTSB_E_INVAL, "nutsb_set_user_names: bad argument%s");
    CK(cudaSetDevice(c->device));
    if (c->have_users && n_users != c->U) return fail(c, NUTSB_E_STATE, "nutsb_set_user_names does not match the population%s");
    for (i32 u = 0; u < n_users; ++u) if (off[u + 1] < off[u]) return fail(c, NUTSB_E_INVAL, "name offsets are not monotone%s");
    const u64 t0 = n_users ? off[0] : 0, t1 = n_users ? off[n_users] : 0;
    if (t1 > t0 && !names) return fail(c, NUTSB_E_INVAL, "names is NULL%s");
    c->names.assign(names ? names + t0 : nullptr, names ? names + t1 : nullptr);
    c->name_off.assign((size_t)n_users + 1, 0);
    for (i32 u = 0; u <= n_users; ++u) c->name_off[u] = n_users ? off[u] - t0 : 0;
    c->sflags.assign(sflags, sflags + n_users);
    TRY(upload(c, c->d_names, c->names.data(), c->names.size()));
    TRY(upload(c, c->d_name_off, c->name_off.data(), c->name_off.size() * 8));
    TRY(upload(c, c->d_sflags, c->sflags.data(), c->sflags.size()));
    CK(cudaStreamSynchronize(c->stream));
    c->have_names = true;
    return NUTSB_OK;
}

NUTSB_API int nutsb_set_ban_swearing(nutsb_ctx *c, int on) { if (!c) return NUTSB_E_INVAL; c->ban_swearing = on != 0; return NUTSB_OK; }

static int speech_ready(nutsb_ctx *c)
{
    if (!c->have_users) return fail(c, NUTSB_E_STATE, "nutsb_set_users has not been called%s");
    if (!c->have_names || (i32)c->sflags.size() != c->U) return fail(c, NUTSB_E_STATE, "nutsb_set_user_names does not match the population%s");
    return NUTSB_OK;
}

// queue tier: composed on the host with the same rules the device composer uses
NUTSB_API int nutsb_q_speech(nutsb_ctx *c, int verb, int32_t user, const char *inpstr)
{
    if (!c || !inpstr) return NUTSB_E_INVAL;
    TRY(speech_ready(c));
    if (verb < 0 || verb >= NUTSB_SPEECH_VERBS) return fail(c, NUTSB_E_INVAL, "unknown speech verb%s");
    if (user < 0 || user >= c->U) return fail(c, NUTSB_E_RANGE, "user index out of range%s");
    const size_t blen = strlen(inpstr);
    const u8 first = blen ? (u8)inpstr[0] : 0, last = blen ? (u8)inpstr[blen - 1] : 0;
    const i32 room = c->user_room[user] < c->R ? c->user_room[user] : -1;
    i32 gate = -1;
    for (u32 sidx = 0; sidx < 3; ++sidx) {
        const SpeechSlot sl = nutsb_speech_slot((u32)verb, sidx, user, room, c->sflags[user], c->ban_swearing, first, last);
        if (sl.kind == NUTSB_OP_NONE) continue;
        std::string text = c->lits[sl.a];
        if (sl.name == 2 || (sl.name == 1 && !(c->sflags[user] & NUTSB_SF_INVIS)))
            text.append((const char *)c->names.data() + c->name_off[user], (size_t)(c->name_off[user + 1] - c->name_off[user]));
        else if (sl.name == 1) text += c->lits[NUTSB_LIT_INVISNAME];
        text += c->lits[sl.b];
        if (sl.body == 1) text.append(inpstr, blen); else if (sl.body == 2 && blen) text.append(inpstr + 1, blen - 1);
        text += c->lits[sl.c];
        if (sl.gated && gate < 0) {    // the line's body joins the swear batch run at flush
            gate = (i32)c->q_sw_off.size() - 1;
            c->q_sw_text.insert(c->q_sw_text.end(), (const u8 *)inpstr, (const u8 *)inpstr + blen);
            c->q_sw_off.push_back((u64)c->q_sw_text.size());
        }
        TRY(q_push(c, sl.kind, sl.target, text.c_str(), sl.except_user, sl.flags, sl.gated ? gate : -1));
        // say, emote and echo record the line to the room in its review buffer (c:4099, c:4209, c:4304) --
        // once it is known not to be refused
        if (sidx == 2 && room >= 0 && (verb == NUTSB_SPEECH_SAY || verb == NUTSB_SPEECH_EMOTE || verb == NUTSB_SPEECH_ECHO))
            c->q_rec.push_back({ room, sl.gated ? gate : -1, text });
    }
    return NUTSB_OK;
}

// tell() c:4128, pemote() c:4234 after their argument checks (the target resolved by get_user, not the
// speaker, not afk / ignoring / offsite: the talker's state), wizshout() c:6527, revtell() c:7699.
static std::string user_name(const nutsb_ctx *c, i32 u)
{ return std::string((const char *)c->names.data() + c->name_off[(size_t)u], (size_t)(c->name_off[(size_t)u + 1] - c->name_off[(size_t)u])); }

static void do_record_tell(nutsb_ctx *c, i32 u, const char *str)     // record_tell(), c:2074
{
    c->revtell[(size_t)u].put(str, strnlen(str, NUTSB_REVIEW_LEN));
}

static int q_private(nutsb_ctx *c, int pemote, i32 user, i32 target, const char *inpstr)
{
    if (!c || !inpstr) return NUTSB_E_INVAL;
    TRY(speech_ready(c));
    if (user < 0 || user >= c->U || target < 0 || target >= c->U) return fail(c, NUTSB_E_RANGE, "user index out of range%s");
    if (c->sflags[(size_t)user] & NUTSB_SF_MUZZLED)
        return nutsb_q_write_user(c, user, pemote ? "You are muzzled, you cannot emote.\n" : "You are muzzled, you cannot tell anyone anything.\n");
    const size_t n = strlen(inpstr);
    const std::string name = (c->sflags[(size_t)user] & NUTSB_SF_INVIS) ? c->lits[NUTSB_LIT_INVISNAME] : user_name(c, user);
    const std::string tname = user_name(c, target), msg(inpstr, n);
    std::string a, b;
    if (pemote) {
        a = "~OL(To " + tname + ")~RS " + name + " " + msg + "\n";                    // c:4281
        b = "~OL>>~RS " + name + " " + msg + "\n";                                     // c:4283
    } else {
        const char *type = (n && inpstr[n - 1] == '?') ? "ask" : "tell";              // c:4175
        a = std::string("~OLYou ") + type + " " + tname + ":~RS " + msg + "\n";        // c:4177
        b = "~OL" + name + " " + type + "s you:~RS " + msg + "\n";                     // c:4180
    }
    TRY(nutsb_q_write_user(c, user, a.c_str()));
    TRY(nutsb_q_write_user(c, target, b.c_str()));
    do_record_tell(c, target, b.c_str());
    return NUTSB_OK;
}
NUTSB_API int nutsb_q_tell(nutsb_ctx *c, int32_t user, int32_t target, const char *inpstr) { return q_private(c, 0, user, target, inpstr); }
NUTSB_API int nutsb_q_pemote(nutsb_ctx *c, int32_t user, int32_t target, const char *inpstr) { return q_private(c, 1, user, target, inpstr); }

// inpstr = the whole line as wizshout() receives it.  lev < 0: no level word, everybody from WIZ up (c:6560-6564);
// else the form "to level <level_name>" (c:6552-6557; lev >= WIZ and <= the speaker's level are the caller's checks):
// the level word is taken off here (remove_first, c:2350) -- after the ban_swearing check, which the reference asks
// of the whole line (c:6541), level word included
NUTSB_API int nutsb_q_wizshout(nutsb_ctx *c, int32_t user, int lev, const char *level_name, const char *inpstr)
{
    if (!c || !inpstr || (lev >= 0 && !level_name)) return NUTSB_E_INVAL;
    TRY(speech_ready(c));
    if (user < 0 || user >= c->U) return fail(c, NUTSB_E_RANGE, "user index out of range%s");
    if (c->sflags[(size_t)user] & NUTSB_SF_MUZZLED) return nutsb_q_write_user(c, user, "You are muzzled, you cannot wizshout.\n");
    const size_t n_all = strlen(inpstr);
    const HostOps::Mark m = c->q.mark();
    const size_t sw_text = c->q_sw_text.size(), sw_off = c->q_sw_off.size();
    i32 gate = -1;
    int rc = NUTSB_OK;
    if (c->ban_swearing) {                                           // c:6541, asked of the whole line
        gate = (i32)c->q_sw_off.size() - 1;
        c->q_sw_text.insert(c->q_sw_text.end(), (const u8 *)inpstr, (const u8 *)inpstr + n_all);
        c->q_sw_off.push_back((u64)c->q_sw_text.size());
        rc = q_push(c, NUTSB_OP_USER, user, c->lits[6].c_str(), -1, NUTSB_OF_GATE_IF_SET, gate);
    }
    const char *body = inpstr;
    if (lev >= 0) {                                                  // remove_first(), c:2350-2358 (char is signed there)
        while ((signed char)*body < 33 && *body) ++body;
        while ((signed char)*body > 32) ++body;
        while ((signed char)*body < 33 && *body) ++body;
    }
    const std::string msg(body), to = lev >= 0 ? std::string(" to level ") + level_name : std::string();
    const std::string a = "~OLYou wizshout" + to + ":~RS " + msg + "\n";
    const std::string b = "~OL" + user_name(c, user) + " wizshouts" + to + ":~RS " + msg + "\n";
    if (rc == NUTSB_OK) rc = q_push(c, NUTSB_OP_USER, user, a.c_str(), -1, 0, gate);
    if (rc == NUTSB_OK) rc = q_push(c, NUTSB_OP_LEVEL, lev >= 0 ? lev : 2 /* WIZ */, b.c_str(), user, NUTSB_OF_ABOVE, gate);
    if (rc != NUTSB_OK) { c->q.rollback(m); c->q_sw_text.resize(sw_text); c->q_sw_off.resize(sw_off); }
    return rc;
}

NUTSB_API int nutsb_q_revtell(nutsb_ctx *c, int32_t user)
{
    if (!c) return NUTSB_E_INVAL;
    if (user < 0 || user >= c->U || (size_t)user >= c->revtell.size()) return fail(c, NUTSB_E_RANGE, "user index out of range%s");
    const auto &rb = c->revtell[(size_t)user];
    int cnt = 0;
    for (int i = 0; i < NUTSB_REVTELL_LINES; ++i) {
        const int line = (rb.line + i) % NUTSB_REVTELL_LINES;
        if (rb.buf[line][0]) {
            if (++cnt == 1) TRY(nutsb_q_write_user(c, user, "\n~BB~FG*** Your revtell buffer ***\n\n"));
            TRY(nutsb_q_write_user(c, user, rb.buf[line]));
        }
    }
    if (!cnt) return nutsb_q_write_user(c, user, "Revtell buffer is empty.\n");
    return nutsb_q_write_user(c, user, "\n~BB~FG*** End ***\n\n");
}

// The records of a composed speech batch (k lines, ops 3j..3j+2 in d_sp_*, verdicts in d_sp_verdict), packed in
// d_rec_out (nutsb_speech.cuh); their size goes to h_small at byte 2048, which run_write's synchronisations make
// readable.  On the main stream: the scans and the sort share its scan state with run_write's planning.
static int speech_records(nutsb_ctx *c, i64 k, const u8 *verb, const SpeechShard &sh, bool shard)
{
    cudaStream_t st = c->stream;
    const u32 R = (u32)c->R;
    u64 *h_total = c->h_small.as<u64>() + 256;
    if (R == 0 || k == 0) { *h_total = 0; return NUTSB_OK; }
    const size_t kk = (size_t)k;
    TRY(ensure(c, c->d_rec_key, kk * 4)); TRY(ensure(c, c->d_rec_line, kk * 4)); TRY(ensure(c, c->d_rec_cnt, 16));
    for (int q = 0; q < 2; ++q) { TRY(ensure(c, c->d_rec_k[q], kk * 4 + 16)); TRY(ensure(c, c->d_rec_v[q], kk * 4 + 16)); }   // radix_sort's sizes
    TRY(ensure(c, c->d_rec_seg, ((size_t)R + 1) * 4)); TRY(ensure(c, c->d_rec_lens, (size_t)R * 16));
    TRY(ensure(c, c->d_rec_bytes, (size_t)R * 4)); TRY(ensure(c, c->d_rec_off, ((size_t)R + 1) * 8));
    const size_t rooms = std::min<size_t>(R, kk), lines = std::min<size_t>(kk, (size_t)R * NUTSB_REVIEW_LINES);
    TRY(ensure(c, c->d_rec_out, rooms * NUTSB_REC_HEAD + lines * NUTSB_REVIEW_LEN + 16));
    u32 *key = c->d_rec_key.as<u32>(), *line = c->d_rec_line.as<u32>(), *cnt = c->d_rec_cnt.as<u32>();
    if (shard) { NUTSB_LAUNCH(cdiv(kk, 256), 256, st, k_speech_rec_mark<true>, verb, sh, k, c->d_sp_kind.as<u8>(), c->d_sp_target.as<i32>(), c->d_sp_gate.as<i32>(), c->d_sp_verdict.as<u8>(), key); }
    else       { NUTSB_LAUNCH(cdiv(kk, 256), 256, st, k_speech_rec_mark<false>, verb, sh, k, c->d_sp_kind.as<u8>(), c->d_sp_target.as<i32>(), c->d_sp_gate.as<i32>(), c->d_sp_verdict.as<u8>(), key); }
    CKL();
    TRY(run_scan(c, InRecKey{key}, OutRec{key, c->d_rec_k[0].as<u32>(), line, cnt, k}, k, nullptr));
    u32 *keys = nullptr, *vals = nullptr;
    TRY(radix_sort(c, c->d_rec_k, c->d_rec_v, k, cnt, bits_for(R), &keys, &vals));
    u32 *seg = c->d_rec_seg.as<u32>();
    NUTSB_LAUNCH(cdiv(kk + 1, 256), 256, st, k_speech_rec_bounds, keys, cnt, k, R, seg); CKL();
    NUTSB_LAUNCH(cdiv((u64)R * 32, 256), 256, st, k_speech_rec_tail, seg, vals, line, c->d_sp_off.as<u64>(), c->d_sp_text.as<u8>(), R,
                 c->d_rec_lens.as<u8>(), c->d_rec_bytes.as<u32>()); CKL();
    TRY(run_scan(c, InU32{c->d_rec_bytes.as<u32>()}, OutU64{c->d_rec_off.as<u64>()}, (i64)R, nullptr));
    NUTSB_LAUNCH(cdiv((u64)R * 32, 256), 256, st, k_speech_rec_pack, seg, vals, line, c->d_sp_off.as<u64>(), c->d_sp_text.as<u8>(), R,
                 c->d_rec_lens.as<u8>(), c->d_rec_off.as<u64>(), c->d_rec_out.as<u8>()); CKL();
    CK(cudaMemcpyAsync(h_total, c->d_rec_off.as<u64>() + R, 8, cudaMemcpyDeviceToHost, st));
    return NUTSB_OK;
}

// The packed records to the host (h_rec) once run_write has synchronised: one copy of the bytes they keep.
static int fetch_records(nutsb_ctx *c)
{
    CK(cudaStreamSynchronize(c->stream));
    const u64 total = c->h_small.as<u64>()[256];
    TRY(ensure_host(c, c->h_rec, (size_t)total + 16));
    if (total) {
        CK(cudaMemcpyAsync(c->h_rec.p, c->d_rec_out.p, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    c->rec_total = total; c->rec_ready = true;
    return NUTSB_OK;
}

// ... and into the rings: room r's c records end at (line + c) % REVIEW_LINES, the last min(c, REVIEW_LINES) of them
// where record() would have put them.
static void apply_records(nutsb_ctx *c)
{
    const u8 *p = c->h_rec.as<u8>(), *end = p + c->rec_total;
    while (p < end) {
        u32 room, cnt;
        memcpy(&room, p, 4); memcpy(&cnt, p + 4, 4);
        const u8 *lens = p + 8;
        const u32 t = std::min<u32>(cnt, NUTSB_REVIEW_LINES);
        const u8 *text = p + NUTSB_REC_HEAD;
        auto &rb = c->rev[room];
        rb.line = (int)((rb.line + (cnt - t)) % NUTSB_REVIEW_LINES);
        for (u32 i = 0; i < t; ++i) { rb.put(text, lens[i]); text += lens[i]; }
        p = text;
    }
    c->rec_ready = false;
}

NUTSB_API int nutsb_set_speech_record(nutsb_ctx *c, int on) { if (!c) return NUTSB_E_INVAL; c->speech_record = on != 0; return NUTSB_OK; }

NUTSB_API int nutsb_get_review_buffer(nutsb_ctx *c, int32_t room, uint8_t *rows, int32_t *line)
{
    if (!c) return NUTSB_E_INVAL;
    if (room < 0 || room >= (i32)c->rev.size()) return fail(c, NUTSB_E_RANGE, "room index out of range%s");
    const auto &rb = c->rev[(size_t)room];
    if (rows) memcpy(rows, rb.buf, sizeof rb.buf);
    if (line) *line = rb.line;
    return NUTSB_OK;
}

// shard: the context is one shard of a nutsb_multi, the speakers are global user indices, and only the lines
// that produce an op on this shard are composed (k_speech_route, then a scan compacts their indices)
static int run_speech(nutsb_ctx *c, i64 n, const u8 *verb, const i32 *speaker, const u8 *bodies, const u64 *body_off, nutsb_streams *out,
                      IovReq *iv, bool shard = false)
{
    TRY(speech_ready(c));
    if (shard && (!c->have_g_names || c->shard < 0)) return fail(c, NUTSB_E_STATE, "nutsb_multi_set_user_names does not match the population%s");
    cudaStream_t st = c->stream;
    c->h_small.as<u64>()[256] = 0;                             // no records until speech_records says otherwise
    if (n == 0) { nutsb_ops o{}; return run_write(c, &o, out, iv); }
    SpeechView v{ n, verb, speaker, bodies, body_off, c->d_names.as<u8>(), c->d_name_off.as<u64>(), c->d_sflags.as<u8>(),
                  c->d_user_room.as<i32>(), c->d_lit.as<u8>(), c->d_lit_off.as<u32>(), c->U, c->R, c->ban_swearing ? 1u : 0u };
    SpeechShard sh{};
    u64 *h64 = c->h_small.as<u64>(); u32 *h32 = c->h_small.as<u32>();
    i64 k = n;                                                 // the lines composed here
    if (shard) {
        v.names = c->d_g_names.as<u8>(); v.name_off = c->d_g_name_off.as<u64>(); v.sflags = c->d_g_sflags.as<u8>(); v.n_users = c->g_U;
        sh = SpeechShard{ nullptr, 0, c->d_g_user_shard.as<i32>(), c->d_g_user_local.as<i32>(), c->d_g_has_room.as<u8>(), c->shard };
        TRY(ensure(c, c->d_sp_keep, (size_t)n)); TRY(ensure(c, c->d_sp_sel, ((size_t)n + 1) * 4));
    }
    const size_t n3 = (size_t)n * 3;
    TRY(ensure(c, c->d_sp_len, n3 * 4)); TRY(ensure(c, c->d_sp_off, (n3 + 1) * 8));
    TRY(ensure(c, c->d_sp_kind, n3)); TRY(ensure(c, c->d_sp_flags, n3));
    TRY(ensure(c, c->d_sp_target, n3 * 4)); TRY(ensure(c, c->d_sp_except, n3 * 4)); TRY(ensure(c, c->d_sp_gate, n3 * 4));
    TRY(ensure(c, c->d_sp_verdict, (size_t)n));
    CK(cudaMemsetAsync(c->d_status.p, 0, 64, st));
    if (shard) {
        i32 *sel = c->d_sp_sel.as<i32>();
        NUTSB_LAUNCH(cdiv(n, 256), 256, st, k_speech_route, v, sh, c->d_sp_keep.as<u8>(), c->d_status.as<u32>()); CKL();
        TRY(run_scan(c, InU8{c->d_sp_keep.as<u8>()}, OutSel{c->d_sp_keep.as<u8>(), sel, n}, n, nullptr));
        CK(cudaMemcpyAsync(h32, sel + n, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        k = (i64)h32[0]; sh.sel = sel; sh.k = k;
        if (k == 0) {                                          // nothing lands here (the line checks still count)
            CK(cudaMemcpyAsync(h32 + 4, c->d_status.p, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            TRY(status_to_error(c, h32[4]));
            nutsb_ops o{}; return run_write(c, &o, out, iv);
        }
    }
    const size_t k3 = (size_t)k * 3;
    if (shard) { NUTSB_LAUNCH(cdiv(k, 256), 256, st, k_speech_measure<true>, v, sh, c->d_sp_len.as<u32>(), c->d_status.as<u32>()); }
    else       { NUTSB_LAUNCH(cdiv(n, 256), 256, st, k_speech_measure<false>, v, sh, c->d_sp_len.as<u32>(), c->d_status.as<u32>()); }
    CKL();
    TRY(run_scan(c, InU32{c->d_sp_len.as<u32>()}, OutU64{c->d_sp_off.as<u64>()}, (i64)k3, nullptr));
    CK(cudaMemcpyAsync(h64, c->d_sp_off.as<u64>() + k3, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h32 + 4, c->d_status.p, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    TRY(status_to_error(c, h32[4]));
    const u64 text_bytes = h64[0];
    TRY(ensure(c, c->d_sp_text, text_bytes + 64));
    if (shard) {
        NUTSB_LAUNCH(cdiv((u64)k * NUTSB_SPEECH_GROUP, 256), 256, st, k_speech_compose<true>, v, sh, c->d_sp_off.as<u64>(), c->d_sp_text.as<u8>(),
                     c->d_sp_kind.as<u8>(), c->d_sp_target.as<i32>(), c->d_sp_except.as<i32>(), c->d_sp_flags.as<u8>(), c->d_sp_gate.as<i32>());
    } else {
        NUTSB_LAUNCH(cdiv((u64)n * NUTSB_SPEECH_GROUP, 256), 256, st, k_speech_compose<false>, v, sh, c->d_sp_off.as<u64>(), c->d_sp_text.as<u8>(),
                     c->d_sp_kind.as<u8>(), c->d_sp_target.as<i32>(), c->d_sp_except.as<i32>(), c->d_sp_flags.as<u8>(), c->d_sp_gate.as<i32>());
    }
    CKL();
    // the verdicts of every line: a shard delivers gated shouts of speakers who live elsewhere (the gates are line indices)
    TRY(verdict_dev(c, V_SWEAR, n, bodies, body_off, c->d_sp_verdict.as<u8>()));
    if (c->speech_record) TRY(speech_records(c, k, verb, sh, shard));
    nutsb_ops o{ (i64)k3, c->d_sp_text.as<u8>(), c->d_sp_off.as<u64>(), c->d_sp_kind.as<u8>(), c->d_sp_target.as<i32>(),
                 c->d_sp_except.as<i32>(), c->d_sp_flags.as<u8>(), c->d_sp_gate.as<i32>(), c->d_sp_verdict.as<u8>() };
    return run_write(c, &o, out, iv);
}

// the n input lines of a speech batch, host memory -> staging buffers in HBM (the pointers are replaced by theirs)
static int upload_speech(nutsb_ctx *c, i64 n, const u8 *&verb, const i32 *&speaker, const u8 *&bodies, const u64 *&body_off)
{
    cudaStream_t st = c->stream;
    TRY(ev_record(c, EV_H2D0, st));
    if (n <= 0) return ev_record(c, EV_H2D1, st);
    const u64 t0 = body_off[0], t1 = body_off[n];
    if (t1 < t0 || (t1 > t0 && !bodies)) return fail(c, NUTSB_E_INVAL, "bad body offsets%s");
    // (offsets that are not monotone inside [t0, t1] are caught on the device: k_speech_measure)
    TRY(ensure(c, c->s_body, (size_t)(t1 - t0) + 64));
    if (t1 > t0) CK(cudaMemcpyAsync(c->s_body.p, bodies + t0, (size_t)(t1 - t0), cudaMemcpyHostToDevice, st));
    TRY(upload(c, c->s_boff, body_off, ((size_t)n + 1) * 8));
    TRY(upload(c, c->s_verb, verb, (size_t)n));
    TRY(upload(c, c->s_speaker, speaker, (size_t)n * 4));
    verb = c->s_verb.as<u8>(); speaker = c->s_speaker.as<i32>(); bodies = c->s_body.as<u8>() - t0; body_off = c->s_boff.as<u64>();
    return ev_record(c, EV_H2D1, st);
}

// A speech batch: the input lines in HBM or (upload) in host memory, composed on the device
static int speech_batch(nutsb_ctx *c, i64 n, const u8 *verb, const i32 *speaker, const u8 *bodies, const u64 *body_off,
                        bool upload, const Result &r, bool shard = false)
{
    if (!c || (!r.st && !r.iov) || n < 0 || (n && (!verb || !speaker || !body_off))) return fail(c, NUTSB_E_INVAL, "bad argument%s");
    c->rec_ready = false;
    if (c->speech_record && !c->q_rec.empty())
        return fail(c, NUTSB_E_STATE, "record() calls are pending in the queue: flush first%s");
    TRY(begin_write(c, false));
    if (upload) TRY(upload_speech(c, n, verb, speaker, bodies, body_off));
    nutsb_streams ds{}; IovReq iv;
    TRY(run_speech(c, n, verb, speaker, bodies, body_off, &ds, r.form == Result::IOV ? &iv : nullptr, shard));
    if (c->speech_record) TRY(fetch_records(c));             // before the result is handed over: an error leaves it untouched
    TRY(deliver(c, upload, ds, iv, r));
    if (c->speech_record && !shard) apply_records(c);          // (nutsb_multi applies every shard's once all have succeeded)
    return NUTSB_OK;
}

NUTSB_API int nutsb_speech_batch_dev(nutsb_ctx *c, int64_t n, const uint8_t *verb, const int32_t *speaker,
                                     const uint8_t *bodies, const uint64_t *body_off, nutsb_streams *out)
{ return speech_batch(c, n, verb, speaker, bodies, body_off, false, { Result::HBM, out, nullptr }); }

NUTSB_API int nutsb_speech_batch(nutsb_ctx *c, int64_t n, const uint8_t *verb, const int32_t *speaker,
                                 const uint8_t *bodies, const uint64_t *body_off, nutsb_streams *out)
{ return speech_batch(c, n, verb, speaker, bodies, body_off, true, { Result::HOST, out, nullptr }); }

// input lines in, gather lists out: the smallest host <-> device traffic the path has (bodies + 5 bytes per
// line one way; each rendering once per colour setting + 16 bytes per piece the other)
NUTSB_API int nutsb_speech_batch_iov(nutsb_ctx *c, int64_t n, const uint8_t *verb, const int32_t *speaker,
                                     const uint8_t *bodies, const uint64_t *body_off, nutsb_iov_streams *out)
{ return speech_batch(c, n, verb, speaker, bodies, body_off, true, { Result::IOV, nullptr, out }); }

#include "nutsb_multi.cuh"
