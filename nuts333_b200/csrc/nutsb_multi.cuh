// nutsb_multi.cuh -- one population, one batch, several GPUs (included at the end of nutsb_lib.cu).
//
// The path shards by room with no exchange step (SURVEY.md 8e): what a user receives depends on the
// ops that name his room, himself or his level, and on nobody else's stream.  So:
//   * rooms are dealt to the shards, heaviest first onto the least loaded shard (weight = the room's
//     population unless the caller gives one per room: population x expected traffic); a room's users go
//     with it; users in no room (user->room == NULL) go to the least loaded shard;
//   * a batch is routed on the host: write_user(u) -> the shard of u; write_room[_except](rm) -> the shard
//     of rm; the all-room forms (rm == NULL: shout, bcast, system messages, nuts333.c:1399-1400,
//     4119-4123, 4783-4787) and write_level (c:1372-1385) are REPLICATED to every shard, each rendering
//     for its own users; user / room indices become the shard's local ones, an excluded user who lives
//     elsewhere becomes "nobody" (he is in none of this shard's rooms); swear verdicts are replicated;
//   * every shard runs on its own device, one host thread each, no collective; the results come back in
//     GLOBAL user order: streams (nutsb_mstreams) or gather lists (nutsb_miov_streams), by pointer
//     bookkeeping over the shards' own results;
//   * a speech batch (nutsb_multi_speech_batch*) is not routed on the host: every shard is given the whole
//     batch and picks the lines that produce an op on it on the device (k_speech_route), by the rule the one-
//     context composer uses (nutsb_speech_slot).
// A shard whose context is absent (nutsb_multi_create_rank: one process per GPU, torchrun) is planned and
// routed but not run: its users' streams are reported empty by this process.
#include <thread>

#ifdef NUTSB_CPUSIM           // the emulator's launch state is process-global: the shards run one after the other there
#define NUTSB_MULTI_SERIAL(th) do { (th).back().join(); (th).pop_back(); } while (0)
#else
#define NUTSB_MULTI_SERIAL(th) do { } while (0)
#endif

struct nutsb_multi {
    int n_shards = 0;
    bool rank = false;                            // nutsb_multi_create_rank: this process runs one shard
    std::vector<nutsb_ctx *> ctx;                 // [n_shards], null = not run by this process
    std::string err;
    // plan
    bool have_users = false;
    i32 U = 0, R = 0;
    std::vector<i32> room_shard, room_local, user_shard, user_local;
    std::vector<std::vector<i32>> shard_users;     // global index of each shard's users, in global order
    std::vector<i32> shard_rooms;                  // rooms per shard
    // speech: the global names / speech flags (nutsb_multi_set_user_names), pushed to the shards with the plan
    bool have_names = false;
    std::vector<u8> names, sflags; std::vector<u64> name_off;
    // routed batch and result, per shard
    struct Routed { HostOps ops; nutsb_streams out{}; nutsb_iov_streams iov{}; nutsb_timing tm{}; int rc = NUTSB_OK; };
    std::vector<Routed> routed;
    // merged result
    std::vector<u64> len; std::vector<const u8 *> ptr;
    std::vector<const nutsb_iovec *> iov; std::vector<u32> count;
    std::vector<u64> dg_local;
    // every room's review buffer in global order, taken from the last plan that was set up whole, until a re-plan
    // succeeds (one that fails half way has already reshaped some shards' buffers: its retry starts from these)
    std::vector<nutsb_ctx::RevBuf> rev_carry; bool carry = false;
};

static int mfail(nutsb_multi *m, int code, const char *msg) { if (m) m->err = msg; return code; }

NUTSB_API const char *nutsb_multi_last_error(const nutsb_multi *m) { return m ? m->err.c_str() : ""; }
NUTSB_API int nutsb_multi_n_shards(const nutsb_multi *m) { return m ? m->n_shards : 0; }
NUTSB_API nutsb_ctx *nutsb_multi_ctx(nutsb_multi *m, int shard) { return (m && shard >= 0 && shard < m->n_shards) ? m->ctx[(size_t)shard] : nullptr; }

NUTSB_API void nutsb_multi_destroy(nutsb_multi *m)
{
    if (!m) return;
    for (nutsb_ctx *c : m->ctx) if (c) nutsb_destroy(c);
    delete m;
}

static int multi_create(nutsb_multi **out, int n_shards, const int *device_ids, int only_shard)
{
    if (!out || n_shards <= 0 || !device_ids) return NUTSB_E_INVAL;
    *out = nullptr;
    nutsb_multi *m = new (std::nothrow) nutsb_multi;
    if (!m) return NUTSB_E_NOMEM;
    m->n_shards = n_shards;
    m->rank = only_shard >= 0;
    m->ctx.assign((size_t)n_shards, nullptr);
    m->routed.resize((size_t)n_shards);
    for (int s = 0; s < n_shards; ++s) {
        if (only_shard >= 0 && s != only_shard) continue;
        const int rc = nutsb_create(&m->ctx[(size_t)s], device_ids[only_shard >= 0 ? 0 : s]);
        if (rc != NUTSB_OK) { nutsb_multi_destroy(m); return rc; }
    }
    *out = m;
    return NUTSB_OK;
}

// one context per entry of device_ids (the same device may be named twice: two shards on one GPU)
NUTSB_API int nutsb_multi_create(nutsb_multi **out, const int *device_ids, int n_devices)
{ return multi_create(out, n_devices, device_ids, -1); }

// one process per GPU: this process runs shard `shard` of `n_shards` on `device`; the other shards are planned
// and routed (every process must be given the same population and the same batches) but not run here
NUTSB_API int nutsb_multi_create_rank(nutsb_multi **out, int n_shards, int shard, int device)
{
    if (shard < 0 || shard >= n_shards) return NUTSB_E_INVAL;
    return multi_create(out, n_shards, &device, shard);
}

#define MEACH(call) do { for (nutsb_ctx *c_ : m->ctx) if (c_) { const int rc_ = (call); if (rc_ != NUTSB_OK) { m->err = nutsb_last_error(c_); return rc_; } } } while (0)

NUTSB_API int nutsb_multi_set_swear_words(nutsb_multi *m, const char *const *words)
{ if (!m) return NUTSB_E_INVAL; MEACH(nutsb_set_swear_words(c_, words)); return NUTSB_OK; }
NUTSB_API int nutsb_multi_set_ban_files(nutsb_multi *m, const void *siteban, size_t sn, const void *userban, size_t un)
{ if (!m) return NUTSB_E_INVAL; MEACH(nutsb_set_ban_files(c_, siteban, sn, userban, un)); return NUTSB_OK; }
NUTSB_API int nutsb_multi_set_profiling(nutsb_multi *m, int on)
{ if (!m) return NUTSB_E_INVAL; MEACH(nutsb_set_profiling(c_, on)); return NUTSB_OK; }

// The speech batch's view of the global population on shard s's device: which shard and local index every user
// has, and whether the user is in a room.
static int shard_tables(nutsb_ctx *c, int s, const nutsb_multi *m, const int32_t *room)
{
    std::vector<u8> has_room((size_t)m->U);
    for (i32 u = 0; u < m->U; ++u) has_room[(size_t)u] = room[u] >= 0;
    c->shard = s; c->g_U = m->U; c->have_g_names = false;
    TRY(upload(c, c->d_g_user_shard, m->user_shard.data(), (size_t)m->U * 4));
    TRY(upload(c, c->d_g_user_local, m->user_local.data(), (size_t)m->U * 4));
    TRY(upload(c, c->d_g_has_room, has_room.data(), (size_t)m->U));
    CK(cudaStreamSynchronize(c->stream));                      // has_room goes out of scope
    return NUTSB_OK;
}

// The names to every shard this process runs: its own users' (nutsb_set_user_names: its queue tier) and the global
// table (the speech batch's names, which a shard needs for the shouts of speakers who live elsewhere).
static int multi_push_names(nutsb_multi *m)
{
    for (int s = 0; s < m->n_shards; ++s) {
        nutsb_ctx *c = m->ctx[(size_t)s];
        if (!c) continue;
        const std::vector<i32> &us = m->shard_users[(size_t)s];
        std::vector<u8> ln, lf(us.size()); std::vector<u64> lo(us.size() + 1, 0);
        for (size_t i = 0; i < us.size(); ++i) {
            const size_t u = (size_t)us[i];
            ln.insert(ln.end(), m->names.begin() + (ptrdiff_t)m->name_off[u], m->names.begin() + (ptrdiff_t)m->name_off[u + 1]);
            lo[i + 1] = ln.size(); lf[i] = m->sflags[u];
        }
        static const u8 zb = 0;
        int rc = nutsb_set_user_names(c, (i32)us.size(), ln.empty() ? &zb : ln.data(), lo.data(), lf.empty() ? &zb : lf.data());
        if (rc == NUTSB_OK) rc = [&]() -> int {
            c->have_g_names = false;
            TRY(upload(c, c->d_g_names, m->names.data(), m->names.size()));
            TRY(upload(c, c->d_g_name_off, m->name_off.data(), m->name_off.size() * 8));
            TRY(upload(c, c->d_g_sflags, m->sflags.data(), m->sflags.size()));
            CK(cudaStreamSynchronize(c->stream));
            c->have_g_names = true;
            return NUTSB_OK;
        }();
        if (rc != NUTSB_OK) { m->err = nutsb_last_error(c); return rc; }
    }
    return NUTSB_OK;
}

// user->name, user->vis, user->muzzled of every user in GLOBAL order (as nutsb_set_user_names); may come before or
// after nutsb_multi_set_users, and is given to the shards whenever the plan changes.
NUTSB_API int nutsb_multi_set_user_names(nutsb_multi *m, int32_t n_users, const uint8_t *names, const uint64_t *off, const uint8_t *sflags)
{
    if (!m || n_users < 0 || (n_users && (!off || !sflags))) return mfail(m, NUTSB_E_INVAL, "nutsb_multi_set_user_names: bad argument");
    if (m->have_users && n_users != m->U) return mfail(m, NUTSB_E_STATE, "nutsb_multi_set_user_names does not match the population");
    for (i32 u = 0; u < n_users; ++u) if (off[u + 1] < off[u]) return mfail(m, NUTSB_E_INVAL, "name offsets are not monotone");
    const u64 t0 = n_users ? off[0] : 0, t1 = n_users ? off[n_users] : 0;
    if (t1 > t0 && !names) return mfail(m, NUTSB_E_INVAL, "names is NULL");
    m->have_names = false;
    m->names.assign(names ? names + t0 : nullptr, names ? names + t1 : nullptr);
    m->name_off.assign((size_t)n_users + 1, 0);
    for (i32 u = 0; u <= n_users; ++u) m->name_off[(size_t)u] = n_users ? off[u] - t0 : 0;
    m->sflags.assign(sflags, sflags + n_users);
    m->have_names = true;
    return m->have_users ? multi_push_names(m) : NUTSB_OK;
}

NUTSB_API int nutsb_multi_set_ban_swearing(nutsb_multi *m, int on)
{ if (!m) return NUTSB_E_INVAL; MEACH(nutsb_set_ban_swearing(c_, on)); return NUTSB_OK; }

// The global population (index = position in the reference's user list).  room_weight: per room, the load it
// is expected to bring (NULL: its population).
NUTSB_API int nutsb_multi_set_users(nutsb_multi *m, int32_t n_users, int32_t n_rooms, const int32_t *room,
                                     const uint8_t *flags, const uint8_t *level, const uint64_t *room_weight)
{
    if (!m || n_users < 0 || n_rooms < 0 || (n_users && (!room || !flags || !level))) return mfail(m, NUTSB_E_INVAL, "nutsb_multi_set_users: bad argument");
    for (i32 u = 0; u < n_users; ++u) {
        if (room[u] >= n_rooms || room[u] < -1) return mfail(m, NUTSB_E_RANGE, "user room out of range");
        if (flags[u] & (NUTSB_UF_CLONE | NUTSB_UF_REMOTE))
            return mfail(m, NUTSB_E_UNSUPPORTED, "clones / remote users: their relays cross rooms (and shards); use one context");
    }
    const int S = m->n_shards;
    // queued ops name users by index (nutsb_set_users refuses them): checked on every shard before anything changes
    for (nutsb_ctx *c : m->ctx)
        if (c && (c->q.n() || !c->q_rec.empty()))
            return mfail(m, NUTSB_E_STATE, "nutsb_multi_set_users with ops still queued on a shard: flush first");
    // every room's review buffer as the old plan holds it (on a shard this process runs), to follow the room to its
    // new shard and local index; a room new to the population starts empty, as on one context
    if (m->have_users) {
        m->rev_carry.assign((size_t)m->R, nutsb_ctx::RevBuf{});
        for (i32 r = 0; r < m->R; ++r) {
            const nutsb_ctx *c = m->ctx[(size_t)m->room_shard[(size_t)r]];
            const size_t l = (size_t)m->room_local[(size_t)r];
            if (c && l < c->rev.size()) m->rev_carry[(size_t)r] = c->rev[l];
        }
        m->carry = true;
    }
    m->have_users = false; m->U = n_users; m->R = n_rooms;
    std::vector<u64> pop((size_t)n_rooms, 0);
    for (i32 u = 0; u < n_users; ++u) if (room[u] >= 0) pop[(size_t)room[u]]++;
    std::vector<u64> w((size_t)n_rooms);
    for (i32 r = 0; r < n_rooms; ++r) w[(size_t)r] = room_weight ? room_weight[r] : pop[(size_t)r];
    // heaviest room first, onto the least loaded shard (ties: lower index -- the plan is the same in every process)
    std::vector<i32> order((size_t)n_rooms); std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](i32 a, i32 b) { return w[(size_t)a] > w[(size_t)b]; });
    std::vector<u64> load((size_t)S, 0), heads((size_t)S, 0);
    m->room_shard.assign((size_t)n_rooms, 0); m->room_local.assign((size_t)n_rooms, 0);
    for (i32 r : order) {
        int best = 0;
        for (int s = 1; s < S; ++s) if (load[(size_t)s] < load[(size_t)best]) best = s;
        m->room_shard[(size_t)r] = best; load[(size_t)best] += w[(size_t)r] ? w[(size_t)r] : 1; heads[(size_t)best] += pop[(size_t)r];
    }
    m->shard_rooms.assign((size_t)S, 0);
    for (i32 r = 0; r < n_rooms; ++r) m->room_local[(size_t)r] = m->shard_rooms[(size_t)m->room_shard[(size_t)r]]++;   // local rooms keep the global order
    m->user_shard.assign((size_t)n_users, 0); m->user_local.assign((size_t)n_users, 0);
    m->shard_users.assign((size_t)S, std::vector<i32>());
    for (i32 u = 0; u < n_users; ++u) {
        int s;
        if (room[u] >= 0) s = m->room_shard[(size_t)room[u]];
        else { s = 0; for (int q = 1; q < S; ++q) if (heads[(size_t)q] < heads[(size_t)s]) s = q; heads[(size_t)s]++; }
        m->user_shard[(size_t)u] = s; m->user_local[(size_t)u] = (i32)m->shard_users[(size_t)s].size();
        m->shard_users[(size_t)s].push_back(u);
    }
    for (int s = 0; s < S; ++s) {
        nutsb_ctx *c = m->ctx[(size_t)s];
        if (!c) continue;
        const std::vector<i32> &us = m->shard_users[(size_t)s];
        std::vector<i32> lr(us.size()); std::vector<u8> lf(us.size()), ll(us.size());
        for (size_t i = 0; i < us.size(); ++i) {
            const i32 u = us[i];
            lr[i] = room[u] >= 0 ? m->room_local[(size_t)room[u]] : -1; lf[i] = flags[u]; ll[i] = level[u];
        }
        static const i32 zi = 0; static const u8 zb = 0;
        int rc = nutsb_set_users(c, (i32)us.size(), m->shard_rooms[(size_t)s], us.empty() ? &zi : lr.data(), us.empty() ? &zb : lf.data(), us.empty() ? &zb : ll.data());
        if (rc == NUTSB_OK) rc = shard_tables(c, s, m, room);
        if (rc != NUTSB_OK) { m->err = nutsb_last_error(c); return rc; }
    }
    for (i32 r = 0; r < n_rooms; ++r)
        if (nutsb_ctx *c = m->ctx[(size_t)m->room_shard[(size_t)r]])
            c->rev[(size_t)m->room_local[(size_t)r]] = m->carry && (size_t)r < m->rev_carry.size() ? m->rev_carry[(size_t)r] : nutsb_ctx::RevBuf{};
    m->rev_carry.clear(); m->carry = false;
    m->len.assign((size_t)n_users, 0); m->ptr.assign((size_t)n_users, nullptr);
    m->iov.assign((size_t)n_users, nullptr); m->count.assign((size_t)n_users, 0);
    m->have_users = true;
    if (m->have_names && (i32)m->sflags.size() == n_users) return multi_push_names(m);       // the plan moved users between shards
    return NUTSB_OK;
}

// where everything went: room_shard[n_rooms], user_shard[n_users], user_local[n_users] (any may be NULL)
NUTSB_API int nutsb_multi_plan(const nutsb_multi *m, int32_t *room_shard, int32_t *user_shard, int32_t *user_local)
{
    if (!m || !m->have_users) return NUTSB_E_STATE;
    if (room_shard) std::copy(m->room_shard.begin(), m->room_shard.end(), room_shard);
    if (user_shard) std::copy(m->user_shard.begin(), m->user_shard.end(), user_shard);
    if (user_local) std::copy(m->user_local.begin(), m->user_local.end(), user_local);
    return NUTSB_OK;
}

// The batch, routed: every shard's ops in the shard's local indices, call order kept.
static int multi_route(nutsb_multi *m, const nutsb_ops *o)
{
    if (!m->have_users) return mfail(m, NUTSB_E_STATE, "nutsb_multi_set_users has not been called");
    if (!o || o->n_ops < 0 || (o->n_ops && (!o->text_off || !o->kind || !o->target || !o->except_user || !o->flags)))
        return mfail(m, NUTSB_E_INVAL, "ops array is NULL");
    const int S = m->n_shards;
    const bool gated = o->gate && o->verdict;
    for (auto &r : m->routed) { r.ops.clear(); r.rc = NUTSB_OK; }
    auto push = [&](int s, i64 i, i32 target, i32 exc) {
        m->routed[(size_t)s].ops.push(o->kind[i], target, o->text + o->text_off[i], (size_t)(o->text_off[i + 1] - o->text_off[i]),
                                      exc, o->flags[i], gated ? o->gate[i] : -1);
    };
    for (i64 i = 0; i < o->n_ops; ++i) {
        const char *why = "";
        if (const int rc = host_op_error(o, i, m->U, m->R, &why)) return mfail(m, rc, why);
        if (o->text_off[i + 1] - o->text_off[i] > NUTSB_MAX_TEXT) return mfail(m, NUTSB_E_RANGE, "string longer than NUTSB_MAX_TEXT (2000) bytes");
        const u8 k = o->kind[i]; const i32 t = o->target[i], x = o->except_user[i];
        if (k == NUTSB_OP_NONE) continue;
        auto local_x = [&](int s) { return (x >= 0 && m->user_shard[(size_t)x] == s) ? m->user_local[(size_t)x] : -1; };
        if (k == NUTSB_OP_USER) {
            if (t < 0) continue;                                       // write_user(NULL, ...): c:1298
            push(m->user_shard[(size_t)t], i, m->user_local[(size_t)t], -1);
        } else if (k == NUTSB_OP_ROOM && t >= 0) {
            const int s = m->room_shard[(size_t)t];
            push(s, i, m->room_local[(size_t)t], local_x(s));
        } else {                                                       // all rooms (c:1399) / write_level: every shard
            for (int s = 0; s < S; ++s) push(s, i, t, local_x(s));
        }
    }
    return NUTSB_OK;
}

// The routed ops of one shard, as host arrays owned by the handle (valid until the next batch): for a caller that
// wants them resident in HBM before it times anything (bench.py), or that runs the shard itself.
NUTSB_API int nutsb_multi_route(nutsb_multi *m, const nutsb_ops *ops, int shard, nutsb_ops *out)
{
    if (!m || !out || shard < 0 || shard >= m->n_shards) return NUTSB_E_INVAL;
    TRY(multi_route(m, ops));
    *out = m->routed[(size_t)shard].ops.view(ops->gate && ops->verdict ? ops->verdict : nullptr);
    return NUTSB_OK;
}

// The result forms of a batch over the shards: streams on the host, streams kept in HBM, gather lists.
enum MForm { M_STREAMS, M_KEEP, M_IOV };

// One batch on every shard this process runs, one host thread each (job: the shard's call, its result into
// r.out / r.iov), then the merge into global user order -- pointer bookkeeping over the shards' own results, no
// byte copied.  If a shard fails: its code and message, and the output is left alone.
template <class Job>
static int multi_batch(nutsb_multi *m, MForm form, Job job, nutsb_mstreams *ms, nutsb_miov_streams *mi)
{
    const int S = m->n_shards;
    std::vector<std::thread> th;
    for (int s = 0; s < S; ++s) {
        if (!m->ctx[(size_t)s]) continue;
        th.emplace_back([m, s, &job] {
            nutsb_multi::Routed &r = m->routed[(size_t)s];
            r.rc = job(m->ctx[(size_t)s], r);
            if (r.rc == NUTSB_OK) nutsb_get_timing(m->ctx[(size_t)s], &r.tm);
        });
        NUTSB_MULTI_SERIAL(th);
    }
    for (auto &t : th) t.join();
    for (int s = 0; s < S; ++s)
        if (m->ctx[(size_t)s] && m->routed[(size_t)s].rc != NUTSB_OK) { m->err = nutsb_last_error(m->ctx[(size_t)s]); return m->routed[(size_t)s].rc; }
    u64 total = 0, deliv = 0;
    std::fill(m->len.begin(), m->len.end(), 0); std::fill(m->ptr.begin(), m->ptr.end(), nullptr);
    std::fill(m->iov.begin(), m->iov.end(), nullptr); std::fill(m->count.begin(), m->count.end(), 0);
    for (int s = 0; s < S; ++s) {
        if (!m->ctx[(size_t)s]) continue;
        const nutsb_multi::Routed &r = m->routed[(size_t)s];
        total += form == M_IOV ? r.iov.total_bytes : r.out.total_bytes;
        deliv += form == M_IOV ? r.iov.n_deliveries : r.out.n_deliveries;
        if (form == M_KEEP) continue;                                  // (the streams stay in HBM: nutsb_multi_stream_digests)
        const u64 *off = form == M_IOV ? r.iov.off : r.out.off;
        const std::vector<i32> &us = m->shard_users[(size_t)s];
        for (size_t i = 0; i < us.size(); ++i) {
            const size_t u = (size_t)us[i];
            m->len[u] = off[i + 1] - off[i];
            if (form == M_IOV) { m->iov[u] = r.iov.iov + r.iov.first[i]; m->count[u] = r.iov.count[i]; }
            else m->ptr[u] = r.out.bytes + off[i];
        }
    }
    if (form == M_IOV) {
        mi->n_users = m->U; mi->total_bytes = total; mi->n_deliveries = deliv;
        mi->len = m->len.data(); mi->iov = m->iov.data(); mi->count = m->count.data();
    } else {
        const bool keep = form == M_KEEP;
        ms->n_users = m->U; ms->total_bytes = total; ms->n_deliveries = deliv;
        ms->len = keep ? nullptr : m->len.data(); ms->ptr = keep ? nullptr : m->ptr.data(); ms->on_device = keep ? 1 : 0;
    }
    return NUTSB_OK;
}

// a routed write batch: every shard's share through the one-context call of the form
static int multi_write(nutsb_multi *m, const nutsb_ops *ops, MForm form, nutsb_mstreams *ms, nutsb_miov_streams *mi)
{
    TRY(multi_route(m, ops));
    const u8 *verdict = ops->gate && ops->verdict ? ops->verdict : nullptr;
    return multi_batch(m, form, [verdict, form](nutsb_ctx *c, nutsb_multi::Routed &r) {
        const nutsb_ops e = r.ops.view(verdict);
        return form == M_IOV ? nutsb_write_batch_iov(c, &e, &r.iov) : form == M_KEEP ? nutsb_write_batch_keep(c, &e, &r.out) : nutsb_write_batch(c, &e, &r.out);
    }, ms, mi);
}

/* keep != 0: the streams stay in HBM (ptr[] NULL); digests through nutsb_multi_stream_digests */
NUTSB_API int nutsb_multi_write_batch(nutsb_multi *m, const nutsb_ops *ops, nutsb_mstreams *out, int keep)
{
    if (!m || !out) return NUTSB_E_INVAL;
    return multi_write(m, ops, keep ? M_KEEP : M_STREAMS, out, nullptr);
}

NUTSB_API int nutsb_multi_write_batch_iov(nutsb_multi *m, const nutsb_ops *ops, nutsb_miov_streams *out)
{
    if (!m || !out) return NUTSB_E_INVAL;
    return multi_write(m, ops, M_IOV, nullptr, out);
}

// A speech batch: the whole batch to every shard, which composes the lines that produce an op on it (run_speech's
// shard mode); speakers are global user indices.
static int multi_speech(nutsb_multi *m, i64 n, const u8 *verb, const i32 *speaker, const u8 *bodies, const u64 *body_off,
                        MForm form, nutsb_mstreams *ms, nutsb_miov_streams *mi)
{
    if (!m->have_users) return mfail(m, NUTSB_E_STATE, "nutsb_multi_set_users has not been called");
    if (!m->have_names || (i32)m->sflags.size() != m->U) return mfail(m, NUTSB_E_STATE, "nutsb_multi_set_user_names does not match the population");
    TRY(multi_batch(m, form, [=](nutsb_ctx *c, nutsb_multi::Routed &r) {
        const Result res = form == M_IOV ? Result{ Result::IOV, nullptr, &r.iov } : Result{ form == M_KEEP ? Result::HBM : Result::HOST, &r.out, nullptr };
        return speech_batch(c, n, verb, speaker, bodies, body_off, true, res, true);
    }, ms, mi));
    for (nutsb_ctx *c : m->ctx) if (c && c->rec_ready) apply_records(c);      // every shard has succeeded: all or nothing
    return NUTSB_OK;
}

// Recording (nutsb_set_speech_record) on every shard: each records its own rooms.  Not in rank mode: a room's buffer
// could not follow it to a shard another process runs.
NUTSB_API int nutsb_multi_set_speech_record(nutsb_multi *m, int on)
{
    if (!m) return NUTSB_E_INVAL;
    if (on && m->rank) return mfail(m, NUTSB_E_UNSUPPORTED, "speech records in rank mode: a room's review buffer cannot follow it to another process");
    MEACH(nutsb_set_speech_record(c_, on));
    return NUTSB_OK;
}

// Global room `room`'s buffer (nutsb_get_review_buffer), from the shard that holds the room.
NUTSB_API int nutsb_multi_get_review_buffer(nutsb_multi *m, int32_t room, uint8_t *rows, int32_t *line)
{
    if (!m) return NUTSB_E_INVAL;
    if (!m->have_users) return mfail(m, NUTSB_E_STATE, "nutsb_multi_set_users has not been called");
    if (room < 0 || room >= m->R) return mfail(m, NUTSB_E_RANGE, "room index out of range");
    nutsb_ctx *c = m->ctx[(size_t)m->room_shard[(size_t)room]];
    if (!c) return mfail(m, NUTSB_E_UNSUPPORTED, "the room lives on a shard another process runs");
    const int rc = nutsb_get_review_buffer(c, m->room_local[(size_t)room], rows, line);
    if (rc != NUTSB_OK) m->err = nutsb_last_error(c);
    return rc;
}

NUTSB_API int nutsb_multi_speech_batch(nutsb_multi *m, int64_t n, const uint8_t *verb, const int32_t *speaker,
                                       const uint8_t *bodies, const uint64_t *body_off, nutsb_mstreams *out, int keep)
{
    if (!m || !out) return NUTSB_E_INVAL;
    return multi_speech(m, n, verb, speaker, bodies, body_off, keep ? M_KEEP : M_STREAMS, out, nullptr);
}

NUTSB_API int nutsb_multi_speech_batch_iov(nutsb_multi *m, int64_t n, const uint8_t *verb, const int32_t *speaker,
                                           const uint8_t *bodies, const uint64_t *body_off, nutsb_miov_streams *out)
{
    if (!m || !out) return NUTSB_E_INVAL;
    return multi_speech(m, n, verb, speaker, bodies, body_off, M_IOV, nullptr, out);
}

// One shard's own result of the last gather-list batch (local user order): the pools the merged pieces point into.
NUTSB_API int nutsb_multi_shard_iov(const nutsb_multi *m, int shard, nutsb_iov_streams *out)
{
    if (!m || !out || shard < 0 || shard >= m->n_shards || !m->ctx[(size_t)shard]) return NUTSB_E_INVAL;
    *out = m->routed[(size_t)shard].iov;
    return NUTSB_OK;
}

// digest[n_users] in global order (nutsb_stream_digests per shard); cont != 0: the fold goes on from the values
// in digest[] (a job that runs in message-ordered chunks).  Users of shards this process does not run are left alone.
NUTSB_API int nutsb_multi_stream_digests(nutsb_multi *m, uint64_t *digest, int cont)
{
    if (!m || !digest || !m->have_users) return NUTSB_E_INVAL;
    std::vector<int> rc((size_t)m->n_shards, NUTSB_OK);
    std::vector<std::vector<u64>> loc((size_t)m->n_shards);
    std::vector<std::thread> th;
    for (int s = 0; s < m->n_shards; ++s) {
        if (!m->ctx[(size_t)s]) continue;
        const std::vector<i32> &us = m->shard_users[(size_t)s];
        loc[(size_t)s].resize(us.size() + 1);
        for (size_t i = 0; i < us.size(); ++i) loc[(size_t)s][i] = digest[us[i]];
        th.emplace_back([m, s, cont, &rc, &loc] {
            rc[(size_t)s] = cont ? nutsb_stream_digests_continue(m->ctx[(size_t)s], loc[(size_t)s].data()) : nutsb_stream_digests(m->ctx[(size_t)s], loc[(size_t)s].data());
        });
        NUTSB_MULTI_SERIAL(th);
    }
    for (auto &t : th) t.join();
    for (int s = 0; s < m->n_shards; ++s) {
        if (!m->ctx[(size_t)s]) continue;
        if (rc[(size_t)s] != NUTSB_OK) { m->err = nutsb_last_error(m->ctx[(size_t)s]); return rc[(size_t)s]; }
        const std::vector<i32> &us = m->shard_users[(size_t)s];
        for (size_t i = 0; i < us.size(); ++i) digest[us[i]] = loc[(size_t)s][i];
    }
    return NUTSB_OK;
}

// Verdict batches: the strings are split by index range over the shards this process runs (SURVEY.md 8e).
static int multi_verdict(nutsb_multi *m, int which, i64 n, const u8 *bytes, const u64 *off, u8 *verdict)
{
    if (!m || n < 0 || (n && (!off || !verdict))) return NUTSB_E_INVAL;
    std::vector<int> live;
    for (int s = 0; s < m->n_shards; ++s) if (m->ctx[(size_t)s]) live.push_back(s);
    if (live.empty() || n == 0) return NUTSB_OK;
    const i64 per = (n + (i64)live.size() - 1) / (i64)live.size();
    std::vector<int> rc(live.size(), NUTSB_OK);
    std::vector<std::thread> th;
    for (size_t k = 0; k < live.size(); ++k) {
        const i64 a = std::min<i64>(n, (i64)k * per), b = std::min<i64>(n, a + per);
        if (b <= a) continue;
        th.emplace_back([=, &rc] {
            nutsb_ctx *c = m->ctx[(size_t)live[k]];
            rc[k] = which == V_SWEAR ? nutsb_contains_swearing_batch(c, b - a, bytes, off + a, verdict + a)
                  : which == V_SITE  ? nutsb_site_banned_batch(c, b - a, bytes, off + a, verdict + a)
                                     : nutsb_user_banned_batch(c, b - a, bytes, off + a, verdict + a);
        });
        NUTSB_MULTI_SERIAL(th);
    }
    for (auto &t : th) t.join();
    for (size_t k = 0; k < live.size(); ++k) if (rc[k] != NUTSB_OK) { m->err = nutsb_last_error(m->ctx[(size_t)live[k]]); return rc[k]; }
    return NUTSB_OK;
}
NUTSB_API int nutsb_multi_contains_swearing_batch(nutsb_multi *m, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return multi_verdict(m, V_SWEAR, n, b, o, v); }
NUTSB_API int nutsb_multi_site_banned_batch(nutsb_multi *m, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return multi_verdict(m, V_SITE, n, b, o, v); }
NUTSB_API int nutsb_multi_user_banned_batch(nutsb_multi *m, int64_t n, const uint8_t *b, const uint64_t *o, uint8_t *v) { return multi_verdict(m, V_USER, n, b, o, v); }

// the last batch's device timings of one shard (nutsb_set_profiling / nutsb_multi_set_profiling)
NUTSB_API int nutsb_multi_get_timing(const nutsb_multi *m, int shard, nutsb_timing *out)
{
    if (!m || !out || shard < 0 || shard >= m->n_shards || !m->ctx[(size_t)shard]) return NUTSB_E_INVAL;
    *out = m->routed[(size_t)shard].tm;
    return NUTSB_OK;
}

// ---- calls in flight: nutsb_pipe ------------------------------------------------------------------
// A host-buffer call is H2D copy -> kernels -> D2H copy, and PCIe is full duplex: with two calls in flight one
// call's H2D and kernels run under the other's D2H (profiles/r01_pcie_probe.json: 57 GB/s either way, 99 GB/s both
// ways at once).  nutsb_pipe keeps `depth` contexts on one device, each with its own worker thread; submit hands a
// call to the next context and returns at once, wait returns its result.  Results are valid until `depth` further
// submissions; a call's input buffers must stay valid until it has been waited for.  Tables and population are
// set once for all contexts (nutsb_pipe_ctx(p, i) gives each of them for anything else).
#include <condition_variable>
#include <functional>
#include <mutex>

struct nutsb_pipe {
    struct Lane {
        nutsb_ctx *ctx = nullptr;
        std::thread th; std::mutex m; std::condition_variable cv;
        std::function<int()> job; bool has_job = false, done = true, quit = false; int rc = NUTSB_OK;
        nutsb_iov_streams out{};
    };
    int depth = 0;
    std::vector<Lane *> lanes;
    uint64_t next = 0;
};

static void pipe_worker(nutsb_pipe::Lane *L)
{
    for (;;) {
        std::function<int()> job;
        {
            std::unique_lock<std::mutex> lk(L->m);
            L->cv.wait(lk, [L] { return L->has_job || L->quit; });
            if (L->quit) return;
            job = L->job; L->has_job = false;
        }
        const int rc = job();
        { std::lock_guard<std::mutex> lk(L->m); L->rc = rc; L->done = true; }
        L->cv.notify_all();
    }
}

NUTSB_API void nutsb_pipe_destroy(nutsb_pipe *p)
{
    if (!p) return;
    for (nutsb_pipe::Lane *L : p->lanes) {
        if (L->th.joinable()) {
            { std::unique_lock<std::mutex> lk(L->m); L->cv.wait(lk, [L] { return L->done; }); L->quit = true; }
            L->cv.notify_all();
            L->th.join();
        }
        if (L->ctx) nutsb_destroy(L->ctx);
        delete L;
    }
    delete p;
}

NUTSB_API int nutsb_pipe_create(nutsb_pipe **out, int device, int depth)
{
    if (!out || depth < 1 || depth > 8) return NUTSB_E_INVAL;
    *out = nullptr;
    nutsb_pipe *p = new (std::nothrow) nutsb_pipe;
    if (!p) return NUTSB_E_NOMEM;
    p->depth = depth;
    for (int i = 0; i < depth; ++i) {
        nutsb_pipe::Lane *L = new (std::nothrow) nutsb_pipe::Lane;
        if (!L) { nutsb_pipe_destroy(p); return NUTSB_E_NOMEM; }
        p->lanes.push_back(L);
        const int rc = nutsb_create(&L->ctx, device);
        if (rc != NUTSB_OK) { nutsb_pipe_destroy(p); return rc; }
#ifndef NUTSB_CPUSIM
        L->th = std::thread(pipe_worker, L);
#endif
    }
    *out = p;
    return NUTSB_OK;
}
NUTSB_API int nutsb_pipe_depth(const nutsb_pipe *p) { return p ? p->depth : 0; }
NUTSB_API nutsb_ctx *nutsb_pipe_ctx(nutsb_pipe *p, int lane) { return (p && lane >= 0 && lane < p->depth) ? p->lanes[(size_t)lane]->ctx : nullptr; }

#define PEACH(call) do { for (nutsb_pipe::Lane *L_ : p->lanes) { nutsb_ctx *c_ = L_->ctx; const int rc_ = (call); if (rc_ != NUTSB_OK) return rc_; } } while (0)
NUTSB_API int nutsb_pipe_set_swear_words(nutsb_pipe *p, const char *const *words) { if (!p) return NUTSB_E_INVAL; PEACH(nutsb_set_swear_words(c_, words)); return NUTSB_OK; }
NUTSB_API int nutsb_pipe_set_users(nutsb_pipe *p, int32_t n_users, int32_t n_rooms, const int32_t *room, const uint8_t *flags, const uint8_t *level)
{ if (!p) return NUTSB_E_INVAL; PEACH(nutsb_set_users(c_, n_users, n_rooms, room, flags, level)); return NUTSB_OK; }
NUTSB_API int nutsb_pipe_set_user_names(nutsb_pipe *p, int32_t n_users, const uint8_t *names, const uint64_t *off, const uint8_t *sflags)
{ if (!p) return NUTSB_E_INVAL; PEACH(nutsb_set_user_names(c_, n_users, names, off, sflags)); return NUTSB_OK; }
NUTSB_API int nutsb_pipe_set_ban_swearing(nutsb_pipe *p, int on) { if (!p) return NUTSB_E_INVAL; PEACH(nutsb_set_ban_swearing(c_, on)); return NUTSB_OK; }

static int pipe_submit(nutsb_pipe *p, std::function<int(nutsb_pipe::Lane *)> fn, uint64_t *ticket)
{
    if (!p || !ticket) return NUTSB_E_INVAL;
    nutsb_pipe::Lane *L = p->lanes[(size_t)(p->next % (uint64_t)p->depth)];
    *ticket = p->next++;
#ifdef NUTSB_CPUSIM                     // the emulator's launch state is process-global: the call runs here and now
    L->rc = fn(L); L->done = true;
#else
    {
        std::unique_lock<std::mutex> lk(L->m);
        L->cv.wait(lk, [L] { return L->done; });             // the lane's previous call (its result is given up by now)
        L->job = [fn, L] { return fn(L); }; L->has_job = true; L->done = false;
    }
    L->cv.notify_all();
#endif
    return NUTSB_OK;
}

// nutsb_speech_batch_iov / nutsb_write_batch_iov, in flight
NUTSB_API int nutsb_pipe_submit_speech_iov(nutsb_pipe *p, int64_t n, const uint8_t *verb, const int32_t *speaker,
                                           const uint8_t *bodies, const uint64_t *body_off, uint64_t *ticket)
{
    return pipe_submit(p, [=](nutsb_pipe::Lane *L) { return nutsb_speech_batch_iov(L->ctx, n, verb, speaker, bodies, body_off, &L->out); }, ticket);
}
NUTSB_API int nutsb_pipe_submit_write_iov(nutsb_pipe *p, const nutsb_ops *ops, uint64_t *ticket)
{
    if (!ops) return NUTSB_E_INVAL;
    const nutsb_ops o = *ops;
    return pipe_submit(p, [o](nutsb_pipe::Lane *L) { return nutsb_write_batch_iov(L->ctx, &o, &L->out); }, ticket);
}
// the result of call `ticket` (one of the last `depth` submitted); its return code is the call's own
NUTSB_API int nutsb_pipe_wait(nutsb_pipe *p, uint64_t ticket, nutsb_iov_streams *out)
{
    if (!p || !out || ticket >= p->next || ticket + (uint64_t)p->depth < p->next) return NUTSB_E_INVAL;
    nutsb_pipe::Lane *L = p->lanes[(size_t)(ticket % (uint64_t)p->depth)];
    {
        std::unique_lock<std::mutex> lk(L->m);
        L->cv.wait(lk, [L] { return L->done; });
    }
    *out = L->out;
    return L->rc;
}
