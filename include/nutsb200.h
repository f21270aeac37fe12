/* nutsb200.h -- C-ABI of the B200-native NUTS 3.3.3 message path.
 *
 * The reference (ToKe79/nuts333) has no plugin/FFI layer: the path is reached by
 * direct C calls inside one translation unit.  The boundary a replacement must
 * honour is the function surface the reference declares in nuts333.h:
 *
 *     void write_user(UR_OBJECT user, char *str);                        nuts333.c:1291
 *     void write_room(RM_OBJECT rm, char *str);                          nuts333.c:1390
 *     void write_room_except(RM_OBJECT rm, char *str, UR_OBJECT user);   nuts333.c:1401
 *     void write_level(int level, int above, char *str, UR_OBJECT user); nuts333.c:1372
 *     int  contains_swearing(char *str);                                 nuts333.c:2540
 *     int  site_banned(char *site);                                      nuts333.c:330
 *     int  user_banned(char *name);                                      nuts333.c:349
 *     void write_sock(int sock, char *str);                              nuts333.c:1281
 *
 * shim/nuts333_shim.c holds bodies with exactly these names over this header (the
 * drop-in; tests/dropin/ links them over the unmodified nuts333.c).
 *
 * This header exposes that surface in three tiers, all `extern "C"`, plain
 * pointers and sizes only:
 *
 *   1. queue tier  (nutsb_q_*, nutsb_flush): one call per reference call, user /
 *      room passed as their index in the reference's lists.  str is copied on
 *      enqueue (callers overwrite the global text[] right after, c:4094-4098).
 *      shim/nuts333_shim.c holds the eight bodies that bind nuts333.c to it.
 *   2. batch tier, host buffers (nutsb_write_batch, nutsb_*_batch): SoA batches
 *      in host memory, results in library-owned pinned host memory.
 *   3. batch tier, device buffers (*_dev): the same on buffers already in HBM.
 * and, over the batch tier, nutsb_multi (one population and one batch over several
 * GPUs, sharded by room, no collective) and nutsb_pipe (calls in flight on one GPU).
 *
 * Semantics are bit-exact with nuts333.c for USER_TYPE recipients, for clones (the
 * relay of c:1416-1426) and for remote users (the MSG/EMSG framing of c:1299-1307):
 * both are made on the host by the queue tier and by the host-buffer batch calls
 * (nutsb_set_clones, nutsb_set_remotes); the device-buffer calls refuse such a
 * population (NUTSB_E_UNSUPPORTED).
 *
 * Errors: every entry point returns 0 or a negative NUTSB_E_* code and never
 * aborts the host; on error outputs are left untouched.  One context per host
 * thread, one context per GPU; not async-signal-safe (the reference enters its
 * write layer from SIGALRM, c:7721 -- a binding must defer those to the main
 * loop).  There is NO CPU fallback: without a CUDA device nutsb_create fails.
 */
#ifndef NUTSB200_H
#define NUTSB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NUTSB_VERSION 0x000100

enum {
    NUTSB_OK            =  0,
    NUTSB_E_INVAL       = -1,  /* bad argument (NULL, negative count, offsets not monotone) */
    NUTSB_E_NOMEM       = -2,  /* host or device allocation failed                          */
    NUTSB_E_CUDA        = -3,  /* CUDA runtime error, see nutsb_last_error()                */
    NUTSB_E_UNSUPPORTED = -4,  /* device-buffer batch over a population with clones / remote users */
    NUTSB_E_RANGE       = -5,  /* string longer than NUTSB_MAX_TEXT, index out of range     */
    NUTSB_E_STATE       = -6   /* call order (e.g. write batch before nutsb_set_users)      */
};

/* text[ARR_SIZE*2] is the largest string the reference can pass (nuts333.h:280). */
#define NUTSB_MAX_TEXT 2000
/* line[82] in site_banned/user_banned (c:334,353): longer tokens overflow there. */
#define NUTSB_MAX_BAN_TOKEN 81
#define NUTSB_REVIEW_LINES 15    /* nuts333.h:37 */
#define NUTSB_REVIEW_LEN   200   /* nuts333.h:39 */
#define NUTSB_REVTELL_LINES 5    /* nuts333.h:38 */

/* recipient flags (nuts333.h:67-85 fields actually read on the path) */
#define NUTSB_UF_COLOUR   0x01u  /* user->colour != 0            */
#define NUTSB_UF_LOGIN    0x02u  /* user->login  != 0            */
#define NUTSB_UF_IGNALL   0x04u  /* user->ignall                 */
#define NUTSB_UF_IGNSHOUT 0x08u  /* user->ignshout               */
#define NUTSB_UF_CLONE    0x10u  /* type==CLONE_TYPE: receives nothing itself; nutsb_set_clones */
#define NUTSB_UF_REMOTE   0x20u  /* type==REMOTE_TYPE: reached through its netlink; nutsb_set_remotes */

/* op kinds: one op == one call of the reference's write surface */
#define NUTSB_OP_USER  0  /* write_user(target, str)                                   */
#define NUTSB_OP_ROOM  1  /* write_room_except(target, str, except); target -1 = NULL  */
#define NUTSB_OP_LEVEL 2  /* write_level(target, above, str, except)                   */
#define NUTSB_OP_NONE  3  /* no call: a branch of a caller that was not taken           */

/* op flags: the globals the reference reads inside the call */
#define NUTSB_OF_FORCE_LISTEN 0x01u  /* force_listen (nuts333.h:293, c:1413)           */
#define NUTSB_OF_SHOUT        0x02u  /* com_num==SHOUT || com_num==SEMOTE (c:1414)     */
#define NUTSB_OF_ABOVE        0x04u  /* write_level's `above`                          */
#define NUTSB_OF_GATE_IF_SET  0x08u  /* with gate>=0: live iff verdict[gate]!=0,
                                        else live iff verdict[gate]==0 (say(), c:4091) */
#define NUTSB_OF_PAGER        0x10u  /* render as the pager more() renders a file line
                                        (nuts333.c:2254-2300): the same byte machine, but
                                        no terminal reset after the string (c:1365 absent) */
#define NUTSB_OF_RAW          0x40u  /* the bytes as they are, no byte machine: what write_user hands to
                                        write_sock for a remote user (nuts333.c:1303-1305)             */
#define NUTSB_OF_PLAIN        0x20u  /* the recipient's colour setting is ignored and taken
                                        as off: more(NULL,sock,file) at login (c:2259,2279) */

typedef struct nutsb_ctx nutsb_ctx;

/* A batch of write calls, in call order.  All arrays have n_ops entries except
 * text_off (n_ops+1, monotone, text_off[0] may be non-zero).  Strings need no
 * NUL terminator and must not contain NUL.  gate/verdict may be NULL. */
typedef struct nutsb_ops {
    int64_t         n_ops;
    const uint8_t  *text;
    const uint64_t *text_off;
    const uint8_t  *kind;         /* NUTSB_OP_*                                         */
    const int32_t  *target;       /* user index | room index (-1 all rooms) | level     */
    const int32_t  *except_user;  /* -1 = none                                          */
    const uint8_t  *flags;        /* NUTSB_OF_*                                         */
    const int32_t  *gate;         /* index into verdict, -1 = unconditional; or NULL    */
    const uint8_t  *verdict;      /* swear verdicts the gates refer to; or NULL         */
} nutsb_ops;

/* Per-user socket streams: user u receives bytes[off[u] .. off[u+1]) -- exactly
 * what the reference would have written to user u's socket over the batch, in
 * call order.  Pointers are owned by the context and stay valid until the next
 * write batch / flush / destroy on it. */
typedef struct nutsb_streams {
    int64_t         n_users;
    uint64_t        total_bytes;
    uint64_t        n_deliveries;   /* (op, recipient) pairs rendered                    */
    const uint64_t *off;            /* n_users + 1                                       */
    const uint8_t  *bytes;
    int32_t         on_device;      /* 1: off/bytes are device pointers                  */
} nutsb_streams;

/* Device-side timings of the last write batch, CUDA events on the context's
 * stream (ms).  Filled only after nutsb_set_profiling(ctx, 1). */
typedef struct nutsb_timing {
    float plan_ms;       /* measure, bucket, prefix, events, offsets, copy plan         */
    float render_ms;     /* k_render: every room/level op rendered once per colour      */
    float fanout_ms;     /* k_fanout: rendered bytes -> recipients' streams (dominant)  */
    float direct_ms;     /* write_user ops rendered straight into the streams           */
    float total_ms;      /* first kernel to last kernel, incl. the two size read-backs  */
    float h2d_ms, d2h_ms;
    uint64_t fanout_bytes_in, fanout_bytes_out;   /* algorithmic bytes of the fan-out kernel:
                                                     rendered slab read once, deliveries written once */
    uint64_t render_bytes_in, slab_bytes;         /* k_render: source bytes read, rendered bytes written */
    uint32_t launches;   /* kernels launched by the last batch call                     */
    uint32_t fanout_launches;
} nutsb_timing;

int         nutsb_version(void);
const char *nutsb_strerror(int code);
const char *nutsb_last_error(const nutsb_ctx *ctx);

int  nutsb_create(nutsb_ctx **out, int device);
void nutsb_destroy(nutsb_ctx *ctx);
int  nutsb_set_profiling(nutsb_ctx *ctx, int on);
int  nutsb_get_timing(const nutsb_ctx *ctx, nutsb_timing *out);
/* 1 (default): k_render and k_direct run on a second stream beside the planning kernels and the
 * fan-out.  0: every kernel on one stream, so that each kernel's own duration can be timed alone. */
int  nutsb_set_overlap(nutsb_ctx *ctx, int on);
/* Use the caller's CUDA stream (a cudaStream_t) instead of the context's own.  The context's own stream has the
 * device's highest priority and its side stream (the renderer, beside the planning kernels) the lowest; a caller's
 * stream created above the lowest priority keeps that order (cudaStreamCreateWithPriority). */
int  nutsb_set_stream(nutsb_ctx *ctx, void *cuda_stream);

/* Clones (nuts333.c:1416-1426): owner[u] = index of the owner of clone u, -1 for everybody else (clones are the
 * users flagged NUTSB_UF_CLONE); hear[u] = clone_hear (0 nothing, 1 swears, 2 all).  Call after
 * nutsb_set_users.  The queue tier then makes the relays: a room op naming a clone's room also queues
 * write_user(owner, "~FT[ <room> ]:~RS <str>") at the clone's place in the user list, unless the clone is
 * filtered like any recipient, hears nothing, its owner ignores everything, or (hear 1) the string does not
 * swear.  The host-buffer batch calls make them too; the device-buffer ones refuse the population (see
 * nutsb_write_batch).  Room names: rm->name, default "room<index>". */
int nutsb_set_clones(nutsb_ctx *ctx, int32_t n_users, const int32_t *owner, const uint8_t *hear);
/* Remote users (nuts333.c:1299-1307): link[u] = index of the pseudo-user whose stream stands for the netlink
 * socket remote user u is reached through (a user in no room, flagged neither clone nor remote; several
 * remote users may share one), -1 for everybody else; old_peer[u] != 0: the peer is older than 3.2 and gets
 * its colour commands stripped (colour_com_strip, c:2588).  Call after nutsb_set_users and
 * nutsb_set_user_names.  The queue tier then frames what write_user would hand to write_sock:
 * "MSG <name>\n<str>[\n]EMSG\n", unrendered (NUTSB_OF_RAW), into the link's stream, for write_user to a remote
 * user and for every remote recipient of a room / level op, in user-list order. */
int nutsb_set_remotes(nutsb_ctx *ctx, int32_t n_users, const int32_t *link, const uint8_t *old_peer);
int nutsb_set_room_names(nutsb_ctx *ctx, int32_t n_rooms, const uint8_t *names, const uint64_t *off);

/* ---- tables ------------------------------------------------------------- */

/* swear_words[] (nuts333.h:275-277): list ends at the first entry starting
 * with '*' or at a NULL pointer.  Default = the stock list. */
int nutsb_set_swear_words(nutsb_ctx *ctx, const char *const *words);

/* Raw FILE BYTES of datafiles/siteban and datafiles/userban; the library
 * applies the fscanf("%s")/feof tokenizer of c:338-342 (a last token not
 * followed by whitespace is never tested).  NULL = file missing (verdict 0). */
int nutsb_set_ban_files(nutsb_ctx *ctx, const void *siteban, size_t siteban_len,
                        const void *userban, size_t userban_len);
/* Ban-list maintenance (nuts333.c:6216-6429) on the lists held by the context: which 0 = siteban,
 * 1 = userban (first byte upper-cased, c:6269); add 1 = ban_site / ban_user: append "token\n" unless a
 * TESTED token equals it (strcmp); add 0 = unban_*: the list rewritten without it, every tested token as
 * "token\n" -- a last token that ran into EOF is dropped (the reference's feof() loop), an emptied list is
 * removed.  The matchers in HBM follow at once.  *result: 0 done, 1 nothing to do ("already banned" /
 * "not currently banned").  The command's own checks (own host, levels, user files) are the talker's.
 * nutsb_get_ban_file: the list as it stands, to be written back to datafiles/ (*present 0: no file). */
int nutsb_ban_edit(nutsb_ctx *ctx, int which, int add, const char *token, int *result);
int nutsb_get_ban_file(nutsb_ctx *ctx, int which, const void **bytes, size_t *len, int *present);

/* Population, index = position in the reference's user list (creation order,
 * c:2683-2691).  room[u] in [0,n_rooms) or -1 (user->room==NULL). */
int nutsb_set_users(nutsb_ctx *ctx, int32_t n_users, int32_t n_rooms, const int32_t *room,
                    const uint8_t *flags, const uint8_t *level);
/* The same when users joined or left (the list positions shift): prev_index[u] = the index user u had in
 * the population before, -1 for a new user (create_user() starts with empty buffers, c:2747); NULL = nobody
 * moved.  Queued ops name users by index, so both calls return NUTSB_E_STATE while anything is queued
 * (nutsb_q_pending() > 0): flush first, then bring the new population in.  The review buffers of the rooms and
 * the revtell buffers of the users live on across the call (the reference clears them only in create_room,
 * create_user and clear_revbuff). */
int nutsb_set_users_remap(nutsb_ctx *ctx, int32_t n_users, int32_t n_rooms, const int32_t *room,
                          const uint8_t *flags, const uint8_t *level, const int32_t *prev_index);

/* ---- batch tier --------------------------------------------------------- */

/* write_user / write_room[_except] / write_level, batched.  Host variant:
 * ops in host memory, streams returned in pinned host memory.  With clones or remote users in the
 * population (NUTSB_UF_CLONE / NUTSB_UF_REMOTE) the host-buffer calls (nutsb_write_batch, nutsb_write_batch_iov)
 * expand every op on the host exactly as the queue tier does -- the relays of nuts333.c:1416-1426 and the
 * MSG/EMSG frames of c:1299-1307, each under the op's own gate -- before the batch runs (needs an empty queue,
 * nutsb_set_clones / nutsb_set_remotes); the device-buffer calls (*_dev, nutsb_write_batch_keep,
 * nutsb_speech_batch*) take ops as they are and return NUTSB_E_UNSUPPORTED for such a population rather than
 * deliver different bytes. */
int nutsb_write_batch(nutsb_ctx *ctx, const nutsb_ops *ops, nutsb_streams *out);
/* Device variant: every pointer in ops is a device pointer; streams stay in HBM.  The packed text is read
 * in aligned 16-byte vectors: it must be readable from the 16-byte boundary at or before its first byte to the
 * one at or after its last (true of any buffer that starts a cudaMalloc allocation, whatever its length). */
int nutsb_write_batch_dev(nutsb_ctx *ctx, const nutsb_ops *ops, nutsb_streams *out);

/* The same streams as gather lists, for a host that hands them to writev(2).  The reference writes the
 * same rendered bytes to every listener of a room (write_room_except's loop, c:1409-1428, calls write_user
 * per recipient); here they cross PCIe once per colour setting instead of once per recipient.  User u's
 * stream is the concatenation of iov[first[u]] .. iov[first[u] + count[u] - 1] (zero-length pieces
 * occur); every piece points into `pool` or `pool2`, pinned host memory owned by the context:
 *     writev(user->socket, (const struct iovec *)(s.iov + s.first[u]), s.count[u]);   (in chunks of IOV_MAX)
 * nutsb_iovec has the layout of struct iovec on LP64.  Concatenated, the pieces are byte for byte the
 * stream nutsb_write_batch returns for u (off[] is the same array).  pool = every room / level op
 * rendered once per colour setting (copied to the host while the device is still planning), pool2 = every
 * write_user op rendered once for its recipient.  With
 * recipients behind a filter (login / ignall / ignshout users, write_level ops in the batch) the pool is
 * the full streams and every user has one piece: same result, no saving.  Valid until the next write
 * batch / flush / destroy on the context. */
typedef struct nutsb_iovec { const void *base; size_t len; } nutsb_iovec;
typedef struct nutsb_iov_streams {
    int64_t            n_users;
    uint64_t           total_bytes;    /* sum of all streams                                 */
    uint64_t           n_deliveries;
    const uint64_t    *off;            /* n_users + 1: off[u+1] - off[u] = length of u's stream */
    const uint64_t    *first;          /* n_users                                            */
    const uint32_t    *count;          /* n_users                                            */
    const nutsb_iovec *iov;
    uint64_t           n_iov;
    const uint8_t     *pool;           /* room / level ops, once per colour setting (or the full streams) */
    uint64_t           pool_bytes;
    const uint8_t     *pool2;          /* write_user ops, once each (NULL when the pool is the streams)    */
    uint64_t           pool2_bytes;
} nutsb_iov_streams;
int nutsb_write_batch_iov(nutsb_ctx *ctx, const nutsb_ops *ops, nutsb_iov_streams *out);

/* contains_swearing / site_banned / user_banned over n packed strings
 * (bytes + off[n+1]); verdict[n] gets 0/1.  *_dev: device pointers. */
int nutsb_contains_swearing_batch(nutsb_ctx *ctx, int64_t n, const uint8_t *bytes,
                                  const uint64_t *off, uint8_t *verdict);
int nutsb_contains_swearing_batch_dev(nutsb_ctx *ctx, int64_t n, const uint8_t *bytes,
                                      const uint64_t *off, uint8_t *verdict);
int nutsb_site_banned_batch(nutsb_ctx *ctx, int64_t n, const uint8_t *bytes,
                            const uint64_t *off, uint8_t *verdict);
int nutsb_site_banned_batch_dev(nutsb_ctx *ctx, int64_t n, const uint8_t *bytes,
                                const uint64_t *off, uint8_t *verdict);
int nutsb_user_banned_batch(nutsb_ctx *ctx, int64_t n, const uint8_t *bytes,
                            const uint64_t *off, uint8_t *verdict);
int nutsb_user_banned_batch_dev(nutsb_ctx *ctx, int64_t n, const uint8_t *bytes,
                                const uint64_t *off, uint8_t *verdict);

/* ---- the callers' composition: say / shout / emote / semote / echo / bcast ------------- */
/* What one input line becomes (nuts333.c:4062-4126, 4188-4232, 4289-4305, 4772-4788):
 * up to three write calls per line -- the refusal ("You are muzzled ...", or noswearing when
 * ban_swearing is on and the body swears), the speaker's own copy, the line to the room(s).
 * The caller-level checks (word_count, command_mode) stay with the caller. */
#define NUTSB_SPEECH_SAY    0   /* say(user,inpstr)     c:4062 */
#define NUTSB_SPEECH_SHOUT  1   /* shout(user,inpstr)   c:4105 */
#define NUTSB_SPEECH_EMOTE  2   /* emote(user,inpstr)   c:4188 */
#define NUTSB_SPEECH_SEMOTE 3   /* semote(user,inpstr)  c:4213 */
#define NUTSB_SPEECH_ECHO   4   /* echo(user,inpstr)    c:4289 */
#define NUTSB_SPEECH_BCAST  5   /* bcast(user,inpstr)   c:4772 */
#define NUTSB_SF_INVIS   0x01u  /* user->vis == 0: others see invisname (nuts333.h:150) */
#define NUTSB_SF_MUZZLED 0x02u  /* user->muzzled                                        */

/* user->name, user->vis, user->muzzled of every user (names packed, off[n_users+1]). */
int nutsb_set_user_names(nutsb_ctx *ctx, int32_t n_users, const uint8_t *names, const uint64_t *off,
                         const uint8_t *speech_flags);
/* the global ban_swearing (nuts333.h:296, config option c:803-808); default off as in init_globals */
int nutsb_set_ban_swearing(nutsb_ctx *ctx, int on);
/* n input lines: verb[n], speaker[n] (user index), bodies packed + off[n+1].  The device
 * runs contains_swearing on the bodies, composes the calls and renders them; streams as
 * for nutsb_write_batch.  *_dev: every pointer is a device pointer, streams stay in HBM.
 * With nutsb_set_speech_record(ctx, 1) the three calls also record what say / emote / echo send to the
 * room in its review buffer, as nutsb_q_speech does (see nutsb_set_speech_record); nutsb_speech_batch_dev
 * then synchronises once more and returns with the records applied.  nutsb_timing of a speech batch describes its
 * write pipeline: the composition and the recording step before it are in neither launches nor total_ms. */
int nutsb_speech_batch(nutsb_ctx *ctx, int64_t n, const uint8_t *verb, const int32_t *speaker,
                       const uint8_t *bodies, const uint64_t *body_off, nutsb_streams *out);
int nutsb_speech_batch_dev(nutsb_ctx *ctx, int64_t n, const uint8_t *verb, const int32_t *speaker,
                           const uint8_t *bodies, const uint64_t *body_off, nutsb_streams *out);
/* Host buffers in, gather lists out (see nutsb_write_batch_iov). */
int nutsb_speech_batch_iov(nutsb_ctx *ctx, int64_t n, const uint8_t *verb, const int32_t *speaker,
                           const uint8_t *bodies, const uint64_t *body_off, nutsb_iov_streams *out);
/* queue tier: one call of the reference's say()/shout()/... ; composed on the host, the swear
 * verdicts of the queued lines are taken in one device batch at nutsb_flush */
int nutsb_q_speech(nutsb_ctx *ctx, int verb, int32_t user, const char *inpstr);
/* 1: nutsb_speech_batch / _iov / _dev record what say / emote / echo send to the room, as nutsb_q_speech does.
 * 0 (default): they leave the review buffers alone, as before.
 * A line is recorded when its room line is sent: the speaker is in a room and not muzzled, and the line is not
 * refused for swearing.  The record is the composed line as record() (c:2062) keeps it.  The records go in batch
 * order after what the buffers held; the buffers change only when the whole call succeeds.  With record() calls
 * still pending in the queue (nutsb_q_speech / nutsb_q_record since the last flush or review) the calls return
 * NUTSB_E_STATE: flush first. */
int nutsb_set_speech_record(nutsb_ctx *ctx, int on);
/* Room `room`'s buffer as the reference holds it: REVIEW_LINES rows of REVIEW_LEN+2 bytes (rm->revbuff, strncpy's
 * NUL padding included) and the ring position (rm->revline).  Records still pending in the queue are not in it
 * until the next flush or review.  Either pointer may be NULL. */
int nutsb_get_review_buffer(nutsb_ctx *ctx, int32_t room, uint8_t *rows, int32_t *line);

/* ---- review buffers (queue tier; record c:2062, review c:5192, clear_revbuff c:2626) ------
 * nutsb_q_speech records what say / emote / echo send to the room (c:4099, c:4209, c:4304), as
 * the reference does: the first REVIEW_LEN bytes of the line ('\n' appended when it was cut).
 * nutsb_q_record is record() for any other caller.  nutsb_q_review queues what review() writes
 * to `user` for `room` (the room is the caller's to resolve: get_room / has_room_access):
 * header, the buffered lines oldest first through write_user again, footer -- or "Review
 * buffer is empty.".  Lines refused for swearing are never recorded: a review (like a flush)
 * first takes the swear verdicts of the lines queued so far.  Buffers are cleared by
 * nutsb_set_users (create_room, c:2799) and nutsb_q_review_clear. */
int nutsb_q_record(nutsb_ctx *ctx, int32_t room, const char *str);
/* tell c:4128 / pemote c:4234 after their argument checks (`target` = what get_user found: not the speaker, not
 * afk / ignoring / offsite -- the talker's state): the muzzle refusal, or the two lines ("~OLYou tell X:~RS ..." /
 * "~OLX tells you:~RS ...", ask for a trailing '?'; "~OL(To X)~RS ..." / "~OL>>~RS ...") and record_tell c:2074.
 * wizshout c:6527: muzzle refusal, ban_swearing branch (asked of the whole line, c:6541), then the speaker's line
 * and write_level(lev or WIZ, 1, line, user); inpstr = the whole line; lev < 0 = no level word, else the level
 * word is taken off inside (remove_first, c:6553) and level_name = level_name[lev].  revtell c:7699 replays the
 * user's five-line buffer through write_user.  Need nutsb_set_user_names. */
int nutsb_q_tell(nutsb_ctx *ctx, int32_t user, int32_t target, const char *inpstr);
int nutsb_q_pemote(nutsb_ctx *ctx, int32_t user, int32_t target, const char *inpstr);
int nutsb_q_wizshout(nutsb_ctx *ctx, int32_t user, int lev, const char *level_name, const char *inpstr);
int nutsb_q_revtell(nutsb_ctx *ctx, int32_t user);
int nutsb_q_review(nutsb_ctx *ctx, int32_t user, int32_t room, const char *room_name);
int nutsb_q_review_clear(nutsb_ctx *ctx, int32_t room);

/* ---- colour_com_count / colour_com_strip (nuts333.c:2563-2610), host buffers ------------- */
/* count[i] = colour_com_count(string i), including its double count ("~FBK" is 2). */
int nutsb_colour_com_count_batch(nutsb_ctx *ctx, int64_t n, const uint8_t *bytes, const uint64_t *off, int32_t *count);
/* string i with every "~XX" (XX a colour command) removed, as colour_com_strip returns it:
 * (*out_bytes)[(*out_off)[i] .. (*out_off)[i+1]); buffers owned by the context. */
int nutsb_colour_com_strip_batch(nutsb_ctx *ctx, int64_t n, const uint8_t *bytes, const uint64_t *off,
                                 const uint8_t **out_bytes, const uint64_t **out_off);

/* Position-weighted 64-bit digest of every user's stream, computed on the
 * device from the last write batch: h = fold(h*0x100000001b3 + byte) over the
 * stream, h0 = 0xcbf29ce484222325.  digest[n_users] is a HOST array.  NUTSB_E_STATE after a
 * gather-list batch that never built the streams (plain listeners: nothing to digest in HBM). */
int nutsb_stream_digests(nutsb_ctx *ctx, uint64_t *digest);

/* The parity digests of SURVEY.md 8(d) for the last write batch whose streams are in HBM (host arrays, either may be
 * NULL): d(m,u) = 64-bit FNV-1a (offset 0xcbf29ce484222325, prime 0x100000001b3) over the rendered bytes of one delivery;
 * per_user[u] = the left fold over u's deliveries in call order, per_op[m] = the same fold over op m's recipients in
 * user-list order (the loop of nuts333.c:1409):  D <- (D * 0x9E3779B97F4A7C15) ^ d ^ len, D0 = 0.  A delivery of no
 * bytes makes no write(2) in the reference and is not folded; an op that was gated off or reached nobody has digest 0.
 * The message-major view of the batch: what each call delivered, without materialising a byte per recipient. */
int nutsb_delivery_digests(nutsb_ctx *ctx, uint64_t *per_user, uint64_t *per_op);
/* Streams left in HBM: ops in host memory, nutsb_streams with device pointers (on_device 1) -- for a caller
 * that only wants digests (nutsb_stream_digests) or copies what it needs later. */
int nutsb_write_batch_keep(nutsb_ctx *ctx, const nutsb_ops *ops, nutsb_streams *out);
/* nutsb_stream_digests continuing from the values in digest[]: the fold over what a user received in earlier
 * batches goes on over this batch's stream (a job run in message-ordered chunks, SURVEY 8d config 5). */
int nutsb_stream_digests_continue(nutsb_ctx *ctx, uint64_t *digest);

/* ---- several GPUs: one population, one batch (SURVEY.md 8e) ------------------------------------
 * The path shards by room with no exchange step.  nutsb_multi holds one context per shard; rooms are dealt to
 * the shards heaviest first onto the least loaded one (weight: the room's population, or room_weight[]), a room's
 * users go with it.  A batch is routed on the host: write_user -> the user's shard, write_room[_except](rm) -> rm's
 * shard, the all-room forms (rm == NULL, nuts333.c:1399-1400: shout c:4119-4123, bcast c:4783-4787) and write_level
 * (c:1372-1385) are replicated to every shard, each rendering for its own users.  Shards run concurrently, one host
 * thread and one device each, no collective; results come back in GLOBAL user order.  Clones / remote users are
 * refused (NUTSB_E_UNSUPPORTED): their relays cross rooms.
 * nutsb_multi_create_rank: one process per GPU (torchrun) -- this process runs shard `shard` only; every process
 * gives the same population and batches, plans and routes identically, and reports its own users' streams
 * (the users of the other shards come back empty). */
typedef struct nutsb_multi nutsb_multi;
typedef struct nutsb_mstreams {
    int64_t         n_users;
    uint64_t        total_bytes;    /* over the shards this process runs                   */
    uint64_t        n_deliveries;
    const uint64_t *len;            /* n_users: length of user u's stream (NULL when kept in HBM) */
    const uint8_t *const *ptr;      /* n_users: its bytes, in the owning shard's pinned buffer     */
    int32_t         on_device;      /* 1: the streams were left in HBM (keep != 0)          */
} nutsb_mstreams;
int  nutsb_multi_create(nutsb_multi **out, const int *device_ids, int n_devices);
int  nutsb_multi_create_rank(nutsb_multi **out, int n_shards, int shard, int device);
void nutsb_multi_destroy(nutsb_multi *m);
const char *nutsb_multi_last_error(const nutsb_multi *m);
int  nutsb_multi_n_shards(const nutsb_multi *m);
nutsb_ctx *nutsb_multi_ctx(nutsb_multi *m, int shard);          /* NULL for a shard this process does not run */
int  nutsb_multi_set_swear_words(nutsb_multi *m, const char *const *words);
int  nutsb_multi_set_ban_files(nutsb_multi *m, const void *siteban, size_t siteban_len, const void *userban, size_t userban_len);
int  nutsb_multi_set_profiling(nutsb_multi *m, int on);
int  nutsb_multi_set_users(nutsb_multi *m, int32_t n_users, int32_t n_rooms, const int32_t *room,
                           const uint8_t *flags, const uint8_t *level, const uint64_t *room_weight);
int  nutsb_multi_plan(const nutsb_multi *m, int32_t *room_shard, int32_t *user_shard, int32_t *user_local);
int  nutsb_multi_route(nutsb_multi *m, const nutsb_ops *ops, int shard, nutsb_ops *out);
int  nutsb_multi_write_batch(nutsb_multi *m, const nutsb_ops *ops, nutsb_mstreams *out, int keep);
int  nutsb_multi_stream_digests(nutsb_multi *m, uint64_t *digest, int cont);
int  nutsb_multi_contains_swearing_batch(nutsb_multi *m, int64_t n, const uint8_t *bytes, const uint64_t *off, uint8_t *verdict);
int  nutsb_multi_site_banned_batch(nutsb_multi *m, int64_t n, const uint8_t *bytes, const uint64_t *off, uint8_t *verdict);
int  nutsb_multi_user_banned_batch(nutsb_multi *m, int64_t n, const uint8_t *bytes, const uint64_t *off, uint8_t *verdict);
int  nutsb_multi_get_timing(const nutsb_multi *m, int shard, nutsb_timing *out);

/* Gather lists over the shards (see nutsb_write_batch_iov), in GLOBAL user order: user u's stream is
 *     writev(sock, (const struct iovec *)s.iov[u], s.count[u]);
 * iov[u] points at u's first piece inside the gather list of u's shard (no byte is copied); pieces point into
 * that shard's pools (nutsb_multi_shard_iov).  Valid until the next batch on the handle. */
typedef struct nutsb_miov_streams {
    int64_t                   n_users;
    uint64_t                  total_bytes, n_deliveries;   /* over the shards this process runs          */
    const uint64_t           *len;     /* n_users: length of user u's stream                          */
    const nutsb_iovec *const *iov;     /* n_users: u's first piece, inside its shard's iov array      */
    const uint32_t           *count;   /* n_users: u's pieces (0, iov[u] NULL: a shard not run here)  */
} nutsb_miov_streams;
int  nutsb_multi_write_batch_iov(nutsb_multi *m, const nutsb_ops *ops, nutsb_miov_streams *out);
/* the last gather-list batch's result of one shard as nutsb_write_batch_iov gives it (local user order, its pools) */
int  nutsb_multi_shard_iov(const nutsb_multi *m, int shard, nutsb_iov_streams *out);

/* Speech batches over the shards (see nutsb_speech_batch).  Names and speech flags in GLOBAL user order, before or
 * after nutsb_multi_set_users; every speaker index is a global one.  Every shard is given the whole batch and picks,
 * on the device, the lines that produce an op on it, by the same rule the one-context composer uses: the refusal,
 * the speaker's own copy and the line to the speaker's room go to the speaker's shard; shout / semote / bcast (all rooms) and echo's
 * write_level(WIZ) go to every shard.  Each shard takes the swear verdicts of the whole batch.  Streams, totals and
 * errors as for nutsb_multi_write_batch (keep != 0: the streams stay in HBM, nutsb_multi_stream_digests);
 * NUTSB_E_STATE when the names do not match the population. */
int  nutsb_multi_set_user_names(nutsb_multi *m, int32_t n_users, const uint8_t *names, const uint64_t *off,
                                const uint8_t *speech_flags);
int  nutsb_multi_set_ban_swearing(nutsb_multi *m, int on);
int  nutsb_multi_speech_batch(nutsb_multi *m, int64_t n, const uint8_t *verb, const int32_t *speaker,
                              const uint8_t *bodies, const uint64_t *body_off, nutsb_mstreams *out, int keep);
int  nutsb_multi_speech_batch_iov(nutsb_multi *m, int64_t n, const uint8_t *verb, const int32_t *speaker,
                                  const uint8_t *bodies, const uint64_t *body_off, nutsb_miov_streams *out);
/* Recording (nutsb_set_speech_record) on every shard: each records the lines of its own rooms, and the buffers change
 * only when every shard has succeeded.  nutsb_multi_set_users carries each room's buffer to its new shard and local
 * index.  Rank mode refuses it (NUTSB_E_UNSUPPORTED): a buffer cannot follow a room into another process.
 * nutsb_multi_get_review_buffer: global room `room`'s buffer (nutsb_get_review_buffer). */
int  nutsb_multi_set_speech_record(nutsb_multi *m, int on);
int  nutsb_multi_get_review_buffer(nutsb_multi *m, int32_t room, uint8_t *rows, int32_t *line);

/* ---- calls in flight on one device -----------------------------------------------------------------
 * A host-buffer call is H2D copy -> kernels -> D2H copy; PCIe is full duplex, so with two calls in flight one call's
 * H2D and kernels run under the other's D2H.  nutsb_pipe holds `depth` contexts on one device with a worker thread
 * each: submit returns at once, wait returns the call's result (valid until `depth` further submissions; the call's
 * input buffers must stay valid until it has been waited for).  The setters reach every context. */
typedef struct nutsb_pipe nutsb_pipe;
int  nutsb_pipe_create(nutsb_pipe **out, int device, int depth);
void nutsb_pipe_destroy(nutsb_pipe *p);
int  nutsb_pipe_depth(const nutsb_pipe *p);
nutsb_ctx *nutsb_pipe_ctx(nutsb_pipe *p, int lane);
int  nutsb_pipe_set_swear_words(nutsb_pipe *p, const char *const *words);
int  nutsb_pipe_set_users(nutsb_pipe *p, int32_t n_users, int32_t n_rooms, const int32_t *room, const uint8_t *flags, const uint8_t *level);
int  nutsb_pipe_set_user_names(nutsb_pipe *p, int32_t n_users, const uint8_t *names, const uint64_t *off, const uint8_t *speech_flags);
int  nutsb_pipe_set_ban_swearing(nutsb_pipe *p, int on);
int  nutsb_pipe_submit_speech_iov(nutsb_pipe *p, int64_t n, const uint8_t *verb, const int32_t *speaker,
                                  const uint8_t *bodies, const uint64_t *body_off, uint64_t *ticket);
int  nutsb_pipe_submit_write_iov(nutsb_pipe *p, const nutsb_ops *ops, uint64_t *ticket);
int  nutsb_pipe_wait(nutsb_pipe *p, uint64_t ticket, nutsb_iov_streams *out);

/* ---- queue tier: the reference's call surface, one call each ------------ */

int nutsb_q_write_user(nutsb_ctx *ctx, int32_t user, const char *str);            /* c:1291 */
int nutsb_q_write_room(nutsb_ctx *ctx, int32_t room, const char *str,
                       int force_listen, int shout);                              /* c:1390 */
int nutsb_q_write_room_except(nutsb_ctx *ctx, int32_t room, const char *str, int32_t except_user,
                              int force_listen, int shout);                       /* c:1401 */
int nutsb_q_write_level(nutsb_ctx *ctx, int level, int above, const char *str,
                        int32_t except_user);                                     /* c:1372 */
/* write_sock(sock, str) (c:1281-1286) to the socket of user `sock_user` (or of a netlink's pseudo-user): the
 * bytes as they are (NUTSB_OF_RAW), in order with everything else queued for that socket.  A socket that is
 * nobody's (accept_connection's refusal, c:280) is the host's own write(2) -- after a flush. */
int nutsb_q_write_sock(nutsb_ctx *ctx, int32_t sock_user, const char *str);
/* One fgets() chunk of a paged file as more() writes it (c:2254-2300): the byte machine of
 * write_user without the closing reset; plain != 0 when more() was called with user==NULL. */
int nutsb_q_page_line(nutsb_ctx *ctx, int32_t sock_user, const char *str, int plain);
/* The pager more(user, sock, filename) (c:2205-2322) over the file's BYTES (file == NULL:
 * fopen failed): queues one page -- the fgets(text,1999) chunks from *filepos until 23
 * screen lines are counted (all of it when user < 0) and, if the file is not finished, the
 * "Press <return>" prompt -- for sock_user, updates *filepos as the reference updates
 * user->filepos, and returns more()'s return value (0 no file, 1 more to come, 2 done) in
 * *retval.  user = -1 stands for user==NULL (login: colour taken as off, no paging). */
int nutsb_q_more(nutsb_ctx *ctx, int32_t user, int32_t sock_user, const void *file, size_t file_len,
                 int64_t *filepos, int *retval);
int64_t nutsb_q_pending(const nutsb_ctx *ctx);
/* Runs everything queued since the last flush; the host then write()s each
 * user's stream to its socket.  The queue is emptied when the batch has run and when it can never run
 * (a validation error); after NUTSB_E_NOMEM / NUTSB_E_CUDA it is kept -- ops, swear bodies, pending
 * record() calls -- so that the flush can be tried again, and the review buffers take the queued lines
 * only once the batch that delivers them has succeeded.  A queue call that fails (NUTSB_E_RANGE: a relay
 * or frame over NUTSB_MAX_TEXT) queues nothing. */
int nutsb_flush(nutsb_ctx *ctx, nutsb_streams *out);
/* The same with gather lists as the result (nutsb_write_batch_iov): the host writev()s each user's list. */
int nutsb_flush_iov(nutsb_ctx *ctx, nutsb_iov_streams *out);

/* Synchronous single-item verdicts (the callers branch on them immediately,
 * c:4091, c:279, c:1496): one tiny launch each, latency-bound by design. */
int nutsb_contains_swearing(nutsb_ctx *ctx, const char *str);                     /* c:2540 */
int nutsb_site_banned(nutsb_ctx *ctx, const char *site);                          /* c:330  */
int nutsb_user_banned(nutsb_ctx *ctx, const char *name);                          /* c:349  */

#ifdef __cplusplus
}
#endif
#endif /* NUTSB200_H */
