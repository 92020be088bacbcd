/* tl/nvl collectives: argument translation, algorithm table, launch + completion.
 * All 16 collective types map onto four kernels:
 *   reduce family   -> nvl_allreduce_oneshot / nvl_reduce_staged (P2P or NVLS)
 *   data movement   -> nvl_exchange (stage + pull)
 *   synchronisation -> nvl_barrier                                                     */
#include "tl_nvl.h"
#include "core/ucc_progress_queue.h"
#include "utils/profile/ucc_profile.h"
#include "utils/ucc_string.h"
#include <strings.h>

#define NVL_LIB(_t) ((_t)->super.super.context->lib)

static int to_nvl_dt(ucc_datatype_t dt)
{
    switch (dt) {
    case UCC_DT_INT8: return NVL_DT_I8; case UCC_DT_INT16: return NVL_DT_I16; case UCC_DT_INT32: return NVL_DT_I32; case UCC_DT_INT64: return NVL_DT_I64;
    case UCC_DT_UINT8: return NVL_DT_U8; case UCC_DT_UINT16: return NVL_DT_U16; case UCC_DT_UINT32: return NVL_DT_U32; case UCC_DT_UINT64: return NVL_DT_U64;
    case UCC_DT_FLOAT16: return NVL_DT_F16; case UCC_DT_FLOAT32: return NVL_DT_F32; case UCC_DT_FLOAT64: return NVL_DT_F64; case UCC_DT_BFLOAT16: return NVL_DT_BF16;
    case UCC_DT_FLOAT32_COMPLEX: return NVL_DT_C64; case UCC_DT_FLOAT64_COMPLEX: return NVL_DT_C128;
    default: return -1;
    }
}
static int to_nvl_op(ucc_reduction_op_t op)
{
    switch (op) {
    case UCC_OP_SUM: return NVL_OP_SUM; case UCC_OP_PROD: return NVL_OP_PROD; case UCC_OP_MAX: return NVL_OP_MAX; case UCC_OP_MIN: return NVL_OP_MIN;
    case UCC_OP_LAND: return NVL_OP_LAND; case UCC_OP_LOR: return NVL_OP_LOR; case UCC_OP_LXOR: return NVL_OP_LXOR; case UCC_OP_BAND: return NVL_OP_BAND;
    case UCC_OP_BOR: return NVL_OP_BOR; case UCC_OP_BXOR: return NVL_OP_BXOR; case UCC_OP_AVG: return NVL_OP_AVG;
    default: return -1;
    }
}
static inline int is_cuda(ucc_memory_type_t mt) { return mt == UCC_MEMORY_TYPE_CUDA; }

/* ------------------------------------------------------------------ */
/* task life cycle                                                     */
/* ------------------------------------------------------------------ */
/* what the most recent launch of this process was (benchmarks print it next to their numbers): "<kernel> grid x block" */
static cudaEvent_t event_get(ucc_tl_nvl_context_t *ctx);
static char nvl_last_launch[128];
UCC_EXPORT const char *ucc_tl_nvl_last_launch_info(void) { return nvl_last_launch; }
static void note_launch(const ucc_tl_nvl_task_t *t)
{
    const char *k = "barrier"; int nb = t->nblocks;
    switch (t->kind) {
    case NVL_TASK_REDUCE_ONESHOT: k = t->u.red.kind == NVL_RED_REDUCE_SCATTER ? "oneshot_rs" : "oneshot"; break;
    case NVL_TASK_REDUCE_STAGED:
        if (t->u.red.direct == NVL_DIRECT_FULL) { k = "twoshot_zcopy(direct)"; nb = t->nblocks_direct; }
        else k = (t->u.red.use_nvls && t->team->nvls) ? "nvls_staged" : "twoshot_staged";
        break;
    case NVL_TASK_REDUCE_STEPS: k = t->u.red.sched == 1 ? "ring" : "rhd"; break;
    case NVL_TASK_REDUCE_PIPE: k = "nvls_pipe"; break;
    case NVL_TASK_REDUCE_SYMM: k = "nvls_symm_inplace"; break;
    case NVL_TASK_AG_SYMM: k = "allgather_symm_mc"; break;
    case NVL_TASK_XCHG: k = (t->use_push && t->u.xchg.direct) ? (t->use_ce ? "exchange_push_copy_engine" : (t->use_bulk ? "exchange_push_bulk(tma)" : "exchange_push")) : (t->u.xchg.direct ? "exchange_pull_zcopy" : (t->u.xchg.use_mc ? "exchange_nvls" : (t->u.xchg.ring ? "exchange_ring" : "exchange_pull_staged"))); break;
    case NVL_TASK_SELF_COPY: k = t->use_bulk ? "self_copy_bulk(tma)" : "self_copy"; break;
    case NVL_TASK_P2P:
        if (t->u.p2p.mode == NVL_P2P_PUSH) { k = "p2p_send_rndv(push)"; nb = nvl_p2p_push_ctas(t->u.p2p.bytes); }
        else if (t->u.p2p.mode == NVL_P2P_WAIT) { k = "p2p_recv_rndv(wait)"; nb = 1; }
        else { k = t->u.p2p.send ? "p2p_send" : "p2p_recv"; nb = nvl_p2p_lanes(t->u.p2p.bytes); }
        break;
    default: nb = 1; break;
    }
    snprintf(nvl_last_launch, sizeof(nvl_last_launch), "%s %dx%d", k, nb, (t->use_bulk && !t->use_ce && (t->kind == NVL_TASK_SELF_COPY || (t->use_push && t->u.xchg.direct))) ? 32 : t->nthreads);
}

static ucc_status_t nvl_launch(ucc_tl_nvl_task_t *t, cudaStream_t s)
{
    cudaError_t e;
    note_launch(t);
    switch (t->kind) {
    case NVL_TASK_REDUCE_ONESHOT:
        e = t->u.red.kind == NVL_RED_REDUCE_SCATTER ? nvl_launch_reduce_scatter_oneshot(&t->u.red, t->nblocks, t->nthreads, s)
                                                    : nvl_launch_allreduce_oneshot(&t->u.red, t->nblocks, t->nthreads, s);
        break;
    case NVL_TASK_REDUCE_STAGED:
        if (t->u.red.direct == NVL_DIRECT_FULL) e = nvl_launch_reduce_direct(&t->u.red, t->nblocks_direct, t->nthreads, s);
        else e = nvl_launch_reduce_staged(&t->u.red, t->nblocks, t->nthreads, s);
        break;
    case NVL_TASK_REDUCE_STEPS: e = nvl_launch_reduce_steps(&t->u.red, t->nblocks, t->nthreads, s); break;
    case NVL_TASK_REDUCE_PIPE: e = nvl_launch_reduce_pipe(&t->u.red, t->nblocks, t->nthreads, s); break;
    case NVL_TASK_REDUCE_SYMM: e = nvl_launch_reduce_symm(&t->u.red, t->nblocks, t->nthreads, s); break;
    case NVL_TASK_AG_SYMM: e = nvl_launch_allgather_symm(&t->u.xchg, t->nblocks, t->nthreads, s); break;
    case NVL_TASK_XCHG:
        if (t->use_push && t->u.xchg.direct) { /* every member's destination resolved: store my blocks straight into them */
            nvl_push_args_t pa;
            memset(&pa, 0, sizeof(pa));
            pa.team = t->u.xchg.team; pa.src = t->u.xchg.src;
            for (int p = 0; p < pa.team.size; p++) {
                pa.send_off[p] = t->push.send_off[p]; pa.send_bytes[p] = t->push.send_bytes[p]; pa.land_off[p] = t->push.land_off[p]; pa.recv_off[p] = t->push.recv_off[p];
                pa.dst_of[p] = p == pa.team.rank ? (char *)t->u.xchg.dst : t->u.xchg.d.dst[p];
            }
            pa.lookup = t->push.lookup;
            /* (every member takes this branch or none: `direct` is decided from what all of them published) */
            if (t->use_ce) {
                /* copy-engine variant (reference tl/cuda alltoallv_ce.c:202-439: cudaMemcpyAsync per peer after an IPC handle
                 * exchange and a host barrier): barrier kernel (every member's stream reached the collective: its dst may be
                 * written) -> one DMA per peer, straight into the mapped destinations; no SM moves a byte -> barrier kernel
                 * (everything has landed).  The landing offsets of alltoallv travelled with the buffer exchange (peer_land). */
                e = nvl_launch_barrier(&t->u.xchg.team, s);
                for (int i = 1; i <= pa.team.size && e == cudaSuccess; i++) {
                    int p = (pa.team.rank + i) % pa.team.size;
                    size_t land = pa.lookup ? t->push.peer_land[p] : pa.land_off[p];
                    if (!pa.send_bytes[p] || pa.dst_of[p] + land == (const char *)pa.src + pa.send_off[p]) continue;
                    e = cudaMemcpyAsync(pa.dst_of[p] + land, (const char *)pa.src + pa.send_off[p], pa.send_bytes[p], cudaMemcpyDeviceToDevice, s);
                }
                if (e == cudaSuccess) e = nvl_launch_barrier(&t->u.xchg.team, s);
                break;
            }
            e = t->use_bulk ? nvl_launch_exchange_push_bulk(&pa, t->nblocks, s) : nvl_launch_exchange_push(&pa, t->nblocks, t->nthreads, s);
        } else e = nvl_launch_exchange(&t->u.xchg, t->nblocks, t->nthreads, s);
        break;
    case NVL_TASK_P2P: e = nvl_launch_p2p(&t->u.p2p, t->nthreads, s); break;
    case NVL_TASK_SELF_COPY:
        if (!t->u.xchg.src_bytes) e = cudaSuccess;
        else if (t->use_bulk) e = nvl_launch_self_copy_bulk(t->u.xchg.dst, t->u.xchg.src, t->u.xchg.src_bytes, t->nblocks, s);
        else e = nvl_launch_self_copy(t->u.xchg.dst, t->u.xchg.src, t->u.xchg.src_bytes, t->nblocks, t->nthreads, s);
        break;
    default: e = nvl_launch_barrier(&t->u.red.team, s); break;
    }
    if (e != cudaSuccess) { tl_error(NVL_LIB(t->team), "kernel launch failed: %s", cudaGetErrorString(e)); return UCC_ERR_NO_MESSAGE; }
    return UCC_OK;
}

/* Kernels of one team must start in post order on every rank (the device-side epochs count launches), even when
 * consecutive posts use different streams: chain them with the completion event of the previous launch. */
static ucc_status_t launch_ordered(ucc_tl_nvl_task_t *t, cudaStream_t s)
{
    ucc_tl_nvl_team_t *team = t->team;
    ucc_status_t st;
    if (t->captured) return nvl_launch(t, s);
    if (t->kind == NVL_TASK_P2P) { /* channel counters, no barrier epochs: independent of the team's collective order */
        st = nvl_launch(t, s);
        if (st != UCC_OK) return st;
        CUDA_CHECK(cudaEventRecord(t->event, s));
        return UCC_OK;
    }
    if (team->last_event[t->lane] && team->last_stream[t->lane] != s) CUDA_CHECK(cudaStreamWaitEvent(s, team->last_event[t->lane], 0));
    st = nvl_launch(t, s);
    if (st != UCC_OK) return st;
    CUDA_CHECK(cudaEventRecord(t->event, s));
    team->last_event[t->lane] = t->event; team->last_stream[t->lane] = s;
    return UCC_OK;
}

/* point the task's device descriptor at its lane: a lane is a complete [control | one-shot | p2p | data] image at
 * lane * lane_stride of every member's heap (and of the multicast mapping), so the kernels need no lane awareness */
static void task_set_lane(ucc_tl_nvl_task_t *t, unsigned lane)
{
    ucc_tl_nvl_team_t *team = t->team;
    nvl_team_dev_t *d = (t->kind == NVL_TASK_XCHG || t->kind == NVL_TASK_AG_SYMM) ? &t->u.xchg.team : &t->u.red.team;
    size_t off = (size_t)lane * team->lane_stride;
    t->lane = lane;
    if (t->kind == NVL_TASK_SELF_COPY || t->kind == NVL_TASK_P2P) return;
    for (int p = 0; p < team->dev.size; p++) d->heap[p] = team->dev.heap[p] + off;
    d->mc_heap = team->dev.mc_heap ? team->dev.mc_heap + off : NULL;
}

/* every member published its buffers for this collective: pick (identically everywhere) the in-place kernel or
 * the staged one and fill the pointer tables */
static ucc_status_t resolve_direct(ucc_tl_nvl_task_t *t)
{
    nvl_direct_t d;
    int ok = ucc_tl_nvl_xb_resolve(t->team, t->cseq, t->need_src, t->need_dst, t->kind != NVL_TASK_XCHG, t->exp_src, t->exp_dst, &d, (t->kind == NVL_TASK_XCHG && t->use_push) ? t->push.peer_land : NULL);
    tl_debug(NVL_LIB(t->team), "exchange %lu: %s (src %d dst %d)", (unsigned long)t->cseq, ok > 0 ? "zero-copy" : (ok ? "MAPPING FAILED" : "staged"), t->need_src, t->need_dst);
    if (ok < 0) {
        tl_error(NVL_LIB(t->team), "cannot map a peer's buffer for the zero-copy kernel (the peers will run it): failing the collective; "
                 "UCC_TL_NVL_ZCOPY=n avoids the zero-copy path");
        return UCC_ERR_NO_RESOURCE;
    }
    if (t->kind == NVL_TASK_XCHG) { t->u.xchg.direct = ok; if (ok) t->u.xchg.d = d; }
    else { t->u.red.direct = ok ? t->want_direct : NVL_DIRECT_NONE; if (ok) t->u.red.d = d; }
    /* persistent request: the buffers are fixed for the lifetime of the request, so every later post of it (same decision on
     * every member - they all re-post the same request) launches straight away with these tables: no handle export, no board
     * round trip, no deferred launch */
    if (UCC_IS_PERSISTENT(t->super.bargs.args)) { t->direct_cached = 1; t->cached_mode = ok ? 1 : 0; t->cached_d = d; }
    return UCC_OK;
}
static void apply_cached_direct(ucc_tl_nvl_task_t *t)
{
    int ok = t->cached_mode;
    if (t->kind == NVL_TASK_XCHG) { t->u.xchg.direct = ok; if (ok) t->u.xchg.d = t->cached_d; }
    else { t->u.red.direct = ok ? t->want_direct : NVL_DIRECT_NONE; if (ok) t->u.red.d = t->cached_d; }
}
static inline int task_is_direct(const ucc_tl_nvl_task_t *t) { return t->want_direct && (t->team->zcopy || t->direct_cached); }

/* Registered buffers: when the collective carries GLOBAL memory handles (one imported ucc_mem_map handle per member) for every
 * side the zero-copy kernel touches, the pointer tables are built right here from the registrations - the per-post exchange is
 * never used for this request.  Every member evaluates the same handles, flags and sizes, so the outcome is the same everywhere;
 * a member that cannot reach some segment could break that symmetry, so reachability of ALL segments is required on import
 * (unreachable -> h->mapped == NULL -> no table, and since the exporter could not produce an IPC handle either, nobody has one). */
static void memh_direct(ucc_tl_nvl_task_t *t, const ucc_coll_args_t *a, const void *my_src, void *my_dst)
{
    ucc_tl_nvl_team_t *team = t->team;
    const ucc_base_context_t *bctx = team->super.super.context;
    ucc_rank_t N = UCC_TL_TEAM_SIZE(team), me = UCC_TL_TEAM_RANK(team);
    int use_src = t->need_src && (a->mask & UCC_COLL_ARGS_FIELD_MEM_MAP_SRC_MEMH) && (a->flags & UCC_COLL_ARGS_FLAG_SRC_MEMH_GLOBAL) && a->src_memh.global_memh;
    int use_dst = t->need_dst && (a->mask & UCC_COLL_ARGS_FIELD_MEM_MAP_DST_MEMH) && (a->flags & UCC_COLL_ARGS_FLAG_DST_MEMH_GLOBAL) && a->dst_memh.global_memh;
    nvl_direct_t d;
    if (!t->want_direct || (t->need_src && !use_src) || (t->need_dst && !use_dst)) return;
    memset(&d, 0, sizeof(d));
    for (int side = 0; side < 2; side++) {
        ucc_mem_map_mem_h *gl = side ? a->dst_memh.global_memh : a->src_memh.global_memh;
        const char *mine = side ? (const char *)my_dst : (const char *)my_src;
        nvl_memh_t *hm;
        size_t off;
        if (side ? !use_dst : !use_src) continue;
        hm = (nvl_memh_t *)ucc_mem_map_tl_handle(gl[me], bctx);
        if (!hm || !hm->mapped || mine < hm->mapped || mine >= hm->mapped + hm->len) return; /* my buffer is not inside my registered segment */
        off = (size_t)(mine - hm->mapped);
        if ((uintptr_t)mine & 15) return;
        for (ucc_rank_t p = 0; p < N; p++) {
            nvl_memh_t *h = (nvl_memh_t *)ucc_mem_map_tl_handle(gl[p], bctx);
            if (!h || !h->mapped || off >= h->len || ((uintptr_t)(h->mapped + off) & 15)) return;
            if (side) d.dst[p] = p == me ? (char *)my_dst : h->mapped + off; else d.src[p] = p == me ? (const char *)my_src : h->mapped + off;
        }
    }
    t->direct_cached = 1; t->cached_mode = 1; t->cached_d = d;
}

/* ------------------------------------------------------------------ */
/* send / recv.  Small messages: eager, through the pair's ring in the receiver's heap, one kernel per side, launched at post.
 * Large messages (P2P_RNDV_THRESH): rendezvous.  The receiver puts (IPC handle, offset) of its buffer on its board - but only
 * once its stream has reached the recv (the sender may write from then on) - and parks a one-warp kernel on its stream that
 * waits for the pair's message counter.  The sender maps the buffer (cached) and launches a kernel that stores into it
 * directly and bumps that counter.  That kernel never waits for anything on the device, and it runs on a per-peer side stream
 * behind an event of the user's stream, so an exchange posted as send + recv on ONE stream on both sides cannot deadlock
 * (with NCCL that shape needs a group).  A receiver whose buffer cannot be exported says so on the board and both sides use
 * the ring for that message.  Sends to one peer are launched strictly in post order. */
static ucc_status_t p2p_side_stream(ucc_tl_nvl_team_t *team, int peer)
{
    if (team->p2p_stream[peer]) return UCC_OK;
    CUDA_CHECK(cudaStreamCreateWithFlags(&team->p2p_stream[peer], cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreateWithFlags(&team->p2p_side_event[peer], cudaEventDisableTiming));
    return UCC_OK;
}
static inline int xb_kind_mappable(int kind) { return kind == NVL_XB_RAW || kind == NVL_XB_IPC; }

static void p2p_try_publish(ucc_tl_nvl_task_t *t)
{
    ucc_tl_nvl_team_t *team = t->team;
    int peer = t->u.p2p.peer;
    ucc_rank_t me = UCC_TL_TEAM_RANK(team);
    nvl_xb_rz_t *e = &team->xb_mine->rz[peer][t->rz_seq % NVL_XB_RZ_SLOTS];
    if (!t->rz_pub_pending || t->rz_seq != team->rz_pub[peer]) return;
    if (t->rz_seq >= NVL_XB_RZ_SLOTS && ucc_load_acquire(&team->xb[peer]->rz_consumed[me]) + NVL_XB_RZ_SLOTS <= t->rz_seq) return;
    if (xb_kind_mappable(t->rz_buf.kind) && !t->rz_stream_idle) { /* my stream must be at the recv: earlier work in it may still use the buffer */
        cudaError_t ce = cudaEventQuery(t->in_event);
        if (ce == cudaErrorNotReady) { (void)cudaGetLastError(); return; }
    }
    e->buf = t->rz_buf;
    ucc_store_release(&e->seq, t->rz_seq + 1);
    team->rz_pub[peer]++; t->rz_pub_pending = 0;
}

static ucc_status_t p2p_try_wait(ucc_tl_nvl_task_t *t)
{
    ucc_tl_nvl_team_t *team = t->team;
    int peer = t->u.p2p.peer;
    ucc_rank_t me = UCC_TL_TEAM_RANK(team);
    ucc_status_t st;
    if (!t->rz_wait_pending || t->rz_pub_pending) return UCC_OK;
    if ((int32_t)(ucc_load_acquire(&team->xb[peer]->rz_launched[me]) - (t->u.p2p.rz_seq + 1)) < 0) return UCC_OK;
    st = nvl_launch(t, t->stream);
    if (st != UCC_OK) return st;
    CUDA_CHECK(cudaEventRecord(t->event, t->stream));
    t->rz_wait_pending = 0;
    return UCC_OK;
}

/* UCC_OK: launched; UCC_INPROGRESS: not its turn / the receiver has not published yet */
static ucc_status_t p2p_try_send(ucc_tl_nvl_task_t *t, int at_post)
{
    ucc_tl_nvl_team_t *team = t->team;
    int peer = t->u.p2p.peer, side = !at_post;
    ucc_rank_t me = UCC_TL_TEAM_RANK(team);
    ucc_status_t st;
    if (t->p2p_order != team->p2p_launch_seq[peer]) return UCC_INPROGRESS;
    t->u.p2p.mode = NVL_P2P_RING;
    if (t->p2p_rndv && !t->captured) {
        const nvl_xb_rz_t *e = &team->xb[peer]->rz[me][t->rz_seq % NVL_XB_RZ_SLOTS];
        if (ucc_load_acquire(&e->seq) != t->rz_seq + 1) return UCC_INPROGRESS;
        if (xb_kind_mappable(e->buf.kind)) {
            char *remote = e->buf.len == t->u.p2p.bytes ? ucc_tl_nvl_xb_import(team, (ucc_rank_t)peer, &e->buf) : NULL;
            if (!remote) {
                tl_error(NVL_LIB(team), "send to %d: %s", peer, e->buf.len == t->u.p2p.bytes ? "cannot map the receiver's buffer" : "message size differs from the posted receive");
                ucc_store_release(&team->xb_mine->rz_consumed[peer], t->rz_seq + 1);
                team->p2p_launch_seq[peer]++;
                return UCC_ERR_NO_RESOURCE;
            }
            t->u.p2p.mode = NVL_P2P_PUSH; t->u.p2p.remote = remote; t->u.p2p.rz_seq = team->rz_zc_tx[peer]++;
            side = 1;   /* all zero-copy sends to a peer share one stream: their completion counter must advance in order */
        }
        ucc_store_release(&team->xb_mine->rz_consumed[peer], t->rz_seq + 1);
    }
    if (side) {
        st = p2p_side_stream(team, peer);
        if (st != UCC_OK) return st;
        CUDA_CHECK(cudaStreamWaitEvent(team->p2p_stream[peer], t->in_event, 0));
        st = nvl_launch(t, team->p2p_stream[peer]);
        if (st != UCC_OK) return st;
        CUDA_CHECK(cudaEventRecord(t->event, team->p2p_stream[peer]));
        CUDA_CHECK(cudaEventRecord(team->p2p_side_event[peer], team->p2p_stream[peer]));
        team->p2p_side_used[peer] = 1;
        if (t->u.p2p.mode == NVL_P2P_PUSH) ucc_store_release(&team->xb_mine->rz_launched[peer], t->u.p2p.rz_seq + 1);
        CUDA_CHECK(cudaStreamWaitEvent(t->stream, t->event, 0));   /* the send is "in" the user's stream from here on */
    } else {
        if (team->p2p_side_used[peer] && !t->captured) CUDA_CHECK(cudaStreamWaitEvent(t->stream, team->p2p_side_event[peer], 0));
        st = nvl_launch(t, t->stream);
        if (st != UCC_OK) return st;
        if (!t->captured) CUDA_CHECK(cudaEventRecord(t->event, t->stream));
    }
    team->p2p_launch_seq[peer]++;
    return UCC_OK;
}

static ucc_status_t p2p_post(ucc_tl_nvl_task_t *t, cudaStream_t s)
{
    ucc_tl_nvl_team_t *team = t->team;
    int peer = t->u.p2p.peer, rndv = t->p2p_rndv && !t->captured;
    ucc_status_t st;
    t->u.p2p.mode = NVL_P2P_RING; t->rz_pub_pending = 0; t->rz_wait_pending = 0;
    tl_debug(NVL_LIB(team), "%s %zu bytes %s %d: %s (P2P_RNDV_THRESH %zu, zero-copy boards %d)", t->u.p2p.send ? "send" : "recv", t->u.p2p.bytes,
             t->u.p2p.send ? "to" : "from", peer, rndv ? "rendezvous" : "eager ring", NVL_CTX(team)->cfg.p2p_rndv_thresh, team->zcopy);
    if (!t->captured && !t->in_event) { t->in_event = event_get(NVL_CTX(team)); if (!t->in_event) return UCC_ERR_NO_RESOURCE; }
    if (t->u.p2p.send) {
        t->p2p_order = team->p2p_post_seq[peer]++;
        if (rndv) t->rz_seq = team->rz_tx[peer]++;
        if (t->captured && t->p2p_order != team->p2p_launch_seq[peer]) {
            tl_error(NVL_LIB(team), "send to %d posted into a capturing stream while earlier sends to it are still waiting for the receiver", peer);
            team->p2p_post_seq[peer]--;
            return UCC_ERR_NOT_SUPPORTED;
        }
        if (!t->captured) CUDA_CHECK(cudaEventRecord(t->in_event, s));
        st = p2p_try_send(t, 1);
        if (st == UCC_INPROGRESS) { t->state = NVL_TASK_P2P_WAIT; st = UCC_OK; }
        return st;
    }
    if (rndv) {
        t->rz_seq = team->rz_rx[peer]++;
        ucc_tl_nvl_xb_export(team, t->u.p2p.buf, t->u.p2p.bytes, &t->rz_buf);
        if (xb_kind_mappable(t->rz_buf.kind)) {
            t->u.p2p.mode = NVL_P2P_WAIT; t->u.p2p.rz_seq = team->rz_zc_rx[peer]++;
            /* an idle stream is at the recv already: publish right away (saves one host poll of the handshake) */
            t->rz_stream_idle = cudaStreamQuery(s) == cudaSuccess;
            if (!t->rz_stream_idle) { (void)cudaGetLastError(); CUDA_CHECK(cudaEventRecord(t->in_event, s)); }
        }
        t->rz_pub_pending = 1;
        p2p_try_publish(t);
        /* the wait kernel goes into the stream only once the sender's push kernel has been LAUNCHED (p2p_try_wait, from progress):
         * a kernel that spins for an unbounded time can stall unrelated streams that share its hardware queue - among them the
         * side stream of this rank's own push, which the peer's wait kernel is waiting for.  The push never waits for anything
         * on the device, so a wait kernel enqueued after its launch spins for the duration of the transfer at most */
        if (t->u.p2p.mode == NVL_P2P_WAIT) { t->rz_wait_pending = 1; return UCC_OK; }
    }
    st = nvl_launch(t, s);
    if (st != UCC_OK) return st;
    if (!t->captured) CUDA_CHECK(cudaEventRecord(t->event, s));
    return UCC_OK;
}

/* head of the launch queue: start it once its buffer exchange (if any) is complete */
static ucc_status_t try_launch_queued(ucc_tl_nvl_task_t *t)
{
    ucc_tl_nvl_team_t *team = t->team;
    cudaStream_t s;
    ucc_status_t st;
    if (ucc_list_head(&team->launch_q, ucc_tl_nvl_task_t, q_elem) != t) return UCC_INPROGRESS;
    if (t->need_xchg) {
        if (!t->published) t->published = ucc_tl_nvl_xb_publish(team, t->cseq, t->exp_src, t->exp_src_len, t->exp_dst, t->exp_dst_len, 1, (t->kind == NVL_TASK_XCHG && t->use_push) ? t->push.recv_off : NULL);
        if (!t->published || !ucc_tl_nvl_xb_ready(team, t->cseq)) return UCC_INPROGRESS;
        st = resolve_direct(t);
        if (st != UCC_OK) { ucc_list_del(&t->q_elem); t->state = NVL_TASK_LAUNCHED; return st; }
    }
    s = t->stream;
    st = launch_ordered(t, s);
    if (st != UCC_OK) return st;
    ucc_list_del(&t->q_elem); t->state = NVL_TASK_LAUNCHED;
    if (t->super.ee) { /* stream-ordered post: only now is the collective really in the user's stream */
        ucc_ev_t post_event;
        post_event.ev_type = UCC_EVENT_COLLECTIVE_POST; post_event.ev_context = NULL; post_event.ev_context_size = 0; post_event.req = &t->super.super;
        ucc_ee_set_event_internal(t->super.ee, &post_event, &t->super.ee->event_out_queue);
    }
    return UCC_OK;
}

static void nvl_progress(ucc_coll_task_t *ct)
{
    ucc_tl_nvl_task_t *t = ucc_derived_of(ct, ucc_tl_nvl_task_t);
    cudaError_t e;
    if (t->kind == NVL_TASK_P2P && (t->rz_pub_pending || t->rz_wait_pending || t->state == NVL_TASK_P2P_WAIT)) {
        ucc_status_t st = UCC_OK;
        ucc_spin_lock(&t->team->launch_lock);
        p2p_try_publish(t);
        st = p2p_try_wait(t);
        if (st != UCC_OK) { ucc_spin_unlock(&t->team->launch_lock); ct->status = st; return; }
        if (t->state == NVL_TASK_P2P_WAIT) {
            st = p2p_try_send(t, 0);
            if (st != UCC_INPROGRESS) t->state = NVL_TASK_LAUNCHED;
        }
        ucc_spin_unlock(&t->team->launch_lock);
        if (st == UCC_INPROGRESS) return;
        if (st != UCC_OK) { ct->status = st; return; }
        /* stream-ordered post: a send is in the user's stream once launched; a receive counts as posted once its buffer is on
         * the board (until then the owner has to keep progressing, nobody else can publish it) */
        if (t->state == NVL_TASK_LAUNCHED && !t->rz_pub_pending && !t->rz_wait_pending && t->super.ee && !t->p2p_ee_done) {
            ucc_ev_t post_event;
            t->p2p_ee_done = 1;
            post_event.ev_type = UCC_EVENT_COLLECTIVE_POST; post_event.ev_context = NULL; post_event.ev_context_size = 0; post_event.req = &t->super.super;
            ucc_ee_set_event_internal(t->super.ee, &post_event, &t->super.ee->event_out_queue);
        }
    }
    if (t->kind == NVL_TASK_P2P && t->rz_wait_pending) return;   /* its event is not recorded yet */
    if (t->state == NVL_TASK_QUEUED) {
        ucc_status_t st;
        ucc_spin_lock(&t->team->launch_lock);
        st = try_launch_queued(t);
        ucc_spin_unlock(&t->team->launch_lock);
        if (st == UCC_INPROGRESS) return;
        if (st != UCC_OK) { ct->status = st; return; }
    }
    if (t->captured) { ct->status = UCC_OK; return; }
    e = cudaEventQuery(t->event);
    if (e == cudaErrorNotReady) { (void)cudaGetLastError(); return; }
    if (e != cudaSuccess) { (void)cudaGetLastError(); tl_error(NVL_LIB(t->team), "collective kernel failed: %s", cudaGetErrorString(e)); ct->status = UCC_ERR_NO_MESSAGE; return; }
    if (ucc_unlikely(*(volatile uint32_t *)t->team->host_err)) {
        tl_error(NVL_LIB(t->team), "device-side wait timed out (a peer did not arrive within TL_NVL_TIMEOUT)");
        ct->status = UCC_ERR_TIMED_OUT; return;
    }
    ct->status = UCC_OK;
}

/* A pipelined parent (cl/hier fragments) changed bargs.args since the last post (UCC_COLL_TASK_FLAG_ARGS_UPDATED).  tl/nvl tasks capture
 * buffers, counts, grids and push tables at init, so the task is rebuilt through the algorithm entry that made it and takes over the fresh
 * state; the core part (listeners, schedule links, callbacks) stays.  Sequence numbers are taken at post, never at init, so nothing is skipped. */
static ucc_status_t nvl_finalize(ucc_coll_task_t *ct);
static ucc_status_t nvl_rebuild(ucc_tl_nvl_task_t *t)
{
    const size_t off = offsetof(ucc_tl_nvl_task_t, team), len = sizeof(*t) - off;
    char tmp[sizeof(ucc_tl_nvl_task_t)];
    ucc_coll_task_t *nct = NULL;
    ucc_status_t st;
    if (!t->super.init_fn) return UCC_ERR_NOT_SUPPORTED;
    st = t->super.init_fn(&t->super.bargs, t->super.team, &nct);
    if (st != UCC_OK) return st;
    if (nct->finalize != nvl_finalize) { nct->finalize(nct); return UCC_ERR_NOT_SUPPORTED; }
    memcpy(tmp, (char *)nct + off, len); memcpy((char *)nct + off, (char *)t + off, len); memcpy((char *)t + off, tmp, len);
    t->super.flags &= ~(uint32_t)UCC_COLL_TASK_FLAG_ARGS_UPDATED;
    return nct->finalize(nct); /* releases the previous state (events go back to the cache, a lane's ordering event is kept alive) */
}

static ucc_status_t nvl_post_on(ucc_tl_nvl_task_t *t, cudaStream_t s)
{
    enum cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    ucc_status_t st;
    UCC_PROFILE_REQUEST_EVENT(t, "nvl_coll_start", 0);
    ucc_tl_nvl_team_t *team = t->team;
    int direct;
    if (ucc_unlikely(t->super.flags & UCC_COLL_TASK_FLAG_ARGS_UPDATED)) { st = nvl_rebuild(t); if (st != UCC_OK) return st; }
    t->stream = s; t->captured = 0; t->state = NVL_TASK_LAUNCHED; t->gated = 0; t->published = 0;
    if (cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive) t->captured = 1;
    ucc_spin_lock(&team->launch_lock);
    /* lanes advance in post order, which UCC requires to be the same on every member; point-to-point and single-member tasks
     * involve no team-wide kernel and take no lane */
    if (t->kind == NVL_TASK_P2P) {
        t->p2p_ee_done = 0;
        st = p2p_post(t, s);
        ucc_spin_unlock(&team->launch_lock);
        if (st != UCC_OK) return st;
        return ucc_progress_queue_enqueue(UCC_TL_CORE_CTX(t->team)->pq, &t->super);
    }
    if (t->kind != NVL_TASK_SELF_COPY) task_set_lane(t, team->lane_seq++ % team->nlanes);
    direct = task_is_direct(t) && !t->direct_cached;   /* cached tables: also fine inside a stream capture, nothing to wait for */
    t->need_xchg = direct;
    if (t->kind == NVL_TASK_XCHG || t->kind == NVL_TASK_AG_SYMM) t->u.xchg.direct = 0; else if (t->kind != NVL_TASK_P2P) t->u.red.direct = NVL_DIRECT_NONE;
    if (task_is_direct(t) && t->direct_cached) apply_cached_direct(t);
    if (direct) {
        /* the exchange sequence advances on every rank in post order; a capturing stream cannot wait for the
         * peers, so it tells them "not usable" and everybody takes the staged kernel for this one */
        t->cseq = team->xb_seq++;
        t->published = ucc_tl_nvl_xb_publish(team, t->cseq, t->exp_src, t->exp_src_len, t->exp_dst, t->exp_dst_len, !t->captured, (t->kind == NVL_TASK_XCHG && t->use_push) ? t->push.recv_off : NULL);
        if (t->captured) { direct = 0; t->need_xchg = 0; if (team->xb_mine->consumed < t->cseq + 1) ucc_store_release(&team->xb_mine->consumed, t->cseq + 1); }
    }
    if (t->captured || t->kind == NVL_TASK_P2P || (ucc_list_is_empty(&team->launch_q) && (!direct || (t->published && ucc_tl_nvl_xb_ready(team, t->cseq))))) {
        st = direct ? resolve_direct(t) : UCC_OK;
        if (st == UCC_OK) st = launch_ordered(t, s);
    } else {
        /* deferred: the kernel is launched (into the same stream) from progress once the peers' buffers are known and
         * the tasks ahead of it are launched.  As with the reference's triggered post, a stream-ordered consumer
         * learns from UCC_EVENT_COLLECTIVE_POST when the collective is really in its stream.  (Parking the user's
         * stream on a cuStreamWaitValue32 gate was tried and dropped: streams share hardware channels, so the
         * parked wait can block the very kernel that is supposed to release it.) */
        st = UCC_OK;
        ucc_list_add_tail(&team->launch_q, &t->q_elem); t->state = NVL_TASK_QUEUED;
    }
    ucc_spin_unlock(&team->launch_lock);
    if (st != UCC_OK) return st;
    return ucc_progress_queue_enqueue(UCC_TL_CORE_CTX(t->team)->pq, &t->super);
}
static ucc_status_t nvl_post(ucc_coll_task_t *ct)
{ ucc_tl_nvl_task_t *t = ucc_derived_of(ct, ucc_tl_nvl_task_t); ct->ee = NULL; return nvl_post_on(t, t->team->stream); }

/* stream-ordered post: the kernel goes straight onto the user's stream (what PyTorch-style
 * consumers use); no host-side dependency resolution is needed */
static ucc_status_t nvl_triggered_post(ucc_ee_h ee, ucc_ev_t *ev, ucc_coll_task_t *ct)
{
    ucc_tl_nvl_task_t *t = ucc_derived_of(ct, ucc_tl_nvl_task_t);
    ucc_ev_t post_event;
    ucc_status_t st;
    (void)ev;
    if (ee->ee_type != UCC_EE_CUDA_STREAM) return UCC_ERR_NOT_SUPPORTED;
    ct->ee = ee;
    st = nvl_post_on(t, (cudaStream_t)ee->ee_context);
    if (st != UCC_OK) return st;
    if (t->state == NVL_TASK_QUEUED || t->state == NVL_TASK_P2P_WAIT || (t->kind == NVL_TASK_P2P && (t->rz_pub_pending || t->rz_wait_pending))) return UCC_OK; /* the post event follows the deferred launch / publication */
    t->p2p_ee_done = 1;
    post_event.ev_type = UCC_EVENT_COLLECTIVE_POST; post_event.ev_context = NULL; post_event.ev_context_size = 0; post_event.req = &ct->super;
    ucc_ee_set_event_internal(ee, &post_event, &ee->event_out_queue);
    return UCC_OK;
}
static void event_put(ucc_tl_nvl_context_t *ctx, cudaEvent_t e);
static ucc_status_t nvl_finalize(ucc_coll_task_t *ct)
{
    ucc_tl_nvl_task_t *t = ucc_derived_of(ct, ucc_tl_nvl_task_t);
    ucc_tl_nvl_team_t *team = t->team;
    ucc_spin_lock(&team->launch_lock);
    if (t->state == NVL_TASK_QUEUED) { /* abandoned before its kernel was launched (timeout / error): release the user's stream */
        ucc_list_del(&t->q_elem); t->state = NVL_TASK_LAUNCHED;
    }
    if (t->state == NVL_TASK_P2P_WAIT) { /* a send given up before the receiver showed up: let the sends behind it proceed */
        if (t->p2p_order == team->p2p_launch_seq[t->u.p2p.peer]) team->p2p_launch_seq[t->u.p2p.peer]++;
        t->state = NVL_TASK_LAUNCHED;
    }
    if (t->event && team->last_event[t->lane] == t->event) { /* the lane still orders its next launch after this event: keep it alive */
        cudaEvent_t spare = team->order_event[t->lane]; team->order_event[t->lane] = t->event; t->event = spare;
    }
    ucc_spin_unlock(&team->launch_lock);
    if (t->in_event) { event_put(NVL_CTX(team), t->in_event); t->in_event = NULL; }
    if (t->event) event_put(NVL_CTX(team), t->event);
    ucc_coll_task_destruct(ct);
    ucc_mpool_put(t);
    return UCC_OK;
}

static cudaEvent_t event_get(ucc_tl_nvl_context_t *ctx)
{
    cudaEvent_t e = NULL;
    ucc_spin_lock(&ctx->ev_lock);
    if (ctx->n_ev_cache) e = ctx->ev_cache[--ctx->n_ev_cache];
    ucc_spin_unlock(&ctx->ev_lock);
    if (!e && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { (void)cudaGetLastError(); return NULL; }
    return e;
}
static void event_put(ucc_tl_nvl_context_t *ctx, cudaEvent_t e)
{
    ucc_spin_lock(&ctx->ev_lock);
    if (ctx->n_ev_cache < NVL_EVENT_CACHE) { ctx->ev_cache[ctx->n_ev_cache++] = e; e = NULL; }
    ucc_spin_unlock(&ctx->ev_lock);
    if (e) cudaEventDestroy(e);
}
static ucc_status_t task_alloc(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_tl_nvl_task_t **tp)
{
    ucc_tl_nvl_team_t *team = ucc_derived_of(b_team, ucc_tl_nvl_team_t);
    ucc_tl_nvl_context_t *ctx = NVL_CTX(team);
    ucc_tl_nvl_task_t *t = (ucc_tl_nvl_task_t *)ucc_mpool_get(&ctx->task_mp);
    if (!t) return UCC_ERR_NO_MEMORY;
    ucc_coll_task_init(&t->super, b, b_team);
    t->team = team; t->event = NULL; t->captured = 0; t->lane = 0; t->in_event = NULL; t->state = NVL_TASK_LAUNCHED; t->want_direct = 0; t->gated = 0; t->use_push = 0; t->use_bulk = 0; t->use_ce = 0;
    t->need_xchg = 0; t->direct_cached = 0; t->cached_mode = 0; t->need_src = t->need_dst = 0; t->exp_src = NULL; t->exp_dst = NULL; t->exp_src_len = t->exp_dst_len = 0; t->nblocks_direct = 0;
    t->nthreads = (int)ctx->cfg.nthreads;
    t->super.post = nvl_post; t->super.progress = nvl_progress; t->super.finalize = nvl_finalize; t->super.triggered_post = nvl_triggered_post;
    t->event = event_get(ctx);
    if (!t->event) { ucc_mpool_put(t); return UCC_ERR_NO_RESOURCE; }
    *tp = t;
    return UCC_OK;
}
static int pick_blocks(ucc_tl_nvl_context_t *ctx, size_t bytes, size_t bytes_per_block)
{
    size_t nb;
    if (ctx->cfg.nblocks != UCC_UUNITS_AUTO && ctx->cfg.nblocks > 0) return (int)ucc_min(ctx->cfg.nblocks, ctx->cfg.max_blocks);
    nb = (bytes + bytes_per_block - 1) / bytes_per_block;
    if (nb < 1) nb = 1;
    if (nb > ctx->cfg.max_blocks) nb = ctx->cfg.max_blocks;
    return (int)nb;
}

/* ------------------------------------------------------------------ */
/* team of one: each collective is at most one local copy (cf. reference tl/self/tl_self_coll.c:49-278, which    */
/* hands the copy to the EC executor); here it is a copy kernel on the caller's stream                          */
/* ------------------------------------------------------------------ */
static ucc_status_t self_init(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p)
{
    ucc_tl_nvl_team_t *team = ucc_derived_of(b_team, ucc_tl_nvl_team_t);
    ucc_tl_nvl_context_t *ctx = NVL_CTX(team);
    ucc_coll_args_t *a = &b->args;
    const void *src = NULL; void *dst = NULL; size_t bytes = 0;
    ucc_memory_type_t smt = UCC_MEMORY_TYPE_CUDA, dmt = UCC_MEMORY_TYPE_CUDA;
    ucc_tl_nvl_task_t *t;
    ucc_status_t st;
    if (!UCC_IS_INPLACE(*a)) {
        switch (a->coll_type) {
        case UCC_COLL_TYPE_ALLGATHER: case UCC_COLL_TYPE_ALLREDUCE: case UCC_COLL_TYPE_ALLTOALL: case UCC_COLL_TYPE_GATHER: case UCC_COLL_TYPE_REDUCE:
        case UCC_COLL_TYPE_REDUCE_SCATTER: case UCC_COLL_TYPE_SCATTER:
            src = a->src.info.buffer; dst = a->dst.info.buffer; bytes = a->dst.info.count * ucc_dt_size(a->dst.info.datatype);
            smt = a->src.info.mem_type; dmt = a->dst.info.mem_type; break;
        case UCC_COLL_TYPE_ALLGATHERV: case UCC_COLL_TYPE_GATHERV: case UCC_COLL_TYPE_REDUCE_SCATTERV:
            src = a->src.info.buffer; bytes = ucc_coll_args_get_count(a, a->dst.info_v.counts, 0) * ucc_dt_size(a->dst.info_v.datatype);
            dst = PTR_OFFSET(a->dst.info_v.buffer, (a->dst.info_v.displacements ? ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, 0) : 0) * ucc_dt_size(a->dst.info_v.datatype));
            smt = a->src.info.mem_type; dmt = a->dst.info_v.mem_type; break;
        case UCC_COLL_TYPE_ALLTOALLV:
            bytes = ucc_coll_args_get_count(a, a->src.info_v.counts, 0) * ucc_dt_size(a->src.info_v.datatype);
            src = PTR_OFFSET(a->src.info_v.buffer, ucc_coll_args_get_displacement(a, a->src.info_v.displacements, 0) * ucc_dt_size(a->src.info_v.datatype));
            dst = PTR_OFFSET(a->dst.info_v.buffer, ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, 0) * ucc_dt_size(a->dst.info_v.datatype));
            smt = a->src.info_v.mem_type; dmt = a->dst.info_v.mem_type; break;
        case UCC_COLL_TYPE_SCATTERV:
            bytes = a->dst.info.count * ucc_dt_size(a->dst.info.datatype); dst = a->dst.info.buffer;
            src = PTR_OFFSET(a->src.info_v.buffer, (a->src.info_v.displacements ? ucc_coll_args_get_displacement(a, a->src.info_v.displacements, 0) : 0) * ucc_dt_size(a->src.info_v.datatype));
            smt = a->src.info_v.mem_type; dmt = a->dst.info.mem_type; break;
        default: break; /* bcast, barrier, fanin, fanout: nothing moves */
        }
    }
    if (bytes && (!is_cuda(smt) || !is_cuda(dmt))) return UCC_ERR_NOT_SUPPORTED;
    st = task_alloc(b, b_team, &t);
    if (st != UCC_OK) return st;
    memset(&t->u.xchg, 0, sizeof(t->u.xchg));
    t->kind = NVL_TASK_SELF_COPY;
    t->u.xchg.src = src; t->u.xchg.dst = dst; t->u.xchg.src_bytes = (src && dst && src != dst) ? bytes : 0;
    t->nblocks = pick_blocks(ctx, bytes, 64 * 1024);
    /* big copies: the TMA engine streams them through shared memory - measured on a B200 at 1 GiB: 3310 GB/s with one one-warp CTA
     * on every second SM against 2930 GB/s for 256 x 512 copying threads and 3270 GB/s for cudaMemcpyAsync; below ~128 MB the
     * thread copy's faster ramp-up wins */
    if (ctx->cfg.bulk != UCC_NO && t->u.xchg.src_bytes >= ((size_t)128 << 20) && !((((uintptr_t)src) | ((uintptr_t)dst)) & 15)) {
        t->use_bulk = 1; t->nblocks = (int)ucc_max(1u, ucc_min((unsigned)ctx->sm_count / 2, ctx->cfg.max_blocks));
    }
    *task_p = &t->super;
    return UCC_OK;
}

/* ------------------------------------------------------------------ */
/* reduce family                                                       */
/* ------------------------------------------------------------------ */
typedef enum { RED_ALG_ONESHOT, RED_ALG_TWOSHOT, RED_ALG_NVLS, RED_ALG_RING, RED_ALG_RHD, RED_ALG_NVLS_PIPE } red_alg_t;

static ucc_status_t red_init(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p, red_alg_t alg)
{
    ucc_tl_nvl_team_t *team = ucc_derived_of(b_team, ucc_tl_nvl_team_t);
    ucc_tl_nvl_context_t *ctx = NVL_CTX(team);
    ucc_coll_args_t *a = &b->args;
    ucc_rank_t N = UCC_TL_TEAM_SIZE(team), me = UCC_TL_TEAM_RANK(team);
    int inplace = UCC_IS_INPLACE(*a), root = (ucc_rank_t)a->root == me;
    ucc_tl_nvl_task_t *t;
    nvl_red_args_t *r;
    ucc_datatype_t dt; ucc_memory_type_t smt, dmt;
    const void *src; void *dst; size_t count, bytes;
    int ndt, nop;
    ucc_status_t st;
    if (team->self) return self_init(b, b_team, task_p);
    switch (a->coll_type) {
    case UCC_COLL_TYPE_ALLREDUCE:
        dt = a->dst.info.datatype; count = a->dst.info.count; dst = a->dst.info.buffer; dmt = a->dst.info.mem_type;
        src = inplace ? dst : a->src.info.buffer; smt = inplace ? dmt : a->src.info.mem_type; break;
    case UCC_COLL_TYPE_REDUCE:
        if (root) { dt = a->dst.info.datatype; count = a->dst.info.count; dst = a->dst.info.buffer; dmt = a->dst.info.mem_type; src = inplace ? dst : a->src.info.buffer; smt = inplace ? dmt : a->src.info.mem_type; }
        else { dt = a->src.info.datatype; count = a->src.info.count; src = a->src.info.buffer; smt = a->src.info.mem_type; dst = NULL; dmt = smt; }
        break;
    case UCC_COLL_TYPE_REDUCE_SCATTER:
        dt = a->dst.info.datatype; dst = a->dst.info.buffer; dmt = a->dst.info.mem_type;
        count = inplace ? a->dst.info.count : a->dst.info.count * N;
        src = inplace ? dst : a->src.info.buffer; smt = inplace ? dmt : a->src.info.mem_type; break;
    case UCC_COLL_TYPE_REDUCE_SCATTERV:
        dt = a->dst.info_v.datatype; dst = a->dst.info_v.buffer; dmt = a->dst.info_v.mem_type;
        count = ucc_coll_args_get_total_count(a, a->dst.info_v.counts, N);
        src = inplace ? dst : a->src.info.buffer; smt = inplace ? dmt : a->src.info.mem_type; break;
    default: return UCC_ERR_NOT_SUPPORTED;
    }
    if (!is_cuda(smt) || !is_cuda(dmt)) return UCC_ERR_NOT_SUPPORTED;
    ndt = to_nvl_dt(dt); nop = to_nvl_op(a->op);
    if (ndt < 0 || nop < 0 || !nvl_dt_supports_op(ndt, nop)) return UCC_ERR_NOT_SUPPORTED;
    bytes = count * ucc_dt_size(dt);
    if (alg == RED_ALG_ONESHOT) {
        /* allreduce: the whole vector goes into a 1 MB slot; reduce_scatter(v): every block does (kernels/nvl_oneshot_rs.cu) */
        size_t need = bytes;
        if (a->coll_type == UCC_COLL_TYPE_REDUCE_SCATTER) need = ucc_div_round_up(count, N) * ucc_dt_size(dt);
        else if (a->coll_type == UCC_COLL_TYPE_REDUCE_SCATTERV) { need = 0; for (ucc_rank_t i = 0; i < N; i++) need = ucc_max(need, ucc_coll_args_get_count(a, a->dst.info_v.counts, i) * ucc_dt_size(dt)); }
        else if (a->coll_type != UCC_COLL_TYPE_ALLREDUCE) return UCC_ERR_NOT_SUPPORTED;
        if (need > NVL_LL_MAX) return UCC_ERR_NOT_SUPPORTED;
    }
    if ((alg == RED_ALG_NVLS || alg == RED_ALG_NVLS_PIPE) && (!team->nvls || !nvl_nvls_supports(ndt, nop))) return UCC_ERR_NOT_SUPPORTED;
    if (alg == RED_ALG_NVLS_PIPE && a->coll_type != UCC_COLL_TYPE_ALLREDUCE) return UCC_ERR_NOT_SUPPORTED;
    if (alg == RED_ALG_RING || alg == RED_ALG_RHD) {
        /* step-structured kernels: allreduce / reduce_scatter(v) whose slices fit one heap round; rhd pairs ranks by xor */
        size_t slice_cap = (ctx->cfg.symmetric_size / N / 16) * 16, need;
        if (a->coll_type == UCC_COLL_TYPE_REDUCE || (alg == RED_ALG_RHD && !ucc_is_pow2(N))) return UCC_ERR_NOT_SUPPORTED;
        if (a->coll_type == UCC_COLL_TYPE_REDUCE_SCATTERV) { need = 0; for (ucc_rank_t i = 0; i < N; i++) need = ucc_max(need, ucc_coll_args_get_count(a, a->dst.info_v.counts, i) * ucc_dt_size(dt)); }
        else need = ucc_div_round_up(count, N) * ucc_dt_size(dt);
        if (ucc_align_up(need, 16) > slice_cap) return UCC_ERR_NOT_SUPPORTED;
    }
    st = task_alloc(b, b_team, &t);
    if (st != UCC_OK) return st;
    r = &t->u.red;
    memset(r, 0, sizeof(*r));
    r->team = team->dev; r->src = src; r->dst = dst; r->count = count; r->dt = ndt; r->op = nop; r->root = (int)a->root; r->use_nvls = (alg == RED_ALG_NVLS || alg == RED_ALG_NVLS_PIPE);
    switch (a->coll_type) {
    case UCC_COLL_TYPE_ALLREDUCE: r->kind = NVL_RED_ALLREDUCE; break;
    case UCC_COLL_TYPE_REDUCE: r->kind = NVL_RED_REDUCE; break;
    default:
        r->kind = NVL_RED_REDUCE_SCATTER;
        { size_t off = 0;
          for (ucc_rank_t i = 0; i < N; i++) {
              size_t c = a->coll_type == UCC_COLL_TYPE_REDUCE_SCATTERV ? ucc_coll_args_get_count(a, a->dst.info_v.counts, i) : ucc_buffer_block_count(count, N, i);
              r->rs_offset[i] = off; r->rs_count[i] = c; off += c;
          }
          /* in-place: the result block stays at its offset inside the buffer */
          if (inplace) r->dst = (char *)dst + r->rs_offset[me] * ucc_dt_size(dt); }
        break;
    }
    if (alg == RED_ALG_ONESHOT) { t->kind = NVL_TASK_REDUCE_ONESHOT; t->nblocks = pick_blocks(ctx, bytes, 16384); if (t->nblocks > 64) t->nblocks = 64; }
    else if (alg == RED_ALG_RING || alg == RED_ALG_RHD) { t->kind = NVL_TASK_REDUCE_STEPS; r->sched = alg == RED_ALG_RING ? 1 : 2; t->nblocks = pick_blocks(ctx, bytes, 64 * 1024); }
    else if (alg == RED_ALG_NVLS_PIPE) { t->kind = NVL_TASK_REDUCE_PIPE; t->nblocks = pick_blocks(ctx, bytes, 32 * 1024); }
    else { t->kind = NVL_TASK_REDUCE_STAGED; t->nblocks = pick_blocks(ctx, bytes, 32 * 1024); }
    /* symmetric user memory (UCC_TL_NVL_USER_SIZE): src and dst sit in the multicast-bound user region of the heap, at the same
     * offset on every member by contract -> reduce in place through the switch, nothing staged, nothing exchanged */
    if ((alg == RED_ALG_TWOSHOT || alg == RED_ALG_NVLS) && r->kind == NVL_RED_ALLREDUCE && team->nvls && ctx->cfg.user_size && nvl_nvls_supports(ndt, nop)) {
        const char *ub = team->heap + team->lane_stride * team->nlanes, *ue = ub + ctx->cfg.user_size;
        const char *s0 = (const char *)src, *d0 = (const char *)dst;
        if (s0 >= ub && s0 + ucc_align_up(bytes, 16) <= ue && d0 >= ub && d0 + bytes <= ue && !(((uintptr_t)s0 | (uintptr_t)d0) & 15)) {
            t->kind = NVL_TASK_REDUCE_SYMM; r->d.src[0] = s0; r->d.dst[0] = (char *)dst; r->use_nvls = 1;
            t->nblocks = pick_blocks(ctx, bytes, 32 * 1024);
            /* nothing is staged here, every thread only issues multimem.ld_reduce / multimem.st: the switch is saturated by few CTAs
             * and slowed down by many (8 x B200, 1 GiB: 32 CTAs 839 GB/s, 64: 837, 256: 705; 64 MB: 700 / 669 / 562 -
             * profiles/r2_n8/matrix.jsonl) */
            if (N > 4 && t->nblocks > 32) t->nblocks = 32;
            *task_p = &t->super;
            return UCC_OK;
        }
    }
    /* reduce_scatter(v) out of a symmetric source (the FSDP / ZeRO gradient shape): every block is reduced in the switch
     * straight into its owner's destination, which may be any local buffer */
    if ((alg == RED_ALG_TWOSHOT || alg == RED_ALG_NVLS) && r->kind == NVL_RED_REDUCE_SCATTER && !inplace && team->nvls && ctx->cfg.user_size && nvl_nvls_supports(ndt, nop)) {
        const char *ub = team->heap + team->lane_stride * team->nlanes, *ue = ub + ctx->cfg.user_size;
        const char *s0 = (const char *)src;
        int aligned = !((uintptr_t)s0 & 15);
        for (ucc_rank_t i = 0; i < N; i++) if ((r->rs_offset[i] * ucc_dt_size(dt)) & 15) aligned = 0;
        if (aligned && s0 >= ub && s0 + ucc_align_up(bytes, 16) <= ue) {
            t->kind = NVL_TASK_REDUCE_SYMM; r->d.src[0] = s0; r->d.dst[0] = NULL; r->use_nvls = 1;
            t->nblocks = pick_blocks(ctx, bytes / N, 32 * 1024);
            *task_p = &t->super;
            return UCC_OK;
        }
    }
    /* zero-copy: every criterion below is evaluated identically on all ranks (sizes / counts are collective
     * arguments); what only the owner knows (can the buffer be exported? is it aligned?) travels with the exchange */
    if ((alg == RED_ALG_TWOSHOT || alg == RED_ALG_NVLS) && team->zcopy && ctx->cfg.zcopy != UCC_NO && bytes >= ctx->cfg.zcopy_thresh) {
        /* the NVLS kernels stay staged: writing the result to N mapped destinations instead of one multicast store was
         * tried (NVL_DIRECT_DST) and measured slower on 8 GPUs - it multiplies the bytes leaving each GPU by 1.75 */
        int mode = alg == RED_ALG_NVLS ? NVL_DIRECT_NONE : NVL_DIRECT_FULL;
        if (mode == NVL_DIRECT_FULL && r->kind == NVL_RED_REDUCE_SCATTER)
            for (ucc_rank_t i = 0; i < N; i++) if ((r->rs_offset[i] * ucc_dt_size(dt)) & 15) mode = NVL_DIRECT_NONE;
        if (mode != NVL_DIRECT_NONE) {
            t->want_direct = mode; t->nblocks_direct = t->nblocks;
            t->need_src = mode == NVL_DIRECT_FULL; t->need_dst = r->kind != NVL_RED_REDUCE_SCATTER;
            t->exp_src = src; t->exp_src_len = bytes;
            t->exp_dst = r->kind == NVL_RED_REDUCE_SCATTER ? NULL : dst; t->exp_dst_len = t->exp_dst ? bytes : 0;
        }
    }
    /* registered buffers make the in-place kernel available without the exchange board (also when it could not be set up) */
    if ((alg == RED_ALG_TWOSHOT) && !t->want_direct && ctx->cfg.zcopy != UCC_NO && bytes >= ctx->cfg.zcopy_thresh && (a->mask & (UCC_COLL_ARGS_FIELD_MEM_MAP_SRC_MEMH | UCC_COLL_ARGS_FIELD_MEM_MAP_DST_MEMH))) {
        int mode = NVL_DIRECT_FULL;
        if (r->kind == NVL_RED_REDUCE_SCATTER) for (ucc_rank_t i = 0; i < N; i++) if ((r->rs_offset[i] * ucc_dt_size(dt)) & 15) mode = NVL_DIRECT_NONE;
        if (mode) { t->want_direct = mode; t->nblocks_direct = t->nblocks; t->need_src = 1; t->need_dst = r->kind != NVL_RED_REDUCE_SCATTER; t->exp_src = src; t->exp_src_len = bytes;
                    t->exp_dst = r->kind == NVL_RED_REDUCE_SCATTER ? NULL : dst; t->exp_dst_len = t->exp_dst ? bytes : 0; }
    }
    if (t->want_direct && r->kind != NVL_RED_REDUCE) memh_direct(t, a, src, dst);
    if (t->want_direct && !t->direct_cached && !team->zcopy) t->want_direct = 0;
    *task_p = &t->super;
    return UCC_OK;
}
static ucc_status_t red_init_oneshot(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return red_init(b, t, p, RED_ALG_ONESHOT); }
static ucc_status_t red_init_twoshot(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return red_init(b, t, p, RED_ALG_TWOSHOT); }
static ucc_status_t red_init_nvls(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return red_init(b, t, p, RED_ALG_NVLS); }
static ucc_status_t red_init_ring(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return red_init(b, t, p, RED_ALG_RING); }
static ucc_status_t red_init_rhd(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return red_init(b, t, p, RED_ALG_RHD); }
static ucc_status_t red_init_nvls_pipe(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return red_init(b, t, p, RED_ALG_NVLS_PIPE); }

/* ------------------------------------------------------------------ */
/* data movement family                                                */
/* ------------------------------------------------------------------ */
static ucc_status_t xchg_init(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p)
{
    ucc_tl_nvl_team_t *team = ucc_derived_of(b_team, ucc_tl_nvl_team_t);
    ucc_tl_nvl_context_t *ctx = NVL_CTX(team);
    ucc_coll_args_t *a = &b->args;
    ucc_rank_t N = UCC_TL_TEAM_SIZE(team), me = UCC_TL_TEAM_RANK(team);
    int inplace = UCC_IS_INPLACE(*a), is_root = (ucc_rank_t)a->root == me;
    size_t cap = ctx->cfg.symmetric_size > NVL_XCHG_TABLE_BYTES ? ctx->cfg.symmetric_size - NVL_XCHG_TABLE_BYTES : 0;
    nvl_xchg_args_t x;
    ucc_tl_nvl_task_t *t;
    size_t moved = 0, dts;
    ucc_status_t st;
    if (team->self) return self_init(b, b_team, task_p);
    memset(&x, 0, sizeof(x));
    x.team = team->dev;
    if (UCC_COLL_ARGS_ACTIVE_SET(a)) {
        /* two-member active set = send / recv (reference tl_cuda_coll.h:156-166 supports exactly this shape): one kernel per
         * side over the pair's heap channel.  Messages between an ordered pair are matched in post order; the tag is not
         * needed for that and larger active sets go to the next TL */
        ucc_rank_t r0 = (ucc_rank_t)a->active_set.start, r1 = (ucc_rank_t)(a->active_set.start + a->active_set.stride), root = (ucc_rank_t)a->root;
        size_t len = a->src.info.count * ucc_dt_size(a->src.info.datatype);
        if (a->coll_type != UCC_COLL_TYPE_BCAST || a->active_set.size != 2 || !is_cuda(a->src.info.mem_type)) return UCC_ERR_NOT_SUPPORTED;
        if ((me != r0 && me != r1) || (root != r0 && root != r1) || r0 >= N || r1 >= N || r0 == r1) return UCC_ERR_NOT_SUPPORTED;
        st = task_alloc(b, b_team, &t);
        if (st != UCC_OK) return st;
        t->kind = NVL_TASK_P2P;
        memset(&t->u.p2p, 0, sizeof(t->u.p2p));
        t->u.p2p.team = team->dev; t->u.p2p.buf = a->src.info.buffer; t->u.p2p.bytes = len;
        t->u.p2p.send = me == root; t->u.p2p.peer = (int)(me == r0 ? r1 : r0);
        t->nblocks = nvl_p2p_lanes(len);
        t->p2p_rndv = team->zcopy && len && len >= ctx->cfg.p2p_rndv_thresh;
        t->u.p2p.spin_ns = (uint64_t)(ctx->cfg.p2p_timeout * 1e9);
        *task_p = &t->super;
        return UCC_OK;
    }
    switch (a->coll_type) {
    case UCC_COLL_TYPE_ALLGATHER: {
        size_t blk = a->dst.info.count / N * ucc_dt_size(a->dst.info.datatype);
        if (!is_cuda(a->dst.info.mem_type) || (!inplace && !is_cuda(a->src.info.mem_type))) return UCC_ERR_NOT_SUPPORTED;
        x.dst = a->dst.info.buffer; x.src = inplace ? (char *)x.dst + me * blk : a->src.info.buffer; x.src_bytes = blk;
        for (ucc_rank_t p = 0; p < N; p++) { x.pull_off[p] = 0; x.pull_bytes[p] = blk; x.dst_off[p] = p * blk; }
        /* destination in the symmetric user region (same offset on every member by contract): multicast my block straight
         * into everybody's dst - nothing staged, pulled or copied out */
        if (team->nvls && ctx->cfg.user_size && blk && !(blk & 15) && !(((uintptr_t)x.src | (uintptr_t)x.dst) & 15)) {
            const char *ub = team->heap + team->lane_stride * team->nlanes, *ue = ub + ctx->cfg.user_size, *d0 = (const char *)x.dst;
            if (d0 >= ub && d0 + blk * N <= ue) {
                st = task_alloc(b, b_team, &t);
                if (st != UCC_OK) return st;
                x.push_off = (size_t)me * blk;
                t->kind = NVL_TASK_AG_SYMM; t->u.xchg = x;
                t->nblocks = pick_blocks(ctx, blk, 32 * 1024);
                *task_p = &t->super;
                return UCC_OK;
            }
        }
        moved = blk * N; break; }
    case UCC_COLL_TYPE_ALLGATHERV: {
        dts = ucc_dt_size(a->dst.info_v.datatype);
        if (!is_cuda(a->dst.info_v.mem_type) || (!inplace && !is_cuda(a->src.info.mem_type))) return UCC_ERR_NOT_SUPPORTED;
        x.dst = a->dst.info_v.buffer;
        for (ucc_rank_t p = 0; p < N; p++) { x.pull_off[p] = 0; x.pull_bytes[p] = ucc_coll_args_get_count(a, a->dst.info_v.counts, p) * dts; x.dst_off[p] = ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, p) * dts; moved += x.pull_bytes[p]; }
        x.src = inplace ? (char *)x.dst + x.dst_off[me] : a->src.info.buffer; x.src_bytes = x.pull_bytes[me];
        break; }
    case UCC_COLL_TYPE_ALLTOALL: {
        size_t blk = a->dst.info.count / N * ucc_dt_size(a->dst.info.datatype);
        if (inplace) return UCC_ERR_NOT_SUPPORTED; /* would need a full private copy: leave to the fallback TL */
        if (!is_cuda(a->dst.info.mem_type) || !is_cuda(a->src.info.mem_type)) return UCC_ERR_NOT_SUPPORTED;
        x.dst = a->dst.info.buffer; x.src = a->src.info.buffer; x.src_bytes = blk * N; x.self_off = me * blk;
        for (ucc_rank_t p = 0; p < N; p++) { x.pull_off[p] = me * blk; x.pull_bytes[p] = blk; x.dst_off[p] = p * blk; }
        moved = blk * N; break; }
    case UCC_COLL_TYPE_ALLTOALLV: {
        size_t sdt = ucc_dt_size(a->src.info_v.datatype), ddt = ucc_dt_size(a->dst.info_v.datatype), end = 0;
        if (inplace) return UCC_ERR_NOT_SUPPORTED;
        if (!is_cuda(a->dst.info_v.mem_type) || !is_cuda(a->src.info_v.mem_type)) return UCC_ERR_NOT_SUPPORTED;
        x.dst = a->dst.info_v.buffer; x.src = a->src.info_v.buffer; x.publish_table = 1;
        for (ucc_rank_t p = 0; p < N; p++) {
            size_t so = ucc_coll_args_get_displacement(a, a->src.info_v.displacements, p) * sdt, sc = ucc_coll_args_get_count(a, a->src.info_v.counts, p) * sdt;
            x.stage_off[p] = so; if (so + sc > end) end = so + sc;
            x.pull_off[p] = NVL_XCHG_LOOKUP; x.pull_bytes[p] = ucc_coll_args_get_count(a, a->dst.info_v.counts, p) * ddt;
            x.dst_off[p] = ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, p) * ddt; moved += x.pull_bytes[p];
        }
        x.src_bytes = end; x.self_off = x.stage_off[me];
        break; }
    case UCC_COLL_TYPE_BCAST: {
        size_t len = a->src.info.count * ucc_dt_size(a->src.info.datatype);
        if (!is_cuda(a->src.info.mem_type)) return UCC_ERR_NOT_SUPPORTED;
        x.dst = a->src.info.buffer; x.src = a->src.info.buffer; x.src_bytes = is_root ? len : 0;
        if (!is_root) { x.pull_off[a->root] = 0; x.pull_bytes[a->root] = len; x.dst_off[a->root] = 0; }
        moved = len; break; }
    case UCC_COLL_TYPE_GATHER: {
        size_t blk = is_root ? a->dst.info.count / N * ucc_dt_size(a->dst.info.datatype) : a->src.info.count * ucc_dt_size(a->src.info.datatype);
        if (is_root ? !is_cuda(a->dst.info.mem_type) || (!inplace && !is_cuda(a->src.info.mem_type)) : !is_cuda(a->src.info.mem_type)) return UCC_ERR_NOT_SUPPORTED;
        if (is_root) {
            x.dst = a->dst.info.buffer; x.src = inplace ? (char *)x.dst + me * blk : a->src.info.buffer;
            for (ucc_rank_t p = 0; p < N; p++) { x.pull_off[p] = 0; x.pull_bytes[p] = blk; x.dst_off[p] = p * blk; }
        } else { x.src = a->src.info.buffer; x.src_bytes = blk; }
        moved = blk * N; break; }
    case UCC_COLL_TYPE_GATHERV: {
        if (is_root ? !is_cuda(a->dst.info_v.mem_type) || (!inplace && !is_cuda(a->src.info.mem_type)) : !is_cuda(a->src.info.mem_type)) return UCC_ERR_NOT_SUPPORTED;
        if (is_root) {
            dts = ucc_dt_size(a->dst.info_v.datatype); x.dst = a->dst.info_v.buffer;
            for (ucc_rank_t p = 0; p < N; p++) { x.pull_off[p] = 0; x.pull_bytes[p] = ucc_coll_args_get_count(a, a->dst.info_v.counts, p) * dts; x.dst_off[p] = ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, p) * dts; moved += x.pull_bytes[p]; }
            x.src = inplace ? (char *)x.dst + x.dst_off[me] : a->src.info.buffer;
        } else { x.src = a->src.info.buffer; x.src_bytes = a->src.info.count * ucc_dt_size(a->src.info.datatype); moved = x.src_bytes * N; }
        break; }
    case UCC_COLL_TYPE_SCATTER: {
        size_t blk = is_root ? a->src.info.count / N * ucc_dt_size(a->src.info.datatype) : a->dst.info.count * ucc_dt_size(a->dst.info.datatype);
        if (is_root ? !is_cuda(a->src.info.mem_type) || (!inplace && !is_cuda(a->dst.info.mem_type)) : !is_cuda(a->dst.info.mem_type)) return UCC_ERR_NOT_SUPPORTED;
        if (is_root) { x.src = a->src.info.buffer; x.src_bytes = blk * N; x.self_off = me * blk; if (!inplace) { x.dst = a->dst.info.buffer; x.pull_bytes[me] = blk; x.dst_off[me] = 0; } }
        else { x.dst = a->dst.info.buffer; x.pull_off[a->root] = me * blk; x.pull_bytes[a->root] = blk; x.dst_off[a->root] = 0; }
        moved = blk * N; break; }
    case UCC_COLL_TYPE_SCATTERV: {
        if (is_root ? !is_cuda(a->src.info_v.mem_type) || (!inplace && !is_cuda(a->dst.info.mem_type)) : !is_cuda(a->dst.info.mem_type)) return UCC_ERR_NOT_SUPPORTED;
        if (is_root) {
            size_t end = 0; dts = ucc_dt_size(a->src.info_v.datatype);
            x.src = a->src.info_v.buffer; x.publish_table = 1;
            for (ucc_rank_t p = 0; p < N; p++) { size_t so = ucc_coll_args_get_displacement(a, a->src.info_v.displacements, p) * dts, sc = ucc_coll_args_get_count(a, a->src.info_v.counts, p) * dts; x.stage_off[p] = so; if (so + sc > end) end = so + sc; }
            x.src_bytes = end; x.self_off = x.stage_off[me]; moved = end;
            if (!inplace) { x.dst = a->dst.info.buffer; x.pull_bytes[me] = ucc_coll_args_get_count(a, a->src.info_v.counts, me) * dts; x.dst_off[me] = 0; }
        } else { x.dst = a->dst.info.buffer; x.pull_off[a->root] = NVL_XCHG_LOOKUP; x.pull_bytes[a->root] = a->dst.info.count * ucc_dt_size(a->dst.info.datatype); x.dst_off[a->root] = 0; moved = x.pull_bytes[a->root] * N; }
        break; }
    default: return UCC_ERR_NOT_SUPPORTED;
    }
    /* the staged payload must fit the heap (every rank evaluates the same bound for symmetric colls;
     * v-variants that exceed it are rejected on the ranks that notice -> use a size hint via TUNE to avoid) */
    if (x.src_bytes > cap) return UCC_ERR_NOT_SUPPORTED;
    st = task_alloc(b, b_team, &t);
    if (st != UCC_OK) return st;
    t->kind = NVL_TASK_XCHG; t->u.xchg = x;
    t->nblocks = pick_blocks(ctx, moved, 64 * 1024);
    /* the grid must be the same on every rank (blocks pair up through per-block flags), but for alltoallv / gatherv /
     * scatterv `moved` is private to a rank: use a fixed grid for those */
    if (a->coll_type == UCC_COLL_TYPE_ALLTOALLV || a->coll_type == UCC_COLL_TYPE_GATHERV || a->coll_type == UCC_COLL_TYPE_SCATTERV)
        t->nblocks = (int)ucc_min(ctx->cfg.max_blocks, (ctx->cfg.nblocks != UCC_UUNITS_AUTO && ctx->cfg.nblocks > 0) ? ctx->cfg.nblocks : 128u);
    if (team->zcopy && ctx->cfg.zcopy != UCC_NO) {
        /* `moved` is the same number on every rank except for the v-collectives whose counts are private to a
         * rank (alltoallv, gatherv, scatterv): those only go zero-copy when it is forced, size-independently */
        int symmetric = a->coll_type != UCC_COLL_TYPE_ALLTOALLV && a->coll_type != UCC_COLL_TYPE_GATHERV && a->coll_type != UCC_COLL_TYPE_SCATTERV;
        /* (asymmetric ones: always - the choice may only depend on what every rank knows, and staging a skewed
         * alltoallv through the heap was 2.4x slower than NCCL at 16 MB on 4 GPUs) */
        if (symmetric ? moved >= (ctx->cfg.zcopy == UCC_YES ? ctx->cfg.zcopy_thresh : ucc_max(ctx->cfg.zcopy_thresh, (size_t)4 << 20)) : 1) { /* below ~4 MB the host-side exchange costs more than the staging copy */
            t->want_direct = NVL_DIRECT_FULL; t->need_src = 1; t->need_dst = 0;
            t->exp_src = x.src_bytes ? x.src : NULL; t->exp_src_len = x.src_bytes;
        }
    }
    *task_p = &t->super;
    return UCC_OK;
}

/* zero-copy PUSH allgather(v) / alltoall (kernels/nvl_push.cu): the destinations travel over the exchange board and every rank
 * stores its blocks straight into them; if a destination cannot be mapped the task falls back to the staged pull it also is */
static ucc_status_t xchg_init_push(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p)
{
    ucc_tl_nvl_team_t *team = ucc_derived_of(b_team, ucc_tl_nvl_team_t);
    ucc_tl_nvl_context_t *ctx = NVL_CTX(team);
    ucc_coll_args_t *a = &b->args;
    ucc_rank_t N = UCC_TL_TEAM_SIZE(team), me = UCC_TL_TEAM_RANK(team);
    ucc_coll_type_t ct = a->coll_type;
    ucc_tl_nvl_task_t *t;
    nvl_xchg_args_t *x;
    size_t dst_len = 0;
    ucc_status_t st;
    if (ct != UCC_COLL_TYPE_ALLGATHER && ct != UCC_COLL_TYPE_ALLGATHERV && ct != UCC_COLL_TYPE_ALLTOALL && ct != UCC_COLL_TYPE_ALLTOALLV) return UCC_ERR_NOT_SUPPORTED;
    if (!team->self && (!team->zcopy || ctx->cfg.zcopy == UCC_NO)) return UCC_ERR_NOT_SUPPORTED;
    if (ct == UCC_COLL_TYPE_ALLTOALL && UCC_IS_INPLACE(*a)) return UCC_ERR_NOT_SUPPORTED;
    st = xchg_init(b, b_team, task_p);
    if (st != UCC_OK) return st;
    t = ucc_derived_of(*task_p, ucc_tl_nvl_task_t); x = &t->u.xchg;
    if (t->kind != NVL_TASK_XCHG) return UCC_OK; /* symmetric destination / single member: nothing to add */
    t->push.lookup = 0;
    for (ucc_rank_t p = 0; p < N; p++) {
        t->push.recv_off[p] = x->dst_off[p];
        if (ct == UCC_COLL_TYPE_ALLTOALLV) {
            /* what I send is described by MY send counts / displacements (x->stage_off); where it lands only the receiver knows:
             * it publishes recv_off[] on the device and the senders look their entry up (the mirror image of the pull kernel's table) */
            size_t sdt = ucc_dt_size(a->src.info_v.datatype);
            t->push.send_off[p] = x->stage_off[p]; t->push.send_bytes[p] = ucc_coll_args_get_count(a, a->src.info_v.counts, p) * sdt;
            t->push.land_off[p] = x->dst_off[me]; t->push.lookup = 1;
        } else if (ct == UCC_COLL_TYPE_ALLTOALL) { t->push.send_off[p] = x->dst_off[p]; t->push.send_bytes[p] = x->pull_bytes[p]; t->push.land_off[p] = x->dst_off[me]; }
        else { t->push.send_off[p] = 0; t->push.send_bytes[p] = x->pull_bytes[me]; t->push.land_off[p] = x->dst_off[me]; } /* my block, at my displacement, in everybody's dst */
        if (x->dst_off[p] + x->pull_bytes[p] > dst_len) dst_len = x->dst_off[p] + x->pull_bytes[p];
    }
    /* alltoallv: one landing-offset table per block at the start of the data region */
    if (t->push.lookup && (size_t)t->nblocks * NVL_MAX_PEERS * sizeof(uint64_t) > ctx->cfg.symmetric_size) { (*task_p)->finalize(*task_p); *task_p = NULL; return UCC_ERR_NOT_SUPPORTED; }
    t->use_push = 1;
    /* data mover: the TMA engine for big transfers (the choice may only depend on what every member knows - sizes of the
     * v-collectives are private, those always take it) */
    { size_t total = 0; int symmetric = ct == UCC_COLL_TYPE_ALLGATHER || ct == UCC_COLL_TYPE_ALLTOALL || ct == UCC_COLL_TYPE_ALLGATHERV;
      for (ucc_rank_t p = 0; p < N; p++) total += x->pull_bytes[p];
      t->use_bulk = ctx->cfg.bulk != UCC_NO && (symmetric ? total >= ctx->cfg.bulk_thresh : 1);
      if (t->use_bulk) t->nblocks = (int)ucc_max(1u, ucc_min(ctx->cfg.bulk_ctas, ctx->cfg.max_blocks)); }
    t->want_direct = NVL_DIRECT_FULL; t->need_src = 0; t->need_dst = 1;
    t->exp_src = NULL; t->exp_src_len = 0; t->exp_dst = x->dst; t->exp_dst_len = dst_len;
    return UCC_OK;
}

/* copy-engine push exchange: same buffer resolution as `push`, the copies are DMAs issued by the host (see nvl_launch) */
static ucc_status_t xchg_init_ce(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p)
{
    ucc_tl_nvl_task_t *t;
    ucc_status_t st = xchg_init_push(b, b_team, task_p);
    if (st != UCC_OK) return st;
    t = ucc_derived_of(*task_p, ucc_tl_nvl_task_t);
    if (t->kind != NVL_TASK_XCHG) return UCC_OK;
    t->use_ce = 1; t->use_bulk = 0; t->nblocks = 1;
    return UCC_OK;
}

/* allgather(v) / bcast through the switch: every rank multicasts its block once (multimem.st), everybody then
 * copies out of its OWN heap.  Same bytes into every GPU as the pull variant, 1/(N-1) of the bytes out. */
static ucc_status_t xchg_init_nvls(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p)
{
    ucc_tl_nvl_team_t *team = ucc_derived_of(b_team, ucc_tl_nvl_team_t);
    ucc_tl_nvl_context_t *ctx = NVL_CTX(team);
    ucc_rank_t N = UCC_TL_TEAM_SIZE(team), me = UCC_TL_TEAM_RANK(team);
    ucc_coll_type_t ct = b->args.coll_type;
    size_t cap = ctx->cfg.symmetric_size > NVL_XCHG_TABLE_BYTES ? ctx->cfg.symmetric_size - NVL_XCHG_TABLE_BYTES : 0, off = 0;
    ucc_tl_nvl_task_t *t;
    nvl_xchg_args_t *x;
    ucc_status_t st;
    if (!team->nvls || (ct != UCC_COLL_TYPE_ALLGATHER && ct != UCC_COLL_TYPE_ALLGATHERV && ct != UCC_COLL_TYPE_BCAST)) return UCC_ERR_NOT_SUPPORTED;
    st = xchg_init(b, b_team, task_p);
    if (st != UCC_OK) return st;
    t = ucc_derived_of(*task_p, ucc_tl_nvl_task_t); x = &t->u.xchg;
    if (t->kind != NVL_TASK_XCHG) return UCC_OK; /* symmetric-destination allgather or single-member copy: already complete */
    t->want_direct = 0;
    if (ct == UCC_COLL_TYPE_BCAST) { x->push_off = 0; off = x->src_bytes; }
    else for (ucc_rank_t p = 0; p < N; p++) { if (p == me) x->push_off = off; x->pull_off[p] = off; off += ucc_align_up(x->pull_bytes[p] ? x->pull_bytes[p] : (p == me ? x->src_bytes : 0), 16); }
    /* NOTE for allgatherv every rank knows all counts, so `off` (and the decisions below) agree everywhere */
    if (off > cap) { (*task_p)->finalize(*task_p); *task_p = NULL; return UCC_ERR_NOT_SUPPORTED; }
    x->use_mc = 1;
    return UCC_OK;
}
/* ring allgather(v): same heap layout as the nvls variant, N-1 neighbour-to-neighbour steps inside one kernel */
static ucc_status_t xchg_init_ring(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p)
{
    ucc_tl_nvl_team_t *team = ucc_derived_of(b_team, ucc_tl_nvl_team_t);
    ucc_tl_nvl_context_t *ctx = NVL_CTX(team);
    ucc_rank_t N = UCC_TL_TEAM_SIZE(team);
    size_t cap = ctx->cfg.symmetric_size > NVL_XCHG_TABLE_BYTES ? ctx->cfg.symmetric_size - NVL_XCHG_TABLE_BYTES : 0, off = 0;
    ucc_tl_nvl_task_t *t; nvl_xchg_args_t *x; ucc_status_t st;
    if (b->args.coll_type != UCC_COLL_TYPE_ALLGATHER && b->args.coll_type != UCC_COLL_TYPE_ALLGATHERV) return UCC_ERR_NOT_SUPPORTED;
    st = xchg_init(b, b_team, task_p);
    if (st != UCC_OK) return st;
    t = ucc_derived_of(*task_p, ucc_tl_nvl_task_t); x = &t->u.xchg;
    if (t->kind != NVL_TASK_XCHG) return UCC_OK; /* symmetric-destination allgather or single-member copy: already complete */
    t->want_direct = 0;
    for (ucc_rank_t p = 0; p < N; p++) { x->pull_off[p] = off; off += ucc_align_up(x->pull_bytes[p], 16); }
    if (off > cap) { (*task_p)->finalize(*task_p); *task_p = NULL; return UCC_ERR_NOT_SUPPORTED; }
    x->ring = 1;
    for (ucc_rank_t p = 0; p < N; p++) { x->ring_order[p] = (int)team->ring_order[p]; if (team->ring_order[p] == UCC_TL_TEAM_RANK(team)) x->ring_pos = (int)p; }
    return UCC_OK;
}

static ucc_status_t barrier_init(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p)
{
    ucc_tl_nvl_task_t *t;
    ucc_status_t st;
    if (ucc_derived_of(b_team, ucc_tl_nvl_team_t)->self) return self_init(b, b_team, task_p);
    st = task_alloc(b, b_team, &t);
    if (st != UCC_OK) return st;
    t->kind = NVL_TASK_BARRIER; t->nblocks = 1;
    memset(&t->u.red, 0, sizeof(t->u.red)); t->u.red.team = ucc_derived_of(b_team, ucc_tl_nvl_team_t)->dev;
    *task_p = &t->super;
    return UCC_OK;
}

/* ------------------------------------------------------------------ */
/* algorithm table / scores                                            */
/* ------------------------------------------------------------------ */
typedef struct nvl_alg { const char *name; const char *desc; ucc_base_coll_init_fn_t init; } nvl_alg_t;
static const nvl_alg_t algs_allreduce[] = {
    {"twoshot", "stage + pull-reduce own slice over NVLink + push result to every peer, one kernel", red_init_twoshot},
    {"oneshot", "push the whole vector to every peer and reduce locally (latency path, <= 64K)", red_init_oneshot},
    {"nvls", "stage + multimem.ld_reduce / multimem.st through the NVSwitch (in-switch reduction)", red_init_nvls},
    {"ring", "ring reduce-scatter + ring allgather through the heaps, neighbour links only, one kernel", red_init_ring},
    {"rhd", "recursive halving + recursive doubling (radix-2 scatter-reduce-allgather), power-of-two teams, one kernel", red_init_rhd},
    {"nvls_pipe", "nvls with three heap buffers: staging, in-switch reduction and copy-out of consecutive chunks overlap (opt-in, not yet measured)", red_init_nvls_pipe}, {NULL}};
static const nvl_alg_t algs_rs[] = {
    {"twoshot", "stage + pull-reduce own slice over NVLink", red_init_twoshot},
    {"nvls", "stage + multimem.ld_reduce own slice in the NVSwitch", red_init_nvls},
    {"ring", "ring reduce-scatter through the heaps, neighbour links only", red_init_ring},
    {"rhd", "recursive halving, power-of-two teams", red_init_rhd},
    {"oneshot", "push every block to its owner and reduce locally: one flag exchange (latency path, blocks <= 1 MB; opt-in, not yet measured)", red_init_oneshot}, {NULL}};
static const nvl_alg_t algs_red[] = {
    {"twoshot", "stage + pull-reduce own slice over NVLink", red_init_twoshot},
    {"nvls", "stage + multimem.ld_reduce own slice in the NVSwitch", red_init_nvls}, {NULL}};
static const nvl_alg_t algs_xchg[] = {{"pull", "stage once, every peer pulls its part over NVLink", xchg_init}, {NULL}};
static const nvl_alg_t algs_xchg_mc[] = {{"pull", "stage once, every peer pulls its part over NVLink", xchg_init},
    {"nvls", "multicast the own block into every member's heap with multimem.st, copy out locally", xchg_init_nvls}, {NULL}};
static const nvl_alg_t algs_ag[] = {{"pull", "stage once, every peer pulls its part over NVLink", xchg_init},
    {"nvls", "multicast the own block into every member's heap with multimem.st, copy out locally", xchg_init_nvls},
    {"ring", "N-1 neighbour-to-neighbour pull steps through the heaps, one kernel", xchg_init_ring},
    {"push", "zero-copy push: every rank stores its block straight into the members' mapped destinations (TMA bulk copies from BULK_THRESH)", xchg_init_push},
    {"ce", "zero-copy push by the copy engines: cudaMemcpyAsync into the members' mapped destinations between two barrier kernels", xchg_init_ce}, {NULL}};
static const nvl_alg_t algs_a2a[] = {{"pull", "stage once, every peer pulls its part over NVLink", xchg_init},
    {"push", "zero-copy push: every rank stores block p straight into member p's mapped destination; alltoallv looks the landing offset up in a table the receiver publishes on the device", xchg_init_push},
    {"ce", "zero-copy push by the copy engines (reference ALLTOALL_USE_COPY_ENGINE): one cudaMemcpyAsync per peer between two barrier kernels", xchg_init_ce}, {NULL}};
static const nvl_alg_t algs_barrier[] = {{"flags", "flag exchange in peer memory", barrier_init}, {NULL}};
static const nvl_alg_t *const nvl_algs[UCC_COLL_TYPE_NUM] = {
    algs_ag, algs_ag, algs_allreduce, algs_a2a, algs_a2a, algs_barrier, algs_xchg_mc, algs_barrier, algs_barrier,
    algs_xchg, algs_xchg, algs_red, algs_rs, algs_rs, algs_xchg, algs_xchg};
static ucc_base_coll_alg_info_t nvl_alg_info[UCC_COLL_TYPE_NUM][8];

void ucc_tl_nvl_register_alg_info(void)
{
    for (int c = 0; c < UCC_COLL_TYPE_NUM; c++) {
        int i;
        for (i = 0; nvl_algs[c][i].name && i < 7; i++) { nvl_alg_info[c][i].id = (unsigned)i; nvl_alg_info[c][i].name = nvl_algs[c][i].name; nvl_alg_info[c][i].desc = nvl_algs[c][i].desc; }
        nvl_alg_info[c][i].name = NULL;
        ucc_tl_nvl.alg_info[c] = nvl_alg_info[c];
    }
}

ucc_status_t ucc_tl_nvl_alg_id_to_init(int alg_id, const char *alg_id_str, ucc_coll_type_t coll_type, ucc_memory_type_t mem_type, ucc_base_coll_init_fn_t *init)
{
    int c = ucc_coll_type_index(coll_type), n = 0;
    (void)mem_type;
    while (nvl_algs[c][n].name) n++;
    if (alg_id_str) { alg_id = -1; for (int i = 0; i < n; i++) if (!strcasecmp(alg_id_str, nvl_algs[c][i].name)) alg_id = i; }
    if (alg_id < 0 || alg_id >= n) return alg_id_str ? UCC_ERR_NOT_SUPPORTED : UCC_ERR_INVALID_PARAM;
    *init = nvl_algs[c][alg_id].init;
    return UCC_OK;
}

ucc_status_t ucc_tl_nvl_coll_init(ucc_base_coll_args_t *b, ucc_base_team_t *team, ucc_coll_task_t **task)
{ return nvl_algs[ucc_coll_type_index(b->args.coll_type)][0].init(b, team, task); }

ucc_status_t ucc_tl_nvl_team_get_scores(ucc_base_team_t *b_team, ucc_coll_score_t **score_p)
{
    ucc_tl_nvl_team_t *team = ucc_derived_of(b_team, ucc_tl_nvl_team_t);
    ucc_tl_nvl_context_t *ctx = NVL_CTX(team);
    ucc_memory_type_t mt[1] = {UCC_MEMORY_TYPE_CUDA};
    ucc_coll_score_team_info_t info = {UCC_TL_NVL_DEFAULT_SCORE, UCC_TL_TEAM_SIZE(team), UCC_TL_NVL_SUPPORTED_COLLS, mt, 1, ucc_tl_nvl_coll_init, ucc_tl_nvl_alg_id_to_init};
    ucc_coll_score_t *score;
    char sel[512], a[32], n[32];
    /* a team of one outranks tl/self (50) for CUDA buffers: its copy is a stream-ordered kernel instead of a blocking memcpy */
    ucc_status_t st = ucc_coll_score_build_default(b_team, team->self ? 60 : UCC_TL_NVL_DEFAULT_SCORE, ucc_tl_nvl_coll_init, UCC_TL_NVL_SUPPORTED_COLLS, mt, 1, &score);
    if (st != UCC_OK) return st;
    if (team->self) { info.default_score = 60; st = ucc_tl_apply_tune(&team->super, score, &info, NULL, ctx->cfg.super.super.score_str); if (st != UCC_OK) { ucc_coll_score_free(score); return st; } *score_p = score; return UCC_OK; }
    snprintf(a, sizeof(a), "%zu", ctx->cfg.oneshot_thresh + 1); /* ranges are end-exclusive, the threshold itself is still one-shot */
    ucc_memunits_to_str(ucc_max(ctx->cfg.nvls_thresh, ctx->cfg.oneshot_thresh + 1), n, sizeof(n));
    /* message-size driven defaults: latency kernel below the threshold, in-switch reduction for big
     * messages when the multicast mapping is live (dt/op it cannot do fall back to twoshot through the
     * score fallback chain because nvls init returns NOT_SUPPORTED) */
    /* with two members the switch has nothing to combine: pulling over P2P moves the same bytes with less overhead */
    /* measured on 8 x B200: zero-copy two-shot wins from 1 MB to a few hundred MB (every byte crosses NVLink once, no
     * staging); beyond that the in-switch reduction with its multicast store moves 1.75x fewer bytes out of each GPU and
     * overtakes it despite the two staging passes (ALLREDUCE_NVLS_THRESH, default 512M) */
    /* 4 x B200: zero-copy two-shot stays ahead at every size (634 GB/s at 256 MB vs 605 for NVLS at 1 GiB), and the
     * NVLS reduce_scatter loses to it because of the staging pass (390 vs NCCL 525 GB/s at 256 MB) - so NVLS is the
     * default only for very large allreduce on teams of more than four; `@nvls` remains selectable for everything */
    /* round 2, 8 x B200, 1 GiB f32 (profiles/r2_n8/matrix.jsonl): staged NVLS 706-716 GB/s, zero-copy two-shot 651, pipelined NVLS
     * (stage / multimem / copy-out of consecutive rounds overlapped, kernels/nvl_pipe.cu) 690 with a 128 MB heap, 770 with 384 MB
     * (three 128 MB round buffers) and 632 with 1 GB; NCCL 723.  Hence the 384 MB default heap and `nvls_pipe` above the threshold
     * whenever the heap is big enough for its round buffers; at 256 MB all four are within 2 % (628-637) and two-shot stays */
    if (team->nvls && UCC_TL_TEAM_SIZE(team) > 4)
        snprintf(sel, sizeof(sel), "allreduce:0-%s:@oneshot#allreduce:%s-inf:@%s", a, n, ctx->cfg.symmetric_size >= ((size_t)192 << 20) ? "nvls_pipe" : "nvls");
    else snprintf(sel, sizeof(sel), "allreduce:0-%s:@oneshot", a);
    /* data movement on teams of more than four (8 x B200, profiles/r2_n8/colls.jsonl): at 16 MB the zero-copy push exchange is at
     * NCCL's speed (allgather 54.8 us, alltoall 56.1 us; NCCL 53.9 / 56.6) where the pull kernel needs 69.3 / 66.7 us; at 1 MB and at
     * 256 MB pull is as good or better; push falls back to pull when a destination cannot be mapped.  (The skewed MoE alltoallv is
     * fastest on the copy engines from a few MB on - 16 MB: 93.9 us vs 144.3 us pull, NCCL 94.6 - but its sizes are private to each
     * member, so the score map cannot select by size (msgsize 0): `UCC_TL_NVL_TUNE=alltoallv:@ce` is the user's call) */
    if (UCC_TL_TEAM_SIZE(team) > 4 && team->zcopy) {
        size_t l = strlen(sel);
        snprintf(sel + l, sizeof(sel) - l, "#allgather:4M-64M:@push#alltoall:4M-64M:@push");
    }
    st = ucc_tl_apply_tune(&team->super, score, &info, sel, ctx->cfg.super.super.score_str);
    if (st != UCC_OK) { ucc_coll_score_free(score); return st; }
    *score_p = score;
    return UCC_OK;
}
