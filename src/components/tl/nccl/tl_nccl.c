/* tl/nccl: the baseline transport — a thin mapping of UCC collectives onto NCCL calls
 * (what reference tl/nccl does, tl_nccl_coll.c:265-951).  It exists for A/B comparison inside the
 * same perftest and as a fallback; its score (20) is below tl/nvl (40).  NCCL is dlopen'ed. */
#include "components/tl/ucc_tl.h"
#include "core/ucc_context.h"
#include "core/ucc_team.h"
#include "core/ucc_ee.h"
#include "core/ucc_service_coll.h"
#include "core/ucc_progress_queue.h"
#include "utils/ucc_mpool.h"
#include "utils/ucc_string.h"
#include "utils/cuda/ucc_cuda_util.h"
#include <nccl.h>
#include <dlfcn.h>
#include <strings.h>

#define UCC_TL_NCCL_DEFAULT_SCORE 20
#define UCC_TL_NCCL_SUPPORTED_COLLS (UCC_COLL_TYPE_ALLGATHER | UCC_COLL_TYPE_ALLGATHERV | UCC_COLL_TYPE_ALLREDUCE | UCC_COLL_TYPE_ALLTOALL | \
    UCC_COLL_TYPE_ALLTOALLV | UCC_COLL_TYPE_BARRIER | UCC_COLL_TYPE_BCAST | UCC_COLL_TYPE_GATHER | UCC_COLL_TYPE_GATHERV | UCC_COLL_TYPE_REDUCE | \
    UCC_COLL_TYPE_REDUCE_SCATTER | UCC_COLL_TYPE_SCATTER | UCC_COLL_TYPE_SCATTERV)

static struct {
    void *h;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *);
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int);
    ncclResult_t (*CommInitRankConfig)(ncclComm_t *, int, ncclUniqueId, int, ncclConfig_t *);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*CommAbort)(ncclComm_t);
    ncclResult_t (*CommGetAsyncError)(ncclComm_t, ncclResult_t *);
    const char  *(*GetErrorString)(ncclResult_t);
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*Reduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*ReduceScatter)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)(void);
    ncclResult_t (*GroupEnd)(void);
} nc;

typedef enum { NCCL_SYNC_AUTO, NCCL_SYNC_EVENT, NCCL_SYNC_DRIVER } nccl_sync_t;
typedef struct ucc_tl_nccl_context_config { ucc_tl_context_config_t super; unsigned sync; int blocking, lazy_init; } ucc_tl_nccl_context_config_t;
typedef struct ucc_tl_nccl_lib { ucc_tl_lib_t super; } ucc_tl_nccl_lib_t;
typedef struct ucc_tl_nccl_context { ucc_tl_context_t super; ucc_tl_nccl_context_config_t cfg; ucc_mpool_t task_mp; int dev; float *barrier_buf; } ucc_tl_nccl_context_t;
typedef enum { NCCL_COMM_UNINIT, NCCL_COMM_INITING, NCCL_COMM_READY, NCCL_COMM_ERROR } nccl_comm_state_t;
/* what every member publishes at team creation: rank 0's unique id + where the member runs, so that all members take
 * the same decision about teams NCCL cannot serve (two members on one GPU) and about members sharing a process */
typedef struct nccl_member_info { ncclUniqueId id; uint64_t host_hash; int32_t pid; int32_t dev; char busid[24]; } nccl_member_info_t;
typedef struct ucc_tl_nccl_team {
    ucc_tl_team_t super; nccl_member_info_t *ids; void *oob_req; ucc_team_oob_coll_t oob; int oob_internal;
    ncclComm_t comm; nccl_comm_state_t state; cudaStream_t stream; nccl_member_info_t my_id; int inproc_peers;
} ucc_tl_nccl_team_t;
typedef struct ucc_tl_nccl_task {
    ucc_coll_task_t super; ucc_tl_nccl_team_t *team; cudaEvent_t event; int captured; int alg;
    volatile uint32_t *host_status; uint32_t *dev_status; void *scratch;
} ucc_tl_nccl_task_t;
extern ucc_tl_iface_t ucc_tl_nccl;
#define NCCL_CTX(_t) ucc_derived_of((_t)->super.super.context, ucc_tl_nccl_context_t)
#define NLIB(_t) ((_t)->super.super.context->lib)
#define NCCLCHECK(_team, _call) do { ncclResult_t _r = (_call); if (_r != ncclSuccess && _r != ncclInProgress) { \
    tl_error(NLIB(_team), "%s failed: %s", #_call, nc.GetErrorString ? nc.GetErrorString(_r) : "?"); return UCC_ERR_NO_MESSAGE; } } while (0)

static const char *sync_names[] = {"auto", "event", "driver", NULL};
static ucc_config_field_t tl_nccl_lib_config_table[] = {{"", "", NULL, 0, UCC_CONFIG_TYPE_TABLE(ucc_tl_lib_config_table)}, {NULL}};
static ucc_config_field_t tl_nccl_context_config_table[] = {
    {"", "", NULL, ucc_offsetof(ucc_tl_nccl_context_config_t, super), UCC_CONFIG_TYPE_TABLE(ucc_tl_context_config_table)},
    {"SYNC", "auto", "Completion detection: event (cudaEventQuery) or driver (stream memory operation writing a host flag)", ucc_offsetof(ucc_tl_nccl_context_config_t, sync), UCC_CONFIG_TYPE_ENUM(sync_names)},
    {"BLOCKING", "yes", "Use blocking NCCL communicator initialisation", ucc_offsetof(ucc_tl_nccl_context_config_t, blocking), UCC_CONFIG_TYPE_BOOL},
    {"LAZY_INIT", "yes", "Create the NCCL communicator at the first collective instead of at team creation", ucc_offsetof(ucc_tl_nccl_context_config_t, lazy_init), UCC_CONFIG_TYPE_BOOL},
    {NULL}};

static ucc_status_t load_nccl(void)
{
    if (nc.h) return UCC_OK;
    /* never pull a second NCCL into a process that will load its own (PyTorch bundles one with the same
     * soname): use the copy that is already mapped, else an explicit override, else the system library */
    nc.h = dlopen("libnccl.so.2", RTLD_LAZY | RTLD_NOLOAD);
    if (!nc.h && getenv("UCC_TL_NCCL_LIB")) nc.h = dlopen(getenv("UCC_TL_NCCL_LIB"), RTLD_LAZY | RTLD_LOCAL);
    if (!nc.h && !getenv("UCC_TL_NCCL_NO_SYSTEM_LIB")) nc.h = dlopen("libnccl.so.2", RTLD_LAZY | RTLD_LOCAL);
    if (!nc.h) return UCC_ERR_NO_RESOURCE;
#define SYM(_f) *(void **)&nc._f = dlsym(nc.h, "nccl" #_f)
    SYM(GetUniqueId); SYM(CommInitRank); SYM(CommInitRankConfig); SYM(CommDestroy); SYM(CommAbort); SYM(CommGetAsyncError); SYM(GetErrorString); SYM(AllReduce); SYM(Broadcast);
    SYM(Reduce); SYM(AllGather); SYM(ReduceScatter); SYM(Send); SYM(Recv); SYM(GroupStart); SYM(GroupEnd);
    return (nc.GetUniqueId && nc.CommInitRank && nc.AllReduce && nc.Send && nc.GroupStart) ? UCC_OK : UCC_ERR_NO_RESOURCE;
}

/* ---- lib / ctx ---- */
static ucc_status_t nccl_lib_init(const ucc_base_lib_params_t *p, const ucc_base_lib_config_t *config, ucc_base_lib_t **lib_p)
{
    ucc_tl_nccl_lib_t *lib; int n = 0; (void)p;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { (void)cudaGetLastError(); return UCC_ERR_NO_RESOURCE; }
    if (load_nccl() != UCC_OK) return UCC_ERR_NO_RESOURCE;
    lib = (ucc_tl_nccl_lib_t *)calloc(1, sizeof(*lib)); if (!lib) return UCC_ERR_NO_MEMORY;
    ucc_tl_lib_init_base(&lib->super, &ucc_tl_nccl, ucc_derived_of(config, ucc_tl_lib_config_t));
    *lib_p = &lib->super.super; return UCC_OK;
}
static void nccl_lib_finalize(ucc_base_lib_t *lib) { free(lib); }
static ucc_status_t nccl_lib_get_attr(const ucc_base_lib_t *lib, ucc_base_lib_attr_t *attr)
{ (void)lib; attr->attr.thread_mode = UCC_THREAD_MULTIPLE; attr->attr.coll_types = UCC_TL_NCCL_SUPPORTED_COLLS; attr->flags = 0; attr->min_team_size = 2; attr->max_team_size = UCC_RANK_MAX; return UCC_OK; }
static ucc_status_t nccl_lib_get_properties(ucc_base_lib_properties_t *p) { p->default_team_size = 2; p->min_team_size = 2; p->max_team_size = UCC_RANK_MAX; return UCC_OK; }
static ucc_status_t nccl_ctx_create(const ucc_base_context_params_t *p, const ucc_base_ctx_config_t *config, ucc_base_context_t **ctx_p)
{
    ucc_tl_nccl_context_t *ctx; int dev;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); return UCC_ERR_NO_RESOURCE; }
    ctx = (ucc_tl_nccl_context_t *)calloc(1, sizeof(*ctx)); if (!ctx) return UCC_ERR_NO_MEMORY;
    ctx->super.super.ucc_context = p->context; ctx->super.super.lib = config->lib; ctx->dev = dev;
    ucc_config_parser_clone_opts(config, &ctx->cfg, tl_nccl_context_config_table);
    if (cudaMalloc((void **)&ctx->barrier_buf, 2 * sizeof(float)) != cudaSuccess) { (void)cudaGetLastError(); free(ctx); return UCC_ERR_NO_MEMORY; }
    ucc_mpool_init(&ctx->task_mp, 0, sizeof(ucc_tl_nccl_task_t), 0, 64, 8, (unsigned)-1, NULL, p->thread_mode, "tl_nccl_tasks");
    *ctx_p = &ctx->super.super; return UCC_OK;
}
static void nccl_ctx_destroy(ucc_base_context_t *b)
{ ucc_tl_nccl_context_t *ctx = ucc_derived_of(b, ucc_tl_nccl_context_t); cudaFree(ctx->barrier_buf); ucc_mpool_cleanup(&ctx->task_mp, 1); ucc_config_parser_release_opts(&ctx->cfg, tl_nccl_context_config_table); free(ctx); }
static ucc_status_t nccl_ctx_get_attr(const ucc_base_context_t *b, ucc_base_ctx_attr_t *attr)
{ (void)b; if (attr->attr.mask & UCC_CONTEXT_ATTR_FIELD_CTX_ADDR_LEN) attr->attr.ctx_addr_len = 0; attr->topo_required = 0; attr->attr.global_work_buffer_size = 0; return UCC_OK; }

/* ---- team ---- */
/* Communicator creation.  Blocking mode (default, one member per process): ncclCommInitRank returns when every member
 * has called it.  Non-blocking mode (UCC_TL_NCCL_BLOCKING=n, or members that share a process - a blocking call issued from
 * the single thread that drives several members would wait for members that are never reached): ncclCommInitRankConfig
 * with blocking=0, then ncclCommGetAsyncError is polled; `wait` = spin here until the communicator is usable. */
static ucc_status_t nccl_comm_init(ucc_tl_nccl_team_t *team, int wait)
{
    int nonblocking = (!NCCL_CTX(team)->cfg.blocking || team->inproc_peers) && nc.CommInitRankConfig && nc.CommGetAsyncError;
    ncclResult_t r, ar;
    if (team->state == NCCL_COMM_READY) return UCC_OK;
    if (team->state == NCCL_COMM_ERROR) return UCC_ERR_NOT_SUPPORTED;
    if (team->state == NCCL_COMM_UNINIT) {
        if (cudaStreamCreateWithFlags(&team->stream, cudaStreamNonBlocking) != cudaSuccess) { (void)cudaGetLastError(); team->state = NCCL_COMM_ERROR; return UCC_ERR_NOT_SUPPORTED; }
        if (nonblocking) {
            ncclConfig_t cfg = NCCL_CONFIG_INITIALIZER;
            cfg.blocking = 0;
            r = nc.CommInitRankConfig(&team->comm, (int)UCC_TL_TEAM_SIZE(team), team->ids[0].id, (int)UCC_TL_TEAM_RANK(team), &cfg);
            if (r != ncclSuccess && r != ncclInProgress) { tl_debug(NLIB(team), "ncclCommInitRankConfig failed"); team->state = NCCL_COMM_ERROR; return UCC_ERR_NOT_SUPPORTED; }
            team->state = NCCL_COMM_INITING;
        } else {
            if (nc.CommInitRank(&team->comm, (int)UCC_TL_TEAM_SIZE(team), team->ids[0].id, (int)UCC_TL_TEAM_RANK(team)) != ncclSuccess) {
                tl_debug(NLIB(team), "ncclCommInitRank failed"); team->state = NCCL_COMM_ERROR; return UCC_ERR_NOT_SUPPORTED; }
            team->state = NCCL_COMM_READY;
            return UCC_OK;
        }
    }
    do {
        ar = ncclSuccess;
        r = nc.CommGetAsyncError(team->comm, &ar);
        if (r != ncclSuccess || (ar != ncclSuccess && ar != ncclInProgress)) { tl_debug(NLIB(team), "NCCL communicator creation failed"); team->state = NCCL_COMM_ERROR; return UCC_ERR_NOT_SUPPORTED; }
        if (ar == ncclSuccess) { team->state = NCCL_COMM_READY; return UCC_OK; }
    } while (wait);
    return UCC_INPROGRESS;
}
static ucc_status_t nccl_team_create_post(ucc_base_context_t *b_ctx, const ucc_base_team_params_t *params, ucc_base_team_t **team_p)
{
    ucc_tl_nccl_team_t *team = (ucc_tl_nccl_team_t *)calloc(1, sizeof(*team));
    ucc_status_t st;
    if (!team) return UCC_ERR_NO_MEMORY;
    team->super.super.context = b_ctx; team->super.super.params = *params;
    if (params->params.mask & UCC_TEAM_PARAM_FIELD_OOB) team->oob = params->params.oob;
    else { ucc_subset_t s; s.map = params->map; s.myrank = params->rank; if (ucc_internal_oob_init(params->team, s, &team->oob) != UCC_OK) { free(team); return UCC_ERR_NOT_SUPPORTED; } team->oob_internal = 1; }
    team->ids = (nccl_member_info_t *)calloc(params->size, sizeof(nccl_member_info_t));
    memset(&team->my_id, 0, sizeof(team->my_id));
    if (params->rank == 0 && nc.GetUniqueId(&team->my_id.id) != ncclSuccess) { free(team->ids); free(team); return UCC_ERR_NO_MESSAGE; }
    team->my_id.host_hash = ucc_local_proc.host_hash; team->my_id.pid = (int32_t)ucc_local_proc.pid; team->my_id.dev = ucc_derived_of(b_ctx, ucc_tl_nccl_context_t)->dev;
    if (cudaDeviceGetPCIBusId(team->my_id.busid, (int)sizeof(team->my_id.busid), team->my_id.dev) != cudaSuccess) { (void)cudaGetLastError(); snprintf(team->my_id.busid, sizeof(team->my_id.busid), "dev%d", team->my_id.dev); }
    st = team->oob.allgather(&team->my_id, team->ids, sizeof(nccl_member_info_t), team->oob.coll_info, &team->oob_req);
    if (st != UCC_OK) { free(team->ids); free(team); return st; }
    *team_p = &team->super.super;
    return UCC_OK;
}
static ucc_status_t nccl_team_create_test(ucc_base_team_t *b)
{
    ucc_tl_nccl_team_t *team = ucc_derived_of(b, ucc_tl_nccl_team_t);
    ucc_rank_t size = UCC_TL_TEAM_SIZE(team), i, j;
    ucc_status_t st;
    if (team->oob_req) {
        st = team->oob.req_test(team->oob_req);
        if (st == UCC_INPROGRESS) return st;
        team->oob.req_free(team->oob_req); team->oob_req = NULL;
        if (st < 0) goto fail;
        /* decisions every member derives from the same gathered table */
        for (i = 0; i < size; i++) for (j = i + 1; j < size; j++) {
            if (team->ids[i].host_hash != team->ids[j].host_hash) continue;
            if (!strncmp(team->ids[i].busid, team->ids[j].busid, sizeof(team->ids[i].busid))) {
                tl_debug(NLIB(team), "members %u and %u share GPU %s: NCCL cannot serve this team", (unsigned)i, (unsigned)j, team->ids[i].busid);
                st = UCC_ERR_NOT_SUPPORTED; goto fail;
            }
            if (team->ids[i].pid == team->ids[j].pid) team->inproc_peers = 1;
        }
    }
    if (!NCCL_CTX(team)->cfg.lazy_init || team->inproc_peers) {
        st = nccl_comm_init(team, 0);
        if (st == UCC_INPROGRESS) return st;
        if (st != UCC_OK) goto fail;
    }
    return UCC_OK;
fail:
    if (team->comm && nc.CommAbort) nc.CommAbort(team->comm);
    if (team->stream) cudaStreamDestroy(team->stream);
    if (team->oob_internal) ucc_internal_oob_finalize(&team->oob);
    free(team->ids); free(team);
    return st;
}
static ucc_status_t nccl_team_destroy(ucc_base_team_t *b)
{
    ucc_tl_nccl_team_t *team = ucc_derived_of(b, ucc_tl_nccl_team_t);
    if (team->comm) { if (team->state == NCCL_COMM_ERROR && nc.CommAbort) nc.CommAbort(team->comm); else nc.CommDestroy(team->comm); }
    if (team->stream) cudaStreamDestroy(team->stream);
    if (team->oob_internal) ucc_internal_oob_finalize(&team->oob);
    free(team->ids); free(team);
    return UCC_OK;
}

/* ---- collectives ---- */
static int to_nccl_dt(ucc_datatype_t dt, ncclDataType_t *o)
{
    switch (dt) {
    case UCC_DT_INT8: *o = ncclInt8; break; case UCC_DT_UINT8: *o = ncclUint8; break; case UCC_DT_INT32: *o = ncclInt32; break; case UCC_DT_UINT32: *o = ncclUint32; break;
    case UCC_DT_INT64: *o = ncclInt64; break; case UCC_DT_UINT64: *o = ncclUint64; break; case UCC_DT_FLOAT16: *o = ncclFloat16; break; case UCC_DT_FLOAT32: *o = ncclFloat32; break;
    case UCC_DT_FLOAT64: *o = ncclFloat64; break; case UCC_DT_BFLOAT16: *o = ncclBfloat16; break; default: return 0;
    }
    return 1;
}
static int to_nccl_op(ucc_reduction_op_t op, ncclRedOp_t *o)
{
    switch (op) { case UCC_OP_SUM: *o = ncclSum; break; case UCC_OP_PROD: *o = ncclProd; break; case UCC_OP_MAX: *o = ncclMax; break; case UCC_OP_MIN: *o = ncclMin; break; case UCC_OP_AVG: *o = ncclAvg; break; default: return 0; }
    return 1;
}
/* complex SUM / AVG work part by part: NCCL reduces them as a real vector twice as long (as the reference's tl/nccl does);
 * returns how many real elements one element of udt is, 0 when NCCL cannot reduce (udt, op) */
static int nccl_red_type(ucc_datatype_t udt, ucc_reduction_op_t uop, ncclDataType_t *dt, ncclRedOp_t *op)
{
    if (!to_nccl_op(uop, op)) return 0;
    if (udt == UCC_DT_FLOAT32_COMPLEX || udt == UCC_DT_FLOAT64_COMPLEX) {
        if (uop != UCC_OP_SUM && uop != UCC_OP_AVG) return 0;
        *dt = udt == UCC_DT_FLOAT32_COMPLEX ? ncclFloat32 : ncclFloat64;
        return 2;
    }
    return to_nccl_dt(udt, dt);
}
static int cuda_mt(ucc_memory_type_t mt) { return mt == UCC_MEMORY_TYPE_CUDA || mt == UCC_MEMORY_TYPE_CUDA_MANAGED; }

/* the NCCL calls of one collective */
static ucc_status_t nccl_issue(ucc_tl_nccl_task_t *t, cudaStream_t s)
{
    ucc_tl_nccl_team_t *team = t->team; ucc_coll_args_t *a = &t->super.bargs.args;
    ucc_rank_t N = UCC_TL_TEAM_SIZE(team), me = UCC_TL_TEAM_RANK(team); int inplace = UCC_IS_INPLACE(*a), root = (ucc_rank_t)a->root == me;
    ncclDataType_t dt = ncclUint8; ncclRedOp_t op = ncclSum; ncclComm_t c = team->comm;
    switch (a->coll_type) {
    case UCC_COLL_TYPE_ALLREDUCE: {
        size_t cnt = a->dst.info.count * nccl_red_type(a->dst.info.datatype, a->op, &dt, &op);
        NCCLCHECK(team, nc.AllReduce(inplace ? a->dst.info.buffer : a->src.info.buffer, a->dst.info.buffer, cnt, dt, op, c, s)); break; }
    case UCC_COLL_TYPE_BARRIER:
        NCCLCHECK(team, nc.AllReduce(NCCL_CTX(team)->barrier_buf, NCCL_CTX(team)->barrier_buf + 1, 1, ncclFloat32, ncclSum, c, s)); break;
    case UCC_COLL_TYPE_ALLGATHER: {
        size_t blk = a->dst.info.count / N * ucc_dt_size(a->dst.info.datatype);
        NCCLCHECK(team, nc.AllGather(inplace ? (char *)a->dst.info.buffer + me * blk : a->src.info.buffer, a->dst.info.buffer, blk, ncclUint8, c, s)); break; }
    case UCC_COLL_TYPE_ALLGATHERV: {
        size_t dts = ucc_dt_size(a->dst.info_v.datatype);
        const void *mine = inplace ? (char *)a->dst.info_v.buffer + ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, me) * dts : a->src.info.buffer;
        if (t->alg == 2) { /* bcast: N grouped broadcasts */
            NCCLCHECK(team, nc.GroupStart());
            for (ucc_rank_t p = 0; p < N; p++) { size_t cnt = ucc_coll_args_get_count(a, a->dst.info_v.counts, p) * dts; void *d = (char *)a->dst.info_v.buffer + ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, p) * dts;
                if (cnt) NCCLCHECK(team, nc.Broadcast(p == me ? mine : d, d, cnt, ncclUint8, (int)p, c, s)); }
            NCCLCHECK(team, nc.GroupEnd());
        } else if (t->alg == 1) { /* bcopy: allgather of max count into scratch, then copy out */
            size_t maxc = ucc_coll_args_get_max_count(a, a->dst.info_v.counts, N) * dts;
            CUDA_CHECK(cudaMemcpyAsync((char *)t->scratch + N * maxc, mine, ucc_coll_args_get_count(a, a->dst.info_v.counts, me) * dts, cudaMemcpyDeviceToDevice, s));
            NCCLCHECK(team, nc.AllGather((char *)t->scratch + N * maxc, t->scratch, maxc, ncclUint8, c, s));
            for (ucc_rank_t p = 0; p < N; p++) CUDA_CHECK(cudaMemcpyAsync((char *)a->dst.info_v.buffer + ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, p) * dts,
                                                                          (char *)t->scratch + p * maxc, ucc_coll_args_get_count(a, a->dst.info_v.counts, p) * dts, cudaMemcpyDeviceToDevice, s));
        } else { /* p2p */
            NCCLCHECK(team, nc.GroupStart());
            for (ucc_rank_t p = 0; p < N; p++) {
                size_t cnt = ucc_coll_args_get_count(a, a->dst.info_v.counts, p) * dts, mycnt = ucc_coll_args_get_count(a, a->dst.info_v.counts, me) * dts;
                if (mycnt) NCCLCHECK(team, nc.Send(mine, mycnt, ncclUint8, (int)p, c, s));
                if (cnt) NCCLCHECK(team, nc.Recv((char *)a->dst.info_v.buffer + ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, p) * dts, cnt, ncclUint8, (int)p, c, s));
            }
            NCCLCHECK(team, nc.GroupEnd());
        }
        break; }
    case UCC_COLL_TYPE_ALLTOALL: {
        size_t blk = a->dst.info.count / N * ucc_dt_size(a->dst.info.datatype);
        NCCLCHECK(team, nc.GroupStart());
        for (ucc_rank_t p = 0; p < N; p++) { NCCLCHECK(team, nc.Send((char *)a->src.info.buffer + p * blk, blk, ncclUint8, (int)p, c, s)); NCCLCHECK(team, nc.Recv((char *)a->dst.info.buffer + p * blk, blk, ncclUint8, (int)p, c, s)); }
        NCCLCHECK(team, nc.GroupEnd()); break; }
    case UCC_COLL_TYPE_ALLTOALLV: {
        size_t sdt = ucc_dt_size(a->src.info_v.datatype), ddt = ucc_dt_size(a->dst.info_v.datatype);
        NCCLCHECK(team, nc.GroupStart());
        for (ucc_rank_t p = 0; p < N; p++) {
            size_t sc = ucc_coll_args_get_count(a, a->src.info_v.counts, p) * sdt, rc = ucc_coll_args_get_count(a, a->dst.info_v.counts, p) * ddt;
            if (sc) NCCLCHECK(team, nc.Send((char *)a->src.info_v.buffer + ucc_coll_args_get_displacement(a, a->src.info_v.displacements, p) * sdt, sc, ncclUint8, (int)p, c, s));
            if (rc) NCCLCHECK(team, nc.Recv((char *)a->dst.info_v.buffer + ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, p) * ddt, rc, ncclUint8, (int)p, c, s));
        }
        NCCLCHECK(team, nc.GroupEnd()); break; }
    case UCC_COLL_TYPE_BCAST:
        if (UCC_COLL_ARGS_ACTIVE_SET(a)) { /* 2-rank style active set: root sends to the other members */
            size_t len = a->src.info.count * ucc_dt_size(a->src.info.datatype);
            NCCLCHECK(team, nc.GroupStart());
            if (root) { for (uint64_t i = 0; i < a->active_set.size; i++) { ucc_rank_t p = (ucc_rank_t)(a->active_set.start + i * a->active_set.stride); if (p != me) NCCLCHECK(team, nc.Send(a->src.info.buffer, len, ncclUint8, (int)p, c, s)); } }
            else NCCLCHECK(team, nc.Recv(a->src.info.buffer, len, ncclUint8, (int)a->root, c, s));
            NCCLCHECK(team, nc.GroupEnd());
        } else NCCLCHECK(team, nc.Broadcast(a->src.info.buffer, a->src.info.buffer, a->src.info.count * ucc_dt_size(a->src.info.datatype), ncclUint8, (int)a->root, c, s));
        break;
    case UCC_COLL_TYPE_REDUCE_SCATTER: {
        size_t cnt = inplace ? a->dst.info.count / N : a->dst.info.count, mine = me * cnt * ucc_dt_size(a->dst.info.datatype);
        cnt *= nccl_red_type(a->dst.info.datatype, a->op, &dt, &op);
        NCCLCHECK(team, nc.ReduceScatter(inplace ? a->dst.info.buffer : a->src.info.buffer, inplace ? (char *)a->dst.info.buffer + mine : a->dst.info.buffer, cnt, dt, op, c, s)); break; }
    case UCC_COLL_TYPE_REDUCE: {
        ucc_datatype_t udt = root ? a->dst.info.datatype : a->src.info.datatype; size_t cnt = root ? a->dst.info.count : a->src.info.count;
        cnt *= nccl_red_type(udt, a->op, &dt, &op);
        NCCLCHECK(team, nc.Reduce((root && inplace) ? a->dst.info.buffer : a->src.info.buffer, root ? a->dst.info.buffer : NULL, cnt, dt, op, (int)a->root, c, s)); break; }
    case UCC_COLL_TYPE_GATHER: case UCC_COLL_TYPE_GATHERV: {
        int v = a->coll_type == UCC_COLL_TYPE_GATHERV;
        NCCLCHECK(team, nc.GroupStart());
        if (root) {
            size_t dts = ucc_dt_size(v ? a->dst.info_v.datatype : a->dst.info.datatype); char *dst = (char *)(v ? a->dst.info_v.buffer : a->dst.info.buffer);
            for (ucc_rank_t p = 0; p < N; p++) {
                size_t cnt = v ? ucc_coll_args_get_count(a, a->dst.info_v.counts, p) * dts : a->dst.info.count / N * dts, off = v ? ucc_coll_args_get_displacement(a, a->dst.info_v.displacements, p) * dts : p * cnt;
                if (p == me) { if (!inplace && cnt) CUDA_CHECK(cudaMemcpyAsync(dst + off, a->src.info.buffer, cnt, cudaMemcpyDeviceToDevice, s)); }
                else if (cnt) NCCLCHECK(team, nc.Recv(dst + off, cnt, ncclUint8, (int)p, c, s));
            }
        } else { size_t cnt = a->src.info.count * ucc_dt_size(a->src.info.datatype); if (cnt) NCCLCHECK(team, nc.Send(a->src.info.buffer, cnt, ncclUint8, (int)a->root, c, s)); }
        NCCLCHECK(team, nc.GroupEnd()); break; }
    case UCC_COLL_TYPE_SCATTER: case UCC_COLL_TYPE_SCATTERV: {
        int v = a->coll_type == UCC_COLL_TYPE_SCATTERV;
        NCCLCHECK(team, nc.GroupStart());
        if (root) {
            size_t dts = ucc_dt_size(v ? a->src.info_v.datatype : a->src.info.datatype); char *src = (char *)(v ? a->src.info_v.buffer : a->src.info.buffer);
            for (ucc_rank_t p = 0; p < N; p++) {
                size_t cnt = v ? ucc_coll_args_get_count(a, a->src.info_v.counts, p) * dts : a->src.info.count / N * dts, off = v ? ucc_coll_args_get_displacement(a, a->src.info_v.displacements, p) * dts : p * cnt;
                if (p == me) { if (!inplace && cnt) CUDA_CHECK(cudaMemcpyAsync(a->dst.info.buffer, src + off, cnt, cudaMemcpyDeviceToDevice, s)); }
                else if (cnt) NCCLCHECK(team, nc.Send(src + off, cnt, ncclUint8, (int)p, c, s));
            }
        } else { size_t cnt = a->dst.info.count * ucc_dt_size(a->dst.info.datatype); if (cnt) NCCLCHECK(team, nc.Recv(a->dst.info.buffer, cnt, ncclUint8, (int)a->root, c, s)); }
        NCCLCHECK(team, nc.GroupEnd()); break; }
    default: return UCC_ERR_NOT_SUPPORTED;
    }
    return UCC_OK;
}

static void nccl_progress(ucc_coll_task_t *ct)
{
    ucc_tl_nccl_task_t *t = ucc_derived_of(ct, ucc_tl_nccl_task_t);
    ncclResult_t ar = ncclSuccess; cudaError_t e;
    if (t->captured) { ct->status = UCC_OK; return; }
    if (nc.CommGetAsyncError && nc.CommGetAsyncError(t->team->comm, &ar) == ncclSuccess && ar != ncclSuccess && ar != ncclInProgress) {
        tl_error(NLIB(t->team), "NCCL async error: %s", nc.GetErrorString(ar)); t->team->state = NCCL_COMM_ERROR; ct->status = UCC_ERR_NO_MESSAGE; return; }
    if (t->host_status) { if (*t->host_status == (uint32_t)UCC_OK) ct->status = UCC_OK; return; }
    e = cudaEventQuery(t->event);
    if (e == cudaErrorNotReady) { (void)cudaGetLastError(); return; }
    ct->status = ucc_cuda_error_to_status(e);
}
static ucc_status_t nccl_post_on(ucc_tl_nccl_task_t *t, cudaStream_t s)
{
    enum cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone; ucc_status_t st;
    t->captured = (cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive);
    st = nccl_issue(t, s); if (st != UCC_OK) return st;
    if (!t->captured) {
        if (t->host_status && ucc_cu.cuStreamWriteValue32) { *t->host_status = (uint32_t)UCC_INPROGRESS; if (ucc_cu.cuStreamWriteValue32((CUstream)s, (CUdeviceptr)(uintptr_t)t->dev_status, (uint32_t)UCC_OK, 0) != CUDA_SUCCESS) return UCC_ERR_NO_MESSAGE; }
        else CUDA_CHECK(cudaEventRecord(t->event, s));
    }
    return ucc_progress_queue_enqueue(UCC_TL_CORE_CTX(t->team)->pq, &t->super);
}
static ucc_status_t nccl_post(ucc_coll_task_t *ct) { ucc_tl_nccl_task_t *t = ucc_derived_of(ct, ucc_tl_nccl_task_t); return nccl_post_on(t, t->team->stream); }
static ucc_status_t nccl_triggered_post(ucc_ee_h ee, ucc_ev_t *ev, ucc_coll_task_t *ct)
{
    ucc_tl_nccl_task_t *t = ucc_derived_of(ct, ucc_tl_nccl_task_t); ucc_ev_t pe; ucc_status_t st; (void)ev;
    if (ee->ee_type != UCC_EE_CUDA_STREAM) return UCC_ERR_NOT_SUPPORTED;
    ct->ee = ee; st = nccl_post_on(t, (cudaStream_t)ee->ee_context); if (st != UCC_OK) return st;
    pe.ev_type = UCC_EVENT_COLLECTIVE_POST; pe.ev_context = NULL; pe.ev_context_size = 0; pe.req = &ct->super;
    ucc_ee_set_event_internal(ee, &pe, &ee->event_out_queue);
    return UCC_OK;
}
static ucc_status_t nccl_finalize(ucc_coll_task_t *ct)
{
    ucc_tl_nccl_task_t *t = ucc_derived_of(ct, ucc_tl_nccl_task_t);
    if (t->event) cudaEventDestroy(t->event);
    if (t->host_status) cudaFreeHost((void *)t->host_status);
    if (t->scratch) cudaFree(t->scratch);
    ucc_coll_task_destruct(ct); ucc_mpool_put(t); return UCC_OK;
}

static ucc_status_t nccl_coll_init_alg(ucc_base_coll_args_t *b, ucc_base_team_t *b_team, ucc_coll_task_t **task_p, int alg)
{
    ucc_tl_nccl_team_t *team = ucc_derived_of(b_team, ucc_tl_nccl_team_t); ucc_tl_nccl_context_t *ctx = NCCL_CTX(team);
    ucc_coll_args_t *a = &b->args; ucc_tl_nccl_task_t *t; ncclDataType_t dt; ncclRedOp_t op; ucc_status_t st;
    ucc_memory_type_t mt = ucc_coll_args_mem_type(a, UCC_TL_TEAM_RANK(team));
    if (!(UCC_TL_NCCL_SUPPORTED_COLLS & a->coll_type)) return UCC_ERR_NOT_SUPPORTED;
    if (a->coll_type != UCC_COLL_TYPE_BARRIER && !cuda_mt(mt)) return UCC_ERR_NOT_SUPPORTED;
    if (ucc_coll_has_reduction(a->coll_type)) {
        int root = (ucc_rank_t)a->root == UCC_TL_TEAM_RANK(team);
        ucc_datatype_t udt = (a->coll_type == UCC_COLL_TYPE_REDUCE && !root) ? a->src.info.datatype : a->dst.info.datatype;
        if (!nccl_red_type(udt, a->op, &dt, &op)) return UCC_ERR_NOT_SUPPORTED;
    }
    if ((a->coll_type & (UCC_COLL_TYPE_ALLTOALL | UCC_COLL_TYPE_ALLTOALLV)) && UCC_IS_INPLACE(*a)) return UCC_ERR_NOT_SUPPORTED;
    if (UCC_COLL_ARGS_ACTIVE_SET(a) && a->coll_type != UCC_COLL_TYPE_BCAST) return UCC_ERR_NOT_SUPPORTED;
    st = nccl_comm_init(team, 1); /* lazy */
    if (st != UCC_OK) return st;
    t = (ucc_tl_nccl_task_t *)ucc_mpool_get(&ctx->task_mp); if (!t) return UCC_ERR_NO_MEMORY;
    ucc_coll_task_init(&t->super, b, b_team);
    t->team = team; t->event = NULL; t->host_status = NULL; t->dev_status = NULL; t->scratch = NULL; t->alg = alg; t->captured = 0;
    t->super.post = nccl_post; t->super.progress = nccl_progress; t->super.finalize = nccl_finalize; t->super.triggered_post = nccl_triggered_post;
    if (ctx->cfg.sync == NCCL_SYNC_DRIVER && ucc_cu_api_load() == UCC_OK && ucc_cu.cuStreamWriteValue32) {
        void *dp = NULL;
        if (cudaHostAlloc((void **)&t->host_status, sizeof(uint32_t), cudaHostAllocMapped) == cudaSuccess && cudaHostGetDevicePointer(&dp, (void *)t->host_status, 0) == cudaSuccess) t->dev_status = (uint32_t *)dp;
        else { (void)cudaGetLastError(); t->host_status = NULL; }
    }
    if (!t->host_status && cudaEventCreateWithFlags(&t->event, cudaEventDisableTiming) != cudaSuccess) { (void)cudaGetLastError(); ucc_mpool_put(t); return UCC_ERR_NO_RESOURCE; }
    if (a->coll_type == UCC_COLL_TYPE_ALLGATHERV && alg == 1) {
        size_t maxc = ucc_coll_args_get_max_count(a, a->dst.info_v.counts, UCC_TL_TEAM_SIZE(team)) * ucc_dt_size(a->dst.info_v.datatype);
        if (cudaMalloc(&t->scratch, (UCC_TL_TEAM_SIZE(team) + 1) * (maxc ? maxc : 1)) != cudaSuccess) { (void)cudaGetLastError(); nccl_finalize(&t->super); return UCC_ERR_NO_MEMORY; }
    }
    *task_p = &t->super;
    return UCC_OK;
}
static ucc_status_t nccl_coll_init(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return nccl_coll_init_alg(b, t, p, 0); }
static ucc_status_t nccl_coll_init_1(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return nccl_coll_init_alg(b, t, p, 1); }
static ucc_status_t nccl_coll_init_2(ucc_base_coll_args_t *b, ucc_base_team_t *t, ucc_coll_task_t **p) { return nccl_coll_init_alg(b, t, p, 2); }

static const ucc_base_coll_alg_info_t allgatherv_algs[] = {{0, "p2p", "grouped ncclSend/ncclRecv"}, {1, "bcopy", "ncclAllGather of the max count into a scratch + copy out"},
                                                           {2, "bcast", "one grouped ncclBroadcast per rank"}, {0, NULL, NULL}};
static ucc_status_t nccl_alg_id_to_init(int alg_id, const char *s, ucc_coll_type_t ct, ucc_memory_type_t mt, ucc_base_coll_init_fn_t *init)
{
    (void)mt;
    if (ct != UCC_COLL_TYPE_ALLGATHERV) return UCC_ERR_NOT_SUPPORTED;
    if (s) { alg_id = -1; for (int i = 0; allgatherv_algs[i].name; i++) if (!strcasecmp(s, allgatherv_algs[i].name)) alg_id = i; }
    if (alg_id < 0 || alg_id > 2) return s ? UCC_ERR_NOT_SUPPORTED : UCC_ERR_INVALID_PARAM;
    *init = alg_id == 0 ? nccl_coll_init : alg_id == 1 ? nccl_coll_init_1 : nccl_coll_init_2;
    return UCC_OK;
}
static ucc_status_t nccl_team_get_scores(ucc_base_team_t *b_team, ucc_coll_score_t **score_p)
{
    ucc_tl_nccl_team_t *team = ucc_derived_of(b_team, ucc_tl_nccl_team_t);
    ucc_memory_type_t mt[2] = {UCC_MEMORY_TYPE_CUDA, UCC_MEMORY_TYPE_CUDA_MANAGED};
    ucc_coll_score_team_info_t info = {UCC_TL_NCCL_DEFAULT_SCORE, UCC_TL_TEAM_SIZE(team), UCC_TL_NCCL_SUPPORTED_COLLS, mt, 2, nccl_coll_init, nccl_alg_id_to_init};
    ucc_coll_score_t *score;
    ucc_status_t st = ucc_coll_score_build_default(b_team, UCC_TL_NCCL_DEFAULT_SCORE, nccl_coll_init, UCC_TL_NCCL_SUPPORTED_COLLS, mt, 2, &score);
    if (st != UCC_OK) return st;
    /* barrier on "host memory" (no buffers) gets the lowest score so a host TL wins when present */
    ucc_coll_score_add_range(score, UCC_COLL_TYPE_BARRIER, UCC_MEMORY_TYPE_HOST, 0, UCC_MSG_MAX, 1, nccl_coll_init, b_team);
    st = ucc_tl_apply_tune(&team->super, score, &info, "allgatherv:0-16k:@p2p#allgatherv:16k-1M:@bcopy#allgatherv:1M-inf:@bcast", NCCL_CTX(team)->cfg.super.super.score_str);
    if (st != UCC_OK) { ucc_coll_score_free(score); return st; }
    *score_p = score;
    return UCC_OK;
}

ucc_tl_iface_t ucc_tl_nccl = {
    .super = {.name = "nccl", .score = UCC_TL_NCCL_DEFAULT_SCORE},
    .tl_lib_config = {"TL_NCCL lib", "TL_NCCL_", tl_nccl_lib_config_table, sizeof(ucc_tl_lib_config_t), {NULL, NULL}},
    .tl_context_config = {"TL_NCCL context", "TL_NCCL_", tl_nccl_context_config_table, sizeof(ucc_tl_nccl_context_config_t), {NULL, NULL}},
    .lib = {nccl_lib_init, nccl_lib_finalize, nccl_lib_get_attr, nccl_lib_get_properties},
    .context = {nccl_ctx_create, NULL, nccl_ctx_destroy, nccl_ctx_get_attr, NULL, NULL, NULL},
    .team = {nccl_team_create_post, nccl_team_create_test, nccl_team_destroy, nccl_team_get_scores},
    .coll = {nccl_coll_init},
};
static void UCC_CTOR tl_nccl_register(void)
{ ucc_config_table_register(&ucc_tl_nccl.tl_lib_config); ucc_config_table_register(&ucc_tl_nccl.tl_context_config); ucc_tl_nccl.alg_info[ucc_coll_type_index(UCC_COLL_TYPE_ALLGATHERV)] = allgatherv_algs; }
