/* C launch interface of the tl/nvl device code (sm_100a).
 *
 * Every collective is ONE kernel that moves data between the team members'
 * symmetric heaps over NVLink (plain ld/st on peer-mapped addresses or
 * multimem.* on the NVLS multicast mapping), reduces in registers with the
 * datatype/operator templates, and synchronises with flag words that live in
 * the peers' heaps — no host involvement between phases, no separate reduce
 * or copy kernel, no NCCL. */
#ifndef UCC_TL_NVL_KERNELS_H_
#define UCC_TL_NVL_KERNELS_H_
#include <stdint.h>
#include <stddef.h>
#include <cuda_runtime_api.h>

#define NVL_MAX_PEERS  16
#define NVL_MAX_BLOCKS 320
#define NVL_LL_MAX     (1024 * 1024)         /* bytes per rank in the one-shot (latency) region */
#define NVL_P2P_MAX_CTAS 16                  /* lanes of a point-to-point channel */
#define NVL_P2P_SLOTS    4                   /* chunks in flight per channel */
#define NVL_P2P_CHUNK    (256 * 1024)
#define NVL_P2P_CHAN_BYTES (NVL_P2P_SLOTS * NVL_P2P_CHUNK)
#define NVL_P2P_LANE_BYTES (NVL_P2P_CHUNK / NVL_P2P_MAX_CTAS)   /* 16 KB: what one CTA moves per ring step */

/* control block at offset 0 of every rank's heap */
typedef struct nvl_ctrl {
    uint32_t flags[NVL_MAX_BLOCKS][NVL_MAX_PEERS];    /* [block][src rank]: barrier signals written by peers */
    uint32_t epoch;                                   /* barrier epoch of this rank (advanced by the last block of a kernel) */
    uint32_t done_blocks;                             /* blocks of the running kernel that reached the end */
    uint32_t rsvd[NVL_MAX_BLOCKS - 2];
    uint32_t ll_flags[NVL_MAX_BLOCKS][NVL_MAX_PEERS]; /* one-shot arrival flags */
    uint32_t ll_seq[NVL_MAX_BLOCKS];                  /* one-shot sequence (parity selects the buffer) */
    uint32_t error;                                   /* set by a kernel whose spin timed out */
    uint32_t pad[31];
    uint64_t mc_arrive[NVL_MAX_BLOCKS];               /* NVLS barrier counters (incremented through the multicast mapping) */
    uint64_t mc_epoch[NVL_MAX_BLOCKS];
    /* point-to-point channels (kernels/nvl_p2p.cu), [peer][lane]; all counters count chunks and only ever grow */
    uint32_t p2p_head[NVL_MAX_PEERS][NVL_P2P_MAX_CTAS]; /* in the RECEIVER's heap: chunks peer has delivered into my ring (written by peer) */
    uint32_t p2p_ack[NVL_MAX_PEERS][NVL_P2P_MAX_CTAS];  /* in the SENDER's heap: chunks peer has drained from its ring (written by peer) */
    uint32_t p2p_tx[NVL_MAX_PEERS][NVL_P2P_MAX_CTAS];   /* local: chunks I produced for peer so far */
    uint32_t p2p_rx[NVL_MAX_PEERS][NVL_P2P_MAX_CTAS];   /* local: chunks I consumed from peer so far */
    /* rendezvous (zero-copy) messages: the sender stores straight into the receiver's buffer */
    uint32_t p2p_rz_done[NVL_MAX_PEERS];                /* in the RECEIVER's heap: zero-copy messages of peer that have completely landed (written by peer) */
    uint32_t p2p_rz_blocks[NVL_MAX_PEERS];              /* local: CTAs of the running push kernel towards peer that are finished */
} nvl_ctrl_t;

#define NVL_CTRL_SIZE  (128 * 1024)
#define NVL_LL_OFFSET  NVL_CTRL_SIZE
#define NVL_LL_SIZE    (2 * NVL_MAX_PEERS * NVL_LL_MAX)
#define NVL_P2P_OFFSET (NVL_LL_OFFSET + NVL_LL_SIZE)       /* per source rank one channel ring */
#define NVL_P2P_SIZE   (NVL_MAX_PEERS * NVL_P2P_CHAN_BYTES)
#define NVL_DATA_OFFSET (NVL_P2P_OFFSET + NVL_P2P_SIZE)

typedef struct nvl_team_dev {
    int      rank, size;
    char    *heap[NVL_MAX_PEERS]; /* unicast mapping of every member's heap in my address space */
    char    *mc_heap;             /* multicast mapping of the same offsets, or NULL */
    size_t   data_size;           /* bytes of the data region */
    uint64_t timeout_ns;          /* spin budget before a kernel gives up */
    uint32_t *host_err;           /* host-mapped word: set when a spin timed out */
} nvl_team_dev_t;

typedef enum { NVL_DT_I8, NVL_DT_I16, NVL_DT_I32, NVL_DT_I64, NVL_DT_U8, NVL_DT_U16, NVL_DT_U32, NVL_DT_U64,
               NVL_DT_F16, NVL_DT_F32, NVL_DT_F64, NVL_DT_BF16, NVL_DT_C64, NVL_DT_C128, NVL_DT_LAST } nvl_dt_t;
typedef enum { NVL_OP_SUM, NVL_OP_PROD, NVL_OP_MAX, NVL_OP_MIN, NVL_OP_LAND, NVL_OP_LOR, NVL_OP_LXOR, NVL_OP_BAND, NVL_OP_BOR,
               NVL_OP_BXOR, NVL_OP_AVG, NVL_OP_LAST } nvl_op_t;

/* what the staged reduction kernel produces */
typedef enum {
    NVL_RED_ALLREDUCE,       /* every rank gets the whole reduced vector */
    NVL_RED_REDUCE_SCATTER,  /* rank r gets block r (counts/offsets in elements) */
    NVL_RED_REDUCE           /* only `root` gets the reduced vector */
} nvl_red_kind_t;

/* zero-copy view of the members' USER buffers (CUDA IPC mappings, or plain pointers inside one process), resolved
 * by the host-side buffer exchange (tl_nvl_direct.c) right before the launch */
typedef struct nvl_direct {
    const char *src[NVL_MAX_PEERS];
    char       *dst[NVL_MAX_PEERS];
} nvl_direct_t;
typedef enum { NVL_DIRECT_NONE = 0, NVL_DIRECT_FULL = 1, NVL_DIRECT_DST = 2 } nvl_direct_mode_t;

typedef struct nvl_red_args {
    nvl_team_dev_t team;
    const void    *src;
    void          *dst;
    size_t         count;       /* elements of the full input vector */
    int            dt, op, kind, root;
    int            use_nvls;    /* reduce in the switch (multimem.ld_reduce) instead of pulling */
    size_t         rs_offset[NVL_MAX_PEERS]; /* REDUCE_SCATTER(V): element offset / count of each rank's block */
    size_t         rs_count[NVL_MAX_PEERS];
    int            sched;       /* step-structured kernel: 1 = ring, 2 = recursive halving / doubling */
    int            direct;      /* nvl_direct_mode_t: FULL = read peers' src and write peers' dst in place (no staging at all);
                                   DST = staged/NVLS reduction whose result goes straight into every member's dst (no copy-out) */
    nvl_direct_t   d;
} nvl_red_args_t;

/* the zero-copy reduction kernel wants the pointer tables relative to the caller: entry i = my i-th right neighbour (i = 0: me) */
static inline void nvl_direct_rotate(nvl_red_args_t *a)
{
    nvl_direct_t r;
    int i, n = a->team.size, me = a->team.rank;
    for (i = 0; i < NVL_MAX_PEERS; i++) { r.src[i] = i < n ? a->d.src[(me + i) % n] : 0; r.dst[i] = i < n ? a->d.dst[(me + i) % n] : 0; }
    a->d = r;
}

/* generic staged exchange: allgather(v), alltoall(v), bcast, gather, scatter */
#define NVL_XCHG_TABLE_BYTES 256 /* published offset table in front of the staged payload */
#define NVL_XCHG_LOOKUP ((size_t)-1)
typedef struct nvl_xchg_args {
    nvl_team_dev_t team;
    const void    *src;          /* local bytes staged into my heap (phase A) */
    size_t         src_bytes;    /* how many bytes of src are staged (0: nothing to publish) */
    size_t         stage_off[NVL_MAX_PEERS]; /* published table: byte offset of the block meant for peer p inside my staged data */
    void          *dst;
    /* phase B: from peer p copy pull_bytes[p] starting at pull_off[p] (offset inside p's staged data,
     * or NVL_XCHG_LOOKUP: read it from p's published table at index `rank`) to dst + dst_off[p];
     * the own block (p == rank) is copied straight from src + self_off */
    size_t         pull_off[NVL_MAX_PEERS], pull_bytes[NVL_MAX_PEERS], dst_off[NVL_MAX_PEERS];
    size_t         self_off;
    int            publish_table;
    int            use_mc;       /* NVLS push: phase A multimem.st's my bytes to offset push_off of EVERY heap, phase B reads my own heap */
    size_t         push_off;
    int            ring;         /* allgather(v) over neighbour links only: pull_off[] is the common heap layout, N-1 pull steps */
    int            ring_order[NVL_MAX_PEERS], ring_pos; /* topology-aware visit order of the ring (ring_order[ring_pos] == rank) */
    int            direct;       /* pull from the peers' user buffers (d.src[p]) instead of their staged copies */
    nvl_direct_t   d;
} nvl_xchg_args_t;

/* zero-copy push exchange (kernels/nvl_push.cu): my block for member p = send_bytes[p] bytes at src + send_off[p], stored at
 * dst_of[p] + land_off[p] (dst_of[p] = p's destination buffer mapped here; dst_of[rank] = my own) */
typedef struct nvl_push_args {
    nvl_team_dev_t team;
    const void    *src;
    size_t         send_off[NVL_MAX_PEERS], send_bytes[NVL_MAX_PEERS], land_off[NVL_MAX_PEERS];
    char          *dst_of[NVL_MAX_PEERS];
    int            lookup;       /* alltoallv: only the receiver knows where a block lands; every rank publishes recv_off[] (offset of
                                    source p's block inside MY dst) at the start of its heap data region and senders read entry [rank] */
    size_t         recv_off[NVL_MAX_PEERS];
} nvl_push_args_t;

/* two-member active-set broadcast = send / recv (kernels/nvl_p2p.cu) */
typedef struct nvl_p2p_args {
    nvl_team_dev_t team;
    void          *buf;
    size_t         bytes;
    int            peer;   /* team rank of the other side */
    int            send;   /* 1: I am the root (sender), 0: receiver */
    int            mode;   /* nvl_p2p_mode_t */
    uint32_t       rz_seq; /* NVL_P2P_PUSH / NVL_P2P_WAIT: index of this zero-copy message between the pair (in post order) */
    char          *remote; /* NVL_P2P_PUSH: the receiver's buffer, mapped here */
    uint64_t       spin_ns;/* budget of a wait for the peer (0: no deadline) */
} nvl_p2p_args_t;
/* NVL_P2P_RING: through the pair's heap channel (eager: the sender never needs the receiver's address);
 * NVL_P2P_PUSH / NVL_P2P_WAIT: rendezvous - the receiver published its buffer, the sender's kernel stores into it directly and
 * bumps p2p_rz_done in the receiver's heap; the receiver's stream only carries a one-warp kernel that waits for that counter */
typedef enum { NVL_P2P_RING = 0, NVL_P2P_PUSH, NVL_P2P_WAIT } nvl_p2p_mode_t;
#define NVL_P2P_PUSH_MAX_CTAS 64

#ifdef __cplusplus
extern "C" {
#endif
int          nvl_p2p_lanes(size_t bytes);
int          nvl_p2p_push_ctas(size_t bytes);
cudaError_t  nvl_launch_p2p(const nvl_p2p_args_t *a, int nthreads, cudaStream_t s);
size_t       nvl_dt_size(int dt);
int          nvl_dt_supports_op(int dt, int op);
int          nvl_nvls_supports(int dt, int op);
/* latency path: one-shot push allreduce, bytes <= NVL_LL_MAX */
cudaError_t  nvl_launch_allreduce_oneshot(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s);
/* bandwidth path: staged two-shot (P2P pull or NVLS) for allreduce / reduce_scatter(v) / reduce */
cudaError_t  nvl_launch_reduce_staged(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s);
/* latency path of reduce_scatter(v): one-shot push of every block to its owner, blocks <= NVL_LL_MAX */
cudaError_t  nvl_launch_reduce_scatter_oneshot(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s);
/* zero-copy two-shot: every rank reduces its slice straight out of the members' src buffers into their dst buffers */
cudaError_t  nvl_launch_reduce_direct(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s);
/* ring / recursive halving-doubling allreduce and reduce_scatter(v) through the heaps (a->sched), single round */
cudaError_t  nvl_launch_reduce_steps(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s);
/* staged NVLS allreduce with three heap buffers: staging / in-switch reduction / copy-out of consecutive chunks overlap */
cudaError_t  nvl_launch_reduce_pipe(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s);
/* in-place NVLS allreduce on symmetric user memory: a->d.src[0] / a->d.dst[0] = local addresses inside my heap mapping */
cudaError_t  nvl_launch_reduce_symm(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s);
/* allgather into a symmetric destination: a->src/src_bytes = my block, a->dst = local address of the gathered buffer in my heap, a->push_off = my offset */
cudaError_t  nvl_launch_allgather_symm(const nvl_xchg_args_t *a, int nblocks, int nthreads, cudaStream_t s);
cudaError_t  nvl_launch_exchange(const nvl_xchg_args_t *a, int nblocks, int nthreads, cudaStream_t s);
cudaError_t  nvl_launch_exchange_push(const nvl_push_args_t *a, int nblocks, int nthreads, cudaStream_t s);
/* same exchange driven by the TMA engine (cp.async.bulk through shared memory): one-warp CTAs */
cudaError_t  nvl_launch_exchange_push_bulk(const nvl_push_args_t *a, int nblocks, cudaStream_t s);
cudaError_t  nvl_launch_barrier(const nvl_team_dev_t *t, cudaStream_t s);
cudaError_t  nvl_launch_self_copy(void *dst, const void *src, size_t bytes, int nblocks, int nthreads, cudaStream_t s); /* team of one */
cudaError_t  nvl_launch_self_copy_bulk(void *dst, const void *src, size_t bytes, int nblocks, cudaStream_t s);      /* same, TMA engine; 16-byte aligned pointers */
cudaError_t  nvl_launch_ctrl_init(void *heap_base, cudaStream_t s);
#ifdef __cplusplus
}
#endif
#endif
