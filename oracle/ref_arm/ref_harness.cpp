/* Reference arm harness (baseline only, NOT product code).
 *
 * openucx/ucc cannot be configured without autotools and UCX/UCS, so `bench.py --impl reference`
 * drives the reference's own sm_100 NVLS kernels - compiled UNMODIFIED from REFERENCE_DIR by build.sh - through the
 * stock host sequence of the reference's tl/cuda:
 *   setup     tl_cuda_nvls.c:296-700   (cuMulticastCreate on rank 0, POSIX fd + pidfd_getfd import, cuMemCreate,
 *                                       UC map, control memset, cuMulticastAddDevice, cuMulticastBindAddr, MC map;
 *                                       max_concurrent slots of NVLS_SYMMETRIC_SIZE + NVLS_CONTROL_SIZE)
 *   allreduce allreduce_nvls.c:59-137  (cudaMemcpyAsync src -> UC slot, post_allreduce_kernel(sm_count, threads),
 *                                       cudaMemcpyAsync UC slot -> dst, event)
 *   reduce_scatter  reduce_scatterv_nvls.c:17-104, allgather  allgatherv_nvls.c:17-95
 * with the reference's defaults (tl_cuda.c:55-66: 512 MB per slot, 4 CTAs x 1024 threads, 8 slots).
 * The OOB exchange (pid/fd allgather, barriers) is done by the Python caller over torch.distributed.
 * This file links nothing from the repo's own libraries. */
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <unistd.h>
#include <sys/syscall.h>
#include <sys/prctl.h>
#include "ucc/api/ucc.h"

extern "C" {
ucc_status_t post_allreduce_kernel(cudaStream_t stream, uint32_t sm_count, uint32_t threads, CUdeviceptr mc_base_addr,
                                   size_t src_size_bytes, CUdeviceptr mc_control_addr, CUdeviceptr uc_control_addr,
                                   uint64_t launch_counter, uint32_t rank, uint32_t tsize, ucc_datatype_t datatype);
ucc_status_t post_reduce_scatter_kernel(cudaStream_t stream, uint32_t sm_count, uint32_t threads, CUdeviceptr dst_ptr,
                                        CUdeviceptr mc_base_addr, CUdeviceptr mc_control_addr, CUdeviceptr uc_control_addr,
                                        uint64_t launch_counter, size_t offset, size_t count, ucc_datatype_t datatype,
                                        uint32_t tsize);
ucc_status_t post_allgatherv_kernel(cudaStream_t stream, uint32_t sm_count, uint32_t threads, CUdeviceptr src_ptr,
                                    CUdeviceptr mc_base_addr, size_t my_offset, size_t my_count, CUdeviceptr mc_control_addr,
                                    CUdeviceptr uc_control_addr, uint64_t launch_counter, uint32_t tsize);
}

#define NVLS_CONTROL_SIZE 1024 /* tl_cuda_coll.h:48 */
#define MAX_SLOTS 64

static struct {
    int      rank, size, device, slots;
    uint32_t sm_count, threads;
    size_t   symm_size, mc_size, gran, min_gran;
    CUmemGenericAllocationHandle mc_handle, mem_handle;
    CUdeviceptr uc_va, mc_va;
    int      mc_fd;
    uint64_t coll_ids[MAX_SLOTS];
    uint64_t seq;
} R;

#define DRV(call) do { CUresult _r = (call); if (_r != CUDA_SUCCESS) { const char *s = 0; cuGetErrorString(_r, &s); \
    fprintf(stderr, "[ref_arm] rank %d: %s failed: %s\n", R.rank, #call, s ? s : "?"); return -1; } } while (0)
#define RT(call) do { cudaError_t _r = (call); if (_r != cudaSuccess) { \
    fprintf(stderr, "[ref_arm] rank %d: %s failed: %s\n", R.rank, #call, cudaGetErrorString(_r)); return -1; } } while (0)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

extern "C" int ref_nvls_create(int rank, int size, int device, size_t symm_size, int slots, int sm_count, int threads)
{
    memset(&R, 0, sizeof(R));
    R.rank = rank; R.size = size; R.device = device; R.slots = slots; R.symm_size = symm_size;
    R.sm_count = sm_count; R.threads = threads; R.mc_fd = -1;
    if (slots > MAX_SLOTS) return -1;
    RT(cudaSetDevice(device));
    RT(cudaFree(0));
    int mc_ok = 0;
    DRV(cuDeviceGetAttribute(&mc_ok, CU_DEVICE_ATTRIBUTE_MULTICAST_SUPPORTED, device));
    if (!mc_ok) { fprintf(stderr, "[ref_arm] device %d has no multicast support\n", device); return -2; }
    CUmulticastObjectProp p; memset(&p, 0, sizeof(p));
    p.numDevices = size; p.size = (size_t)slots * (symm_size + NVLS_CONTROL_SIZE);
    p.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
    DRV(cuMulticastGetGranularity(&R.min_gran, &p, CU_MULTICAST_GRANULARITY_MINIMUM));
    DRV(cuMulticastGetGranularity(&R.gran, &p, CU_MULTICAST_GRANULARITY_RECOMMENDED));
    R.mc_size = align_up(p.size, R.gran);
    p.size = R.mc_size;
    if (rank == 0) {
        DRV(cuMulticastCreate(&R.mc_handle, &p));
        DRV(cuMemExportToShareableHandle(&R.mc_fd, R.mc_handle, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0));
        prctl(PR_SET_PTRACER, PR_SET_PTRACER_ANY);
    }
    return 0;
}

extern "C" int ref_nvls_local_fd(void) { return R.mc_fd; }

extern "C" int ref_nvls_import(int root_pid, int root_fd)
{
    if (R.rank == 0) return 0;
    int pidfd = (int)syscall(SYS_pidfd_open, root_pid, 0);
    if (pidfd < 0) { perror("[ref_arm] pidfd_open"); return -1; }
    int fd = (int)syscall(SYS_pidfd_getfd, pidfd, root_fd, 0);
    close(pidfd);
    if (fd < 0) { perror("[ref_arm] pidfd_getfd"); return -1; }
    DRV(cuMemImportFromShareableHandle(&R.mc_handle, (void *)(uintptr_t)fd, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR));
    close(fd);
    return 0;
}

extern "C" int ref_nvls_add_device(void)
{
    CUmemAllocationProp prop; memset(&prop, 0, sizeof(prop));
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = R.device;
    prop.requestedHandleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
    DRV(cuMemCreate(&R.mem_handle, R.mc_size, &prop, 0));
    CUmemAccessDesc ad; memset(&ad, 0, sizeof(ad));
    ad.location.type = CU_MEM_LOCATION_TYPE_DEVICE; ad.location.id = R.device; ad.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    DRV(cuMemAddressReserve(&R.uc_va, R.mc_size, R.min_gran, 0, 0));
    DRV(cuMemMap(R.uc_va, R.mc_size, 0, R.mem_handle, 0));
    DRV(cuMemSetAccess(R.uc_va, R.mc_size, &ad, 1));
    RT(cudaMemset2D((void *)(R.uc_va + R.symm_size), R.symm_size + NVLS_CONTROL_SIZE, 0, NVLS_CONTROL_SIZE, R.slots));
    RT(cudaDeviceSynchronize());
    DRV(cuMulticastAddDevice(R.mc_handle, R.device));
    return 0;
}

extern "C" int ref_nvls_bind(void)
{
    CUmemAccessDesc ad; memset(&ad, 0, sizeof(ad));
    ad.location.type = CU_MEM_LOCATION_TYPE_DEVICE; ad.location.id = R.device; ad.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    DRV(cuMulticastBindAddr(R.mc_handle, 0, R.uc_va, R.mc_size, 0));
    DRV(cuMemAddressReserve(&R.mc_va, R.mc_size, R.min_gran, 0, 0));
    DRV(cuMemMap(R.mc_va, R.mc_size, 0, R.mc_handle, 0));
    DRV(cuMemSetAccess(R.mc_va, R.mc_size, &ad, 1));
    return 0;
}

/* slot rotation as in tl_cuda_coll.h:168 (coll_id = seq_num % max_concurrent), per-slot launch counter as in
 * allreduce_nvls.c: team->nvls.coll_ids[task->coll_id]++ */
static inline void next_slot(CUdeviceptr *uc, CUdeviceptr *mc, CUdeviceptr *uc_ctl, CUdeviceptr *mc_ctl, uint64_t *launch)
{
    int    slot = (int)(R.seq++ % R.slots);
    size_t off  = (size_t)slot * (R.symm_size + NVLS_CONTROL_SIZE);
    *uc = R.uc_va + off; *mc = R.mc_va + off;
    *uc_ctl = *uc + R.symm_size; *mc_ctl = *mc + R.symm_size;
    *launch = R.coll_ids[slot]++;
}

extern "C" int ref_allreduce(const void *src, void *dst, size_t bytes, int dt, void *stream)
{
    cudaStream_t s = (cudaStream_t)stream;
    size_t kernel_size = align_up(bytes, 16 * (size_t)R.size);
    if (kernel_size > R.symm_size) return -3; /* the reference returns UCC_ERR_NOT_SUPPORTED -> next TL (tl_nccl) */
    CUdeviceptr uc, mc, ucc_, mcc; uint64_t lc;
    next_slot(&uc, &mc, &ucc_, &mcc, &lc);
    RT(cudaMemcpyAsync((void *)uc, src, bytes, cudaMemcpyDeviceToDevice, s));
    if (post_allreduce_kernel(s, R.sm_count, R.threads, mc, kernel_size, mcc, ucc_, lc, R.rank, R.size, (ucc_datatype_t)dt) != UCC_OK) return -1;
    RT(cudaMemcpyAsync(dst, (void *)uc, bytes, cudaMemcpyDeviceToDevice, s));
    return 0;
}

/* src: size * count_bytes, dst: count_bytes (this rank's block); units of the kernel are uint32 */
extern "C" int ref_reduce_scatter(const void *src, void *dst, size_t block_bytes, int dt, void *stream)
{
    cudaStream_t s = (cudaStream_t)stream;
    size_t total = block_bytes * R.size;
    if (total > R.symm_size || block_bytes % 16) return -3;
    CUdeviceptr uc, mc, ucc_, mcc; uint64_t lc;
    next_slot(&uc, &mc, &ucc_, &mcc, &lc);
    RT(cudaMemcpyAsync((void *)uc, src, total, cudaMemcpyDeviceToDevice, s));
    if (post_reduce_scatter_kernel(s, R.sm_count, R.threads, (CUdeviceptr)dst, mc, mcc, ucc_, lc, (block_bytes / 4) * R.rank, block_bytes / 4,
                                   (ucc_datatype_t)dt, R.size) != UCC_OK) return -1;
    return 0;
}

extern "C" int ref_allgather(const void *src, void *dst, size_t block_bytes, void *stream)
{
    cudaStream_t s = (cudaStream_t)stream;
    size_t total = block_bytes * R.size;
    if (total > R.symm_size || block_bytes % 16) return -3;
    CUdeviceptr uc, mc, ucc_, mcc; uint64_t lc;
    next_slot(&uc, &mc, &ucc_, &mcc, &lc);
    if (post_allgatherv_kernel(s, R.sm_count, R.threads, (CUdeviceptr)src, mc, (block_bytes / 4) * R.rank, block_bytes / 4, mcc, ucc_, lc, R.size) != UCC_OK) return -1;
    RT(cudaMemcpyAsync(dst, (void *)uc, total, cudaMemcpyDeviceToDevice, s));
    return 0;
}

extern "C" int ref_nvls_destroy(void)
{
    cudaDeviceSynchronize();
    if (R.mc_va) { cuMemUnmap(R.mc_va, R.mc_size); cuMemAddressFree(R.mc_va, R.mc_size); }
    if (R.uc_va) { cuMulticastUnbind(R.mc_handle, R.device, 0, R.mc_size); cuMemUnmap(R.uc_va, R.mc_size); cuMemAddressFree(R.uc_va, R.mc_size); }
    if (R.mem_handle) cuMemRelease(R.mem_handle);
    if (R.mc_handle) cuMemRelease(R.mc_handle);
    if (R.mc_fd >= 0) close(R.mc_fd);
    memset(&R, 0, sizeof(R));
    return 0;
}
