"""Reference arm driver (baseline only): the reference's own tl/cuda NVLS kernels, compiled unmodified into
oracle/_ref/libref_tlcuda.so by build.sh, driven through the stock host sequence (see ref_harness.cpp), plus the two
other transports the reference's score map would pick on this box:

  * team size 1            -> tl/self: cudaMemcpyAsync src -> dst   (reference tl/self/tl_self_coll.c copy path)
  * padded size > NVLS_SYMMETRIC_SIZE (512 MB default, tl_cuda.c:55) or no multicast
                           -> tl/nccl: ncclAllReduce               (reference tl_nccl_coll.c; here torch's NCCL binding)

Nothing of the repo's own library is imported or loaded here."""
import ctypes
import os

import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "..", "_ref", "libref_tlcuda.so")

# ucc_datatype_t predefined ids (reference src/ucc/api/ucc.h: UCC_PREDEFINED_DT(id) = id << 3); the ucc.h the arm is built
# from is pinned by its sha256 in tests/golden/ref_arm_sources.sha256
UCC_DT = {torch.int32: 2 << 3, torch.int64: 3 << 3, torch.float32: 11 << 3, torch.bfloat16: 13 << 3}


class RefTlCuda:
    """tl/cuda NVLS team of the reference: one multicast-bound symmetric region of `slots` x (symm_size + 1 KB)."""

    def __init__(self, rank, world, device, symm_size=512 << 20, slots=8, sm_count=4, threads=1024):
        self.rank, self.world, self.symm_size = rank, world, symm_size
        self.lib = ctypes.CDLL(LIB)
        L = self.lib
        L.ref_nvls_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int]
        L.ref_nvls_import.argtypes = [ctypes.c_int, ctypes.c_int]
        L.ref_allreduce.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]
        L.ref_reduce_scatter.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]
        L.ref_allgather.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        self.ok = False
        st = L.ref_nvls_create(rank, world, device, symm_size, slots, sm_count, threads)
        info = [None] * world
        dist.all_gather_object(info, (os.getpid(), L.ref_nvls_local_fd(), st))
        if any(i[2] != 0 for i in info):
            return
        st = L.ref_nvls_import(info[0][0], info[0][1])
        st = st or L.ref_nvls_add_device()
        if not self._agree(st):
            return
        st = L.ref_nvls_bind()
        if not self._agree(st):
            return
        self.ok = True

    def _agree(self, st):
        flags = [None] * self.world
        dist.all_gather_object(flags, int(st))
        return all(f == 0 for f in flags)

    def allreduce(self, src, dst, stream):
        return self.lib.ref_allreduce(src.data_ptr(), dst.data_ptr(), src.numel() * src.element_size(), UCC_DT[src.dtype], stream.cuda_stream)

    def reduce_scatter(self, src, dst, stream):
        return self.lib.ref_reduce_scatter(src.data_ptr(), dst.data_ptr(), dst.numel() * dst.element_size(), UCC_DT[src.dtype], stream.cuda_stream)

    def allgather(self, src, dst, stream):
        return self.lib.ref_allgather(src.data_ptr(), dst.data_ptr(), src.numel() * src.element_size(), stream.cuda_stream)

    def destroy(self):
        self.lib.ref_nvls_destroy()
