// sm_100a building blocks: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM / commit), descriptors.
// Hand-written PTX wrappers; no CUTLASS.  Encodings follow the PTX ISA "tcgen05" chapter:
//   shared-memory matrix descriptor (64 bit) and instruction descriptor (32 bit) for .kind::f16.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ----------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// ----------------------------------------------------------------------------- TMA loads
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
        "%6}], [%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// ----------------------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // whole warp, ncols pow2 >= 32
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives once all previously issued tcgen05 ops of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i gets TMEM lane (base_lane + i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
        "[%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle (rows of 64 bf16 = 128 B, 8-row / 1024 B
// swizzle atoms stacked along M/N): start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major) |
// SBO>>4 [32,46) = 1024 B | version=1 [46,48) | layout=SWIZZLE_128B(2) [61,64).
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

// Instruction descriptor for kind::f16: D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1, A/B K-major (bits 15,16 = 0),
// N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ __forceinline__ uint32_t make_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
           (static_cast<uint32_t>(M >> 4) << 24);
}
// The same with fp16 operands: A/B format 0 = f16 (fp32 accumulation either way).
__host__ __device__ __forceinline__ uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}
// Instruction descriptor for operand type T (bf16 or f16)
template <typename T> __host__ __device__ __forceinline__ uint32_t make_idesc(int M, int N);
template <> __host__ __device__ __forceinline__ uint32_t make_idesc<bf16>(int M, int N) { return make_idesc_bf16(M, N); }
template <> __host__ __device__ __forceinline__ uint32_t make_idesc<f16>(int M, int N) { return make_idesc_f16(M, N); }

}  // namespace tc

// ----------------------------------------------------------------------------- host: tensor-map encode
// cuTensorMapEncodeTiled is fetched through the runtime (no link-time dependency on libcuda, so the library
// also loads on a machine without a driver).
typedef CUresult (*cab_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
cab_encode_tiled_fn cab_get_encode_tiled();

// Tensor map of 2-byte elements (elem_dtype CABINET_BF16 or CABINET_F16), rank <= 5, 128B swizzle, zero OOB fill.
// dims/strides innermost first; strides in BYTES for dims 1..rank-1 (dim 0 is contiguous).
int cab_make_tmap_2b(CUtensorMap* map, int elem_dtype, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box,
                     CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B);
static inline int cab_make_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                                     const uint64_t* strides_bytes, const uint32_t* box,
                                     CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                     CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
    return cab_make_tmap_2b(map, CABINET_BF16, base, rank, dims, strides_bytes, box, promo, swizzle);
}

namespace tc {
// ----------------------------------------------------------------------------- TMA stores (smem -> global, bulk group)
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N> __device__ __forceinline__ void bulk_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
}  // namespace tc

namespace tc {
// 32 lanes x 32 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
}  // namespace tc

namespace tc {
// Warp-uniform issue helpers: EVERY lane of the MMA warp executes these with identical operands (so the compiler can
// keep descriptors in uniform registers and emit straight-line code); the tcgen05 instruction itself is predicated on
// `leader` (one elected lane) inside the asm.
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred)::"memory");
    return pred;
}
__device__ __forceinline__ void umma_bf16_if(uint32_t leader, uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                             uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void umma_commit_if(uint32_t leader, uint64_t* bar) {
    asm volatile(
        "{\n\t"
        ".reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(leader)
        : "memory");
}
}  // namespace tc

namespace tc {
// Explicit shared-space accesses (32-bit shared addresses).  Pointers derived from the dynamic smem base through
// integer alignment arithmetic lose their address space and compile to generic LD/ST (slow path); these do not.
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ float2 lds64f(uint32_t a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const uint4& v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
}  // namespace tc
