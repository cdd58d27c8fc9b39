// sm100.cuh — thin inline-PTX wrappers for the Blackwell (sm_100a) features the dense kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (TMEM alloc / mma / commit / ld), proxy fences.
// Bit layouts of the UMMA shared-memory and instruction descriptors follow the PTX ISA tables
// ("tcgen05 matrix descriptor", "instruction descriptor" for .kind::tf32).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace xb {
namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }

// ------------------------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// 1 in exactly one lane of the (fully converged) warp, 0 in the others
__device__ __forceinline__ uint32_t elect_one_pred() {
    uint32_t e;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(e));
    return e;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    // bounded: a protocol bug traps (launch error) instead of hanging the GPU
    uint32_t done = 0, spins = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!done && ++spins > (1u << 24)) __trap();
    }
}

// ------------------------------------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_dst), "l"((uint64_t)map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
// Predicated forms for a fully converged warp in which ONE lane (`elected`, from elect_one_pred) issues: the operands stay
// warp-uniform, so ptxas feeds the uniform-datapath instruction (UTMALDG / UTMASTG / UTCHMMA / UTCBAR) from uniform registers.
// Inside `if (lane == 0)` the same operands are per-thread registers and every such instruction is wrapped in an
// ELECT + R2UR.BROADCAST "waterfall" loop (~80 cycles each, measured on the tcgen05.mma stream).
__device__ __forceinline__ void tma_load_2d_if(uint32_t elected, uint32_t smem_dst, const CUtensorMap* map, int c0, int c1,
                                               uint32_t bar) {
    asm volatile(
        "{\n"
        ".reg .pred pe;\n"
        "setp.ne.b32 pe, %5, 0;\n"
        "@pe cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n"
        "}\n" ::"r"(smem_dst), "l"((uint64_t)map), "r"(c0), "r"(c1), "r"(bar), "r"(elected)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx_if(uint32_t elected, uint32_t bar, uint32_t bytes) {
    asm volatile(
        "{\n"
        ".reg .pred pe;\n"
        "setp.ne.b32 pe, %2, 0;\n"
        "@pe mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n"
        "}\n" ::"r"(bar), "r"(bytes), "r"(elected)
        : "memory");
}
__device__ __forceinline__ void tma_store_2d_commit_if(uint32_t elected, const CUtensorMap* map, uint32_t smem_src, int c0,
                                                       int c1) {
    asm volatile(
        "{\n"
        ".reg .pred pe;\n"
        "setp.ne.b32 pe, %4, 0;\n"
        "@pe cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];\n"
        "@pe cp.async.bulk.commit_group;\n"
        "}\n" ::"l"((uint64_t)map), "r"(c0), "r"(c1), "r"(smem_src), "r"(elected)
        : "memory");
}
// shared -> global tile store, tracked by the issuing thread's bulk async-group (commit_group / wait_group)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"((uint64_t)map),
                 "r"(c0), "r"(c1), "r"(smem_src)
                 : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (TMA / tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ tcgen05 / TMEM
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result_addr) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {            // the same warp that allocated
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], TF32 inputs, FP32 accumulate; issued by ONE thread.
__device__ __forceinline__ void mma_tf32_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// predicated forms for a converged warp with one issuing lane (see tma_load_2d_if)
__device__ __forceinline__ void mma_tf32_ss_if(uint32_t elected, uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p, pe;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.ne.b32 pe, %5, 0;\n"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(elected)
        : "memory");
}
__device__ __forceinline__ void mma_commit_if(uint32_t elected, uint32_t bar) {
    asm volatile(
        "{\n"
        ".reg .pred pe;\n"
        "setp.ne.b32 pe, %1, 0;\n"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
        "}\n" ::"r"(bar), "r"(elected)
        : "memory");
}
// all previously issued tcgen05.mma of this thread complete -> one arrival on the mbarrier
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 columns of 32-bit: thread i of the warp receives lane (row) base+i, columns c..c+31.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor, SWIZZLE_128B (the layout TMA writes with CU_TENSOR_MAP_SWIZZLE_128B):
//   bits [0,14) start address >> 4 | [16,30) leading byte offset >> 4 | [32,46) stride byte offset >> 4 |
//   [46,48) version = 1 | [61,64) layout type = 2 (SWIZZLE_128B)
// K-major operand : rows of 128 B (32 tf32 along K); SBO = 1024 B between 8-row groups; LBO unused.
// MN-major operand: rows of 128 B (32 tf32 along M/N), one row per K index; LBO = bytes between consecutive
//                   32-element M/N blocks; SBO = bytes between 8-row K groups.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                             uint32_t layout_type) {
    uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout_type << 61;
    return d;
}
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return umma_desc(smem_addr, lbo_bytes, sbo_bytes, 2u);
}
// MN-major 32-bit (tf32) operands must use layout type 1, SWIZZLE_128B_BASE32B: 32-byte chunks of a 128-byte row are
// XOR-ed with (row & 3) (TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B); the atom is 4 K-rows x 128 B, so one K = 8 MMA
// spans two atoms: SBO = 512 B between them, LBO = bytes between consecutive 32-element M/N blocks.
__device__ __forceinline__ uint64_t umma_desc_sw128_base32(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return umma_desc(smem_addr, lbo_bytes, sbo_bytes, 1u);
}
// Instruction descriptor for .kind::tf32, fp32 accumulate: c_format F32 (1) at [4,6), a/b format TF32 (2) at [7,10) /
// [10,13), a/b major (0 = K, 1 = MN) at 15 / 16, N >> 3 at [17,23), M >> 4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// x = hi + lo with hi exactly representable in TF32 (round-to-nearest); lo = x - hi is exact in fp32.
// cvt.rna.tf32.f32 (nearest, ties away from zero) is emulated in SASS as add 0x1000 / Inf-NaN guard (FSETP + SEL) / mask: the
// guard is dropped here — the operands are finite activations, weights and gradients — which leaves IADD + LOP3 + FADD per
// element instead of five instructions (the operand warps of the dense kernels are instruction-bound); bit-identical to
// cvt.rna for every finite x below 2^128 - 2^104.
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
    lo = x - hi;
}

__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float4 v) {
    // no "memory" clobber: ordered against the other volatile asm (loads, fences, barriers) but plain C++ loads of
    // read-only tables (bias, head weights) may be scheduled across it
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
}
__device__ __forceinline__ float2 lds64(uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts64(uint32_t addr, float x, float y) {
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(x), "f"(y));
}
__device__ __forceinline__ void bar_sync_named(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void bar_arrive_named(int id, int nthreads) {   // signals without waiting (release ordering)
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace sm100

// ------------------------------------------------------------------------------------------------ host: tensor maps
typedef CUresult (*XbEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline XbEncodeTiledFn xb_encode_tiled_fn() {
    static XbEncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (XbEncodeTiledFn)ptr;
    }
    return fn;
}

// fp32 row-major [rows][cols] (row pitch `ld` floats), box = [box_rows][box_cols], SWIZZLE_128B when box_cols == 32.
// swizzle: 0 none, 1 = SWIZZLE_128B (16-byte chunks), 2 = SWIZZLE_128B_ATOM_32B (32-byte chunks)
static inline bool xb_make_map_f32_2d(CUtensorMap* map, const float* base, int64_t rows, int64_t cols, int64_t ld,
                                      int box_rows, int box_cols, int swizzle) {
    XbEncodeTiledFn fn = xb_encode_tiled_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle == 1 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : (swizzle == 2 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_NONE),
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

}  // namespace xb
