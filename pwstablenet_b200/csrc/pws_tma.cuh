// pws_tma.cuh -- TMA (cp.async.bulk.tensor) + mbarrier plumbing of libpwswarp for sm_100a.
//
// Thin inline-PTX wrappers (SASS: UTMALDG / UTMASTG / UTMAREDG, SYNCS.*) and the host-side
// tensor-map encoder.  libcuda is not linked: cuTensorMapEncodeTiled is resolved through
// cudaGetDriverEntryPoint at first use.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace pws {
namespace tma {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// make mbarrier.init visible to the async proxy (TMA completes transactions on them)
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// order generic-proxy shared-memory writes before a following async-proxy (TMA store / reduce) read
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: the warp sleeps in hardware until the phase completes (or the hint
// expires) instead of burning issue slots in a poll loop
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
    return ok != 0;
}
// non-blocking: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// try_wait comes back after a few tens of nanoseconds whatever the hint says (ncu: ~80 retries per waited tile, 4 % of the
// backward's instructions).  A pause between retries (PWS_WAIT_NS / PWS_WAIT_RELAXED_NS > 0) was measured: the backward does
// not change (0.429 ms with 0 / 64 / 150 ns: the scheduler serves the retries only when nobody else is ready) and the
// forward loses 1-2 %, so the default is none.
#ifndef PWS_WAIT_NS
#define PWS_WAIT_NS 0
#endif
#ifndef PWS_WAIT_RELAXED_NS
#define PWS_WAIT_RELAXED_NS 0
#endif
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) { if (PWS_WAIT_NS) __nanosleep(PWS_WAIT_NS); }
}
// for the roles that run stages ahead (producer, scouts)
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) { if (PWS_WAIT_RELAXED_NS) __nanosleep(PWS_WAIT_RELAXED_NS); }
}

__device__ __forceinline__ void prefetch_desc(const CUtensorMap *tm)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

// global -> shared box load, completion counted in bytes on `bar`; out-of-range elements arrive as zero
__device__ __forceinline__ void load_3d(void *dst, const CUtensorMap *tm, uint64_t *bar, int c0, int c1, int c2)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void load_4d(void *dst, const CUtensorMap *tm, uint64_t *bar, int c0, int c1, int c2, int c3)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void load_2d(void *dst, const CUtensorMap *tm, uint64_t *bar, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// ---- L2 eviction priorities ------------------------------------------------------------------
// Streaming operands are loaded evict_first, accumulators that are revisited (grad_input between its
// zero-fill and its last RED) are written evict_last, so the stream does not push them out of L2.
__device__ __forceinline__ uint64_t policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_normal()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void load_3d_hint(void *dst, const CUtensorMap *tm, uint64_t *bar, int c0, int c1, int c2, uint64_t pol)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)), "l"(pol)
        : "memory");
}
__device__ __forceinline__ void load_4d_hint(void *dst, const CUtensorMap *tm, uint64_t *bar, int c0, int c1, int c2, int c3, uint64_t pol)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4, %5}], [%6], %7;"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar)), "l"(pol)
        : "memory");
}
// fire-and-forget float add (no L2 policy operand: the default priority needs none, and a policy costs the SASS two
// R2UR per instruction for the descriptor)
__device__ __forceinline__ void red_add_f32(float *p, float v)
{
    asm volatile("red.relaxed.gpu.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void st_f32_hint(float *p, float v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_zero_v4_hint(float4 *p, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %1, %1, %1}, %2;" ::"l"(p), "f"(0.0f), "l"(pol) : "memory");
}

// shared -> global box store / f32 add-reduction (out-of-range elements are dropped); bulk-group completion
__device__ __forceinline__ void store_3d(const CUtensorMap *tm, const void *src, int c0, int c1, int c2)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];"
        ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(src))
        : "memory");
}
__device__ __forceinline__ void reduce_add_3d(const CUtensorMap *tm, const void *src, int c0, int c1, int c2)
{
    asm volatile(
        "cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2, %3}], [%4];"
        ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(src))
        : "memory");
}
__device__ __forceinline__ void commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups still have to READ their shared-memory source
template <int N> __device__ __forceinline__ void wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N> __device__ __forceinline__ void wait_group() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int threads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

// ---- host ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// General fp32 tiled map: `rank` dims (fastest first), element strides of dims 1..rank-1, box extents.
// Requirements (the encoder rejects violations): base 16-byte aligned, every stride a multiple of 4
// elements, box[0] a multiple of 4, every box extent <= 256.
// elem_bytes = 4 (fp32) or 2 (dtype16: CU_TENSOR_MAP_DATA_TYPE_FLOAT16 / _BFLOAT16): for 16-bit elements the
// alignment rules read "8 elements" instead of "4".
inline bool encode_elems(CUtensorMap *tm, CUtensorMapDataType dt, int elem_bytes, const void *base, int rank, const uint64_t *dims,
                         const uint64_t *strides_elems, const uint32_t *box,
                         CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B)
{
    EncodeTiledFn fn = encode_fn();
    if (!fn || rank < 1 || rank > 5) return false;
    cuuint64_t d[5], st[4];
    cuuint32_t b[5], es[5];
    for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; es[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) st[i] = strides_elems[i] * (uint64_t)elem_bytes;
    return fn(tm, dt, (cuuint32_t)rank, const_cast<void *>(base), d, st, b, es,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
inline bool encode_f32(CUtensorMap *tm, const void *base, int rank, const uint64_t *dims, const uint64_t *strides_elems,
                       const uint32_t *box, CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B)
{
    return encode_elems(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, rank, dims, strides_elems, box, promo);
}

// rank-3 tiled map over (d0 fastest, d1, d2) with element strides s1, s2 (s0 == 1); elem = 4 bytes.
// Requirements (checked by the caller): base 16-byte aligned, s1*4 and s2*4 multiples of 16, box0*4 multiple of 16,
// every box extent <= 256.
inline bool encode_3d_f32(CUtensorMap *tm, const void *base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1, uint64_t s2,
                          uint32_t b0, uint32_t b1, uint32_t b2, CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B)
{
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {s1 * 4, s2 * 4};
    cuuint32_t box[3] = {b0, b1, b2};
    cuuint32_t es[3] = {1, 1, 1};
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void *>(base), dims, strides, box, es,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tma
}  // namespace pws
