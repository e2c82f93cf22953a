// mbarrier / bulk-copy (TMA 1-D) PTX wrappers, the data-dependent stage-release predicates, and the stack test and
// launch sequence shared by the four 8-bit tile kernels (hdr_merge_staged.cu, hdr_merge_staged_lut.cu,
// hdr_merge_stream.cu, hdr_merge_stream_lut.cu).
#pragma once

#include <algorithm>

#include "hdr_merge.cuh"

namespace cl {
namespace staged {

__device__ __forceinline__ uint32_t smem_addr(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_addr(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (-> launch error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) __trap();
    }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_addr(dst)),
        "l"(src), "r"(bytes), "r"(smem_addr(bar))
        : "memory");
}

// Releasing a shared-memory stage right after ISSUING the loads that read it is not enough: with
// 16 warps woken by the same bulk-copy completion the LSU queue can hold the loads for longer than
// the refill takes to arrive, and the refill then overtakes in-flight reads (seen at a ~1e-4 rate
// on full-size stacks, never on small ones).  The release is therefore predicated on a value
// computed FROM the loaded data -- always true (sums of weights / squares are never < 0, and a NaN
// compares false), but the compiler cannot prove it, so the mbarrier arrive is ordered after the
// arithmetic that consumed the loads and the scoreboard guarantees they have returned.
__device__ __forceinline__ bool consumed(double a, double b, double c) { return !((a + b) + c < 0.0); }
// Same idea on the integer pipe for the per-exposure release (the FP64 pipe is the busier one): the
// variance accumulators are sums of squares, i.e. >= +0 -- or NaN of EITHER sign (FP64 arithmetic passes
// an input NaN's sign and payload through, and x86 / NumPy's 0/0 is the negative quiet NaN, so an
// uncertainty image can hold one).  With m = OR of the three high words the test "m < 0x80000000 or
// m >= 0xFFF00000" is true for every such value (a set sign bit can only come from a NaN, whose high word is
// >= 0xFFF00000, and OR-ing more bits in keeps it there) and false only for negative finite numbers, which
// cannot occur: always true, never provable, NaN safe.
__device__ __forceinline__ bool consumed_nonneg(double a, double b, double c) {
    const uint32_t m = (uint32_t)(__double2hiint(a) | __double2hiint(b) | __double2hiint(c));
    return m + 0x00100000u < 0x80100000u;
}

// What every tile kernel needs of the stack: 8-bit DNs (256-row tables), C = 3 or 1 (mono runs as virtual RGB), at
// least one full 512-pixel tile, 32-bit sample indices, and the uncertainty of every exposure from an image
// (std_images) or of none (the STD table).  The flat's DN bytes are bulk-copied; its uncertainties are too when the
// kernel streams uncertainty images, the STD-table kernels load them per sample.
inline bool tile_stack(const MergeParams& p, bool std_images) {
    if ((p.C != 3 && p.C != 1) || p.bits != 256) return false;
    const int64_t n_samples = (int64_t)p.H * p.W * p.C;
    if (n_samples < kStagedTilePx * 3 || n_samples >= 0xFFFFFFFFll) return false;
    if (!std_images && !p.std_lut) return false;
    for (int k = 0; k < p.n; ++k)
        if ((p.std[k] != nullptr) != std_images) return false;
    return !p.flat_bytes || (aligned(p.flat, 16) && aligned(p.flat_std, std_images ? 16 : 8));
}

// The launch sequence of a tile kernel: [dark scan | work-list clear], the kernel on the full tiles (one CTA per SM, at
// most one per tile), the generic kernel on the ragged tail, [fix-up].  The single-pass kernels (p.stream_mode != 0)
// also file cancelled samples in the work list, so they always clear or fill it and always run the fix-up; the
// two-pass kernels use it only for the bad pixels of dark frames.  CL_ERR_WORKSPACE, with nothing enqueued, when the
// sequence needs the work list and the workspace held none.
template <typename Layout>
int launch_tile_kernel(const MergeParams& p, void (*kernel)(MergeParams, Layout, int), int threads, const Layout& L,
                       cudaStream_t stream) {
    const bool single_pass = p.stream_mode != 0;
    if ((single_pass || p.any_dark) && !p.hot_list) return CL_ERR_WORKSPACE;
    const int64_t n_samples = (int64_t)p.H * p.W * p.C;
    const int n_tiles = (int)(n_samples / (kStagedTilePx * 3));
    int st = CL_OK;
    if (p.any_dark) st = launch_dark_scan(p, stream);           // (the scan clears the list too)
    else if (single_pass) st = clear_hot_list(p, stream);
    if (st != CL_OK) return st;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total);
    if (e != cudaSuccess) return cuda_status(e);
    kernel<<<std::min(sm_count(), n_tiles), threads, L.total, stream>>>(p, L, n_tiles);
    st = launched();
    if (st != CL_OK) return st;
    // pixels past the last full tile (< 512) go through the generic kernel; both kernels run identical arithmetic
    const int64_t tail_first_sample = (int64_t)n_tiles * kStagedTilePx * 3;
    if (tail_first_sample < n_samples) {
        st = launch_merge_generic_range(p, tail_first_sample / 4, stream);
        if (st != CL_OK) return st;
    }
    return single_pass || p.any_dark ? launch_merge_fixup(p, stream) : CL_OK;
}

}  // namespace staged
}  // namespace cl
