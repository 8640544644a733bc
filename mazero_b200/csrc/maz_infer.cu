// maz_infer.cu -- fused network forward for the search (tcgen05 / TMEM / bulk-TMA, sm_100a).
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <string>

#include "../../include/maz_infer.h"
#include "umma.cuh"
#include "infer_fused.cuh"
#include "infer_hmma.cuh"
#include "infer_twin.cuh"

using namespace maz;
using namespace maz::umma;

extern "C" const char *maz_last_error(void);
namespace maz { int set_last_error(int code, const std::string &msg); bool pdl_enabled(); int pdl_mask(); }
namespace maz { namespace twin {     // maz_infer_wide.cu: the wide instance of the two-tiles-in-flight kernel
const void *wide_kernel();
cudaError_t launch_wide(const cudaLaunchConfig_t &cfg, const maz_infer_desc &d);
} }

// ---------------------------------------------------------------------------------------------------------
// Self-test kernel: one GEMM stage exactly as the fused kernel runs it.
//   threads: 128 (4 warps); thread r owns token row r.
__global__ void __launch_bounds__(128, 1) k_dbg_umma_gemm(const float *__restrict__ a, const __nv_bfloat16 *__restrict__ wp,
                                                          float *__restrict__ out, int N, int K)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar_w, bar_mma;
    __shared__ uint32_t tmem_base_s;
    uint8_t *sA = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);   // 1 KB aligned (swizzled tiles)
    uint8_t *sW = smem + operand_bytes(128, K);           // N x K bf16
    const int tid = threadIdx.x, warp = tid >> 5;

    if (tid == 0) {
        mbar_init(&bar_w, 1);
        mbar_init(&bar_mma, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_base_s, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (tid == 0) {
        mbar_expect_tx(&bar_w, operand_bytes(N, K));
        bulk_g2s(sW, wp, operand_bytes(N, K), &bar_w);
    }
    // activations: fp32 global row -> bf16 operand layout
    for (int k8 = 0; k8 < K / 8; ++k8) {
        const float4 lo = *reinterpret_cast<const float4 *>(a + (size_t)tid * K + k8 * 8);
        const float4 hi = *reinterpret_cast<const float4 *>(a + (size_t)tid * K + k8 * 8 + 4);
        __nv_bfloat162 p0 = __floats2bfloat162_rn(lo.x, lo.y), p1 = __floats2bfloat162_rn(lo.z, lo.w);
        __nv_bfloat162 p2 = __floats2bfloat162_rn(hi.x, hi.y), p3 = __floats2bfloat162_rn(hi.z, hi.w);
        uint4 v;
        v.x = *reinterpret_cast<uint32_t *>(&p0);
        v.y = *reinterpret_cast<uint32_t *>(&p1);
        v.z = *reinterpret_cast<uint32_t *>(&p2);
        v.w = *reinterpret_cast<uint32_t *>(&p3);
        *reinterpret_cast<uint4 *>(sA + operand_chunk_off(tid, k8, K, 128)) = v;
    }
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
        mbar_wait(&bar_w, 0);
        tc_fence_after();
        issue_gemm(tmem_base, smem_u32(sA), K, 0, smem_u32(sW), K, 0, K, N, false);
        mma_commit(&bar_mma);
    }
    mbar_wait(&bar_mma, 0);
    tc_fence_after();
    const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);
    for (int c = 0; c < N; c += 16) {
        float v[16];
        tmem_ld16(lane_base + c, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) out[(size_t)tid * N + c + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 256);
}

extern "C" int maz_dbg_umma_gemm(const float *a, const void *w_packed, float *out, int n, int k, void *stream)
{
    if (!a || !w_packed || !out || n % 16 || k % 16 || n < 16 || n > 256 || k < 16 || k > 512)
        return set_last_error(1, "maz_dbg_umma_gemm: bad arguments");
    const size_t dyn = operand_bytes(128, k) + operand_bytes(n, k) + 2048;
    cudaError_t e = cudaFuncSetAttribute(k_dbg_umma_gemm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return set_last_error(2, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    k_dbg_umma_gemm<<<1, 128, dyn, static_cast<cudaStream_t>(stream)>>>(a, static_cast<const __nv_bfloat16 *>(w_packed), out, n, k);
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_last_error(2, std::string("k_dbg_umma_gemm: ") + cudaGetErrorString(e));
    return 0;
}

extern "C" int maz_infer_configure(int vec_floats, int ka);

extern "C" int maz_infer_recurrent(const maz_infer_desc *d, void *stream)
{
    if (!d) return set_last_error(1, "maz_infer_recurrent: NULL descriptor");
    if (d->B <= 0 || d->N <= 0 || d->N > 32 || d->A <= 0 || d->A > hmma::KA_WIDE || d->KA % 16 || d->KA < d->A || d->KA > hmma::KA_WIDE ||
        d->NAP != d->KA)
        return set_last_error(3, "maz_infer_recurrent: unsupported shape (agents <= 32, actions <= 128)");
    if (d->tc_layout == 0 && d->A > hmma::KA_NARROW)
        return set_last_error(3, "maz_infer_recurrent: the first-generation kernel (tc_layout 0) supports at most 48 actions; use tc_layout 1");
    if (!d->pool || !d->actions || !d->next_hidden || !d->reward || !d->value || !d->probs || !d->beta || !d->wpk || !d->vec)
        return set_last_error(1, "maz_infer_recurrent: NULL tensor");
    if (d->vec_floats <= 0 || d->vec_floats % 4) return set_last_error(1, "maz_infer_recurrent: vec_floats must be a positive multiple of 4");
    const bool tw = d->tc_layout == 1, wide = d->KA > hmma::KA_NARROW;
    if (d->tc_layout != 0 && !tw) return set_last_error(1, "maz_infer_recurrent: unknown tc_layout");
    if (tw && (d->o_oh_in <= 0 || d->o_oh_dyn <= 0 || d->o_oh_rg <= 0 || d->o_oh_rg + d->A * 64 > d->vec_floats))
        return set_last_error(1, "maz_infer_recurrent: tc_layout 1 needs the one-hot weight tables behind vec");
    const size_t dyn = tw ? twin::smem_bytes() : fused::smem_bytes(d->KA, d->vec_floats);
    if (dyn > 227 * 1024) return set_last_error(3, "maz_infer_recurrent: parameters do not fit in shared memory");
    if (int rc = maz_infer_configure(d->vec_floats, d->KA)) return rc;
    const int roots_per_tile = 4 * (32 / d->N);
    int tiles = (d->B + roots_per_tile - 1) / roots_per_tile;
    if (tw) tiles = (tiles + 1) / 2;                      // a CTA of the second-generation kernel owns two tiles
    // programmatic dependent of the tree kernel: TMEM allocation, barrier set-up and the weight / parameter
    // streaming overlap the predecessor's tail; the epilogue warps call griddepcontrol.wait before they read it
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)tiles);
    cfg.blockDim = dim3(fused::NTHREADS);
    cfg.dynamicSmemBytes = dyn;
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (maz::pdl_mask() & 1) ? 1 : 0;
    cudaError_t e = !tw ? cudaLaunchKernelEx(&cfg, fused::k_recurrent_inference, *d)
                    : wide ? twin::launch_wide(cfg, *d)
                           : cudaLaunchKernelEx(&cfg, twin::k_recurrent_inference_twin<false>, *d);
    if (e != cudaSuccess) return set_last_error(2, std::string("k_recurrent_inference: ") + cudaGetErrorString(e));
    return 0;
}

// Small-batch variant (infer_hmma.cuh): 32-row tiles on warp-level MMAs.  `d->wpk` / chunk tables must be in the
// row-major padded layout of mazero_b200/fused.py::HmmaParams.  KA > 48 launches the wide instance.
extern "C" int maz_infer_small_nq(void) { return hmma::NQ; }

// Opt both kernels into the device's maximum dynamic shared memory, once per device.  (cudaFuncSetAttribute SETS the limit: a
// per-launch "raise when larger than last time" scheme lowered it when another caller had configured a smaller network in
// between, and the next launch of the larger one failed with cudaErrorInvalidValue.)
extern "C" int maz_infer_configure(int vec_floats, int ka)
{
    (void)vec_floats; (void)ka;
    static bool done[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_last_error(2, "no CUDA device available (libmaz_b200 has no CPU fallback)");
    if (dev < 0 || dev >= 64 || done[dev]) return 0;
    int optin = 227 * 1024;
    cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    const void *kernels[] = {(const void *)hmma::k_recurrent_inference_small<false>, (const void *)hmma::k_recurrent_inference_small<true>,
                             (const void *)fused::k_recurrent_inference, (const void *)twin::k_recurrent_inference_twin<false>,
                             twin::wide_kernel()};
    cudaError_t e = cudaSuccess;
    for (const void *k : kernels) {
        cudaFuncAttributes fa;
        if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, k);     // (the opt-in limit covers static + dynamic)
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
    }
    if (e != cudaSuccess) return set_last_error(2, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    done[dev] = true;
    return 0;
}

extern "C" int maz_infer_recurrent_small(const maz_infer_desc *d, void *stream)
{
    if (!d) return set_last_error(1, "maz_infer_recurrent_small: NULL descriptor");
    if (d->B <= 0 || d->N <= 0 || d->N > 32 || d->A <= 0 || d->A > hmma::KA_WIDE || d->KA % 16 || d->KA < d->A || d->KA > hmma::KA_WIDE ||
        d->NAP != d->KA)
        return set_last_error(3, "maz_infer_recurrent_small: unsupported shape (agents <= 32, actions <= 128)");
    if (!d->pool || !d->actions || !d->next_hidden || !d->reward || !d->value || !d->probs || !d->beta || !d->wpk || !d->vec)
        return set_last_error(1, "maz_infer_recurrent_small: NULL tensor");
    if (d->vec_floats <= 0 || d->vec_floats % 4) return set_last_error(1, "maz_infer_recurrent_small: vec_floats must be a positive multiple of 4");
    for (int c = 0; c < MAZ_INFER_NCHUNK; ++c)
        if (d->chunk_bytes[c] == 0 || d->chunk_bytes[c] > hmma::SLOT_BYTES || d->chunk_bytes[c] % 16 || d->chunk_off[c] % 16)
            return set_last_error(1, "maz_infer_recurrent_small: bad weight chunk table");
    const size_t dyn = hmma::smem_bytes(d->vec_floats);
    if (dyn > 227 * 1024) return set_last_error(3, "maz_infer_recurrent_small: parameters do not fit in shared memory");
    if (int rc = maz_infer_configure(d->vec_floats, d->KA)) return rc;
    const int rpt = hmma::TM / d->N;
    const int tiles = (d->B + rpt - 1) / rpt;
    // optionally a programmatic dependent of the tree kernel (MAZ_PDL bit 0): barrier set-up, the parameter copy and the first
    // weight chunks overlap the predecessor's tail; the compute warps call griddepcontrol.wait before they touch its outputs
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)tiles);
    cfg.blockDim = dim3(hmma::NTHREADS);
    cfg.dynamicSmemBytes = dyn;
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (maz::pdl_mask() & 1) ? 1 : 0;
    cudaError_t e = d->KA > hmma::KA_NARROW ? cudaLaunchKernelEx(&cfg, hmma::k_recurrent_inference_small<true>, *d)
                                            : cudaLaunchKernelEx(&cfg, hmma::k_recurrent_inference_small<false>, *d);
    if (e != cudaSuccess) return set_last_error(2, std::string("k_recurrent_inference_small: ") + cudaGetErrorString(e));
    return 0;
}
