// maz_infer_initial.cu -- maz_infer_initial (include/maz_infer.h): the root inference of the search, one launch of
// k_initial_inference_small (infer_initial.cuh).  A translation unit of its own, so that the one-step and persistent instances
// of the small-batch stages (maz_infer.cu, maz_search.cu) are compiled exactly as before.
#include <cuda_runtime.h>

#include <string>

#define MAZ_HMMA_NO_KERNEL
#include "../../include/maz_infer.h"
#include "infer_initial.cuh"

using namespace maz;

namespace maz { int set_last_error(int code, const std::string &msg); }

// the small-batch chunks of the heads that the root variant consumes (mazero_b200/fused.py: value graph net layer 1, fc_policy.0,
// value graph net layer 2, fc_policy.3)
static const int kHeadChunks[4] = {27, 28, 30, 31};

extern "C" int maz_infer_initial(const maz_initial_desc *d, void *stream)
{
    if (!d) return set_last_error(1, "maz_infer_initial: NULL descriptor");
    if (!d->obs || !d->hidden || !d->value || !d->policy_logits || !d->rep_wpk || !d->rep_vec || !d->wpk || !d->vec)
        return set_last_error(1, "maz_infer_initial: NULL pointer");
    if (d->B <= 0 || d->N < 1 || d->N > 30 || d->A <= 0 || d->obs_dim <= 0)
        return set_last_error(1, "maz_infer_initial: bad shape (B >= 1, 1 <= N <= 30, A >= 1, obs_dim >= 1)");
    if (d->H != hmma::H || d->A > hmma::KA_WIDE || d->obs_dim > hmma::OBS_MAX)
        return set_last_error(3, "maz_infer_initial: unsupported shape (hidden 128, actions <= 128, obs_dim <= 640)");
    const int KA = (d->A + 15) / 16 * 16, kp = (d->obs_dim + 15) / 16 * 16;
    if (d->vec_floats <= 0 || d->vec_floats % 4 || d->o_vg < 0 || d->o_vg % 4 || d->o_pol < d->o_vg ||
        d->o_vg + 4 * hmma::GH + hmma::SUP * hmma::GH + 16 > d->vec_floats || d->o_pol + 3 * hmma::PH + KA > d->vec_floats)
        return set_last_error(1, "maz_infer_initial: bad parameter vector (vec_floats, o_vg, o_pol)");
    for (int c : kHeadChunks)
        if (d->chunk_bytes[c] == 0 || d->chunk_bytes[c] > hmma::SLOT_BYTES || d->chunk_bytes[c] % 16 || d->chunk_off[c] % 16)
            return set_last_error(1, "maz_infer_initial: bad weight chunk table");

    hmma::InitialArgs a = {};
    hmma::Desc &h = a.d;
    h.B = d->B; h.N = d->N; h.A = d->A; h.KA = KA; h.NAP = KA;
    h.Nt = d->N; h.cur = -1; h.inv_tau = 1.f;
    h.vec = d->vec + d->o_vg;                        // the heads' parameters only: value graph net, then fc_policy
    h.vec_floats = d->vec_floats - d->o_vg;
    h.o_rg = h.o_vg = 0;
    h.o_pol = d->o_pol - d->o_vg;
    a.obs = d->obs; a.hidden = d->hidden; a.value = d->value; a.logits = d->policy_logits;
    a.obs_dim = d->obs_dim; a.kp = kp;
    a.rep_vec = d->rep_vec; a.rep_floats = 2 * kp + 7 * hmma::H;
    const uint8_t *rw = static_cast<const uint8_t *>(d->rep_wpk);
    for (int k0 = 0; k0 < kp; k0 += 128) {           // mlp.0 column blocks [128][kc + 8], then mlp.3, mlp.6 [128][136]
        const int kc = kp - k0 < 128 ? kp - k0 : 128;
        a.chunk_src[a.nchunk] = rw;
        a.chunk_bytes[a.nchunk++] = 128u * (kc + hmma::PAD) * 2u;
        rw += 128u * (kc + hmma::PAD) * 2u;
    }
    for (int i = 0; i < 2; ++i) {
        a.chunk_src[a.nchunk] = rw;
        a.chunk_bytes[a.nchunk++] = hmma::SLOT_BYTES;
        rw += hmma::SLOT_BYTES;
    }
    for (int c : kHeadChunks) {
        a.chunk_src[a.nchunk] = static_cast<const uint8_t *>(d->wpk) + d->chunk_off[c];
        a.chunk_bytes[a.nchunk++] = d->chunk_bytes[c];
    }
    const size_t dyn = hmma::initial_smem_bytes(h.vec_floats, a.rep_floats);
    if (dyn > 227 * 1024) return set_last_error(3, "maz_infer_initial: parameters do not fit in shared memory");

    // opt the two instances into the device's maximum dynamic shared memory, once per device (as maz_infer_configure)
    static bool done[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_last_error(2, "no CUDA device available (libmaz_b200 has no CPU fallback)");
    cudaError_t e = cudaSuccess;
    if (dev < 0 || dev >= 64 || !done[dev]) {
        int optin = 227 * 1024;
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        const void *kernels[] = {(const void *)hmma::k_initial_inference_small<false>, (const void *)hmma::k_initial_inference_small<true>};
        for (const void *k : kernels) {
            cudaFuncAttributes fa;
            if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, k);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
        }
        if (e != cudaSuccess) return set_last_error(2, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
        if (dev >= 0 && dev < 64) done[dev] = true;
    }
    const int rpt = hmma::TM / d->N;
    const unsigned tiles = (unsigned)((d->B + rpt - 1) / rpt);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (KA > hmma::KA_NARROW) hmma::k_initial_inference_small<true><<<tiles, hmma::NTHREADS, dyn, s>>>(a);
    else hmma::k_initial_inference_small<false><<<tiles, hmma::NTHREADS, dyn, s>>>(a);
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_last_error(2, std::string("k_initial_inference_small: ") + cudaGetErrorString(e));
    return 0;
}
