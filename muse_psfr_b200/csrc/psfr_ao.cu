// Strehl ratio of every PSF of the fused pipeline (DESIGN.md 5.5).
//
//  otf_sum_kernel : sum of the telescope OTF over the full N x N grid, once per context.
//  strehl_kernel  : S = (raw sample at the PSF origin) / otf_sum for every PSF of a chunk.
//
// Why one sample is enough: the row and column passes of run_pruned_psf form the unnormalised 2-D DFT of
// exp(-c D) * OTF_tel (c = (2 pi / lambda_nm)^2 / 2, so exp(-c D_unit) = exp(-D_lambda / 2)), and the column pass
// writes S[img][x][j] = scale * (-1)^(kc + k_j) * P[k_j][kc].  Sample x = j = 40 has kc = k_j = 0 (pixel 20 of
// set_lambda_tables has bilinear weight exactly 1 there), so its sign is +1 and P[0][0] is the plain sum over the
// grid: S[img][40][40] = scale * sum_d sum_f OTF_tel(f) exp(-D_d(f) / 2) with scale = 1 / ndir in field-mean mode
// and 1 per plane in field mode.  The constant between the sample and the Strehl numerator is therefore 1 (the
// mean over the directions in field-mean mode), with OTF_tel in the units of d_otf (its origin is 1 / N^2).
#include "psfr_internal.h"

namespace psfr {

constexpr int kOtfSumThreads = 1024;

// d_otf holds the half-plane rows o = 0 .. N/2 (row N/2 the zero frequency, row 0 the frequency -N/2, both their
// own mirror) and a zero pad row; row o in 1 .. N/2 - 1 stands for itself and its point mirror N - o.  Thread t
// adds a fixed strided subset in order, then a fixed tree: the same bits on every run.
__global__ void __launch_bounds__(kOtfSumThreads) otf_sum_kernel(const double* __restrict__ otf, int kN, double* out) {
    __shared__ double red[kOtfSumThreads];
    const int t = threadIdx.x, kNH = kN / 2;
    const size_t live = (size_t)(kNH + 1) * kN;
    double s = 0.0;
    for (size_t i = t; i < live; i += kOtfSumThreads) {
        const int row = (int)(i / kN);
        const double v = __ldg(otf + i);
        s += (row == 0 || row == kNH) ? v : 2.0 * v;
    }
    red[t] = s;
    for (int w = kOtfSumThreads / 2; w > 0; w >>= 1) {
        __syncthreads();
        if (t < w) red[t] += red[t + w];
    }
    if (t == 0) *out = red[0];
}

int run_otf_sum(Ctx* c, cudaStream_t s) {
    double* d_sum = c->d_misc;   // scratch: nothing else lives in d_misc at context creation
    otf_sum_kernel<<<1, kOtfSumThreads, 0, s>>>(c->d_otf, c->N, d_sum);
    PSFR_LAUNCH_CHECK(c);
    PSFR_CUDA(c, cudaMemcpyAsync(&c->otf_sum, d_sum, sizeof(double), cudaMemcpyDeviceToHost, s));
    PSFR_CUDA(c, cudaStreamSynchronize(s));
    if (!(c->otf_sum > 0)) return set_error(c, PSFR_E_CUDA, "telescope OTF sum is %g", c->otf_sum);
    return PSFR_OK;
}

__global__ void strehl_kernel(const double* __restrict__ samp, int nimg, double otf_sum, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nimg) out[i] = __ldg(samp + (size_t)i * kNS * kNS + kPSF * kNS + kPSF) / otf_sum;
}

int run_strehl(Ctx* c, int nimg, double* out_dev, cudaStream_t s) {
    strehl_kernel<<<(nimg + 127) / 128, 128, 0, s>>>(c->d_samp, nimg, c->otf_sum, out_dev);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

}  // namespace psfr
