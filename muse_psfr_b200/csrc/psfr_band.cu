// Band images: filter-weighted sums of the wavelength planes of every image set (DESIGN.md 5.6).
//
//  band_kernel : one thread per (set, pixel).  It walks the nlam planes of its set in ascending k, reading each
//                pixel once, and carries all PSFR_MAX_BANDS accumulators in registers:
//                acc[b] = fma(w[b][k], C[k][pix], acc[b]) from acc = 0, then B[b][pix] = acc[b] / W_b.
//                Unused bands have zero weights; the array is fully unrolled so it never goes to local memory.
//                The weights come through shared memory in tiles of kBandTile wavelengths, stored k-major
//                ([nlam][PSFR_MAX_BANDS], zero-padded), so every thread of a CTA reads the same word (broadcast).
#include <algorithm>
#include "psfr_internal.h"

namespace psfr {

constexpr int kBandThreads = 256;
constexpr int kBandTile = 64;   // wavelengths per weight tile: 64 x 16 doubles = 8 KB of shared memory

__global__ void __launch_bounds__(kBandThreads)
band_kernel(const double* __restrict__ in, long long nset, int nlam, int npix, int nband,
            const double* __restrict__ w, BandSums wsum, double* __restrict__ out) {
    __shared__ double ws[kBandTile * PSFR_MAX_BANDS];
    const long long total = nset * npix;
    const long long stride = (long long)gridDim.x * kBandThreads;
    // the trip count is the same for every thread of a CTA: the tile loop below synchronises
    for (long long base = (long long)blockIdx.x * kBandThreads; base < total; base += stride) {
        const long long i = base + threadIdx.x;
        const bool live = i < total;
        const long long set = live ? i / npix : 0;
        const int pix = live ? (int)(i - set * npix) : 0;
        const double* src = in + set * nlam * (long long)npix + pix;
        double acc[PSFR_MAX_BANDS];
#pragma unroll
        for (int b = 0; b < PSFR_MAX_BANDS; ++b) acc[b] = 0.0;
        for (int k0 = 0; k0 < nlam; k0 += kBandTile) {
            const int nk = min(kBandTile, nlam - k0);
            __syncthreads();
            for (int j = threadIdx.x; j < nk * PSFR_MAX_BANDS; j += kBandThreads)
                ws[j] = __ldg(w + (size_t)k0 * PSFR_MAX_BANDS + j);
            __syncthreads();
            if (live)
                for (int k = 0; k < nk; ++k) {
                    const double v = __ldg(src + (long long)(k0 + k) * npix);
#pragma unroll
                    for (int b = 0; b < PSFR_MAX_BANDS; ++b) acc[b] = fma(ws[k * PSFR_MAX_BANDS + b], v, acc[b]);
                }
        }
        if (live) {
            double* dst = out + set * nband * (long long)npix + pix;
#pragma unroll
            for (int b = 0; b < PSFR_MAX_BANDS; ++b)
                if (b < nband) dst[(long long)b * npix] = acc[b] / wsum.w[b];
        }
    }
}

int run_band(Ctx* c, long long nset, int nlam, int npix, int nband, const BandSums& sums, const double* in_dev,
             double* out_dev, cudaStream_t s) {
    const long long total = nset * npix;
    const long long want = (total + kBandThreads - 1) / kBandThreads;
    const int blocks = (int)std::min<long long>(want, (long long)c->sm_count * 16);
    band_kernel<<<blocks, kBandThreads, 0, s>>>(in_dev, nset, nlam, npix, nband, c->d_bandw, sums, out_dev);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

}  // namespace psfr
