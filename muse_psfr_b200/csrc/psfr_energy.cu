// Encircled energy of every image: EE at given radii, the total, and the radii at given fractions of the total
// (psfr_encircled_energy, psfr_compute_energy; definition in DESIGN.md section 5.4).
#include <math_constants.h>
#include "psfr_internal.h"
#include "ee_geometry.h"

namespace psfr {

namespace {

constexpr int kEeWarps = 4;
constexpr int kEeMaxIter = 200;           // bisection alone needs 38 steps from 29 px down to 1e-10 px
constexpr double kEeTol = 1e-10;          // bracket width [px] at which the radius solve stops
// resident CTAs per SM the kernel is compiled for: at 4 it fits in 116 registers without spills (at the
// default bound ptxas picks 80 and spills)
#ifndef PSFR_EE_MINBLOCKS
#define PSFR_EE_MINBLOCKS 4
#endif

// EE(r) of one image in shared memory, and with kDeriv dEE/dr = sum img * (circle length inside the pixel).
// Every lane walks its pixels lane, lane + 32, ... in order and adds the value of each pixel wholly inside the
// disc; the pixels the circle crosses are listed (lst, in that order) and their overlaps summed afterwards by
// all lanes at once, so that the few lanes holding one do not serialise the warp.  Rows the disc cannot reach
// are skipped (they would add nothing).  The warp adds the lanes' partial sums with the xor-shuffle tree: all
// lanes end with the same bits, and once the circle contains every pixel nothing is listed and the additions
// are exactly those of r = +inf (TOTAL).
template <bool kDeriv>
__device__ __forceinline__ double ee_eval(const double* img, unsigned short* lst, int ny, int nx, double y0,
                                          double x0, double r, double* dee) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const double r2 = r * r;
    int p0, p1;
    ee::row_window(y0, r, ny, &p0, &p1);
    const int i0 = p0 * nx, i1 = p1 * nx;
    double t = 0.0;
    int nst = 0;
    int i = (i0 & ~31) + lane;
    int p = i / nx, q = i - p * nx;
    for (; i - lane < i1; i += 32) {
        bool cross = false;
        if (i >= i0 && i < i1) {
            double near2, far2;
            ee::pixel_dist2(p - y0, q - x0, &near2, &far2);
            if (r2 >= far2) t += img[i];
            else cross = r2 > near2;
        }
        const unsigned m = __ballot_sync(0xffffffffu, cross);
        if (cross) lst[nst + __popc(m & lt)] = (unsigned short)i;
        nst += __popc(m);
        for (q += 32; q >= nx; q -= nx) ++p;
    }
    __syncwarp();
    double s = 0.0, g = 0.0;
    for (int j = lane; j < nst; j += 32) {
        const int k = lst[j], pk = k / nx;
        const double v = img[k];
        if (kDeriv) {
            double arc;
            s = fma(v, ee::pixel_area_arc(pk - y0, (k - pk * nx) - x0, r, &arc), s);
            g = fma(v, arc, g);
        } else {
            s = fma(v, ee::pixel_area(pk - y0, (k - pk * nx) - x0, r), s);
        }
    }
    __syncwarp();
    t += s;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        t += __shfl_xor_sync(0xffffffffu, t, o);
        if (kDeriv) g += __shfl_xor_sync(0xffffffffu, g, o);
    }
    if (kDeriv) *dee = g;
    return t;
}

// One warp per image, images handed out by a global counter (the radius solve takes a varying number of
// steps).  par: radii [nrad] then fractions [nfrac]; centres [nimg][2] (row, column) or nullptr for
// (ny / 2, nx / 2).  out [nimg][nrad + 1 + nfrac]: EE at each radius, TOTAL, radius at each fraction.
__global__ void __launch_bounds__(kEeWarps * 32, PSFR_EE_MINBLOCKS)
ee_kernel(const double* __restrict__ imgs, int nimg, int ny, int nx, const double* __restrict__ centres,
          const double* __restrict__ par, int nrad, int nfrac, double* __restrict__ out, int* __restrict__ next_image) {
    extern __shared__ double sm[];
    const int npx = ny * nx, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rec = nrad + 1 + nfrac;
    double* img = sm + (size_t)warp * npx;
    unsigned short* lst = reinterpret_cast<unsigned short*>(sm + (size_t)kEeWarps * npx) + (size_t)warp * npx;
#pragma unroll 1
    for (;;) {
        int image = 0;
        if (lane == 0) image = atomicAdd(next_image, 1);
        image = __shfl_sync(0xffffffffu, image, 0);
        if (image >= nimg) return;
        __syncwarp();
        const double* src = imgs + (size_t)image * npx;
        for (int i = lane; i < npx; i += 32) img[i] = src[i];
        __syncwarp();
        const double y0 = centres ? centres[2 * (size_t)image] : (double)(ny / 2);
        const double x0 = centres ? centres[2 * (size_t)image + 1] : (double)(nx / 2);
        double* o = out + (size_t)image * rec;
        const double total = ee_eval<false>(img, lst, ny, nx, y0, x0, CUDART_INF, nullptr);
        for (int k = 0; k < nrad; ++k) {
            const double e = ee_eval<false>(img, lst, ny, nx, y0, x0, par[k], nullptr);
            if (lane == 0) o[k] = e;
        }
        if (lane == 0) o[nrad] = total;
        __syncwarp();
        // farthest pixel corner: EE there is TOTAL, bit for bit
        const double fy = fmax(y0 + 0.5, ny - 0.5 - y0), fx = fmax(x0 + 0.5, nx - 0.5 - x0);
        const double rmax = sqrt(fy * fy + fx * fx);
        // r where EE crosses frac * TOTAL from below (the smallest such r when no pixel is negative).  The bracket
        // [lo, hi] keeps EE(lo) < target <= EE(hi); it starts from the tabulated radii, and the first trial point
        // interpolates inside it.  Newton steps inside the bracket, bisection when Newton leaves it or does not
        // halve the step of two iterations back, and a step of tol / 2 across the root once Newton's steps are
        // that small, which closes the bracket.
        for (int j = 0; j < nfrac; ++j) {
            double res = CUDART_NAN;
            if (total > 0.0) {
                const double target = par[nrad + j] * total;
                double lo, hi, elo, ehi;
                ee::fraction_bracket(par, o, nrad, target, rmax, total, &lo, &elo, &hi, &ehi);
                double x = lo + (target - elo) / (ehi - elo) * (hi - lo);
                if (!(x > lo && x < hi)) x = 0.5 * (lo + hi);
                double dx = hi - lo, dxold = dx;
                for (int it = 0; it < kEeMaxIter && hi - lo > kEeTol; ++it) {
                    double d;
                    const double f = ee_eval<true>(img, lst, ny, nx, y0, x0, x, &d) - target;
                    if (f >= 0.0) hi = x; else lo = x;
                    if (hi - lo <= kEeTol) break;
                    double xn = d > 0.0 ? x - f / d : lo;
                    const bool newton = xn > lo && xn < hi && fabs(xn - x) <= 0.5 * fabs(dxold);
                    dxold = dx;
                    if (newton) {
                        if (fabs(xn - x) < 0.5 * kEeTol) xn = f >= 0.0 ? x - 0.5 * kEeTol : x + 0.5 * kEeTol;
                    } else {
                        xn = 0.5 * (lo + hi);
                    }
                    dx = xn - x;
                    x = xn;
                }
                res = hi;
            }
            if (lane == 0) o[nrad + 1 + j] = res;
        }
        __syncwarp();
    }
}

}  // namespace

int run_ee(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* centres_dev, int nrad, int nfrac,
           double* out_dev, cudaStream_t s) {
    // per warp: the image, and the list of pixels the circle crosses
    const size_t smem = (size_t)kEeWarps * ny * nx * (sizeof(double) + sizeof(unsigned short));
    if (smem > 200 * 1024)
        return set_error(c, PSFR_E_UNSUPPORTED, "image %dx%d too large for the encircled-energy kernel", ny, nx);
    if (int rc = ensure_dynamic_smem(c, ee_kernel, smem)) return rc;
    int grid = (nimg + kEeWarps - 1) / kEeWarps;
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ee_kernel, kEeWarps * 32, smem) != cudaSuccess ||
        per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    const int resident = c->sm_count * per_sm;
    if (grid > resident) grid = resident;
    PSFR_CUDA(c, cudaMemsetAsync(c->d_counter + 3, 0, sizeof(int), s));
    ee_kernel<<<grid, kEeWarps * 32, smem, s>>>(img_dev, nimg, ny, nx, centres_dev, c->d_eepar, nrad, nfrac, out_dev,
                                                 c->d_counter + 3);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

}  // namespace psfr
