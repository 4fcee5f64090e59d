// convolve_final_psf (psfrec.py:874-930) by FFT, the way the reference itself does it
// (scipy.signal.fftconvolve(psf, K[None], 'same'), :916-917, :927-928).
//
// A 40x40 plane convolved with a 41x41 kernel has an 80x80 linear support, so one 80x80
// circular convolution is exact; 'same' keeps rows/columns 20..59.  One CTA per image, all
// data in shared memory:
//   rows    : two real rows packed in one 80-point complex transform, untangled into the
//             half spectrum W[y][kx], kx = 0..40
//   columns : forward transform, times the kernel spectrum (precomputed once per draw for the
//             tip-tilt kernel, once per wavelength for the MUSE kernel), inverse transform,
//             keeping output rows 20..59
//   rows    : Hermitian pair -> two real rows, columns 20..59 kept
// and the same again for the second kernel (zero-padded linear convolution, cropped after
// each: not associative, so the two are applied in sequence like the reference).
// This costs ~0.5 M FP64 operations per image against 5.4 M FMAs for the direct sum.
//
// 80-point transform = 16 x 5 across threads: n = 5 n1 + n2, k = k1 + 16 k2;
//   pass A (thread = line, n2): radix-16 (4 x 4) over n1 in registers, times w80^(n2 k1)
//   pass B (thread = line, k1): radix-5 over n2
#include "psfr_internal.h"

namespace psfr {

namespace {

constexpr int kF = 80;            // transform length
constexpr int kFH = kF / 2 + 1;   // 41 half-spectrum columns
constexpr int kConvThreads = 256;

__device__ __forceinline__ double2 cxadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 cxsub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 cxmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 cxconj(double2 a) { return make_double2(a.x, -a.y); }
// a * (SGN * i)
template <int SGN>
__device__ __forceinline__ double2 mul_si(double2 a) {
    return SGN > 0 ? make_double2(-a.y, a.x) : make_double2(a.y, -a.x);
}
// a * (c + SGN i s)
template <int SGN>
__device__ __forceinline__ double2 mul_cs(double2 a, double c, double s) {
    return SGN > 0 ? make_double2(a.x * c - a.y * s, a.x * s + a.y * c)
                   : make_double2(a.x * c + a.y * s, a.y * c - a.x * s);
}

// X[k] = sum_n x[n] exp(SGN 2 pi i n k / 4)
template <int SGN>
__device__ __forceinline__ void dft4s(double2& x0, double2& x1, double2& x2, double2& x3) {
    const double2 a = cxadd(x0, x2), b = cxsub(x0, x2), c = cxadd(x1, x3), d = mul_si<SGN>(cxsub(x1, x3));
    x0 = cxadd(a, c);
    x2 = cxsub(a, c);
    x1 = cxadd(b, d);
    x3 = cxsub(b, d);
}

template <int SGN>
__device__ __forceinline__ void dft5s(double2& x0, double2& x1, double2& x2, double2& x3, double2& x4) {
    const double c1 = 0.30901699437494742410, c2_ = -0.80901699437494742410;
    const double s1 = 0.95105651629515357212, s2 = 0.58778525229247312917;
    const double2 t1 = cxadd(x1, x4), t2 = cxadd(x2, x3), t3 = cxsub(x1, x4), t4 = cxsub(x2, x3);
    const double2 a1 = make_double2(x0.x + c1 * t1.x + c2_ * t2.x, x0.y + c1 * t1.y + c2_ * t2.y);
    const double2 a2 = make_double2(x0.x + c2_ * t1.x + c1 * t2.x, x0.y + c2_ * t1.y + c1 * t2.y);
    const double2 b1 = mul_si<SGN>(make_double2(s1 * t3.x + s2 * t4.x, s1 * t3.y + s2 * t4.y));
    const double2 b2 = mul_si<SGN>(make_double2(s2 * t3.x - s1 * t4.x, s2 * t3.y - s1 * t4.y));
    x0 = make_double2(x0.x + t1.x + t2.x, x0.y + t1.y + t2.y);
    x1 = cxadd(a1, b1);
    x4 = cxsub(a1, b1);
    x2 = cxadd(a2, b2);
    x3 = cxsub(a2, b2);
}

// 16-point transform, v[4a + b] = x[4a + b] in; on exit position 4c + d holds X[c + 4d]
template <int SGN>
__device__ __forceinline__ void dft16s(double2* v) {
    const double h = 0.70710678118654752440, cA = 0.92387953251128673848, sA = 0.38268343236508978178;
#pragma unroll
    for (int b = 0; b < 4; ++b) dft4s<SGN>(v[b], v[4 + b], v[8 + b], v[12 + b]);   // position 4c + b = y[b][c]
    // y[b][c] *= w16^(b c)
    v[4 * 1 + 1] = mul_cs<SGN>(v[4 * 1 + 1], cA, sA);     // e = 1
    v[4 * 1 + 2] = mul_cs<SGN>(v[4 * 1 + 2], h, h);       // e = 2
    v[4 * 1 + 3] = mul_cs<SGN>(v[4 * 1 + 3], sA, cA);     // e = 3
    v[4 * 2 + 1] = mul_cs<SGN>(v[4 * 2 + 1], h, h);       // e = 2
    v[4 * 2 + 2] = mul_si<SGN>(v[4 * 2 + 2]);             // e = 4
    v[4 * 2 + 3] = mul_cs<SGN>(v[4 * 2 + 3], -h, h);      // e = 6
    v[4 * 3 + 1] = mul_cs<SGN>(v[4 * 3 + 1], sA, cA);     // e = 3
    v[4 * 3 + 2] = mul_cs<SGN>(v[4 * 3 + 2], -h, h);      // e = 6
    v[4 * 3 + 3] = mul_cs<SGN>(v[4 * 3 + 3], -cA, -sA);   // e = 9
#pragma unroll
    for (int c = 0; c < 4; ++c) dft4s<SGN>(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
}
__device__ __forceinline__ constexpr int k1_of_pos(int pos) { return (pos >> 2) + 4 * (pos & 3); }

// Every pass works in place.  Forward (decimation in time, n = 5 n1 + n2, k = k1 + 16 k2):
//   pass A (thread n2): 16 slots 5 n1 + n2 -> radix-16 -> Y[n2][k1] in slot 5 k1 + n2
//   pass B (thread k1): 5 slots 5 k1 + n2, times w80^(n2 k1) -> radix-5 -> X[k1 + 16 k2] in slot 5 k1 + k2
// so a natural-order line comes out with X[k] in slot P(k) = 5 (k mod 16) + k / 16.
// Inverse of a P-ordered line (decimation in frequency, n = a + 16 b in slot 5 a + b, k = c + 5 d):
//   pass B' (thread a): 5 slots 5 a + b -> radix-5 -> times w80^(-a c) -> slot 5 a + c
//   pass A' (thread c): 16 slots 5 a + c -> radix-16 -> X[c + 5 d] in slot 5 d + c, i.e. natural order.
// No staging registers, one barrier per pass, stride-5 / unit-stride addressing only.
__device__ __forceinline__ constexpr int perm_p(int k) { return 5 * (k & 15) + (k >> 4); }

// radix-16 over 16 loaded values; output index j = k1_of_pos(pos) is stored at base[j * stride5 + off]
template <int SGN>
__device__ __forceinline__ void pass16(double2* v, double2* base, int stride) {
    dft16s<SGN>(v);
#pragma unroll
    for (int pos = 0; pos < 16; ++pos) base[k1_of_pos(pos) * stride] = v[pos];
}

// z * w80^(SGN e), tw[e] = exp(-2 pi i e / 80)
template <int SGN>
__device__ __forceinline__ double2 twmul(double2 z, const double2* tw, int e) {
    double2 w = tw[e];
    if (SGN > 0) w.y = -w.y;
    return cxmul(z, w);
}

constexpr int kIST = kKW;      // row stride of the real plane: odd, so a column of rows spreads over the banks
constexpr int kLS = kF + 1;    // stride of the row-pass scratch lines (odd number of 16-byte slots)

struct ConvSmem {
    double2 W[kF * kFH];     // half spectrum / scratch lines
    double img[kKW * kKW];   // real plane (40x40, stride 41) or kernel (41x41)
    double2 tw[kF];
};

// ---- rows, forward: real rows (p, p + NP) of img packed in one transform -> half spectra W[r][kx]
template <int NIN>
__device__ __noinline__ void rows_forward(ConvSmem& S) {
    constexpr int NP = (NIN + 1) / 2;   // row pairs
    const int tid = threadIdx.x;
    for (int it = tid; it < NP * 5; it += kConvThreads) {
        const int p = it % NP, n2 = it / NP;
        const bool has2 = p + NP < NIN;
        double2 v[16];
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
            const int n = 5 * n1 + n2;
            v[n1] = n < NIN ? make_double2(S.img[p * kIST + n], has2 ? S.img[(p + NP) * kIST + n] : 0.0)
                            : make_double2(0.0, 0.0);
        }
        pass16<-1>(v, S.W + p * kLS + n2, 5);
    }
    __syncthreads();
    for (int it = tid; it < NP * 16; it += kConvThreads) {
        const int p = it % NP, k1 = it / NP;
        double2* line = S.W + p * kLS + 5 * k1;
        double2 z0 = line[0], z1 = twmul<-1>(line[1], S.tw, k1), z2 = twmul<-1>(line[2], S.tw, 2 * k1),
                z3 = twmul<-1>(line[3], S.tw, 3 * k1), z4 = twmul<-1>(line[4], S.tw, 4 * k1);
        dft5s<-1>(z0, z1, z2, z3, z4);
        line[0] = z0, line[1] = z1, line[2] = z2, line[3] = z3, line[4] = z4;     // Z[k1 + 16 k2] in slot 5 k1 + k2
    }
    __syncthreads();
    // untangle: A[kx] = (Z[kx] + conj Z[-kx]) / 2 -> row p, B[kx] = (Z[kx] - conj Z[-kx]) / 2i -> row p + NP
    // (the target rows overlap other pairs' scratch lines: all loads, barrier, all stores)
    constexpr int RU = (NP * kFH + kConvThreads - 1) / kConvThreads;
    double2 za[RU], zb[RU];
#pragma unroll
    for (int rd = 0; rd < RU; ++rd) {
        const int it = tid + rd * kConvThreads;
        if (it < NP * kFH) {
            const int kx = it % kFH, p = it / kFH;
            const double2* line = S.W + p * kLS;
            za[rd] = line[perm_p(kx)];
            zb[rd] = line[perm_p((kF - kx) % kF)];
        }
    }
    __syncthreads();
#pragma unroll
    for (int rd = 0; rd < RU; ++rd) {
        const int it = tid + rd * kConvThreads;
        if (it < NP * kFH) {
            const int kx = it % kFH, p = it / kFH;
            S.W[p * kFH + kx] = make_double2(0.5 * (za[rd].x + zb[rd].x), 0.5 * (za[rd].y - zb[rd].y));
            if (p + NP < NIN)
                S.W[(p + NP) * kFH + kx] = make_double2(0.5 * (za[rd].y + zb[rd].y), 0.5 * (zb[rd].x - za[rd].x));
        }
    }
    __syncthreads();
}

// ---- columns, forward: W[0..NIN)[kx] (rows >= NIN are zero) -> spectrum; ky ends up in row P(ky).
// MUL: times khat[ky][kx], kept in shared memory; otherwise written to gout[ky][kx] in natural order.
template <int NIN, bool MUL>
__device__ __noinline__ void cols_forward(ConvSmem& S, const double2* __restrict__ khat, double2* __restrict__ gout) {
    const int tid = threadIdx.x;
    for (int it = tid; it < kFH * 5; it += kConvThreads) {
        const int kx = it % kFH, n2 = it / kFH;
        double2 v[16];
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
            const int n = 5 * n1 + n2;
            v[n1] = n < NIN ? S.W[n * kFH + kx] : make_double2(0.0, 0.0);
        }
        pass16<-1>(v, S.W + n2 * kFH + kx, 5 * kFH);
    }
    __syncthreads();
    for (int it = tid; it < kFH * 16; it += kConvThreads) {
        const int kx = it % kFH, k1 = it / kFH;
        double2* col = S.W + (5 * k1) * kFH + kx;
        double2 z[5], kh[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            z[q] = q ? twmul<-1>(col[q * kFH], S.tw, q * k1) : col[0];
            if (MUL) kh[q] = __ldg(khat + (k1 + 16 * q) * kFH + kx);
        }
        dft5s<-1>(z[0], z[1], z[2], z[3], z[4]);
#pragma unroll
        for (int k2 = 0; k2 < 5; ++k2) {
            if (MUL) col[k2 * kFH] = cxmul(z[k2], kh[k2]);
            else gout[(k1 + 16 * k2) * kFH + kx] = z[k2];
        }
    }
    __syncthreads();
}

// ---- columns, inverse (decimation in frequency): spectrum with ky in row P(ky) -> spatial row y in row y
__device__ __noinline__ void cols_inverse(ConvSmem& S) {
    const int tid = threadIdx.x;
    for (int it = tid; it < kFH * 16; it += kConvThreads) {
        const int kx = it % kFH, a = it / kFH;
        double2* col = S.W + (5 * a) * kFH + kx;
        double2 z[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) z[q] = col[q * kFH];
        dft5s<1>(z[0], z[1], z[2], z[3], z[4]);
#pragma unroll
        for (int c = 0; c < 5; ++c) col[c * kFH] = c ? twmul<1>(z[c], S.tw, a * c) : z[0];
    }
    __syncthreads();
    for (int it = tid; it < kFH * 5; it += kConvThreads) {
        const int kx = it % kFH, c = it / kFH;
        double2 v[16];
#pragma unroll
        for (int a = 0; a < 16; ++a) v[a] = S.W[(5 * a + c) * kFH + kx];
        pass16<1>(v, S.W + c * kFH + kx, 5 * kFH);       // y = c + 5 d -> row 5 d + c
    }
    __syncthreads();
}

// ---- rows, inverse: half spectra of output rows (p, p + 20), i.e. rows y = p + 20 and p + 40 of the
// full convolution -> two real rows, columns 20..59, times scale
__device__ __noinline__ void rows_inverse(ConvSmem& S, double scale) {
    constexpr int NP = kPSF / 2, OFF = kPSF / 2;
    const int tid = threadIdx.x;
    double2 v[16];
    const int p = tid % NP, n2 = tid / NP;
    const bool active = tid < NP * 5;
    if (active) {
        const double2* A = S.W + (p + OFF) * kFH;
        const double2* B = S.W + (p + NP + OFF) * kFH;
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
            const int n = 5 * n1 + n2;
            if (n <= kF / 2) {
                const double2 a = A[n], b = B[n];
                v[n1] = make_double2(a.x - b.y, a.y + b.x);            // A + i B
            } else {
                const double2 a = A[kF - n], b = B[kF - n];
                v[n1] = make_double2(a.x + b.y, b.x - a.y);            // conj A + i conj B
            }
        }
    }
    __syncthreads();   // the scratch lines overlap rows other pairs still read
    if (active) pass16<1>(v, S.W + p * kLS + n2, 5);
    __syncthreads();
    for (int it = tid; it < NP * 16; it += kConvThreads) {
        const int pp = it % NP, k1 = it / NP;
        const double2* line = S.W + pp * kLS + 5 * k1;
        double2 z0 = line[0], z1 = twmul<1>(line[1], S.tw, k1), z2 = twmul<1>(line[2], S.tw, 2 * k1),
                z3 = twmul<1>(line[3], S.tw, 3 * k1), z4 = twmul<1>(line[4], S.tw, 4 * k1);
        dft5s<1>(z0, z1, z2, z3, z4);
        const double2 z[5] = {z0, z1, z2, z3, z4};
#pragma unroll
        for (int k2 = 0; k2 < 5; ++k2) {
            const int x = k1 + 16 * k2;
            if (x >= OFF && x < OFF + kPSF) {
                S.img[pp * kIST + x - OFF] = scale * z[k2].x;
                S.img[(pp + NP) * kIST + x - OFF] = scale * z[k2].y;
            }
        }
    }
    __syncthreads();
}

__device__ void load_twiddles(ConvSmem& S) {
    for (int k = threadIdx.x; k < kF; k += kConvThreads) {
        double s, c;
        sincospi(2.0 * k / kF, &s, &c);
        S.tw[k] = make_double2(c, -s);
    }
}

// spectrum of one 41x41 kernel: khat[ky][kx], ky < 80, kx <= 40
__global__ void __launch_bounds__(kConvThreads)
kernel_spectrum_kernel(const double* __restrict__ kern, double2* __restrict__ khat) {
    extern __shared__ __align__(16) unsigned char conv_smem_raw[];
    ConvSmem& S = *reinterpret_cast<ConvSmem*>(conv_smem_raw);
    const int k = blockIdx.x;
    load_twiddles(S);
    for (int i = threadIdx.x; i < kKW * kKW; i += kConvThreads) S.img[i] = kern[(size_t)k * kKW * kKW + i];
    __syncthreads();
    rows_forward<kKW>(S);
    cols_forward<kKW, false>(S, nullptr, khat + (size_t)k * kF * kFH);
}

__global__ void __launch_bounds__(kConvThreads, 3)
fft_convolve_kernel(const double* __restrict__ in, const double2* __restrict__ khat_tt,
                    const double2* __restrict__ khat_mu, int nlam, int per_draw, double* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char conv_smem_raw[];
    ConvSmem& S = *reinterpret_cast<ConvSmem*>(conv_smem_raw);
    // a draw owns per_draw consecutive images (its field positions x wavelengths) and one tip-tilt spectrum
    const int img = blockIdx.x, draw = img / per_draw, lam = img % nlam;
    constexpr int kImg = kPSF * kPSF;
    load_twiddles(S);
    for (int i = threadIdx.x; i < kImg; i += kConvThreads) S.img[(i / kPSF) * kIST + i % kPSF] = in[(size_t)img * kImg + i];
    __syncthreads();
    const double scale = 1.0 / (kF * kF);
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        const double2* kh = pass == 0 ? khat_tt + (size_t)draw * kF * kFH : khat_mu + (size_t)lam * kF * kFH;
        rows_forward<kPSF>(S);
        cols_forward<kPSF, true>(S, kh, nullptr);
        cols_inverse(S);
        rows_inverse(S, scale);
    }
    for (int i = threadIdx.x; i < kImg; i += kConvThreads) out[(size_t)img * kImg + i] = S.img[(i / kPSF) * kIST + i % kPSF];
}

}  // namespace

int run_kernel_spectra(Ctx* c, int nk, const double* kern_dev, double2* khat_dev, cudaStream_t s) {
    if (int rc = ensure_dynamic_smem(c, kernel_spectrum_kernel, sizeof(ConvSmem))) return rc;
    kernel_spectrum_kernel<<<nk, kConvThreads, sizeof(ConvSmem), s>>>(kern_dev, khat_dev);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

int run_fft_convolve(Ctx* c, int ndraw, int ndir, int nlam, const double* in_dev, double* out_dev, cudaStream_t s) {
    if (int rc = ensure_dynamic_smem(c, fft_convolve_kernel, sizeof(ConvSmem))) return rc;
    fft_convolve_kernel<<<ndraw * ndir * nlam, kConvThreads, sizeof(ConvSmem), s>>>(in_dev, c->d_khat_tt, c->d_khat_mu,
                                                                                     nlam, ndir * nlam, out_dev);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

}  // namespace psfr
