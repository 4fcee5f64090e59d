// Exact overlap of a disc and an axis-aligned rectangle (encircled energy, DESIGN.md section 5.4).
// __host__ __device__ so that the same code runs in psfr_energy.cu and in the CPU check tools/ee_check.cu.
//
// The disc of radius r is centred at the origin.  A rectangle is folded into the first quadrant by the disc's
// symmetry (a rectangle across an axis is split there), and a first-quadrant rectangle [a, b] x [c, d] is
// integrated column by column: the chord height s(x) = sqrt(r^2 - x^2) clipped to [c, d].  Every term of the
// result is non-negative, so nothing cancels: the area under the arc between x = u and x = v is the trapezoid
// under the chord plus the circular segment r^2 (phi - sin phi) / 2, with phi from atan2 of the half chord and
// phi - sin phi from its series at small phi.  FP64 throughout, no supersampling.
#pragma once
#include <cmath>

#if defined(__CUDACC__)
#define EE_HD __host__ __device__ __forceinline__
#else
#define EE_HD inline
#endif

namespace ee {

// phi - sin(phi) for phi in [0, pi/2]; the series below 1 keeps full relative precision where the
// difference cancels (its first omitted term is below 1e-17 of the sum)
EE_HD double phi_minus_sin(double phi) {
    if (phi >= 1.0) return phi - sin(phi);
    const double z = phi * phi;
    // phi^3 (1/3! - z/5! + z^2/7! - ...), nine terms, Horner from the highest
    double p = 1.0 / 121645100408832000.0;                 // 1/19!
    p = fma(p, -z, 1.0 / 355687428096000.0);               // 1/17!
    p = fma(p, -z, 1.0 / 1307674368000.0);                 // 1/15!
    p = fma(p, -z, 1.0 / 6227020800.0);                    // 1/13!
    p = fma(p, -z, 1.0 / 39916800.0);                      // 1/11!
    p = fma(p, -z, 1.0 / 362880.0);                        // 1/9!
    p = fma(p, -z, 1.0 / 5040.0);                          // 1/7!
    p = fma(p, -z, 1.0 / 120.0);                           // 1/5!
    p = fma(p, -z, 1.0 / 6.0);                             // 1/3!
    return p * z * phi;
}

// sqrt(r^2 - x^2) for 0 <= x <= r, formed as sqrt((r - x)(r + x)) (no cancellation in r^2 - x^2)
EE_HD double half_chord(double r, double x) {
    const double t = (r - x) * (r + x);
    return t > 0.0 ? sqrt(t) : 0.0;
}

// Area of the disc x^2 + y^2 <= r^2 inside [a, b] x [c, d], 0 <= a <= b, 0 <= c <= d, and with kArc the length
// of the circle inside it: the circle crosses such a rectangle in one arc, from (u, su) to (v, sv), of length
// r phi.
template <bool kArc>
EE_HD double quadrant_area(double a, double b, double c, double d, double r, double* arc) {
    if (kArc) *arc = 0.0;
    if (!(a < b) || !(c < d) || !(r > 0.0)) return 0.0;
    // s(x) >= d for x <= xd (full height), s(x) <= c for x >= xc (nothing)
    const double xd = r > d ? half_chord(r, d) : 0.0;
    const double xc = r > c ? half_chord(r, c) : 0.0;
    double area = 0.0;
    if (a < xd) area = (fmin(b, xd) - a) * (d - c);
    double u, su, v, sv;
    if (a < xd) { u = xd; su = d; } else { u = a; su = 0.0; }
    if (b > xc) { v = xc; sv = c; } else { v = b; sv = 0.0; }
    if (u < v) {
        if (!(a < xd)) su = half_chord(r, u);
        if (!(b > xc)) sv = half_chord(r, v);
        // trapezoid under the chord from (u, su) to (v, sv), above y = c, plus the segment beyond the chord
        const double w = v - u;
        const double l = 0.5 * sqrt(w * w + (su - sv) * (su - sv));      // half chord length
        const double phi = 2.0 * atan2(l, half_chord(r, l));
        area += w * (0.5 * ((su - c) + (sv - c))) + 0.5 * r * r * phi_minus_sin(phi);
        if (kArc) *arc = r * phi;
    }
    return area;
}

// Area (and with kArc the circle length) of the disc of radius r centred at the origin inside
// [x0, x1] x [y0, y1]: the parts of the rectangle in the four quadrants, each folded into the first.
template <bool kArc>
EE_HD double rect_overlap(double x0, double x1, double y0, double y1, double r, double* arc) {
    // the parts of [x0, x1] below and above 0, and of [y0, y1], as first-quadrant intervals
    const bool xn = x0 < 0.0, xp = x1 > 0.0, yn = y0 < 0.0, yp = y1 > 0.0;
    const double xna = x1 < 0.0 ? -x1 : 0.0, xnb = -x0, xpa = x0 > 0.0 ? x0 : 0.0, xpb = x1;
    const double yna = y1 < 0.0 ? -y1 : 0.0, ynb = -y0, ypa = y0 > 0.0 ? y0 : 0.0, ypb = y1;
    double area = 0.0, len = 0.0;
    auto add = [&](bool on, double a, double b, double c, double d) {
        if (!on) return;
        double l = 0.0;
        area += quadrant_area<kArc>(a, b, c, d, r, &l);
        if (kArc) len += l;
    };
    add(xn && yn, xna, xnb, yna, ynb);
    add(xn && yp, xna, xnb, ypa, ypb);
    add(xp && yn, xpa, xpb, yna, ynb);
    add(xp && yp, xpa, xpb, ypa, ypb);
    if (kArc) *arc = len;
    return area;
}

// Overlap of the unit pixel centred at (dy, dx) from the disc's centre with the disc of radius r.
EE_HD double pixel_area(double dy, double dx, double r) {
    return rect_overlap<false>(dx - 0.5, dx + 0.5, dy - 0.5, dy + 0.5, r, nullptr);
}
EE_HD double pixel_area_arc(double dy, double dx, double r, double* arc) {
    return rect_overlap<true>(dx - 0.5, dx + 0.5, dy - 0.5, dy + 0.5, r, arc);
}

// Squared distances from the disc's centre to the nearest and the farthest point of that pixel.
EE_HD void pixel_dist2(double dy, double dx, double* near2, double* far2) {
    const double ay = fabs(dy), ax = fabs(dx);
    const double ny = fmax(ay - 0.5, 0.0), nx = fmax(ax - 0.5, 0.0);
    *near2 = ny * ny + nx * nx;
    *far2 = (ay + 0.5) * (ay + 0.5) + (ax + 0.5) * (ax + 0.5);
}

// Rows [*p0, *p1) of an image of ny rows that the disc of radius r about row y0 can reach: row p spans
// [p - 1/2, p + 1/2], so it is reached when y0 - r - 1/2 <= p <= y0 + r + 1/2; the window keeps a row of margin
// on each side against rounding.  Both ends are clamped to [0, ny] in double before the conversion to int, so a
// centre far outside the image gives an empty window (*p0 >= *p1) and nothing overflows; r may be +inf.
EE_HD void row_window(double y0, double r, int ny, int* p0, int* p1) {
    *p0 = (int)fmin(fmax(0.0, floor(y0 - r - 0.5)), (double)ny);
    *p1 = (int)fmax(0.0, fmin((double)ny, ceil(y0 + r + 0.5) + 1.0));
}

// Starting bracket of the radius at which EE reaches target > 0, from n tabulated radii r[k] with e[k] = EE(r[k])
// and the farthest pixel corner rmax, where EE = total >= target: *hi is the smallest tabulated radius with
// EE >= target (rmax if there is none), *lo the largest tabulated radius below *hi with EE < target (0 if there is
// none, where EE = 0).  So lo < hi and EE(lo) < target <= EE(hi) also where EE falls (negative pixels), and the
// bracket does not depend on the order of the radii.
EE_HD void fraction_bracket(const double* r, const double* e, int n, double target, double rmax, double total,
                            double* lo, double* elo, double* hi, double* ehi) {
    *hi = rmax;
    *ehi = total;
    for (int k = 0; k < n; ++k)
        if (e[k] >= target && r[k] < *hi) { *hi = r[k]; *ehi = e[k]; }
    *lo = 0.0;
    *elo = 0.0;
    for (int k = 0; k < n; ++k)
        if (e[k] < target && r[k] < *hi && r[k] > *lo) { *lo = r[k]; *elo = e[k]; }
}

}  // namespace ee
