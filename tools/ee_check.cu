// CPU driver of the __host__ __device__ overlap geometry in csrc/ee_geometry.h (tests/test_energy_host.py):
// reads lines "dy dx r" from stdin and prints, for each, the overlap area of the unit pixel centred at
// (dy, dx) with the disc of radius r about the origin, and the length of the circle inside that pixel.
//   nvcc -O2 -I muse_psfr_b200/csrc tools/ee_check.cu -o ee_check
#include <cstdio>
#include "ee_geometry.h"

int main() {
    double dy, dx, r;
    while (std::scanf("%lf %lf %lf", &dy, &dx, &r) == 3) {
        double arc = 0.0;
        const double a = ee::pixel_area_arc(dy, dx, r, &arc);
        const double b = ee::pixel_area(dy, dx, r);
        std::printf("%.17g %.17g %.17g\n", a, arc, b);
    }
    return 0;
}
