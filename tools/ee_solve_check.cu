// CPU driver of the radius-solve helpers in csrc/ee_geometry.h (tests/test_energy_window_host.py).  Reads lines
//   w y0 r ny                              -> prints "p0 p1", the row window of ee::row_window
//   b target rmax total n r_1 e_1 ... r_n e_n -> prints "lo elo hi ehi", the bracket of ee::fraction_bracket
//   nvcc -O2 -I muse_psfr_b200/csrc tools/ee_solve_check.cu -o ee_solve_check
#include <cstdio>
#include <vector>
#include "ee_geometry.h"

int main() {
    char op;
    while (std::scanf(" %c", &op) == 1) {
        if (op == 'w') {
            double y0, r;
            int ny, p0, p1;
            if (std::scanf("%lf %lf %d", &y0, &r, &ny) != 3) return 1;
            ee::row_window(y0, r, ny, &p0, &p1);
            std::printf("%d %d\n", p0, p1);
        } else if (op == 'b') {
            double target, rmax, total, lo, elo, hi, ehi;
            int n;
            if (std::scanf("%lf %lf %lf %d", &target, &rmax, &total, &n) != 4 || n < 0) return 1;
            std::vector<double> r(n), e(n);
            for (int k = 0; k < n; ++k)
                if (std::scanf("%lf %lf", &r[k], &e[k]) != 2) return 1;
            ee::fraction_bracket(r.data(), e.data(), n, target, rmax, total, &lo, &elo, &hi, &ehi);
            std::printf("%.17g %.17g %.17g %.17g\n", lo, elo, hi, ehi);
        } else {
            return 1;
        }
    }
    return 0;
}
