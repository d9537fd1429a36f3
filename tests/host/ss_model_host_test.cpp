// Host-side check of the closed forms of gpcc_b200/csrc/ss_model.h (plain C++ behind GPCC_HD): reads lines
// "kid rho dt" from stdin and prints A, Q, dA/drho, dQ/drho (row-major, %.17g) on one line each.
#include "ss_model.h"
#include <cstdio>
#include <initializer_list>
using namespace gpcc;

template <int KID>
static void run(double rho, double dt) {
    constexpr int d = ss::Dim<KID>::d;
    ss::Coef<d> c;
    ss::setup<KID>(rho, c);
    double A[d][d], Q[d][d], dA[d][d], dQ[d][d];
    ss::step<KID, true>(c, dt, A, Q, dA, dQ);
    for (auto* M : {&A, &Q, &dA, &dQ})
        for (int i = 0; i < d; ++i)
            for (int j = 0; j < d; ++j) printf("%.17g ", (*M)[i][j]);
    printf("\n");
}

int main() {
    int kid;
    double rho, dt;
    while (scanf("%d %lf %lf", &kid, &rho, &dt) == 3) {
        if (kid == 0) run<0>(rho, dt);
        else if (kid == 2) run<2>(rho, dt);
        else run<3>(rho, dt);
    }
    return 0;
}
