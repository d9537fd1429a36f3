// Host-side check of ss::noise_factor (gpcc_b200/csrc/ss_model.h): reads "kid rho D" lines; prints Q(D) of ss::step and its
// factor C, each d x d row-major, on one line.
#include "ss_model.h"
#include <cstdio>
using namespace gpcc;

template <int KID>
static void run(double rho, double D) {
    constexpr int d = ss::Dim<KID>::d;
    ss::Coef<d> c;
    ss::setup<KID>(rho, c);
    double A[d][d], Q[d][d], dA[d][d], dQ[d][d], C[d][d];
    ss::step<KID, false>(c, D, A, Q, dA, dQ);
    ss::noise_factor<d>(Q, C);
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) printf("%.17g ", Q[i][j]);
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) printf("%.17g ", C[i][j]);
    printf("\n");
}

int main() {
    int kid;
    double rho, D;
    while (scanf("%d %lf %lf", &kid, &rho, &D) == 3) {
        if (kid == 0) run<0>(rho, D);
        else if (kid == 2) run<2>(rho, D);
        else run<3>(rho, D);
    }
    return 0;
}
