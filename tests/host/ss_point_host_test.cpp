// Host-side check of ss::point_moments (gpcc_b200/csrc/ss_model.h): reads "kid L l a rho dt1 later dt2" followed by m (D),
// P (packed, D(D+1)/2), and when later != 0 lam (D) and Lam (packed); prints the smoothed mean and variance of h'x.
#include "ss_model.h"
#include <cstdio>
#include <vector>
using namespace gpcc;

template <int KID, int L>
static void run(int l, double a, double rho, double dt1, int later, double dt2) {
    constexpr int d = ss::Dim<KID>::d, D = d + L, NP = D * (D + 1) / 2;
    double m[D], P[NP], lam[D], Lam[NP];
    for (double& v : m) scanf("%lf", &v);
    for (double& v : P) scanf("%lf", &v);
    if (later) {
        for (double& v : lam) scanf("%lf", &v);
        for (double& v : Lam) scanf("%lf", &v);
    }
    ss::Coef<d> c;
    ss::setup<KID>(rho, c);
    double mean, var;
    ss::point_moments<KID, L>(c, l, a, m, P, dt1, later ? lam : nullptr, later ? Lam : nullptr, dt2, mean, var);
    printf("%.17g %.17g\n", mean, var);
}

template <int KID, int L = 1>
static void dispatch(int nb, int l, double a, double rho, double dt1, int later, double dt2) {
    if (nb == L) return run<KID, L>(l, a, rho, dt1, later, dt2);
    if constexpr (L < 8) dispatch<KID, L + 1>(nb, l, a, rho, dt1, later, dt2);
}

int main() {
    int kid, nb, l, later;
    double a, rho, dt1, dt2;
    while (scanf("%d %d %d %lf %lf %lf %d %lf", &kid, &nb, &l, &a, &rho, &dt1, &later, &dt2) == 8) {
        if (kid == 0) dispatch<0>(nb, l, a, rho, dt1, later, dt2);
        else if (kid == 2) dispatch<2>(nb, l, a, rho, dt1, later, dt2);
        else dispatch<3>(nb, l, a, rho, dt1, later, dt2);
    }
    return 0;
}
