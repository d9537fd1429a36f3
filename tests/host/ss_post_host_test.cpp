// Host-side check of ss::point_mean_weights (gpcc_b200/csrc/ss_model.h): reads "kid L l a rho dt1 later dt2" followed by m
// (D), P (packed, D(D+1)/2), and when later != 0 lam (D) and Lam (packed); prints the smoothed mean of ss::point_moments and
// c1'm - w'lam from the weights.
#include "ss_model.h"
#include <cstdio>
using namespace gpcc;

template <int KID, int L>
static void run(int l, double a, double rho, double dt1, int later, double dt2) {
    constexpr int d = ss::Dim<KID>::d, D = d + L, NP = D * (D + 1) / 2;
    double m[D], P[NP], P2[NP], lam[D], Lam[NP], c1[D], w[D];
    for (double& v : m) scanf("%lf", &v);
    for (int i = 0; i < NP; ++i) { scanf("%lf", &P[i]); P2[i] = P[i]; }
    for (int i = 0; i < D; ++i) lam[i] = 0.0;
    for (int i = 0; i < NP; ++i) Lam[i] = 0.0;
    if (later) {
        for (double& v : lam) scanf("%lf", &v);
        for (double& v : Lam) scanf("%lf", &v);
    }
    ss::Coef<d> c;
    ss::setup<KID>(rho, c);
    double m1[D];
    for (int i = 0; i < D; ++i) m1[i] = m[i];
    double mean, var;
    ss::point_moments<KID, L>(c, l, a, m1, P, dt1, later ? lam : nullptr, later ? Lam : nullptr, dt2, mean, var);
    ss::point_mean_weights<KID, L>(c, l, a, P2, dt1, later != 0, dt2, c1, w);
    double lin = 0.0;
    for (int i = 0; i < D; ++i) lin += c1[i] * m[i] - w[i] * lam[i];
    printf("%.17g %.17g\n", mean, lin);
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
