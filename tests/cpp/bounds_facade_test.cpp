// bounds_facade_test.cpp — SDF::Octree::QueryBounds through the C++ facade: boxes around a sphere tree enclose Query at their
// corners and centres, a box outside the root gets DBL_MAX, an inverted box NaN, and a copy of the tree gives the same bits.
// Build: g++ -std=c++17 -I include tests/cpp/bounds_facade_test.cpp -L <pkg>/lib -lhpsdf ; run on a GPU box.
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>
#include "hpsdf.hpp"

int main()
{
    SDF::Config cfg;
    cfg.targetErrorThreshold = 1e-6;
    SDF::Program prog;
    prog.Sphere(0.1, 0.0, 0.0, 0.3);
    SDF::Octree t;
    t.Create(cfg, prog);
    const int n = 64;
    std::vector<double> lo(3 * n + 6), hi(3 * n + 6);
    for (int i = 0; i < n; ++i)
        for (int a = 0; a < 3; ++a)
        {
            lo[3 * i + a] = -0.5 + ((i * 7 + a * 3) % 16) / 16.0;
            hi[3 * i + a] = lo[3 * i + a] + 1.0 / (1 + (i % 5));
        }
    const double extra[6] = { 0.7, 0.7, 0.7, 0.9, 0.9, 0.9 };       // outside the root
    const double inv[6] = { 0.2, 0.0, 0.0, 0.1, 0.1, 0.1 };         // inverted on x
    std::memcpy(&lo[3 * n], extra, 24); std::memcpy(&hi[3 * n], extra + 3, 24);
    std::memcpy(&lo[3 * n + 3], inv, 24); std::memcpy(&hi[3 * n + 3], inv + 3, 24);
    std::vector<double> fLo(n + 2), fHi(n + 2);
    t.QueryBounds(lo.data(), hi.data(), n + 2, fLo.data(), fHi.data());
    int bad = 0;
    for (int i = 0; i < n; ++i)
    {
        double pts[27];
        for (int c = 0; c < 9; ++c)
            for (int a = 0; a < 3; ++a)
                pts[3 * c + a] = c == 8 ? 0.5 * (lo[3 * i + a] + hi[3 * i + a]) : ((c >> a) & 1) ? hi[3 * i + a] : lo[3 * i + a];
        double q[9];
        t.Query(pts, 9, q);
        for (int c = 0; c < 9; ++c)
            if (!(fLo[i] <= q[c] && q[c] <= fHi[i])) { std::printf("box %d point %d: %g outside [%g, %g]\n", i, c, q[c], fLo[i], fHi[i]); ++bad; }
    }
    if (fLo[n] != DBL_MAX || fHi[n] != DBL_MAX) { std::printf("outside box: [%g, %g]\n", fLo[n], fHi[n]); ++bad; }
    if (!std::isnan(fLo[n + 1]) || !std::isnan(fHi[n + 1])) { std::printf("inverted box: [%g, %g]\n", fLo[n + 1], fHi[n + 1]); ++bad; }
    SDF::Octree copy(t);
    std::vector<double> gLo(n + 2), gHi(n + 2);
    copy.QueryBounds(lo.data(), hi.data(), n + 2, gLo.data(), gHi.data());
    if (std::memcmp(gLo.data(), fLo.data(), 8 * n) || std::memcmp(gHi.data(), fHi.data(), 8 * n)) { std::printf("copy differs\n"); ++bad; }
    std::printf(bad ? "FAILED\n" : "All bounds tests passed!\n");
    return bad ? 1 : 0;
}
