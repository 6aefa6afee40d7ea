// Host driver of the Sturm-count bisection of secedo_b200/csrc/sturm.hpp (the code the device runs one eigenvalue index
// per thread). Input file: u32 n, then n doubles d and n - 1 doubles e. Output file: the n eigenvalues, ascending.
// With --count x: prints count_below(x) instead.
#include "../secedo_b200/csrc/sturm.hpp"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

int main(int argc, char **argv) {
    const bool count = argc == 5 && std::strcmp(argv[1], "--count") == 0;
    if (argc != 3 && !count) {
        std::fprintf(stderr, "usage: %s in.bin out.bin | --count in.bin x -\n", argv[0]);
        return 2;
    }
    FILE *f = std::fopen(count ? argv[2] : argv[1], "rb");
    uint32_t n = 0;
    if (!f || std::fread(&n, 4, 1, f) != 1 || n == 0) {
        return 1;
    }
    std::vector<double> d(n), e(n, 0.0), e2(n, 0.0), w(n);
    if (std::fread(d.data(), 8, n, f) != n || std::fread(e.data(), 8, n - 1, f) != n - 1) {
        return 1;
    }
    std::fclose(f);
    for (uint32_t i = 0; i + 1 < n; ++i) {
        e2[i] = e[i] * e[i];
    }
    const double pmin = sturm::pivmin(e2.data(), n);
    if (count) {
        std::printf("%u\n", sturm::count_below(d.data(), e2.data(), n, std::strtod(argv[3], nullptr), pmin));
        return 0;
    }
    const sturm::Interval iv = sturm::gershgorin(d.data(), e.data(), n, pmin);
    for (uint32_t k = 0; k < n; ++k) {
        w[k] = sturm::bisect(d.data(), e2.data(), n, k, iv, pmin);
    }
    FILE *o = std::fopen(argv[2], "wb");
    if (!o || std::fwrite(w.data(), 8, n, o) != n) {
        return 1;
    }
    std::fclose(o);
    return 0;
}
