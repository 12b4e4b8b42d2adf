// Test driver for the writable settings of include/eicos.hpp: EiCOS::Solver and EiCOS::BatchSolver take their
// settings through getSettings(), the way a user of the reference's interface writes them.  Reads a problem,
// one set of settings and a batch of (h, b) from a binary file written by tests/test_runtime_settings.py, solves
// the problem once with Solver and the batch with BatchSolver, and prints every result as the hex image of its
// float64 bits so that the Python side can compare bit for bit.  The test compiles it against the CPU emulator of
// the kernels and against the CUDA library.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "eicos.hpp"

namespace
{
FILE *in;

template <class T>
std::vector<T> read(size_t k)
{
    std::vector<T> v(k);
    if (k && fread(v.data(), sizeof(T), k, in) != k)
    {
        fprintf(stderr, "settings_driver: truncated input\n");
        exit(3);
    }
    return v;
}

void print(const char *tag, const double *v, size_t k)
{
    printf("%s", tag);
    for (size_t i = 0; i < k; i++)
    {
        uint64_t u;
        std::memcpy(&u, v + i, 8);
        printf(" %016llx", (unsigned long long)u);
    }
    printf("\n");
}

void apply(EiCOS::Settings &s, const std::vector<double> &d, const std::vector<int> &i)
{
    s.feastol = d[0], s.abstol = d[1], s.reltol = d[2];
    s.feastol_inacc = d[3], s.abstol_inacc = d[4], s.reltol_inacc = d[5];
    s.linsysacc = d[6], s.irerrfact = d[7];
    s.gamma = d[8], s.stepmin = d[9], s.stepmax = d[10];
    s.sigmamin = d[11], s.sigmamax = d[12];
    s.safeguard = (size_t)d[13];
    s.nitref = (size_t)i[0], s.iter_max = (size_t)i[1];
}
} // namespace

int main(int argc, char **argv)
{
    if (argc < 2 || !(in = fopen(argv[1], "rb")))
    {
        fprintf(stderr, "usage: settings_driver <script>\n");
        return 2;
    }
    const std::vector<int> dims = read<int>(7); // n m p l ncones nnzG nnzA
    const int n = dims[0], m = dims[1], p = dims[2], l = dims[3], nc = dims[4], nG = dims[5], nA = dims[6];
    std::vector<int> q = read<int>(nc), Gjc = read<int>(n + 1), Gir = read<int>(nG), Ajc = read<int>(n + 1), Air = read<int>(nA);
    std::vector<double> Gpr = read<double>(nG), Apr = read<double>(nA), c = read<double>(n), h = read<double>(m), b = read<double>(p);
    const std::vector<double> sd = read<double>(14);
    const std::vector<int> si = read<int>(2);
    const int batch = read<int>(1)[0];
    const std::vector<double> hs = read<double>((size_t)batch * m), bs = read<double>((size_t)batch * p);
    fclose(in);
    try
    {
        EiCOS::Solver S(n, m, p, l, nc, q.data(), nG ? Gpr.data() : nullptr, nG ? Gjc.data() : nullptr, nG ? Gir.data() : nullptr,
                        nA ? Apr.data() : nullptr, nA ? Ajc.data() : nullptr, nA ? Air.data() : nullptr, c.data(), h.data(), b.data());
        apply(S.getSettings(), sd, si);
        const int code = (int)S.solve();
        const EiCOS::Information &I = S.getInfo();
        printf("solve %d %zu %zu\n", code, I.iter, I.iter_max);
        print("x", S.solution().data(), (size_t)n);

        EiCOS::BatchSolver B(n, m, p, l, nc, q.data(), nG ? Gpr.data() : nullptr, nG ? Gjc.data() : nullptr, nG ? Gir.data() : nullptr,
                             nA ? Apr.data() : nullptr, nA ? Ajc.data() : nullptr, nA ? Air.data() : nullptr, c.data(), h.data(), b.data());
        apply(B.getSettings(), sd, si);
        const EiCOS::BatchSolver::Result r = B.solve(batch, nullptr, hs.data(), p ? bs.data() : nullptr);
        for (int k = 0; k < batch; k++)
        {
            const eicos_info &i = r.info[(size_t)k];
            printf("batch %d %d %d %d %d %d\n", r.exitflag[(size_t)k], i.iter, i.iter_max, i.nitref1, i.nitref2, i.nitref3);
            print("x", r.x.data() + (size_t)k * n, (size_t)n);
            print("z", r.z.data() + (size_t)k * m, (size_t)m);
        }
        // an out-of-range value is rejected at the next solve, naming the field
        B.getSettings().gamma = 1.5;
        try
        {
            B.solve(batch, nullptr, hs.data(), p ? bs.data() : nullptr);
            printf("rejected none\n");
        }
        catch (const std::runtime_error &e)
        {
            printf("rejected %s\n", std::strstr(e.what(), "gamma") ? "gamma" : "other");
        }
    }
    catch (const std::exception &e)
    {
        fprintf(stderr, "settings_driver: %s\n", e.what());
        return 1;
    }
    return 0;
}
