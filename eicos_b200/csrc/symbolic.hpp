// Host-side, once-per-sparsity-pattern analysis for the batched B200 SOCP engine.
//
// Replaces (reference = EmbersArc/EiCOS, /root/reference):
//   - Solver::build dims                      src/eicos.cpp:132-187
//   - setEquilibration (shared G/A values)    src/eicos.cpp:302-374
//   - setupKKT + cacheIndices                 src/eicos.cpp:1734-1988  (index maps instead of pointer tables)
//   - Eigen::SimplicialLDLT::analyzePattern   call site src/eicos.cpp:897 (AMD ordering, elimination
//                                             tree, column counts) - run ONCE per pattern here instead of
//                                             once per solve()
// and adds what only the GPU needs: CSR views of G, A and L (the programs the numeric kernels run
// are compiled from these by streams.cpp).
#pragma once

#include <cstdint>
#include <vector>

namespace eicos
{

typedef std::vector<int> ivec;
typedef std::vector<double> dvec;

// Tunable constants of the reference (include/eicos.hpp:23-47); all compile-time there as well.  Here they are
// the defaults of KSettings, except deltastat and equil_iters, which enter the shared KKT values, the programs'
// constants and the equilibration at setup and so stay fixed for the life of a handle.
struct Settings
{
    static constexpr double gamma = 0.99, deltastat = 7e-8;
    static constexpr double feastol = 1e-8, abstol = 1e-8, reltol = 1e-8;
    static constexpr double feastol_inacc = 1e-4, abstol_inacc = 5e-5, reltol_inacc = 5e-5;
    static constexpr int nitref = 9, equil_iters = 3, iter_max = 100;
    static constexpr double linsysacc = 1e-14, irerrfact = 6, stepmin = 1e-6, stepmax = 0.999;
    static constexpr double sigmamin = 1e-4, sigmamax = 1.0, safeguard = 500;
};

// The settings the kernels read at run time (KArgs::settings), one set per handle.  Plain doubles and ints:
// passed inside the __grid_constant__ KArgs, every field is read from the constant bank.
struct KSettings
{
    double feastol, abstol, reltol;
    double feastol_inacc, abstol_inacc, reltol_inacc;
    double linsysacc, irerrfact;
    double gamma, stepmin, stepmax;
    double sigmamin, sigmamax;
    double safeguard;
    int nitref, iter_max;
};

inline KSettings default_settings()
{
    KSettings k;
    k.feastol = Settings::feastol, k.abstol = Settings::abstol, k.reltol = Settings::reltol;
    k.feastol_inacc = Settings::feastol_inacc, k.abstol_inacc = Settings::abstol_inacc, k.reltol_inacc = Settings::reltol_inacc;
    k.linsysacc = Settings::linsysacc, k.irerrfact = Settings::irerrfact;
    k.gamma = Settings::gamma, k.stepmin = Settings::stepmin, k.stepmax = Settings::stepmax;
    k.sigmamin = Settings::sigmamin, k.sigmamax = Settings::sigmamax;
    k.safeguard = Settings::safeguard;
    k.nitref = Settings::nitref, k.iter_max = Settings::iter_max;
    return k;
}

struct Csc
{
    int rows = 0, cols = 0;
    ivec p{0}, i;
    dvec x;
    int nnz() const { return (int)i.size(); }
};

// CSR view of a CSC matrix: row r has entries [p[r], p[r+1]) with column j[k] and value slot v[k]
// (v indexes the CSC value array, so only ONE copy of the values exists on the device).
struct CsrView
{
    ivec p, j, v;
};

struct Symbolic
{
    // ---- dimensions (src/eicos.cpp:152-165)
    int n = 0, p = 0, m = 0, l = 0, nc = 0, N = 0, mt = 0; // mt = m + 2 nc
    ivec q;                                                   // cone dims
    ivec cone_z, cone_k, cone_q;                              // first index of cone c in z-space / expanded space / q-storage
    int qtot = 0;                                             // sum(dim-1)
    ivec zk;                                                  // z index -> expanded index (K row = n+p+zk[i])

    // ---- problem matrices (equilibrated values live in G.x / A.x) and equilibration vectors
    Csc G, A;
    CsrView Gr, Ar;
    dvec xeq, Aeq, Geq;

    // ---- KKT pattern, upper triangle, CSC with sorted rows (src/eicos.cpp:1734-1890)
    ivec Kp, Ki;
    ivec AGslot; // K slot of k-th value in [At columns..., Gt columns...] order (cacheIndices :1899-1942)
    ivec Vslot;  // K slot of k-th scaling value (cacheIndices :1946-1987)
    ivec Kvidx;  // per K slot: index into the per-instance V array, or -1 if the value is shared
    dvec Kshared; // per K slot: value shared by the whole batch (delta, -delta, A', G'); 0 where Kvidx>=0
    ivec AGsrc;   // per AGslot entry: >=0 -> index into A.x ; <0 -> -(index into G.x)-1

    // ---- ordering + symbolic factor (Eigen analyzePattern)
    ivec pinv; // pinv[k] = original index of k-th pivot (AMD output, Eigen m_Pinv)
    ivec P;    // P[old] = new (Eigen m_P)
    ivec parent, Lp, Li;
    CsrView Lr; // rows of L: Lr.j = column, Lr.v = position in the CSC arrays
    int nnzL = 0;

    // ---- permuted KKT, lower-triangular by columns: what column j of the factorisation consumes
    ivec KLp, KLslot, KLpos; // entry range per column; K slot; position inside L column j (-1 = diagonal)

    // ---- shape of the factor
    ivec level;              // etree height of every column (0 = leaf)
    int height = 0, maxcol = 0;
    long long fma_count = 0; // multiply-adds of one numeric factorisation
};

// Row/column infinity-norm equilibration of G and A in place (src/eicos.cpp:302-362); cones share
// one row scale.  c/h/b are NOT touched here (they are per instance).
void equilibrate(Csc &G, Csc &A, int l, const ivec &q, dvec &xeq, dvec &Aeq, dvec &Geq);

// Builds everything above from the (unequilibrated) problem matrices.
void analyze(Symbolic &S, int n, int m, int p, int ncones, const int *q,
             const double *Gpr, const int *Gjc, const int *Gir,
             const double *Apr, const int *Ajc, const int *Air);

// Undo the equilibration of the stored G/A values by multiplying the scales back in
// (restore(), src/eicos.cpp:376-392 - not bit-exact with the original data, like the reference).
void unequilibrate(Symbolic &S);

// Overwrite the stored G/A values where a pointer is given, then equilibrate what is stored and
// re-derive the shared KKT values (updateData, src/eicos.cpp:2032-2082); the pattern and every
// index map are reused.  Whatever is stored for a NULL argument is equilibrated AGAIN, so callers
// either pass both matrices or call unequilibrate() first (which is what the reference does).
void refresh_values(Symbolic &S, const double *Gpr, const double *Apr);

// The ordering itself (exposed for tests): full symmetric pattern with diagonal, sorted columns.
ivec amd_ordering(int n, const ivec &Ap, const ivec &Ai);

} // namespace eicos
