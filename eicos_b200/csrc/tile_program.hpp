// The per-tile interior-point program: every step of EiCOS's Solver::solve (reference
// src/eicos.cpp:848-1262) for TILE = LANES x VEC instances at a time.
//
// One CTA owns one tile.  Lane l of a warp owns VEC consecutive instances of the tile, so a row of a
// per-instance array is moved with ONE 16-byte access per lane (512 B per warp for VEC = 2): every
// index decode, address computation and loop step is amortised over VEC instances, and the
// sparsity pattern never diverges inside a warp.
//   * Program kernels (numeric LDL', triangular sweeps, KKT mat-vecs): ONE warp per tile interprets
//     machine code compiled on the host (machine.hpp, streams.hpp): bundles of independent 3-address
//     operations on shared-memory rows.  Global reads arrive through a cp.async ring whose rows the
//     code names directly; intermediate values sit in shared-memory slots for their live range; the
//     code itself and its load list arrive by TMA bulk copies.  Nothing inside such a kernel needs a barrier.
//   * Vector kernels (statistics, scalings, right-hand sides, line search, iterate update): the
//     warps ("workers") of the CTA split the rows; per-instance reductions run down the rows in
//     each worker and are combined through shared memory in a fixed order, so every warp holds
//     bit-identical per-instance scalars and all control flow is uniform across the CTA.
//
// The same source compiles two ways:
//   * nvcc (default): LANES = 32, workers = warps of the CTA  -> the product.
//   * -DEICOS_EMU (tests/emu only): LANES = 1, workers = host threads, plain C++ -> lets the
//     CPU-only test tier execute the kernel logic against the oracle.  Never linked into the product.
#pragma once

#include "layout.hpp"
#include "streams.hpp"
#include "symbolic.hpp"

#include <cfloat>
#include <cmath>

#ifdef EICOS_EMU
#include <barrier>
#define EI_DEV inline
#define EI_LDG(p) (*(p))
#define EI_CLOCK() 0ll
#else
#include <cuda_runtime.h>
#define EI_DEV __device__ __forceinline__
#define EI_LDG(p) __ldg(p)
#define EI_CLOCK() clock64()
#endif

#ifndef EICOS_VEC
#define EICOS_VEC 2
#endif

namespace eicos
{

#ifdef EICOS_EMU
constexpr int LANES = 1;
#else
constexpr int LANES = 32;
#endif
constexpr int VEC = EICOS_VEC;       // instances per lane
constexpr int TILE = LANES * VEC;    // instances per tile = doubles per row
constexpr int KRED = 7;              // rows per worker in the shared reduction buffer

// ------------------------------------------------------------------ VEC-wide values
struct alignas(VEC >= 2 ? 16 : 8) vd
{
    double v[VEC];
};
struct vb
{
    bool v[VEC];
};
#define VFOR for (int c_ = 0; c_ < VEC; c_++)

EI_DEV vd vset(double s)
{
    vd r;
    VFOR r.v[c_] = s;
    return r;
}
EI_DEV vd operator+(vd a, vd b) { VFOR a.v[c_] += b.v[c_]; return a; }
EI_DEV vd operator-(vd a, vd b) { VFOR a.v[c_] -= b.v[c_]; return a; }
EI_DEV vd operator*(vd a, vd b) { VFOR a.v[c_] *= b.v[c_]; return a; }
EI_DEV vd operator/(vd a, vd b) { VFOR a.v[c_] /= b.v[c_]; return a; }
EI_DEV vd operator-(vd a) { VFOR a.v[c_] = -a.v[c_]; return a; }
EI_DEV vd operator+(vd a, double b) { VFOR a.v[c_] += b; return a; }
EI_DEV vd operator-(vd a, double b) { VFOR a.v[c_] -= b; return a; }
EI_DEV vd operator+(double b, vd a) { VFOR a.v[c_] = b + a.v[c_]; return a; }
EI_DEV vd operator-(double b, vd a) { VFOR a.v[c_] = b - a.v[c_]; return a; }
EI_DEV vd operator*(vd a, double b) { VFOR a.v[c_] *= b; return a; }
EI_DEV vd operator*(double b, vd a) { VFOR a.v[c_] = b * a.v[c_]; return a; }
EI_DEV vd operator/(vd a, double b) { VFOR a.v[c_] /= b; return a; }
EI_DEV vd operator/(double b, vd a) { VFOR a.v[c_] = b / a.v[c_]; return a; }
EI_DEV vd &operator+=(vd &a, vd b) { VFOR a.v[c_] += b.v[c_]; return a; }
EI_DEV vd &operator-=(vd &a, vd b) { VFOR a.v[c_] -= b.v[c_]; return a; }
// v - a * b with one rounding, spelled out so that every code path (and the CPU emulator) fuses alike
EI_DEV vd vfnma(vd v, vd a, vd b)
{
    VFOR v.v[c_] = fma(-a.v[c_], b.v[c_], v.v[c_]);
    return v;
}
EI_DEV vd vfnma(vd v, double a, vd b)
{
    VFOR v.v[c_] = fma(-a, b.v[c_], v.v[c_]);
    return v;
}
// a * b + c and a * b with one rounding each.  A value recomputed in registers that used to be stored and read
// back has to round like the stored one, whatever else now uses its parts: these spell out which products the
// compilers fused where the value was stored (a product whose only use is one add).
EI_DEV vd vfma(vd a, vd b, vd c)
{
    VFOR c.v[c_] = fma(a.v[c_], b.v[c_], c.v[c_]);
    return c;
}
EI_DEV vd vmul_rn(vd a, vd b)
{
#ifdef EICOS_EMU
    VFOR
    {
        a.v[c_] *= b.v[c_];
        asm("" : "+x"(a.v[c_])); // g++: the product is opaque to -ffp-contract
    }
#else
    VFOR a.v[c_] = __dmul_rn(a.v[c_], b.v[c_]);
#endif
    return a;
}
EI_DEV vd vsqrt(vd a) { VFOR a.v[c_] = sqrt(a.v[c_]); return a; }
EI_DEV vd vabs(vd a) { VFOR a.v[c_] = fabs(a.v[c_]); return a; }
EI_DEV bool ei_isnan(double v) { return v != v; }
EI_DEV double dmax(double a, double b) { return a > b ? a : b; } // std::max(a,b) semantics (returns a on ties / NaN in b)
EI_DEV double dmin(double a, double b) { return b < a ? b : a; } // std::min(a,b)
EI_DEV vd vmax(vd a, vd b) { VFOR a.v[c_] = dmax(a.v[c_], b.v[c_]); return a; }
EI_DEV vd vmin(vd a, vd b) { VFOR a.v[c_] = dmin(a.v[c_], b.v[c_]); return a; }
EI_DEV vd vsel(vb m, vd a, vd b) { VFOR a.v[c_] = m.v[c_] ? a.v[c_] : b.v[c_]; return a; }
EI_DEV vb vbset(bool s)
{
    vb r;
    VFOR r.v[c_] = s;
    return r;
}
EI_DEV vb operator&&(vb a, vb b) { VFOR a.v[c_] = a.v[c_] && b.v[c_]; return a; }
EI_DEV vb operator||(vb a, vb b) { VFOR a.v[c_] = a.v[c_] || b.v[c_]; return a; }
EI_DEV vb operator!(vb a) { VFOR a.v[c_] = !a.v[c_]; return a; }
EI_DEV bool vany(vb a)
{
    bool r = false;
    VFOR r = r || a.v[c_];
    return r;
}
EI_DEV bool vall(vb a)
{
    bool r = true;
    VFOR r = r && a.v[c_];
    return r;
}

EI_DEV vd vload(const double *p) { return *reinterpret_cast<const vd *>(p); }
EI_DEV void vstore(double *p, vd v) { *reinterpret_cast<vd *>(p) = v; }

// 16-byte record of an instruction stream, read by the whole warp from one address (one broadcast
// transaction through the read-only path; the line stays in L1 for the next three records)
#ifdef EICOS_EMU
struct i4
{
    int x, y, z, w;
};
EI_DEV i4 ldg4(const int *p) { return i4{p[0], p[1], p[2], p[3]}; }
#else
typedef int4 i4;
EI_DEV i4 ldg4(const int *p) { return __ldg(reinterpret_cast<const int4 *>(p)); }
#endif
struct alignas(16) d2
{
    double x, y;
};
EI_DEV d2 ldg2(const double *p)
{
#ifdef EICOS_EMU
    return d2{p[0], p[1]};
#else
    const double2 v = __ldg(reinterpret_cast<const double2 *>(p));
    return d2{v.x, v.y};
#endif
}

// proxy for one row of the tile as seen by this lane (VEC instances)
struct RowRef
{
    double *p;
    EI_DEV operator vd() const { return vload(p); }
    EI_DEV void operator=(vd v) const { vstore(p, v); }
    EI_DEV void operator=(double s) const { vstore(p, vset(s)); }
    EI_DEV void operator+=(vd v) const { vstore(p, vload(p) + v); }
    EI_DEV void operator-=(vd v) const { vstore(p, vload(p) - v); }
    EI_DEV void operator*=(double s) const { vstore(p, vload(p) * s); }
    EI_DEV void operator*=(vd s) const { vstore(p, vload(p) * s); }
    EI_DEV void operator=(const RowRef &o) const { vstore(p, vload(o.p)); }
};
#define ROWD(base, r) (RowRef{(base) + (size_t)(r) * TILE})
#define ROWC(base, r, c) ((base)[(size_t)(r) * TILE + (c)])

struct KArgs
{
    DevPattern P;
    Layout L;
    double *ws; // [tiles][rows_total][TILE]
    int *iws;   // [tiles][irows_total][TILE]
    int batch;  // instances handled by this launch's chunk
    int first;  // global index (within the device's batch) of the chunk's first instance
    // instance-major device buffers for load/store (any may be null)
    const double *in_c, *in_h, *in_b;
    const double *base_c, *base_h, *base_b; // raw vectors shared by the batch (used when in_* is null)
    const double *in_G, *in_A;              // per-instance-matrices mode: instance-major raw G / A values (may be null)
    const double *base_G, *base_A;          // ... and the raw values shared by the batch (used when in_G / in_A is null)
    double *out_x, *out_y, *out_z, *out_s;
    int *out_exit, *out_iter;
    double *out_info; // [batch][S_WORK_END]
    int *out_iinfo;   // [batch][J_WORK_END]
    // solveKKT parameters
    // solveKKT jobs of this launch: CTA = (tile, job).  set 0: rhs1 -> sol1, set 1: rhs2 -> sol2 (LdVariant)
    struct KktJob
    {
        int rhs, sol, nitrow, set;
    } job[2];
    int njobs, initialize;
    int variant; // which ring depth of the programs this launch runs (streams.hpp: M_VARIANT_GROUPS)
    int part_doubles; // wide launches: shared memory (doubles) of one warp's machine
    int keep_sticky;
    KSettings settings; // the handle's solver settings (tolerances, iteration limit, refinement, step control)
    int pre_equilibrated; // inputs are already divided by the equilibration vectors
    unsigned int *active_count; // device counter: instances still iterating after the head step
    unsigned long long *ir_rounds; // device counters: [0] solve rounds executed (tile-rounds), [1..5] cycles per solve_kkt phase
};

struct Team
{
    int lane;      // element offset of this lane inside a row (= physical lane * VEC)
    int pl;        // physical lane inside the warp
    int wk, nwk;
    int job;       // eicos_solve_kkt: which of the launch's solveKKT jobs this CTA runs
    double *red;   // [nwk][KRED][TILE]
    double *pbuf;  // worker 0: shared memory of the FMA machine (no lane offset)
#ifdef EICOS_EMU
    std::barrier<> *bar; // workers of a tile are real threads in the emulator
    void sync() const
    {
        if (bar)
            bar->arrive_and_wait();
    }
    bool all(vb v) const { return vall(v); }
    bool any(vb v) const { return vany(v); }
#else
    __device__ __forceinline__ void sync() const { __syncthreads(); }
    __device__ __forceinline__ bool all(vb v) const { return __all_sync(0xffffffffu, vall(v)); }
    __device__ __forceinline__ bool any(vb v) const { return __any_sync(0xffffffffu, vany(v)); }
#endif
};

// ------------------------------------------------------------------ block reductions (fixed order)
template <int K, class Op>
EI_DEV void team_reduce(const Team &tm, vd (&v)[K], Op op)
{
    if (tm.nwk == 1)
        return;
    for (int i0 = 0; i0 < K; i0 += KRED)
    { // the shared buffer holds KRED rows per worker: wide reductions go through it in rounds
        const int kn = K - i0 < KRED ? K - i0 : KRED;
        tm.sync();
        for (int i = 0; i < kn; i++)
            vstore(tm.red + (size_t)(tm.wk * KRED + i) * TILE + tm.lane, v[i0 + i]);
        tm.sync();
        for (int i = 0; i < kn; i++)
        {
            vd s = vload(tm.red + (size_t)i * TILE + tm.lane);
            for (int w = 1; w < tm.nwk; w++)
                s = op(s, vload(tm.red + (size_t)(w * KRED + i) * TILE + tm.lane));
            v[i0 + i] = s;
        }
    }
}
template <int K>
EI_DEV void team_sum(const Team &tm, vd (&v)[K])
{
    team_reduce<K>(tm, v, [](vd a, vd b) { return a + b; });
}
template <int K>
EI_DEV void team_max(const Team &tm, vd (&v)[K])
{
    team_reduce<K>(tm, v, [](vd a, vd b) { return vmax(a, b); });
}
template <int K>
EI_DEV void team_min(const Team &tm, vd (&v)[K])
{
    team_reduce<K>(tm, v, [](vd a, vd b) { return vmin(a, b); });
}

struct TileMem
{
    double *T;        // tile base + this lane's element offset
    int *I;
    const double *Tb; // tile base (row 0, lane 0): source of whole-row bulk copies
};

// Base pointers of a tile as seen by this lane: the lane's element offset is folded in once, so a
// row access is base + row * TILE (one IMAD.WIDE).
EI_DEV TileMem tile_mem(const Team &tm, const KArgs &a, int tile)
{
    TileMem t;
    t.Tb = a.ws + (size_t)tile * a.L.rows_total * TILE;
    t.T = a.ws + (size_t)tile * a.L.rows_total * TILE + tm.lane;
    t.I = a.iws + (size_t)tile * a.L.irows_total * TILE + tm.lane;
    return t;
}

EI_DEV vb lane_active(const Team &tm, const TileMem &t)
{
    vb r;
    VFOR r.v[c_] = ROWC(t.I, J_STATUS, c_) == ST_ACTIVE;
    return r;
}

EI_DEV const double *rowp(const Team &, const double *T, int row) { return T + (size_t)row * TILE; }

// Elementwise pass over `count` rows with NIN input arrays (row offsets in[k]): a worker takes U
// consecutive rows at a time and loads ALL their operands before computing, so U*NIN vector loads
// are in flight per warp instead of one.  body(row, x) gets x[k] = in[k][row] and does the stores.
template <int NIN, int U, class F>
EI_DEV void ew_rows(const Team &tm, const double *T, int count, const int (&in)[NIN], F body)
{
    constexpr int UE = (U * 2 / VEC) > 0 ? (U * 2 / VEC) : 1; // U is quoted for VEC = 2; keep the register footprint constant
    for (int base = tm.wk * UE; base < count; base += tm.nwk * UE)
    {
        vd x[UE][NIN];
#pragma unroll
        for (int u = 0; u < UE; u++)
            if (base + u < count)
#pragma unroll
                for (int k = 0; k < NIN; k++)
                    x[u][k] = vload(rowp(tm, T, in[k] + base + u));
#pragma unroll
        for (int u = 0; u < UE; u++)
            if (base + u < count)
                body(base + u, x[u]);
    }
}

// ------------------------------------------------------------------ W products (src/eicos.cpp:485-507)
// out = W * in for the instances' current scalings; in/out are z-shaped (expanded) row offsets.
EI_DEV void cone_scale(const Team &tm, const KArgs &a, double *T, int in, int out, vb write, bool lp = true)
{
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    if (lp)
    {
        const int ins[3] = {L.lpw, in, out};
        ew_rows<3, 4>(tm, T, P.l, ins, [&](int k, const vd *x) { ROWD(T, out + k) = vsel(write, x[0] * x[1], x[2]); });
    }
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    {
        const int d = EI_LDG(P.cone_dim + c), ks = EI_LDG(P.cone_k + c), qo = EI_LDG(P.cone_q + c);
        VFOR
        {
            const double eta = ROWC(T, L.cpar + c * CP_COUNT + CP_ETA, c_), ca = ROWC(T, L.cpar + c * CP_COUNT + CP_A, c_);
            double zeta = 0.0;
            for (int k = 1; k < d; k++)
                zeta += ROWC(T, L.cq + qo + k - 1, c_) * ROWC(T, in + ks + k, c_);
            const double z0 = ROWC(T, in + ks, c_);
            const double factor = z0 + zeta / (1. + ca);
            if (write.v[c_])
            {
                ROWC(T, out + ks, c_) = eta * (ca * z0 + zeta);
                for (int k = 1; k < d; k++)
                    ROWC(T, out + ks + k, c_) = eta * (ROWC(T, in + ks + k, c_) + factor * ROWC(T, L.cq + qo + k - 1, c_));
            }
        }
    }
}

// ------------------------------------------------------------------ line search (src/eicos.cpp:1380-1469)
// lambda, ds, dz are z-shaped row offsets.  Returns the clamped step for every instance.
// lp = false: the caller has already folded the LP rows into m0 = min ds/lambda, m1 = min dz/lambda.
//
// The reference walks the cones with a running offset and `continue`s past a cone whose lambda has left the
// cone (lknorm2 <= 0) WITHOUT advancing that offset (:1423-1424 against :1462): every later cone is then read
// at the skipped cone's position, with its own dimension.  cone_step() evaluates one cone at a given compact
// z offset; the fast path below uses every cone's own offset, and only instances that hit the `continue` are
// walked again sequentially with the reference's running offset (line_search_misaligned).
struct ConeStep
{
    bool skipped; // lknorm2 <= 0
    double inv;   // 1 / conic_step, or DBL_MAX when the cone does not bound the step
};
// entry k of the cone evaluated at compact z offset `cs`: expanded row zk[cs + k]
template <class RowOf>
EI_DEV ConeStep cone_step(double *T, int lam, int ds, int dz, int d, RowOf row, int c_)
{
    ConeStep r;
    r.skipped = false;
    r.inv = DBL_MAX;
    const double l0 = ROWC(T, lam + row(0), c_);
    double sq = 0.0;
    for (int k = 1; k < d; k++)
    {
        const double v = ROWC(T, lam + row(k), c_);
        sq += v * v;
    }
    const double lknorm2 = l0 * l0 - sq;
    if (lknorm2 <= 0.)
    {
        r.skipped = true;
        return r;
    }
    const double lknorm = sqrt(lknorm2);
    const double lknorminv = 1. / lknorm;
    const double lk0 = l0 / lknorm;
    double dsdot = 0.0, dzdot = 0.0;
    for (int k = 1; k < d; k++)
    {
        const double lkb = ROWC(T, lam + row(k), c_) / lknorm;
        dsdot += lkb * ROWC(T, ds + row(k), c_);
        dzdot += lkb * ROWC(T, dz + row(k), c_);
    }
    const double ds0 = ROWC(T, ds + row(0), c_), dz0 = ROWC(T, dz + row(0), c_);
    const double lds = lk0 * ds0 - dsdot, ldz = lk0 * dz0 - dzdot;
    const double rho0 = lknorminv * lds, sig0 = lknorminv * ldz;
    const double frho = (lds + ds0) / (lk0 + 1.), fsig = (ldz + dz0) / (lk0 + 1.);
    double ar = 0.0, as = 0.0;
    for (int k = 1; k < d; k++)
    {
        const double lkb = ROWC(T, lam + row(k), c_) / lknorm;
        const double rr = lknorminv * (ROWC(T, ds + row(k), c_) - frho * lkb);
        const double ss = lknorminv * (ROWC(T, dz + row(k), c_) - fsig * lkb);
        ar += rr * rr;
        as += ss * ss;
    }
    const double rhonorm = sqrt(ar) - rho0, signorm = sqrt(as) - sig0;
    const double conic_step = dmax(0., dmax(signorm, rhonorm));
    if (conic_step != 0.)
        r.inv = 1. / conic_step;
    return r;
}
// One instance (element c_ of this lane), all cones in order with the reference's running offset.
EI_DEV double line_search_misaligned(const KArgs &a, double *T, int lam, int ds, int dz, int c_)
{
    const DevPattern &P = a.P;
    double best = DBL_MAX;
    int cs = P.l; // compact z offset (the LP rows come first)
    for (int c = 0; c < P.nc; c++)
    {
        const int d = EI_LDG(P.cone_dim + c);
        const int base = cs;
        // (a misaligned cone may reach past the last z entry in the reference - undefined behaviour there; here the
        //  walk stops at the end of z)
        if (base + d > P.m)
            break;
        const ConeStep r = cone_step(T, lam, ds, dz, d, [&](int k) { return EI_LDG(P.zk + base + k); }, c_);
        if (r.skipped)
            continue; // the offset stays where it is
        best = dmin(best, r.inv);
        cs += d;
    }
    return best;
}
EI_DEV vd line_search(const Team &tm, const KArgs &a, double *T, int lam, int ds, int dz,
                      vd tau, vd dtau, vd kap, vd dkap, bool lp = true, vd m0 = vset(DBL_MAX), vd m1 = vset(DBL_MAX))
{
    const DevPattern &P = a.P;
    vd mn[3] = {m0, m1, vset(DBL_MAX)}; // rhomin, sigmamin, min over cones of 1/conic_step
    if (lp)
    {
        const int ins[3] = {lam, ds, dz};
        ew_rows<3, 4>(tm, T, P.l, ins, [&](int, const vd *x) {
            mn[0] = vmin(mn[0], x[1] / x[0]);
            mn[1] = vmin(mn[1], x[2] / x[0]);
        });
    }
    vd skipped[1] = {vset(0.0)}; // 1 where an instance has hit the `continue` with cones still to come
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    {
        const int d = EI_LDG(P.cone_dim + c), zs = EI_LDG(P.cone_k + c);
        VFOR
        {
            const ConeStep r = cone_step(T, lam, ds, dz, d, [&](int k) { return zs + k; }, c_);
            if (r.skipped)
            {
                if (c + 1 < P.nc)
                    skipped[0].v[c_] = 1.0;
                continue;
            }
            mn[2].v[c_] = dmin(mn[2].v[c_], r.inv);
        }
    }
    team_max<1>(tm, skipped);
    {
        vb sk;
        VFOR sk.v[c_] = skipped[0].v[c_] != 0.0;
        if (tm.any(sk))
        { // rare: walk those instances again the way the reference does (every worker computes the same values)
            team_min<3>(tm, mn);
            VFOR if (sk.v[c_]) mn[2].v[c_] = line_search_misaligned(a, T, lam, ds, dz, c_);
        }
    }
    team_min<3>(tm, mn);
    vd res;
    VFOR
    {
        double alpha;
        if (P.l > 0)
        {
            const double rhomin = mn[0].v[c_], sigmamin = mn[1].v[c_];
            const double eps = 1e-13;
            if (-sigmamin > -rhomin)
                alpha = sigmamin < 0. ? 1. / (-sigmamin) : 1. / eps;
            else
                alpha = rhomin < 0. ? 1. / (-rhomin) : 1. / eps;
        }
        else
            alpha = 10.;
        const double mt = -tau.v[c_] / dtau.v[c_], mk = -kap.v[c_] / dkap.v[c_];
        if (mt > 0. && mt < alpha)
            alpha = mt;
        if (mk > 0. && mk < alpha)
            alpha = mk;
        alpha = dmin(mn[2].v[c_], alpha);
        // std::clamp(alpha, stepmin, stepmax)
        if (alpha < a.settings.stepmin)
            alpha = a.settings.stepmin;
        else if (a.settings.stepmax < alpha)
            alpha = a.settings.stepmax;
        res.v[c_] = alpha;
    }
    return res;
}

// ------------------------------------------------------------------ TMA bulk copies and mbarriers (sm_100a)
#ifndef EICOS_EMU
EI_DEV void mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
EI_DEV void mbar_inval(unsigned bar) { asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar) : "memory"); }
EI_DEV void mbar_arrive(unsigned bar)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
EI_DEV void mbar_arrive_expect(unsigned bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
EI_DEV bool mbar_try_wait(unsigned bar, unsigned parity)
{
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
    return ok != 0;
}
EI_DEV void mbar_wait(unsigned bar, unsigned parity)
{
    while (!mbar_try_wait(bar, parity))
    {
    }
}
// one row (or one chunk of a record stream) global -> shared, completion counted on the mbarrier
EI_DEV void bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
#endif

// ------------------------------------------------------------------ the FMA machine (machine.hpp)
// Shared memory of one program warp: [ops ring][load-list ring][mbarriers][rows: 0, -0, scratch, slots, data ring].
constexpr int ROW_BYTES = TILE * (int)sizeof(double);
constexpr int M_CHUNK_BYTES = M_CHUNK_WORDS * 4;
constexpr int M_OPS_RING_BYTES = M_CHUNKS * M_CHUNK_BYTES;
constexpr int M_LD_CHUNK_BYTES = M_LD_CHUNK_WORDS * 4;
constexpr int M_LD_RING_BYTES = M_LD_CHUNKS * M_LD_CHUNK_BYTES;
#ifndef EICOS_TMA_RING
#define EICOS_TMA_RING 0 // 1: data ring fed by bulk copies (one lane per row, one mbarrier per group) - measured slower, DESIGN.md section 4; 0: cp.async per lane
#endif
constexpr int M_BAR_BYTES = 192; // M_CHUNKS + M_LD_CHUNKS mbarriers, then one per ring group (M_MAX_RING_GROUPS)
static_assert((M_CHUNKS + M_LD_CHUNKS + M_MAX_RING_GROUPS) * 8 <= M_BAR_BYTES, "mbarriers");
constexpr int M_HEAD_DOUBLES = (M_OPS_RING_BYTES + M_LD_RING_BYTES + M_BAR_BYTES) / 8;
constexpr int M_BUNDLE_BYTES = M_BUNDLE_WORDS * 4;
#ifndef EICOS_EMU
static_assert(ROW_BYTES == (1 << M_FIELD_SHIFT), "a field is the byte offset of a 512-byte row");
#endif
inline size_t machine_smem_doubles(int slot_budget, int ring_groups, int nr = 1)
{
    return M_HEAD_DOUBLES + (size_t)(m_row_slot0(nr) + nr * slot_budget + ring_groups * M_RING_GROUP) * TILE;
}

// what the interpreter compiles in for a kernel (everything else costs no instructions)
enum : int
{
    MC_CONST = 1,  // MF_ACONST / MF_CCONST
    MC_POS = 2,    // MF_POS
    MC_BKEEP = 4,  // MF_BKEEP
    MC_RECIP = 8,  // MF_RECIP
    MC_FIN = 16,   // MF_FIN
    MC_OUT2 = 32,  // MF_OUT2
    MC_AONE = 64,  // MF_AONE
    MC_X3 = 128    // finish functors read a fourth operand (field w6), loaded with the other operands
};

// one run of a program on a tile
struct MRun
{
    DevMachine prog;
    const int *ld;     // materialised load list of this use
    const double *Tb;  // tile base (row 0, lane 0)
    double *out, *out2; // out bases (+ this lane's element offset)
    double *outB, *out2B; // ... of the second job (two-job programs)
    bool a_one;
};

EI_DEV double words_double(int lo, int hi)
{
#ifdef EICOS_EMU
    double v;
    const int w[2] = {lo, hi};
    std::memcpy(&v, w, 8);
    return v;
#else
    return __hiloint2double(hi, lo);
#endif
}

struct Machine
{
#ifdef EICOS_EMU
    double *rows;
    EI_DEV void init(const Team &, double *mem) { rows = mem + M_HEAD_DOUBLES; }
    EI_DEV vd ld(int f) const { return vload(rows + (size_t)(f >> M_FIELD_SHIFT) * TILE); }
    EI_DEV void st(int f, vd v) const { vstore(rows + (size_t)(f >> M_FIELD_SHIFT) * TILE, v); }

    template <int CFG, int NR, class Fin>
    EI_DEV void run(const Team &, const MRun &r, Fin &fin)
    {
        for (int c = 0; c < VEC; c++)
            for (int j = 0; j < NR; j++)
            {
                rows[(size_t)(M_ROW_ZERO + j) * TILE + c] = 0.0;
                rows[(size_t)(m_row_negzero(NR) + j) * TILE + c] = -0.0;
            }
        const int ring_rows = r.prog.ring_groups * M_RING_GROUP;
        long long issued = 0; // ring groups copied so far
        const auto refill = [&]() {
            for (int k = 0; k < M_RING_GROUP; k++)
            {
                const long long idx = issued * M_RING_GROUP + k;
                const int w = r.ld[idx];
                std::memcpy(rows + (size_t)(r.prog.ring_row0 + idx % ring_rows) * TILE, r.Tb + (size_t)w * TILE, ROW_BYTES);
            }
            issued++;
        };
        for (int g = 0; g < r.prog.ring_groups; g++)
            refill();
        const int *rec = r.prog.ops;
        const int JB = 1 << M_FIELD_SHIFT; // field offset of the second job's row
        for (;; rec += M_BUNDLE_WORDS)
        {
            const int ctrl = rec[4];
            vd res[M_U][NR], bv[M_U][NR], xv[M_U][NR];
            for (int u = 0; u < M_U; u++)
            {
                const int *w = rec + u * M_REC_WORDS;
                const int f = w[4];
                const double cst = words_double(w[6], w[7]);
                vd a = (CFG & MC_CONST) && (f & MF_ACONST) ? vset(cst) : ld(w[0]);
                if ((CFG & MC_AONE) && (f & MF_AONE) && r.a_one)
                    a = vset(1.0);
                if ((CFG & MC_POS) && f < 0)
                    a = -a;
                for (int j = 0; j < NR; j++)
                {
                    xv[u][j] = (CFG & MC_X3) && (f & MF_X3) ? ld(w[6] + j * JB) : vset(0.0);
                    const vd b = ld(w[1] + j * JB);
                    const vd c = (CFG & MC_CONST) && (f & MF_CCONST) ? vset(cst) : ld(w[2] + j * JB);
                    vd v = vfnma(c, a, b);
                    if ((CFG & MC_RECIP) && (f & MF_RECIP))
                        v = 1.0 / c;
                    res[u][j] = v;
                    bv[u][j] = b;
                }
            }
            for (int u = 0; u < M_U; u++)
            {
                const int *w = rec + u * M_REC_WORDS;
                const int f = w[4];
                for (int j = 0; j < NR; j++)
                {
                    st(w[3] + j * JB, res[u][j]);
                    if (f & MF_OUT)
                    {
                        double *o = (CFG & MC_OUT2) && (f & MF_OUT2) ? (j ? r.out2B : r.out2) : (j ? r.outB : r.out);
                        vstore(o + (size_t)w[5] * TILE, res[u][j]);
                    }
                    if ((CFG & MC_BKEEP) && (f & MF_BKEEP))
                        st(w[5] + j * JB, bv[u][j]);
                }
                if ((CFG & MC_FIN) && (f & MF_FIN))
                    fin((f >> MF_KIND_SHIFT) & 15, w[5], res[u], bv[u], xv[u]);
            }
            for (int k = (ctrl >> MF_NREL_SHIFT) & 31; k > 0; k--)
                refill();
            if (ctrl & MF_END)
                break;
        }
    }
#else
    unsigned rows; // shared address of the rows region + this lane's 16 bytes
    unsigned opsb; // shared address of the ops ring
    unsigned ldb;  // shared address of the load-list ring
    unsigned bars; // mbarriers: M_CHUNKS of the ops chunks, then M_LD_CHUNKS of the load-list chunks
    int pl;
    // data ring: every lane moves its 16 bytes of a row (cp.async), one commit group per ring group
    const char *Tl;   // tile base + this lane's 16 bytes
    const char *Tb0;  // tile base
    unsigned ring0;   // shared address of ring row 0 (+ lane)
    int rg;           // ring groups
    unsigned gbar;    // TMA ring: mbarriers of the ring groups
    int gslot, gphase, gwaited; // ... group the consumer waits for next (its ring position and phase parity), groups waited for
    int gneed;        // ... groups the bundles so far have asked for (sum of their NEWG fields)
    int head;         // ring group the next refill lands in
    int lgroup;       // load-list group the next refill reads
    const int *ldg;   // global pointer of the next load-list chunk to fetch
    int ld_nchunks, ld_fetched;
    // ops ring: the record stream arrives in 1 KB chunks by TMA bulk copies (one elected lane)
    const int *opsg;  // global pointer of the next chunk to fetch
    int nchunks, fetched;

    __device__ __forceinline__ void init(const Team &tm, double *mem)
    {
        pl = tm.pl;
        opsb = (unsigned)__cvta_generic_to_shared(mem);
        ldb = opsb + M_OPS_RING_BYTES;
        bars = ldb + M_LD_RING_BYTES;
        rows = bars + M_BAR_BYTES + 16u * pl;
    }
    static __device__ __forceinline__ i4 lds4(unsigned a)
    {
        i4 r;
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(a));
        return r;
    }
    __device__ __forceinline__ vd ld(int f) const
    {
        vd r;
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(r.v[0]), "=d"(r.v[1]) : "r"(rows + (unsigned)f));
        return r;
    }
    __device__ __forceinline__ void st(int f, vd v) const
    {
        asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(rows + (unsigned)f), "d"(v.v[0]), "d"(v.v[1]) : "memory");
    }
    // the row behind it (the second job's row of a vector operand)
    __device__ __forceinline__ vd ldB(int f) const
    {
        vd r;
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+512];" : "=d"(r.v[0]), "=d"(r.v[1]) : "r"(rows + (unsigned)f));
        return r;
    }
    __device__ __forceinline__ void stB(int f, vd v) const
    {
        asm volatile("st.shared.v2.f64 [%0+512], {%1, %2};" ::"r"(rows + (unsigned)f), "d"(v.v[0]), "d"(v.v[1]) : "memory");
    }
    __device__ __forceinline__ void issue_row(unsigned dst, int w) const
    { // ring row <- workspace row w of the tile (padding words of the materialised list name row 0).
      // One IMAD.WIDE for the address: left to itself the compiler re-derives it from the tile index (7 instructions).
        unsigned long long src;
        asm volatile("mad.wide.s32 %0, %1, 512, %2;" : "=l"(src) : "r"(w), "l"(Tl));
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
    }
    static __device__ __forceinline__ void out_row(const double *base, int w, vd v)
    { // global row w behind an out base (one IMAD.WIDE for the address, like issue_row)
        unsigned long long dst;
        asm volatile("mad.wide.s32 %0, %1, 512, %2;" : "=l"(dst) : "r"(w), "l"(base));
        asm volatile("st.global.v2.f64 [%0], {%1, %2};" ::"l"(dst), "d"(v.v[0]), "d"(v.v[1]) : "memory");
    }
    __device__ __forceinline__ void fetch_ld_chunk()
    { // next chunk of the load list into its ring position
        if (pl == 0)
        {
            const unsigned slot = (unsigned)ld_fetched % M_LD_CHUNKS;
            const unsigned bar = bars + 8u * (M_CHUNKS + slot);
            mbar_arrive_expect(bar, M_LD_CHUNK_BYTES);
            bulk_g2s(ldb + slot * M_LD_CHUNK_BYTES, ldg, M_LD_CHUNK_BYTES, bar);
        }
        ld_fetched++;
        ldg += M_LD_CHUNK_WORDS;
    }
    __device__ __forceinline__ void issue_group()
    { // the next M_RING_GROUP words of the load list into ring group `head`
        const int gc = lgroup % M_LD_CHUNK_GROUPS;
        if (gc == 0)
        { // entering a new chunk of the load list: the one before it is free, this one must have landed
            const int c = lgroup / M_LD_CHUNK_GROUPS;
            // (the words of the chunk being replaced were read - and used - long ago: no cross-proxy fence needed
            //  between those generic reads and the bulk copy's write; a fence here waits for every copy in flight)
            if (c > 0 && ld_fetched < ld_nchunks)
                fetch_ld_chunk();
            mbar_wait(bars + 8u * (M_CHUNKS + (unsigned)c % M_LD_CHUNKS), ((unsigned)c / M_LD_CHUNKS) & 1u);
        }
        const unsigned la = ldb + (unsigned)(lgroup % (M_LD_CHUNKS * M_LD_CHUNK_GROUPS)) * (M_RING_GROUP * 4);
#if EICOS_TMA_RING
        // lane k < 8 copies row k of the group: one arrival (+512 bytes expected) and one bulk copy each; the group's
        // mbarrier (8 arrivals) completes when all eight rows have landed
        // (a group that only padding pops ran over is released without ever having been read: its mbarrier must
        //  still have been waited for before the ring position is armed again)
        while (gwaited + rg <= lgroup)
            wait_next_group();
        if (pl < M_RING_GROUP)
        {
            int w;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w) : "r"(la + 4u * (unsigned)pl));
            unsigned long long src;
            asm volatile("mad.wide.s32 %0, %1, 512, %2;" : "=l"(src) : "r"(w), "l"(Tb0));
            const unsigned bar = gbar + 8u * (unsigned)head;
            mbar_arrive_expect(bar, ROW_BYTES);
            bulk_g2s(ring0 + (unsigned)head * (M_RING_GROUP * ROW_BYTES) + (unsigned)pl * (ROW_BYTES - 16), (const void *)src, ROW_BYTES, bar);
        }
        lgroup++;
        head = head + 1 == rg ? 0 : head + 1;
        return;
#endif
        const i4 nw0 = lds4(la), nw1 = lds4(la + 16);
        lgroup++;
        const unsigned d = ring0 + (unsigned)head * (M_RING_GROUP * ROW_BYTES);
        issue_row(d, nw0.x);
        issue_row(d + ROW_BYTES, nw0.y);
        issue_row(d + 2 * ROW_BYTES, nw0.z);
        issue_row(d + 3 * ROW_BYTES, nw0.w);
        issue_row(d + 4 * ROW_BYTES, nw1.x);
        issue_row(d + 5 * ROW_BYTES, nw1.y);
        issue_row(d + 6 * ROW_BYTES, nw1.z);
        issue_row(d + 7 * ROW_BYTES, nw1.w);
        asm volatile("cp.async.commit_group;" ::: "memory");
        head = head + 1 == rg ? 0 : head + 1;
    }
    __device__ __forceinline__ void issue_chunk()
    { // next chunk of the record stream into its ring position (lane 0 only)
        const unsigned slot = (unsigned)fetched % M_CHUNKS;
        const unsigned bar = bars + 8u * slot;
        mbar_arrive_expect(bar, M_CHUNK_BYTES);
        bulk_g2s(opsb + slot * M_CHUNK_BYTES, opsg, M_CHUNK_BYTES, bar);
    }
    __device__ __forceinline__ void wait_next_group()
    { // TMA ring: the next group in load-list order has landed
        mbar_wait(gbar + 8u * (unsigned)gslot, (unsigned)gphase);
        gwaited++;
        if (++gslot == rg)
            gslot = 0, gphase ^= 1;
    }
    static __device__ __forceinline__ void wait_groups(int code)
    { // machine.hpp: M_WAIT_N.  Called only when code > 0 (most bundles read rows of groups that were waited for
      // already: one test instead of seven); the shallow ring's codes first.
        static_assert(M_WAIT_N[1] == 0 && M_WAIT_N[2] == 1 && M_WAIT_N[3] == 2 && M_WAIT_N[4] == 3 && M_WAIT_N[5] == 5 &&
                          M_WAIT_N[6] == 8 && M_WAIT_N[7] == 12,
                      "wait codes");
        if (code == 3)
            asm volatile("cp.async.wait_group 2;" ::: "memory");
        else if (code == 2)
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        else if (code == 1)
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        else if (code == 4)
            asm volatile("cp.async.wait_group 3;" ::: "memory");
        else if (code == 5)
            asm volatile("cp.async.wait_group 5;" ::: "memory");
        else if (code == 6)
            asm volatile("cp.async.wait_group 8;" ::: "memory");
        else
            asm volatile("cp.async.wait_group 12;" ::: "memory");
    }

    template <int CFG, int NR, class Fin>
    __device__ __forceinline__ void run(const Team &, const MRun &r, Fin &fin)
    {
        static_assert(ROW_BYTES == 512, "ldB / stB address the next row as +512");
        __syncwarp();
        if (pl == 0)
        { // (every run invalidates its barriers when it is done, so the memory may be another machine's next time)
            for (int b = 0; b < M_CHUNKS + M_LD_CHUNKS; b++)
                mbar_init(bars + 8u * b, 1);
#if EICOS_TMA_RING
            for (int b = 0; b < M_MAX_RING_GROUPS; b++)
                mbar_init(bars + 8u * (M_CHUNKS + M_LD_CHUNKS + b), M_RING_GROUP);
#endif
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        st(M_ROW_ZERO * ROW_BYTES, vset(0.0));
        st((NR * ROW_BYTES), vset(-0.0));
        if (NR == 2)
        {
            stB(M_ROW_ZERO * ROW_BYTES, vset(0.0));
            stB((NR * ROW_BYTES), vset(-0.0));
        }
        // ops ring and load-list ring
        nchunks = r.prog.nchunks;
        opsg = r.prog.ops;
        fetched = 0;
        for (int c = 0; c < M_CHUNKS && c < nchunks; c++)
        {
            if (pl == 0)
                issue_chunk();
            fetched++;
            opsg += M_CHUNK_WORDS;
        }
        ld_nchunks = r.prog.nld_chunks;
        ldg = r.ld;
        ld_fetched = 0;
        for (int c = 0; c < M_LD_CHUNKS && c < ld_nchunks; c++)
            fetch_ld_chunk();
        // data ring: the first groups of the load list (the list is padded with M_LD_NONE)
        Tl = (const char *)r.Tb + 16 * pl;
        Tb0 = (const char *)r.Tb;
        gbar = bars + 8u * (M_CHUNKS + M_LD_CHUNKS);
        gslot = 0, gphase = 0, gwaited = 0, gneed = 0;
        rg = r.prog.ring_groups;
        ring0 = rows + (unsigned)r.prog.ring_row0 * ROW_BYTES;
        head = 0;
        lgroup = 0;
        for (int g = 0; g < rg; g++)
            issue_group();
        mbar_wait(bars, 0);
        unsigned pos = 0; // byte position of the current bundle in the ops ring
        int cons = 0;     // chunk being consumed
        const int aone_mask = r.a_one ? MF_AONE : 0;
        i4 ra[M_U], rb[M_U];
#pragma unroll
        for (int u = 0; u < M_U; u++)
        {
            ra[u] = lds4(opsb + 32u * u);
            rb[u] = lds4(opsb + 32u * u + 16u);
        }
        for (;;)
        {
            const int ctrl = rb[0].x;
#if EICOS_TMA_RING
            gneed += (ctrl >> MF_NEWG_SHIFT) & 31;
            while (gwaited < gneed)
                wait_next_group();
#else
            if (ctrl & (7 << MF_WAIT_SHIFT))
                wait_groups((ctrl >> MF_WAIT_SHIFT) & 7);
#endif
            // ---- operand loads (A: one row; B, C, x3: one row per job)
            vd a[M_U], b[M_U][NR], c[M_U][NR], x3[M_U][NR];
            int fl[M_U], kf[M_U], w5[M_U];
#pragma unroll
            for (int u = 0; u < M_U; u++)
            {
                fl[u] = rb[u].x;
                kf[u] = ra[u].w;
                w5[u] = rb[u].y;
                b[u][0] = ld(ra[u].y);
                if (NR == 2)
                    b[u][NR - 1] = ldB(ra[u].y);
                if (CFG & MC_X3)
                {
                    if (fl[u] & MF_X3)
                    {
                        x3[u][0] = ld(rb[u].z);
                        if (NR == 2)
                            x3[u][NR - 1] = ldB(rb[u].z);
                    }
                    else
                    {
#pragma unroll
                        for (int j = 0; j < NR; j++)
                            x3[u][j] = vset(0.0);
                    }
                }
                if (CFG & MC_CONST)
                {
                    const double cst = __hiloint2double(rb[u].w, rb[u].z);
                    if (fl[u] & MF_ACONST)
                        a[u] = vset(cst);
                    else
                        a[u] = ld(ra[u].x);
                    if (fl[u] & MF_CCONST)
                    {
#pragma unroll
                        for (int j = 0; j < NR; j++)
                            c[u][j] = vset(cst);
                    }
                    else
                    {
                        c[u][0] = ld(ra[u].z);
                        if (NR == 2)
                            c[u][NR - 1] = ldB(ra[u].z);
                    }
                }
                else
                {
                    a[u] = ld(ra[u].x);
                    c[u][0] = ld(ra[u].z);
                    if (NR == 2)
                        c[u][NR - 1] = ldB(ra[u].z);
                }
            }
            // ---- the records of the next bundle (the chunk behind a boundary was fetched M_CHUNKS - 1 chunks ago)
            const bool last = (ctrl & MF_END) != 0;
            pos += M_BUNDLE_BYTES;
            if ((pos & (M_CHUNK_BYTES - 1)) == 0)
            {
                // the chunk just read is free: it takes the next chunk of the stream
                if (fetched < nchunks)
                {
                    if (pl == 0)
                        issue_chunk();
                    fetched++;
                    opsg += M_CHUNK_WORDS;
                }
                cons++;
                if (cons < nchunks)
                    mbar_wait(bars + 8u * ((unsigned)cons % M_CHUNKS), ((unsigned)cons / M_CHUNKS) & 1u);
                pos &= M_OPS_RING_BYTES - 1;
            }
#pragma unroll
            for (int u = 0; u < M_U; u++)
            {
                ra[u] = lds4(opsb + pos + 32u * u);
                rb[u] = lds4(opsb + pos + 32u * u + 16u);
            }
            // ---- multiply-adds
            vd res[M_U][NR];
#pragma unroll
            for (int u = 0; u < M_U; u++)
            {
                vd av = a[u];
                if ((CFG & MC_AONE) && (fl[u] & aone_mask))
                    av = vset(1.0);
                if (CFG & MC_POS)
                { // flip the sign of A where the flag (bit 31) is set
                    VFOR av.v[c_] = __hiloint2double(__double2hiint(av.v[c_]) ^ (fl[u] & (int)0x80000000), __double2loint(av.v[c_]));
                }
#pragma unroll
                for (int j = 0; j < NR; j++)
                    res[u][j] = vfnma(c[u][j], av, b[u][j]);
                if ((CFG & MC_RECIP) && (fl[u] & MF_RECIP))
                { // (a real branch: the division is long and rare)
                    asm volatile("" ::: "memory");
#pragma unroll
                    for (int j = 0; j < NR; j++)
                        res[u][j] = 1.0 / c[u][j];
                }
            }
            // ---- stores
#pragma unroll
            for (int u = 0; u < M_U; u++)
            {
                st(kf[u], res[u][0]);
                if (NR == 2)
                    stB(kf[u], res[u][NR - 1]);
                if (fl[u] & MF_OUT)
                {
                    const bool second = (CFG & MC_OUT2) && (fl[u] & MF_OUT2);
                    out_row(second ? r.out2 : r.out, w5[u], res[u][0]);
                    if (NR == 2)
                        out_row(second ? r.out2B : r.outB, w5[u], res[u][NR - 1]);
                }
                if ((CFG & MC_BKEEP) && (fl[u] & MF_BKEEP))
                {
                    st(w5[u], b[u][0]);
                    if (NR == 2)
                        stB(w5[u], b[u][NR - 1]);
                }
                if ((CFG & MC_FIN) && (fl[u] & MF_FIN))
                    fin((fl[u] >> MF_KIND_SHIFT) & 15, w5[u], res[u], b[u], x3[u]);
            }
            // ---- refills of the ring groups this bundle finished with
#if EICOS_TMA_RING
            if (ctrl & MF_FENCE)
            { // a row this refill copies was written by the program (other lanes' generic stores): order them in
              // front of the async proxy's reads
                __syncwarp();
                asm volatile("fence.proxy.async;" ::: "memory");
            }
#endif
            for (int k = (ctrl >> MF_NREL_SHIFT) & 31; k > 0; k--)
                issue_group();
            if (last)
                break;
        }
        // nothing may still be in flight when the machine is re-opened or the CTA exits
#if EICOS_TMA_RING
        while (gwaited < lgroup)
            wait_next_group();
#else
        asm volatile("cp.async.wait_all;" ::: "memory");
#endif
        for (int c = cons + 1; c < fetched; c++)
            mbar_wait(bars + 8u * ((unsigned)c % M_CHUNKS), ((unsigned)c / M_CHUNKS) & 1u);
        for (int c = (lgroup + M_LD_CHUNK_GROUPS - 1) / M_LD_CHUNK_GROUPS; c < ld_fetched; c++)
            mbar_wait(bars + 8u * (M_CHUNKS + (unsigned)c % M_LD_CHUNKS), ((unsigned)c / M_LD_CHUNKS) & 1u);
        __syncwarp();
        if (pl == 0)
            for (int b = 0; b < M_CHUNKS + M_LD_CHUNKS + (EICOS_TMA_RING ? M_MAX_RING_GROUPS : 0); b++)
                mbar_inval(bars + 8u * b);
        __syncwarp();
    }
#endif
};

// finish functors see (kind, w5, result[NR], B[NR], x3[NR])
struct NoFin
{
    template <int NR>
    EI_DEV void operator()(int, int, const vd (&)[NR], const vd (&)[NR], const vd (&)[NR]) {}
};

// ------------------------------------------------------------------ numeric LDL' (Eigen factorize, src/eicos.cpp:900,1164)
// Right-looking in elimination order, one warp per tile, as a machine program (streams.cpp: build_factor):
// HBM traffic is the scaling block V in, L and 1/D out.  Like Eigen the factorisation fails only on an
// exactly zero pivot (the reciprocal is infinite).
struct PivotFin
{
    vb zero_pivot;
    EI_DEV void operator()(int, int, const vd (&res)[1], const vd (&)[1], const vd (&)[1])
    {
        VFOR zero_pivot.v[c_] = zero_pivot.v[c_] || fabs(res[0].v[c_]) > DBL_MAX;
    }
};
EI_DEV void tile_factor(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const vb act = lane_active(tm, t);
    if (!tm.any(act))
        return;
    if (tm.wk != 0)
        return;
    Machine mm;
    mm.init(tm, tm.pbuf);
    PivotFin fin;
    fin.zero_pivot = vbset(false);
    MRun r;
    r.prog = a.P.fa[a.variant];
    r.ld = a.P.fa_ld[a.variant];
    r.Tb = t.Tb;
    r.out = r.out2 = r.outB = r.out2B = t.T;
    r.a_one = false;
    mm.run<MC_CONST | MC_POS | MC_BKEEP | MC_RECIP | MC_FIN, 1>(tm, r, fin);
    VFOR if (fin.zero_pivot.v[c_] && act.v[c_]) ROWC(t.I, J_STATUS, c_) = EXIT_FATAL;
}

// ------------------------------------------------------------------ triangular solves and KKT residual (machine programs)
// forward:  xw = L^-1 P rhs         rows of L in dot form, ascending columns (the summation order of Eigen's
//                                   forward substitution); the permutation is folded into the loads.
// backward: out = P' L^-T D^-1 xw   columns in reverse order, dot form; results land in KKT order; the
//                                   accumulating form also does x += out for the instances with `cont`.
// residual: e = rhs - Ktrue * x     with the un-regularised scaling block (src/eicos.cpp:1511-1576)
// All three are programs of the FMA machine (streams.cpp: build_forward / build_backward / build_matvec).
template <int NR>
struct AccFin
{
    vb cont[NR];
    double *x[NR]; // accumulated solutions (+ lane)
    EI_DEV void operator()(int, int row, const vd (&res)[NR], const vd (&)[NR], const vd (&xa)[NR])
    {
#pragma unroll
        for (int j = 0; j < NR; j++)
            vstore(x[j] + (size_t)row * TILE, xa[j] + vsel(cont[j], res[j], vset(0.0)));
    }
};
template <int NR>
struct AbsMaxFin
{
    vd nerr[NR];
    EI_DEV void operator()(int, int, const vd (&res)[NR], const vd (&)[NR], const vd (&)[NR])
    {
#pragma unroll
        for (int j = 0; j < NR; j++)
            nerr[j] = vmax(nerr[j], vabs(res[j]));
    }
};

// e[j] = rhs[j] - Ktrue * x[j], nerr[j] = ||e[j]||_inf per instance.  mvld: the materialised mat-vec load list of this use.
// set: job set of a one-job solve (selects the load lists of the part programs in a wide launch)
template <int NR>
EI_DEV void kkt_residual(const Team &tm, const KArgs &a, Machine &mm, const TileMem &t, const DevMachine &prog, const int *mvld,
                         const int (&x)[NR], const int (&erow)[NR], bool initialize, vd (&nerr)[NR], int set = 0)
{
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    const double delta = Settings::deltastat;
    const int zb = P.n + P.p;
#pragma unroll
    for (int j = 0; j < NR; j++)
        nerr[j] = vset(0.0);
    // wide launch (one-job solves only): the rows are split into M_MV_PARTS independent programs, one warp each, every
    // warp with a machine of its own; max |e| is combined by team_max below (order-independent: same bits as one warp)
    const bool wide = NR == 1 && tm.nwk >= M_MV_PARTS;
    if ((wide ? tm.wk < M_MV_PARTS : tm.wk == 0) && P.mv_rows > 0)
    {
        AbsMaxFin<NR> fin;
#pragma unroll
        for (int j = 0; j < NR; j++)
            fin.nerr[j] = vset(0.0);
        Machine mw;
        if (wide)
            mw.init(tm, tm.pbuf + (size_t)tm.wk * a.part_doubles);
        Machine &mrun = wide ? mw : mm;
        MRun r;
        r.prog = wide ? P.mvw[tm.wk] : prog;
        r.ld = wide ? P.mvw_ld[set][tm.wk] : mvld;
        r.Tb = t.Tb;
        r.out = r.out2 = T + (size_t)erow[0] * TILE;
        r.outB = r.out2B = T + (size_t)erow[NR - 1] * TILE;
        r.a_one = false;
        mrun.template run<MC_CONST | MC_BKEEP | MC_FIN, NR>(tm, r, fin);
#pragma unroll
        for (int j = 0; j < NR; j++)
            nerr[j] = fin.nerr[j];
    }
    if (P.nc > 0)
    {
        tm.sync(); // (workers > 1) the partial cone rows written by the program warps are visible
        for (int c = tm.wk; c < P.nc; c += tm.nwk)
        {
            const int d = EI_LDG(P.cone_dim + c), ks = EI_LDG(P.cone_k + c), qo = EI_LDG(P.cone_q + c);
            const int kb = zb + ks; // KKT row of the cone's first entry
            const int cp = L.cpar + c * CP_COUNT;
            const vd eta2 = ROWD(T, cp + CP_ETA2), d1 = ROWD(T, cp + CP_D1), u0 = ROWD(T, cp + CP_U0);
            const vd u1 = ROWD(T, cp + CP_U1), v1 = ROWD(T, cp + CP_V1);
            for (int j = 0; j < NR; j++)
            {
                const int xj = x[j], ej = erow[j];
                const vd x1 = ROWD(T, xj + kb), x3 = ROWD(T, xj + kb + d), x4 = ROWD(T, xj + kb + d + 1);
                vd qtx2 = vset(0.0);
                for (int k = 1; k < d; k++)
                    qtx2 += vd(ROWD(T, L.cq + qo + k - 1)) * vd(ROWD(T, xj + kb + k));
                const vd vu = v1 * x3 + u1 * x4;
                for (int k = 0; k < d; k++)
                {
                    const vd xk = ROWD(T, xj + kb + k);
                    vd v = ROWD(T, ej + kb + k); // rhs - G x from the mat-vec program
                    if (k < d - 1)
                        v += delta * xk;
                    else
                        v -= delta * xk;
                    if (initialize)
                        v += xk;
                    else if (k == 0)
                        v += eta2 * (d1 * x1 + u0 * x4);
                    else
                        v += eta2 * (xk + vu * vd(ROWD(T, L.cq + qo + k - 1)));
                    ROWD(T, ej + kb + k) = v;
                    nerr[j] = vmax(nerr[j], vabs(v));
                }
                const vd e3 = initialize ? x3 : eta2 * (v1 * qtx2 + x3);
                const vd e4 = initialize ? x4 : eta2 * (u0 * x1 + u1 * qtx2 - x4);
                ROWD(T, ej + kb + d) = e3;
                ROWD(T, ej + kb + d + 1) = e4;
                nerr[j] = vmax(nerr[j], vmax(vabs(e3), vabs(e4)));
            }
        }
    }
    team_max<NR>(tm, nerr);
}

// ------------------------------------------------------------------ solveKKT (src/eicos.cpp:1471-1620)
// sol = K^-1 rhs followed by up to nitref refinement rounds; every instance stops on its own
// criterion, the tile loops until all of its instances have stopped.
//   NR = 1: CTA = (tile, job) - the two solves of an iteration that share the factor (rhs1 -> sol1,
//           rhs2 -> sol2) run side by side as separate CTAs (few tiles: twice the parallelism);
//   NR = 2: one CTA runs both in ONE pass over L per sweep (two-job programs: every record is decoded
//           once for two right-hand sides; a job whose instances have all stopped rides along with its
//           accumulation masked off) - the form for a full machine.
template <int NR>
EI_DEV void tile_solve_kkt(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const vb act = lane_active(tm, t);
    if (!tm.any(act))
        return;
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    const bool init = a.initialize != 0;
    int sol[NR], xw[NR], dxr[NR], erow[NR], nitrow[NR];
    vd threshold[NR];
#pragma unroll
    for (int j = 0; j < NR; j++)
    {
        const KArgs::KktJob jb = a.job[NR == 1 ? tm.job : j];
        const int set = jb.set; // (jb.rhs is baked into the materialised load lists of the set)
        sol[j] = jb.sol;
        nitrow[j] = jb.nitrow;
        xw[j] = set ? L.xw2 : L.xw;
        dxr[j] = set ? L.dxr2 : L.dxr;
        erow[j] = set ? L.e2 : L.e;
        // max |rhs| is kept up to date by the kernels that write the right-hand sides (src/eicos.cpp:1590)
        threshold[j] = (1. + vd(ROWD(T, L.sc + (set ? S_RHSMAX2 : S_RHSMAX1)))) * a.settings.linsysacc;
    }
    const int set0 = a.job[NR == 1 ? tm.job : 0].set, v = a.variant;
    // programs and load lists of this launch: [first solve | refinement round]
    const DevMachine &pfw = NR == 1 ? P.fw[v] : P.fw2, &pbw = NR == 1 ? P.bw[v] : P.bw2;
    const DevMachine &pbwp = NR == 1 ? P.bwp[v] : P.bwp2, &pmv = NR == 1 ? P.mv[v] : P.mv2;
    const int *fw_ld[2], *bw_ld[2], *mv_ld;
    if (NR == 1)
    {
        fw_ld[0] = P.fw_ld[v][set0][0], fw_ld[1] = P.fw_ld[v][set0][1];
        bw_ld[0] = P.bw_ld[v][set0][0], bw_ld[1] = P.bw_ld[v][set0][1];
        mv_ld = P.mv_ld[v][set0];
    }
    else
    {
        fw_ld[0] = P.fw2_ld[0], fw_ld[1] = P.fw2_ld[1];
        bw_ld[0] = P.bw2_ld[0], bw_ld[1] = P.bw2_ld[1];
        mv_ld = P.mv2_ld;
    }
    Machine mm;
    mm.init(tm, tm.pbuf);

    long long ck[5] = {0, 0, 0, 0, 0}, c0 = EI_CLOCK(), c1;
#define EI_PHASE(k) (c1 = EI_CLOCK(), ck[k] += c1 - c0, c0 = c1)
    const auto sweeps = [&](int round, bool accumulate, const vb (&cont)[NR]) {
        MRun r;
        r.Tb = t.Tb;
        r.a_one = false;
        r.prog = pfw;
        r.ld = fw_ld[round];
        r.out = r.out2 = T + (size_t)xw[0] * TILE;
        r.outB = r.out2B = T + (size_t)xw[NR - 1] * TILE;
        NoFin nofin;
        mm.run<0, NR>(tm, r, nofin);
        EI_PHASE(1);
        if (accumulate)
        {
            AccFin<NR> fin;
#pragma unroll
            for (int j = 0; j < NR; j++)
            {
                fin.cont[j] = cont[j];
                fin.x[j] = T + (size_t)sol[j] * TILE;
            }
            r.prog = pbw;
            r.ld = bw_ld[1];
            r.out = r.out2 = T + (size_t)dxr[0] * TILE;
            r.outB = r.out2B = T + (size_t)dxr[NR - 1] * TILE;
            mm.run<MC_POS | MC_FIN | MC_X3, NR>(tm, r, fin);
        }
        else
        {
            r.prog = pbwp;
            r.ld = bw_ld[0];
            r.out = r.out2 = T + (size_t)sol[0] * TILE;
            r.outB = r.out2B = T + (size_t)sol[NR - 1] * TILE;
            mm.run<MC_POS, NR>(tm, r, nofin);
        }
        EI_PHASE(2);
    };
    vb nocont[NR];
#pragma unroll
    for (int j = 0; j < NR; j++)
        nocont[j] = vbset(false);
    if (tm.wk == 0)
        sweeps(0, false, nocont);
    tm.sync();

    vd nerr_prev[NR];
    int kref[NR][VEC];
    vb done[NR];
#pragma unroll
    for (int j = 0; j < NR; j++)
    {
        nerr_prev[j] = vset(DBL_MAX);
        done[j] = !act;
        VFOR kref[j][c_] = 0;
    }
    unsigned rounds = 0;
    for (;;)
    {
        vd nerr[NR];
        kkt_residual<NR>(tm, a, mm, t, pmv, mv_ld, sol, erow, init, nerr, set0);
        EI_PHASE(3);
        bool all_done = true;
#pragma unroll
        for (int j = 0; j < NR; j++)
        {
            vb rollback = vbset(false);
            VFOR
            {
                if (done[j].v[c_])
                    continue;
                if (kref[j][c_] > 0 && nerr[j].v[c_] > nerr_prev[j].v[c_])
                {
                    rollback.v[c_] = true;
                    kref[j][c_]--;
                    done[j].v[c_] = true;
                }
                else if (kref[j][c_] == a.settings.nitref || nerr[j].v[c_] < threshold[j].v[c_] ||
                         (kref[j][c_] > 0 && nerr_prev[j].v[c_] < a.settings.irerrfact * nerr[j].v[c_]))
                    done[j].v[c_] = true;
                else
                    nerr_prev[j].v[c_] = nerr[j].v[c_];
            }
            if (tm.any(rollback))
            { // x -= dx_ref for the instances whose last refinement made things worse
                for (int r = tm.wk; r < P.N; r += tm.nwk)
                    ROWD(T, sol[j] + r) -= vsel(rollback, ROWD(T, dxr[j] + r), vset(0.0));
            }
            all_done = all_done && tm.all(done[j]);
        }
        if (all_done)
            break;
        tm.sync(); // e complete before the forward sweep loads it
        EI_PHASE(4);
        if (tm.wk == 0)
        {
            vb cont[NR];
#pragma unroll
            for (int j = 0; j < NR; j++)
                cont[j] = !done[j];
            sweeps(1, true, cont);
        }
        tm.sync();
#pragma unroll
        for (int j = 0; j < NR; j++)
            VFOR if (!done[j].v[c_]) kref[j][c_]++;
        rounds++;
    }
    tm.sync();
    if (tm.wk == 0)
    {
#pragma unroll
        for (int j = 0; j < NR; j++)
            if (nitrow[j] >= 0)
                VFOR if (act.v[c_]) ROWC(t.I, nitrow[j], c_) = kref[j][c_];
#ifndef EICOS_EMU
        if (a.ir_rounds)
        {
            // [0] tile-rounds (sweep pairs x jobs), [6] lane-rounds: sweep pairs each instance needed
            int lane_rounds = 0;
#pragma unroll
            for (int j = 0; j < NR; j++)
                VFOR if (act.v[c_]) lane_rounds += kref[j][c_] + 1;
            for (int o = 16; o > 0; o >>= 1)
                lane_rounds += __shfl_xor_sync(0xffffffffu, lane_rounds, o);
            if (tm.pl == 0)
            {
                atomicAdd(a.ir_rounds, (unsigned long long)(rounds + 1) * NR);
                atomicAdd(a.ir_rounds + 6, (unsigned long long)lane_rounds);
                EI_PHASE(4);
                for (int k = 0; k < 5; k++)
                    atomicAdd(a.ir_rounds + 1 + k, (unsigned long long)ck[k]);
            }
        }
#endif
    }
#undef EI_PHASE
}

// ------------------------------------------------------------------ start of a solve (src/eicos.cpp:855-894)
EI_DEV void tile_init(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    const int n = P.n, zb = P.n + P.p;
    if (tm.wk == 0)
    {
        VFOR
        {
            const bool valid = tile * TILE + tm.lane + c_ < a.batch;
            ROWC(t.I, J_STATUS, c_) = valid ? (int)ST_ACTIVE : (int)EXIT_FATAL;
            ROWC(t.I, J_INST, c_) = valid ? a.first + tile * TILE + tm.lane + c_ : -1;
            ROWC(t.I, J_STORED, c_) = 0;
            if (!a.keep_sticky)
            {
                ROWC(t.I, J_HAS_PINFRES, c_) = 0;
                ROWC(t.I, J_HAS_DINFRES, c_) = 0;
                ROWC(t.I, J_HAS_RELGAP, c_) = 0;
                ROWC(T, L.sc + S_PINFRES, c_) = 0.0;
                ROWC(T, L.sc + S_DINFRES, c_) = 0.0;
                ROWC(T, L.sc + S_RELGAP, c_) = 0.0;
            }
        }
    }
    for (int k = tm.wk; k < P.nnzV; k += tm.nwk)
    { // resetKKTScalings :807-846
        const int kind = EI_LDG(P.Vkind + k);
        ROWD(T, L.V + k) = kind == 0 ? -1.0 : (kind == 1 ? 0.0 : 1.0);
    }
    // the LP scalings as the refinement residual reads them: MINUS w^2 (the mat-vec program then needs neither a sign
    // flag nor a special case for the identity scalings of the initial solves, src/eicos.cpp:1557-1559)
    for (int k = tm.wk; k < P.l; k += tm.nwk)
        ROWD(T, L.lpv + k) = -1.0;
    // rhs1 = [0; b; h], rhs2 = [-c; 0; 0]; resx0.. = max(1, ||c||), ... (:865-894)
    vd nr[3] = {vset(0.0), vset(0.0), vset(0.0)};
    vd mx[2] = {vset(0.0), vset(0.0)}; // max |rhs1|, max |rhs2| (solveKKT's stopping threshold, src/eicos.cpp:1590)
    for (int r = tm.wk; r < n; r += tm.nwk)
    {
        const vd v = ROWD(T, L.chb + r);
        ROWD(T, L.rhs1 + r) = 0.0;
        ROWD(T, L.rhs2 + r) = -v;
        nr[0] += v * v;
        mx[1] = vmax(mx[1], vabs(v));
    }
    for (int r = n + tm.wk; r < zb; r += tm.nwk)
    {
        const vd v = ROWD(T, L.chb + r);
        ROWD(T, L.rhs1 + r) = v;
        ROWD(T, L.rhs2 + r) = 0.0;
        nr[1] += v * v;
        mx[0] = vmax(mx[0], vabs(v));
    }
    for (int r = zb + tm.wk; r < P.N; r += tm.nwk)
    {
        const vd v = ROWD(T, L.chb + r);
        ROWD(T, L.rhs1 + r) = v;
        ROWD(T, L.rhs2 + r) = 0.0;
        nr[2] += v * v;
        mx[0] = vmax(mx[0], vabs(v));
    }
    team_sum<3>(tm, nr);
    team_max<2>(tm, mx);
    if (tm.wk == 0)
    {
        ROWD(T, L.sc + S_RESX0) = vmax(vset(1.), vsqrt(nr[0]));
        ROWD(T, L.sc + S_RESY0) = vmax(vset(1.), vsqrt(nr[1]));
        ROWD(T, L.sc + S_RESZ0) = vmax(vset(1.), vsqrt(nr[2]));
        ROWD(T, L.sc + S_RHSMAX1) = mx[0];
        ROWD(T, L.sc + S_RHSMAX2) = mx[1];
    }
}

// bringToCone (src/eicos.cpp:761-805): dst = sign*src + (1+alpha) e ; src, dst z-shaped row offsets
EI_DEV void bring_to_cone(const Team &tm, const KArgs &a, double *T, int src, double sign, int dst, vb write)
{
    const DevPattern &P = a.P;
    vd al[1] = {vset(-a.settings.gamma)};
    for (int k = tm.wk; k < P.l; k += tm.nwk)
    {
        const vd r = sign * vd(ROWD(T, src + k));
        VFOR if (r.v[c_] <= 0 && -r.v[c_] > al[0].v[c_]) al[0].v[c_] = -r.v[c_];
    }
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    {
        const int d = EI_LDG(P.cone_dim + c), kb = EI_LDG(P.cone_k + c);
        vd sq = vset(0.0);
        for (int k = 1; k < d; k++)
        {
            const vd v = sign * vd(ROWD(T, src + kb + k));
            sq += v * v;
        }
        const vd cres = sign * vd(ROWD(T, src + kb)) - vsqrt(sq);
        VFOR if (cres.v[c_] <= 0 && -cres.v[c_] > al[0].v[c_]) al[0].v[c_] = -cres.v[c_];
    }
    team_max<1>(tm, al);
    const vd alpha = al[0] + 1.;
    for (int k = tm.wk; k < P.l; k += tm.nwk)
        ROWD(T, dst + k) = vsel(write, sign * vd(ROWD(T, src + k)) + alpha, ROWD(T, dst + k));
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    {
        const int d = EI_LDG(P.cone_dim + c), kb = EI_LDG(P.cone_k + c);
        ROWD(T, dst + kb) = vsel(write, sign * vd(ROWD(T, src + kb)) + alpha, ROWD(T, dst + kb));
        for (int k = 1; k < d; k++)
            ROWD(T, dst + kb + k) = vsel(write, sign * vd(ROWD(T, src + kb + k)), ROWD(T, dst + kb + k));
    }
}

// initial point (src/eicos.cpp:933-992), after the two initial KKT solves
EI_DEV void tile_init_point(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const vb act = lane_active(tm, t);
    if (!tm.any(act))
        return;
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    const int n = P.n, zb = P.n + P.p;
    for (int j = tm.wk; j < n; j += tm.nwk)
    {
        ROWD(T, L.w + j) = vsel(act, ROWD(T, L.sol1 + j), ROWD(T, L.w + j));
        ROWD(T, L.rhs1 + j) = -vd(ROWD(T, L.chb + j));
    }
    for (int i = tm.wk; i < P.p; i += tm.nwk)
        ROWD(T, L.w + n + i) = vsel(act, ROWD(T, L.sol2 + n + i), ROWD(T, L.w + n + i));
    bring_to_cone(tm, a, T, L.sol1 + zb, -1.0, L.s, act);
    bring_to_cone(tm, a, T, L.sol2 + zb, 1.0, L.w + zb, act);
    if (tm.wk == 0)
        VFOR if (act.v[c_])
        {
            ROWC(T, L.sc + S_KAP, c_) = 1.;
            ROWC(T, L.sc + S_TAU, c_) = 1.;
            ROWC(T, L.sc + S_STEP, c_) = 0.;
            ROWC(T, L.sc + S_STEP_AFF, c_) = 0.;
            ROWC(T, L.sc + S_PRES_PREV, c_) = DBL_MAX;
            // rhs1 = [-c; b; h] from here on (S_RHSMAX2 still holds max |c| from eicos_init)
            ROWC(T, L.sc + S_RHSMAX1, c_) = dmax(ROWC(T, L.sc + S_RHSMAX1, c_), ROWC(T, L.sc + S_RHSMAX2, c_));
            ROWC(t.I, J_PINF, c_) = 0;
            ROWC(t.I, J_DINF, c_) = 0;
            ROWC(t.I, J_ITER, c_) = 0;
        }
}

// ------------------------------------------------------------------ per-instance scalar state of `Work` + `Information`
struct WState
{
    double d[S_WORK_END];
    int i[J_WORK_END];
};

EI_DEV void ws_load(const Team &tm, const double *T, const int *I, int sc, int soff, int ioff, int c, WState &w)
{
    for (int k = 0; k < S_WORK_END; k++)
        w.d[k] = ROWC(T, sc + soff + k, c);
    for (int k = 0; k < J_WORK_END; k++)
        w.i[k] = ROWC(I, ioff + k, c);
}
EI_DEV void ws_store(const Team &tm, double *T, int *I, int sc, int soff, int ioff, int c, const WState &w)
{
    for (int k = 0; k < S_WORK_END; k++)
        ROWC(T, sc + soff + k, c) = w.d[k];
    for (int k = 0; k < J_WORK_END; k++)
        ROWC(I, ioff + k, c) = w.i[k];
}

// Information::isBetterThan (src/eicos.cpp:23-68)
EI_DEV bool ws_better(const WState &a, const WState &o)
{
    const bool gapmu = (a.d[S_GAP] > 0. && o.d[S_GAP] > 0. && a.d[S_GAP] < o.d[S_GAP]) &&
                       (a.d[S_MU] > 0. && a.d[S_MU] < o.d[S_MU]);
    if (a.i[J_HAS_PINFRES] && a.d[S_KAPOVERT] > 1.)
    {
        if (o.i[J_HAS_PINFRES])
            return gapmu && (a.d[S_PINFRES] > 0. && a.d[S_PINFRES] < o.d[S_PRES]);
        return gapmu;
    }
    return gapmu && (a.d[S_PRES] > 0. && a.d[S_PRES] < o.d[S_PRES]) &&
           (a.d[S_DRES] > 0. && a.d[S_DRES] < o.d[S_DRES]) &&
           (a.d[S_KAPOVERT] > 0. && a.d[S_KAPOVERT] < o.d[S_KAPOVERT]);
}

// checkExitConditions (src/eicos.cpp:526-641).  An empty std::optional compares "less than"
// any double there, which is what the (!has || v < tol) terms reproduce.
EI_DEV int ws_check_exit(const KSettings &st, WState &w, bool reduced)
{
    const double feastol = reduced ? st.feastol_inacc : st.feastol;
    const double abstol = reduced ? st.abstol_inacc : st.abstol;
    const double reltol = reduced ? st.reltol_inacc : st.reltol;
    const double tau = w.d[S_TAU], kap = w.d[S_KAP];
    if ((-w.d[S_CX] > 0. || -w.d[S_BY] - w.d[S_HZ] >= -abstol) &&
        (w.d[S_PRES] < feastol && w.d[S_DRES] < feastol) &&
        (w.d[S_GAP] < abstol || !w.i[J_HAS_RELGAP] || w.d[S_RELGAP] < reltol))
    {
        w.i[J_PINF] = 0;
        w.i[J_DINF] = 0;
        return reduced ? EXIT_OPTIMAL + EXIT_INACC : EXIT_OPTIMAL;
    }
    else if (w.i[J_HAS_DINFRES] && w.d[S_DINFRES] < feastol && tau < kap)
    {
        w.i[J_PINF] = 0;
        w.i[J_DINF] = 1;
        return reduced ? EXIT_DINF + EXIT_INACC : EXIT_DINF;
    }
    else if ((w.i[J_HAS_PINFRES] && w.d[S_PINFRES] < feastol && tau < kap) ||
             (tau < feastol && kap < feastol && (!w.i[J_HAS_PINFRES] || w.d[S_PINFRES] < feastol)))
    {
        w.i[J_PINF] = 1;
        w.i[J_DINF] = 0;
        return reduced ? EXIT_PINF + EXIT_INACC : EXIT_PINF;
    }
    return EXIT_NOT_CONVERGED;
}

// ------------------------------------------------------------------ NT scaling of one cone, one instance (src/eicos.cpp:419-474)
struct ConeScaling
{
    int stage; // 0 ok, 1 failed the residual test (nothing assigned), 2 failed c^2/u0^2 - d (eta, q assigned)
    double eta, eta2, a, d1, u0, u1, v1, w, snorm, znorm, gamma;
};

EI_DEV ConeScaling cone_scaling(const Team &tm, const double *T, int srow, int zrow, int d, int c)
{
    ConeScaling r;
    const double s0 = ROWC(T, srow, c), z0 = ROWC(T, zrow, c);
    double ss = 0.0, zz = 0.0;
    for (int k = 1; k < d; k++)
    {
        const double sv = ROWC(T, srow + k, c), zv = ROWC(T, zrow + k, c);
        ss += sv * sv;
        zz += zv * zv;
    }
    const double sres = s0 * s0 - ss, zres = z0 * z0 - zz;
    r.stage = 0;
    if (sres <= 0 || zres <= 0)
    {
        r.stage = 1;
        return r;
    }
    r.snorm = sqrt(sres);
    r.znorm = sqrt(zres);
    r.eta2 = r.snorm / r.znorm;
    r.eta = sqrt(r.eta2);
    double g = 0.0;
    for (int k = 0; k < d; k++)
        g += (ROWC(T, srow + k, c) / r.snorm) * (ROWC(T, zrow + k, c) / r.znorm);
    g = sqrt(0.5 * (1. + g));
    r.gamma = g;
    const double av = (0.5 / g) * (s0 / r.snorm + z0 / r.znorm);
    double w = 0.0;
    for (int k = 1; k < d; k++)
    {
        const double qk = (0.5 / g) * (ROWC(T, srow + k, c) / r.snorm - ROWC(T, zrow + k, c) / r.znorm);
        w += qk * qk;
    }
    const double cc = (1. + av) + w / (1. + av);
    const double dd = 1. + 2. / (1. + av) + w / ((1. + av) * (1. + av));
    const double d1 = dmax(0., 0.5 * (av * av + w * (1. - (cc * cc) / (1. + w * dd))));
    const double u0sq = av * av + w - d1;
    const double c2byu02 = (cc * cc) / u0sq;
    if (c2byu02 - dd <= 0)
    {
        r.stage = 2;
        return r;
    }
    r.d1 = d1;
    r.u0 = sqrt(u0sq);
    r.u1 = sqrt(c2byu02);
    r.v1 = sqrt(c2byu02 - dd);
    r.a = av;
    r.w = w;
    return r;
}

// ------------------------------------------------------------------ computeResiduals (src/eicos.cpp:643-689)
// rx = -A'y - G'z, ry = A x, rz = s + G x (each before and after the tau terms) and the sums the
// statistics need; one warp per tile runs the machine program of streams.cpp: build_resid, whose
// finish functor keeps the fourteen sums; results in `r` and the S_RED rows.
enum { RS_HX2, RS_RX2, RS_CX, RS_NX2, RS_HY2, RS_RY2, RS_BY, RS_NY2, RS_HZ2, RS_RZ2, RS_HZ, RS_NZ2, RS_NS2, RS_GAP, RS_NRED };
struct ResidFin
{
    vd r[RS_NRED];
    EI_DEV void operator()(int kind, int, const vd (&resv)[1], const vd (&bv)[1], const vd (&ownv)[1])
    {
        const vd res = resv[0], b = bv[0], own = ownv[0];
        // PRE: res = the row before its tau term; FIN: res = the finished row, b = c_j / b_i / h_i, f3 -> x_j / y_i / z_i;
        // FIRST_Z: res = s_i, f3 -> z_i
        if (kind == RS_PRE_X)
            r[RS_HX2] += res * res;
        else if (kind == RS_PRE_Y)
            r[RS_HY2] += res * res;
        else if (kind == RS_PRE_Z)
            r[RS_HZ2] += res * res;
        else
        {
            if (kind == RS_FIN_X)
            {
                r[RS_RX2] += res * res;
                r[RS_CX] += b * own;
                r[RS_NX2] += own * own;
            }
            else if (kind == RS_FIN_Y)
            {
                r[RS_RY2] += res * res;
                r[RS_BY] += b * own;
                r[RS_NY2] += own * own;
            }
            else if (kind == RS_FIN_Z)
            {
                r[RS_RZ2] += res * res;
                r[RS_HZ] += b * own;
                r[RS_NZ2] += own * own;
            }
            else
            { // RS_FIRST_Z, RS_FIRST_PRE_Z
                r[RS_NS2] += res * res;
                r[RS_GAP] += res * own;
                if (kind == RS_FIRST_PRE_Z)
                    r[RS_HZ2] += res * res;
            }
        }
    }
};

EI_DEV void tile_resid(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const vb act = lane_active(tm, t);
    if (!tm.any(act))
        return;
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    // The program exists in M_MV_PARTS independent parts (streams.cpp).  A wide launch (one warp per part, each with a
    // machine of its own) runs them side by side, a one-warp launch one after the other; the fourteen sums are the
    // parts' sums added in part order either way, so both launches give the same bits.
    const bool wide = tm.nwk >= M_MV_PARTS;
    vd tot[RS_NRED];
    for (int k = 0; k < RS_NRED; k++)
        tot[k] = vset(0.0);
    const auto run_part = [&](int part, double *mem) {
        ResidFin fin;
        for (int k = 0; k < RS_NRED; k++)
            fin.r[k] = vset(0.0);
        Machine mm;
        mm.init(tm, mem);
        MRun r;
        r.prog = P.rs[part];
        r.ld = P.rs_ld[part];
        r.Tb = t.Tb;
        r.out = r.out2 = r.outB = r.out2B = T + (size_t)L.r * TILE;
        r.a_one = false;
        mm.run<MC_CONST | MC_POS | MC_BKEEP | MC_FIN | MC_X3, 1>(tm, r, fin);
        for (int k = 0; k < RS_NRED; k++)
            tot[k] = part == 0 || wide ? fin.r[k] : tot[k] + fin.r[k];
    };
    if (P.mv_rows > 0)
    {
        if (wide)
        {
            if (tm.wk < M_MV_PARTS)
                run_part(tm.wk, tm.pbuf + (size_t)tm.wk * a.part_doubles);
            team_sum<RS_NRED>(tm, tot); // worker order = part order
        }
        else if (tm.wk == 0)
            for (int part = 0; part < M_MV_PARTS; part++)
                run_part(part, tm.pbuf);
    }
    if (tm.wk == 0)
        for (int k = 0; k < RS_NRED; k++)
            ROWD(T, L.sc + S_RED + k) = tot[k];
}

// lambda = W z of the LP rows.  Without second-order cones it is never stored: its readers take z and recompute
// lpw * z, rounded alone like the head's product.  With cones the head's cone_scale() writes the rows, and keeps
// their old values for an instance whose cone scaling failed, so they are read.
EI_DEV int lp_lambda_row(const DevPattern &P, const Layout &L) { return P.nc == 0 ? L.w + P.n + P.p : L.lam; }
EI_DEV vd lp_lambda(const DevPattern &P, vd lpw, vd row) { return P.nc == 0 ? vmul_rn(lpw, row) : row; }

// ------------------------------------------------------------------ head of an iteration
// computeResiduals + updateStatistics + safeguards / exit tests + best-iterate bookkeeping
// (src/eicos.cpp:997-1158), then for the instances that keep iterating: updateScalings,
// updateKKTScalings and RHSaffine (:1160-1162, :1176).  Instances that stop are back-scaled in place.
EI_DEV void tile_head(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const vb act = lane_active(tm, t);
    if (!tm.any(act))
        return;
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    int *I = t.I;
    const int n = P.n, p = P.p, zb = P.n + P.p;
    const vd tau = ROWD(T, L.sc + S_TAU), kap = ROWD(T, L.sc + S_KAP);
    enum { HX2, RX2, CX, NX2, HY2, RY2, BY, NY2, HZ2, RZ2, HZ, NZ2, NS2, GAP, NRED };
    static_assert(NRED == 14, "S_RED holds 14 rows");
    vd r[NRED];
    for (int k = 0; k < NRED; k++)
        r[k] = ROWD(T, L.sc + S_RED + k);

    // ---- per instance: updateStatistics (:691-728), safeguards, exit tests, best iterate (:1010-1158).
    //      Every warp computes the same values; warp 0 writes them back.
    vb restore = vbset(false), save = vbset(false), fin = vbset(false), cont = vbset(false);
    vd ftau = tau;
    WState wsv[VEC], bsv[VEC];
    double rtv[VEC], ppv[VEC];
    int codev[VEC];
    VFOR
    {
        const int c = c_;
        WState &w = wsv[c], &best = bsv[c];
        ws_load(tm, T, I, L.sc, 0, 0, c, w);
        ws_load(tm, T, I, L.sc, S_BEST, J_BEST, c, best);
        const double tau_c = tau.v[c], kap_c = kap.v[c];
        const double hresx = sqrt(r[HX2].v[c]), hresy = sqrt(r[HY2].v[c]), hresz = sqrt(r[HZ2].v[c]);
        const double nx = sqrt(r[NX2].v[c]), ny = sqrt(r[NY2].v[c]), nz = sqrt(r[NZ2].v[c]), ns = sqrt(r[NS2].v[c]);
        const double cx = r[CX].v[c], by = p > 0 ? r[BY].v[c] : 0., hz = r[HZ].v[c];
        const double rt = kap_c + cx + by + hz;
        w.d[S_CX] = cx;
        w.d[S_BY] = by;
        w.d[S_HZ] = hz;
        w.d[S_GAP] = r[GAP].v[c];
        w.d[S_MU] = (r[GAP].v[c] + kap_c * tau_c) / ((P.l + P.nc) + 1);
        w.d[S_KAPOVERT] = kap_c / tau_c;
        w.d[S_PCOST] = cx / tau_c;
        w.d[S_DCOST] = -(hz + by) / tau_c;
        if (w.d[S_PCOST] < 0.)
        {
            w.i[J_HAS_RELGAP] = 1;
            w.d[S_RELGAP] = w.d[S_GAP] / (-w.d[S_PCOST]);
        }
        else if (w.d[S_DCOST] > 0.)
        {
            w.i[J_HAS_RELGAP] = 1;
            w.d[S_RELGAP] = w.d[S_GAP] / w.d[S_DCOST];
        }
        else
            w.i[J_HAS_RELGAP] = 0;
        const double resx0 = ROWC(T, L.sc + S_RESX0, c), resy0 = ROWC(T, L.sc + S_RESY0, c), resz0 = ROWC(T, L.sc + S_RESZ0, c);
        const double nry = p > 0 ? sqrt(r[RY2].v[c]) / dmax(resy0 + nx, 1.) : 0.;
        const double nrz = sqrt(r[RZ2].v[c]) / dmax(resz0 + nx + ns, 1.);
        w.d[S_PRES] = dmax(nry, nrz) / tau_c;
        w.d[S_DRES] = sqrt(r[RX2].v[c]) / dmax(resx0 + ny + nz, 1.) / tau_c;
        if ((hz + by) / dmax(ny + nz, 1.) < -a.settings.reltol)
        {
            w.i[J_HAS_PINFRES] = 1;
            w.d[S_PINFRES] = hresx / dmax(ny + nz, 1.);
        }
        if (cx / dmax(nx, 1.) < -a.settings.reltol)
        {
            w.i[J_HAS_DINFRES] = 1;
            w.d[S_DINFRES] = dmax(hresy / dmax(nx, 1.), hresz / dmax(nx + ns, 1.));
        }

        const int iter = w.i[J_ITER];
        double pres_prev = ROWC(T, L.sc + S_PRES_PREV, c);
        int code = ST_ACTIVE;
        bool rst = false, sav = false;
        if (act.v[c])
        {
            if (iter > 0 && (w.d[S_PRES] > a.settings.safeguard * pres_prev || w.d[S_GAP] < 0.))
            {
                rst = true;
                w = best;
                code = ws_check_exit(a.settings, w, true);
                if (code == EXIT_NOT_CONVERGED)
                    code = EXIT_NUMERICS;
            }
            else
            {
                pres_prev = w.d[S_PRES];
                code = ws_check_exit(a.settings, w, false);
                if (code == EXIT_NOT_CONVERGED)
                {
                    if (iter > 0 && w.d[S_STEP] == a.settings.stepmin * a.settings.gamma)
                    {
                        rst = true;
                        w = best;
                        code = ws_check_exit(a.settings, w, true);
                        if (code == EXIT_NOT_CONVERGED)
                            code = EXIT_NUMERICS;
                    }
                    else if (iter == a.settings.iter_max)
                    {
                        if (!ws_better(w, best))
                        {
                            rst = true;
                            w = best;
                        }
                        code = ws_check_exit(a.settings, w, true);
                        if (code == EXIT_NOT_CONVERGED)
                            code = EXIT_MAXIT;
                    }
                    else if (ei_isnan(w.d[S_PCOST]))
                    {
                        if (!(iter == 0 || ws_better(w, best)))
                        {
                            rst = true;
                            w = best;
                            code = ws_check_exit(a.settings, w, true);
                            if (code == EXIT_NOT_CONVERGED)
                                code = EXIT_NUMERICS;
                        } // else: the reference leaves not_converged_yet (-87) in place (:1117-1121)
                    }
                    else
                        code = ST_ACTIVE;
                }
            }
            if (code == ST_ACTIVE && (iter == 0 || ws_better(w, best)))
            {
                sav = true;
                best = w;
            }
        }
        restore.v[c] = rst;
        save.v[c] = sav;
        fin.v[c] = act.v[c] && code != ST_ACTIVE;
        cont.v[c] = act.v[c] && code == ST_ACTIVE;
        ftau.v[c] = w.d[S_TAU];
        rtv[c] = rt;
        ppv[c] = pres_prev;
        codev[c] = code;
    }
    tm.sync(); // every warp has read the old state rows before warp 0 overwrites them
    if (tm.wk == 0)
        VFOR if (act.v[c_])
        {
            ws_store(tm, T, I, L.sc, 0, 0, c_, wsv[c_]);
            if (save.v[c_])
                ws_store(tm, T, I, L.sc, S_BEST, J_BEST, c_, bsv[c_]);
            ROWC(T, L.sc + S_RT, c_) = rtv[c_];
            ROWC(T, L.sc + S_PRES_PREV, c_) = ppv[c_];
            ROWC(I, J_STATUS, c_) = codev[c_];
        }

    // ---- vector part of `w = w_best` / `w_best = w`, and backscale (:1271-1277) for finished instances.
    //      lambda is not part of the best iterate here: an instance that restores it always stops, and the lambda
    //      of a stopped instance is read by nothing.
    if (!tm.any(restore || fin) && tm.all(save || !act))
    { // common case: every active instance improves its best iterate and nobody stops -> plain copies
        // (inactive lanes of w_best are never read again)
        const int ins[1] = {L.w};
        ew_rows<1, 8>(tm, T, P.N, ins, [&](int q, const vd *x) { ROWD(T, L.wb + q) = x[0]; });
        const int inz[1] = {L.s};
        ew_rows<1, 8>(tm, T, P.mt, inz, [&](int e, const vd *x) { ROWD(T, L.bs + e) = x[0]; });
    }
    else if (tm.any(restore || save || fin))
    {
        const bool any_fin = tm.any(fin);
        {
            const int ins[2] = {L.w, L.wb};
            ew_rows<2, 6>(tm, T, P.N, ins, [&](int q, const vd *x) {
                vd v = vsel(restore, x[1], x[0]);
                ROWD(T, L.wb + q) = vsel(save, v, x[1]);
                if (any_fin && P.pim)
                    v = vsel(fin, v / (vd(ROWD(T, L.eq + q)) * ftau), v);
                else if (any_fin)
                {
                    const double eq = q < n ? EI_LDG(P.xeq + q) : (q < zb ? EI_LDG(P.Aeq + q - n) : EI_LDG(P.GeqE + q - zb));
                    v = vsel(fin, v / (eq * ftau), v);
                }
                ROWD(T, L.w + q) = v;
            });
        }
        {
            const int ins[2] = {L.s, L.bs};
            ew_rows<2, 6>(tm, T, P.mt, ins, [&](int e, const vd *x) {
                vd sv = vsel(restore, x[1], x[0]);
                ROWD(T, L.bs + e) = vsel(save, sv, x[1]);
                if (any_fin && P.pim)
                    sv = vsel(fin, sv * (vd(ROWD(T, L.eq + zb + e)) / ftau), sv);
                else if (any_fin)
                    sv = vsel(fin, sv * (EI_LDG(P.GeqE + e) / ftau), sv);
                ROWD(T, L.s + e) = sv;
            });
        }
    }
    if (!tm.any(cont))
        return;
    tm.sync(); // restored / back-scaled rows are in place
#ifndef EICOS_EMU
    if (tm.wk == 0 && a.active_count)
    {
        int mine = 0;
        VFOR mine += cont.v[c_] ? 1 : 0;
        for (int o = 16; o > 0; o >>= 1)
            mine += __shfl_xor_sync(0xffffffffu, mine, o);
        if (tm.pl == 0)
            atomicAdd(a.active_count, (unsigned)mine);
    }
#else
    if (tm.wk == 0 && a.active_count)
        VFOR if (cont.v[c_]) *a.active_count += 1;
#endif

    // ---- updateScalings (:411-479); its return value is ignored by the caller (:1160), so after a
    // failure at cone c the LP part and cones < c are new, cone c is partly new and lambda is stale.
    const int sz = L.w + zb; // z rows of the iterate
    const bool lp_only = P.nc == 0; // then scale()'s lambda = W z is not stored (lp_lambda)
    if (lp_only && tm.all(cont))
    {
        const int ins[2] = {L.s, sz};
        ew_rows<2, 6>(tm, T, P.l, ins, [&](int k, const vd *x) {
            const vd v = x[0] / x[1];
            ROWD(T, L.lpv + k) = -v;
            ROWD(T, L.lpw + k) = vsqrt(v);
            ROWD(T, L.V + k) = -v - Settings::deltastat; // updateKKTScalings, LP part (:1696-1699)
        });
    }
    else
    {
        const int ins[4] = {L.s, sz, L.lpv, L.lpw};
        ew_rows<4, 3>(tm, T, P.l, ins, [&](int k, const vd *x) {
            const vd v = x[0] / x[1];
            const vd nvn = vsel(cont, -v, x[2]); // (lpv holds -w^2)
            ROWD(T, L.lpv + k) = nvn;
            ROWD(T, L.lpw + k) = vsel(cont, vsqrt(v), x[3]);
            ROWD(T, L.V + k) = nvn - Settings::deltastat; // updateKKTScalings, LP part (:1696-1699)
        });
    }
    vb nofail = vbset(true);
    if (P.nc > 0)
    {
        vd ff[1] = {vset((double)P.nc)};
        for (int c = tm.wk; c < P.nc; c += tm.nwk)
        {
            const int ks = EI_LDG(P.cone_k + c), d = EI_LDG(P.cone_dim + c);
            VFOR
            {
                const ConeScaling cs = cone_scaling(tm, T, L.s + ks, sz + ks, d, c_);
                if (cs.stage != 0)
                    ff[0].v[c_] = dmin(ff[0].v[c_], (double)c);
            }
        }
        team_min<1>(tm, ff);
        VFOR nofail.v[c_] = (int)ff[0].v[c_] == P.nc;
        for (int c = tm.wk; c < P.nc; c += tm.nwk)
        {
            const int d = EI_LDG(P.cone_dim + c), ks = EI_LDG(P.cone_k + c), qo = EI_LDG(P.cone_q + c);
            const int cp = L.cpar + c * CP_COUNT;
            VFOR
            {
                if (!cont.v[c_] || c > (int)ff[0].v[c_])
                    continue;
                const ConeScaling cs = cone_scaling(tm, T, L.s + ks, sz + ks, d, c_);
                if (cs.stage == 1)
                    continue;
                ROWC(T, cp + CP_ETA2, c_) = cs.eta2;
                ROWC(T, cp + CP_ETA, c_) = cs.eta;
                for (int k = 1; k < d; k++)
                    ROWC(T, L.cq + qo + k - 1, c_) = (0.5 / cs.gamma) * (ROWC(T, L.s + ks + k, c_) / cs.snorm - ROWC(T, sz + ks + k, c_) / cs.znorm);
                if (cs.stage == 2)
                    continue;
                ROWC(T, cp + CP_D1, c_) = cs.d1;
                ROWC(T, cp + CP_U0, c_) = cs.u0;
                ROWC(T, cp + CP_U1, c_) = cs.u1;
                ROWC(T, cp + CP_V1, c_) = cs.v1;
                ROWC(T, cp + CP_A, c_) = cs.a;
                ROWC(T, cp + CP_W, c_) = cs.w;
            }
        }
    }
    tm.sync(); // scalings complete (rows are distributed differently in the passes below)
    if (!lp_only)
        cone_scale(tm, a, T, sz, L.lam, cont && nofail);

    // ---- updateKKTScalings (:1691-1732) into the V rows, RHSaffine (:1670-1689) into rhs2
    const double delta = Settings::deltastat;
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    {
        const int d = EI_LDG(P.cone_dim + c), ks = EI_LDG(P.cone_k + c), qo = EI_LDG(P.cone_q + c);
        const int cp = L.cpar + c * CP_COUNT;
        const vd eta2 = ROWD(T, cp + CP_ETA2), d1 = ROWD(T, cp + CP_D1), u0 = ROWD(T, cp + CP_U0);
        const vd u1 = ROWD(T, cp + CP_U1), v1 = ROWD(T, cp + CP_V1);
        // cones before c contributed sum(3 dim + 1) V entries; ks - 2c - l = sum of their dims
        int vb_ = L.V + P.l + 3 * (ks - 2 * c - P.l) + c;
        ROWD(T, vb_++) = -(eta2 * d1) - delta;
        for (int k = 1; k < d; k++)
            ROWD(T, vb_++) = -eta2 - delta;
        ROWD(T, vb_++) = -eta2;
        for (int k = 1; k < d; k++)
            ROWD(T, vb_++) = -(eta2 * v1) * vd(ROWD(T, L.cq + qo + k - 1));
        ROWD(T, vb_++) = eta2 + delta;
        ROWD(T, vb_++) = -(eta2 * u0);
        for (int k = 1; k < d; k++)
            ROWD(T, vb_++) = -(eta2 * u1) * vd(ROWD(T, L.cq + qo + k - 1));
    }
    {
        vd mx[1] = {vset(0.0)}; // max |rhs2| for the affine solve
        const int ins[1] = {L.r};
        ew_rows<1, 8>(tm, T, zb, ins, [&](int q, const vd *x) {
            ROWD(T, L.rhs2 + q) = q < n ? x[0] : -x[0];
            mx[0] = vmax(mx[0], vabs(x[0]));
        });
        const int inz[2] = {L.s, L.r + zb}; // s - rz; the slot rows of s and rz are zero
        ew_rows<2, 6>(tm, T, P.mt, inz, [&](int e, const vd *x) {
            const vd v = x[0] - x[1];
            ROWD(T, L.rhs2 + zb + e) = v;
            mx[0] = vmax(mx[0], vabs(v));
        });
        team_max<1>(tm, mx);
        if (tm.wk == 0)
            ROWD(T, L.sc + S_RHSMAX2) = vsel(cont, mx[0], ROWD(T, L.sc + S_RHSMAX2));
    }
}

// ------------------------------------------------------------------ affine step -> centering -> combined RHS
// (src/eicos.cpp:1181-1210 with RHScombined :1282-1325, conicProduct :1357, conicDivision :1330)
EI_DEV void tile_mid(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const vb act = lane_active(tm, t);
    if (!tm.any(act))
        return;
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    const int n = P.n, p = P.p, zb = P.n + P.p;
    const vd tau = ROWD(T, L.sc + S_TAU), kap = ROWD(T, L.sc + S_KAP), rt = ROWD(T, L.sc + S_RT);
    const vd mu = ROWD(T, L.sc + S_MU);

    // c'dx, b'dy, h'dz for both solutions; the slot rows of h are zero but are skipped anyway
    vd dt[6];
    for (int k = 0; k < 6; k++)
        dt[k] = vset(0.0);
    {
        const int ix[3] = {L.chb, L.sol1, L.sol2};
        ew_rows<3, 4>(tm, T, n, ix, [&](int, const vd *x) {
            dt[0] += x[0] * x[1];
            dt[3] += x[0] * x[2];
        });
        const int iy[3] = {L.chb + n, L.sol1 + n, L.sol2 + n};
        ew_rows<3, 4>(tm, T, p, iy, [&](int, const vd *x) {
            dt[1] += x[0] * x[1];
            dt[4] += x[0] * x[2];
        });
        const int iz[3] = {L.chb + zb, L.sol1 + zb, L.sol2 + zb};
        ew_rows<3, 4>(tm, T, P.l, iz, [&](int, const vd *x) {
            dt[2] += x[0] * x[1];
            dt[5] += x[0] * x[2];
        });
    }
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    {
        const int d = EI_LDG(P.cone_dim + c), kb = zb + EI_LDG(P.cone_k + c);
        for (int k = 0; k < d; k++)
        {
            const vd hv = ROWD(T, L.chb + kb + k);
            dt[2] += hv * vd(ROWD(T, L.sol1 + kb + k));
            dt[5] += hv * vd(ROWD(T, L.sol2 + kb + k));
        }
    }
    team_sum<6>(tm, dt);
    const vd dtau_denom = kap / tau - dt[0] - dt[1] - dt[2];
    const vd dtauaff = (rt - kap + dt[3] + dt[4] + dt[5]) / dtau_denom;
    // LP rows in one pass: dz = dz2 + dtauaff * dz1, W dz, ds = -(W dz) - lambda, min ratios of the line search.
    // Nothing is stored: RHScombined below recomputes the three rows, and the combined solve overwrites sol2.
    const int lrow = lp_lambda_row(P, L);
    vd m0 = vset(DBL_MAX), m1 = vset(DBL_MAX);
    {
        const int ins[4] = {L.sol2 + zb, L.sol1 + zb, L.lpw, lrow};
        ew_rows<4, 3>(tm, T, P.l, ins, [&](int, const vd *x) {
            const vd lk = lp_lambda(P, x[2], x[3]);
            const vd wd = vmul_rn(x[2], vfma(dtauaff, x[1], x[0]));
            const vd ds = -wd - lk;
            m0 = vmin(m0, ds / lk);
            m1 = vmin(m1, wd / lk);
        });
    }
    if (P.mt > P.l)
    { // cone rows: the same steps, pass by pass (slot rows are never read again)
        const int cz = zb + P.l, nr = P.mt - P.l;
        const int ins[2] = {L.sol2 + cz, L.sol1 + cz};
        ew_rows<2, 6>(tm, T, nr, ins, [&](int e, const vd *x) { ROWD(T, L.sol2 + cz + e) = x[0] + dtauaff * x[1]; });
        tm.sync();
        cone_scale(tm, a, T, L.sol2 + zb, L.wdz, vbset(true), false);
        tm.sync();
        const int in2[2] = {L.wdz + P.l, L.lam + P.l};
        ew_rows<2, 6>(tm, T, nr, in2, [&](int e, const vd *x) { ROWD(T, L.dsw + P.l + e) = -x[0] - x[1]; });
        tm.sync();
    }
    const vd dkapaff = -kap - kap / tau * dtauaff;
    const vd step_aff = line_search(tm, a, T, L.lam, L.dsw, L.wdz, tau, dtauaff, kap, dkapaff, false, m0, m1);
    vd sigma;
    VFOR
    {
        const double om = 1. - step_aff.v[c_];
        double sg = om * om * om; // std::pow(x, 3)
        if (sg < a.settings.sigmamin)
            sg = a.settings.sigmamin;
        else if (a.settings.sigmamax < sg)
            sg = a.settings.sigmamax;
        sigma.v[c_] = sg;
    }
    if (tm.wk == 0)
        VFOR if (act.v[c_])
        {
            ROWC(T, L.sc + S_DTAU_DENOM, c_) = dtau_denom.v[c_];
            ROWC(T, L.sc + S_DTAUAFF, c_) = dtauaff.v[c_];
            ROWC(T, L.sc + S_DKAPAFF, c_) = dkapaff.v[c_];
            ROWC(T, L.sc + S_STEP_AFF, c_) = step_aff.v[c_];
            ROWC(T, L.sc + S_SIGMA, c_) = sigma.v[c_];
        }

    // RHScombined
    const vd sigmamu = sigma * mu, oms = 1. - sigma;
    vd mx[1] = {vset(0.0)}; // max |rhs2| for the combined solve
    {
        const int ins[1] = {L.rhs2};
        ew_rows<1, 8>(tm, T, n + p, ins, [&](int r, const vd *x) {
            const vd v = x[0] * oms;
            ROWD(T, L.rhs2 + r) = v;
            mx[0] = vmax(mx[0], vabs(v));
        });
        const int inl[5] = {lrow, L.sol2 + zb, L.sol1 + zb, L.r + zb, L.lpw};
        ew_rows<5, 2>(tm, T, P.l, inl, [&](int k, const vd *x) {
            const vd lk = lp_lambda(P, x[4], x[0]);
            const vd wd = vmul_rn(x[4], vfma(dtauaff, x[2], x[1])); // the affine pass's W dz and ds
            const vd ds = -wd - lk;
            vd d1 = lk * lk;
            d1 += ds * wd;
            d1 -= sigmamu;
            const vd q = d1 / lk; // conicDivision, LP part
            ROWD(T, L.dsw + k) = q;
            const vd v = -oms * x[3] + x[4] * q;
            ROWD(T, L.rhs2 + zb + k) = v;
            mx[0] = vmax(mx[0], vabs(v));
        });
    }
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    {
        const int d = EI_LDG(P.cone_dim + c), zs = EI_LDG(P.cone_k + c), qo = EI_LDG(P.cone_q + c);
        const int kb = zb + zs;
        const int cp = L.cpar + c * CP_COUNT;
        const vd eta = ROWD(T, cp + CP_ETA), ca = ROWD(T, cp + CP_A);
        // ds1 = lambda o lambda ; ds2 = (W\ds_aff) o (W dz_aff)
        const vd l0 = ROWD(T, L.lam + zs), u0 = ROWD(T, L.dsw + zs), v0 = ROWD(T, L.wdz + zs);
        vd ll = vset(0.0), uv = vset(0.0);
        for (int k = 0; k < d; k++)
        {
            const vd lk = ROWD(T, L.lam + zs + k);
            ll += lk * lk;
            uv += vd(ROWD(T, L.dsw + zs + k)) * vd(ROWD(T, L.wdz + zs + k));
        }
        vd w0 = ll - sigmamu;
        w0 += uv;
        ROWD(T, L.ds1 + zs) = w0;
        for (int k = 1; k < d; k++)
        {
            const vd lk = ROWD(T, L.lam + zs + k);
            vd v = l0 * lk + l0 * lk;
            v += u0 * vd(ROWD(T, L.wdz + zs + k)) + v0 * vd(ROWD(T, L.dsw + zs + k));
            ROWD(T, L.ds1 + zs + k) = v;
        }
        // dsw = lambda \ ds1
        vd rho = vset(0.0), zeta = vset(0.0);
        for (int k = 1; k < d; k++)
        {
            const vd lk = ROWD(T, L.lam + zs + k);
            rho += lk * lk;
            zeta += lk * vd(ROWD(T, L.ds1 + zs + k));
        }
        rho = l0 * l0 - rho;
        const vd factor = (zeta / l0 - w0) / rho;
        const vd q0 = (l0 * w0 - zeta) / rho;
        ROWD(T, L.dsw + zs) = q0;
        for (int k = 1; k < d; k++)
            ROWD(T, L.dsw + zs + k) = factor * vd(ROWD(T, L.lam + zs + k)) + vd(ROWD(T, L.ds1 + zs + k)) / l0;
        // ds1 = W * dsw, then the cone rows of rhs2
        vd zt = vset(0.0);
        for (int k = 1; k < d; k++)
            zt += vd(ROWD(T, L.cq + qo + k - 1)) * vd(ROWD(T, L.dsw + zs + k));
        const vd fz = q0 + zt / (1. + ca);
        {
            const vd v = -oms * vd(ROWD(T, L.r + kb)) + eta * (ca * q0 + zt);
            ROWD(T, L.rhs2 + kb) = v;
            mx[0] = vmax(mx[0], vabs(v));
        }
        for (int k = 1; k < d; k++)
        {
            const vd v = -oms * vd(ROWD(T, L.r + kb + k)) +
                         eta * (vd(ROWD(T, L.dsw + zs + k)) + fz * vd(ROWD(T, L.cq + qo + k - 1)));
            ROWD(T, L.rhs2 + kb + k) = v;
            mx[0] = vmax(mx[0], vabs(v));
        }
        ROWD(T, L.rhs2 + kb + d) = 0.0;
        ROWD(T, L.rhs2 + kb + d + 1) = 0.0;
    }
    team_max<1>(tm, mx);
    if (tm.wk == 0)
        ROWD(T, L.sc + S_RHSMAX2) = vsel(act, mx[0], ROWD(T, L.sc + S_RHSMAX2));
}

// ------------------------------------------------------------------ combined step and iterate update (src/eicos.cpp:1214-1252)
EI_DEV void tile_tail(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const vb act = lane_active(tm, t);
    if (!tm.any(act))
        return;
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    const int n = P.n, zb = P.n + P.p;
    const vd tau = ROWD(T, L.sc + S_TAU), kap = ROWD(T, L.sc + S_KAP), rt = ROWD(T, L.sc + S_RT);
    const vd mu = ROWD(T, L.sc + S_MU), sigma = ROWD(T, L.sc + S_SIGMA);
    const vd dtau_denom = ROWD(T, L.sc + S_DTAU_DENOM), dtauaff = ROWD(T, L.sc + S_DTAUAFF);
    const vd dkapaff = ROWD(T, L.sc + S_DKAPAFF);

    vd dt[3] = {vset(0.0), vset(0.0), vset(0.0)};
    {
        const int ix[2] = {L.chb, L.sol2};
        ew_rows<2, 6>(tm, T, n, ix, [&](int, const vd *x) { dt[0] += x[0] * x[1]; });
        const int iy[2] = {L.chb + n, L.sol2 + n};
        ew_rows<2, 6>(tm, T, P.p, iy, [&](int, const vd *x) { dt[1] += x[0] * x[1]; });
        const int iz[2] = {L.chb + zb, L.sol2 + zb};
        ew_rows<2, 6>(tm, T, P.l, iz, [&](int, const vd *x) { dt[2] += x[0] * x[1]; });
    }
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    {
        const int d = EI_LDG(P.cone_dim + c), kb = zb + EI_LDG(P.cone_k + c);
        for (int k = 0; k < d; k++)
            dt[2] += vd(ROWD(T, L.chb + kb + k)) * vd(ROWD(T, L.sol2 + kb + k));
    }
    team_sum<3>(tm, dt);
    const vd bkap = kap * tau + dkapaff * dtauaff - sigma * mu;
    const vd dtau = ((1. - sigma) * rt - bkap / tau + dt[0] + dt[1] + dt[2]) / dtau_denom;
    // LP rows in one pass: dz = dz2 + dtau * dz1, W dz, ds = -(ds + W dz), min ratios of the line search.
    // Nothing is stored: the update pass below recomputes dz and ds (and dx, dy) in registers.
    vd m0 = vset(DBL_MAX), m1 = vset(DBL_MAX);
    {
        const int ins[5] = {L.sol2 + zb, L.sol1 + zb, L.lpw, L.dsw, lp_lambda_row(P, L)};
        ew_rows<5, 2>(tm, T, P.l, ins, [&](int, const vd *x) {
            const vd lk = lp_lambda(P, x[2], x[4]);
            const vd wd = vmul_rn(x[2], vfma(dtau, x[1], x[0]));
            const vd ds = -(x[3] + wd);
            m0 = vmin(m0, ds / lk);
            m1 = vmin(m1, wd / lk);
        });
    }
    if (P.mt > P.l)
    { // cone rows: pass by pass
        const int cz = zb + P.l, nr = P.mt - P.l;
        const int ins[2] = {L.sol2 + cz, L.sol1 + cz};
        ew_rows<2, 6>(tm, T, nr, ins, [&](int e, const vd *x) { ROWD(T, L.sol2 + cz + e) = x[0] + dtau * x[1]; });
        tm.sync();
        cone_scale(tm, a, T, L.sol2 + zb, L.wdz, vbset(true), false);
        tm.sync();
        const int in2[2] = {L.dsw + P.l, L.wdz + P.l};
        ew_rows<2, 6>(tm, T, nr, in2, [&](int e, const vd *x) { ROWD(T, L.dsw + P.l + e) = -(x[0] + x[1]); });
        tm.sync();
    }
    const vd dkap = -(bkap + kap * dtau) / tau;
    const vd step = a.settings.gamma * line_search(tm, a, T, L.lam, L.dsw, L.wdz, tau, dtau, kap, dkap, false, m0, m1);
    if (P.mt > P.l)
    {
        cone_scale(tm, a, T, L.dsw, L.dsaff, vbset(true), false);
        tm.sync();
    }
    {
        // x, y += step * (dxy2 + dtau * dxy1)
        const int ins[3] = {L.w, L.sol2, L.sol1};
        ew_rows<3, 4>(tm, T, zb, ins, [&](int q, const vd *x) { ROWD(T, L.w + q) = vsel(act, x[0] + step * (x[1] + dtau * x[2]), x[0]); });
        // LP rows: z += step * dz and s += step * (W ds) in one pass, dz and ds as in the pass before the line search
        const int inl[6] = {L.w + zb, L.sol2 + zb, L.sol1 + zb, L.s, L.lpw, L.dsw};
        ew_rows<6, 2>(tm, T, P.l, inl, [&](int k, const vd *x) {
            const vd dz = vfma(dtau, x[2], x[1]);
            const vd ds = -(x[5] + vmul_rn(x[4], dz));
            ROWD(T, L.w + zb + k) = vsel(act, vfma(step, dz, x[0]), x[0]);
            ROWD(T, L.s + k) = vsel(act, vfma(step, vmul_rn(x[4], ds), x[3]), x[3]);
        });
    }
    for (int c = tm.wk; c < P.nc; c += tm.nwk)
    { // cone rows of z; the expansion slots of the iterate stay zero
        const int d = EI_LDG(P.cone_dim + c), kb = zb + EI_LDG(P.cone_k + c);
        for (int k = 0; k < d; k++)
            ROWD(T, L.w + kb + k) = vsel(act, vd(ROWD(T, L.w + kb + k)) + step * vd(ROWD(T, L.sol2 + kb + k)), ROWD(T, L.w + kb + k));
    }
    if (P.mt > P.l)
    {
        const int ins[2] = {L.s + P.l, L.dsaff + P.l};
        ew_rows<2, 6>(tm, T, P.mt - P.l, ins, [&](int e, const vd *x) { ROWD(T, L.s + P.l + e) = vsel(act, x[0] + step * x[1], x[0]); });
    }
    if (tm.wk == 0)
        VFOR if (act.v[c_])
        {
            ROWC(T, L.sc + S_KAP, c_) = kap.v[c_] + step.v[c_] * dkap.v[c_];
            ROWC(T, L.sc + S_TAU, c_) = tau.v[c_] + step.v[c_] * dtau.v[c_];
            ROWC(T, L.sc + S_STEP, c_) = step.v[c_];
            ROWC(t.I, J_ITER, c_) += 1;
        }
}

// ------------------------------------------------------------------ data in / results out
// Inputs are instance-major (what the C ABI receives); they are equilibrated on the way in
// (c / x_equil, h / G_equil, b / A_equil : src/eicos.cpp:364-371) and land KKT-shaped in `chb`.
EI_DEV void tile_load(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    const int n = P.n, zb = P.n + P.p;
    VFOR
    {
        int inst = tile * TILE + tm.lane + c_;
        if (inst >= a.batch)
            inst = a.batch - 1; // padding instances replay the last one; their results are never stored
        const size_t g = (size_t)a.first + inst;
        if (P.pim)
        { // raw data in; eicos_equilibrate scales matrices and vectors per instance
            for (int j = tm.wk; j < n; j += tm.nwk)
                ROWC(t.T, L.chb + j, c_) = a.in_c ? a.in_c[g * n + j] : EI_LDG(a.base_c + j);
            for (int i = tm.wk; i < P.p; i += tm.nwk)
                ROWC(t.T, L.chb + n + i, c_) = a.in_b ? a.in_b[g * P.p + i] : EI_LDG(a.base_b + i);
            for (int i = tm.wk; i < P.m; i += tm.nwk)
                ROWC(t.T, L.chb + zb + EI_LDG(P.zk + i), c_) = a.in_h ? a.in_h[g * P.m + i] : EI_LDG(a.base_h + i);
            for (int k = tm.wk; k < P.nnzG; k += tm.nwk)
                ROWC(t.T, L.Gx + k, c_) = a.in_G ? a.in_G[g * P.nnzG + k] : EI_LDG(a.base_G + k);
            for (int k = tm.wk; k < P.nnzA; k += tm.nwk)
                ROWC(t.T, L.Ax + k, c_) = a.in_A ? a.in_A[g * P.nnzA + k] : EI_LDG(a.base_A + k);
            continue;
        }
        for (int j = tm.wk; j < n; j += tm.nwk)
        {
            const double v = a.in_c ? a.in_c[g * n + j] : EI_LDG(a.base_c + j);
            ROWC(t.T, L.chb + j, c_) = a.pre_equilibrated ? v : v / EI_LDG(P.xeq + j);
        }
        for (int i = tm.wk; i < P.p; i += tm.nwk)
        {
            const double v = a.in_b ? a.in_b[g * P.p + i] : EI_LDG(a.base_b + i);
            ROWC(t.T, L.chb + n + i, c_) = a.pre_equilibrated ? v : v / EI_LDG(P.Aeq + i);
        }
        for (int i = tm.wk; i < P.m; i += tm.nwk)
        {
            const double v = a.in_h ? a.in_h[g * P.m + i] : EI_LDG(a.base_h + i);
            const int e = EI_LDG(P.zk + i);
            ROWC(t.T, L.chb + zb + e, c_) = a.pre_equilibrated ? v : v / EI_LDG(P.GeqE + e);
        }
    }
}

// ------------------------------------------------------------------ on-device equilibration (per-instance-matrices mode)
// max |row| over the entries k0..k1-1 of an index walk, folded into mx in walk order; the row loads of
// four entries are issued before the first compare so that they overlap (the walk is latency-bound).
template <class RowOf>
EI_DEV vd equil_max_abs(const double *T, int k0, int k1, vd mx, RowOf row)
{
    int k = k0;
    for (; k + 4 <= k1; k += 4)
    {
        vd v[4];
#pragma unroll
        for (int u = 0; u < 4; u++)
            v[u] = vload(T + (size_t)row(k + u) * TILE);
#pragma unroll
        for (int u = 0; u < 4; u++)
            mx = vmax(vabs(v[u]), mx);
    }
    for (; k < k1; k++)
        mx = vmax(vabs(vload(T + (size_t)row(k) * TILE)), mx);
    return mx;
}

// entries k0..k1-1 of a CSC column: value /= row scale, then /= column scale (two divisions, src/eicos.cpp:353-356)
EI_DEV void equil_scale_column(double *T, int val0, int scale0, const int *rows, int k0, int k1, vd cj)
{
    int k = k0;
    for (; k + 4 <= k1; k += 4)
    {
        vd v[4], r[4];
#pragma unroll
        for (int u = 0; u < 4; u++)
        {
            v[u] = vload(T + (size_t)(val0 + k + u) * TILE);
            r[u] = vload(T + (size_t)(scale0 + EI_LDG(rows + k + u)) * TILE);
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
            vstore(T + (size_t)(val0 + k + u) * TILE, v[u] / r[u] / cj);
    }
    for (; k < k1; k++)
        ROWD(T, val0 + k) = vd(ROWD(T, val0 + k)) / vd(ROWD(T, scale0 + EI_LDG(rows + k))) / cj;
}

// setEquilibration (src/eicos.cpp:302-374) for every instance of the tile: equil_iters rounds of
// column / row infinity-norm scaling of [A; G] (the rows of a second-order cone share the sum of
// their norms), rows first then columns as two separate divisions, scales accumulated into
// x_equil / A_equil / G_equil; then c, b, h are divided by them.  Work vectors: xw.
EI_DEV void tile_equil(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    const int n = P.n, p = P.p, zb = P.n + P.p;
    const int cs = L.xw, ra = L.xw + n, rg = L.xw + zb; // column scales, row scales of A, of G (z index, not expanded)
    const auto root = [](vd v) {
        VFOR v.v[c_] = fabs(v.v[c_]) < 1e-6 ? 1.0 : sqrt(v.v[c_]);
        return v;
    };
    for (int r = tm.wk; r < P.N; r += tm.nwk)
        ROWD(T, L.eq + r) = 1.0;
    tm.sync();
    for (int round = 0; round < Settings::equil_iters; round++)
    {
        for (int j = tm.wk; j < n; j += tm.nwk)
        { // maxCols over A then G (:267)
            vd mx = equil_max_abs(T, EI_LDG(P.Ap + j), EI_LDG(P.Ap + j + 1), vset(0.0), [&](int k) { return L.Ax + k; });
            ROWD(T, cs + j) = equil_max_abs(T, EI_LDG(P.Gp + j), EI_LDG(P.Gp + j + 1), mx, [&](int k) { return L.Gx + k; });
        }
        for (int i = tm.wk; i < p; i += tm.nwk) // maxRows (:256)
            ROWD(T, ra + i) = equil_max_abs(T, EI_LDG(P.Arp + i), EI_LDG(P.Arp + i + 1), vset(0.0),
                                            [&](int q) { return L.Ax + EI_LDG(P.Arv + q); });
        for (int i = tm.wk; i < P.m; i += tm.nwk)
            ROWD(T, rg + i) = equil_max_abs(T, EI_LDG(P.Grp + i), EI_LDG(P.Grp + i + 1), vset(0.0),
                                            [&](int q) { return L.Gx + EI_LDG(P.Grv + q); });
        tm.sync();
        for (int c = tm.wk; c < P.nc; c += tm.nwk)
        { // every row of a cone gets the sum over the cone (:338-344)
            const int d = EI_LDG(P.cone_dim + c), z0 = EI_LDG(P.cone_z + c);
            vd tot = vset(0.0);
            for (int k = 0; k < d; k++)
                tot += vd(ROWD(T, rg + z0 + k));
            for (int k = 0; k < d; k++)
                ROWD(T, rg + z0 + k) = tot;
        }
        tm.sync();
        for (int r = tm.wk; r < zb + P.m; r += tm.nwk)
            ROWD(T, cs + r) = root(ROWD(T, cs + r));
        tm.sync();
        for (int j = tm.wk; j < n; j += tm.nwk)
        { // rows first, then columns: two divisions per entry (:353-356)
            const vd cj = ROWD(T, cs + j);
            equil_scale_column(T, L.Ax, ra, P.Ai, EI_LDG(P.Ap + j), EI_LDG(P.Ap + j + 1), cj);
            equil_scale_column(T, L.Gx, rg, P.Gi, EI_LDG(P.Gp + j), EI_LDG(P.Gp + j + 1), cj);
            ROWD(T, L.eq + j) *= cj;
        }
        for (int i = tm.wk; i < p; i += tm.nwk)
            ROWD(T, L.eq + n + i) *= vd(ROWD(T, ra + i));
        for (int i = tm.wk; i < P.m; i += tm.nwk)
            ROWD(T, L.eq + zb + EI_LDG(P.zk + i)) *= vd(ROWD(T, rg + i));
        tm.sync();
    }
    for (int j = tm.wk; j < n; j += tm.nwk)
        ROWD(T, L.chb + j) = vd(ROWD(T, L.chb + j)) / vd(ROWD(T, L.eq + j));
    for (int i = tm.wk; i < p; i += tm.nwk)
        ROWD(T, L.chb + n + i) = vd(ROWD(T, L.chb + n + i)) / vd(ROWD(T, L.eq + n + i));
    for (int i = tm.wk; i < P.m; i += tm.nwk)
    {
        const int e = EI_LDG(P.zk + i);
        ROWD(T, L.chb + zb + e) = vd(ROWD(T, L.chb + zb + e)) / vd(ROWD(T, L.eq + zb + e));
    }
}

EI_DEV void tile_store(const Team &tm, const KArgs &a, int tile)
{
    // Writes the results of every instance of the tile that has finished and has not been stored yet
    // (called once at the end, and before a compaction frees the slots of finished instances).
    const TileMem t = tile_mem(tm, a, tile);
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    const int n = P.n, zb = P.n + P.p;
    VFOR
    {
        const int inst = ROWC(t.I, J_INST, c_);
        if (inst < 0 || ROWC(t.I, J_STORED, c_) || ROWC(t.I, J_STATUS, c_) == ST_ACTIVE)
            continue;
        const size_t g = (size_t)inst;
        if (a.out_x)
            for (int j = tm.wk; j < n; j += tm.nwk)
                a.out_x[g * n + j] = ROWC(t.T, L.w + j, c_);
        if (a.out_y)
            for (int i = tm.wk; i < P.p; i += tm.nwk)
                a.out_y[g * P.p + i] = ROWC(t.T, L.w + n + i, c_);
        if (a.out_z)
            for (int i = tm.wk; i < P.m; i += tm.nwk)
                a.out_z[g * P.m + i] = ROWC(t.T, L.w + zb + EI_LDG(P.zk + i), c_);
        if (a.out_s)
            for (int i = tm.wk; i < P.m; i += tm.nwk)
                a.out_s[g * P.m + i] = ROWC(t.T, L.s + EI_LDG(P.zk + i), c_);
        if (tm.wk == 0)
        {
            if (a.out_exit)
                a.out_exit[g] = ROWC(t.I, J_STATUS, c_);
            if (a.out_iter)
                a.out_iter[g] = ROWC(t.I, J_ITER, c_);
            if (a.out_info)
                for (int k = 0; k < S_WORK_END; k++)
                    a.out_info[g * S_WORK_END + k] = ROWC(t.T, L.sc + k, c_);
            if (a.out_iinfo)
                for (int k = 0; k < J_WORK_END; k++)
                    a.out_iinfo[g * J_WORK_END + k] = ROWC(t.I, k, c_);
        }
    }
    tm.sync();
    if (tm.wk == 0)
        VFOR if (ROWC(t.I, J_INST, c_) >= 0 && ROWC(t.I, J_STATUS, c_) != ST_ACTIVE) ROWC(t.I, J_STORED, c_) = 1;
}

// ------------------------------------------------------------------ debug: lineSearch on caller data (unit tests)
// in_h / in_G / in_A: lambda, ds, dz (instance-major, compact z order); in_b: tau, dtau, kap, dkap per instance;
// out_x: the step length.  Lets a test drive the line search into states a solve hardly ever reaches.
EI_DEV void tile_debug_line_search(const Team &tm, const KArgs &a, int tile)
{
    const TileMem t = tile_mem(tm, a, tile);
    const DevPattern &P = a.P;
    const Layout &L = a.L;
    double *T = t.T;
    const int base = tile * TILE + tm.lane;
    for (int i = tm.wk; i < P.m; i += tm.nwk)
    {
        const int e = EI_LDG(P.zk + i);
        VFOR
        {
            const int inst = base + c_;
            const bool ok = inst < a.batch;
            ROWC(T, L.lam + e, c_) = ok ? a.in_h[(size_t)inst * P.m + i] : 1.0;
            ROWC(T, L.dsw + e, c_) = ok ? a.in_G[(size_t)inst * P.m + i] : 0.0;
            ROWC(T, L.wdz + e, c_) = ok ? a.in_A[(size_t)inst * P.m + i] : 0.0;
        }
    }
    tm.sync();
    vd sc[4];
    for (int k = 0; k < 4; k++)
        VFOR sc[k].v[c_] = base + c_ < a.batch ? a.in_b[(size_t)(base + c_) * 4 + k] : 1.0;
    const vd alpha = line_search(tm, a, T, L.lam, L.dsw, L.wdz, sc[0], sc[1], sc[2], sc[3]);
    if (tm.wk == 0)
        VFOR if (base + c_ < a.batch) a.out_x[base + c_] = alpha.v[c_];
}

// ------------------------------------------------------------------ active-set compaction
// Moves one still-active instance from slot `src` to the free slot `dst` (slot = tile * TILE + lane
// position): the rows that carry state across iterations are copied, everything else is recomputed.
struct MoveRanges
{
    int n;        // number of (first row, rows) pairs
    int r[14];
};
EI_DEV void compact_move(const KArgs &a, const MoveRanges &mr, int src, int dst, int tid, int nthreads)
{
    const size_t st = (size_t)(src / TILE), dt = (size_t)(dst / TILE);
    const int sl = src % TILE, dl = dst % TILE;
    const double *S = a.ws + st * a.L.rows_total * TILE + sl;
    double *D = a.ws + dt * a.L.rows_total * TILE + dl;
    for (int q = 0; q < mr.n; q++)
        for (int r = mr.r[2 * q] + tid, e = mr.r[2 * q] + mr.r[2 * q + 1]; r < e; r += nthreads)
            D[(size_t)r * TILE] = S[(size_t)r * TILE];
    int *SI = a.iws + st * a.L.irows_total * TILE + sl, *DI = a.iws + dt * a.L.irows_total * TILE + dl;
    for (int r = tid; r < J_COUNT; r += nthreads)
        DI[(size_t)r * TILE] = SI[(size_t)r * TILE];
}
EI_DEV void compact_vacate(const KArgs &a, int src)
{ // the source slot becomes an empty, already-stored, inactive slot
    int *SI = a.iws + (size_t)(src / TILE) * a.L.irows_total * TILE + src % TILE;
    SI[(size_t)J_STATUS * TILE] = EXIT_FATAL;
    SI[(size_t)J_INST * TILE] = -1;
    SI[(size_t)J_STORED * TILE] = 1;
}

} // namespace eicos
