// Host orchestration of the batched interior-point loop + the __global__ entry points.
// Compiled by nvcc for sm_100a (product) or by g++ with -DEICOS_EMU (tests/emu only).
#include "engine.hpp"
#include "backend.hpp"
#include "tile_program.hpp"

#include <algorithm>
#include <cstdint>
#ifdef EICOS_EMU
#include <thread>
#endif

namespace eicos
{

#ifndef EICOS_EMU
// thin named wrappers so that profilers show one kernel name per step of the algorithm
#define EI_DEFINE_KERNEL(name, fn, minblocks) EI_DEFINE_KERNEL_(name, fn, EI_MAX_THREADS, minblocks, 0)
/* one-warp program kernels: no register cap below the hardware's (a handful of CTAs per SM, limited by shared memory) */
#define EI_DEFINE_KERNEL1(name, fn) EI_DEFINE_KERNEL_(name, fn, 32, 8, 0)
#define EI_DEFINE_KERNEL_(name, fn, maxthreads, minblocks, JOBS)                                           \
    __global__ void __launch_bounds__(maxthreads, minblocks) name(const __grid_constant__ KArgs a) \
    {                                                                                          \
        extern __shared__ double smem[];                                                       \
        Team tm;                                                                               \
        tm.pl = threadIdx.x & 31;                                                              \
        tm.lane = tm.pl * VEC;                                                                 \
        tm.wk = threadIdx.x >> 5;                                                              \
        tm.nwk = blockDim.x >> 5;                                                              \
        tm.red = smem;                                                                         \
        /* vector kernels (several warps): [reduction rows]; program kernels (one warp): the shared  \
           memory of the FMA machine (ops ring, mbarriers, rows) at pbuf */                          \
        tm.pbuf = smem + (size_t)(tm.nwk > 1 ? tm.nwk * KRED : 0) * TILE;                           \
        tm.job = JOBS ? (int)(blockIdx.x % (unsigned)a.njobs) : 0;                                 \
        fn(tm, a, JOBS ? (int)(blockIdx.x / (unsigned)a.njobs) : (int)blockIdx.x);                                                                 \
    }
#define EI_MAX_THREADS 256
EI_DEFINE_KERNEL(eicos_load_inputs, tile_load, 2)
EI_DEFINE_KERNEL(eicos_equilibrate, tile_equil, 2)
EI_DEFINE_KERNEL(eicos_init, tile_init, 2)
EI_DEFINE_KERNEL1(eicos_ldl_factor, tile_factor)
EI_DEFINE_KERNEL_(eicos_solve_kkt, tile_solve_kkt<1>, 32, 8, 1) /* CTA = (tile, job): one solveKKT each */
EI_DEFINE_KERNEL_(eicos_solve_kkt_pair, tile_solve_kkt<2>, 32, 7, 0) /* two solveKKT that share the factor, one pass over L */
/* few tiles: four warps per CTA, the residual rows split over them (M_MV_PARTS machines side by side) */
EI_DEFINE_KERNEL_(eicos_solve_kkt_wide, tile_solve_kkt<1>, 32 * M_MV_PARTS, 2, 1)
EI_DEFINE_KERNEL_(eicos_residuals_wide, tile_resid, 32 * M_MV_PARTS, 2, 0)
EI_DEFINE_KERNEL(eicos_init_point, tile_init_point, 2)
EI_DEFINE_KERNEL1(eicos_residuals, tile_resid)
EI_DEFINE_KERNEL(eicos_iter_head, tile_head, 2)
EI_DEFINE_KERNEL(eicos_iter_mid, tile_mid, 2)
EI_DEFINE_KERNEL(eicos_iter_tail, tile_tail, 2)
EI_DEFINE_KERNEL(eicos_store_outputs, tile_store, 2)
EI_DEFINE_KERNEL(eicos_debug_line_search, tile_debug_line_search, 2)

#define EI_LAUNCH(name, fn, tiles, threads, smem, stream, args) name<<<(tiles), (threads), (smem), (stream)>>>(args)
#define EI_LAUNCH_JOBS(name, fn, tiles, njobs, threads, smem, stream, args) \
    name<<<(tiles) * (njobs), (threads), (smem), (stream)>>>(args)

__global__ void eicos_compact(const __grid_constant__ KArgs a, const __grid_constant__ MoveRanges mr, const int *moves)
{
    const int src = moves[2 * blockIdx.x], dst = moves[2 * blockIdx.x + 1];
    compact_move(a, mr, src, dst, threadIdx.x, blockDim.x);
    __syncthreads();
    if (threadIdx.x == 0)
        compact_vacate(a, src);
}
#else
#define EI_MAX_THREADS 256
// emulator: one std::thread per worker of a tile, CTA barrier = std::barrier
#define EI_LAUNCH(name, fn, tiles, threads, smem, stream, args) EI_LAUNCH_JOBS(name, fn, tiles, 1, threads, smem, stream, args)
#define EI_LAUNCH_JOBS(name, fn, tiles, njobs, threads, smem, stream, args)                       \
    do                                                                                            \
    {                                                                                             \
        const int nw_ = (threads), nj_ = (njobs);                                                                \
        std::vector<double> red_((size_t)nw_ * KRED * TILE + 8);                                  \
        std::vector<double> pb_(M_MV_PARTS * machine_smem_doubles(std::max(std::max((args).P.sw_budget, (args).P.fa_budget), (args).P.pair_budget), M_MAX_RING_GROUPS, 2) + 8); \
        for (int cta_ = 0; cta_ < (tiles) * nj_; cta_++)                                          \
        {                                                                                         \
            const int tile_ = cta_ / nj_;                                                         \
            std::barrier<> bar_(nw_);                                                             \
            auto body_ = [&](int wk_) {                                                           \
                Team tm_;                                                                         \
                tm_.lane = 0;                                                                     \
                tm_.pl = 0;                                                                       \
                tm_.wk = wk_;                                                                     \
                tm_.nwk = nw_;                                                                    \
                tm_.job = cta_ % nj_;                                                             \
                tm_.red = red_.data();                                                            \
                tm_.pbuf = pb_.data();                                                            \
                tm_.bar = nw_ > 1 ? &bar_ : nullptr;                                              \
                fn(tm_, (args), tile_);                                                           \
            };                                                                                    \
            std::vector<std::thread> th_;                                                         \
            for (int wk_ = 1; wk_ < nw_; wk_++)                                                   \
                th_.emplace_back(body_, wk_);                                                     \
            body_(0);                                                                             \
            for (auto &t_ : th_)                                                                  \
                t_.join();                                                                        \
        }                                                                                         \
    } while (0)
#endif

#ifdef EICOS_EMU
static void eicos_compact_emu(const KArgs &a, const MoveRanges &mr, const int *moves, int nmoves)
{
    for (int q = 0; q < nmoves; q++)
    {
        compact_move(a, mr, moves[2 * q], moves[2 * q + 1], 0, 1);
        compact_vacate(a, moves[2 * q]);
    }
}
#endif

// slot budgets of the machine programs (a slot = one row of TILE doubles; two rows in the two-job programs).
// With the shallow ring (24 rows) a solveKKT / residual CTA takes 25 KB of shared memory: 9 per SM; a factor CTA 29 KB: 7 per SM,
// one wave for the 1024 tiles of the benchmark batch.
constexpr int MAX_SW_SLOTS = 16, MAX_FA_SLOTS = 24;

int Engine::tile_width() { return TILE; }

// A launch of `ctas` one-warp CTAs runs the deep-ring programs when all of them are resident at the deep
// ring's shared-memory footprint (then nothing is lost by giving each tile more rows in flight).
// The two solves of an iteration that share the factor run as CTAs (tile, job); EICOS_PAIR_SOLVES = 1 runs them as ONE
// CTA per tile with the two-job programs instead (one pass over L for both right-hand sides: less HBM traffic, but on
// B200 the wider operations cost more shared-memory bandwidth than the shared L saves - measured slower, kept as an
// option and as a parity check of the two-job machine).
bool Engine::pair_solves(int) const { return force_pair_ > 0; }

// Ring depth of a launch.  The bytes ONE tile has in flight bound its pace when few tiles share an SM (a sweep of
// MPC02 copies 11 MB per tile through a ring of 12 KB: 12 KB per memory latency); with the machine full the shallow
// ring's smaller footprint (9 tiles per SM instead of 6) wins (65 536 instances: 41.0 k solves/s at 3 groups, 37.6 k at
// 5 or 6).  Measured crossover: every launch deep gains 5.7 % at 16 384 instances (512 CTAs in the paired solve) and
// loses 4.5 % at 32 768 (1 024 CTAs: two waves at the deep footprint), so a launch takes the deep programs when all
// its CTAs are resident with them; the wide launches always do for their sweeps.  EICOS_RING_VARIANT = 0 / 1 pins the choice for every launch.
bool Engine::deep_ring(int ctas) const
{
    if (force_variant_ >= 0)
        return force_variant_ > 0;
    // ... when all of its CTAs are resident at the deep programs' footprint (MPC02: six per SM; measured 4 / 5 / 6 per
    // SM: 44.29 k / 44.30 k / 44.50 k solves/s at 65 536 instances, 39.96 k / 40.04 k / 40.36 k at 49 152)
    long long per_sm = (long long)((size_t)227 * 1024 / (smem_prog_[M_VARIANTS - 1] + 1024));
    if (const char *v = std::getenv("EICOS_DEEP_CTAS_PER_SM")) // (diagnostics)
        per_sm = std::atoi(v);
    return (long long)ctas <= per_sm * sms_;
}

// A launch with few CTAs (all resident at the wide kernels' shared-memory footprint) runs the wide kernels: four warps
// per CTA, the rows of the mat-vec programs split over them.  EICOS_WIDE = 0 / 1 pins the choice.
bool Engine::wide_launch(int ctas) const
{
    if (force_wide_ >= 0)
        return force_wide_ > 0;
    const long long per_sm = (long long)((size_t)227 * 1024 / (smem_wide_ + 1024));
    return per_sm > 0 && (long long)ctas <= per_sm * sms_;
}

namespace
{
template <class T>
T *upload(const std::vector<T> &v, std::vector<void *> &owned, be::stream_t s)
{
    T *d = (T *)be::alloc(v.size() * sizeof(T));
    be::h2d(d, v.data(), v.size() * sizeof(T), s);
    owned.push_back(d);
    return d;
}
inline be::stream_t S_(void *p) { return (be::stream_t)(intptr_t)p; }

dvec expanded_geq(const Symbolic &S)
{
    dvec g(S.mt, 1.0);
    for (int i = 0; i < S.m; i++)
        g[S.zk[i]] = S.Geq[i];
    return g;
}
} // namespace

void Engine::build_layout(const Symbolic &S, bool acc_rows)
{
    int at = 0;
    auto take = [&](int rows) {
        const int o = at;
        at += rows;
        return o;
    };
    Layout &L = L_;
    L.chb = take(S.N);
    L.w = take(S.N);
    L.s = take(S.mt);
    L.lam = take(S.mt);
    L.wb = take(S.N);
    L.bs = take(S.mt);
    L.r = take(S.N);
    L.lpv = take(S.l);
    L.lpw = take(S.l);
    L.cpar = take(S.nc * CP_COUNT);
    L.cq = take(S.qtot);
    L.V = take((int)S.Vslot.size());
    L.Lx = take(S.nnzL);
    L.D = take(S.N);
    L.Dinv = take(S.N);
    L.rhs1 = take(S.N);
    L.rhs2 = take(S.N);
    L.sol1 = take(S.N);
    L.sol2 = take(S.N);
    L.xw = take(S.N);
    L.dxr = take(S.N);
    L.e = take(S.N);
    L.xw2 = take(S.N);
    L.dxr2 = take(S.N);
    L.e2 = take(S.N);
    L.dsw = take(S.mt);
    L.wdz = take(S.mt);
    L.dsaff = take(S.mt);
    L.ds1 = take(S.mt);
    L.Gx = take(pim_ ? S.G.nnz() : 0);
    L.Ax = take(pim_ ? S.A.nnz() : 0);
    L.eq = take(pim_ ? S.N : 0);
    L.sc = take(S_COUNT);
    L.acc = acc_rows ? take(S.nnzL) : -1;
    L.rows_total = at;
    L.irows_total = J_COUNT;
}

void Engine::upload_pattern(const Symbolic &S)
{
    be::stream_t st = S_(stream_);
    // slot budgets; the environment overrides exist for the tests, which shrink them to force the
    // far-gather / direct-operand / general-form paths on small patterns
    int sw_budget = MAX_SW_SLOTS, fa_budget = MAX_FA_SLOTS;
    if (const char *v = std::getenv("EICOS_MAX_SW_SLOTS"))
        sw_budget = std::max(1, std::min(MAX_SW_SLOTS, std::atoi(v)));
    if (const char *v = std::getenv("EICOS_MAX_FA_SLOTS"))
        fa_budget = std::max(1, std::min(MAX_FA_SLOTS, std::atoi(v)));
    try
    {
        build_streams(S, L_, workers_, sw_budget, fa_budget, H_, pim_);
    }
    catch (const MachineOutOfSlots &)
    { // the factorisation's accumulators do not fit the slots: give them home rows
        if (L_.acc >= 0)
            throw;
        build_layout(S, true);
        build_streams(S, L_, workers_, sw_budget, fa_budget, H_, pim_);
    }
    Lp_ = S.Lp;
    DevPattern &P = P_;
    P.n = S.n;
    P.p = S.p;
    P.m = S.m;
    P.l = S.l;
    P.nc = S.nc;
    P.N = S.N;
    P.mt = S.mt;
    P.qtot = S.qtot;
    P.nnzL = S.nnzL;
    P.nnzV = (int)S.Vslot.size();
    P.maxcol = S.maxcol;
    P.pim = pim_ ? 1 : 0;
    P.nnzG = S.G.nnz();
    P.nnzA = S.A.nnz();
    if (pim_)
    {
        P.Gp = upload(S.G.p, owned_, st);
        P.Gi = upload(S.G.i, owned_, st);
        P.Ap = upload(S.A.p, owned_, st);
        P.Ai = upload(S.A.i, owned_, st);
        P.Grp = upload(S.Gr.p, owned_, st);
        P.Grv = upload(S.Gr.v, owned_, st);
        P.Arp = upload(S.Ar.p, owned_, st);
        P.Arv = upload(S.Ar.v, owned_, st);
        P.cone_z = upload(S.cone_z, owned_, st);
    }
    P.cone_dim = upload(S.q, owned_, st);
    P.cone_k = upload(S.cone_k, owned_, st);
    P.cone_q = upload(S.cone_q, owned_, st);
    P.zk = upload(S.zk, owned_, st);
    P.xeq = dxeq_ = upload(S.xeq, owned_, st);
    P.Aeq = dAeq_ = upload(S.Aeq, owned_, st);
    P.GeqE = dGeq_ = upload(expanded_geq(S), owned_, st);
    // machine programs: record streams as they are, load lists materialised per use
    // (selector -> row offset of the vector it stands for, streams.hpp; M_LD_NONE stays)
    const auto prog = [&](const MachineCode &h, DevMachine &d, int **keep = nullptr) {
        int *o = upload(h.ops, owned_, st);
        d.ops = o;
        d.nchunks = h.nchunks;
        d.nld_chunks = h.nld_chunks;
        d.ring_groups = h.ring_groups;
        d.ring_row0 = m_row_slot0(h.nr) + h.nr * h.slot_budget;
        if (keep)
            *keep = o;
    };
    // offsets of the vectors the selectors 1.. stand for: job A, then job B (two-job programs)
    const auto variant = [&](const ivec &list, std::initializer_list<int> va, std::initializer_list<int> vb = {}) {
        ivec out(list.size());
        int off[16] = {0};
        int k = 1;
        for (int o : va)
            off[k++] = o;
        k = 9;
        for (int o : vb)
            off[k++] = o;
        for (size_t q = 0; q < list.size(); q++)
        { // (padding words copy row 0 of the tile into a ring row nobody reads: cheaper than a test per copy)
            const int w = list[q];
            out[q] = w == M_LD_NONE ? 0 : (w & M_LD_ROW_MASK) + off[(((unsigned)w >> M_LD_SEL_SHIFT) & 7) + ((w & M_LD_JOB_B) ? 8 : 0)];
        }
        return upload(out, owned_, st);
    };
    P.sw_budget = H_.fw[0].slot_budget;
    P.fa_budget = H_.fa[0].slot_budget;
    const int rhs[2] = {L_.rhs1, L_.rhs2}, sol[2] = {L_.sol1, L_.sol2}, xw[2] = {L_.xw, L_.xw2};
    const int dxr[2] = {L_.dxr, L_.dxr2}, er[2] = {L_.e, L_.e2};
    for (int v = 0; v < M_VARIANTS; v++)
    {
        prog(H_.fw[v], P.fw[v]);
        prog(H_.bw[v], P.bw[v]);
        prog(H_.bwp[v], P.bwp[v]);
        prog(H_.mv[v], P.mv[v], &dmv_ops_[v]);
        prog(H_.fa[v], P.fa[v], &dfa_ops_[v]);
        for (int set = 0; set < 2; set++)
        { // forward: 1 = right-hand side, 3 = xw; backward: 1 = output, 2 = accumulated solution, 3 = xw
            P.fw_ld[v][set][0] = variant(H_.fw[v].ld, {rhs[set], 0, xw[set]});
            P.fw_ld[v][set][1] = variant(H_.fw[v].ld, {er[set], 0, xw[set]});
            P.bw_ld[v][set][0] = variant(H_.bwp[v].ld, {sol[set], 0, xw[set], rhs[set]});
            P.bw_ld[v][set][1] = variant(H_.bw[v].ld, {dxr[set], sol[set], xw[set], er[set]});
            P.mv_ld[v][set] = variant(H_.mv[v].ld, {rhs[set], sol[set], L_.lpv, er[set]});
        }
        P.fa_ld[v] = variant(H_.fa[v].ld, {});
    }
    // the mat-vec programs in parts
    for (int k = 0; k < M_MV_PARTS; k++)
    {
        prog(H_.rs[k], P.rs[k], &drs_ops_[k]);
        prog(H_.mvw[k], P.mvw[k], &dmvw_ops_[k]);
        P.rs_ld[k] = variant(H_.rs[k].ld, {L_.chb, L_.w, L_.s, L_.r, L_.sc});
        for (int set = 0; set < 2; set++)
            P.mvw_ld[set][k] = variant(H_.mvw[k].ld, {rhs[set], sol[set], L_.lpv, er[set]});
    }
    // two-job programs: job A = set 0 (rhs1 / sol1), job B = set 1 (rhs2 / sol2)
    P.pair_budget = H_.pair_budget;
    prog(H_.fw2, P.fw2);
    prog(H_.bw2, P.bw2);
    prog(H_.bwp2, P.bwp2);
    prog(H_.mv2, P.mv2, &dmv2_ops_);
    P.fw2_ld[0] = variant(H_.fw2.ld, {rhs[0], 0, xw[0]}, {rhs[1], 0, xw[1]});
    P.fw2_ld[1] = variant(H_.fw2.ld, {er[0], 0, xw[0]}, {er[1], 0, xw[1]});
    P.bw2_ld[0] = variant(H_.bwp2.ld, {sol[0], 0, xw[0], rhs[0]}, {sol[1], 0, xw[1], rhs[1]});
    P.bw2_ld[1] = variant(H_.bw2.ld, {dxr[0], sol[0], xw[0], er[0]}, {dxr[1], sol[1], xw[1], er[1]});
    P.mv2_ld = variant(H_.mv2.ld, {rhs[0], sol[0], L_.lpv, er[0]}, {rhs[1], sol[1], L_.lpv, er[1]});
    P.mv_rows = H_.mv_rows;
    ivec vk;
    for (int k = 0; k < S.l; k++)
        vk.push_back(0);
    for (int d : S.q)
    {
        for (int k = 0; k < d + 1; k++)
            vk.push_back(0); // D block and the v diagonal: -1
        for (int k = 1; k < d; k++)
            vk.push_back(1); // v: 0
        vk.push_back(2);     // u diagonal: +1
        for (int k = 0; k < d; k++)
            vk.push_back(1); // u: 0
    }
    P.Vkind = upload(vk, owned_, st);
    be::sync(st);
}

void Engine::upload_values(const Symbolic &S)
{
    be::stream_t st = S_(stream_);
    be::set_device(device_);
    refresh_stream_values(S, L_, H_, pim_);
    const dvec ge = expanded_geq(S);
    be::h2d(dxeq_, S.xeq.data(), S.xeq.size() * sizeof(double), st);
    be::h2d(dAeq_, S.Aeq.data(), S.Aeq.size() * sizeof(double), st);
    be::h2d(dGeq_, ge.data(), ge.size() * sizeof(double), st);
    // the mat-vec and factor programs carry the shared coefficients inline
    for (int v = 0; v < M_VARIANTS; v++)
    {
        be::h2d(dmv_ops_[v], H_.mv[v].ops.data(), H_.mv[v].ops.size() * sizeof(int), st);
        be::h2d(dfa_ops_[v], H_.fa[v].ops.data(), H_.fa[v].ops.size() * sizeof(int), st);
    }
    be::h2d(dmv2_ops_, H_.mv2.ops.data(), H_.mv2.ops.size() * sizeof(int), st);
    for (int k = 0; k < M_MV_PARTS; k++)
    {
        be::h2d(drs_ops_[k], H_.rs[k].ops.data(), H_.rs[k].ops.size() * sizeof(int), st);
        be::h2d(dmvw_ops_[k], H_.mvw[k].ops.data(), H_.mvw[k].ops.size() * sizeof(int), st);
    }
    be::sync(st);
}

Engine::Engine(const Symbolic &S, int device, long long capacity_instances, int workers, bool instance_matrices)
    : device_(device), workers_(std::max(1, std::min(workers, EI_MAX_THREADS / 32 > 0 ? EI_MAX_THREADS / 32 : 1))),
      pim_(instance_matrices), nnzG_(S.G.nnz()), nnzA_(S.A.nnz())
{
    be::set_device(device_);
    if (const char *v = std::getenv("EICOS_RING_VARIANT")) // (diagnostics / tests) pin the ring depth of every launch
        force_variant_ = std::atoi(v);
    if (const char *v = std::getenv("EICOS_PAIR_SOLVES")) // ... and the form of the paired solves
        force_pair_ = std::atoi(v);
    if (const char *v = std::getenv("EICOS_WIDE")) // ... and the wide kernels
        force_wide_ = std::atoi(v);
    stream_ = (void *)(intptr_t)be::make_stream();
    build_layout(S, false);
    upload_pattern(S);
    cap_tiles_ = std::max<long long>(1, (capacity_instances + TILE - 1) / TILE);
    ws_bytes_ = (size_t)cap_tiles_ * L_.rows_total * TILE * sizeof(double);
    ws_ = (double *)be::alloc(ws_bytes_);
    const size_t ib = (size_t)cap_tiles_ * L_.irows_total * TILE * sizeof(int);
    iws_ = (int *)be::alloc(ib);
    be::zero(ws_, ws_bytes_, S_(stream_));
    be::zero(iws_, ib, S_(stream_));
    base_vec_ = (double *)be::alloc((size_t)(S.n + S.m + S.p) * sizeof(double));
    if (pim_)
        base_mat_ = (double *)be::alloc((size_t)(nnzG_ + nnzA_ + 1) * sizeof(double));
    active_count_ = (unsigned int *)be::alloc(sizeof(unsigned int));
    ir_rounds_ = (unsigned long long *)be::alloc(8 * sizeof(unsigned long long)); // [0] rounds, [1..5] phase cycles
    host_pinned_ = (unsigned int *)be::pinned(12 * sizeof(unsigned long long));
    const size_t slots = (size_t)cap_tiles_ * TILE;
    moves_dev_ = (int *)be::alloc(2 * slots * sizeof(int));
    status_host_ = (int *)be::pinned(slots * sizeof(int));
    moves_host_ = (int *)be::pinned(2 * slots * sizeof(int));
    // program kernels (one warp per tile): the shared memory of the FMA machine; vector kernels: reduction rows only
    for (int v = 0; v < M_VARIANTS; v++)
    {
        // (the programs of a variant share one machine: its slots are the largest budget among them)
        const int sw_v = std::max(std::max(H_.fw[v].slot_budget, H_.bw[v].slot_budget), std::max(H_.bwp[v].slot_budget, H_.mv[v].slot_budget));
        smem_prog_[v] = machine_smem_doubles(sw_v, variant_groups(v)) * sizeof(double);
        smem_factor_[v] = machine_smem_doubles(P_.fa_budget, variant_groups(v)) * sizeof(double);
    }
    smem_pair_ = machine_smem_doubles(P_.pair_budget, M_PAIR_GROUPS, 2) * sizeof(double);
    // one-warp residual kernel: the parts one after the other in one machine; wide kernels: reduction rows + one machine per
    // warp (the sweeps' machine of warp 0 lies over the same memory: it is idle while the parts run)
    part_doubles_ = machine_smem_doubles(P_.sw_budget, M_PART_GROUPS);
    smem_resid_ = part_doubles_ * sizeof(double);
    smem_wide_ = ((size_t)M_MV_PARTS * KRED * TILE +
                  std::max((size_t)M_MV_PARTS * part_doubles_, std::max(smem_prog_[0], smem_prog_[M_VARIANTS - 1]) / sizeof(double))) *
                 sizeof(double);
    smem_common_ = workers_ > 1 ? (size_t)workers_ * KRED * TILE * sizeof(double) : 0;
#ifndef EICOS_EMU
    {
        if (smem_pair_ > 48 * 1024)
            EI_CUDA(cudaFuncSetAttribute(eicos_solve_kkt_pair, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pair_));
        if (smem_wide_ > 48 * 1024)
        {
            EI_CUDA(cudaFuncSetAttribute(eicos_solve_kkt_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_wide_));
            EI_CUDA(cudaFuncSetAttribute(eicos_residuals_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_wide_));
        }
        if (smem_resid_ > 48 * 1024)
            EI_CUDA(cudaFuncSetAttribute(eicos_residuals, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_resid_));
        const size_t top_f = std::max(smem_factor_[0], smem_factor_[M_VARIANTS - 1]), top_p = std::max(smem_prog_[0], smem_prog_[M_VARIANTS - 1]);
        if (top_f > 48 * 1024)
            EI_CUDA(cudaFuncSetAttribute(eicos_ldl_factor, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)top_f));
        if (top_p > 48 * 1024)
        {
            EI_CUDA(cudaFuncSetAttribute(eicos_solve_kkt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)top_p));
            EI_CUDA(cudaFuncSetAttribute(eicos_residuals, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)top_p));
        }
        int dev_sms = 148;
        EI_CUDA(cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, device_));
        sms_ = dev_sms;
    }
    if (smem_common_ > 48 * 1024)
    {
        const void *ks[] = {(const void *)eicos_load_inputs, (const void *)eicos_equilibrate, (const void *)eicos_init,
                            (const void *)eicos_init_point,
                            (const void *)eicos_iter_head, (const void *)eicos_iter_mid, (const void *)eicos_iter_tail,
                            (const void *)eicos_store_outputs};
        for (const void *k : ks)
            EI_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_common_));
    }
#endif
    be::sync(S_(stream_));
}

Engine::~Engine()
{
    be::set_device(device_);
#ifndef EICOS_EMU
    for (void *e : events_)
        cudaEventDestroy((cudaEvent_t)e);
#endif
    for (void *p : owned_)
        be::dfree(p);
    be::dfree(ws_);
    be::dfree(iws_);
    be::dfree(base_vec_);
    be::dfree(base_mat_);
    be::dfree(active_count_);
    be::dfree(ir_rounds_);
    be::unpin(host_pinned_);
    be::dfree(moves_dev_);
    be::unpin(status_host_);
    be::unpin(moves_host_);
    be::drop_stream(S_(stream_));
}

void Engine::set_matrices(const double *d_G, const double *d_A, const double *base_G, const double *base_A)
{
    if (!pim_)
        throw std::invalid_argument("the handle was not set up for per-instance matrices");
    be::set_device(device_);
    be::stream_t st = S_(stream_);
    mat_dG_ = d_G;
    mat_dA_ = d_A;
    if ((!d_G && nnzG_ && !base_G) || (!d_A && nnzA_ && !base_A))
        throw std::invalid_argument("missing matrix values: neither stacked nor base data given");
    if (base_G)
        be::h2d(base_mat_, base_G, (size_t)nnzG_ * sizeof(double), st);
    if (base_A)
        be::h2d(base_mat_ + nnzG_, base_A, (size_t)nnzA_ * sizeof(double), st);
    be::sync(st);
}

void Engine::debug_line_search(int batch, const double *h_lambda, const double *h_ds, const double *h_dz, const double *h_scalars,
                               double *h_alpha)
{
    be::set_device(device_);
    be::stream_t st = S_(stream_);
    if (batch <= 0 || batch > cap_tiles_ * TILE)
        throw std::invalid_argument("debug_line_search: batch exceeds workspace capacity");
    const size_t zm = (size_t)batch * P_.m;
    double *d = (double *)be::alloc((3 * zm + 5 * (size_t)batch) * sizeof(double));
    be::h2d(d, h_lambda, zm * sizeof(double), st);
    be::h2d(d + zm, h_ds, zm * sizeof(double), st);
    be::h2d(d + 2 * zm, h_dz, zm * sizeof(double), st);
    be::h2d(d + 3 * zm, h_scalars, 4 * (size_t)batch * sizeof(double), st);
    KArgs a;
    std::memset(&a, 0, sizeof(a));
    a.P = P_;
    a.L = L_;
    a.ws = ws_;
    a.iws = iws_;
    a.settings = settings_;
    a.batch = batch;
    a.in_h = d;
    a.in_G = d + zm;
    a.in_A = d + 2 * zm;
    a.in_b = d + 3 * zm;
    a.out_x = d + 3 * zm + 4 * (size_t)batch;
    const int tiles = (batch + TILE - 1) / TILE;
    const int threads = workers_ * (LANES == 1 ? 1 : 32);
    (void)threads;
    EI_LAUNCH(eicos_debug_line_search, tile_debug_line_search, tiles, threads, smem_common_, st, a);
    be::d2h(h_alpha, a.out_x, (size_t)batch * sizeof(double), st);
    be::sync(st);
    be::dfree(d);
}

ProgramStats Engine::program_stats() const
{
    ProgramStats p;
    p.sw_slots = H_.sw_slots;
    p.fa_slots = H_.fa_slots;
    p.fa_fast = 1;
    p.sw_far = H_.sw_far;
    p.sw_direct = 0;
    p.fa_home = H_.fa_home;
    p.fw_loads = H_.fw[0].nld - (int)H_.fw[0].pads;
    p.bw_loads = H_.bw[0].nld - (int)H_.bw[0].pads;
    p.fa_loads = H_.fa[0].nld - (int)H_.fa[0].pads;
    p.mv_loads = H_.mv[0].nld - (int)H_.mv[0].pads;
    return p;
}

void Engine::solve(int batch, const double *d_c, const double *d_h, const double *d_b,
                   const double *base_c, const double *base_h, const double *base_b,
                   double *d_x, double *d_y, double *d_z, double *d_s,
                   int *d_exit, int *d_iter, double *d_info, int *d_iinfo,
                   bool keep_sticky, bool pre_equilibrated, bool timing, SolveStats *stats)
{
    be::set_device(device_);
    be::stream_t st = S_(stream_);
    SolveStats local;
    SolveStats &stt = stats ? *stats : local;
    stt = SolveStats();
    if (batch <= 0)
        return;
    if (keep_sticky && batch > cap_tiles_ * TILE)
        throw std::invalid_argument("keep_sticky needs the whole batch resident");

    KArgs a;
    std::memset(&a, 0, sizeof(a));
    a.P = P_;
    a.L = L_;
    a.ws = ws_;
    a.iws = iws_;
    a.settings = settings_;
    a.in_c = d_c;
    a.in_h = d_h;
    a.in_b = d_b;
    a.base_c = base_vec_;
    a.base_h = base_vec_ + P_.n;
    a.base_b = base_vec_ + P_.n + P_.m;
    if ((!d_c && P_.n && !base_c) || (!d_h && P_.m && !base_h) || (!d_b && P_.p && !base_b))
        throw std::invalid_argument("missing problem vector: neither stacked nor base data given");
    if (base_c)
        be::h2d(base_vec_, base_c, P_.n * sizeof(double), st);
    if (base_h)
        be::h2d(base_vec_ + P_.n, base_h, P_.m * sizeof(double), st);
    if (base_b)
        be::h2d(base_vec_ + P_.n + P_.m, base_b, P_.p * sizeof(double), st);
    be::sync(st); // base_* may be pageable host memory owned by the caller
    a.in_G = mat_dG_;
    a.in_A = mat_dA_;
    a.base_G = base_mat_;
    a.base_A = base_mat_ ? base_mat_ + nnzG_ : nullptr;
    a.out_x = d_x;
    a.out_y = d_y;
    a.out_z = d_z;
    a.out_s = d_s;
    a.out_exit = d_exit;
    a.out_iter = d_iter;
    a.out_info = d_info;
    a.out_iinfo = d_iinfo;
    a.keep_sticky = keep_sticky ? 1 : 0;
    a.pre_equilibrated = pre_equilibrated ? 1 : 0;
    a.active_count = active_count_;
    a.ir_rounds = ir_rounds_;
    a.njobs = 1;
    be::zero(ir_rounds_, 8 * sizeof(unsigned long long), st);

    const int threads = workers_ * (LANES == 1 ? 1 : 32), threads1 = LANES == 1 ? 1 : 32;
    const int threads_wide = M_MV_PARTS * (LANES == 1 ? 1 : 32);
    (void)threads;
    (void)threads1;
    (void)threads_wide;
    a.part_doubles = (int)part_doubles_;

#ifndef EICOS_EMU
    // event pool for per-class device timing
    size_t ev_used = 0;
    auto ev = [&]() -> cudaEvent_t {
        if (ev_used == events_.size())
        {
            cudaEvent_t e;
            EI_CUDA(cudaEventCreate(&e));
            events_.push_back(e);
        }
        return (cudaEvent_t)events_[ev_used++];
    };
    struct Span
    {
        cudaEvent_t a, b;
        int cls;
    };
    std::vector<Span> spans;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    if (timing)
    {
        ev_begin = ev();
        EI_CUDA(cudaEventRecord(ev_begin, st));
    }
#define EI_TIMED(cls_, stmt)                                  \
    do                                                        \
    {                                                         \
        if (timing && (cls_) >= 0)                            \
        {                                                     \
            Span sp_{ev(), ev(), (cls_)};                     \
            EI_CUDA(cudaEventRecord(sp_.a, st));              \
            stmt;                                             \
            EI_CUDA(cudaEventRecord(sp_.b, st));              \
            spans.push_back(sp_);                             \
        }                                                     \
        else                                                  \
        {                                                     \
            stmt;                                             \
        }                                                     \
        stt.launches++;                                       \
    } while (0)
#else
#define EI_TIMED(cls_, stmt) \
    do                       \
    {                        \
        stmt;                \
        stt.launches++;      \
    } while (0)
#endif

    for (long long first = 0; first < batch; first += cap_tiles_ * TILE)
    {
        const int nb = (int)std::min<long long>(batch - first, cap_tiles_ * TILE);
        int tiles = (nb + TILE - 1) / TILE;
        a.batch = nb;
        a.first = (int)first;
        stt.chunks++;

        // ring depth of a launch: deep when its CTAs would leave most of the machine's shared memory idle
        auto pick = [&](int ctas) { a.variant = deep_ring(ctas) ? M_VARIANTS - 1 : 0; };
        auto factor = [&]() {
            pick(tiles);
            EI_TIMED(0, EI_LAUNCH(eicos_ldl_factor, tile_factor, tiles, threads1, smem_factor_[a.variant], st, a));
                    stt.factor_launches++;
            stt.factor_launch_tiles += tiles;
        };
        // solveKKT launches: one job, or the two solves of an iteration that share the factor and do
        // not depend on each other (rhs1 -> sol1 and rhs2 -> sol2), as CTAs (tile, job) of one launch -
        // same traffic when the machine is full, half the latency when it is not
        auto kkt_pair = [&](int init, int nit1, int nit2) {
            a.job[0] = {L_.rhs1, L_.sol1, nit1, 0};
            a.job[1] = {L_.rhs2, L_.sol2, nit2, 1};
            a.njobs = 2;
            a.initialize = init;
            pick(2 * tiles);
            if (pair_solves(tiles))
            { // both solves in one pass over L (one CTA per tile)
                a.njobs = 1;
                EI_TIMED(1, EI_LAUNCH(eicos_solve_kkt_pair, tile_solve_kkt<2>, tiles, threads1, smem_pair_, st, a));
            }
            else if (wide_launch(2 * tiles))
            {
                a.variant = force_variant_ == 0 ? 0 : M_VARIANTS - 1; // (the sweeps of warp 0: deep ring)
                EI_TIMED(1, EI_LAUNCH_JOBS(eicos_solve_kkt_wide, tile_solve_kkt<1>, tiles, 2, threads_wide, smem_wide_, st, a));
            }
            else
                EI_TIMED(1, EI_LAUNCH_JOBS(eicos_solve_kkt, tile_solve_kkt<1>, tiles, 2, threads1, smem_prog_[a.variant], st, a));
            stt.solve_launches++;
            stt.solve_launch_tiles += (long long)tiles * 2;
        };
        auto kkt_rhs2 = [&](int nitrow) {
            a.job[0] = {L_.rhs2, L_.sol2, nitrow, 1};
            a.njobs = 1;
            a.initialize = 0;
            pick(tiles);
            if (wide_launch(tiles))
            {
                a.variant = force_variant_ == 0 ? 0 : M_VARIANTS - 1; // (the sweeps of warp 0: deep ring)
                EI_TIMED(1, EI_LAUNCH_JOBS(eicos_solve_kkt_wide, tile_solve_kkt<1>, tiles, 1, threads_wide, smem_wide_, st, a));
            }
            else
                EI_TIMED(1, EI_LAUNCH_JOBS(eicos_solve_kkt, tile_solve_kkt<1>, tiles, 1, threads1, smem_prog_[a.variant], st, a));
            stt.solve_launches++;
            stt.solve_launch_tiles += tiles;
        };

        EI_TIMED(2, EI_LAUNCH(eicos_load_inputs, tile_load, tiles, threads, smem_common_, st, a));
        if (pim_)
            EI_TIMED(2, EI_LAUNCH(eicos_equilibrate, tile_equil, tiles, threads, smem_common_, st, a));
        EI_TIMED(2, EI_LAUNCH(eicos_init, tile_init, tiles, threads, smem_common_, st, a));
        factor();
        kkt_pair(1, J_NIT1, J_NIT2);
        EI_TIMED(2, EI_LAUNCH(eicos_init_point, tile_init_point, tiles, threads, smem_common_, st, a));

        for (int it = 0; it <= settings_.iter_max + 1; it++)
        {
            be::zero(active_count_, sizeof(unsigned int), st);
            if (wide_launch(tiles))
                EI_TIMED(3, EI_LAUNCH(eicos_residuals_wide, tile_resid, tiles, threads_wide, smem_wide_, st, a));
            else
                EI_TIMED(3, EI_LAUNCH(eicos_residuals, tile_resid, tiles, threads1, smem_resid_, st, a));
            EI_TIMED(4, EI_LAUNCH(eicos_iter_head, tile_head, tiles, threads, smem_common_, st, a));
            stt.resid_launches++, stt.vector_launches++;
            stt.resid_launch_tiles += tiles, stt.vector_launch_tiles += tiles;
            stt.ipm_iterations++;
            be::d2h(host_pinned_, active_count_, sizeof(unsigned int), st);
            be::sync(st);
            const long long nactive = host_pinned_[0];
            if (nactive == 0)
                break;
            // ---- active-set compaction: when enough instances have finished, store their results and
            // pack the survivors into the leading tiles so that later launches cover fewer tiles
            if (compaction_ && !keep_sticky && tiles >= 8 && nactive * 4 <= (long long)tiles * TILE * 3)
            {
                EI_TIMED(2, EI_LAUNCH(eicos_store_outputs, tile_store, tiles, threads, smem_common_, st, a));
                be::d2h_2d(status_host_, TILE * sizeof(int), iws_ + (size_t)J_STATUS * TILE,
                           (size_t)L_.irows_total * TILE * sizeof(int), TILE * sizeof(int), tiles, st);
                be::sync(st);
                const int new_tiles = (int)((nactive + TILE - 1) / TILE);
                int nmoves = 0, hole = 0;
                const int keep = new_tiles * TILE;
                for (int src = keep; src < tiles * TILE; src++)
                {
                    if (status_host_[src] != ST_ACTIVE)
                        continue;
                    while (hole < keep && status_host_[hole] == ST_ACTIVE)
                        hole++;
                    if (hole >= keep)
                        throw std::logic_error("compaction: no free slot");
                    moves_host_[2 * nmoves] = src;
                    moves_host_[2 * nmoves + 1] = hole++;
                    nmoves++;
                }
                if (nmoves > 0)
                {
                    be::h2d(moves_dev_, moves_host_, 2 * (size_t)nmoves * sizeof(int), st);
                    MoveRanges mr;
                    // rows that are live between the head step and the rest of the iteration (everything
                    // else - factor, solutions, work vectors - is recomputed): problem data, iterate and best
                    // iterate (contiguous), residuals, scalings + scaling block (contiguous), both right-hand
                    // sides (contiguous), scalars
                    // (per-instance matrices: also the equilibrated G / A values and the equilibration vectors)
                    const int rr[14] = {L_.chb, P_.N,
                                        L_.w, (L_.bs + P_.mt) - L_.w,
                                        L_.r, P_.N,
                                        L_.lpv, (L_.V + P_.nnzV) - L_.lpv,
                                        L_.rhs1, 2 * P_.N,
                                        L_.sc, S_COUNT,
                                        L_.Gx, L_.sc - L_.Gx};
                    mr.n = 7;
                    for (int k = 0; k < 14; k++)
                        mr.r[k] = rr[k];
#ifndef EICOS_EMU
                    eicos_compact<<<nmoves, 128, 0, st>>>(a, mr, moves_dev_);
#else
                    eicos_compact_emu(a, mr, moves_dev_, nmoves);
#endif
                    stt.launches++;
                    stt.compactions++;
                }
                tiles = new_tiles;
            }
            factor();
            kkt_pair(0, -1, -1);
            EI_TIMED(4, EI_LAUNCH(eicos_iter_mid, tile_mid, tiles, threads, smem_common_, st, a));
            kkt_rhs2(J_NIT3);
            EI_TIMED(4, EI_LAUNCH(eicos_iter_tail, tile_tail, tiles, threads, smem_common_, st, a));
            stt.vector_launches += 2;
            stt.vector_launch_tiles += 2 * (long long)tiles;
        }
        EI_TIMED(2, EI_LAUNCH(eicos_store_outputs, tile_store, tiles, threads, smem_common_, st, a));
    }
    be::d2h(host_pinned_ + 2, ir_rounds_, 8 * sizeof(unsigned long long), st);
#ifndef EICOS_EMU
    if (timing)
    {
        ev_end = ev();
        EI_CUDA(cudaEventRecord(ev_end, st));
    }
    EI_CUDA(cudaGetLastError());
#endif
    be::sync(st);
    std::memcpy(&stt.ir_rounds, host_pinned_ + 2, sizeof(unsigned long long));
    std::memcpy(&stt.lane_rounds, host_pinned_ + 2 + 2 * 6, sizeof(unsigned long long));
    std::memcpy(stt.kkt_phase_cycles, host_pinned_ + 4, 5 * sizeof(unsigned long long));
#ifndef EICOS_EMU
    if (timing)
    {
        float ms = 0;
        EI_CUDA(cudaEventElapsedTime(&ms, ev_begin, ev_end));
        stt.ms_total = ms;
        for (const Span &sp : spans)
        {
            EI_CUDA(cudaEventElapsedTime(&ms, sp.a, sp.b));
            (sp.cls == 0 ? stt.ms_factor : sp.cls == 1 ? stt.ms_solve : stt.ms_other) += ms;
            if (sp.cls == 3)
                stt.ms_resid += ms;
            if (sp.cls == 4)
                stt.ms_vector += ms;
        }
    }
#endif
#undef EI_TIMED
}

void Engine::debug_factor_init(int batch, const double *d_c, const double *d_h, const double *d_b,
                               const double *base_c, const double *base_h, const double *base_b,
                               double *h_Lx, double *h_D, double *h_sol1, double *h_sol2, int *h_nit)
{
    be::set_device(device_);
    be::stream_t st = S_(stream_);
    if (batch > cap_tiles_ * TILE)
        throw std::invalid_argument("debug_factor_init: batch exceeds workspace capacity");
    KArgs a;
    std::memset(&a, 0, sizeof(a));
    a.P = P_;
    a.L = L_;
    a.ws = ws_;
    a.iws = iws_;
    a.settings = settings_;
    a.in_c = d_c;
    a.in_h = d_h;
    a.in_b = d_b;
    a.base_c = base_vec_;
    a.base_h = base_vec_ + P_.n;
    a.base_b = base_vec_ + P_.n + P_.m;
    if (base_c)
        be::h2d(base_vec_, base_c, P_.n * sizeof(double), st);
    if (base_h)
        be::h2d(base_vec_ + P_.n, base_h, P_.m * sizeof(double), st);
    if (base_b)
        be::h2d(base_vec_ + P_.n + P_.m, base_b, P_.p * sizeof(double), st);
    be::sync(st);
    a.batch = batch;
    a.first = 0;
    const int tiles = (batch + TILE - 1) / TILE;
    const int threads = workers_ * (LANES == 1 ? 1 : 32), threads1 = LANES == 1 ? 1 : 32;
    (void)threads;
    (void)threads1;
    a.in_G = mat_dG_;
    a.in_A = mat_dA_;
    a.base_G = base_mat_;
    a.base_A = base_mat_ ? base_mat_ + nnzG_ : nullptr;
    EI_LAUNCH(eicos_load_inputs, tile_load, tiles, threads, smem_common_, st, a);
    if (pim_)
        EI_LAUNCH(eicos_equilibrate, tile_equil, tiles, threads, smem_common_, st, a);
    EI_LAUNCH(eicos_init, tile_init, tiles, threads, smem_common_, st, a);
    a.variant = deep_ring(2 * tiles) ? M_VARIANTS - 1 : 0;
    EI_LAUNCH(eicos_ldl_factor, tile_factor, tiles, threads1, smem_factor_[a.variant], st, a);
    a.initialize = 1;
    a.njobs = 2;
    a.job[0] = {L_.rhs1, L_.sol1, J_NIT1, 0};
    a.job[1] = {L_.rhs2, L_.sol2, J_NIT2, 1};
    if (pair_solves(tiles))
    {
        a.njobs = 1;
        EI_LAUNCH(eicos_solve_kkt_pair, tile_solve_kkt<2>, tiles, threads1, smem_pair_, st, a);
    }
    else
        EI_LAUNCH_JOBS(eicos_solve_kkt, tile_solve_kkt<1>, tiles, 2, threads1, smem_prog_[a.variant], st, a);
    be::sync(st);
    // gather rows back to instance-major host arrays; L comes back in CSC order
    const size_t tile_doubles = (size_t)L_.rows_total * TILE;
    std::vector<double> buf(tile_doubles);
    std::vector<int> ibuf((size_t)L_.irows_total * TILE);
    for (int t = 0; t < tiles; t++)
    {
        be::d2h(buf.data(), ws_ + t * tile_doubles, tile_doubles * sizeof(double), st);
        be::d2h(ibuf.data(), iws_ + (size_t)t * L_.irows_total * TILE, ibuf.size() * sizeof(int), st);
        be::sync(st);
        for (int lane = 0; lane < TILE; lane++)
        {
            const long long inst = (long long)t * TILE + lane;
            if (inst >= batch)
                break;
            auto grab = [&](double *dst, int row0, int rows) {
                if (dst)
                    for (int r = 0; r < rows; r++)
                        dst[inst * rows + r] = buf[(size_t)(row0 + r) * TILE + lane];
            };
            if (h_Lx)
                for (int u = 0; u < P_.nnzL; u++)
                    h_Lx[inst * P_.nnzL + u] = buf[(size_t)(L_.Lx + u) * TILE + lane];
            if (h_D) // the factorisation keeps 1 / D only (what the sweeps read)
                for (int r = 0; r < P_.N; r++)
                    h_D[inst * P_.N + r] = 1.0 / buf[(size_t)(L_.Dinv + r) * TILE + lane];
            grab(h_sol1, L_.sol1, P_.N);
            grab(h_sol2, L_.sol2, P_.N);
            if (h_nit)
            {
                h_nit[inst * 2 + 0] = ibuf[(size_t)J_NIT1 * TILE + lane];
                h_nit[inst * 2 + 1] = ibuf[(size_t)J_NIT2 * TILE + lane];
            }
        }
    }
}

} // namespace eicos
