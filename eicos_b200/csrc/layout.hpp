// Device-side views of the shared (per-pattern) index data and of the per-instance workspace.
//
// HBM layout ("tiled structure of arrays", batch innermost):
//   an instance belongs to tile t = b / TILE and lane = b % TILE.  Every per-instance array is a run
//   of ROWS; row r of tile t is the TILE consecutive doubles  ws[(t*rows_total + r)*TILE + lane].
//   A warp that walks rows therefore issues one fully coalesced 256-byte access per row whatever the
//   row index is, and all rows of one tile are contiguous (column slices of L are contiguous runs).
//   Index data (instruction streams, see streams.hpp) is shared by the whole batch.
//
// Index spaces: "KKT space" = [x (n) | y (p) | z expanded (mt = m + 2 nc)], the row order of the
// reference's KKT matrix (src/eicos.cpp:1776-1819): every second-order cone of dimension d owns d
// rows followed by 2 expansion slots.  ALL z-shaped vectors (z, s, lambda, h, rz, ...) use the
// expanded index here, with the slot rows held at zero, so that one gather index serves the
// iterate, the residuals and the KKT-space solution vectors alike.
#pragma once

#include <cstddef>

namespace eicos
{

// per-instance status while the interior-point loop is running
enum : int
{
    ST_ACTIVE = -1000,
    EXIT_OPTIMAL = 0,
    EXIT_PINF = 1,
    EXIT_DINF = 2,
    EXIT_MAXIT = -1,
    EXIT_NUMERICS = -2,
    EXIT_OUTCONE = -3,
    EXIT_FATAL = -7,
    EXIT_INACC = 10,
    EXIT_NOT_CONVERGED = -87
}; // include/eicos.hpp:8-21 of the reference

// scalar rows (doubles), one row each
enum ScalarRow : int
{
    S_KAP, S_TAU, S_CX, S_BY, S_HZ, // Work scalars (include/eicos.hpp:107-111)
    S_PCOST, S_DCOST, S_PRES, S_DRES, S_PINFRES, S_DINFRES, S_GAP, S_RELGAP,
    S_SIGMA, S_MU, S_STEP, S_STEP_AFF, S_KAPOVERT, // Information doubles (:51-65)
    S_WORK_END,
    S_BEST = S_WORK_END,                 // same 18 rows again for w_best
    S_BEST_END = S_BEST + S_WORK_END,
    S_RT = S_BEST_END, S_NX, S_NY, S_NZ, S_NS, S_HRESX, S_HRESY, S_HRESZ,
    S_RESX0, S_RESY0, S_RESZ0, S_PRES_PREV,
    S_DTAU_DENOM, S_DTAUAFF, S_DKAPAFF,
    S_RHSMAX1, S_RHSMAX2,  // max |rhs1|, max |rhs2|: kept by the kernels that write the right-hand sides (solveKKT's stopping threshold)
    S_RED,                 // the 14 sums of computeResiduals, handed from eicos_residuals to eicos_iter_head
    S_COUNT = S_RED + 14
};

// integer rows
enum IntRow : int
{
    J_ITER, J_PINF, J_DINF, J_HAS_PINFRES, J_HAS_DINFRES, J_HAS_RELGAP, J_NIT1, J_NIT2, J_NIT3, // Information ints
    J_WORK_END,
    J_BEST = J_WORK_END,
    J_BEST_END = J_BEST + J_WORK_END,
    J_STATUS = J_BEST_END, // ST_ACTIVE or the exit code
    J_INST,                // index of the instance inside the device batch (-1: padding / vacated slot)
    J_STORED,              // results already written to the output buffers
    J_COUNT
};

// Row offsets of every per-instance array inside a tile's workspace block.
struct Layout
{
    int chb;                        // [c | b | h] equilibrated problem vectors, KKT-shaped (N rows)
    int w;                          // current iterate [x | y | z] (N rows)
    int s, lam;                     // slacks, scaled variable (mt rows each)
    int wb, bs;                     // best iterate (w_best; lambda is not kept: an instance that restores it stops)
    int r;                          // residuals [rx | ry | rz] (N rows)
    int lpv, lpw;                   // LP cone scalings (l rows each)
    int cpar, cq;                   // SOC scalings: CP_COUNT rows per cone, q vectors
    int V;                          // scaling block values of the KKT matrix (cacheIndices order)
    int Lx, D, Dinv;                // factor: L column-major (CSC order of the symbolic pattern), pivots, reciprocals
    int rhs1, rhs2, sol1, sol2;     // KKT-space vectors (N rows)
    int xw, dxr, e;                 // triangular-solve work vector, refinement step, residual (N rows)
    int xw2, dxr2, e2;              // the same for the second of two concurrent solves (job set 1)
    int dsw, wdz, dsaff, ds1;       // dsaff_by_W, W_times_dzaff, dsaff, scratch (mt rows)
    int Gx, Ax, eq;                 // per-instance-matrices mode: equilibrated G / A values (CSC order), and the
                                    // equilibration vectors KKT-shaped [x_equil | A_equil | G_equil expanded] (N rows)
    int sc;                         // S_COUNT scalar rows
    int acc;                        // home rows of the factorisation's accumulators (nnzL rows), or -1: they live in slots only
    int rows_total;
    int irows_total;                // integer rows (J_COUNT)
};

// one program of the FMA machine on the device (machine.hpp: MachineCode)
struct DevMachine
{
    const int *ops;
    int nchunks;     // 1 KB chunks of the record stream
    int nld_chunks;  // 1 KB chunks of its load lists
    int ring_groups; // depth of the data ring it was compiled for
    int ring_row0;   // shared-memory row the ring starts at
};

enum ConeParam : int
{
    CP_ETA, CP_ETA2, CP_A, CP_D1, CP_U0, CP_U1, CP_V1, CP_W, CP_COUNT
};

// Shared index data on the device (all pointers are device pointers).
struct DevPattern
{
    int n, p, m, l, nc, N, mt, qtot, nnzL, nnzV, maxcol;
    const int *cone_dim, *cone_k, *cone_q; // per cone: dimension, first expanded index, first q row
    const int *zk;                         // compact z index -> expanded index (load / store only)
    const double *xeq, *Aeq, *GeqE;        // equilibration vectors (GeqE is expanded, 1 in the slots)
    // Machine programs (machine.hpp, streams.cpp) and their load lists, materialised per use (absolute rows
    // of the tile): a job set is (rhs1, sol1) with work vectors xw / dxr / e (set 0) or (rhs2, sol2) with
    // xw2 / dxr2 / e2 (set 1); [set][first solve | refinement round].  The backward sweep of a first solve
    // runs the plain program bwp, a refinement round the accumulating program bw.
    // Every program exists for two depths of the data ring (first index; streams.hpp: M_VARIANT_GROUPS).
    DevMachine fw[2], bw[2], bwp[2], mv[2];
    const int *fw_ld[2][2][2], *bw_ld[2][2][2], *mv_ld[2][2];
    // computeResiduals, and the refinement residual once more, in 4 independent parts (streams.hpp: M_MV_PARTS)
    DevMachine rs[4], mvw[4];
    const int *rs_ld[4], *mvw_ld[2][4]; // mvw_ld: [set][part]
    // two-job programs (both job sets in one pass, shallow ring): [first solve | refinement round]
    DevMachine fw2, bw2, bwp2, mv2;
    const int *fw2_ld[2], *bw2_ld[2], *mv2_ld;
    int mv_rows;
    int sw_budget, fa_budget, pair_budget; // slots of the solveKKT / residual programs, the factor program, the two-job programs
    // factor program (absolute rows: its load list needs no materialisation)
    DevMachine fa[2];
    const int *fa_ld[2];
    // per-instance-matrices mode (every instance has its own G / A values): 1, and the index arrays
    // the on-device equilibration walks (CSC of G and A, their CSR views as row pointer + value index)
    int pim, nnzG, nnzA;
    const int *Gp, *Gi, *Ap, *Ai, *Grp, *Grv, *Arp, *Arv, *cone_z;
    const int *Vkind; // per V entry: what resetKKTScalings writes (0 -> -1, 1 -> 0, 2 -> +1)
};

} // namespace eicos
