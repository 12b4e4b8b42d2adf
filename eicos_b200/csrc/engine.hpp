// Batched interior-point engine for one device: owns the shared pattern data, the per-instance
// workspace (tiled SoA, see layout.hpp) and the launch sequence of Solver::solve
// (reference src/eicos.cpp:848-1262).
#pragma once

#include "layout.hpp"
#include "streams.hpp"
#include "symbolic.hpp"

#include <cstddef>
#include <vector>

namespace eicos
{

struct SolveStats
{
    int chunks = 0, compactions = 0;
    int ipm_iterations = 0;          // head launches over all chunks
    long long launches = 0;          // kernels launched
    unsigned long long ir_rounds = 0; // triangular-solve rounds executed (tile-rounds, all solveKKT calls)
    unsigned long long kkt_phase_cycles[5] = {0, 0, 0, 0, 0}; // norm, forward, backward, residual, bookkeeping (summed over tiles)
    double ms_total = 0, ms_factor = 0, ms_solve = 0, ms_other = 0; // device time by kernel class (CUDA events)
    long long factor_launch_tiles = 0, solve_launch_tiles = 0;      // tiles covered by the timed launches
    int factor_launches = 0, solve_launches = 0;
    double ms_resid = 0, ms_vector = 0; // part of ms_other: eicos_residuals / the three per-iteration vector kernels
    long long resid_launch_tiles = 0, vector_launch_tiles = 0;
    int resid_launches = 0, vector_launches = 0;
    unsigned long long lane_rounds = 0; // solve rounds the instances needed themselves (ir_rounds counts whole tiles)

    SolveStats &operator+=(const SolveStats &o)
    { // a batch solved in several segments (capi.cu)
        chunks += o.chunks, compactions += o.compactions, ipm_iterations += o.ipm_iterations;
        launches += o.launches, ir_rounds += o.ir_rounds;
        for (int k = 0; k < 5; k++)
            kkt_phase_cycles[k] += o.kkt_phase_cycles[k];
        ms_total += o.ms_total, ms_factor += o.ms_factor, ms_solve += o.ms_solve, ms_other += o.ms_other;
        factor_launch_tiles += o.factor_launch_tiles, solve_launch_tiles += o.solve_launch_tiles;
        factor_launches += o.factor_launches, solve_launches += o.solve_launches;
        ms_resid += o.ms_resid, ms_vector += o.ms_vector;
        resid_launch_tiles += o.resid_launch_tiles, vector_launch_tiles += o.vector_launch_tiles;
        resid_launches += o.resid_launches, vector_launches += o.vector_launches;
        lane_rounds += o.lane_rounds;
        return *this;
    }
};

// what the program compiler (streams.cpp) produced for this pattern
struct ProgramStats
{
    int sw_slots = 0, fa_slots = 0, fa_fast = 0; // fa_fast: the factorisation is a machine program (always 1)
    long long sw_far = 0, sw_direct = 0, fa_home = 0; // operands served by far gathers / direct loads / home rows
    int fw_loads = 0, bw_loads = 0, fa_loads = 0, mv_loads = 0; // rows each program reads from HBM per run
};

class Engine
{
  public:
    // capacity_instances: how many instances the workspace holds at once (larger batches are
    // processed in chunks); workers: warps per CTA.
    // instance_matrices: every instance brings its own G / A values (same pattern); they are
    // equilibrated on the device and the programs read them as rows of the workspace.
    Engine(const Symbolic &S, int device, long long capacity_instances, int workers, bool instance_matrices = false);
    ~Engine();
    Engine(const Engine &) = delete;
    Engine &operator=(const Engine &) = delete;

    // per-instance-matrices mode: the matrices of the NEXT solve().  d_G / d_A: instance-major DEVICE
    // arrays of raw values [batch x nnzG], [batch x nnzA], or null to use base_G / base_A (host arrays
    // of raw values shared by all instances).
    void set_matrices(const double *d_G, const double *d_A, const double *base_G, const double *base_A);
    bool instance_matrices() const { return pim_; }

    // re-upload the shared numeric values after refresh_values() (updateData with new G/A)
    void upload_values(const Symbolic &S);

    // Solve `batch` instances.  d_c/d_h/d_b: instance-major DEVICE arrays of raw (unequilibrated)
    // data, or null to use base_* (host arrays, shared by all instances).  Outputs are DEVICE
    // arrays (instance-major), any may be null.  Blocks until the results are complete.
    void solve(int batch, const double *d_c, const double *d_h, const double *d_b,
               const double *base_c, const double *base_h, const double *base_b,
               double *d_x, double *d_y, double *d_z, double *d_s,
               int *d_exit, int *d_iter, double *d_info, int *d_iinfo,
               bool keep_sticky, bool pre_equilibrated, bool timing, SolveStats *stats);

    // debug entry points (GPU unit tests): run the initial factorisation / one KKT solve for
    // instance-major data and copy raw factor values back (host pointers, may be null)
    void debug_factor_init(int batch, const double *d_c, const double *d_h, const double *d_b,
                           const double *base_c, const double *base_h, const double *base_b,
                           double *h_Lx, double *h_D, double *h_sol1, double *h_sol2, int *h_nit);

    // lineSearch (src/eicos.cpp:1380-1469) on caller data: lambda, ds, dz instance-major in compact z order [batch x m],
    // scalars = tau, dtau, kap, dkap per instance [batch x 4]; all host pointers
    void debug_line_search(int batch, const double *h_lambda, const double *h_ds, const double *h_dz, const double *h_scalars,
                           double *h_alpha);

    ProgramStats program_stats() const;
    void *stream() const { return stream_; }
    int device() const { return device_; }
    int workers() const { return workers_; }
    void set_compaction(bool on) { compaction_ = on; }
    // solver settings of every later solve (tolerances, iteration limit, refinement, step control); the caller
    // validates them (capi.cu)
    void set_settings(const KSettings &k) { settings_ = k; }
    const KSettings &settings() const { return settings_; }
    long long capacity() const { return cap_tiles_ * (long long)tile_width(); }
    size_t workspace_bytes() const { return ws_bytes_; }
    const Layout &layout() const { return L_; }
    static int tile_width();

  private:
    void build_layout(const Symbolic &S, bool acc_rows);
    void upload_pattern(const Symbolic &S);

    int device_ = 0, workers_ = 4;
    bool pim_ = false;
    const double *mat_dG_ = nullptr, *mat_dA_ = nullptr; // matrices of the next solve (pim)
    double *base_mat_ = nullptr;                         // device copy of the shared raw G | A values (pim)
    int nnzG_ = 0, nnzA_ = 0;
    long long cap_tiles_ = 0;
    size_t ws_bytes_ = 0;
    void *stream_ = nullptr;
    Layout L_{};
    DevPattern P_{};
    double *ws_ = nullptr;
    int *iws_ = nullptr;
    double *base_vec_ = nullptr; // device copy of base c|h|b
    unsigned int *active_count_ = nullptr;
    unsigned long long *ir_rounds_ = nullptr;
    unsigned int *host_pinned_ = nullptr;
    int *moves_dev_ = nullptr, *status_host_ = nullptr, *moves_host_ = nullptr; // active-set compaction
    bool compaction_ = true;
    size_t smem_factor_[M_VARIANTS] = {0, 0}, smem_common_ = 0, smem_prog_[M_VARIANTS] = {0, 0}; // factor kernel / vector kernels / solveKKT + residual kernels (per ring variant)
    size_t smem_pair_ = 0; // two-job solveKKT kernel
    size_t smem_resid_ = 0, smem_wide_ = 0, part_doubles_ = 0; // one-warp residual kernel; wide kernels; one part machine (doubles)
    int force_wide_ = -1;
    KSettings settings_ = default_settings();
    bool wide_launch(int ctas) const;
    int sms_ = 148, force_variant_ = -1, force_pair_ = -1;
    bool deep_ring(int ctas) const;
    bool pair_solves(int tiles) const;
    std::vector<void *> owned_; // device allocations holding pattern data
    // positions of value arrays that upload_values() rewrites
    double *dxeq_ = nullptr, *dAeq_ = nullptr, *dGeq_ = nullptr;
    int *dmv_ops_[M_VARIANTS] = {nullptr, nullptr}, *drs_ops_[M_MV_PARTS] = {nullptr, nullptr, nullptr, nullptr}, *dmvw_ops_[M_MV_PARTS] = {nullptr, nullptr, nullptr, nullptr}, *dfa_ops_[M_VARIANTS] = {nullptr, nullptr}, *dmv2_ops_ = nullptr;
    HostStreams H_;        // host copy of the instruction streams (value streams are rebuilt on updateData)
    std::vector<int> Lp_;  // column pointers of L (debug extraction)
    std::vector<void *> events_;
};

} // namespace eicos
