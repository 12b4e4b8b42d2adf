// eicos.hpp - C++ facade over the C ABI (eicos_b200.h): the public interface of EmbersArc/EiCOS
// (reference include/eicos.hpp:5-21 exitcode, :23-47 Settings, :49-73 Information, :137-163 Solver)
// with the B200 engine behind it, plus the batched overload for many instances of one sparsity
// pattern.  Header-only; link against libeicos_b200.so.  There is no CPU implementation behind this
// header: constructors throw std::runtime_error when the engine cannot be created (no CUDA device,
// out of memory, malformed pattern).
//
// Differences a user of the reference will notice:
//  * solution() returns a pointer-backed view (VectorView) instead of `const Eigen::VectorXd &`;
//    with Eigen present (EICOS_B200_WITH_EIGEN, set automatically when <Eigen/Sparse> is found) the
//    Eigen-typed constructor / updateData exist and VectorView converts to Eigen::Map.
//  * Settings can be changed: getSettings().feastol = 1e-6 takes effect at the next solve().  The reference
//    declares every numeric field `const` (include/eicos.hpp:25-46); here the tolerances, nitref, iter_max and
//    the step and centering controls are writable and checked when solve() hands them to the engine (an
//    out-of-range value throws std::runtime_error naming the field).  deltastat and equil_iters stay `const`:
//    they are baked into a handle at setup.  delta, eps and maxit are not read (the reference does not read them
//    either); `verbose` is accepted and ignored (printing is out of scope).
//  * getInfo() carries the scalar fields of Information; the iterate vectors are reached through
//    solution() / duals().
#pragma once

#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "eicos_b200.h"

#if !defined(EICOS_B200_WITH_EIGEN) && defined(__has_include)
#if __has_include(<Eigen/Sparse>)
#define EICOS_B200_WITH_EIGEN 1
#endif
#endif
#ifdef EICOS_B200_WITH_EIGEN
#include <Eigen/Sparse>
#endif

namespace EiCOS
{

// reference include/eicos.hpp:8-21
enum class exitcode
{
    optimal = 0,
    primal_infeasible = 1,
    dual_infeasible = 2,
    maxit = -1,
    numerics = -2,
    outcone = -3,
    fatal = -7,
    close_to_optimal = 10,
    close_to_primal_infeasible = 11,
    close_to_dual_infeasible = 12,
    not_converged_yet = -87
};

// reference include/eicos.hpp:23-47, same defaults.  The writable fields go to the engine before every solve
// (eicos_settings); the const ones are fixed at setup (deltastat, equil_iters) or unused (delta, eps, maxit).
struct Settings
{
    double gamma = 0.99;
    const double delta = 2e-7;
    const double deltastat = 7e-8;
    const double eps = 1e13;
    double feastol = 1e-8;
    double abstol = 1e-8;
    double reltol = 1e-8;
    double feastol_inacc = 1e-4;
    double abstol_inacc = 5e-5;
    double reltol_inacc = 5e-5;
    size_t nitref = 9;
    const size_t maxit = 100;
    bool verbose = false;
    double linsysacc = 1e-14;
    double irerrfact = 6;
    double stepmin = 1e-6;
    double stepmax = 0.999;
    double sigmamin = 1e-4;
    double sigmamax = 1.;
    const size_t equil_iters = 3;
    size_t iter_max = 100;
    size_t safeguard = 500;

    // the engine's form (values past INT_MAX saturate, so that the range check rejects them)
    eicos_settings to_c() const
    {
        const auto narrow = [](size_t v) { return v > 0x7fffffff ? 0x7fffffff : (int)v; };
        eicos_settings o;
        o.feastol = feastol, o.abstol = abstol, o.reltol = reltol;
        o.feastol_inacc = feastol_inacc, o.abstol_inacc = abstol_inacc, o.reltol_inacc = reltol_inacc;
        o.linsysacc = linsysacc, o.irerrfact = irerrfact;
        o.gamma = gamma, o.stepmin = stepmin, o.stepmax = stepmax;
        o.sigmamin = sigmamin, o.sigmamax = sigmamax;
        o.safeguard = (double)safeguard;
        o.nitref = narrow(nitref), o.iter_max = narrow(iter_max);
        return o;
    }
};

// reference include/eicos.hpp:49-73
struct Information
{
    double pcost = 0, dcost = 0, pres = 0, dres = 0;
    bool pinf = false, dinf = false;
    std::optional<double> pinfres, dinfres;
    double gap = 0;
    std::optional<double> relgap;
    double sigma = 0, mu = 0, step = 0, step_aff = 0, kapovert = 0;
    size_t iter = 0, iter_max = 0, nitref1 = 0, nitref2 = 0, nitref3 = 0;

    static Information from(const eicos_info &i)
    {
        Information o;
        o.pcost = i.pcost, o.dcost = i.dcost, o.pres = i.pres, o.dres = i.dres;
        o.pinf = i.pinf != 0, o.dinf = i.dinf != 0;
        if (i.has_pinfres)
            o.pinfres = i.pinfres;
        if (i.has_dinfres)
            o.dinfres = i.dinfres;
        o.gap = i.gap;
        if (i.has_relgap)
            o.relgap = i.relgap;
        o.sigma = i.sigma, o.mu = i.mu, o.step = i.step, o.step_aff = i.step_aff, o.kapovert = i.kapovert;
        o.iter = (size_t)i.iter, o.iter_max = (size_t)i.iter_max;
        o.nitref1 = (size_t)i.nitref1, o.nitref2 = (size_t)i.nitref2, o.nitref3 = (size_t)i.nitref3;
        return o;
    }
};

// A read-only vector owned by the solver (valid until the next solve / updateData / destruction).
struct VectorView
{
    const double *ptr = nullptr;
    size_t len = 0;
    const double *data() const { return ptr; }
    size_t size() const { return len; }
    double operator[](size_t i) const { return ptr[i]; }
    double operator()(size_t i) const { return ptr[i]; }
    const double *begin() const { return ptr; }
    const double *end() const { return ptr + len; }
#ifdef EICOS_B200_WITH_EIGEN
    operator Eigen::Map<const Eigen::VectorXd>() const { return {ptr, (Eigen::Index)len}; }
#endif
};

namespace detail
{
inline void check(int rc, const char *what)
{
    if (rc < 0)
        throw std::runtime_error(std::string(what) + ": " + eicos_last_error());
}
} // namespace detail

// reference include/eicos.hpp:137-163
class Solver
{
  public:
    // traditional interface (reference include/eicos.hpp:151-154)
    Solver(int n, int m, int p, int l, int ncones, int *q,
           double *Gpr, int *Gjc, int *Gir,
           double *Apr, int *Ajc, int *Air,
           double *c, double *h, double *b, int device = 0)
        : n_(n), m_(m), p_(p)
    {
        h_ = eicos_setup(n, m, p, l, ncones, q, Gpr, Gjc, Gir, Apr, Ajc, Air, c, h, b, device);
        if (!h_)
            throw std::runtime_error(std::string("EiCOS::Solver: ") + eicos_last_error());
    }
    // reference include/eicos.hpp:155-156 (NULL = keep; h follows Gpr, b follows Apr, src/eicos.cpp:2053-2082)
    void updateData(double *Gpr, double *Apr, double *c, double *h, double *b)
    {
        detail::check(eicos_update_data(h_, Gpr, Apr, c, h, b), "EiCOS::Solver::updateData");
    }

#ifdef EICOS_B200_WITH_EIGEN
    // reference include/eicos.hpp:138-143; G and A must be compressed column-major (they are in the reference too)
    Solver(const Eigen::SparseMatrix<double> &G, const Eigen::SparseMatrix<double> &A,
           const Eigen::VectorXd &c, const Eigen::VectorXd &h, const Eigen::VectorXd &b,
           const Eigen::VectorXi &soc_dims, int device = 0)
        : n_((int)c.size()), m_((int)h.size()), p_((int)b.size())
    {
        if (!G.isCompressed() || !A.isCompressed())
            throw std::invalid_argument("EiCOS::Solver: G and A must be compressed");
        h_ = eicos_setup(n_, m_, p_, m_ - (int)soc_dims.sum(), (int)soc_dims.size(), soc_dims.data(),
                         G.valuePtr(), G.outerIndexPtr(), G.innerIndexPtr(),
                         A.valuePtr(), A.outerIndexPtr(), A.innerIndexPtr(),
                         c.data(), h.data(), b.data(), device);
        if (!h_)
            throw std::runtime_error(std::string("EiCOS::Solver: ") + eicos_last_error());
    }
    // reference include/eicos.hpp:144-148 (same pattern, new values; src/eicos.cpp:2032-2051)
    void updateData(const Eigen::SparseMatrix<double> &G, const Eigen::SparseMatrix<double> &A,
                    const Eigen::VectorXd &c, const Eigen::VectorXd &h, const Eigen::VectorXd &b)
    {
        detail::check(eicos_update_data_full(h_, G.valuePtr(), A.valuePtr(), c.data(), h.data(), b.data()),
                      "EiCOS::Solver::updateData");
    }
#endif
    // the value arrays of the Eigen overload without Eigen: all five required (src/eicos.cpp:2032-2051)
    void updateDataFull(const double *Gpr, const double *Apr, const double *c, const double *h, const double *b)
    {
        detail::check(eicos_update_data_full(h_, Gpr, Apr, c, h, b), "EiCOS::Solver::updateData");
    }

    ~Solver() { eicos_cleanup(h_); }
    Solver(const Solver &) = delete;
    Solver &operator=(const Solver &) = delete;
    Solver(Solver &&o) noexcept : h_(o.h_), n_(o.n_), m_(o.m_), p_(o.p_), settings_(o.settings_) { o.h_ = nullptr; }

    // reference include/eicos.hpp:158; runs with the current getSettings()
    exitcode solve(bool verbose = false)
    {
        (void)verbose;
        const eicos_settings st = settings_.to_c();
        detail::check(eicos_set_settings(h_, &st), "EiCOS::Solver::solve");
        const int rc = eicos_solve(h_);
        if (rc <= EICOS_ERR_INVALID)
            throw std::runtime_error(std::string("EiCOS::Solver::solve: ") + eicos_last_error());
        eicos_info i;
        if (eicos_get_info(h_, &i) == 0)
            info_ = Information::from(i);
        return static_cast<exitcode>(rc);
    }

    // reference include/eicos.hpp:160
    VectorView solution() const { return {eicos_solution(h_), (size_t)n_}; }

    // y, z, s of the reference's private `w` (include/eicos.hpp:176)
    void duals(std::vector<double> &y, std::vector<double> &z, std::vector<double> &s) const
    {
        y.assign((size_t)p_, 0.0), z.assign((size_t)m_, 0.0), s.assign((size_t)m_, 0.0);
        detail::check(eicos_get_duals(h_, y.data(), z.data(), s.data()), "EiCOS::Solver::duals");
    }

    Settings &getSettings() { return settings_; }           // include/eicos.hpp:162
    const Information &getInfo() const { return info_; }     // include/eicos.hpp:163
    eicos_solver *handle() const { return h_; }

  private:
    eicos_solver *h_ = nullptr;
    int n_ = 0, m_ = 0, p_ = 0;
    Settings settings_;
    Information info_;
};

// The batched overload (BASELINE.json north_star): one pattern, `batch` instances, stacked
// instance-major data.  What the reference does with one Solver and updateData + solve per instance
// (src/run.cpp:34-49).  Every instance is solved as a fresh Solver would (no sticky state).
class BatchSolver
{
  public:
    struct Result
    {
        int batch = 0, n = 0, m = 0, p = 0;
        std::vector<double> x, y, z, s; // [batch x n], [batch x p], [batch x m], [batch x m]
        std::vector<int> exitflag;      // exitcode values
        std::vector<eicos_info> info;
        exitcode code(int b) const { return static_cast<exitcode>(exitflag[(size_t)b]); }
        VectorView solution(int b) const { return {x.data() + (size_t)b * n, (size_t)n}; }
    };

    // instance_matrices: instances may bring their own G / A values (solve(..., Gs, As)); they are
    // equilibrated per instance on the device (setEquilibration, src/eicos.cpp:302-374).
    BatchSolver(int n, int m, int p, int l, int ncones, const int *q,
                const double *Gpr, const int *Gjc, const int *Gir,
                const double *Apr, const int *Ajc, const int *Air,
                const double *c, const double *h, const double *b,
                bool instance_matrices = false, int device = 0, long long capacity = 0, int workers = 0)
        : n_(n), m_(m), p_(p), nnzG_(Gjc ? Gjc[n] : 0), nnzA_(Ajc ? Ajc[n] : 0)
    {
        h_ = eicos_batch_setup_ex(n, m, p, l, ncones, q, Gpr, Gjc, Gir, Apr, Ajc, Air, c, h, b, device, capacity, workers,
                                  instance_matrices ? EICOS_BATCH_INSTANCE_MATRICES : 0);
        if (!h_)
            throw std::runtime_error(std::string("EiCOS::BatchSolver: ") + eicos_last_error());
    }
    // several GPUs of one node: the batch is cut into contiguous slices, one per entry of `devices` (eicos_multi_*:
    // one device handle and one host thread per slice, results gathered into the Result; no collective)
    BatchSolver(int n, int m, int p, int l, int ncones, const int *q,
                const double *Gpr, const int *Gjc, const int *Gir,
                const double *Apr, const int *Ajc, const int *Air,
                const double *c, const double *h, const double *b,
                const std::vector<int> &devices, bool instance_matrices = false, long long capacity = 0, int workers = 0)
        : n_(n), m_(m), p_(p), nnzG_(Gjc ? Gjc[n] : 0), nnzA_(Ajc ? Ajc[n] : 0)
    {
        mh_ = eicos_multi_setup(n, m, p, l, ncones, q, Gpr, Gjc, Gir, Apr, Ajc, Air, c, h, b, (int)devices.size(), devices.data(),
                                capacity, workers, instance_matrices ? EICOS_BATCH_INSTANCE_MATRICES : 0);
        if (!mh_)
            throw std::runtime_error(std::string("EiCOS::BatchSolver: ") + eicos_last_error());
    }
    ~BatchSolver()
    {
        eicos_batch_cleanup(h_);
        eicos_multi_cleanup(mh_);
    }
    BatchSolver(const BatchSolver &) = delete;
    BatchSolver &operator=(const BatchSolver &) = delete;

    // new matrix values shared by every instance (updateData with Gpr / Apr, src/eicos.cpp:2076-2081)
    void updateMatrices(const double *Gpr, const double *Apr)
    {
        if (mh_)
            throw std::runtime_error("EiCOS::BatchSolver::updateMatrices: not available on a multi-device solver");
        detail::check(eicos_batch_update_matrices(h_, Gpr, Apr), "EiCOS::BatchSolver::updateMatrices");
    }

    // cs [batch x n], hs [batch x m], bs [batch x p], Gs [batch x nnzG], As [batch x nnzA]; NULL = the setup data
    Result solve(int batch, const double *cs, const double *hs, const double *bs,
                 const double *Gs = nullptr, const double *As = nullptr, bool want_duals = true, bool want_info = true)
    {
        Result r;
        r.batch = batch, r.n = n_, r.m = m_, r.p = p_;
        const size_t B = (size_t)batch;
        r.x.assign(B * n_, 0.0);
        if (want_duals)
            r.y.assign(B * p_, 0.0), r.z.assign(B * m_, 0.0), r.s.assign(B * m_, 0.0);
        r.exitflag.assign(B, (int)exitcode::not_converged_yet);
        if (want_info)
            r.info.resize(B);
        double *y = want_duals ? r.y.data() : nullptr, *z = want_duals ? r.z.data() : nullptr, *s = want_duals ? r.s.data() : nullptr;
        eicos_info *info = want_info ? r.info.data() : nullptr;
        const eicos_settings st = settings_.to_c();
        detail::check(mh_ ? eicos_multi_set_settings(mh_, &st) : eicos_batch_set_settings(h_, &st), "EiCOS::BatchSolver::solve");
        detail::check(mh_ ? eicos_multi_solve(mh_, batch, Gs, As, cs, hs, bs, r.x.data(), y, z, s, r.exitflag.data(), info)
                          : eicos_batch_solve_matrices(h_, batch, Gs, As, cs, hs, bs, r.x.data(), y, z, s, r.exitflag.data(), info),
                      "EiCOS::BatchSolver::solve");
        return r;
    }

    // settings of every instance of the next solve() (reference include/eicos.hpp:162)
    Settings &getSettings() { return settings_; }
    int nnzG() const { return nnzG_; }
    int nnzA() const { return nnzA_; }
    eicos_batch *handle() const { return h_; }
    int devices() const { return mh_ ? eicos_multi_ngpu(mh_) : 1; }

  private:
    eicos_batch *h_ = nullptr;
    eicos_multi *mh_ = nullptr; // set instead of h_ by the multi-device constructor
    int n_ = 0, m_ = 0, p_ = 0, nnzG_ = 0, nnzA_ = 0;
    Settings settings_;
};

} // namespace EiCOS
