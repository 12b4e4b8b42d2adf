// C ABI (include/eicos_b200.h) over the engine.  Host logic that mirrors the reference's
// Solver object: data ownership, updateData semantics, Information.
#include "../../include/eicos_b200.h"
#include "backend.hpp"
#include "engine.hpp"
#include "symbolic.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <thread>
#include <string>
#include <vector>

using namespace eicos;

namespace
{
thread_local std::string g_error;

int fail(int code, const std::string &msg)
{
    g_error = msg;
    return code;
}

void info_from_rows(const double *d, const int *i, int iter_max, eicos_info *o)
{
    o->pcost = d[S_PCOST];
    o->dcost = d[S_DCOST];
    o->pres = d[S_PRES];
    o->dres = d[S_DRES];
    o->pinfres = d[S_PINFRES];
    o->dinfres = d[S_DINFRES];
    o->gap = d[S_GAP];
    o->relgap = d[S_RELGAP];
    o->sigma = d[S_SIGMA];
    o->mu = d[S_MU];
    o->step = d[S_STEP];
    o->step_aff = d[S_STEP_AFF];
    o->kapovert = d[S_KAPOVERT];
    o->pinf = i[J_PINF];
    o->dinf = i[J_DINF];
    o->has_pinfres = i[J_HAS_PINFRES];
    o->has_dinfres = i[J_HAS_DINFRES];
    o->has_relgap = i[J_HAS_RELGAP];
    o->iter = i[J_ITER];
    o->iter_max = iter_max;
    o->nitref1 = i[J_NIT1];
    o->nitref2 = i[J_NIT2];
    o->nitref3 = i[J_NIT3];
}

// eicos_settings <-> KSettings: the same fields under the same names
#define EICOS_SETTINGS_FIELDS(X)                                                                                       \
    X(feastol) X(abstol) X(reltol) X(feastol_inacc) X(abstol_inacc) X(reltol_inacc) X(linsysacc) X(irerrfact)         \
        X(gamma) X(stepmin) X(stepmax) X(sigmamin) X(sigmamax) X(safeguard) X(nitref) X(iter_max)

void settings_out(const KSettings &k, eicos_settings *o)
{
#define EICOS_COPY(f) o->f = k.f;
    EICOS_SETTINGS_FIELDS(EICOS_COPY)
#undef EICOS_COPY
}

// Checks every field; on success fills *k and returns 0, otherwise fails naming the first bad field.
int settings_in(const eicos_settings *s, KSettings *k)
{
    if (!s)
        return fail(EICOS_ERR_INVALID, "null settings");
    const auto bad = [](const char *field, const char *rule) {
        return fail(EICOS_ERR_INVALID, std::string("eicos_settings.") + field + ": must be " + rule);
    };
#define EICOS_FINITE(f)                                                                                               \
    if (!std::isfinite((double)s->f))                                                                                  \
        return bad(#f, "finite");
    EICOS_SETTINGS_FIELDS(EICOS_FINITE)
#undef EICOS_FINITE
#define EICOS_POSITIVE(f)                                                                                             \
    if (!(s->f > 0.))                                                                                                  \
        return bad(#f, "> 0");
    EICOS_POSITIVE(feastol) EICOS_POSITIVE(abstol) EICOS_POSITIVE(reltol)
    EICOS_POSITIVE(feastol_inacc) EICOS_POSITIVE(abstol_inacc) EICOS_POSITIVE(reltol_inacc)
    EICOS_POSITIVE(linsysacc) EICOS_POSITIVE(irerrfact)
#undef EICOS_POSITIVE
    if (!(s->gamma > 0. && s->gamma <= 1.))
        return bad("gamma", "in (0, 1]");
    if (!(s->stepmin > 0. && s->stepmin <= s->stepmax))
        return bad("stepmin", "in (0, stepmax]");
    if (!(s->stepmax <= 1.))
        return bad("stepmax", "<= 1");
    if (!(s->sigmamin >= 0. && s->sigmamin <= s->sigmamax))
        return bad("sigmamin", "in [0, sigmamax]");
    if (!(s->sigmamax <= 1.))
        return bad("sigmamax", "<= 1");
    if (!(s->safeguard >= 1.))
        return bad("safeguard", ">= 1");
    if (s->nitref < 0 || s->nitref > 32)
        return bad("nitref", "in [0, 32]");
    if (s->iter_max < 1 || s->iter_max > 1000)
        return bad("iter_max", "in [1, 1000]");
#define EICOS_COPY(f) k->f = s->f;
    EICOS_SETTINGS_FIELDS(EICOS_COPY)
#undef EICOS_COPY
    return 0;
}

struct DeviceBuffer
{
    void *p = nullptr;
    size_t bytes = 0;
    void ensure(size_t n)
    {
        if (n > bytes)
        {
            be::dfree(p);
            p = be::alloc(n);
            bytes = n;
        }
    }
    ~DeviceBuffer() { be::dfree(p); }
};
} // namespace

struct eicos_batch
{
    Symbolic S;
    std::unique_ptr<Engine> eng;
    dvec rawG, rawA, c, h, b; // unequilibrated data as given by the caller
    int device = 0, workers = 4;
    bool timing = false;
    SolveStats stats;
    DeviceBuffer din, dout, dint, dmat;
};

struct eicos_solver
{
    // The reference keeps c,h,b in equilibrated form and (un)equilibrates in place; so do we.
    Symbolic S;
    std::unique_ptr<Engine> eng;
    dvec c, h, b;
    bool equilibrated = false;
    dvec x, y, z, s;
    eicos_info info;
    DeviceBuffer dout, dint;
    int device = 0;
};

// Warps per CTA of the vector kernels (= workers per tile).  The factorisation, the triangular
// sweeps and the KKT mat-vecs are programs run by ONE warp per tile (streams.hpp); the remaining
// kernels are element-wise passes and reductions over the rows of a tile, split over `workers` warps.
static int default_workers(long long instances)
{
    (void)instances;
    return 8; // measured on B200 (profiles/r02a): 8 against 4 warps per tile, +5 % at 8 192 instances, +1 % at 65 536
}

extern "C"
{

const char *eicos_last_error(void) { return g_error.c_str(); }

void eicos_default_settings(eicos_settings *out)
{
    if (out)
        settings_out(default_settings(), out);
}

int eicos_device_count(void)
{
#ifndef EICOS_EMU
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess)
        return 0;
    return n;
#else
    return 1;
#endif
}

/* ------------------------------------------------------------------ batched */
eicos_batch *eicos_batch_setup(int n, int m, int p, int l, int ncones, const int *q,
                               const double *Gpr, const int *Gjc, const int *Gir,
                               const double *Apr, const int *Ajc, const int *Air,
                               const double *c, const double *h, const double *b,
                               int device, long long capacity, int workers)
{
    return eicos_batch_setup_ex(n, m, p, l, ncones, q, Gpr, Gjc, Gir, Apr, Ajc, Air, c, h, b, device, capacity, workers, 0);
}

eicos_batch *eicos_batch_setup_ex(int n, int m, int p, int l, int ncones, const int *q,
                                  const double *Gpr, const int *Gjc, const int *Gir,
                                  const double *Apr, const int *Ajc, const int *Air,
                                  const double *c, const double *h, const double *b,
                                  int device, long long capacity, int workers, int flags)
{
    (void)l;
    const bool pim = (flags & EICOS_BATCH_INSTANCE_MATRICES) != 0;
    try
    {
        if (n < 0 || m < 0 || p < 0 || ncones < 0 || (n > 0 && !c))
            throw std::invalid_argument("eicos_batch_setup: negative dimension or missing c");
        std::unique_ptr<eicos_batch> bt(new eicos_batch());
        bt->device = device;
        analyze(bt->S, n, m, p, ncones, q, Gpr, Gjc, Gir, Apr, Ajc, Air);
        const Symbolic &S = bt->S;
        if (S.G.nnz())
            bt->rawG.assign(Gpr, Gpr + S.G.nnz());
        if (S.A.nnz())
            bt->rawA.assign(Apr, Apr + S.A.nnz());
        bt->c.assign(c, c + S.n);
        if (S.m)
        {
            if (!h)
                throw std::invalid_argument("eicos_batch_setup: h missing");
            bt->h.assign(h, h + S.m);
        }
        if (S.p)
        {
            if (!b)
                throw std::invalid_argument("eicos_batch_setup: b missing");
            bt->b.assign(b, b + S.p);
        }
        be::set_device(device);
        if (capacity <= 0)
        { // default: what fits 80 % of the free device memory; -r: that divided by r (r handles share the device)
            const long long share = capacity < 0 ? -capacity : 1;
            (void)share;
            capacity = 4096;
#ifndef EICOS_EMU
            size_t fr = 0, tot = 0;
            EI_CUDA(cudaMemGetInfo(&fr, &tot));
            // rows_total is only known to the engine; estimate it from the symbolic sizes
            const double per_inst = 8.0 * (2.0 * S.nnzL + 13.0 * S.N + 12.0 * S.m + 4.0 * S.n + 4.0 * S.p + 2.0 * S.l +
                                           S.Vslot.size() + 8.0 * S.nc + S.qtot + S_COUNT + J_COUNT +
                                           (pim ? (double)S.G.nnz() + S.A.nnz() + S.N : 0.0));
            capacity = (long long)(0.80 * (double)fr / std::max(per_inst, 8.0)) / share;
            capacity = std::max<long long>(32, std::min<long long>(capacity, 1 << 20));
            capacity -= capacity % 32;
#endif
        }
        bt->workers = workers > 0 ? workers : default_workers(capacity);
        bt->eng.reset(new Engine(bt->S, device, capacity, bt->workers, pim));
        bt->workers = bt->eng->workers();
        return bt.release();
    }
    catch (const std::exception &e)
    {
        g_error = e.what();
        return nullptr;
    }
}

int eicos_batch_update_matrices(eicos_batch *bt, const double *Gpr, const double *Apr)
{
    if (!bt)
        return fail(EICOS_ERR_INVALID, "null handle");
    try
    {
        if (Gpr)
            bt->rawG.assign(Gpr, Gpr + bt->S.G.nnz());
        if (Apr)
            bt->rawA.assign(Apr, Apr + bt->S.A.nnz());
        refresh_values(bt->S, bt->rawG.data(), bt->rawA.data());
        bt->eng->upload_values(bt->S);
        return 0;
    }
    catch (const std::exception &e)
    {
        return fail(EICOS_ERR_DEVICE, e.what());
    }
}

int eicos_batch_solve_device(eicos_batch *bt, int batch,
                             const double *d_cs, const double *d_hs, const double *d_bs,
                             double *d_x, double *d_y, double *d_z, double *d_s,
                             int *d_exitflag, int *d_iters)
{
    return eicos_batch_solve_matrices_device(bt, batch, nullptr, nullptr, d_cs, d_hs, d_bs, d_x, d_y, d_z, d_s,
                                             d_exitflag, d_iters);
}

int eicos_batch_solve_matrices_device(eicos_batch *bt, int batch, const double *d_Gs, const double *d_As,
                                      const double *d_cs, const double *d_hs, const double *d_bs,
                                      double *d_x, double *d_y, double *d_z, double *d_s,
                                      int *d_exitflag, int *d_iters)
{
    if (!bt || batch < 0)
        return fail(EICOS_ERR_INVALID, "null handle or negative batch");
    if ((d_Gs || d_As) && !bt->eng->instance_matrices())
        return fail(EICOS_ERR_INVALID, "per-instance matrices need a handle from eicos_batch_setup_ex(..., EICOS_BATCH_INSTANCE_MATRICES)");
    try
    {
        if (bt->eng->instance_matrices())
            bt->eng->set_matrices(d_Gs, d_As, bt->rawG.data(), bt->rawA.data());
        bt->eng->solve(batch, d_cs, d_hs, d_bs, bt->c.data(), bt->h.data(), bt->b.data(),
                       d_x, d_y, d_z, d_s, d_exitflag, d_iters, nullptr, nullptr,
                       /*keep_sticky=*/false, /*pre_equilibrated=*/false, bt->timing, &bt->stats);
        return 0;
    }
    catch (const std::invalid_argument &e)
    {
        return fail(EICOS_ERR_INVALID, e.what());
    }
    catch (const std::exception &e)
    {
        return fail(EICOS_ERR_DEVICE, e.what());
    }
}

int eicos_batch_solve(eicos_batch *bt, int batch,
                      const double *cs, const double *hs, const double *bs,
                      double *x, double *y, double *z, double *s,
                      int *exitflag, eicos_info *info)
{
    return eicos_batch_solve_matrices(bt, batch, nullptr, nullptr, cs, hs, bs, x, y, z, s, exitflag, info);
}

int eicos_batch_solve_matrices(eicos_batch *bt, int batch, const double *Gs, const double *As,
                               const double *cs, const double *hs, const double *bs,
                               double *x, double *y, double *z, double *s,
                               int *exitflag, eicos_info *info)
{
    if (!bt || batch < 0)
        return fail(EICOS_ERR_INVALID, "null handle or negative batch");
    if ((Gs || As) && !bt->eng->instance_matrices())
        return fail(EICOS_ERR_INVALID, "per-instance matrices need a handle from eicos_batch_setup_ex(..., EICOS_BATCH_INSTANCE_MATRICES)");
    try
    {
        const Symbolic &S = bt->S;
        be::set_device(bt->device);
        be::stream_t st = (be::stream_t)(intptr_t)bt->eng->stream();
        // The device staging buffers hold one SEGMENT of at most `capacity` instances (= one resident
        // chunk of the engine), so their size is bounded by the handle, not by the caller's batch.
        const size_t cap = (size_t)std::max<long long>(1, bt->eng->capacity());
        const size_t nG = (size_t)S.G.nnz(), nA = (size_t)S.A.nnz();
        SolveStats total;
        for (size_t first = 0; first < (size_t)batch || first == 0; first += cap)
        {
            const size_t B = std::min(cap, (size_t)batch - first);
            if (bt->eng->instance_matrices())
            { // stacks of raw matrix values (instance-major); missing ones fall back to the setup matrices
                const size_t ng = Gs ? B * nG : 0, na = As ? B * nA : 0;
                bt->dmat.ensure((ng + na) * sizeof(double));
                double *dm = (double *)bt->dmat.p;
                be::h2d(dm, Gs ? Gs + first * nG : nullptr, ng * sizeof(double), st);
                be::h2d(dm + ng, As ? As + first * nA : nullptr, na * sizeof(double), st);
                bt->eng->set_matrices(Gs ? dm : nullptr, As ? dm + ng : nullptr, bt->rawG.data(), bt->rawA.data());
            }
            const size_t nc_ = cs ? B * S.n : 0, nh_ = hs ? B * S.m : 0, nb_ = bs ? B * S.p : 0;
            bt->din.ensure((nc_ + nh_ + nb_) * sizeof(double));
            double *din = (double *)bt->din.p;
            double *dc = cs ? din : nullptr, *dh = hs ? din + nc_ : nullptr, *db = bs ? din + nc_ + nh_ : nullptr;
            be::h2d(dc, cs ? cs + first * S.n : nullptr, nc_ * sizeof(double), st);
            be::h2d(dh, hs ? hs + first * S.m : nullptr, nh_ * sizeof(double), st);
            be::h2d(db, bs ? bs + first * S.p : nullptr, nb_ * sizeof(double), st);
            const size_t ox = x ? B * S.n : 0, oy = y ? B * S.p : 0, oz = z ? B * S.m : 0, os = s ? B * S.m : 0;
            const size_t oi = info ? B * S_WORK_END : 0;
            bt->dout.ensure((ox + oy + oz + os + oi) * sizeof(double));
            double *dout = (double *)bt->dout.p;
            double *dx = x ? dout : nullptr, *dy = y ? dout + ox : nullptr, *dz = z ? dout + ox + oy : nullptr;
            double *dsl = s ? dout + ox + oy + oz : nullptr, *dinfo = info ? dout + ox + oy + oz + os : nullptr;
            const size_t ie = B, ii = info ? B * J_WORK_END : 0;
            bt->dint.ensure((ie + ii) * sizeof(int));
            int *dexit = (int *)bt->dint.p, *diinfo = info ? dexit + ie : nullptr;
            bt->eng->solve((int)B, dc, dh, db, bt->c.data(), bt->h.data(), bt->b.data(),
                           dx, dy, dz, dsl, dexit, nullptr, dinfo, diinfo,
                           false, false, bt->timing, &bt->stats);
            be::d2h(x ? x + first * S.n : nullptr, dx, ox * sizeof(double), st);
            be::d2h(y ? y + first * S.p : nullptr, dy, oy * sizeof(double), st);
            be::d2h(z ? z + first * S.m : nullptr, dz, oz * sizeof(double), st);
            be::d2h(s ? s + first * S.m : nullptr, dsl, os * sizeof(double), st);
            std::vector<int> hexit(ie), hii(ii);
            std::vector<double> hinfo(oi);
            be::d2h(hexit.data(), dexit, ie * sizeof(int), st);
            be::d2h(hii.data(), diinfo, ii * sizeof(int), st);
            be::d2h(hinfo.data(), dinfo, oi * sizeof(double), st);
            be::sync(st);
            if (exitflag)
                std::copy(hexit.begin(), hexit.end(), exitflag + first);
            if (info)
                for (size_t k = 0; k < B; k++)
                    info_from_rows(hinfo.data() + k * S_WORK_END, hii.data() + k * J_WORK_END, bt->eng->settings().iter_max, info + first + k);
            total += bt->stats;
            if (batch == 0)
                break;
        }
        bt->stats = total;
        return 0;
    }
    catch (const std::invalid_argument &e)
    {
        return fail(EICOS_ERR_INVALID, e.what());
    }
    catch (const std::exception &e)
    {
        return fail(EICOS_ERR_DEVICE, e.what());
    }
}

int eicos_batch_set_timing(eicos_batch *bt, int enabled)
{
    if (!bt)
        return fail(EICOS_ERR_INVALID, "null handle");
    bt->timing = enabled != 0;
    return 0;
}

int eicos_batch_set_compaction(eicos_batch *bt, int enabled)
{
    if (!bt)
        return fail(EICOS_ERR_INVALID, "null handle");
    bt->eng->set_compaction(enabled != 0);
    return 0;
}

int eicos_batch_get_stats(const eicos_batch *bt, eicos_batch_stats *o)
{
    if (!bt || !o)
        return fail(EICOS_ERR_INVALID, "null argument");
    const SolveStats &s = bt->stats;
    o->chunks = s.chunks;
    o->ipm_iterations = s.ipm_iterations;
    o->launches = s.launches;
    o->ir_rounds = s.ir_rounds;
    o->ms_total = s.ms_total;
    o->ms_factor = s.ms_factor;
    o->ms_solve = s.ms_solve;
    o->ms_other = s.ms_other;
    o->factor_launch_tiles = s.factor_launch_tiles;
    o->solve_launch_tiles = s.solve_launch_tiles;
    o->factor_launches = s.factor_launches;
    o->solve_launches = s.solve_launches;
    o->compactions = s.compactions;
    for (int k = 0; k < 5; k++)
        o->kkt_phase_cycles[k] = s.kkt_phase_cycles[k];
    o->ms_resid = s.ms_resid;
    o->ms_vector = s.ms_vector;
    o->resid_launch_tiles = s.resid_launch_tiles;
    o->vector_launch_tiles = s.vector_launch_tiles;
    o->resid_launches = s.resid_launches;
    o->vector_launches = s.vector_launches;
    o->lane_rounds = s.lane_rounds;
    return 0;
}

int eicos_batch_get_dims(const eicos_batch *bt, eicos_batch_dims *o)
{
    if (!bt || !o)
        return fail(EICOS_ERR_INVALID, "null argument");
    const Symbolic &S = bt->S;
    o->n = S.n;
    o->m = S.m;
    o->p = S.p;
    o->l = S.l;
    o->ncones = S.nc;
    o->dim_K = S.N;
    o->nnzK = (int)S.Ki.size();
    o->nnzL = S.nnzL;
    o->nnzV = (int)S.Vslot.size();
    o->nnzG = S.G.nnz();
    o->nnzA = S.A.nnz();
    o->etree_height = S.height;
    o->max_col = S.maxcol;
    o->tile_width = Engine::tile_width();
    o->workers = bt->workers;
    o->ldl_fma = S.fma_count;
    o->capacity = bt->eng->capacity();
    o->workspace_bytes = (long long)bt->eng->workspace_bytes();
    o->rows_per_instance = bt->eng->layout().rows_total;
    return 0;
}

int eicos_batch_get_program_stats(const eicos_batch *bt, eicos_program_stats *o)
{
    if (!bt || !o)
        return fail(EICOS_ERR_INVALID, "null argument");
    const ProgramStats p = bt->eng->program_stats();
    o->sw_slots = p.sw_slots;
    o->fa_slots = p.fa_slots;
    o->fa_fast = p.fa_fast;
    o->sw_far = p.sw_far;
    o->sw_direct = p.sw_direct;
    o->fa_home = p.fa_home;
    o->fw_loads = p.fw_loads;
    o->bw_loads = p.bw_loads;
    o->fa_loads = p.fa_loads;
    o->mv_loads = p.mv_loads;
    return 0;
}

int eicos_batch_get_symbolic(const eicos_batch *bt, int *pinv, int *parent, int *Lp, int *Li, int *Kp, int *Ki)
{
    if (!bt)
        return fail(EICOS_ERR_INVALID, "null handle");
    const Symbolic &S = bt->S;
    if (pinv)
        std::copy(S.pinv.begin(), S.pinv.end(), pinv);
    if (parent)
        std::copy(S.parent.begin(), S.parent.end(), parent);
    if (Lp)
        std::copy(S.Lp.begin(), S.Lp.end(), Lp);
    if (Li)
        std::copy(S.Li.begin(), S.Li.end(), Li);
    if (Kp)
        std::copy(S.Kp.begin(), S.Kp.end(), Kp);
    if (Ki)
        std::copy(S.Ki.begin(), S.Ki.end(), Ki);
    return 0;
}

int eicos_batch_debug_init(eicos_batch *bt, int batch, const double *cs, const double *hs, const double *bs,
                           double *Lx, double *D, double *sol1, double *sol2, int *nitref)
{
    if (!bt || batch <= 0)
        return fail(EICOS_ERR_INVALID, "null handle or empty batch");
    try
    {
        const Symbolic &S = bt->S;
        be::set_device(bt->device);
        be::stream_t st = (be::stream_t)(intptr_t)bt->eng->stream();
        const size_t B = (size_t)batch;
        const size_t nc_ = cs ? B * S.n : 0, nh_ = hs ? B * S.m : 0, nb_ = bs ? B * S.p : 0;
        bt->din.ensure((nc_ + nh_ + nb_) * sizeof(double));
        double *din = (double *)bt->din.p;
        double *dc = cs ? din : nullptr, *dh = hs ? din + nc_ : nullptr, *db = bs ? din + nc_ + nh_ : nullptr;
        be::h2d(dc, cs, nc_ * sizeof(double), st);
        be::h2d(dh, hs, nh_ * sizeof(double), st);
        be::h2d(db, bs, nb_ * sizeof(double), st);
        be::sync(st);
        if (bt->eng->instance_matrices()) // the shared raw matrices stand in for every instance
            bt->eng->set_matrices(nullptr, nullptr, bt->rawG.data(), bt->rawA.data());
        bt->eng->debug_factor_init(batch, dc, dh, db, bt->c.data(), bt->h.data(), bt->b.data(), Lx, D, sol1, sol2, nitref);
        return 0;
    }
    catch (const std::invalid_argument &e)
    {
        return fail(EICOS_ERR_INVALID, e.what());
    }
    catch (const std::exception &e)
    {
        return fail(EICOS_ERR_DEVICE, e.what());
    }
}

int eicos_batch_debug_line_search(eicos_batch *bt, int batch, const double *lambda, const double *ds, const double *dz,
                                  const double *scalars, double *alpha)
{
    if (!bt || batch <= 0 || !lambda || !ds || !dz || !scalars || !alpha)
        return fail(EICOS_ERR_INVALID, "null argument or empty batch");
    try
    {
        bt->eng->debug_line_search(batch, lambda, ds, dz, scalars, alpha);
        return 0;
    }
    catch (const std::invalid_argument &e)
    {
        return fail(EICOS_ERR_INVALID, e.what());
    }
    catch (const std::exception &e)
    {
        return fail(EICOS_ERR_DEVICE, e.what());
    }
}

int eicos_batch_debug_set_iter_max(eicos_batch *bt, int iter_max)
{
    if (!bt)
        return fail(EICOS_ERR_INVALID, "null handle");
    KSettings k = bt->eng->settings();
    k.iter_max = iter_max > 0 ? std::min(iter_max, (int)Settings::iter_max) : (int)Settings::iter_max;
    bt->eng->set_settings(k);
    return 0;
}

int eicos_batch_set_settings(eicos_batch *bt, const eicos_settings *settings)
{
    if (!bt)
        return fail(EICOS_ERR_INVALID, "null handle");
    KSettings k;
    if (const int rc = settings_in(settings, &k))
        return rc;
    bt->eng->set_settings(k);
    return 0;
}

int eicos_batch_get_settings(const eicos_batch *bt, eicos_settings *out)
{
    if (!bt || !out)
        return fail(EICOS_ERR_INVALID, "null argument");
    settings_out(bt->eng->settings(), out);
    return 0;
}

// ---------------------------------------------------------------- several devices behind one handle
struct eicos_multi
{
    std::vector<eicos_batch *> part;
    int n = 0, m = 0, p = 0, nnzG = 0, nnzA = 0;
};

static void multi_slice(int batch, int parts, int k, int &first, int &count)
{ // contiguous, sizes differ by at most one (the same cut as eicos_b200/sharding.py: shard_range)
    const int base = batch / parts, rem = batch % parts;
    first = k * base + std::min(k, rem);
    count = base + (k < rem ? 1 : 0);
}

eicos_multi *eicos_multi_setup(int n, int m, int p, int l, int ncones, const int *q,
                               const double *Gpr, const int *Gjc, const int *Gir,
                               const double *Apr, const int *Ajc, const int *Air,
                               const double *c, const double *h, const double *b,
                               int ngpu, const int *devices, long long capacity, int workers, int flags)
{
    if (ngpu < 1)
    {
        g_error = "eicos_multi_setup: ngpu must be at least 1";
        return nullptr;
    }
    std::unique_ptr<eicos_multi> mt(new eicos_multi());
    for (int k = 0; k < ngpu; k++)
    {
        // default capacity on a device that is listed r times: 1 / r of what fits it, taken while its first handle is built
        long long cap_k = capacity;
        if (capacity <= 0 && devices)
        {
            int later = 0;
            for (int j = k; j < ngpu; j++)
                later += devices[j] == devices[k];
            cap_k = -(long long)later; // (the earlier handles of this device have taken their share of the free memory already)
        }
        eicos_batch *bt = eicos_batch_setup_ex(n, m, p, l, ncones, q, Gpr, Gjc, Gir, Apr, Ajc, Air, c, h, b,
                                               devices ? devices[k] : k, cap_k, workers, flags);
        if (!bt)
        { // g_error says why
            for (eicos_batch *o : mt->part)
                eicos_batch_cleanup(o);
            return nullptr;
        }
        mt->part.push_back(bt);
    }
    const Symbolic &S = mt->part[0]->S;
    mt->n = S.n, mt->m = S.m, mt->p = S.p, mt->nnzG = S.G.nnz(), mt->nnzA = S.A.nnz();
    return mt.release();
}

int eicos_multi_ngpu(const eicos_multi *mt) { return mt ? (int)mt->part.size() : 0; }

int eicos_multi_slice(const eicos_multi *mt, int batch, int k, int *first, int *count)
{
    if (!mt || k < 0 || k >= (int)mt->part.size() || batch < 0 || !first || !count)
        return fail(EICOS_ERR_INVALID, "eicos_multi_slice: bad argument");
    multi_slice(batch, (int)mt->part.size(), k, *first, *count);
    return 0;
}

int eicos_multi_solve(eicos_multi *mt, int batch, const double *Gs, const double *As,
                      const double *cs, const double *hs, const double *bs,
                      double *x, double *y, double *z, double *s, int *exitflag, eicos_info *info)
{
    if (!mt || batch <= 0)
        return fail(EICOS_ERR_INVALID, "null handle or empty batch");
    const int parts = (int)mt->part.size();
    std::vector<int> rc(parts, 0);
    std::vector<std::string> err(parts);
    std::vector<std::thread> th;
    const auto run = [&](int k) {
        int first, count;
        multi_slice(batch, parts, k, first, count);
        if (count == 0)
            return;
        const size_t f = (size_t)first;
        const auto at = [&](const double *ptr, int width) { return ptr ? ptr + f * (size_t)width : nullptr; };
        const auto atw = [&](double *ptr, int width) { return ptr ? ptr + f * (size_t)width : nullptr; };
        rc[k] = eicos_batch_solve_matrices(mt->part[k], count, at(Gs, mt->nnzG), at(As, mt->nnzA), at(cs, mt->n), at(hs, mt->m),
                                           at(bs, mt->p), atw(x, mt->n), atw(y, mt->p), atw(z, mt->m), atw(s, mt->m),
                                           exitflag ? exitflag + f : nullptr, info ? info + f : nullptr);
        if (rc[k] != 0)
            err[k] = g_error; // (thread-local: carried back to the caller's thread below)
    };
    for (int k = 1; k < parts; k++)
        th.emplace_back(run, k);
    run(0);
    for (std::thread &t : th)
        t.join();
    for (int k = 0; k < parts; k++)
        if (rc[k] != 0)
            return fail(rc[k], ("device slice " + std::to_string(k) + ": " + err[k]).c_str());
    return 0;
}

int eicos_multi_set_settings(eicos_multi *mt, const eicos_settings *settings)
{
    if (!mt)
        return fail(EICOS_ERR_INVALID, "null handle");
    KSettings k;
    if (const int rc = settings_in(settings, &k))
        return rc;
    for (eicos_batch *bt : mt->part)
        bt->eng->set_settings(k);
    return 0;
}

int eicos_multi_get_settings(const eicos_multi *mt, eicos_settings *out)
{
    if (!mt || !out)
        return fail(EICOS_ERR_INVALID, "null argument");
    settings_out(mt->part[0]->eng->settings(), out);
    return 0;
}

void eicos_multi_cleanup(eicos_multi *mt)
{
    if (!mt)
        return;
    for (eicos_batch *bt : mt->part)
        eicos_batch_cleanup(bt);
    delete mt;
}

void *eicos_batch_stream(const eicos_batch *bt) { return bt ? bt->eng->stream() : nullptr; }

void eicos_batch_cleanup(eicos_batch *bt)
{
    if (bt)
    {
        be::set_device(bt->device);
        delete bt;
    }
}

/* ------------------------------------------------------------------ single instance */
static void equilibrate_vectors(eicos_solver *s)
{ // src/eicos.cpp:364-373
    for (int k = 0; k < s->S.n; k++)
        s->c[k] /= s->S.xeq[k];
    for (int k = 0; k < s->S.p; k++)
        s->b[k] /= s->S.Aeq[k];
    for (int k = 0; k < s->S.m; k++)
        s->h[k] /= s->S.Geq[k];
    s->equilibrated = true;
}

eicos_solver *eicos_setup(int n, int m, int p, int l, int ncones, const int *q,
                          const double *Gpr, const int *Gjc, const int *Gir,
                          const double *Apr, const int *Ajc, const int *Air,
                          const double *c, const double *h, const double *b, int device)
{
    (void)l;
    try
    {
        if (n < 0 || m < 0 || p < 0 || ncones < 0 || (n > 0 && !c))
            throw std::invalid_argument("eicos_setup: negative dimension or missing c");
        std::unique_ptr<eicos_solver> s(new eicos_solver());
        s->device = device;
        std::memset(&s->info, 0, sizeof(s->info));
        analyze(s->S, n, m, p, ncones, q, Gpr, Gjc, Gir, Apr, Ajc, Air);
        const Symbolic &S = s->S;
        s->c.assign(c, c + S.n);
        if (S.m)
        {
            if (!h)
                throw std::invalid_argument("eicos_setup: h missing");
            s->h.assign(h, h + S.m);
        }
        if (S.p)
        {
            if (!b)
                throw std::invalid_argument("eicos_setup: b missing");
            s->b.assign(b, b + S.p);
        }
        equilibrate_vectors(s.get());
        s->x.assign(S.n, 0.0);
        s->y.assign(S.p, 0.0);
        s->z.assign(S.m, 0.0);
        s->s.assign(S.m, 0.0);
        be::set_device(device);
        s->eng.reset(new Engine(s->S, device, 1, default_workers(1)));
        return s.release();
    }
    catch (const std::exception &e)
    {
        g_error = e.what();
        return nullptr;
    }
}

static int update_common(eicos_solver *s, bool full, const double *Gpr, const double *Apr,
                         const double *c, const double *h, const double *b)
{
    if (!s)
        return fail(EICOS_ERR_INVALID, "null handle");
    try
    {
        Symbolic &S = s->S;
        if (full)
        { // Eigen overload: everything overwritten, no un-equilibration needed (src/eicos.cpp:2038-2045)
            if ((S.G.nnz() && !Gpr) || (S.A.nnz() && !Apr) || (S.n && !c) || (S.m && !h) || (S.p && !b))
                throw std::invalid_argument("eicos_update_data_full: all arrays are required");
            s->c.assign(c, c + S.n);
            if (S.m)
                s->h.assign(h, h + S.m);
            if (S.p)
                s->b.assign(b, b + S.p);
            refresh_values(S, Gpr, Apr);
        }
        else
        { // pointer overload (src/eicos.cpp:2053-2082)
            // every argument is checked before anything is touched: a rejected update leaves the solver as it was
            if (Gpr && S.m && !h)
                throw std::invalid_argument("eicos_update_data: h must accompany Gpr");
            if (Apr && S.p && !b)
                throw std::invalid_argument("eicos_update_data: b must accompany Apr");
            if (s->equilibrated)
            { // unsetEquilibration :389-404
                unequilibrate(S);
                for (int k = 0; k < S.n; k++)
                    s->c[k] *= S.xeq[k];
                for (int k = 0; k < S.p; k++)
                    s->b[k] *= S.Aeq[k];
                for (int k = 0; k < S.m; k++)
                    s->h[k] *= S.Geq[k];
                s->equilibrated = false;
            }
            if (Gpr && S.m)
                s->h.assign(h, h + S.m);
            if (Apr && S.p)
                s->b.assign(b, b + S.p);
            if (c)
                s->c.assign(c, c + S.n);
            refresh_values(S, Gpr, Apr);
        }
        equilibrate_vectors(s);
        s->eng->upload_values(S);
        return 0;
    }
    catch (const std::invalid_argument &e)
    {
        return fail(EICOS_ERR_INVALID, e.what());
    }
    catch (const std::exception &e)
    {
        return fail(EICOS_ERR_DEVICE, e.what());
    }
}

int eicos_update_data(eicos_solver *s, const double *Gpr, const double *Apr,
                      const double *c, const double *h, const double *b)
{
    return update_common(s, false, Gpr, Apr, c, h, b);
}

int eicos_update_data_full(eicos_solver *s, const double *Gpr, const double *Apr,
                           const double *c, const double *h, const double *b)
{
    return update_common(s, true, Gpr, Apr, c, h, b);
}

int eicos_set_settings(eicos_solver *s, const eicos_settings *settings)
{
    if (!s)
        return fail(EICOS_ERR_INVALID, "null handle");
    KSettings k;
    if (const int rc = settings_in(settings, &k))
        return rc;
    s->eng->set_settings(k);
    return 0;
}

int eicos_get_settings(const eicos_solver *s, eicos_settings *out)
{
    if (!s || !out)
        return fail(EICOS_ERR_INVALID, "null argument");
    settings_out(s->eng->settings(), out);
    return 0;
}

int eicos_solve(eicos_solver *s)
{
    if (!s)
        return fail(EICOS_ERR_INVALID, "null handle");
    try
    {
        const Symbolic &S = s->S;
        be::set_device(s->device);
        be::stream_t st = (be::stream_t)(intptr_t)s->eng->stream();
        const size_t nd = (size_t)S.n + S.p + 2 * (size_t)S.m + S_WORK_END;
        s->dout.ensure(nd * sizeof(double));
        s->dint.ensure((1 + J_WORK_END) * sizeof(int));
        double *dx = (double *)s->dout.p, *dy = dx + S.n, *dz = dy + S.p, *dsl = dz + S.m, *dinfo = dsl + S.m;
        int *dexit = (int *)s->dint.p, *dii = dexit + 1;
        s->eng->solve(1, nullptr, nullptr, nullptr, s->c.data(), s->h.data(), s->b.data(),
                      dx, dy, dz, dsl, dexit, nullptr, dinfo, dii,
                      /*keep_sticky=*/true, /*pre_equilibrated=*/true, false, nullptr);
        double hinfo[S_WORK_END];
        int hi[1 + J_WORK_END];
        be::d2h(s->x.data(), dx, S.n * sizeof(double), st);
        be::d2h(s->y.data(), dy, S.p * sizeof(double), st);
        be::d2h(s->z.data(), dz, S.m * sizeof(double), st);
        be::d2h(s->s.data(), dsl, S.m * sizeof(double), st);
        be::d2h(hinfo, dinfo, sizeof(hinfo), st);
        be::d2h(hi, dexit, sizeof(hi), st);
        be::sync(st);
        info_from_rows(hinfo, hi + 1, s->eng->settings().iter_max, &s->info);
        return hi[0];
    }
    catch (const std::exception &e)
    {
        g_error = e.what();
        return EXIT_FATAL;
    }
}

const double *eicos_solution(const eicos_solver *s) { return s ? s->x.data() : nullptr; }

int eicos_get_duals(const eicos_solver *s, double *y, double *z, double *slack)
{
    if (!s)
        return fail(EICOS_ERR_INVALID, "null handle");
    if (y)
        std::copy(s->y.begin(), s->y.end(), y);
    if (z)
        std::copy(s->z.begin(), s->z.end(), z);
    if (slack)
        std::copy(s->s.begin(), s->s.end(), slack);
    return 0;
}

int eicos_get_info(const eicos_solver *s, eicos_info *out)
{
    if (!s || !out)
        return fail(EICOS_ERR_INVALID, "null argument");
    *out = s->info;
    return 0;
}

void eicos_cleanup(eicos_solver *s)
{
    if (s)
    {
        be::set_device(s->device);
        delete s;
    }
}

} // extern "C"
