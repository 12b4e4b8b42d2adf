"""Gradients of batched solves (eicos_batch_adjoint, BatchSolver.adjoint, eicos_b200.autograd.EiCOSLayer).

The checks are independent of the engine: K0 = [0 A' G'; A 0 0; G 0 -W^2] is assembled in numpy from the returned
x, y, z, s with W^2 from its closed forms in the original scaling (LP rows: s / z; a cone: eta^2 (2 w w' - J)).
The CPU tier runs on the emulator library; the gpu tier repeats the checks on the CUDA library and compares the two.
"""
import numpy as np
import pytest

import oracle
from eicos_b200.binding import BatchSolver
from eicos_b200.workloads import MPC_REL, perturbed, perturbed_matrices, soc_mpc, soc_mpc_batch

DELTA = 7e-8  # static regularisation of the KKT matrix (Settings::deltastat)
EICOS_ERR_INVALID = -100


# ------------------------------------------------------------------ workloads
def _workload(name):
    """(problem, batch, stacked data for solve(), instance-matrices handle?)"""
    if name == "MPC02x16":
        P = oracle.load_fixture("MPC02")
        W = perturbed(P, 16, rel=MPC_REL, seed=5)
        return P, 16, {"hs": W["hs"], "bs": W["bs"]}, False
    if name == "soc_mpc":
        P = soc_mpc(T=6)
        W = soc_mpc_batch(P, 12)
        return P, 12, {"hs": W["hs"], "bs": W["bs"]}, False
    if name == "MPC02_matrices":
        P = oracle.load_fixture("MPC02")
        W = perturbed_matrices(P, 8, rel=0.01, seed=11, scale_spread=0.5)
        return P, 8, {k: W[k] for k in ("Gs", "As", "hs", "bs")}, True
    P = oracle.load_fixture(name)
    W = perturbed(P, 4, rel=0.02, seed=9, vary=("h", "b"))
    return P, 4, {"hs": W["hs"], "bs": W["bs"]}, False


WORKLOADS = ["update_data_1", "issue98", "lp_afiro", "MPC02x16", "soc_mpc", "MPC02_matrices"]
# issue98 ends at x = s = 0 with all eleven constraints active on five variables: W^2 ~ 1e-10 lies below the static
# regularisation, K0 has a condition number of about 2e10, and the refined solve stops at a relative residual of about
# 1e-8 (measured on the emulator); every other workload meets 1e-9 against K0 itself
RESIDUAL_BOUND = {"issue98": 1e-7}


def _cones(P):
    q = P.get("q")
    return int(P["l"]), [] if q is None else [int(d) for d in np.asarray(q)]


def _matrices(P, data, b):
    Gv = data["Gs"][b] if data.get("Gs") is not None else np.asarray(P["Gpr"], float)
    Av = data["As"][b] if data.get("As") is not None else (np.asarray(P["Apr"], float) if P.get("Apr") is not None else np.zeros(0))
    return Gv, Av


def _dense(P, vals, kind):
    n = int(P["n"])
    rows = int(P["m"]) if kind == "G" else int(P["p"])
    M = np.zeros((rows, n))
    if vals.size:
        jc, ir = np.asarray(P[kind + "jc"]), np.asarray(P[kind + "ir"])
        for j in range(n):
            for k in range(jc[j], jc[j + 1]):
                M[ir[k], j] = vals[k]
    return M


def w_squared(P, s, z):
    l, q = _cones(P)
    m = s.size
    W = np.zeros((m, m))
    W[range(l), range(l)] = s[:l] / z[:l]
    k = l
    for d in q:
        sc, zc = s[k:k + d], z[k:k + d]
        J = -np.eye(d)
        J[0, 0] = 1.0
        sn, zn = np.sqrt(sc @ J @ sc), np.sqrt(zc @ J @ zc)
        sb, zb = sc / sn, zc / zn
        w = (sb + J @ zb) / (2.0 * np.sqrt(0.5 * (1.0 + zb @ sb)))
        W[k:k + d, k:k + d] = (sn / zn) * (2.0 * np.outer(w, w) - J)
        k += d
    return W


def kkt0(P, x, y, z, s, Gv, Av):
    n, m, p = int(P["n"]), int(P["m"]), int(P["p"])
    G, A = _dense(P, Gv, "G"), _dense(P, Av, "A")
    K = np.zeros((n + p + m, n + p + m))
    K[:n, n:n + p], K[n:n + p, :n] = A.T, A
    K[:n, n + p:], K[n + p:, :n] = G.T, G
    K[n + p:, n + p:] = -w_squared(P, s, z)
    return K


def regularisation(P, Gv, Av):
    """Diagonal the solve adds to K0: the solver's static regularisation on the equilibrated matrix, D (delta S) D with
    S = +1 (x), -1 (y), -1 (z; +1 on the last row of every cone, as the reference's refinement residual has it)."""
    Q = dict(P)
    Q["Gpr"] = Gv
    if Av.size:
        Q["Apr"] = Av
    xe, Ae, Ge = oracle.OracleSolver(Q).equil()
    l, q = _cones(P)
    sz = -np.ones(int(P["m"]))
    k = l
    for d in q:
        k += d
        sz[k - 1] = 1.0
    D = np.concatenate([xe, Ae, Ge])
    return DELTA * D * D * np.concatenate([np.ones(xe.size), -np.ones(Ae.size), sz])


def _random_g(batch, n, p, m, seed=3):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((batch, n)), rng.standard_normal((batch, p)), rng.standard_normal((batch, m))


def _solve_and_adjoint(lib, name, capacity=64):
    P, batch, data, pim = _workload(name)
    bs = BatchSolver(P, capacity=capacity, lib=lib, instance_matrices=pim)
    out = bs.solve(batch, **data)
    g = _random_g(batch, bs.n, bs.p, bs.m)
    res = bs.adjoint(out, *g, Gs=data.get("Gs"), As=data.get("As"))
    return P, data, bs, out, g, res


def check_linear_system(lib, name):
    """Per instance: K0 u = g to the accuracy of the regularised solve; dG / dA are the outer-product formulas."""
    P, data, bs, out, (gx, gy, gz), res = _solve_and_adjoint(lib, name)
    n, p = bs.n, bs.p
    assert np.all(out["exit"] == 0), out["exit"]
    assert np.all(res["status"] == 0), res["status"]
    worst0 = worstr = 0.0
    for b in range(out["exit"].size):
        x, y, z, s = (out[k][b] for k in "xyzs")
        Gv, Av = _matrices(P, data, b)
        K = kkt0(P, x, y, z, s, Gv, Av)
        u = np.concatenate([-res["c"][b], res["b"][b], res["h"][b]])
        g = np.concatenate([gx[b], gy[b], gz[b]])
        scale = np.abs(K).sum(1).max() * np.abs(u).max() + np.abs(g).max()
        r0 = np.abs(K @ u - g).max() / scale
        rr = np.abs(K @ u + regularisation(P, Gv, Av) * u - g).max() / scale
        worst0, worstr = max(worst0, r0), max(worstr, rr)
        assert rr <= RESIDUAL_BOUND.get(name, 1e-9), (b, rr, r0)
        # the outer products, entry by entry
        G, A = _dense(P, np.arange(1, Gv.size + 1.0), "G"), _dense(P, np.arange(1, Av.size + 1.0), "A")
        for M, d, dual, uk in ((G, res["G"][b], z, res["h"][b]), (A, res["A"][b], y, res["b"][b])):
            i, j = np.nonzero(M)
            order = np.argsort(M[i, j])
            i, j = i[order], j[order]
            ux = -res["c"][b]
            ref = -(dual[i] * ux[j] + uk[i] * x[j])
            bound = 1e-14 * (np.abs(dual[i] * ux[j]) + np.abs(uk[i] * x[j]))
            assert np.all(np.abs(d - ref) <= bound), (b, np.max(np.abs(d - ref) - bound))
    print(f"\n{name}: worst ||K0 u - g|| / (||K0|| ||u|| + ||g||) = {worst0:.2e}; with the solve's regularisation {worstr:.2e}")
    return worst0


def check_status(lib):
    """MPC02 with h, b +-5 %: optimal and primal-infeasible instances; each optimal instance's gradients equal those of
    the same instance differentiated alone, bit for bit; a slack off the interior gives status 2."""
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 24, rel=0.05, seed=4)
    bs = BatchSolver(P, capacity=64, lib=lib)
    out = bs.solve(24, hs=W["hs"], bs=W["bs"])
    opt = (out["exit"] == 0) | (out["exit"] == 10)
    assert opt.any() and (~opt).any(), out["exit"]
    g = _random_g(24, bs.n, bs.p, bs.m)
    res = bs.adjoint(out, *g)
    assert np.all(res["status"][~opt] == 1)
    assert np.all(res["status"][opt] == 0)
    for k in ("c", "h", "b", "G", "A"):
        assert np.all(res[k][~opt] == 0.0), k
    for b in np.nonzero(opt)[0][:4]:
        one = {k: out[k][b:b + 1] for k in ("x", "y", "z", "s", "exit")}
        alone = bs.adjoint(one, *(v[b:b + 1] for v in g))
        for k in ("c", "h", "b", "G", "A"):
            assert np.array_equal(alone[k][0], res[k][b]), (b, k)
    bad = {k: out[k].copy() for k in ("x", "y", "z", "s", "exit")}
    b0 = int(np.nonzero(opt)[0][0])
    bad["s"][b0, 0] = 0.0
    res2 = bs.adjoint(bad, *g)
    assert res2["status"][b0] == 2
    assert np.all(res2["c"][b0] == 0.0)
    keep = np.arange(24) != b0
    assert np.array_equal(res2["c"][keep], res["c"][keep])
    return res


def check_chunking(lib):
    """capacity 64, batch 200 (four chunks) against one chunk: the same bits."""
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 200, rel=MPC_REL, seed=8)
    big = BatchSolver(P, capacity=256, lib=lib)
    out = big.solve(200, hs=W["hs"], bs=W["bs"])
    g = _random_g(200, big.n, big.p, big.m, seed=4)
    one = big.adjoint(out, *g)
    small = BatchSolver(P, capacity=64, lib=lib)
    four = small.adjoint(out, *g)
    for k in ("c", "h", "b", "G", "A", "status"):
        assert np.array_equal(one[k], four[k]), k
    assert np.all(one["status"][out["exit"] == 0] == 0)


# ------------------------------------------------------------------ CPU tier (emulator)
@pytest.mark.parametrize("name", WORKLOADS)
def test_linear_system(emu_lib, name):
    worst0 = check_linear_system(emu_lib, name)
    assert worst0 <= RESIDUAL_BOUND.get(name, 1e-9), worst0


def _apex(P, s):
    l, q = _cones(P)
    starts = l + np.concatenate([[0], np.cumsum(q)[:-1]]).astype(int) if q else np.zeros(0, int)
    return min((abs(s[k]) for k in starts), default=np.inf) / max(1.0, np.max(np.abs(s))) <= 1e-5


@pytest.mark.parametrize("pim", [False, True], ids=["shared", "instance_matrices"])
def test_finite_differences(emu_lib, pim):
    """<grad L, v> against central differences of L = <gx, x> + <gy, y> + <gz, z> at theta +- eps v (one batch call
    per direction), for directions in c, h, b and, with per-instance matrices, in G and A."""
    P = oracle.load_fixture("update_data_1")
    batch, eps = 6, 1e-6
    bs = BatchSolver(P, capacity=64, lib=emu_lib, instance_matrices=pim)
    bs.set_settings(feastol=1e-11, abstol=1e-11, reltol=1e-11)
    W = perturbed(P, batch, rel=0.05, seed=21)
    theta = {"cs": np.tile(np.asarray(P["c"], float), (batch, 1)), "hs": W["hs"], "bs": W["bs"]}
    if pim:
        M = perturbed_matrices(P, batch, rel=0.02, seed=22)
        theta["Gs"], theta["As"] = M["Gs"], M["As"]
    theta = {k: v for k, v in theta.items() if v is not None and v.size}
    out = bs.solve(batch, **theta)
    g = _random_g(batch, bs.n, bs.p, bs.m, seed=5)
    res = bs.adjoint(out, *g, Gs=theta.get("Gs"), As=theta.get("As"))
    apex = np.array([_apex(P, out["s"][b]) for b in range(batch)])
    print(f"\n{int(apex.sum())} of {batch} instances excluded: a cone's slack at its apex")
    rng = np.random.default_rng(6)
    worst = 0.0
    for k, v0 in theta.items():
        v = rng.standard_normal(v0.shape) * np.abs(v0)
        st = {kk: np.concatenate([vv, vv]) for kk, vv in theta.items()}
        st[k] = np.concatenate([v0 + eps * v, v0 - eps * v])
        o2 = bs.solve(2 * batch, **st)
        L = sum((o2[a] * np.concatenate([gg, gg])).sum(1) for a, gg in zip("xyz", g))
        fd = (L[:batch] - L[batch:]) / (2 * eps)
        ad = (res[k[0]] * v).sum(1)
        ok = (res["status"] == 0) & (o2["exit"][:batch] == 0) & (o2["exit"][batch:] == 0) & ~apex
        assert ok.sum() >= batch // 2, k
        rel = np.abs(fd - ad)[ok] / np.maximum(np.abs(fd), np.abs(ad))[ok]
        worst = max(worst, rel.max())
        assert np.all(rel <= 1e-3), (k, rel)
    print(f"worst relative difference to central differences: {worst:.2e} (bound 1e-3)")


def test_status(emu_lib):
    check_status(emu_lib)


def test_chunking(emu_lib):
    check_chunking(emu_lib)


def test_bad_input(emu_lib):
    import ctypes as C
    P = oracle.load_fixture("update_data_1")
    shared = BatchSolver(P, capacity=64, lib=emu_lib)
    out = shared.solve(2)
    L = emu_lib.L

    def call(bs, batch, Gs=None, drop=None):
        a = {k: np.ascontiguousarray(out[k]) for k in ("x", "y", "z", "s")}
        ex = np.ascontiguousarray(out["exit"], np.int32)
        ptr = {k: a[k].ctypes.data_as(C.POINTER(C.c_double)) for k in a}
        exp = ex.ctypes.data_as(C.POINTER(C.c_int))
        if drop == "exit":
            exp = None
        elif drop:
            ptr[drop] = None
        return L.eicos_batch_adjoint(bs.h, batch, Gs, None, ptr["x"], ptr["y"], ptr["z"], ptr["s"], exp,
                                     None, None, None, None, None, None, None, None, None)

    assert call(shared, 2) == 0
    assert call(shared, 0) == EICOS_ERR_INVALID
    assert call(shared, -1) == EICOS_ERR_INVALID
    for k in ("x", "z", "s", "exit"):
        assert call(shared, 2, drop=k) == EICOS_ERR_INVALID, k
    Gs = np.tile(np.asarray(P["Gpr"], float), (2, 1))
    assert call(shared, 2, Gs=Gs.ctypes.data_as(C.POINTER(C.c_double))) == EICOS_ERR_INVALID
    with pytest.raises(RuntimeError):
        shared.adjoint(out, Gs=Gs)
    with pytest.raises(ValueError):
        shared.adjoint(out, gx=np.zeros(3))
    with pytest.raises(ValueError):
        shared.adjoint({**out, "x": out["x"][:, :-1]})
    with pytest.raises(ValueError):
        shared.adjoint(out, want=("c", "q"))


def _layer_vs_adjoint(lib, device):
    torch = pytest.importorskip("torch")
    from eicos_b200.autograd import EiCOSLayer
    P = oracle.load_fixture("MPC02")
    W = perturbed_matrices(P, 8, rel=0.01, seed=13)
    bs = BatchSolver(P, capacity=64, lib=lib, instance_matrices=True)
    hs = perturbed(P, 8, rel=MPC_REL, seed=14)["hs"]
    t = {k: torch.tensor(v, dtype=torch.float64, device=device, requires_grad=True) for k, v in (("h", hs), ("G", W["Gs"]))}
    layer = EiCOSLayer(bs)
    x, y, z, ex = layer(h=t["h"], G=t["G"])
    assert not ex.requires_grad
    g = [torch.tensor(v, device=device) for v in _random_g(8, bs.n, bs.p, bs.m, seed=15)]
    loss = (x * g[0]).sum() + (y * g[1]).sum() + (z * g[2]).sum()
    dh, dG = torch.autograd.grad(loss, (t["h"], t["G"]))
    out = bs.solve(8, hs=hs, Gs=W["Gs"])
    for k, v in (("x", x), ("y", y), ("z", z)):
        assert np.array_equal(v.detach().cpu().numpy(), out[k]), k
    ref = bs.adjoint(out, *(v.cpu().numpy() for v in g), Gs=W["Gs"])
    assert np.array_equal(dh.cpu().numpy(), ref["h"])
    assert np.array_equal(dG.cpu().numpy(), ref["G"])
    # inputs left as None get no gradient; a tensor given without requires_grad neither
    c0 = torch.tensor(np.tile(np.asarray(P["c"], float), (8, 1)), device=device)
    x2, _, _, _ = layer(c=c0, h=t["h"])
    (dh2,) = torch.autograd.grad((x2 * g[0]).sum(), (t["h"],))
    assert dh2.shape == t["h"].shape
    return layer, bs, P


def test_torch_layer(emu_lib):
    _layer_vs_adjoint(emu_lib, "cpu")


# ------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@pytest.mark.parametrize("name", WORKLOADS)
def test_gpu_linear_system(gpu_lib, name):
    worst0 = check_linear_system(gpu_lib, name)
    assert worst0 <= RESIDUAL_BOUND.get(name, 1e-9), worst0


@pytest.mark.gpu
def test_gpu_status(gpu_lib):
    check_status(gpu_lib)


@pytest.mark.gpu
def test_gpu_chunking(gpu_lib):
    check_chunking(gpu_lib)


# The two libraries round differently (summation order of the sweeps, FMA contraction); both solves meet the residual
# check, and their difference is that residual times the conditioning of K0.  The SOC MPC's K0 has a condition number
# of 2e11 - 4e13 (measured on the emulator), and the gradients differ by up to 1.1e-5 relative (dG, measured on a B200).
AGREEMENT_BOUND = {"soc_mpc": 1e-4}


@pytest.mark.gpu
@pytest.mark.parametrize("name", WORKLOADS)
def test_gpu_matches_emulator(gpu_lib, emu_lib, name):
    """The same x, y, z, s and g through both libraries: gradients agree to 1e-8 relative per block."""
    P, data, bs, out, g, res = _solve_and_adjoint(gpu_lib, name)
    emu = BatchSolver(P, capacity=64, lib=emu_lib, instance_matrices=bs.instance_matrices)
    ref = emu.adjoint(out, *g, Gs=data.get("Gs"), As=data.get("As"))
    assert np.array_equal(res["status"], ref["status"])
    err = {k: float(np.max(np.abs(res[k] - ref[k])) / max(1.0, np.max(np.abs(ref[k])))) for k in ("c", "h", "b", "G", "A")
           if res[k].size}
    print(f"\n{name}: GPU against emulator, relative difference per block {err}")
    assert max(err.values()) <= AGREEMENT_BOUND.get(name, 1e-8), err


@pytest.mark.gpu
def test_gpu_torch_layer(gpu_lib):
    _layer_vs_adjoint(gpu_lib, "cuda")


@pytest.mark.gpu
def test_gpu_torch_stream_order(gpu_lib):
    """Inputs written by a torch kernel on a side stream just before the call give what a synchronised call gives."""
    torch = pytest.importorskip("torch")
    from eicos_b200.autograd import EiCOSLayer
    P = oracle.load_fixture("MPC02")
    batch = 4096
    hs = torch.tensor(perturbed(P, batch, rel=MPC_REL, seed=16)["hs"], device="cuda")
    bs = BatchSolver(P, capacity=batch, lib=gpu_lib)
    layer = EiCOSLayer(bs)
    g = torch.randn(batch, bs.n, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    h_sync = (hs * 1.0).requires_grad_(True)
    torch.cuda.synchronize()
    x_ref, _, _, _ = layer(h=h_sync)
    (d_ref,) = torch.autograd.grad((x_ref * g).sum(), (h_sync,))
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        h = torch.zeros_like(hs)
        for _ in range(20):  # a queue of work that is still running when the solve is called
            h = h + hs / 20.0
        h = (h - h + hs).requires_grad_(True)
        x, _, _, _ = layer(h=h)
        (d,) = torch.autograd.grad((x * g).sum(), (h,))
        side.synchronize()
    assert torch.equal(x, x_ref)
    assert torch.equal(d, d_ref)


@pytest.mark.gpu
def test_gpu_full_size(gpu_lib):
    """MPC02 x 65 536 device-resident: every optimal instance differentiated with finite gradients; a sample of 64
    instances passes the residual check."""
    torch = pytest.importorskip("torch")
    P = oracle.load_fixture("MPC02")
    batch = 65536
    W = perturbed(P, batch, rel=MPC_REL, seed=17)
    bs = BatchSolver(P, lib=gpu_lib)
    n, m, p = bs.n, bs.m, bs.p
    f = dict(dtype=torch.float64, device="cuda")
    hs, bsv = torch.tensor(W["hs"], **f), torch.tensor(W["bs"], **f)
    x, y, z, s = (torch.empty(batch, k, **f) for k in (n, p, m, m))
    ex = torch.empty(batch, dtype=torch.int32, device="cuda")
    bs.solve_device(batch, d_hs=hs.data_ptr(), d_bs=bsv.data_ptr(), d_x=x.data_ptr(), d_y=y.data_ptr(),
                    d_z=z.data_ptr(), d_s=s.data_ptr(), d_exit=ex.data_ptr())
    gen = torch.Generator("cuda").manual_seed(2)
    g = [torch.randn(batch, k, generator=gen, **f) for k in (n, p, m)]
    out = {k: torch.empty(batch, d, **f) for k, d in (("c", n), ("h", m), ("b", p), ("G", bs.nnzG), ("A", bs.nnzA))}
    st = torch.empty(batch, dtype=torch.int32, device="cuda")
    bs.adjoint_device(batch, d_x=x.data_ptr(), d_y=y.data_ptr(), d_z=z.data_ptr(), d_s=s.data_ptr(), d_exit=ex.data_ptr(),
                      d_gx=g[0].data_ptr(), d_gy=g[1].data_ptr(), d_gz=g[2].data_ptr(), d_dc=out["c"].data_ptr(),
                      d_dh=out["h"].data_ptr(), d_db=out["b"].data_ptr(), d_dG=out["G"].data_ptr(),
                      d_dA=out["A"].data_ptr(), d_status=st.data_ptr())
    exn, stn = ex.cpu().numpy(), st.cpu().numpy()
    opt = (exn == 0) | (exn == 10)
    assert np.all(stn[opt] == 0), np.bincount(stn[opt])
    for k, v in out.items():
        assert bool(torch.isfinite(v).all()), k
    for b in np.random.default_rng(3).choice(batch, 64, replace=False):
        if not opt[b]:
            continue
        xb, yb, zb, sb = (t[b].cpu().numpy() for t in (x, y, z, s))
        K = kkt0(P, xb, yb, zb, sb, np.asarray(P["Gpr"], float), np.asarray(P["Apr"], float))
        u = np.concatenate([-out["c"][b].cpu().numpy(), out["b"][b].cpu().numpy(), out["h"][b].cpu().numpy()])
        gg = np.concatenate([v[b].cpu().numpy() for v in g])
        r = np.abs(K @ u - gg).max() / (np.abs(K).sum(1).max() * np.abs(u).max() + np.abs(gg).max())
        assert r <= 1e-9, (b, r)
