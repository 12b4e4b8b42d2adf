"""Tangents of batched solves (eicos_batch_tangent, BatchSolver.tangent, forward-mode AD through EiCOSLayer).

As in test_adjoint.py the checks are independent of the engine: K0 and the right-hand side
r = [-dc - dA'y - dG'z; db - dA x; dh - dG x] are assembled in numpy from the returned x, y, z, s, and W^2 from its
closed forms.  The dot-product identity <g, J v> = <J'g, v> ties the tangent to the adjoint on every workload, smooth
or not.  The CPU tier runs on the emulator library; the gpu tier repeats the checks on the CUDA library.
"""
import numpy as np
import pytest

import oracle
from eicos_b200.binding import BatchSolver
from eicos_b200.workloads import MPC_REL, perturbed, perturbed_matrices
from test_adjoint import (EICOS_ERR_INVALID, RESIDUAL_BOUND, WORKLOADS, _apex, _dense, _matrices, _random_g, _workload,
                          kkt0, regularisation, w_squared)

BLOCKS = ("c", "h", "b", "G", "A")


def _random_v(bs, batch, seed=7):
    rng = np.random.default_rng(seed)
    dims = {"c": bs.n, "h": bs.m, "b": bs.p, "G": bs.nnzG, "A": bs.nnzA}
    return {k: rng.standard_normal((batch, dims[k])) for k in BLOCKS}


def _tangent(bs, out, v, data):
    return bs.tangent(out, dc=v["c"], dh=v["h"], db=v["b"], dG=v["G"], dA=v["A"], Gs=data.get("Gs"), As=data.get("As"))


def _solve_and_tangent(lib, name, capacity=64):
    P, batch, data, pim = _workload(name)
    bs = BatchSolver(P, capacity=capacity, lib=lib, instance_matrices=pim)
    out = bs.solve(batch, **data)
    v = _random_v(bs, batch)
    return P, data, bs, out, v, _tangent(bs, out, v, data)


def _rhs(P, x, y, z, v, b):
    dG = _dense(P, v["G"][b], "G")
    dA = _dense(P, v["A"][b], "A") if v["A"].size else np.zeros((int(P["p"]), int(P["n"])))
    return np.concatenate([-v["c"][b] - dA.T @ y - dG.T @ z, v["b"][b] - dA @ x, v["h"][b] - dG @ x]), dG


def check_linear_system(lib, name):
    """Per instance: K0 [dx; dy; dz] = r to the accuracy of the regularised solve; ds = -W^2 dz; and the third block
    row G dx + ds = dh - dG x, which holds up to the regularisation the solve adds to the z block."""
    P, data, bs, out, v, res = _solve_and_tangent(lib, name)
    n, p = bs.n, bs.p
    assert np.all(out["exit"] == 0), out["exit"]
    assert np.all(res["status"] == 0), res["status"]
    bound = RESIDUAL_BOUND.get(name, 1e-9)
    worst = {"K0": 0.0, "K0+reg": 0.0, "ds": 0.0, "row3": 0.0}
    for b in range(out["exit"].size):
        x, y, z, s = (out[k][b] for k in "xyzs")
        Gv, Av = _matrices(P, data, b)
        K = kkt0(P, x, y, z, s, Gv, Av)
        r, dG = _rhs(P, x, y, z, v, b)
        u = np.concatenate([res["x"][b], res["y"][b], res["z"][b]])
        reg = regularisation(P, Gv, Av)
        scale = np.abs(K).sum(1).max() * np.abs(u).max() + np.abs(r).max()
        r0 = np.abs(K @ u - r).max() / scale
        rr = np.abs(K @ u + reg * u - r).max() / scale
        # ds against numpy's W^2: on a cone whose z is near its boundary W^2 is large and -W^2 dz cancels, so the
        # difference is measured against |W^2| |dz|
        W = w_squared(P, s, z)
        dz = res["z"][b]
        eds = np.max(np.abs(res["s"][b] + W @ dz) / np.maximum(np.abs(W) @ np.abs(dz), 1e-300))
        # G dx + ds - (dh - dG x) = -reg_z dz (the solve's regularisation), with the returned ds, to the accuracy of
        # the solve: relative to the same scale |K0| |u| + |r| as the residual above
        row3 = _dense(P, Gv, "G") @ res["x"][b] + res["s"][b] + reg[n + p:] * dz - r[n + p:]
        e3 = np.max(np.abs(row3)) / scale
        for k, e in (("K0", r0), ("K0+reg", rr), ("ds", eds), ("row3", e3)):
            worst[k] = max(worst[k], e)
        assert rr <= bound, (b, rr, r0)
        assert eds <= 1e-9, (b, eds)
        assert e3 <= bound, (b, e3)
    print(f"\n{name}: worst relative residuals {({k: f'{e:.1e}' for k, e in worst.items()})}")
    return worst["K0"]


# <g, J v> = <J'g, v>, relative to |g| |Jv| + |J'g| |v|.  Both sides are one regularised solve of the same system, so
# the identity holds to the solves' accuracy times the conditioning of K0.  Measured on the emulator: soc_mpc (condition
# number 2e11 - 4e13) reaches 2.8e-14, issue98 (about 2e10) 2.8e-17, every other workload 3e-17 or less.  soc_mpc's bound
# keeps the room its GPU-against-emulator agreement needs (test_adjoint.AGREEMENT_BOUND).
DOT_BOUND = {"soc_mpc": 1e-10}


def check_dot_product(lib, name):
    P, data, bs, out, v, res = _solve_and_tangent(lib, name)
    batch = out["exit"].size
    g = dict(zip("xyz", _random_g(batch, bs.n, bs.p, bs.m, seed=12)))
    adj = bs.adjoint(out, g["x"], g["y"], g["z"], Gs=data.get("Gs"), As=data.get("As"))
    assert np.all(adj["status"] == 0) and np.all(res["status"] == 0)
    worst = 0.0
    for b in range(batch):
        lhs = sum(g[k][b] @ res[k][b] for k in "xyz")
        rhs = sum(adj[k][b] @ v[k][b] for k in BLOCKS if v[k].size)
        gn = np.sqrt(sum(g[k][b] @ g[k][b] for k in "xyz"))
        jv = np.sqrt(sum(res[k][b] @ res[k][b] for k in "xyz"))
        jtg = np.sqrt(sum(adj[k][b] @ adj[k][b] for k in BLOCKS if v[k].size))
        vn = np.sqrt(sum(v[k][b] @ v[k][b] for k in BLOCKS if v[k].size))
        e = abs(lhs - rhs) / (gn * jv + jtg * vn)
        worst = max(worst, e)
        assert e <= DOT_BOUND.get(name, 1e-9), (b, e)
    print(f"\n{name}: worst |<g, Jv> - <J'g, v>| / (|g||Jv| + |J'g||v|) = {worst:.1e}")


def check_status(lib):
    """MPC02 with h, b +-5 %: non-optimal instances get status 1 and zeros; an instance alone gives the bits it gets in
    the mixed batch; a slack set to 0 gives status 2 and leaves every other instance's bits alone."""
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 24, rel=0.05, seed=4)
    bs = BatchSolver(P, capacity=64, lib=lib)
    out = bs.solve(24, hs=W["hs"], bs=W["bs"])
    opt = (out["exit"] == 0) | (out["exit"] == 10)
    assert opt.any() and (~opt).any(), out["exit"]
    v = _random_v(bs, 24, seed=8)
    res = _tangent(bs, out, v, {})
    assert np.all(res["status"][~opt] == 1)
    assert np.all(res["status"][opt] == 0)
    for k in "xyzs":
        assert np.all(res[k][~opt] == 0.0), k
    for b in np.nonzero(opt)[0][:4]:
        one = {k: out[k][b:b + 1] for k in ("x", "y", "z", "s", "exit")}
        alone = _tangent(bs, one, {k: a[b:b + 1] for k, a in v.items()}, {})
        for k in "xyzs":
            assert np.array_equal(alone[k][0], res[k][b]), (b, k)
    bad = {k: out[k].copy() for k in ("x", "y", "z", "s", "exit")}
    b0 = int(np.nonzero(opt)[0][0])
    bad["s"][b0, 0] = 0.0
    res2 = _tangent(bs, bad, v, {})
    assert res2["status"][b0] == 2
    for k in "xyzs":
        assert np.all(res2[k][b0] == 0.0), k
    keep = np.arange(24) != b0
    for k in ("x", "y", "z", "s", "status"):
        assert np.array_equal(res2[k][keep], res[k][keep]), k
    return res


def check_chunking(lib):
    """capacity 64, batch 200 (four chunks) against one chunk: the same bits."""
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 200, rel=MPC_REL, seed=8)
    big = BatchSolver(P, capacity=256, lib=lib)
    out = big.solve(200, hs=W["hs"], bs=W["bs"])
    v = _random_v(big, 200, seed=9)
    one = _tangent(big, out, v, {})
    four = _tangent(BatchSolver(P, capacity=64, lib=lib), out, v, {})
    for k in ("x", "y", "z", "s", "status"):
        assert np.array_equal(one[k], four[k]), k
    assert np.all(one["status"][out["exit"] == 0] == 0)


# ------------------------------------------------------------------ CPU tier (emulator)
@pytest.mark.parametrize("name", WORKLOADS)
def test_linear_system(emu_lib, name):
    worst0 = check_linear_system(emu_lib, name)
    assert worst0 <= RESIDUAL_BOUND.get(name, 1e-9), worst0


@pytest.mark.parametrize("name", WORKLOADS)
def test_dot_product(emu_lib, name):
    check_dot_product(emu_lib, name)


@pytest.mark.parametrize("pim", [False, True], ids=["shared", "instance_matrices"])
def test_finite_differences(emu_lib, pim):
    """The tangent along v against central differences of (x, y, z) at theta +- eps v, for directions in c, h, b and,
    with per-instance matrices, G and A (one direction per block; one batch call each)."""
    P = oracle.load_fixture("update_data_1")
    batch, eps = 6, 1e-6
    bs = BatchSolver(P, capacity=64, lib=emu_lib, instance_matrices=pim)
    bs.set_settings(feastol=1e-11, abstol=1e-11, reltol=1e-11)
    W = perturbed(P, batch, rel=0.05, seed=21)
    theta = {"cs": np.tile(np.asarray(P["c"], float), (batch, 1)), "hs": W["hs"], "bs": W["bs"]}
    if pim:
        M = perturbed_matrices(P, batch, rel=0.02, seed=22)
        theta["Gs"], theta["As"] = M["Gs"], M["As"]
    theta = {k: a for k, a in theta.items() if a is not None and a.size}
    out = bs.solve(batch, **theta)
    apex = np.array([_apex(P, out["s"][b]) for b in range(batch)])
    rng = np.random.default_rng(6)
    worst = 0.0
    for k, v0 in theta.items():
        dv = rng.standard_normal(v0.shape) * np.abs(v0)
        res = bs.tangent(out, **{"d" + k[0]: dv}, Gs=theta.get("Gs"), As=theta.get("As"))
        st = {kk: np.concatenate([vv, vv]) for kk, vv in theta.items()}
        st[k] = np.concatenate([v0 + eps * dv, v0 - eps * dv])
        o2 = bs.solve(2 * batch, **st)
        ok = (res["status"] == 0) & (o2["exit"][:batch] == 0) & (o2["exit"][batch:] == 0) & ~apex
        assert ok.sum() >= batch // 2, k
        # per instance over (x, y, z) together: at an LP vertex x hardly moves with c while y and z do
        fd = np.concatenate([(o2[blk][:batch] - o2[blk][batch:]) / (2 * eps) for blk in "xyz"], axis=1)
        tg = np.concatenate([res[blk] for blk in "xyz"], axis=1)
        rel = (np.abs(fd - tg).max(1) / np.maximum(np.abs(fd).max(1), np.abs(tg).max(1)))[ok]
        worst = max(worst, rel.max())
        assert np.all(rel <= 1e-3), (k, rel)
    print(f"\n{int(apex.sum())} of {batch} instances excluded (apex); worst relative difference {worst:.2e} (bound 1e-3)")


def test_status(emu_lib):
    check_status(emu_lib)


def test_chunking(emu_lib):
    check_chunking(emu_lib)


def check_workers(lib):
    """The summation order of every row is fixed: the same solutions and direction give the same bits with 4 and 8
    workers per tile."""
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 24, rel=0.05, seed=4)
    out = BatchSolver(P, capacity=64, lib=lib).solve(24, hs=W["hs"], bs=W["bs"])
    v = _random_v(BatchSolver(P, capacity=64, lib=lib), 24, seed=8)
    a, b = (_tangent(BatchSolver(P, capacity=64, lib=lib, workers=w), out, v, {}) for w in (4, 8))
    for k in ("x", "y", "z", "s", "status"):
        assert np.array_equal(a[k], b[k]), k


def test_workers(emu_lib):
    check_workers(emu_lib)


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
        return L.eicos_batch_tangent(bs.h, batch, Gs, None, ptr["x"], ptr["y"], ptr["z"], ptr["s"], exp,
                                     None, None, None, None, None, None, None, None, None, None)

    assert call(shared, 2) == 0
    assert call(shared, 0) == EICOS_ERR_INVALID
    assert call(shared, -1) == EICOS_ERR_INVALID
    for k in ("x", "z", "s", "exit"):
        assert call(shared, 2, drop=k) == EICOS_ERR_INVALID, k
    Gs = np.tile(np.asarray(P["Gpr"], float), (2, 1))
    assert call(shared, 2, Gs=Gs.ctypes.data_as(C.POINTER(C.c_double))) == EICOS_ERR_INVALID
    with pytest.raises(RuntimeError):
        shared.tangent(out, Gs=Gs)
    with pytest.raises(ValueError):
        shared.tangent(out, dc=np.zeros(3))
    with pytest.raises(ValueError):
        shared.tangent(out, dG=np.zeros((2, 3)))
    with pytest.raises(ValueError):
        shared.tangent({**out, "z": out["z"][:, :-1]})
    with pytest.raises(ValueError):
        shared.tangent(out, want=("x", "c"))
    # all five NULL: zeros
    none = shared.tangent(out)
    assert np.all(none["status"] == 0) and all(np.all(none[k] == 0.0) for k in "xyzs")


@pytest.mark.parametrize("pim", [False, True], ids=["shared", "instance_matrices"])
def test_null_equals_zero(emu_lib, pim):
    """A NULL direction component gives the bits of a zero one (dG / dA on both kinds of handle)."""
    P, batch, data, _ = _workload("MPC02_matrices")
    bs = BatchSolver(P, capacity=64, lib=emu_lib, instance_matrices=pim)
    if not pim:
        data = {k: data[k] for k in ("hs", "bs")}
    out = bs.solve(batch, **data)
    v = _random_v(bs, batch, seed=10)
    for k in BLOCKS:
        w = dict(v)
        w[k] = np.zeros_like(v[k])
        zero = _tangent(bs, out, w, data)
        w[k] = None
        null = bs.tangent(out, **{"d" + kk: a for kk, a in w.items()}, Gs=data.get("Gs"), As=data.get("As"))
        for blk in ("x", "y", "z", "s", "status"):
            assert np.array_equal(zero[blk], null[blk]), (k, blk)


def _forward_ad(lib, device):
    torch = pytest.importorskip("torch")
    import torch.autograd.forward_ad as fwAD
    from eicos_b200.autograd import EiCOSLayer
    P = oracle.load_fixture("MPC02")
    W = perturbed_matrices(P, 8, rel=0.01, seed=13)
    bs = BatchSolver(P, capacity=64, lib=lib, instance_matrices=True)
    hs = perturbed(P, 8, rel=MPC_REL, seed=14)["hs"]
    v = _random_v(bs, 8, seed=15)
    f = dict(dtype=torch.float64, device=device)
    th, tG = torch.tensor(hs, **f), torch.tensor(W["Gs"], **f)
    layer = EiCOSLayer(bs)
    out = bs.solve(8, hs=hs, Gs=W["Gs"])
    ref = bs.tangent(out, dh=v["h"], dG=v["G"], Gs=W["Gs"])
    with fwAD.dual_level():
        x, y, z, ex = layer(h=fwAD.make_dual(th, torch.tensor(v["h"], **f)), G=fwAD.make_dual(tG, torch.tensor(v["G"], **f)))
        for k, t in (("x", x), ("y", y), ("z", z)):
            p, tan = fwAD.unpack_dual(t)
            assert np.array_equal(p.cpu().numpy(), out[k]), k
            assert np.array_equal(tan.cpu().numpy(), ref[k]), k
        assert fwAD.unpack_dual(ex).tangent is None
        # a tensor given without a tangent contributes nothing
        c0 = torch.tensor(np.tile(np.asarray(P["c"], float), (8, 1)), **f)
        x2, _, _, _ = layer(c=c0, h=fwAD.make_dual(th, torch.tensor(v["h"], **f)), G=tG)
        only_h = bs.tangent(out, dh=v["h"], Gs=W["Gs"])
        assert np.array_equal(fwAD.unpack_dual(x2).tangent.cpu().numpy(), only_h["x"])
    # reverse mode through the same layer is unchanged
    tr = {k: a.clone().requires_grad_(True) for k, a in (("h", th), ("G", tG))}
    x, y, z, _ = layer(h=tr["h"], G=tr["G"])
    g = [torch.tensor(a, device=device) for a in _random_g(8, bs.n, bs.p, bs.m, seed=16)]
    dh, dG = torch.autograd.grad((x * g[0]).sum() + (y * g[1]).sum() + (z * g[2]).sum(), (tr["h"], tr["G"]))
    adj = bs.adjoint(out, *(a.cpu().numpy() for a in g), Gs=W["Gs"])
    assert np.array_equal(dh.cpu().numpy(), adj["h"])
    assert np.array_equal(dG.cpu().numpy(), adj["G"])


def test_forward_ad(emu_lib):
    _forward_ad(emu_lib, "cpu")


# ------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@pytest.mark.parametrize("name", WORKLOADS)
def test_gpu_linear_system(gpu_lib, name):
    worst0 = check_linear_system(gpu_lib, name)
    assert worst0 <= RESIDUAL_BOUND.get(name, 1e-9), worst0


@pytest.mark.gpu
@pytest.mark.parametrize("name", WORKLOADS)
def test_gpu_dot_product(gpu_lib, name):
    check_dot_product(gpu_lib, name)


@pytest.mark.gpu
def test_gpu_status(gpu_lib):
    check_status(gpu_lib)


@pytest.mark.gpu
def test_gpu_chunking(gpu_lib):
    check_chunking(gpu_lib)


@pytest.mark.gpu
def test_gpu_workers(gpu_lib):
    check_workers(gpu_lib)


# The two libraries round differently in the factorisation and the sweeps; their difference is the solves' residual
# times the conditioning of K0 (the SOC MPC: 2e11 - 4e13), as for the adjoint (test_adjoint.AGREEMENT_BOUND).
AGREEMENT_BOUND = {"soc_mpc": 1e-4}


@pytest.mark.gpu
@pytest.mark.parametrize("name", WORKLOADS)
def test_gpu_matches_emulator(gpu_lib, emu_lib, name):
    P, data, bs, out, v, res = _solve_and_tangent(gpu_lib, name)
    emu = BatchSolver(P, capacity=64, lib=emu_lib, instance_matrices=bs.instance_matrices)
    ref = _tangent(emu, out, v, data)
    assert np.array_equal(res["status"], ref["status"])
    err = {k: float(np.max(np.abs(res[k] - ref[k])) / max(1.0, np.max(np.abs(ref[k])))) for k in "xyzs" if res[k].size}
    print(f"\n{name}: GPU against emulator, relative difference per block {err}")
    assert max(err.values()) <= AGREEMENT_BOUND.get(name, 1e-8), err


@pytest.mark.gpu
def test_gpu_forward_ad(gpu_lib):
    _forward_ad(gpu_lib, "cuda")


@pytest.mark.gpu
def test_gpu_forward_ad_stream_order(gpu_lib):
    """Inputs and tangents written by torch kernels on a side stream just before the call give what a synchronised
    call gives."""
    torch = pytest.importorskip("torch")
    import torch.autograd.forward_ad as fwAD
    from eicos_b200.autograd import EiCOSLayer
    P = oracle.load_fixture("MPC02")
    batch = 4096
    hs = torch.tensor(perturbed(P, batch, rel=MPC_REL, seed=16)["hs"], device="cuda")
    bs = BatchSolver(P, capacity=batch, lib=gpu_lib)
    layer = EiCOSLayer(bs)
    dh = torch.randn(batch, bs.m, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    torch.cuda.synchronize()
    with fwAD.dual_level():
        x_ref, _, _, _ = layer(h=fwAD.make_dual(hs * 1.0, dh * 1.0))
        p_ref, t_ref = (a.clone() for a in fwAD.unpack_dual(x_ref))
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        h, d = torch.zeros_like(hs), torch.zeros_like(dh)
        for _ in range(20):  # a queue of work that is still running when the solve is called
            h, d = h + hs / 20.0, d + dh / 20.0
        h, d = h - h + hs, d - d + dh
        with fwAD.dual_level():
            x, _, _, _ = layer(h=fwAD.make_dual(h, d))
            p, t = (a.clone() for a in fwAD.unpack_dual(x))
        side.synchronize()
    assert torch.equal(p, p_ref)
    assert torch.equal(t, t_ref)


@pytest.mark.gpu
def test_gpu_full_size(gpu_lib):
    """MPC02 x 65 536 device-resident, directions in c, h, b, G and A: every optimal instance has status 0 and finite
    outputs; a sample of 64 instances passes the linear-system check."""
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
    v = {k: torch.randn(batch, d, generator=gen, **f) for k, d in (("c", n), ("h", m), ("b", p), ("G", bs.nnzG), ("A", bs.nnzA))}
    o = {k: torch.empty(batch, d, **f) for k, d in (("x", n), ("y", p), ("z", m), ("s", m))}
    st = torch.empty(batch, dtype=torch.int32, device="cuda")
    bs.tangent_device(batch, d_x=x.data_ptr(), d_y=y.data_ptr(), d_z=z.data_ptr(), d_s=s.data_ptr(), d_exit=ex.data_ptr(),
                      d_dc=v["c"].data_ptr(), d_dh=v["h"].data_ptr(), d_db=v["b"].data_ptr(), d_dG=v["G"].data_ptr(),
                      d_dA=v["A"].data_ptr(), d_ox=o["x"].data_ptr(), d_oy=o["y"].data_ptr(), d_oz=o["z"].data_ptr(),
                      d_os=o["s"].data_ptr(), d_status=st.data_ptr())
    exn, stn = ex.cpu().numpy(), st.cpu().numpy()
    opt = (exn == 0) | (exn == 10)
    assert np.all(stn[opt] == 0), np.bincount(stn[opt])
    for k, a in o.items():
        assert bool(torch.isfinite(a).all()), k
    Gv, Av = np.asarray(P["Gpr"], float), np.asarray(P["Apr"], float)
    for b in np.random.default_rng(3).choice(batch, 64, replace=False):
        if not opt[b]:
            continue
        xb, yb, zb, sb = (t[b].cpu().numpy() for t in (x, y, z, s))
        vb = {k: a[b:b + 1].cpu().numpy() for k, a in v.items()}
        K = kkt0(P, xb, yb, zb, sb, Gv, Av)
        r, _ = _rhs(P, xb, yb, zb, vb, 0)
        u = np.concatenate([o[k][b].cpu().numpy() for k in "xyz"])
        e = np.abs(K @ u + regularisation(P, Gv, Av) * u - r).max() / (np.abs(K).sum(1).max() * np.abs(u).max() + np.abs(r).max())
        assert e <= 1e-9, (b, e)
