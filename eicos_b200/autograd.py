"""PyTorch autograd layer over a batched solve, its adjoint and its tangent (eicos_batch_solve*_device,
eicos_batch_adjoint_device, eicos_batch_tangent_device).

    layer = EiCOSLayer(BatchSolver(problem))
    x, y, z, exitflag = layer(c=cs, h=hs, b=bs)      # float64 tensors [batch, k]
    loss(x, y, z).backward()                          # cs.grad, hs.grad, bs.grad

Forward mode (torch.autograd.forward_ad) runs the tangent: one call per direction, for every instance at once.

    with fwAD.dual_level():
        x, y, z, _ = layer(h=fwAD.make_dual(hs, dh))
        dx = fwAD.unpack_dual(x).tangent                # derivative of x along dh

Inputs that are not dual contribute nothing and are never read as tangents.  torch.func.jvp is not supported: it
passes tensors without storage to forward(), and the library needs the tensors' memory.

Inputs left as None use the handle's setup data and get no gradient; G / A (per-instance matrix values in CSC order)
need a handle made with instance_matrices=True.  The forward keeps (x, y, z, s, exitflag) for the backward pass; s is
not returned.  Instances whose adjoint status is not 0 (not optimal, not interior, not finite; include/eicos_b200.h)
get zero gradients (and zero tangents).

The library reads and writes the tensors' memory directly: CUDA tensors with the CUDA library, CPU tensors with a
library built for the host.  Before each call the engine's stream waits for the caller's current stream, so work
queued there that produces the inputs is complete first; each call returns after the engine has drained.
"""
import torch

from .binding import PRODUCT_LIB

_NAMES = ("c", "h", "b", "G", "A")


def _ptr(t):
    return 0 if t is None else t.data_ptr()


class EiCOSLayer:
    def __init__(self, solver):
        self.solver = solver
        self.dims = {"c": solver.n, "h": solver.m, "b": solver.p, "G": solver.nnzG, "A": solver.nnzA}

    def _prepare(self, data):
        given = {k: v for k, v in data.items() if v is not None}
        if not given:
            raise ValueError("EiCOSLayer: give at least one of c, h, b, G, A (the batch size comes from them)")
        if ("G" in given or "A" in given) and not self.solver.instance_matrices:
            raise ValueError("EiCOSLayer: G / A need a BatchSolver made with instance_matrices=True")
        first = next(iter(given.values()))
        batch, device = first.shape[0], first.device
        for k, v in given.items():
            if v.dtype != torch.float64 or v.dim() != 2 or v.shape != (batch, self.dims[k]):
                raise ValueError(f"EiCOSLayer: {k} must be a float64 tensor of shape [{batch}, {self.dims[k]}]")
            if v.device != device:
                raise ValueError("EiCOSLayer: all inputs must be on one device")
        if device.type == "cpu" and self.solver.lib.path == PRODUCT_LIB:
            raise ValueError("EiCOSLayer: the CUDA library needs CUDA tensors")
        return batch, device

    def _wait(self, device):
        """Order the engine's stream after the caller's current stream (CUDA tensors only)."""
        if device.type == "cuda":
            engine = torch.cuda.ExternalStream(self.solver.stream(), device=device)
            engine.wait_stream(torch.cuda.current_stream(device))

    def __call__(self, c=None, h=None, b=None, G=None, A=None):
        return _SolveFn.apply(self, c, h, b, G, A)


class _SolveFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, layer, c, h, b, G, A):
        data = dict(zip(_NAMES, (c, h, b, G, A)))
        batch, device = layer._prepare(data)
        data = {k: (None if v is None else v.detach().contiguous()) for k, v in data.items()}
        bs = layer.solver
        f64 = dict(dtype=torch.float64, device=device)
        x, y = torch.empty(batch, bs.n, **f64), torch.empty(batch, bs.p, **f64)
        z, s = torch.empty(batch, bs.m, **f64), torch.empty(batch, bs.m, **f64)
        ex = torch.empty(batch, dtype=torch.int32, device=device)
        layer._wait(device)
        bs.solve_device(batch, d_cs=_ptr(data["c"]), d_hs=_ptr(data["h"]), d_bs=_ptr(data["b"]), d_x=_ptr(x), d_y=_ptr(y),
                        d_z=_ptr(z), d_s=_ptr(s), d_exit=_ptr(ex), d_Gs=_ptr(data["G"]), d_As=_ptr(data["A"]))
        ctx.layer, ctx.batch, ctx.device = layer, batch, device
        ctx.given = tuple(data[k] is not None for k in _NAMES)
        ctx.save_for_backward(x, y, z, s, ex, data["G"], data["A"])
        ctx.save_for_forward(x, y, z, s, ex, data["G"], data["A"])
        # tangents of inputs that are not dual arrive as None (NULL: a G / A stack of zeros is never read); gradients
        # that were not computed also arrive as None, which the adjoint takes as zero
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(ex)
        return x, y, z, ex

    @staticmethod
    def jvp(ctx, _dlayer, dc, dh, db, dG, dA):
        x, y, z, s, ex, G, A = ctx.saved_tensors
        layer, batch, device = ctx.layer, ctx.batch, ctx.device
        bs = layer.solver
        v = [None if t is None else t.contiguous() for t in (dc, dh, db, dG, dA)]
        f64 = dict(dtype=torch.float64, device=device)
        dx, dy, dz = torch.empty(batch, bs.n, **f64), torch.empty(batch, bs.p, **f64), torch.empty(batch, bs.m, **f64)
        layer._wait(device)
        bs.tangent_device(batch, d_x=_ptr(x), d_y=_ptr(y), d_z=_ptr(z), d_s=_ptr(s), d_exit=_ptr(ex),
                          d_dc=_ptr(v[0]), d_dh=_ptr(v[1]), d_db=_ptr(v[2]), d_dG=_ptr(v[3]), d_dA=_ptr(v[4]),
                          d_ox=_ptr(dx), d_oy=_ptr(dy), d_oz=_ptr(dz), d_Gs=_ptr(G), d_As=_ptr(A))
        return dx, dy, dz, None

    @staticmethod
    def backward(ctx, gx, gy, gz, _gex):
        x, y, z, s, ex, G, A = ctx.saved_tensors
        layer, batch, device = ctx.layer, ctx.batch, ctx.device
        bs = layer.solver
        want = [ctx.needs_input_grad[1 + k] and ctx.given[k] for k in range(5)]
        outs = [torch.empty(batch, layer.dims[k], dtype=torch.float64, device=device) if w else None
                for k, w in zip(_NAMES, want)]
        if not any(want):
            return (None,) * 6
        g = [None if v is None else v.contiguous() for v in (gx, gy, gz)]
        layer._wait(device)
        bs.adjoint_device(batch, d_x=_ptr(x), d_y=_ptr(y), d_z=_ptr(z), d_s=_ptr(s), d_exit=_ptr(ex),
                          d_gx=_ptr(g[0]), d_gy=_ptr(g[1]), d_gz=_ptr(g[2]),
                          d_dc=_ptr(outs[0]), d_dh=_ptr(outs[1]), d_db=_ptr(outs[2]), d_dG=_ptr(outs[3]),
                          d_dA=_ptr(outs[4]), d_Gs=_ptr(G), d_As=_ptr(A))
        return (None,) + tuple(outs)
