"""Batched MPC solves as a differentiable PyTorch operation (not reference behaviour).

    out8, traj, obj, status = udacitympc_b200.autograd.solve(mpc, states, coeffs, cost_params=None, model_params=None)

The forward pass is one batched solve (b200mpc_solve_batch_warm[_device] from the default start point, which also
returns the multipliers); the backward pass is one adjoint solve at that solution (b200mpc_solve_batch_vjp[_device]).
With cost_params the two calls are b200mpc_solve_batch_cost[_device] and b200mpc_solve_batch_vjp_cost[_device], with
model_params b200mpc_solve_batch_model[_device] and b200mpc_solve_batch_vjp_model[_device].  Forward-mode AD
(torch.autograd.forward_ad) runs one tangent solve at the solution (b200mpc_solve_batch_jvp[_device]).
CUDA tensors stay on the device and run on torch's current stream of their device, which must be the MPC handle's
device; CPU tensors go through the host entry points.  The only module of the package that imports torch.
"""
import torch

__all__ = ["solve"]


def _ptr(t):
    return t.data_ptr() if t is not None else 0


def _stream(dev):
    """torch's current stream on dev as the library's stream argument.  torch's default stream is the legacy default
    stream, handle 0, which the library reads as "the handle's own stream": pass cudaStreamLegacy (1) for it instead, so
    the library's work is ordered with torch's."""
    return torch.cuda.current_stream(dev).cuda_stream or 1


def _fields(t):
    """(B, k) -> the field-major (k, B) float64 buffer the device entry points take."""
    return t.detach().to(torch.float64).t().contiguous()


def _rows(t, B, k, name):
    """(B, k) or (k,) -> the (B, k) float64 rows, or None."""
    if t is None:
        return None
    if t.shape not in ((k,), (B, k)):
        raise ValueError(f"{name} must be (B, {k}) or ({k},)")
    return t.detach().to(torch.float64).expand(B, k)


class _Solve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mpc, states, coeffs, cost_params, model_params):
        B = states.shape[0]
        shared = coeffs.dim() == 1
        cf = coeffs.detach().to(torch.float64).expand(B, -1) if shared else coeffs.detach().to(torch.float64)
        st = states.detach().to(torch.float64)
        c8 = _rows(cost_params, B, 8, "cost_params")
        m4 = _rows(model_params, B, 4, "model_params")
        nv, nm = mpc.num_vars, mpc.num_mults
        if states.is_cuda:
            if states.device.index != mpc.device or coeffs.device != states.device or any(
                    r is not None and r.device != states.device for r in (c8, m4)):
                raise ValueError(f"states / coeffs / cost_params / model_params must be on cuda:{mpc.device}, the MPC "
                                 "handle's device")
            dev = states.device
            st_f, cf_f = _fields(st), _fields(cf)
            out8 = torch.empty(8, B, dtype=torch.float64, device=dev)
            traj = torch.empty(nv, B, dtype=torch.float64, device=dev)
            mult = torch.empty(nm, B, dtype=torch.float64, device=dev)
            obj = torch.empty(B, dtype=torch.float64, device=dev)
            status = torch.empty(B, dtype=torch.int32, device=dev)
            if m4 is not None:
                c8_f, m4_f = None if c8 is None else _fields(c8), _fields(m4)
                mpc.solve_batch_model_device(B, _ptr(st_f), _ptr(cf_f), cf.shape[1], _ptr(c8_f), _ptr(m4_f), 0, 0, 0.0,
                                             _ptr(out8), _ptr(traj), _ptr(mult), _ptr(obj), _ptr(status), 0, _stream(dev))
            elif c8 is None:
                mpc.solve_batch_warm_device(B, _ptr(st_f), _ptr(cf_f), cf.shape[1], 0, 0, 0.0, _ptr(out8), _ptr(traj),
                                            _ptr(mult), _ptr(obj), _ptr(status), 0, _stream(dev))
            else:
                c8_f = _fields(c8)
                mpc.solve_batch_cost_device(B, _ptr(st_f), _ptr(cf_f), cf.shape[1], _ptr(c8_f), 0, 0, 0.0, _ptr(out8),
                                            _ptr(traj), _ptr(mult), _ptr(obj), _ptr(status), 0, _stream(dev))
            out8, traj, mult = out8.t(), traj.t(), mult.t()
        else:
            r = mpc.solve_batch(st.numpy(), cf.contiguous().numpy(), want_traj=True, want_mult=True,
                                cost_params=None if c8 is None else c8.contiguous().numpy(),
                                model_params=None if m4 is None else m4.contiguous().numpy())
            out8, traj, mult = torch.from_numpy(r["out8"]), torch.from_numpy(r["traj"]), torch.from_numpy(r["mult"])
            obj, status = torch.from_numpy(r["cost"]), torch.from_numpy(r["status"])
        ctx.mpc, ctx.shared = mpc, shared
        ctx.dtypes = tuple(None if t is None else t.dtype for t in (states, coeffs, cost_params, model_params))
        ctx.cost_shared = cost_params is not None and cost_params.dim() == 1
        ctx.model_shared = model_params is not None and model_params.dim() == 1
        ctx.save_for_backward(st, cf, traj, mult, status, c8, m4)
        ctx.save_for_forward(st, cf, traj, mult, status, c8, m4)
        ctx.mark_non_differentiable(status)
        dt = states.dtype
        return out8.to(dt), traj.to(dt), obj.to(dt), status

    @staticmethod
    def backward(ctx, g_out8, g_traj, g_obj, _g_status):
        st, cf, traj, mult, status, c8, m4 = ctx.saved_tensors
        mpc = ctx.mpc
        B, ncoef = cf.shape
        g = [None if v is None else v.detach().to(torch.float64) for v in (g_out8, g_traj, g_obj)]
        gp = gm = None
        if st.is_cuda:
            dev = st.device
            gs = torch.empty(6, B, dtype=torch.float64, device=dev)
            gc = torch.empty(ncoef, B, dtype=torch.float64, device=dev)
            vs = torch.empty(B, dtype=torch.int32, device=dev)
            keep = [_fields(st), _fields(cf), traj.t().contiguous(), mult.t().contiguous(),
                    None if g[0] is None else _fields(g[0]), None if g[1] is None else _fields(g[1]),
                    None if g[2] is None else g[2].contiguous()]
            if m4 is not None:
                c8_f, m4_f = None if c8 is None else _fields(c8), _fields(m4)
                gp = None if c8 is None else torch.empty(8, B, dtype=torch.float64, device=dev)
                gm = torch.empty(4, B, dtype=torch.float64, device=dev)
                mpc.solve_batch_vjp_model_device(B, *[_ptr(k) for k in keep[:2]], ncoef, _ptr(c8_f), _ptr(m4_f),
                                                 *[_ptr(k) for k in keep[2:]], _ptr(gs), _ptr(gc), _ptr(gp), _ptr(gm),
                                                 _ptr(vs), _stream(dev))
                gp = None if gp is None else gp.t()
                gm = gm.t()
            elif c8 is None:
                mpc.solve_batch_vjp_device(B, *[_ptr(k) for k in keep[:2]], ncoef, *[_ptr(k) for k in keep[2:]], _ptr(gs),
                                           _ptr(gc), 0, _ptr(vs), _stream(dev))
            else:
                c8_f = _fields(c8)
                gp = torch.empty(8, B, dtype=torch.float64, device=dev)
                mpc.solve_batch_vjp_cost_device(B, *[_ptr(k) for k in keep[:2]], ncoef, _ptr(c8_f),
                                                *[_ptr(k) for k in keep[2:]], _ptr(gs), _ptr(gc), _ptr(gp), _ptr(vs),
                                                _stream(dev))
                gp = gp.t()
            gs, gc = gs.t(), gc.t()
        else:
            r = mpc.solve_batch_vjp(st.numpy(), cf.contiguous().numpy(), traj.numpy(), mult.numpy(),
                                    *[None if v is None else v.numpy() for v in g], want_params=c8 is not None,
                                    cost_params=None if c8 is None else c8.contiguous().numpy(),
                                    model_params=None if m4 is None else m4.contiguous().numpy(), want_model=m4 is not None)
            gs, gc = torch.from_numpy(r["grad_state6"]), torch.from_numpy(r["grad_coeffs"])
            if c8 is not None:
                gp = torch.from_numpy(r["grad_params"])
            if m4 is not None:
                gm = torch.from_numpy(r["grad_model"])
        # the derivative exists only at a converged solution
        bad = ~((status == 0) | (status == 1))
        gs = gs.masked_fill(bad[:, None], float("nan"))
        gc = gc.masked_fill(bad[:, None], float("nan"))
        if ctx.shared:
            gc = gc.sum(0)
        if gp is not None:
            gp = gp.masked_fill(bad[:, None], float("nan"))
            if ctx.cost_shared:
                gp = gp.sum(0)
            gp = gp.to(ctx.dtypes[2])
        if gm is not None:
            gm = gm.masked_fill(bad[:, None], float("nan"))
            if ctx.model_shared:
                gm = gm.sum(0)
            gm = gm.to(ctx.dtypes[3])
        return None, gs.to(ctx.dtypes[0]), gc.to(ctx.dtypes[1]), gp, gm

    @staticmethod
    def jvp(ctx, _t_mpc, t_states, t_coeffs, t_cost, t_model):
        st, cf, traj, mult, status, c8, m4 = ctx.saved_tensors
        mpc = ctx.mpc
        B, ncoef = cf.shape
        shapes = ((B, 6), (B, ncoef), (B, 8), (B, 4))
        t = [None if v is None else v.detach().to(torch.float64).expand(*s) for v, s in
             zip((t_states, t_coeffs, t_cost, t_model), shapes)]
        dt = ctx.dtypes[0]
        # the derivative exists only at a converged solution.  The tangents are masked in place and keep the layout of
        # their primal outputs (on CUDA, transposes of field-major buffers), which forward-mode AD requires.
        bad = ~((status == 0) | (status == 1))
        nan = float("nan")
        if st.is_cuda:
            dev = st.device
            to8 = torch.empty(8, B, dtype=torch.float64, device=dev)
            tt = torch.empty(mpc.num_vars, B, dtype=torch.float64, device=dev)
            tob = torch.empty(B, dtype=torch.float64, device=dev)
            vs = torch.empty(B, dtype=torch.int32, device=dev)
            keep = [_fields(st), _fields(cf), None if c8 is None else _fields(c8), None if m4 is None else _fields(m4),
                    traj.t().contiguous(), mult.t().contiguous()] + [None if v is None else _fields(v) for v in t]
            mpc.solve_batch_jvp_device(B, _ptr(keep[0]), _ptr(keep[1]), ncoef, *[_ptr(k) for k in keep[2:]], _ptr(to8),
                                       _ptr(tt), _ptr(tob), _ptr(vs), _stream(dev))
            to8, tt = to8.masked_fill_(bad[None, :], nan).t(), tt.masked_fill_(bad[None, :], nan).t()
        else:
            r = mpc.solve_batch_jvp(st.numpy(), cf.contiguous().numpy(), traj.numpy(), mult.numpy(),
                                    *[None if v is None else v.contiguous().numpy() for v in t],
                                    cost_params=None if c8 is None else c8.contiguous().numpy(),
                                    model_params=None if m4 is None else m4.contiguous().numpy())
            to8, tt, tob = (torch.from_numpy(r[k]) for k in ("t_out8", "t_traj", "t_obj"))
            to8, tt = to8.masked_fill_(bad[:, None], nan), tt.masked_fill_(bad[:, None], nan)
        tob.masked_fill_(bad, nan)
        return to8.to(dt), tt.to(dt), tob.to(dt), None


def solve(mpc, states, coeffs, cost_params=None, model_params=None):
    """Differentiable batched solve on the MPC handle `mpc`: states (B, 6), coeffs (B, ncoef) or (ncoef,) shared by all
    problems, torch tensors on the CPU or on the handle's CUDA device.  cost_params (B, 8) or (8,) shared, in the order
    PARAM_NAMES (ref_v, w_cte, w_epsi, w_v, w_delta, w_a, w_ddelta, w_da), on the same device, replaces the handle's
    cost parameters problem by problem (None: the handle's, not differentiated).  Returns (out8 (B, 8), traj (B, 8N-2),
    obj (B,), status (B,) int32, not differentiable).  Backpropagating into states / coeffs / cost_params runs one
    adjoint solve (MPC.solve_batch_vjp); problems whose status is not 0 or 1 get NaN gradients, and gradients of shared
    coeffs / cost_params are summed over the batch.  model_params (B, 4) or (4,) shared, in the order MODEL_NAMES (dt, Lf,
    delta_max, a_max), likewise replaces the handle's vehicle model and actuator limits and is differentiated.
    Forward-mode AD (torch.autograd.forward_ad) through the solve runs one tangent solve (MPC.solve_batch_jvp) per
    call: tangents of out8, traj and obj, NaN for problems whose status is not 0 or 1; tangents of shared coeffs /
    cost_params / model_params apply to every problem."""
    return _Solve.apply(mpc, states, coeffs, cost_params, model_params)
