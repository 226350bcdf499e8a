"""Host-side mirror of the reference's loss classes (/root/reference/losses.py) over the C ABI.

Same class names, constructor arguments, forward contracts and ``get_last_losses`` tuples:

    Point2Point_Loss / P2P_Loss (losses.py:10-85, 121-129)
    KLD_Loss                    (losses.py:87-118)
    P2PKLD_Loss                 (losses.py:131-145)

and, with no counterpart in the reference (run.py:629-630 only names it as an option), the Chamfer reconstruction loss against a
point set without vertex correspondence: chamfer_distance, Chamfer_Loss, ChamferKLD_Loss (csrc/gin_chamfer.cuh).

The pole averaging (losses.py:22-31,49-51), vertex normals, Laplacian and the three reductions run
as one fused CUDA pipeline (csrc/gin_loss.cuh); the scalar read-backs the reference does with
``.item()`` inside forward are deferred to ``get_last_losses`` so forward itself never syncs.
"""
import torch

from . import _lib
from .ico_conv import get_plan, pixel_strides, _stream, _require_cuda_f32


class _P2PFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inputs, target, level, factors):
        _require_cuda_f32(inputs, 'Point2Point_Loss')
        _require_cuda_f32(target, 'Point2Point_Loss')
        B, C, H, W = inputs.shape
        n = 2 ** level
        V = 10 * 4 ** level + 2
        if C != 3 or H != 5 * n or W != 2 * n:
            raise ValueError('Point2Point_Loss(level %d): expected inputs [B,3,%d,%d], got %s' % (level, 5 * n, 2 * n, tuple(inputs.shape)))
        if tuple(target.shape) != (B, 9, V):
            raise ValueError('Point2Point_Loss: expected target [%d,9,%d], got %s' % (B, V, tuple(target.shape)))
        plan = get_plan(_lib.PLAN_LOSS, level, 1, 'average', inputs.device)
        xs, sb, sp, sc = pixel_strides(inputs)
        tgt = target.contiguous()
        out = torch.empty(4, dtype=torch.float32, device=inputs.device)
        ws = torch.empty(_lib.lib.gin_p2p_ws_bytes(B, level), dtype=torch.uint8, device=inputs.device)
        f_pos, f_nor, f_lap = factors
        _lib.check(_lib.lib.gin_p2p_loss_fwd(plan.host_ptr, plan.dev_ptr, xs.data_ptr(), sb, sp, sc, tgt.data_ptr(),
                                             f_pos, f_nor, f_lap, out.data_ptr(), ws.data_ptr(), B, _stream()), 'gin_p2p_loss_fwd')
        ctx.plan, ctx.strides, ctx.factors, ctx.level = plan, (sb, sp, sc), factors, level
        ctx.save_for_backward(xs, tgt)
        ctx.mark_non_differentiable(out)
        return out[3].clone(), out

    @staticmethod
    def backward(ctx, dloss, _dout):
        xs, tgt = ctx.saved_tensors
        B = xs.shape[0]
        sb, sp, sc = ctx.strides
        dx = torch.empty_strided(xs.shape, xs.stride(), dtype=torch.float32, device=xs.device)
        ws = torch.empty(_lib.lib.gin_p2p_ws_bytes(B, ctx.level), dtype=torch.uint8, device=xs.device)
        g = dloss.reshape(1).contiguous().float()
        f_pos, f_nor, f_lap = ctx.factors
        _lib.check(_lib.lib.gin_p2p_loss_bwd(ctx.plan.host_ptr, ctx.plan.dev_ptr, xs.data_ptr(), sb, sp, sc, tgt.data_ptr(),
                                             f_pos, f_nor, f_lap, g.data_ptr(), dx.data_ptr(), ws.data_ptr(), B, _stream()),
                   'gin_p2p_loss_bwd')
        return dx, None, None, None


class _KLDFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mu, logvar):
        _require_cuda_f32(mu, 'KLD_Loss')
        _require_cuda_f32(logvar, 'KLD_Loss')
        if mu.shape != logvar.shape:
            raise ValueError('KLD_Loss: mu %s and logvar %s differ in shape' % (tuple(mu.shape), tuple(logvar.shape)))
        # the reduction is a plain mean over every element, so any common dense layout works
        if mu.stride() != logvar.stride() or not (mu.is_contiguous() or mu.is_contiguous(memory_format=torch.channels_last)):
            mu, logvar = mu.contiguous(), logvar.contiguous()
        out = torch.empty(1, dtype=torch.float32, device=mu.device)
        ws = torch.empty(4096, dtype=torch.uint8, device=mu.device)
        _lib.check(_lib.lib.gin_kld_fwd(mu.data_ptr(), logvar.data_ptr(), out.data_ptr(), ws.data_ptr(), mu.numel(), _stream()), 'gin_kld_fwd')
        ctx.save_for_backward(mu, logvar)
        return out[0].clone()

    @staticmethod
    def backward(ctx, dout):
        mu, logvar = ctx.saved_tensors
        dmu, dlv = torch.empty_like(mu), torch.empty_like(logvar)
        g = dout.reshape(1).contiguous().float()
        _lib.check(_lib.lib.gin_kld_bwd(mu.data_ptr(), logvar.data_ptr(), g.data_ptr(), 1.0, dmu.data_ptr(), dlv.data_ptr(),
                                        mu.numel(), _stream()), 'gin_kld_bwd')
        return dmu, dlv


class Point2Point_Loss(torch.nn.Module):
    def __init__(self, subdivisions, factor_pos, factor_nor, factor_lap):
        super().__init__()
        self.subdivisions = int(subdivisions)
        self.factor_pos, self.factor_nor, self.factor_lap = float(factor_pos), float(factor_nor), float(factor_lap)
        self._last = None
        self._last_total = None

    def forward(self, inputs, target):
        loss, parts = _P2PFn.apply(inputs, target, self.subdivisions, (self.factor_pos, self.factor_nor, self.factor_lap))
        self._last = parts
        return loss

    def _parts(self):
        if self._last is None:
            return 0., 0., 0., 0.
        return tuple(float(v) for v in self._last.tolist())     # one device->host read

    def get_last_losses(self):
        mse, cos, lap, total = self._parts()
        return mse, cos, lap, total


class KLD_Loss(torch.nn.Module):
    """mean_b( -0.5 * mean_i(1 + logvar - mu^2 - exp(logvar)) )  (losses.py:105; a mean, not the sum of the comment)."""

    def __init__(self):
        super().__init__()
        self.factor_kl = 1.0

    def forward(self, output, target):
        _, mu, logvar = output
        if self.factor_kl:
            self.loss = _KLDFn.apply(mu, logvar)
        else:
            self.loss = torch.tensor(0.)
        return self.loss

    def get_last_losses(self):
        return 0, 0, 0, 0, -self.loss.item()

    def get_factor(self):
        return self.factor_kl

    def update_factor(self, epoch, factor_step_size, factor_gamma):
        if epoch % factor_step_size == 0:
            self.factor_kl *= factor_gamma


class P2P_Loss(Point2Point_Loss):
    def get_last_losses(self):
        mse, cos, lap, total = self._parts()
        return mse, cos, lap, 0., total


class P2PKLD_Loss(P2P_Loss, KLD_Loss):
    def __init__(self, subdivisions, factor_pos, factor_nor, factor_lap, factor_kl):
        P2P_Loss.__init__(self, subdivisions, factor_pos, factor_nor, factor_lap)
        self.factor_kl = factor_kl

    def forward(self, output, target):
        self.kld_loss = KLD_Loss.forward(self, output, target)
        recon, _, _ = output
        self.recons_loss = P2P_Loss.forward(self, recon, target)
        self.loss = self.recons_loss + self.factor_kl * self.kld_loss.to(self.recons_loss.device)
        return self.loss

    def get_last_losses(self):
        return self.recons_loss.item(), 0, 0, -self.kld_loss.item(), self.loss.item()


class _ChamferFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, want_xy, want_yx):
        for name, t in (('x', x), ('y', y)):
            _require_cuda_f32(t, 'chamfer_distance')
            if t.dim() != 3 or t.shape[-1] != 3:
                raise ValueError('chamfer_distance: %s must be [B,n,3], got %s' % (name, tuple(t.shape)))
        if x.shape[0] != y.shape[0]:
            raise ValueError('chamfer_distance: batch sizes differ (%d vs %d)' % (x.shape[0], y.shape[0]))
        B, N, M = x.shape[0], x.shape[1], y.shape[1]
        dev = x.device
        d_xy = torch.empty((B, N), dtype=torch.float32, device=dev) if want_xy else None
        i_xy = torch.empty((B, N), dtype=torch.int32, device=dev) if want_xy else None
        d_yx = torch.empty((B, M), dtype=torch.float32, device=dev) if want_yx else None
        i_yx = torch.empty((B, M), dtype=torch.int32, device=dev) if want_yx else None
        ws = torch.empty(max(1, _lib.lib.gin_chamfer_ws_bytes(B, N, M)), dtype=torch.uint8, device=dev)
        p = lambda t: None if t is None else t.data_ptr()
        _lib.check(_lib.lib.gin_chamfer_fwd(x.data_ptr(), *x.stride(), y.data_ptr(), *y.stride(), p(d_xy), p(i_xy), p(d_yx), p(i_yx),
                                            ws.data_ptr(), B, N, M, _stream()), 'gin_chamfer_fwd')
        ctx.save_for_backward(x, y, i_xy, i_yx)
        ctx.set_materialize_grads(False)
        for t in (i_xy, i_yx):
            if t is not None:
                ctx.mark_non_differentiable(t)
        return d_xy, i_xy, d_yx, i_yx

    @staticmethod
    def backward(ctx, g_xy, _gi_xy, g_yx, _gi_yx):
        x, y, i_xy, i_yx = ctx.saved_tensors
        want_dx, want_dy = ctx.needs_input_grad[:2]
        if (g_xy is None and g_yx is None) or not (want_dx or want_dy):
            return None, None, None, None
        B, N, M = x.shape[0], x.shape[1], y.shape[1]
        g_xy = None if g_xy is None else g_xy.contiguous()
        g_yx = None if g_yx is None else g_yx.contiguous()
        dx = torch.empty((B, N, 3), dtype=torch.float32, device=x.device) if want_dx else None
        dy = torch.empty((B, M, 3), dtype=torch.float32, device=x.device) if want_dy else None
        ws = torch.empty(max(1, _lib.lib.gin_chamfer_ws_bytes(B, N, M)), dtype=torch.uint8, device=x.device)
        p = lambda t: None if t is None else t.data_ptr()
        _lib.check(_lib.lib.gin_chamfer_bwd(x.data_ptr(), *x.stride(), y.data_ptr(), *y.stride(), p(i_xy), p(g_xy), p(i_yx), p(g_yx),
                                            p(dx), p(dy), ws.data_ptr(), B, N, M, _stream()), 'gin_chamfer_bwd')
        return dx, dy, None, None


def chamfer_distance(x, y, xy=True, yx=True):
    """Nearest neighbours between the point sets x [B,N,3] and y [B,M,3] (float32 CUDA, any strides) on the GPU (gin_chamfer_fwd).

    Returns (d_xy [B,N], idx_xy [B,N], d_yx [B,M], idx_yx [B,M]): the squared distance of every point of x to its nearest point of
    y and that point's index (int32; the lowest index among equal distances), and the same from y towards x.  A direction switched
    off with xy=False / yx=False is not computed and returned as None.  Differentiable in x and y through the two distance tensors."""
    if not (xy or yx):
        raise ValueError('chamfer_distance: at least one direction is needed')
    return _ChamferFn.apply(x, y, bool(xy), bool(yx))


def _target_points(target, what):
    """A point set [B,M,3] as is, or the xyz rows of a data-path target [B,9,V] as a [B,V,3] view (no copy)."""
    if target.dim() == 3 and target.shape[-1] == 3:
        return target
    if target.dim() == 3 and target.shape[1] == 9:
        return target[:, :3, :].transpose(1, 2)
    raise ValueError('%s: expected a point set [B,M,3] or a target [B,9,V], got %s' % (what, tuple(target.shape)))


class Chamfer_Loss(torch.nn.Module):
    """Chamfer reconstruction loss between the output vertices and a point set without vertex correspondence:

        mean_b( factor_xy * mean_i d_xy  +  factor_yx * mean_j d_yx )

    with d_xy the squared distance of output vertex i (output2vertices: the grid plus the two averaged poles) to its nearest target
    point and d_yx that of target point j to its nearest output vertex.  `target` is a point set [B,M,3] (a scan, surface samples)
    or the data-path target [B,9,P+2], whose xyz rows are used.  A direction whose factor is 0 is not computed (one-sided loss for
    partial scans).  forward never synchronises with the host."""

    def __init__(self, subdivisions, factor_xy=1.0, factor_yx=1.0):
        super().__init__()
        self.subdivisions = int(subdivisions)
        self.factor_xy, self.factor_yx = float(factor_xy), float(factor_yx)
        if not (self.factor_xy or self.factor_yx):
            raise ValueError('Chamfer_Loss: factor_xy and factor_yx are both 0')
        self._last = None

    def forward(self, inputs, target):
        v = output2vertices(self.subdivisions, inputs)
        y = _target_points(target, 'Chamfer_Loss')
        if y.shape[0] != v.shape[0]:
            raise ValueError('Chamfer_Loss: batch sizes differ (%d vs %d)' % (v.shape[0], y.shape[0]))
        d_xy, _, d_yx, _ = chamfer_distance(v, y, xy=self.factor_xy != 0, yx=self.factor_yx != 0)
        zero = v.new_zeros(())
        l_xy = d_xy.mean() if d_xy is not None else zero
        l_yx = d_yx.mean() if d_yx is not None else zero
        loss = self.factor_xy * l_xy + self.factor_yx * l_yx
        self._last = torch.stack([l_xy, l_yx, loss]).detach()
        return loss

    def get_last_losses(self):
        if self._last is None:
            return 0., 0., 0., 0., 0.
        l_xy, l_yx, total = (float(v) for v in self._last.tolist())     # one device->host read
        return l_xy, l_yx, 0., 0., total


class ChamferKLD_Loss(Chamfer_Loss, KLD_Loss):
    """Chamfer_Loss on the reconstruction plus factor_kl * KLD_Loss, composed as P2PKLD_Loss composes P2P_Loss."""

    def __init__(self, subdivisions, factor_xy, factor_yx, factor_kl):
        Chamfer_Loss.__init__(self, subdivisions, factor_xy, factor_yx)
        self.factor_kl = factor_kl

    def forward(self, output, target):
        self.kld_loss = KLD_Loss.forward(self, output, target)
        recon, _, _ = output
        self.recons_loss = Chamfer_Loss.forward(self, recon, target)
        self.loss = self.recons_loss + self.factor_kl * self.kld_loss.to(self.recons_loss.device)
        return self.loss

    def get_last_losses(self):
        return self.recons_loss.item(), 0, 0, -self.kld_loss.item(), self.loss.item()


def output2vertices(subdivisions, output):
    """ico_utils.py:10-24: [B,C,5n,2n] -> [B,P+2,C] with the two pole vertices appended (row a7)."""
    return _PoleVerticesFn.apply(output, int(subdivisions))


class _PoleVerticesFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, level):
        _require_cuda_f32(x, 'output2vertices')
        B, C, H, W = x.shape
        n = 2 ** level
        if H != 5 * n or W != 2 * n:
            raise ValueError('output2vertices(level %d): expected [B,C,%d,%d], got %s' % (level, 5 * n, 2 * n, tuple(x.shape)))
        plan = get_plan(_lib.PLAN_LOSS, level, 1, 'average', x.device)
        xs, sb, sp, sc = pixel_strides(x)
        v = torch.empty((B, 10 * 4 ** level + 2, C), dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib.gin_pole_vertices_fwd(plan.host_ptr, plan.dev_ptr, xs.data_ptr(), sb, sp, sc, v.data_ptr(), B, C, _stream()),
                   'gin_pole_vertices_fwd')
        ctx.plan, ctx.meta = plan, (xs.shape, xs.stride(), sb, sp, sc)
        return v

    @staticmethod
    def backward(ctx, dv):
        shape, stride, sb, sp, sc = ctx.meta
        dv = dv.contiguous()
        dx = torch.empty_strided(shape, stride, dtype=torch.float32, device=dv.device)
        _lib.check(_lib.lib.gin_pole_vertices_bwd(ctx.plan.host_ptr, ctx.plan.dev_ptr, dv.data_ptr(), dx.data_ptr(), sb, sp, sc,
                                                  shape[0], shape[1], _stream()), 'gin_pole_vertices_bwd')
        return dx, None
