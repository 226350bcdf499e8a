"""Normal and Laplacian terms of the Chamfer loss on the GPU (gin_chamfer_terms_fwd / _bwd, Chamfer_Loss(factor_nor, factor_lap),
ChamferKLD_Loss): the float64 oracle given the kernel's own indices, equality with P2P_Loss when the target is the output grid,
exact scatter and determinism, no change when the terms are off, a graphed VAE step and latent fitting to a scan with normals."""
import contextlib
import copy
import os
import re

import pytest
import torch

from geniconet_b200 import _lib, data, losses, models as gm
from geniconet_b200.graph import GraphedStep
from geniconet_b200.optim import Adam
from oracle import chamfer_terms_ref as ref

pytestmark = pytest.mark.gpu
TERMS = ('nor_xy', 'nor_yx', 'lap_xy', 'lap_yx')


def _mesh_rows(level, B, first):
    """The data-path target [B, 9, V] of synthetic level-`level` meshes (xyz, normals, Laplacians) on the GPU."""
    _, t = data.synthetic_batch(level, first, B)
    return t.cuda()


def _output_vertices(level, B, seed):
    """Output vertices [B, V, 3]: a synthetic mesh with noise, so n and L differ from any target's."""
    v = _mesh_rows(level, B, 0)[:, :3].transpose(1, 2)
    g = torch.Generator().manual_seed(seed)
    return (v + 5e-3 * torch.randn(v.shape, generator=g).cuda()).contiguous()


def _targets(level, B, seed):
    """The three target layouts: a noisy permuted subset as [B,M,6] and [B,M,9], and the data-path [B,9,V] read in place."""
    t = _mesh_rows(level, B, 7)
    V = t.shape[2]
    g = torch.Generator().manual_seed(seed)
    pick = torch.randperm(V, generator=g)[: max(12, 2 * V // 3)].cuda()
    rows = t.transpose(1, 2)[:, pick].clone()
    rows[..., :3] += 2e-3 * torch.randn(rows[..., :3].shape, generator=g).cuda()
    return {'points6': rows[..., :6].contiguous(), 'points9': rows.contiguous(), 'datapath': t}


def _np64(t):
    return t.detach().double().cpu()


def _run_terms(level, v, target, xy, yx, weights):
    """The four terms and dv of sum_k w_k term_k, with the kernel's own nearest-neighbour indices."""
    y, tn, tl = losses._target_rows(target, 'test')
    _, i_xy, _, i_yx = losses.chamfer_distance(v, y, xy=xy, yx=yx)
    vg = v.clone().requires_grad_(True)
    out = losses._ChamferTermsFn.apply(vg, tn, tl, i_xy, i_yx, level)
    (out * weights).sum().backward()
    return out, vg.grad, (tn, tl, i_xy, i_yx)


def _oracle(level, v, tn, tl, i_xy, i_yx, weights):
    v64 = _np64(v).requires_grad_(True)
    c = lambda t: None if t is None else t.cpu()
    terms = ref.chamfer_terms(level, v64, None if tn is None else _np64(tn), None if tl is None else _np64(tl), c(i_xy), c(i_yx))
    sum(w * t for w, t in zip(weights.double().cpu(), terms)).backward()
    return torch.stack([t.detach() for t in terms]), v64.grad


def _check_grad(got, want):
    err = (got.double().cpu() - want).abs().max().item()
    assert err <= 1e-4 * want.abs().max().item() + 1e-9, (err, want.abs().max().item())


# ------------------------------------------------------------------------------------------------------------- 1. the fp64 oracle
@pytest.mark.parametrize('direction', ['both', 'xy', 'yx'])
@pytest.mark.parametrize('level,B', [(1, 3), (2, 3), (3, 2), (4, 2), (5, 1)])
def test_terms_match_the_float64_oracle(level, B, direction):
    v = _output_vertices(level, B, level)
    weights = torch.tensor([0.7, 1.3, 2.1, 0.4], device='cuda')
    for name, target in _targets(level, B, 10 + level).items():
        out, dv, (tn, tl, i_xy, i_yx) = _run_terms(level, v, target, direction != 'yx', direction != 'xy', weights)
        want, grad = _oracle(level, v, tn, tl, i_xy, i_yx, weights)
        got = out.double().cpu()
        for k in range(4):
            off = (tl is None and k >= 2) or (i_xy is None and k % 2 == 0) or (i_yx is None and k % 2 == 1)
            if off:
                assert got[k] == 0 and want[k] == 0, (name, TERMS[k])
            else:
                assert abs(got[k] - want[k]) <= 2e-5 * abs(want[k]), (name, TERMS[k], got[k].item(), want[k].item())
        _check_grad(dv, grad)


@pytest.mark.parametrize('fxy,fyx', [(1.0, 1.0), (0.6, 0.0), (0.0, 1.0)])
def test_loss_class_combines_the_terms(fxy, fyx):
    level, B = 3, 2
    x, _ = data.synthetic_batch(level, 0, B)
    out = (x[:, :3] * 0.95).cuda()
    target = _targets(level, B, 4)['points9']
    crit = losses.Chamfer_Loss(level, fxy, fyx, factor_nor=0.2, factor_lap=0.3)
    loss = crit(out, target)
    l_xy, l_yx, l_nor, l_lap, total = crit.get_last_losses()
    v = losses.output2vertices(level, out)
    d_xy, i_xy, d_yx, i_yx = losses.chamfer_distance(v, target[..., :3], xy=fxy != 0, yx=fyx != 0)
    t = ref.chamfer_terms(level, _np64(v), _np64(target[..., 3:6]), _np64(target[..., 6:9]),
                          None if i_xy is None else i_xy.cpu(), None if i_yx is None else i_yx.cpu())
    k = (fxy != 0) + (fyx != 0)
    want_nor, want_lap = float(t[0] + t[1]) / k, float(t[2] + t[3]) / k
    assert abs(l_nor - want_nor) <= 2e-5 * want_nor and abs(l_lap - want_lap) <= 2e-5 * want_lap
    pos = fxy * (d_xy.mean().item() if fxy else 0.) + fyx * (d_yx.mean().item() if fyx else 0.)
    want = pos + 0.2 * want_nor + 0.3 * want_lap
    assert abs(total - want) <= 2e-5 * want and total == loss.item()


# ------------------------------------------------------------------------------------------------- 2. the output grid as target
@pytest.mark.parametrize('level,B', [(3, 3), (5, 2)])
def test_output_grid_as_target_gives_p2p_terms(level, B):
    x, _ = data.synthetic_batch(level, 0, B)
    out = (x[:, :3] * 0.9).cuda()
    t = _mesh_rows(level, B, 9).clone()                       # normals and Laplacians of another mesh ...
    t[:, :3] = losses.output2vertices(level, out).transpose(1, 2)   # ... at the output's own vertices
    v = losses.output2vertices(level, out)
    _, i_xy, _, _ = losses.chamfer_distance(v, losses._target_points(t, 'test'), yx=False)
    assert torch.equal(i_xy.long(), torch.arange(v.shape[1], device='cuda').expand(B, -1))
    fn, fl = 0.2, 0.2
    grads, parts = {}, {}
    for label, crit in (('chamfer', losses.Chamfer_Loss(level, 1.0, 0.0, factor_nor=fn, factor_lap=fl)),
                        ('p2p', losses.P2P_Loss(level, 1.0, fn, fl))):
        xg = out.clone().requires_grad_(True)
        crit(xg, t).backward()
        grads[label], parts[label] = xg.grad, crit.get_last_losses()
    c, p = parts['chamfer'], parts['p2p']
    assert c[0] == 0. and p[0] == 0.                          # the position terms vanish on both sides
    for got, want in ((c[2], p[1]), (c[3], p[2]), (c[4], p[4])):
        assert abs(got - want) <= 2e-5 * abs(want), (got, want)
    want = grads['p2p'].double()
    err = (grads['chamfer'].double() - want).abs().max().item()
    assert err <= 1e-4 * want.abs().max().item() + 1e-9, err


# -------------------------------------------------------------------------------------------- 3. exact scatter and determinism
def _scatter_heavy(level=3, B=2, M=6000, seed=5):
    """Half of the target points share one nearest output vertex (vertex 5)."""
    v = _output_vertices(level, B, 1)
    g = torch.Generator().manual_seed(seed)
    far = _mesh_rows(level, B, 3)[:, :3].transpose(1, 2)
    pick = torch.randint(0, far.shape[1], (M - M // 2,), generator=g).cuda()
    pts = torch.cat([v[:, 5:6] + 1e-4 * torch.randn(B, M // 2, 3, generator=g).cuda(),
                     far[:, pick] + 1e-3 * torch.randn(B, M - M // 2, 3, generator=g).cuda()], 1)
    tn = torch.randn(B, M, 3, generator=g).cuda()
    tl = 1e-2 * torch.randn(B, M, 3, generator=g).cuda()
    return v, torch.cat([pts, tn, tl], -1).contiguous()


def test_scatter_heavy_gradient_matches_the_oracle():
    level = 3
    v, target = _scatter_heavy(level)
    weights = torch.tensor([0.0, 1.7, 0.0, 2.3], device='cuda')
    out, dv, (tn, tl, i_xy, i_yx) = _run_terms(level, v, target, False, True, weights)
    assert (i_yx[:, : target.shape[1] // 2] == 5).all()
    want, grad = _oracle(level, v, tn, tl, i_xy, i_yx, weights)
    assert torch.allclose(out.double().cpu(), want, rtol=2e-5, atol=0)
    _check_grad(dv, grad)


def test_two_runs_are_bit_identical():
    level = 3
    v, target = _scatter_heavy(level)
    weights = torch.tensor([0.3, 1.7, 0.9, 2.3], device='cuda')
    runs = [_run_terms(level, v, target, True, True, weights)[:2] for _ in range(2)]
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_no_floating_point_atomics_in_the_terms_kernels():
    import shutil
    import subprocess
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    sass = subprocess.run([cuobjdump, '-sass', _lib.LIB_PATH], capture_output=True, text=True).stdout
    current, seen, dirty, integer_atomics = None, set(), set(), set()
    for line in sass.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            current = m.group(1)
            if '13chamfer_terms' in current:
                seen.add(current)
            continue
        if current in seen:
            if re.search(r'(REDG?|ATOMG?)\.E\.ADD\.F(16|32|64)|ATOMS\.(CAST|ADD\.F)', line):
                dirty.add(current)
            if re.search(r'(REDG?|ATOMG?)\.E\.(ADD|MIN|MAX)', line):
                integer_atomics.add(current)
    assert len(seen) == 5, sorted(seen)                        # forward, final, two scatter passes, cotangents
    assert not dirty, sorted(dirty)
    assert len(integer_atomics) == 2, sorted(integer_atomics)   # the two scatter passes


# -------------------------------------------------------------------------------------------------------- 4. no change when off
@pytest.mark.parametrize('fxy,fyx', [(1.0, 1.0), (0.7, 0.0), (0.0, 2.0)])
def test_terms_off_is_the_position_only_composition(fxy, fyx):
    level, B = 4, 3
    x, t = data.synthetic_batch(level, 0, B)
    out, t = (x[:, :3] * 0.9).cuda(), t.cuda()
    res = {}
    for label in ('class', 'composed'):
        xg = out.clone().requires_grad_(True)
        n0 = _lib.launch_count()
        if label == 'class':
            loss = losses.Chamfer_Loss(level, fxy, fyx, factor_nor=0.0, factor_lap=0.0)(xg, t)
        else:
            v = losses.output2vertices(level, xg)
            d_xy, _, d_yx, _ = losses.chamfer_distance(v, losses._target_points(t, 'test'), xy=fxy != 0, yx=fyx != 0)
            zero = v.new_zeros(())
            loss = fxy * (d_xy.mean() if d_xy is not None else zero) + fyx * (d_yx.mean() if d_yx is not None else zero)
        loss.backward()
        res[label] = (loss, xg.grad, _lib.launch_count() - n0)
    (la, ga, na), (lb, gb, nb) = res['class'], res['composed']
    assert torch.equal(la, lb) and torch.equal(ga, gb) and na == nb


# ---------------------------------------------------------------------------------------------------------- 5. missing target rows
def test_missing_target_rows_raise():
    level, B = 2, 2
    x, t = data.synthetic_batch(level, 0, B)
    out, t = x[:, :3].cuda(), t.cuda()
    pts = t.transpose(1, 2).contiguous()
    with pytest.raises(ValueError, match='normals'):
        losses.Chamfer_Loss(level, factor_nor=0.2)(out, pts[..., :3])
    with pytest.raises(ValueError, match='Laplacians'):
        losses.Chamfer_Loss(level, factor_lap=0.2)(out, pts[..., :6])
    with pytest.raises(ValueError, match='Laplacians'):
        mu = torch.zeros(B, 512, 5, 2, device='cuda')
        losses.ChamferKLD_Loss(level, 1.0, 1.0, 0.1, factor_lap=0.2)((out, mu, mu), pts[..., :3])
    with pytest.raises(ValueError, match='expected'):
        losses.Chamfer_Loss(level)(out, pts[..., :5])
    losses.Chamfer_Loss(level, factor_nor=0.2)(out, pts[..., :6])     # normals suffice for the normal term
    losses.Chamfer_Loss(level, factor_nor=0.2, factor_lap=0.2)(out, t)


# ------------------------------------------------------------------------------------------------------------- 6. integration
def test_graphed_vae_training_step_with_the_terms_replays_like_eager():
    level, B = 5, 4
    params = gm.default_params('ico2ico_vae', level)
    torch.manual_seed(0)
    a = gm.ico2ico_vae(params).cuda().train()
    b = copy.deepcopy(a)
    x, t = data.synthetic_batch(level, 0, B)
    x, t = x.cuda(), t.cuda()
    n = 2 ** (level - 3)
    eps = torch.randn(B, 512, 5 * n, 2 * n, generator=torch.Generator().manual_seed(3)).cuda()

    def make(m):
        # one fixed noise draw for both runs: the graph's device-side noise counter advances differently from eager draws
        m.reparameterize = lambda mu, logvar: mu + eps * torch.exp(0.5 * logvar)
        crit = losses.ChamferKLD_Loss(level, 0.6, 0.6, 1e-3, factor_nor=0.2, factor_lap=0.2)
        opt = Adam(m.parameters(), lr=1e-4)
        opt.prepare()

        def step(xs, ts):
            for p in m.parameters():
                if p.grad is not None:
                    p.grad.zero_()
            loss = crit(m(xs), ts)
            loss.backward()
            opt.step()
            return loss
        return step
    sa = make(a)
    for _ in range(3 + 4):                                      # GraphedStep's three warm-up steps, then four replays
        sa(x, t)
    graphed = GraphedStep(make(b), (x, t), warmup=3)
    for _ in range(4):
        graphed()
    torch.cuda.synchronize()
    for (k, p), q in zip(a.named_parameters(), b.parameters()):
        assert torch.equal(p, q), k
    for (k, p), q in zip(a.named_buffers(), b.buffers()):
        assert torch.equal(p, q), k


@contextlib.contextmanager
def _switch(fused_on, frozen):
    saved = gm._FUSED, gm._HEAD, gm._INFER, gm._FROZEN
    gm.set_fused(fused_on, frozen=frozen)
    try:
        yield
    finally:
        gm._FUSED, gm._HEAD, gm._INFER, gm._FROZEN = saved


def test_latent_gradient_of_a_one_sided_normal_term_on_the_frozen_chain():
    level = 5
    pv = gm.default_params('ico2ico_vae', level)
    torch.manual_seed(1)
    dec = gm.enc2ico_vae(pv).cuda().train()
    n = 2 ** (level - 3)
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():                                       # non-trivial running statistics
        for _ in range(2):
            dec.decode(torch.randn(2, 512, 5 * n, 2 * n, generator=g).cuda())
    dec.eval()
    for p in dec.parameters():
        p.requires_grad_(False)
    z0 = torch.randn(1, 512, 5 * n, 2 * n, generator=g).cuda()
    scan = _targets(level, 1, 12)['points6']                    # a partial scan with normals: two thirds of a surface, noisy
    crit = losses.Chamfer_Loss(level, 0.0, 1.0, factor_nor=0.5)  # one-sided: every scan point to its nearest output vertex
    grads = {}
    for label, on in (('frozen', True), ('module', False)):
        z = z0.clone().requires_grad_(True)
        with _switch(on, frozen=on):
            crit(dec.decode(z), scan).backward()
        grads[label] = z.grad.double().flatten()
    a, b = grads['frozen'], grads['module']
    cos = (a @ b / (a.norm() * b.norm())).item()
    print('one-sided Chamfer + normal term latent gradient, frozen chain vs module path: cosine %.5f' % cos)
    assert cos >= 0.99
