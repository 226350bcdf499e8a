"""Chamfer distance on the GPU (gin_chamfer_fwd / _bwd, losses.chamfer_distance, Chamfer_Loss, ChamferKLD_Loss,
ico_utils.computeDistance(mode='chamfer')): known answers, the float64 oracle, gradients, determinism, graphs, latent fitting."""
import contextlib
import copy
import os
import re

import numpy as np
import pytest
import torch

from geniconet_b200 import _lib, data, ico_utils, losses, models as gm
from geniconet_b200.graph import GraphedStep
from geniconet_b200.optim import Adam
from oracle import chamfer_ref as ref

pytestmark = pytest.mark.gpu
L = _lib.lib


def _cd(x, y, xy=True, yx=True):
    return losses.chamfer_distance(x, y, xy=xy, yx=yx)


def _np(t):
    return t.detach().double().cpu().numpy()


def _check_direction(x, y, d, idx):
    """Reported distance = fp64 distance of the reported pair (1e-6 relative); that pair is within fp32 rounding of the fp64 minimum."""
    xn, yn = _np(x), _np(y)
    idx = idx.long().cpu().numpy()
    assert idx.min() >= 0 and idx.max() < yn.shape[1]
    d_pair = ref.pair_distance(xn, yn, idx)
    d = _np(d)
    assert np.all(np.abs(d - d_pair) <= 1e-6 * d_pair + 1e-30), np.abs(d - d_pair).max()
    d_min, _ = ref.nearest(xn, yn)
    scale = (xn ** 2).sum(-1) + (yn ** 2).sum(-1).max(1, keepdims=True)
    assert np.all(d_pair - d_min <= 2e-6 * scale + 1e-30), (d_pair - d_min).max()


def _check(x, y):
    d_xy, i_xy, d_yx, i_yx = _cd(x, y)
    _check_direction(x, y, d_xy, i_xy)
    _check_direction(y, x, d_yx, i_yx)
    return d_xy, i_xy, d_yx, i_yx


# ------------------------------------------------------------------------------------------------------------- 1. known answers
def test_hand_computed_neighbours():
    x = torch.tensor([[[0., 0., 0.], [1., 0., 0.], [5., 5., 5.]]], device='cuda')
    y = torch.tensor([[[1., 0., 0.], [0., 0., 2.], [4., 5., 5.], [0., 3., 0.]]], device='cuda')
    d_xy, i_xy, d_yx, i_yx = _cd(x, y)
    assert d_xy.tolist() == [[1., 0., 1.]] and i_xy.tolist() == [[0, 0, 2]]
    assert d_yx.tolist() == [[0., 4., 1., 9.]] and i_yx.tolist() == [[1, 0, 2, 0]]


def test_exact_tie_takes_the_lowest_index():
    x = torch.zeros(1, 1, 3, device='cuda')
    y = torch.tensor([[[0., 2., 0.], [1., 0., 0.], [-1., 0., 0.], [0., 0., 1.]]], device='cuda')
    d, i, _, _ = _cd(x, y, yx=False)
    assert d.item() == 1. and i.item() == 1
    # the same tie across candidate tiles and CTA splits (B = 1: the candidates are split over several CTAs)
    M = 9000
    y = torch.full((1, M, 3), 50., device='cuda')
    y[0, 7000] = torch.tensor([0., 0., -0.5])
    y[0, 4100] = torch.tensor([0., 0.5, 0.])
    y[0, 8999] = torch.tensor([0.5, 0., 0.])
    d, i, _, _ = _cd(x, y, yx=False)
    assert d.item() == 0.25 and i.item() == 4100


def test_one_sided_calls():
    g = torch.Generator().manual_seed(3)
    x, y = torch.rand(2, 37, 3, generator=g).cuda(), torch.rand(2, 1000, 3, generator=g).cuda()
    full = _cd(x, y)
    d_xy, i_xy, d_yx, i_yx = _cd(x, y, yx=False)
    assert d_yx is None and i_yx is None
    assert torch.equal(d_xy, full[0]) and torch.equal(i_xy, full[1])
    d_xy, i_xy, d_yx, i_yx = _cd(x, y, xy=False)
    assert d_xy is None and torch.equal(d_yx, full[2]) and torch.equal(i_yx, full[3])
    # the C entry point with the index output left out
    ws = torch.empty(L.gin_chamfer_ws_bytes(2, 37, 1000), dtype=torch.uint8, device='cuda')
    d = torch.empty(2, 37, device='cuda')
    _lib.check(L.gin_chamfer_fwd(x.data_ptr(), *x.stride(), y.data_ptr(), *y.stride(), d.data_ptr(), None, None, None, ws.data_ptr(),
                                 2, 37, 1000, torch.cuda.current_stream().cuda_stream))
    assert torch.equal(d, full[0])


@pytest.mark.parametrize('N', [1, 37])
@pytest.mark.parametrize('M', [5, 1000])
def test_sizes_off_the_tiles(N, M):
    g = torch.Generator().manual_seed(N * 1000 + M)
    x, y = torch.randn(3, N, 3, generator=g).cuda(), torch.randn(3, M, 3, generator=g).cuda()
    _check(x, y)


def test_empty_batch_is_a_no_op():
    x, y = torch.empty(0, 5, 3, device='cuda'), torch.empty(0, 7, 3, device='cuda')
    d_xy, i_xy, d_yx, i_yx = _cd(x, y)
    assert d_xy.shape == (0, 5) and d_yx.shape == (0, 7)


# ------------------------------------------------------------------------------------------------------------- 2. the fp64 oracle
def _mesh(level, B, first=0):
    """[B, P+2, 3] vertices of synthetic level-`level` meshes (the xyz rows of the data-path target)."""
    _, t = data.synthetic_batch(level, first, B)
    return t[:, :3, :].transpose(1, 2).contiguous().cuda()


def _variants(v, seed):
    g = torch.Generator().manual_seed(seed)
    B, V, _ = v.shape
    perm = torch.randperm(V, generator=g).cuda()
    out = {'perturbed': v + 1e-3 * torch.randn(v.shape, generator=g).cuda(),
           'permuted': v[:, perm],
           'subsampled': v[:, perm[: max(1, V // 3)]] + 2e-3 * torch.randn(B, max(1, V // 3), 3, generator=g).cuda()}
    far = v[:, :7] * 30. + 10.
    out['outliers'] = torch.cat([out['perturbed'], far], 1)
    return out


@pytest.mark.parametrize('level,B', [(1, 4), (2, 4), (3, 4), (4, 2), (5, 1)])
def test_against_the_float64_oracle(level, B):
    v = _mesh(level, B)
    for name, y in _variants(v, level).items():
        d_xy, _, d_yx, _ = _check(v, y)
        if name == 'permuted':                                 # every vertex finds itself, at distance exactly 0
            assert torch.count_nonzero(d_xy) == 0 and torch.count_nonzero(d_yx) == 0


def test_benchmarked_size_on_sampled_rows():
    B, level = 36, 5
    v = _mesh(level, B)
    y = _variants(v, 7)['perturbed']
    d_xy, i_xy, d_yx, i_yx = _cd(v, y)
    rows = torch.randperm(v.shape[1], generator=torch.Generator().manual_seed(1))[:192].cuda()
    for a, b, d, i in ((v, y, d_xy, i_xy), (y, v, d_yx, i_yx)):
        q = a[:, rows].double()
        full = torch.stack([((q[s][:, None, :] - b[s].double()[None]) ** 2).sum(-1) for s in range(B)])      # fp64 on the GPU
        dmin = full.min(-1).values
        dpair = full.gather(-1, i[:, rows].long()[..., None])[..., 0]
        assert torch.all((d[:, rows].double() - dpair).abs() <= 1e-6 * dpair + 1e-30)
        scale = (q ** 2).sum(-1) + (b.double() ** 2).sum(-1).max(1, keepdim=True).values
        assert torch.all(dpair - dmin <= 2e-6 * scale)


def test_strided_inputs_read_without_a_copy():
    level, B = 4, 3
    x, t = data.synthetic_batch(level, 0, B)
    t = t.cuda()
    y_view = losses._target_points(t, 'test')                 # xyz rows of [B, 9, V]: strides (9V, 1, V)
    assert y_view.stride() == (9 * t.shape[2], 1, t.shape[2]) and y_view.data_ptr() == t.data_ptr()
    out = (x[:, :3] * 0.9).cuda()                              # an NCHW output and its channels-last twin
    nchw = out.flatten(2).transpose(1, 2)
    cl = out.contiguous(memory_format=torch.channels_last).permute(0, 2, 3, 1).reshape(B, -1, 3)
    ref_out = _cd(nchw.contiguous(), y_view.contiguous())
    for q in (nchw, cl):
        for a, b in zip(_cd(q, y_view), ref_out):
            assert torch.equal(a, b)
    _check(nchw, y_view)


# ------------------------------------------------------------------------------------------------------------- 3. gradients
def _grads(x, y, g_xy, g_yx):
    xg, yg = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    d_xy, i_xy, d_yx, i_yx = _cd(xg, yg, xy=g_xy is not None, yx=g_yx is not None)
    loss = 0.
    if g_xy is not None:
        loss = loss + (d_xy * g_xy).sum()
    if g_yx is not None:
        loss = loss + (d_yx * g_yx).sum()
    loss.backward()
    return xg.grad, yg.grad, i_xy, i_yx


def _rel(a, b):
    return float(np.linalg.norm(_np(a) - b) / max(np.linalg.norm(b), 1e-300))


def _scatter_heavy(N=2000, M=6000, B=2, seed=5):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, N, 3, generator=g)
    y = torch.randn(B, M, 3, generator=g)
    y[:, : M // 2] = x[:, :1] * 3.0 + 0.01 * torch.randn(B, M // 2, 3, generator=g)     # half of y shares one nearest x
    x[:, 0] *= 3.0
    return x.cuda(), y.cuda()


@pytest.mark.parametrize('case', ['mesh', 'scatter_heavy', 'one_sided_xy', 'one_sided_yx'])
def test_gradients_match_the_oracle(case):
    if case == 'mesh':
        x = _mesh(3, 3)
        y = _variants(x, 11)['subsampled']
    else:
        x, y = _scatter_heavy()
    g = torch.Generator().manual_seed(2)
    g_xy = torch.rand(x.shape[:2], generator=g).cuda() if case != 'one_sided_yx' else None
    g_yx = torch.rand(y.shape[:2], generator=g).cuda() if case != 'one_sided_xy' else None
    dx, dy, i_xy, i_yx = _grads(x, y, g_xy, g_yx)
    if case == 'scatter_heavy':
        assert (i_yx[:, : y.shape[1] // 2] == 0).all()
    rx, ry = ref.chamfer_backward(_np(x), _np(y), None if i_xy is None else i_xy.cpu().numpy(), None if i_yx is None else i_yx.cpu().numpy(),
                                  None if g_xy is None else _np(g_xy), None if g_yx is None else _np(g_yx))
    assert _rel(dx, rx) <= 1e-5 and _rel(dy, ry) <= 1e-5, (_rel(dx, rx), _rel(dy, ry))


# ------------------------------------------------------------------------------------------------------------- 4. determinism
@pytest.mark.parametrize('case', ['scatter_heavy', 'split_candidates'])
def test_two_runs_are_bit_identical(case):
    if case == 'scatter_heavy':
        x, y = _scatter_heavy()
    else:                                                      # B = 1, M = 1e5: the candidates are split across CTAs
        x = _mesh(5, 1)
        y = torch.randn(1, 100000, 3, generator=torch.Generator().manual_seed(9)).cuda()
        y = y / y.norm(dim=-1, keepdim=True) * (1 + 0.05 * torch.rand(1, 100000, 1, generator=torch.Generator().manual_seed(8)).cuda())
    gw = torch.Generator().manual_seed(4)
    g_xy, g_yx = torch.rand(x.shape[:2], generator=gw).cuda(), torch.rand(y.shape[:2], generator=gw).cuda()
    runs = []
    for _ in range(2):
        xg, yg = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        d_xy, i_xy, d_yx, i_yx = _cd(xg, yg)
        ((d_xy * g_xy).sum() + (d_yx * g_yx).sum()).backward()
        runs.append((d_xy, i_xy, d_yx, i_yx, xg.grad, yg.grad))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_no_floating_point_atomics_in_the_chamfer_kernels():
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
            if '7chamfer' in current:
                seen.add(current)
            continue
        if current in seen:
            if re.search(r'(REDG?|ATOMG?)\.E\.ADD\.F(16|32|64)|ATOMS\.(CAST|ADD\.F)', line):
                dirty.add(current)
            if re.search(r'(REDG?|ATOMG?)\.E\.(ADD|MIN|MAX)', line):
                integer_atomics.add(current)
    assert len(seen) == 4, sorted(seen)                        # nearest neighbours, scatter exponents, scatter sums, finish
    assert not dirty, sorted(dirty)
    assert len(integer_atomics) == 3, sorted(integer_atomics)   # the detector sees the integer atomics the kernels do use


# ------------------------------------------------------------------------------------------------------------- 5. loss classes
def _oracle_loss(v, y, fxy, fyx):
    d_xy, _, d_yx, _ = ref.chamfer_forward(_np(v), _np(y))
    return fxy * d_xy.mean(1).mean() + fyx * d_yx.mean(1).mean(), d_xy.mean(), d_yx.mean()


@pytest.mark.parametrize('fxy,fyx', [(1.0, 1.0), (0.7, 0.0), (0.0, 2.0)])
def test_chamfer_loss_matches_the_oracle(fxy, fyx):
    level, B = 3, 4
    x, t = data.synthetic_batch(level, 0, B)
    x, t = x.cuda(), t.cuda()
    out = x[:, :3] * 0.95
    crit = losses.Chamfer_Loss(level, fxy, fyx)
    v = losses.output2vertices(level, out)
    pts = _variants(_mesh(level, B, first=1), 3)['subsampled']
    for target, y in ((t, t[:, :3].transpose(1, 2)), (pts, pts)):
        loss = crit(out, target)
        want, lxy, lyx = _oracle_loss(v, y, fxy, fyx)
        assert abs(loss.item() - want) <= 1e-5 * want
        parts = crit.get_last_losses()
        assert len(parts) == 5 and parts[2] == parts[3] == 0.
        assert abs(parts[4] - want) <= 1e-5 * want
        assert (abs(parts[0] - lxy) <= 1e-5 * lxy) if fxy else parts[0] == 0.
        assert (abs(parts[1] - lyx) <= 1e-5 * lyx) if fyx else parts[1] == 0.


def test_chamfer_loss_is_zero_on_a_permutation_of_the_output():
    level, B = 4, 2
    x, _ = data.synthetic_batch(level, 0, B)
    out = (x[:, :3] * 1.1).cuda()
    v = losses.output2vertices(level, out)
    perm = torch.randperm(v.shape[1], generator=torch.Generator().manual_seed(0)).cuda()
    assert losses.Chamfer_Loss(level)(out, v[:, perm].contiguous()).item() == 0.0


def test_chamferkld_is_chamfer_plus_kld():
    level, B = 3, 4
    x, t = data.synthetic_batch(level, 0, B)
    out, t = (x[:, :3] * 0.9).cuda(), t.cuda()
    g = torch.Generator().manual_seed(6)
    mu, lv = (0.3 * torch.randn(B, 512, 5, 2, generator=g)).cuda(), (0.2 * torch.randn(B, 512, 5, 2, generator=g)).cuda()
    fkl = 0.25
    both = losses.ChamferKLD_Loss(level, 1.0, 0.5, fkl)
    loss = both((out, mu, lv), t)
    rec = losses.Chamfer_Loss(level, 1.0, 0.5)(out, t)
    kld = losses.KLD_Loss()((out, mu, lv), t)
    assert torch.equal(loss, rec + fkl * kld)
    r, _, _, k, total = both.get_last_losses()
    assert r == rec.item() and k == -kld.item() and total == loss.item()


def test_compute_distance_modes():
    level = 3
    v = _mesh(level, 2)
    out, refv = v[0], v[1]
    faces = torch.as_tensor(_lib.ico_faces(level))
    got = ico_utils.computeDistance(out, refv, faces, None, mode='chamfer')
    d_xy, _, d_yx, _ = ref.chamfer_forward(_np(out)[None], _np(refv)[None])
    want = d_xy.mean() + d_yx.mean()
    assert abs(float(got) - want) <= 1e-5 * want
    p2m = ico_utils.computeDistance(out, refv, faces, None, mode='point2mesh')
    dist, _ = ico_utils.point_to_mesh_distance(out[None], refv[None], faces)
    assert float(p2m) == float(torch.mean(dist).cpu().numpy())
    assert ico_utils.computeDistance(out, refv, faces, None) is None


# ------------------------------------------------------------------------------------------------------------- 6. integration
def test_graphed_training_step_with_chamfer_replays_like_eager():
    level, B = 3, 4
    params = gm.default_params('ico2ico', level)
    torch.manual_seed(0)
    a = gm.ico2ico(params).cuda().train()
    b = copy.deepcopy(a)
    x, t = data.synthetic_batch(level, 0, B)
    x, t = x.cuda(), t.cuda()

    def make(m):
        crit = losses.Chamfer_Loss(level, 1.0, 0.5)
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


def test_latent_gradient_of_one_sided_chamfer_on_the_frozen_chain():
    level, B = 5, 2
    pv = gm.default_params('ico2ico_vae', level)
    torch.manual_seed(1)
    dec = gm.enc2ico_vae(pv).cuda().train()
    n = 2 ** (level - 3)
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():                                       # non-trivial running statistics
        for _ in range(2):
            dec.decode(torch.randn(B, 512, 5 * n, 2 * n, generator=g).cuda())
    dec.eval()
    for p in dec.parameters():
        p.requires_grad_(False)
    z0 = torch.randn(B, 512, 5 * n, 2 * n, generator=g).cuda()
    scan = _variants(_mesh(level, B), 12)['subsampled']           # a partial scan: one third of the surface, noisy
    crit = losses.Chamfer_Loss(level, 0.0, 1.0)                 # one-sided: every scan point to its nearest output vertex
    grads = {}
    for label, on in (('frozen', True), ('module', False)):
        z = z0.clone().requires_grad_(True)
        with _switch(on, frozen=on):
            crit(dec.decode(z), scan).backward()
        grads[label] = z.grad.double().flatten()
    a, b = grads['frozen'], grads['module']
    cos = (a @ b / (a.norm() * b.norm())).item()
    print('one-sided Chamfer latent gradient, frozen chain vs module path: cosine %.5f' % cos)
    assert cos >= 0.99
