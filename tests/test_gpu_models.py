"""GPU parity of the whole graphs (run with -m gpu): ico2ico / ico2ico_vae through the CUDA layers vs the
same graph over the CPU oracle layers, same weights, same inputs (SURVEY 4.2 item 7)."""
import pytest
import torch

import oracle_models as om

pytestmark = pytest.mark.gpu


def _grads(model):
    return {k: p.grad.detach().cpu().clone() for k, p in model.named_parameters() if p.grad is not None}


def _compare_grads(gc, gr, cos_min, what):
    assert set(gc) == set(gr)
    worst = 1.0
    for k in gr:
        a, b = gc[k].flatten().double(), gr[k].flatten().double()
        if b.norm() < 1e-6:          # e.g. conv biases in front of a BatchNorm: the true gradient is zero, both sides are rounding noise
            continue
        cos = (a @ b / (a.norm() * b.norm())).item()
        worst = min(worst, cos)
        assert cos >= cos_min, '%s: gradient cosine of %s = %.5f' % (what, k, cos)
    return worst


# Measured on B200 (tests/diag/diag_parity.py, profiles/r01_parity_by_layer.txt): the fp32 CUDA-core path tracks the fp32
# oracle to 4e-6 on activations and cosine 1.000000 on every gradient; the tcgen05 path rounds every conv operand to
# bf16, which accumulates to 2e-2 on the output and, through 25 layers of backward at batch 2, to cosine 0.984 on the
# first layer's weight gradient (0.996 at batch 8).  Tolerances below are those measurements with ~2x head-room.
@pytest.mark.parametrize('impl,loss_tol,cos_min', [('simt', 2e-4, 0.9995), ('auto', 2e-2, 0.97)])
def test_ico2ico_step_matches_oracle(impl, loss_tol, cos_min):
    from geniconet_b200 import models as gm, losses, data
    from geniconet_b200.ico_conv import set_impl
    level, B = 5, 2
    torch.backends.cudnn.allow_tf32 = False      # the stock 1x1 Conv2d head (models.py:151) would otherwise run in TF32
    torch.backends.cuda.matmul.allow_tf32 = False
    params = gm.default_params('ico2ico', level)
    ref = om.fill_params_deterministic(om.build_oracle_model('ico2ico', params))
    mod = gm.ico2ico(params)
    mod.load_state_dict(ref.state_dict())
    mod = set_impl(mod.cuda(), impl)
    x, tgt = data.synthetic_batch(level, 0, B)
    out_r = ref(x)
    loss_r, _ = om.ref_p2p_loss(level, out_r, tgt, 1., 0., 0.)
    loss_r.backward()
    crit = losses.P2P_Loss(level, 1., 0., 0.)
    out_c = mod(x.cuda())
    assert out_c.shape == out_r.shape
    loss_c = crit(out_c, tgt.cuda())
    loss_c.backward()
    torch.cuda.synchronize()
    assert abs(loss_c.item() - loss_r.item()) <= loss_tol * abs(loss_r.item()), (loss_c.item(), loss_r.item())
    rel = ((out_c.detach().cpu() - out_r.detach()).norm() / out_r.detach().norm()).item()
    assert rel <= (1e-4 if impl == 'simt' else 5e-2), rel          # measured: 3e-5 (fp32 path), 2e-2 (bf16 operands)
    _compare_grads(_grads(mod), _grads(ref), cos_min, impl)


def test_ico2ico_vae_step_matches_oracle():
    from geniconet_b200 import models as gm, losses, data
    from geniconet_b200.ico_conv import set_impl
    from geniconet_b200 import reparam
    level, B = 5, 2
    torch.backends.cudnn.allow_tf32 = False
    params = gm.default_params('ico2ico_vae', level)
    ref = om.fill_params_deterministic(om.build_oracle_model('ico2ico_vae', params))
    mod = gm.ico2ico_vae(params)
    mod.load_state_dict(ref.state_dict())
    mod = set_impl(mod.cuda(), 'simt')
    x, tgt = data.synthetic_batch(level, 3, B)
    # CUDA first: take its eps and feed the same noise to the oracle graph
    eps_box = {}
    orig = gm._reparameterize

    def capture(mu, logvar):
        z, eps = reparam.reparameterize(mu, logvar, seed=42, offset=1, return_eps=True)
        eps_box['eps'] = eps.detach().cpu()
        return z
    gm._reparameterize = capture
    try:
        rec_c, mu_c, lv_c = mod(x.cuda())
    finally:
        gm._reparameterize = orig
    crit = losses.P2PKLD_Loss(level, 0.6, 0.2, 0.2, 1.0)
    loss_c = crit((rec_c, mu_c, lv_c), tgt.cuda())
    loss_c.backward()
    rec_r, mu_r, lv_r = ref(x, eps=eps_box['eps'])
    loss_r = om.ref_p2p_loss(level, rec_r, tgt, 0.6, 0.2, 0.2)[0] + om.ref_kld(mu_r, lv_r)
    loss_r.backward()
    torch.cuda.synchronize()
    assert abs(loss_c.item() - loss_r.item()) <= 1e-3 * abs(loss_r.item()), (loss_c.item(), loss_r.item())
    last = crit.get_last_losses()
    assert abs(last[4] - loss_r.item()) <= 1e-3 * abs(loss_r.item())
    _compare_grads(_grads(mod), _grads(ref), 0.999, 'vae')


def test_reference_style_training_loop_decreases_loss():
    """run.py:240-250 step semantics through the public API: 8 Adam steps on one batch reduce the loss."""
    from geniconet_b200 import models as gm, losses, data
    params = gm.default_params('ico2ico', 5)
    torch.manual_seed(0)
    model = gm.ico2ico(params).cuda()
    crit = losses.P2P_Loss(5, 1., 0., 0.)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    x, tgt = data.synthetic_batch(5, 0, 4)
    x, tgt = x.cuda(), tgt.cuda()
    hist = []
    for _ in range(8):
        opt.zero_grad()
        loss = crit(model(x), tgt)
        loss.backward()
        opt.step()
        hist.append(crit.get_last_losses()[-1])
    assert hist[-1] < 0.7 * hist[0], hist


def test_cuda_path_reproduces_reference_golden():
    """tests/golden/reference_over_oracle.json was produced by the reference's OWN models.py + losses.py (over the oracle
    layers) in the build container; the CUDA path must land on the same loss, outputs and gradient norms."""
    import json
    import os
    from geniconet_b200 import models as gm, losses
    from geniconet_b200.ico_conv import set_impl
    torch.backends.cudnn.allow_tf32 = False
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_over_oracle.json')))
    g = gold['ico2ico']
    gen = torch.Generator().manual_seed(g['input_seed'])
    x = torch.randn(g['batch'], 3, 160, 64, generator=gen) * 0.3
    tgt = torch.randn(g['batch'], 9, 10242, generator=gen) * 0.5
    for impl, tol in (('simt', 1e-4), ('auto', 2e-2)):
        mod = om.fill_params_deterministic(gm.ico2ico(gm.default_params('ico2ico')))
        mod = set_impl(mod.cuda(), impl)
        crit = losses.P2P_Loss(5, 1., 0., 0.)
        y = mod(x.cuda())
        loss = crit(y, tgt.cuda())
        loss.backward()
        assert abs(loss.item() - g['loss']) <= tol * abs(g['loss']), (impl, loss.item(), g['loss'])
        f = y.detach().flatten().cpu()
        samp = f[torch.linspace(0, f.numel() - 1, 64).long()]
        assert (samp - torch.tensor(g['output_sample'])).abs().max().item() <= (2e-4 if impl == 'simt' else 5e-2)
        last = crit.get_last_losses()
        for a, b in zip(last, g['last_losses']):
            assert abs(a - b) <= max(tol, 1e-4) * max(1.0, abs(b)), (impl, last, g['last_losses'])
        # a conv bias that feeds a BatchNorm has a mathematically ZERO gradient (the batch mean absorbs it): its golden
        # "norm" is fp32 rounding noise (~1e-7), so it is only required to stay noise-sized, not to match
        noise = 1e-5 * max(g['grad_norms'].values())
        for k, p in mod.named_parameters():
            want = g['grad_norms'][k]
            got = p.grad.norm().item()
            if want < noise:
                assert got < (10 if impl == 'simt' else 1e3) * noise, (impl, k, got, want)
            else:
                assert abs(got - want) <= (1e-2 if impl == 'simt' else 0.25) * want, (impl, k, got, want)
    # the loss kernels alone, all three terms live (losses.py:71-80)
    g3 = gold['p2p_level3']
    gen = torch.Generator().manual_seed(g3['input_seed'])
    x3 = (torch.randn(g3['batch'], 3, 40, 16, generator=gen) * 0.3).cuda().requires_grad_(True)
    t3 = (torch.randn(g3['batch'], 9, 642, generator=gen) * 0.5).cuda()
    c3 = losses.P2P_Loss(3, 0.6, 0.2, 0.2)
    l3 = c3(x3, t3)
    l3.backward()
    assert abs(l3.item() - g3['loss']) <= 1e-5 * abs(g3['loss'])
    assert abs(x3.grad.norm().item() - g3['grad_norm']) <= 1e-4 * g3['grad_norm']


def _seeded_step(name, level, x, tgt, factors, fused, impl, head=None):
    """One forward + loss + backward from the deterministic parameter fill; returns (loss, grads, buffers)."""
    from geniconet_b200 import models as gm, losses, reparam
    from geniconet_b200.ico_conv import set_impl
    params = gm.default_params(name, level)
    gm.set_fused(fused, head)
    torch.manual_seed(3)
    mod = set_impl(om.fill_params_deterministic(getattr(gm, name)(params)).cuda().train(), impl)
    crit = losses.P2PKLD_Loss(level, *factors, 1.0) if name == 'ico2ico_vae' else losses.P2P_Loss(level, *factors)
    reparam.manual_seed(11)
    loss = crit(mod(x), tgt)
    loss.backward()
    torch.cuda.synchronize()
    return loss.item(), _grads(mod), {k: b.detach().cpu().clone() for k, b in mod.named_buffers()}


@pytest.mark.parametrize('name', ['ico2ico', 'ico2ico_vae'])
def test_fused_chain_matches_modulewise(name):
    """geniconet_b200/fused.py (one Function per encoder/decoder body: sibling convs as one GEMM, fused BatchNorm + ReLU + add +
    bf16 cast, the 1x1 head through gin_head_*) against the module-by-module path over the SAME tcgen05 kernels and against the
    fp32 CUDA-core path: identical weights, inputs and reparam noise.  Both bf16 paths are judged by their distance to the fp32
    gradients, parameter by parameter, under the position (+ KLD) loss.  The VAE's normal / Laplacian terms are left out of the
    gradient comparison: on the near-degenerate mesh a random-init network emits, their gradient is chaotic (ANY rounding
    difference, even a TF32 head, re-draws ~40 % of it -- profiles/r01_vae_grad_conditioning.txt), so there only the loss and
    the finiteness of the gradients are compared; the loss kernels themselves are checked against the oracle in
    tests/test_gpu_layers.py."""
    from geniconet_b200 import models as gm, data
    level, B = 5, 3
    params = gm.default_params(name, level)
    x, tgt = data.synthetic_batch(level, 0, B)
    x, tgt = x.cuda(), tgt.cuda()
    f_ref = (params['ico']['factor_pos'], params['ico']['factor_nor'], params['ico']['factor_lap'])
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False                  # the module-wise paths keep the stock 1x1 head: make it real fp32
    try:
        res = {tag: _seeded_step(name, level, x, tgt, (1.0, 0.0, 0.0), fused, impl)
               for tag, fused, impl in (('fp32', False, 'simt'), ('tc', False, 'auto'), ('fused', True, 'auto'))}
        full = {tag: _seeded_step(name, level, x, tgt, f_ref, fused, impl) for tag, fused, impl in (('tc', False, 'auto'), ('fused', True, 'auto'))}
    finally:
        gm.set_fused(True, True)
        torch.backends.cudnn.allow_tf32 = tf32
    (l0, g0, b0), (l1, g1, b1), (l2, g2, b2) = res['fp32'], res['tc'], res['fused']
    assert abs(l2 - l0) <= 2e-3 * abs(l0) and abs(l2 - l1) <= 2e-3 * abs(l1), (l0, l1, l2)
    assert abs(full['fused'][0] - full['tc'][0]) <= 2e-3 * abs(full['tc'][0])
    assert all(torch.isfinite(g).all() for g in full['fused'][1].values())

    def cos(a, b):
        a, b = a.flatten().double(), b.flatten().double()
        return (a @ b / (a.norm() * b.norm())).item()
    cs_tc, cs_fused = [], []
    for k, ref in g0.items():
        if ref.norm() < 1e-6:
            continue
        c_tc, c_fused = cos(g1[k], ref), cos(g2[k], ref)
        cs_tc.append(c_tc)
        cs_fused.append(c_fused)
        assert c_fused >= 0.985 and c_fused >= c_tc - 0.01, (k, c_tc, c_fused)       # measured: >= 0.9938, |fused - tc| <= 6e-4
        assert 0.93 <= (g2[k].norm() / ref.norm()).item() <= 1.07, k
    assert sum(cs_fused) / len(cs_fused) >= sum(cs_tc) / len(cs_tc) - 0.002, (sum(cs_fused) / len(cs_fused), sum(cs_tc) / len(cs_tc))
    for k in b0:
        if k.endswith('running_mean') or k.endswith('running_var'):
            assert torch.allclose(b2[k], b0[k], rtol=2e-2, atol=2e-3), k
        if k.endswith('num_batches_tracked'):
            assert int(b2[k]) == int(b0[k]) == 1, k
    # a conv bias in front of a BatchNorm: exactly zero on the fused path
    assert float(g2['encoder.3.conv00.bias'].abs().max()) == 0.0


@pytest.mark.parametrize('name', ['ico2ico', 'ico2ico_vae'])
def test_fused_step_is_reproducible(name):
    """The same seeded training step twice, the allocator's free blocks overwritten in between: loss and every gradient must be
    bit-identical.  No kernel on the path combines partial results with atomics (conv-epilogue BatchNorm sums, seam rows,
    split-K and per-CTA reductions all add in a fixed order); a last-bit difference would not stay small -- every bf16 operand
    cast downstream re-rounds, so it grows to the bf16 noise floor within three blocks (profiles/r01_vae_grad_conditioning.txt)."""
    from geniconet_b200 import models as gm, data
    level, B = 5, 5                                          # odd batch: a ragged last sample group
    params = gm.default_params(name, level)
    x, tgt = data.synthetic_batch(level, 0, B)
    x, tgt = x.cuda(), tgt.cuda()
    f = (params['ico']['factor_pos'], params['ico']['factor_nor'], params['ico']['factor_lap'])
    try:
        _seeded_step(name, level, x, tgt, f, True, 'auto')                               # warm-up: plans, caches
        l0, g0, _ = _seeded_step(name, level, x, tgt, f, True, 'auto')
        junk = torch.full((1 << 30,), 0xFF, dtype=torch.uint8, device='cuda')
        del junk
        l1, g1, _ = _seeded_step(name, level, x, tgt, f, True, 'auto')
    finally:
        gm.set_fused(True, True)
    assert l0 == l1
    differing = [k for k in g0 if not torch.equal(g0[k], g1[k])]
    assert not differing, differing


@pytest.mark.parametrize('name,level,B', [('ico2ico', 5, 36), ('ico2ico_vae', 5, 36), ('ico2ico', 6, 16)])
def test_bench_configurations_run_and_agree(name, level, B):
    """The BASELINE.json configurations at their FULL sizes (tile counts, kernel selections and shared-memory plans depend on the
    batch): one fused and one module-wise training step from the same weights must give the same loss and finite gradients."""
    from geniconet_b200 import models as gm, losses, data, reparam
    params = gm.default_params(name, level)
    x, tgt = data.synthetic_batch(level, 0, 2)
    x = x.repeat((B + 1) // 2, 1, 1, 1)[:B].cuda()
    tgt = tgt.repeat((B + 1) // 2, 1, 1)[:B].cuda()
    f = (params['ico']['factor_pos'], params['ico']['factor_nor'], params['ico']['factor_lap'])
    vals = {}
    try:
        for fused in (True, False):
            gm.set_fused(fused)
            torch.manual_seed(5)
            mod = getattr(gm, name)(params).cuda().train()
            crit = losses.P2PKLD_Loss(level, *f, 1.0) if name == 'ico2ico_vae' else losses.P2P_Loss(level, *f)
            reparam.manual_seed(7)
            loss = crit(mod(x), tgt)
            loss.backward()
            torch.cuda.synchronize()
            assert all(torch.isfinite(p.grad).all() for p in mod.parameters())
            vals[fused] = loss.item()
            del mod, loss
            torch.cuda.empty_cache()
    finally:
        gm.set_fused(True)
    assert abs(vals[True] - vals[False]) <= 5e-3 * abs(vals[False]), vals


def test_hook_inside_a_training_chain_runs_the_modules():
    """A forward or forward-pre hook on a module inside a chain sends the chain to the modules in train mode with grad too: both
    hooks fire and the output is bit for bit that of set_fused(False)."""
    import copy
    from geniconet_b200 import models as gm, data
    level, B = 5, 3
    a = om.fill_params_deterministic(gm.ico2ico(gm.default_params('ico2ico', level))).cuda().train()
    b = copy.deepcopy(a)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    fired = []
    a.encoder[3].conv01.register_forward_hook(lambda m, i, o: fired.append('conv01'))
    a.decoder[0].icobn01.register_forward_pre_hook(lambda m, i: fired.append('icobn01'))
    try:
        gm.set_fused(True, head=False)                       # the module head on both sides
        y_a = a(x)
        gm.set_fused(False)
        y_b = b(x)
    finally:
        gm.set_fused(True, True)
    assert fired == ['conv01', 'icobn01']
    assert torch.equal(y_a, y_b)


def test_fused_chain_returns_the_xyz_input_gradient():
    """d loss / d input through the fused chain (the xyz stem's dgrad) against the module-wise fp32 path."""
    from geniconet_b200 import models as gm, losses, data
    from geniconet_b200.ico_conv import set_impl
    level, B = 5, 2
    params = gm.default_params('ico2ico', level)
    x, tgt = data.synthetic_batch(level, 0, B)
    grads = {}
    try:
        for tag, fused, impl in (('fused', True, 'auto'), ('fp32', False, 'simt')):
            gm.set_fused(fused)
            mod = set_impl(om.fill_params_deterministic(gm.ico2ico(params)).cuda().train(), impl)
            xi = x.cuda().requires_grad_(True)
            losses.P2P_Loss(level, 1., 0., 0.)(mod(xi), tgt.cuda()).backward()
            grads[tag] = xi.grad.detach().double().flatten().cpu()
    finally:
        gm.set_fused(True)
    a, b = grads['fused'], grads['fp32']
    assert torch.isfinite(a).all() and a.shape == b.shape
    cos = (a @ b / (a.norm() * b.norm())).item()
    assert cos >= 0.98, cos
