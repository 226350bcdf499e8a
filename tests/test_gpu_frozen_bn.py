"""Eval-mode BatchNorm with grad enabled (fused.run_frozen_chain, gin_bn_eval_bwd / _pair) on the GPU: the kernels against an fp64
reference, the chain against the fp32 oracle, frozen state and parameters, routing, the optimizer's version bump, graphs."""
import contextlib
import copy
import os
import re

import pytest
import torch

import oracle_models as om
from geniconet_b200 import _lib, data, fused, models as gm
from geniconet_b200.graph import GraphedStep
from geniconet_b200.ico_conv import cast_bf16, get_plan

pytestmark = pytest.mark.gpu
L = _lib.lib


@contextlib.contextmanager
def switch(fused_on=True, frozen=True):
    saved = gm._FUSED, gm._HEAD, gm._INFER, gm._FROZEN
    gm.set_fused(fused_on, frozen=frozen)
    try:
        yield
    finally:
        gm._FUSED, gm._HEAD, gm._INFER, gm._FROZEN = saved


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm()).item()


def _cos(a, b):
    a, b = a.detach().double().flatten().cpu(), b.detach().double().flatten().cpu()
    return (a @ b / (a.norm() * b.norm())).item()


def _models(name, level, corner_mode='average', warm_batches=3, B=4):
    """(CUDA model, oracle model on the GPU) with equal weights and non-trivial running statistics, both in eval mode."""
    params = gm.default_params(name, level, corner_mode)
    ref = om.fill_params_deterministic(om.build_oracle_model(name, params)).cuda().train()
    with torch.no_grad():
        for k in range(warm_batches):
            x, _ = data.synthetic_batch(level, 10 + k * B, B)
            ref(x.cuda())
    mod = getattr(gm, name)(params)
    mod.load_state_dict(ref.state_dict())
    return mod.cuda().eval(), ref.eval()


def _target(shape, seed=1):
    return (0.5 * torch.randn(shape, generator=torch.Generator().manual_seed(seed))).cuda()


def _loss(out, t):
    return ((out - t) ** 2).mean()


def _buffers(m):
    return {k: v.detach().clone() for k, v in m.named_buffers()}


# ---------------------------------------------------------------------------------------------------------- 1. the kernels
def _bn_shapes():
    """(level, C) of every BatchNorm of the chains of ico2ico / ico2ico_vae at I5 and I6."""
    shapes = set()
    for top in (5, 6):
        for kind in ('ae', 'vae'):
            enc, dec = gm._ENC_WIDTHS[kind], gm._DEC_WIDTHS[kind]
            shapes.add((top, enc[0]))
            shapes.update((top - d - 1, enc[d + 1]) for d in range(len(enc) - 1))
            shapes.update((top - 2 + d, dec[d + 1]) for d in range(3))
    return sorted(shapes)


def _consts(C, seed):
    g = torch.Generator().manual_seed(seed)
    bn = torch.nn.BatchNorm2d(C).cuda().eval()
    with torch.no_grad():
        bn.weight.copy_(1 + 0.3 * torch.randn(C, generator=g))
        bn.weight[::7] *= -1                                   # negative gammas too
        bn.bias.copy_(0.2 * torch.randn(C, generator=g))
        bn.running_mean.copy_(0.3 * torch.randn(C, generator=g))
        bn.running_var.copy_(0.5 + torch.rand(C, generator=g))
    return fused._eval_consts([(bn, None)])[0][2].clone().view(4, C)      # stat [4][C]


def test_eval_consts_follow_the_width_at_the_same_addresses():
    """The constants cache (fused._bn_table) must not hand a BatchNorm the table of another width that had the same id() and storage
    addresses, as one created after another died can have (the caching allocator reuses the blocks).  Modelled here by one module
    narrowed in place to the leading half of its own storages."""
    bn = torch.nn.BatchNorm2d(128).cuda().eval()
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        bn.weight.copy_(1 + 0.3 * torch.randn(128, generator=g))
        bn.bias.copy_(0.2 * torch.randn(128, generator=g))
        bn.running_mean.copy_(0.3 * torch.randn(128, generator=g))
        bn.running_var.copy_(0.5 + torch.rand(128, generator=g))
    assert fused._eval_consts([(bn, None)])[0][2].numel() == 4 * 128
    bn.weight, bn.bias = torch.nn.Parameter(bn.weight.data[:64]), torch.nn.Parameter(bn.bias.data[:64])
    bn.running_mean, bn.running_var, bn.num_features = bn.running_mean[:64], bn.running_var[:64], 64
    scale, shift, stat = fused._eval_consts([(bn, None)])[0]
    assert (scale.numel(), shift.numel(), stat.numel()) == (64, 64, 4 * 64)
    want = bn.weight.detach() / torch.sqrt(bn.running_var + bn.eps)
    torch.testing.assert_close(scale, want, rtol=1e-5, atol=0)
    torch.testing.assert_close(shift, bn.bias.detach() - bn.running_mean * want, rtol=1e-5, atol=1e-6)


def _ptr(t, off=0):
    return t.data_ptr() + off if t is not None else None


@pytest.mark.parametrize('y16', [True, False], ids=['y_fp16', 'y_fp32'])
@pytest.mark.parametrize('shape', _bn_shapes(), ids=lambda s: 'L%d_C%d' % s)
def test_eval_bwd_kernels_match_fp64(shape, y16):
    level, C = shape
    B, dev = 2, torch.device('cuda')
    rows = B * 10 * 4 ** level
    g = torch.Generator().manual_seed(level * 1000 + C)
    ydt = torch.float16 if y16 else torch.float32
    stA, stB = _consts(C, 1), _consts(C, 2)
    yA = (torch.randn(rows, C, generator=g) * 1.3).to(dev).to(ydt)
    ycat = (torch.randn(rows, 2 * C, generator=g) * 1.3).to(dev).to(ydt)       # yB = its right half, row stride 2C
    dout = torch.randn(rows, C, generator=g).to(dev)
    plan = get_plan(_lib.PLAN_HEXCONV, level, 1, 'average', dev)
    n = 2 ** level
    f16 = 1 if y16 else 0
    s = fused._stream()
    ws = torch.empty(L.gin_bn_eval_bwd_ws_bytes(C), dtype=torch.uint8, device=dev)

    def cast1(dy_f):
        return cast_bf16(dy_f.view(B, 5 * n, 2 * n, C).permute(0, 3, 1, 2), plan, 1, level).view(torch.int16).view(-1, C)

    def fwd(two):
        out_f = torch.empty(rows, C, device=dev)
        mask = torch.empty(rows + 2 * B, C, dtype=torch.bfloat16, device=dev)
        _lib.check(L.gin_bn_act_fwd(yA.data_ptr(), C, stA.data_ptr(), _ptr(ycat, ycat.element_size() * C) if two else None, 2 * C,
                                    stB.data_ptr() if two else None, f16, 1, None, out_f.data_ptr(), mask.data_ptr(), B, level, C, s), 'fwd')
        return out_f, mask

    def ref_sums(y, st, gm64):
        yh = (y.double() - st[0].double()) * st[1].double()
        sg = gm64.sum(0)
        return torch.cat([sg, (gm64 * yh).sum(0), st[2].double() * sg])

    # ---- one BatchNorm + ReLU
    out_f, mask = fwd(False)
    gmask = torch.where(out_f > 0, dout, torch.zeros_like(dout))     # masked entries are +0, as in the kernels
    dy_ref32 = stA[2] * gmask                                   # the fp32 product the kernel forms
    outs = {}
    for from_y in (1, 0):
        dy_b = torch.empty(rows + 2 * B, C, dtype=torch.bfloat16, device=dev)
        dy_f = torch.empty(rows, C, device=dev)
        bsum = torch.empty(3 * C, device=dev)
        _lib.check(L.gin_bn_eval_bwd(dout.data_ptr(), C, mask.data_ptr(), yA.data_ptr(), C, f16, stA.data_ptr(), bsum.data_ptr(),
                                     dy_b.data_ptr(), C, dy_f.data_ptr(), C, ws.data_ptr(), B, level, C, from_y, s), 'gin_bn_eval_bwd')
        outs[from_y] = (dy_b, dy_f, bsum)
    dy_b, dy_f, bsum = outs[1]
    for a, b in zip(outs[0], outs[1]):                          # mask read == mask re-evaluated, bit for bit
        assert torch.equal(a.view(torch.int16) if a.dtype == torch.bfloat16 else a, b.view(torch.int16) if b.dtype == torch.bfloat16 else b)
    assert _rel(dy_f, stA[2].double() * gmask.double()) <= 1e-6
    assert torch.equal(dy_f, dy_ref32)
    assert torch.equal(dy_b.view(torch.int16), cast1(dy_f)), 'bf16 gradient copy (pole rows included)'
    assert _rel(bsum, ref_sums(yA, stA, gmask.double())) <= 1e-5
    # NULL sums: the same gradient, and the workspace is not touched
    ws.fill_(0x5a)
    dy_b2 = torch.empty_like(dy_b)
    _lib.check(L.gin_bn_eval_bwd(dout.data_ptr(), C, None, yA.data_ptr(), C, f16, stA.data_ptr(), None, dy_b2.data_ptr(), C, None, 0,
                                 ws.data_ptr(), B, level, C, 1, s), 'gin_bn_eval_bwd')
    assert torch.equal(dy_b2.view(torch.int16), dy_b.view(torch.int16))
    assert bool((ws == 0x5a).all())

    # ---- the residual pair relu(bnA(yA) + bnB(yB))
    out_f, mask = fwd(True)
    gmask = torch.where(out_f > 0, dout, torch.zeros_like(dout))
    outs = {}
    for from_y, red in ((1, True), (0, True), (1, False)):
        dyA = torch.empty(rows + 2 * B, C, dtype=torch.bfloat16, device=dev)
        dycat = torch.zeros(rows + 2 * B, 2 * C, dtype=torch.bfloat16, device=dev)
        bA, bB = (torch.empty(3 * C, device=dev), torch.empty(3 * C, device=dev)) if red else (None, None)
        ws.fill_(0x5a)
        _lib.check(L.gin_bn_eval_bwd_pair(dout.data_ptr(), C, mask.data_ptr(), yA.data_ptr(), C, stA.data_ptr(), _ptr(bA), dyA.data_ptr(), C,
                                          ycat.data_ptr() + ycat.element_size() * C, 2 * C, stB.data_ptr(), _ptr(bB), dycat.data_ptr() + 2 * C,
                                          2 * C, f16, ws.data_ptr(), B, level, C, from_y, s), 'gin_bn_eval_bwd_pair')
        if not red:
            assert bool((ws == 0x5a).all())
        outs[(from_y, red)] = (dyA, dycat, bA, bB)
    dyA, dycat, bA, bB = outs[(1, True)]
    for key in ((0, True), (1, False)):
        assert torch.equal(outs[key][0].view(torch.int16), dyA.view(torch.int16)), key
        assert torch.equal(outs[key][1].view(torch.int16), dycat.view(torch.int16)), key
    assert torch.equal(outs[(0, True)][2], bA) and torch.equal(outs[(0, True)][3], bB)
    assert torch.equal(dycat[:, :C].view(torch.int16), torch.zeros_like(dycat[:, :C]).view(torch.int16))     # left half untouched
    assert torch.equal(dyA.view(torch.int16), cast1(stA[2] * gmask))
    assert torch.equal(dycat[:, C:].contiguous().view(torch.int16), cast1(stB[2] * gmask))
    assert _rel(dyA[:rows].float(), stA[2].double() * gmask.double()) <= 1e-2      # bf16
    assert _rel(bA, ref_sums(yA, stA, gmask.double())) <= 1e-5
    assert _rel(bB, ref_sums(ycat[:, C:], stB, gmask.double())) <= 1e-5


def test_no_floating_point_atomics_in_the_eval_backward_kernels():
    import shutil
    import subprocess
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    sass = subprocess.run([cuobjdump, '-sass', _lib.LIB_PATH], capture_output=True, text=True).stdout
    current, seen, dirty = None, set(), set()
    for line in sass.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            current = m.group(1)
            if 'eval_bwd' in current:
                seen.add(current)
            continue
        if current in seen and re.search(r'(REDG?|ATOMG?)\.E\.ADD\.F(16|32|64)|ATOMS\.(CAST|ADD\.F)', line):
            dirty.add(current)
    assert len(seen) == 9, sorted(seen)                       # 2 x 2 x 2 streaming kernels + the final sum
    assert not dirty, sorted(dirty)


# ---------------------------------------------------------------------------------------------------------- 2. parity with the oracle
def _param_grads(m):
    return {k: p.grad for k, p in m.named_parameters() if p.grad is not None}


@pytest.mark.parametrize('level,B,corner_mode', [(5, 36, 'average'), (5, 36, 'zeros'), (6, 16, 'average')])
def test_frozen_ico2ico_matches_oracle(level, B, corner_mode):
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    mod, ref = _models('ico2ico', level, corner_mode)
    before = _buffers(mod)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    xc, xr = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    t = _target((B, 3) + tuple(x.shape[2:]))
    with switch():
        out = mod(xc)
        loss = _loss(out, t)
        loss.backward()
    out_r = ref(xr)
    loss_r = _loss(out_r, t)
    loss_r.backward()
    assert abs(loss.item() - loss_r.item()) <= 2e-2 * abs(loss_r.item())
    assert _rel(out, out_r) <= 5e-2
    gc, gr = _param_grads(mod), _param_grads(ref)
    assert set(gc) == set(gr) == {k for k, _ in mod.named_parameters()}
    worst = min((_cos(gc[k], gr[k]), k) for k in gr)
    print('frozen ico2ico I%d B=%d %s: worst gradient cosine %.5f (%s), input %.5f' % (level, B, corner_mode, worst[0], worst[1],
                                                                                       _cos(xc.grad, xr.grad)))
    assert worst[0] >= 0.99, worst
    assert _cos(xc.grad, xr.grad) >= 0.99
    for k in gr:                                                # eval mode: conv biases in front of a BatchNorm get real gradients
        if k.endswith('.bias') and 'conv' in k:
            assert gc[k].norm() > 0 and gr[k].norm() > 0, k
    after = _buffers(mod)
    for k in before:                                            # running statistics and num_batches_tracked bit-identical
        assert torch.equal(before[k], after[k]), k


def test_frozen_vae_decode_matches_oracle():
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    level, B = 5, 36
    mod, ref = _models('ico2ico_vae', level)
    before = _buffers(mod)
    n = 2 ** (level - 3)
    z0 = torch.randn(B, 512, 5 * n, 2 * n, generator=torch.Generator().manual_seed(4)).cuda()
    zc, zr = z0.clone().requires_grad_(True), z0.clone().requires_grad_(True)
    t = _target((B, 3, 5 * 2 ** level, 2 ** (level + 1)))
    with switch():
        loss = _loss(mod.decode(zc), t)
        loss.backward()
    loss_r = _loss(ref.final_layer(ref.decoder(zr)), t)
    loss_r.backward()
    assert abs(loss.item() - loss_r.item()) <= 2e-2 * abs(loss_r.item())
    gc, gr = _param_grads(mod), _param_grads(ref)
    assert set(gc) == set(gr)
    cos = [_cos(gc[k], gr[k]) for k in gr]
    print('frozen VAE decode: z cosine %.5f, parameter cosine mean %.5f min %.5f' % (_cos(zc.grad, zr.grad), sum(cos) / len(cos), min(cos)))
    assert _cos(zc.grad, zr.grad) >= 0.99
    assert sum(cos) / len(cos) >= 0.99 and min(cos) >= 0.98
    after = _buffers(mod)
    for k in before:
        assert torch.equal(before[k], after[k]), k


# ---------------------------------------------------------------------------------------------------------- 3. frozen parameters
def test_latent_fitting_computes_no_weight_gradients():
    level, B = 5, 8
    mod, ref = _models('ico2ico_vae', level)
    for p in mod.parameters():
        p.requires_grad_(False)
    n = 2 ** (level - 3)
    z0 = torch.randn(B, 512, 5 * n, 2 * n, generator=torch.Generator().manual_seed(5)).cuda()
    t = _target((B, 3, 5 * 2 ** level, 2 ** (level + 1)))

    def run(z):
        with switch():
            _loss(mod.decode(z), t).backward()

    def kernels(z):
        run(z)                                                  # warm
        z.grad = None
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(z)
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]

    zc = z0.clone().requires_grad_(True)
    names = kernels(zc)
    assert any('eval_bwd' in k for k in names), 'the frozen chain ran'
    assert not any('wgrad_patch' in k for k in names), sorted({k for k in names if 'wgrad' in k})
    assert all(p.grad is None for p in mod.parameters())
    for p in ref.parameters():
        p.requires_grad_(False)
    zr = z0.clone().requires_grad_(True)
    _loss(ref.final_layer(ref.decoder(zr)), t).backward()
    assert _cos(zc.grad, zr.grad) >= 0.99
    # with the decoder trainable the same profile does list the weight-gradient kernels
    for p in mod.decoder.parameters():
        p.requires_grad_(True)
    assert any('wgrad_patch' in k for k in kernels(z0.clone().requires_grad_(True)))


# ---------------------------------------------------------------------------------------------------------- 4. routing
def _refuse(*a, **k):
    raise AssertionError('the frozen chain must not run here')


def test_default_off_and_hook_fallback(monkeypatch):
    level, B = 5, 4
    mod, _ = _models('ico2ico', level)
    vae, _ = _models('ico2ico_vae', level)
    p = gm.default_params('ico2ico', level)
    enc, dec = gm.ico2enc(p).cuda().eval(), gm.enc2ico(p).cuda().eval()
    enc.encoder.load_state_dict(mod.encoder.state_dict())
    dec.decoder.load_state_dict(mod.decoder.state_dict())
    dec.enc2icoConv.load_state_dict(mod.enc2icoConv.state_dict())
    pv = gm.default_params('ico2ico_vae', level)
    venc, vdec = gm.ico2enc_vae(pv).cuda().eval(), gm.enc2ico_vae(pv).cuda().eval()
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda().requires_grad_(True)
    z = torch.randn(B, 512, 20, 8, device='cuda', requires_grad=True)          # the decoder's input level, top - 3
    if os.environ.get('GIN_FUSED_FROZEN') is None:
        assert not gm._FROZEN                                  # off unless asked for
    calls = []
    real = fused.run_frozen_chain

    def counting(*a, **k):
        calls.append(1)
        return real(*a, **k)

    def everything():
        outs = [mod(x), vae.decode(z), vae.encode(x)[0], enc(x), dec(enc(x)), venc(x)[0], vdec.decode(z)]
        sum(o.float().sum() for o in outs).backward()
        return outs
    with switch(True, False):
        monkeypatch.setattr(fused, 'run_frozen_chain', _refuse)
        off = everything()
    monkeypatch.setattr(fused, 'run_frozen_chain', counting)
    with switch():
        on = everything()
    assert len(calls) >= 8
    assert not torch.equal(on[0], off[0])                      # the switch does take the fused path
    # a hook inside a chain sends that chain to the modules
    monkeypatch.setattr(fused, 'run_frozen_chain', _refuse)
    h = mod.encoder[3].conv01.register_forward_hook(lambda m, i, o: None)
    h2 = mod.decoder[0].icobn01.register_forward_pre_hook(lambda m, i: None)
    try:
        with switch():
            y = mod(x)
    finally:
        h.remove()
        h2.remove()
    assert torch.equal(y, off[0])


def test_frozen_decoder_bn_in_train_mode_model_keeps_running_stats():
    """model.train() then bn.eval() on the decoder's BatchNorms, grad enabled, default switches: the decoder's running statistics stay
    as they are and the output matches the module path."""
    level, B = 5, 8
    mod, _ = _models('ico2ico', level)
    mod.train()
    for m in mod.decoder.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eval()
    other = copy.deepcopy(mod)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    dec_before = _buffers(mod.decoder)
    y = mod(x)
    y.sum().backward()
    for k, v in _buffers(mod.decoder).items():
        assert torch.equal(v, dec_before[k]), k
    with switch(False, False):
        y_mod = other(x)
    assert _rel(y, y_mod) <= 5e-2
    for k, v in _buffers(other).items():                       # encoder statistics updated the same way on both paths
        if 'running' in k:
            assert _rel(_buffers(mod)[k], v) <= 1e-2, k


def test_frozen_encoder_trained_decoder_matches_module_path():
    level, B = 5, 16
    mod, _ = _models('ico2ico', level)
    mod.decoder.train()
    other = copy.deepcopy(mod)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    t = _target((B, 3) + tuple(x.shape[2:]))
    with switch():
        loss = _loss(mod(x), t)
        loss.backward()
    with switch(False, False):
        loss_m = _loss(other(x), t)
        loss_m.backward()
    assert abs(loss.item() - loss_m.item()) <= 2e-2 * abs(loss_m.item())
    ga, gb = _param_grads(mod), _param_grads(other)
    assert set(ga) == set(gb)
    for k in gb:
        if k.startswith('decoder') and 'conv' in k and k.endswith('bias'):
            continue                        # in front of a train-mode BatchNorm: zero up to rounding on both paths
        assert _cos(ga[k], gb[k]) >= 0.99, k


# ---------------------------------------------------------------------------------------------------------- 5. optimizer
def test_adam_steps_are_seen_by_the_module_path():
    from geniconet_b200.optim import Adam
    level, B = 5, 4
    mod, _ = _models('ico2ico', level)
    mod.train()
    opt = Adam(mod.parameters(), lr=1e-3)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    t = _target((B, 3) + tuple(x.shape[2:]))
    with switch(False, False):
        for _ in range(3):
            opt.zero_grad()
            _loss(mod(x), t).backward()
            opt.step()
        mod.eval()
        fresh = gm.ico2ico(gm.default_params('ico2ico', level)).cuda()
        fresh.load_state_dict(mod.state_dict())
        fresh.eval()
        with torch.no_grad():
            assert torch.equal(mod(x), fresh(x))


# ---------------------------------------------------------------------------------------------------------- 6. reproducibility, graphs
def test_reproducible_and_constants_private_to_each_forward():
    level, B = 5, 8
    mod, _ = _models('ico2ico', level)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    t = _target((B, 3) + tuple(x.shape[2:]))

    def grads():
        mod.zero_grad(set_to_none=True)
        with switch():
            _loss(mod(x), t).backward()
        return {k: g.clone() for k, g in _param_grads(mod).items()}
    g1, g2 = grads(), grads()
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k
    # a second forward on the same parameters rewrites the shared constants buffer before the first one's backward
    mod.zero_grad(set_to_none=True)
    with switch():
        loss = _loss(mod(x), t)
        with torch.no_grad():
            for m in mod.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.running_var.mul_(1.5)
        mod(x)
        loss.backward()
    for k, g in _param_grads(mod).items():
        assert torch.equal(g, g1[k]), k


def test_graphed_fine_tune_step_replays_like_eager():
    from geniconet_b200.optim import Adam
    level, B = 5, 8
    a, _ = _models('ico2ico', level)
    b = copy.deepcopy(a)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    t = _target((B, 3) + tuple(x.shape[2:]))

    def make(m):
        opt = Adam(m.parameters(), lr=1e-4)
        opt.prepare()

        def step(xs, ts):
            for p in m.parameters():
                if p.grad is not None:
                    p.grad.zero_()
            loss = _loss(m(xs), ts)
            loss.backward()
            opt.step()
            return loss
        return step
    with switch():
        sa = make(a)
        for _ in range(3 + 4):                                  # GraphedStep's three warm-up steps, then four replays
            sa(x, t)
        graphed = GraphedStep(make(b), (x, t), warmup=3)
        for _ in range(4):
            graphed()
    torch.cuda.synchronize()
    for (k, p), q in zip(a.named_parameters(), b.parameters()):
        assert torch.equal(p, q), k
