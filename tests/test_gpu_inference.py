"""Forward-only fused inference (fused.infer_chain, gin_hexconv_fwd_affine, gin_bn_eval_consts) on the GPU."""
import contextlib
import os
import re

import pytest
import torch

import oracle_models as om
from geniconet_b200 import _lib, data, fused, models as gm
from geniconet_b200.graph import GraphedStep
from geniconet_b200.ico_conv import as_channels_last, cast_bf16, get_plan

pytestmark = pytest.mark.gpu


@contextlib.contextmanager
def switch(fused_on=True, inference=True):
    saved = gm._FUSED, gm._HEAD, gm._INFER
    gm.set_fused(fused_on, inference=inference)
    try:
        yield
    finally:
        gm._FUSED, gm._HEAD, gm._INFER = saved


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm()).item()


def _models(name, level, corner_mode='average', warm_batches=3, B=4):
    """(CUDA model, oracle model on the GPU) with equal weights and non-trivial running statistics, both in eval mode."""
    params = gm.default_params(name, level, corner_mode)
    ref = om.fill_params_deterministic(om.build_oracle_model(name, params)).cuda().train()
    with torch.no_grad():
        for k in range(warm_batches):                     # running statistics from a few train-mode passes
            x, _ = data.synthetic_batch(level, 10 + k * B, B)
            ref(x.cuda())
    mod = getattr(gm, name)(params)
    mod.load_state_dict(ref.state_dict())
    return mod.cuda().eval(), ref.eval()


# ---------------------------------------------------------------------------------------------------------- 1. parity with the oracle
@pytest.mark.parametrize('level,B,corner_mode', [(5, 36, 'average'), (5, 36, 'zeros'), (6, 16, 'average'), (6, 16, 'zeros'),
                                                 (5, 1, 'average'), (5, 3, 'zeros')])
def test_eval_ico2ico_matches_oracle(level, B, corner_mode):
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    mod, ref = _models('ico2ico', level, corner_mode)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    with torch.no_grad(), switch():
        out = mod(x)
        out_r = ref(x)
    rel = _rel(out, out_r)
    print('eval parity ico2ico I%d B=%d %s: rel L2 %.3e' % (level, B, corner_mode, rel))
    assert rel <= 5e-2


def test_eval_ico2ico_vae_matches_oracle():
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    level, B = 5, 36
    mod, ref = _models('ico2ico_vae', level)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    box = {}
    orig = gm._reparameterize

    def capture(mu, logvar):
        from geniconet_b200 import reparam
        z, eps = reparam.reparameterize(mu, logvar, seed=7, offset=1, return_eps=True)
        box['eps'] = eps
        return z
    gm._reparameterize = capture
    try:
        with torch.no_grad(), switch():
            rec, mu, lv = mod(x)
            rec_r, mu_r, lv_r = ref(x, eps=box['eps'])
    finally:
        gm._reparameterize = orig
    for what, a, b in (('mu', mu, mu_r), ('logvar', lv, lv_r), ('decode', rec, rec_r)):
        rel = _rel(a, b)
        print('eval parity ico2ico_vae I5 B=36 %s: rel L2 %.3e' % (what, rel))
        assert rel <= 5e-2, what


# ---------------------------------------------------------------------------------------------------------- 2./3. the affine launches
def _launch_shapes():
    """(level_in, stride, Cin, Cout, split, relu_split, residual) of every affine launch of ico2ico I5 / I6 and the VAE latent heads."""
    shapes = set()
    for top in (5, 6):
        for kind in ('ae', 'vae'):
            enc, dec = gm._ENC_WIDTHS[kind], gm._DEC_WIDTHS[kind]
            for d in range(len(enc) - 1):
                shapes.add((top - d, 2, enc[d], 2 * enc[d + 1], enc[d + 1], enc[d + 1], False))
                shapes.add((top - d - 1, 1, enc[d + 1], enc[d + 1], enc[d + 1], 0, True))
            for d in range(3):
                lvl = top - 2 + d
                shapes.add((lvl, 1, dec[d], 2 * dec[d + 1], dec[d + 1], dec[d + 1], False))
                shapes.add((lvl, 1, dec[d + 1], dec[d + 1], dec[d + 1], 0, True))
        shapes.add((top - 2, 2, 256, 1024, 512, 0, False))
    return sorted(shapes)


def _bn_consts(C, seed, bias=True):
    g = torch.Generator().manual_seed(seed)
    bn = torch.nn.BatchNorm2d(C).cuda().eval()
    with torch.no_grad():
        bn.weight.copy_(1 + 0.2 * torch.randn(C, generator=g))
        bn.bias.copy_(0.1 * torch.randn(C, generator=g))
        bn.running_mean.copy_(0.3 * torch.randn(C, generator=g))
        bn.running_var.copy_(0.5 + torch.rand(C, generator=g))
    cb = (0.05 * torch.randn(C, generator=g)).cuda() if bias else None
    return bn, cb


def _problem(shape, B=2, seed=0):
    lvl_in, stride, cin, cout, split, relu_split, residual = shape
    lvl = lvl_in - 1 if stride == 2 else lvl_in
    dev = torch.device('cuda')
    g = torch.Generator().manual_seed(seed)
    plan = get_plan(_lib.PLAN_HEXCONV, lvl_in, stride, 'average', dev)
    n = 2 ** lvl_in
    x = torch.randn(B, cin, 5 * n, 2 * n, generator=g).cuda()
    xb = cast_bf16(as_channels_last(x), plan, 0, lvl_in)
    w = (torch.randn(cout, cin, 7, generator=g) * (1.5 / (7 * cin)) ** 0.5).cuda()
    packed = fused._pack_many([(w, None, cin)])[0]
    pairs = [_bn_consts(split, seed + 1)] + ([_bn_consts(cout - split, seed + 2)] if split < cout else [])
    consts = fused._eval_consts(pairs)
    scale, shift = fused._span(consts[0][0], cout), fused._span(consts[0][1], cout)
    bias = torch.cat([cb for _, cb in pairs])
    res = torch.randn(B * 10 * 4 ** lvl, cout, generator=g).cuda() if residual else None
    return dict(plan=plan, xb=xb, packed=packed, B=B, cin=cin, cout=cout, lvl=lvl, scale=scale, shift=shift, bias=bias, res=res,
                split=split, relu_split=relu_split, consts=consts)


def _affine(p, want0, want1=(False, False), res=None):
    return fused._conv_affine(p['plan'], p['xb'], p['packed'], p['B'], p['cin'], p['cout'], p['lvl'], p['scale'], p['shift'],
                              p['relu_split'], p['split'], want0, want1, res=res)


@pytest.mark.parametrize('shape', _launch_shapes(), ids=lambda s: 'L%d_s%d_%dx%d_split%d%s' % (s[0], s[1], s[2], s[3], s[4], '_res' if s[6] else ''))
def test_affine_operand_copy_equals_cast_of_its_fp32_map(shape):
    p = _problem(shape)
    two = p['split'] < p['cout']
    out = _affine(p, (True, True), (True, True) if two else (False, False), res=p['res'])
    assert out is not None, 'the affine epilogue must support every launch the models make'
    n = 2 ** p['lvl']
    for d in range(2 if two else 1):
        op, f = out[2 * d], out[2 * d + 1]
        C = f.shape[1]
        ref = cast_bf16(f.view(p['B'], 5 * n, 2 * n, C).permute(0, 3, 1, 2), get_plan(_lib.PLAN_HEXCONV, p['lvl'], 1, 'average', f.device), 0,
                        p['lvl'])
        assert torch.equal(op.view(-1).view(torch.int16), ref.view(-1).view(torch.int16)), 'destination %d' % d


@pytest.mark.parametrize('shape', _launch_shapes(), ids=lambda s: 'L%d_s%d_%dx%d_split%d%s' % (s[0], s[1], s[2], s[3], s[4], '_res' if s[6] else ''))
def test_affine_matches_stats2_plus_bn_act(shape):
    """The epilogue against the composition stats2 (fp32 y, conv bias) -> gin_bn_act_fwd with the same eval constants."""
    import ctypes
    p = _problem(shape, seed=3)
    B, cout, split, lvl = p['B'], p['cout'], p['split'], p['lvl']
    two = split < cout
    out = _affine(p, (False, True), (False, True) if two else (False, False), res=p['res'])
    rows = B * 10 * 4 ** lvl
    y = torch.empty(rows, cout, device='cuda')
    parts = torch.empty(_lib.lib.gin_hexconv_stats_ws_bytes(cout) // 4, device='cuda')
    nparts = ctypes.c_int(0)
    _lib.check(_lib.lib.gin_hexconv_fwd_bf16_stats2(p['plan'].host_ptr, p['plan'].dev_ptr, p['xb'].data_ptr(), p['packed'].data_ptr(),
                                                   p['bias'].data_ptr(), None, 0, y.data_ptr(), 0, B, p['cin'], cout, parts.data_ptr(),
                                                   ctypes.addressof(nparts), fused._stream()), 'stats2')
    stats = [c[2] for c in p['consts']]
    for d, (c0, C, st) in enumerate(((0, split, stats[0]), (split, cout - split, stats[-1]))[:2 if two else 1]):
        ref = torch.empty(rows, C, device='cuda')
        relu = 1 if c0 < p['relu_split'] else 0
        if p['res'] is not None:            # relu(bn(y) + R): R enters gin_bn_act_fwd as a second map with unit scale
            ident = torch.zeros(4, C, device='cuda')
            ident[2] = 1
            args = (p['res'].data_ptr(), cout, ident.data_ptr())
            relu = 1
        else:
            args = (None, 0, None)
        _lib.check(_lib.lib.gin_bn_act_fwd(y.data_ptr() + 4 * c0, cout, st.data_ptr(), *args, 0, relu, None, ref.data_ptr(), None, B, lvl, C,
                                          fused._stream()), 'bn_act_fwd')
        rel = _rel(out[2 * d + 1], ref)
        assert rel <= 1e-6, (d, rel)


def test_affine_fp16_residual():
    shape = (5, 1, 64, 64, 64, 0, True)
    p = _problem(shape, seed=5)
    r16 = p['res'].half()
    a = _affine(p, (False, True), res=r16)[1]
    b = _affine(p, (False, True), res=r16.float())[1]
    assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------- 4. train mode under no_grad
def _state(m):
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def test_train_mode_no_grad_is_the_training_forward():
    level, B = 5, 8
    import copy
    a, _ = _models('ico2ico', level)
    a.train()
    b = copy.deepcopy(a)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    mods = list(a.encoder) + list(a.decoder)
    out_a = fused.run_chain(x, mods)                      # the training chain (autograd Function)
    with torch.no_grad(), switch():
        out_b, _ = fused.infer_chain(x, list(b.encoder) + list(b.decoder))
    assert torch.equal(out_a.detach(), out_b)
    sa, sb = a.state_dict(), b.state_dict()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    # and through the model: same output, same buffers as the module path gets from the training chain
    with torch.no_grad(), switch():
        y_b = b(x)
    y_a = a(x)
    assert torch.equal(y_a.detach(), y_b)


def test_eval_mode_leaves_parameters_and_buffers_untouched():
    mod, _ = _models('ico2ico_vae', 5)
    before = _state(mod)
    x, _ = data.synthetic_batch(5, 0, 4)
    with torch.no_grad(), switch():
        mod(x.cuda())
    after = mod.state_dict()
    for k in before:
        assert torch.equal(before[k], after[k]), k


# ---------------------------------------------------------------------------------------------------------- 5. default off, hooks
def test_default_off_and_hook_fallback():
    params = gm.default_params('ico2ico', 5)
    full, _ = _models('ico2ico', 5)
    enc = gm.ico2enc(params).cuda().eval()
    enc.encoder.load_state_dict(full.encoder.state_dict())
    x, _ = data.synthetic_batch(5, 0, 4)
    x = x.cuda()
    if os.environ.get('GIN_FUSED_INFER') is None:
        assert not gm._INFER                              # off unless asked for
    with torch.no_grad():
        for train in (False, True):                       # eval mode, and train mode under no_grad
            enc.train(train)
            with switch(True, False):
                y0 = enc(x)
            with switch(False, False):
                y1 = enc(x)
            assert torch.equal(y0, y1)
        enc.eval()
        with switch(False, False):
            y1 = enc(x)
        with switch():
            y_fused = enc(x)
        assert not torch.equal(y_fused, y1)              # the switch does take the fused path
        h = enc.encoder[3].conv01.register_forward_hook(lambda m, i, o: None)
        try:
            with switch():
                y2 = enc(x)
        finally:
            h.remove()
        assert torch.equal(y2, y1)


# ---------------------------------------------------------------------------------------------------------- 6. graphs and split models
def test_graph_replay_and_reproducibility():
    mod, _ = _models('ico2ico', 5)
    x, _ = data.synthetic_batch(5, 0, 36)
    xs = x.cuda()

    def fwd(inp):
        with torch.no_grad():
            return mod(inp)
    with switch():
        e1 = fwd(xs).clone()
        e2 = fwd(xs).clone()
        step = GraphedStep(fwd, (xs,))
        r1 = step().clone()
        # a later in-place load_state_dict is followed by the captured graph (constants are computed on the device)
        with torch.no_grad():
            for m in mod.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.running_var.mul_(1.5)
        r2 = step().clone()
        e3 = fwd(xs)
    assert torch.equal(e1, e2) and torch.equal(e1, r1)
    assert torch.equal(r2, e3) and not torch.equal(r2, r1)


def test_split_models_reproduce_the_whole_model():
    level, B = 5, 4
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    full, _ = _models('ico2ico', level)
    p = gm.default_params('ico2ico', level)
    enc, dec = gm.ico2enc(p).cuda().eval(), gm.enc2ico(p).cuda().eval()
    enc.encoder.load_state_dict(full.encoder.state_dict())
    dec.decoder.load_state_dict(full.decoder.state_dict())
    dec.enc2icoConv.load_state_dict(full.enc2icoConv.state_dict())
    vae, _ = _models('ico2ico_vae', level)
    pv = gm.default_params('ico2ico_vae', level)
    venc, vdec = gm.ico2enc_vae(pv).cuda().eval(), gm.enc2ico_vae(pv).cuda().eval()
    for k in ('encoder', 'mu', 'logvar'):
        getattr(venc, k).load_state_dict(getattr(vae, k).state_dict())
    vdec.decoder.load_state_dict(vae.decoder.state_dict())
    vdec.final_layer.load_state_dict(vae.final_layer.state_dict())
    with torch.no_grad(), switch():
        assert torch.equal(dec(enc(x)), full(x))
        mu, lv = vae.encode(x)
        mu2, lv2 = venc(x)
        assert torch.equal(mu, mu2) and torch.equal(lv, lv2)
        z = mu + 0.1 * lv
        assert torch.equal(vdec.decode(z), vae.decode(z))
        assert torch.equal(vdec(z)[0], vae.decode(z))


# ---------------------------------------------------------------------------------------------------------- 7. no float atomics
def test_no_floating_point_atomics_in_the_inference_kernels():
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
            if 'pole_mean_kernel' in current or 'eval_consts_kernel' in current or re.search(r'patch_conv_kernel.*Lb1EEEv', current):
                seen.add(current)
            continue
        if current in seen and re.search(r'(REDG?|ATOMG?)\.E\.ADD\.F(16|32|64)|ATOMS\.(CAST|ADD\.F)', line):
            dirty.add(current)
    assert len(seen) >= 2 + 6, sorted(seen)
    assert not dirty, sorted(dirty)
