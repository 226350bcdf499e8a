"""Exact-arithmetic parity of every tensor-core hex-conv launch of a fused training step, at the benchmarked batch sizes.

The tcgen05 kernels pick their variant from the batch: the N tile (cv2_pick_ntile), the tile-pair kernel (cv2_pair_ok), the rounds
of the persistent grid and the wgrad split-K slicing (wg2::launch) all follow from the tile count ceil(B / group) * ntiles.  The
small-batch layer tests see one variant only, and the whole-model tests compare with bf16 tolerances that a dropped tile or a
double-counted slice fits inside.  Here every operand is in {-1, 0, +1} and every bias a small integer, so each product and each
partial sum is an integer below 2^24 and the fp32 accumulators are exact whatever the tiling or summation order: the kernels must
equal the float64 oracle bit for bit (fp32 outputs equal ref.float(), fp16 outputs ref.half()).

  * the problems are those of bench.conv_calls(model, fused=True) for ico2ico I5 B=36, ico2ico_vae I5 B=36, ico2ico I6 B=16 and
    ico2ico I5 B=36 with corner_mode='zeros', launched through the wrappers the chain uses (fused._conv_fwd / _conv_dgrad /
    _conv_wgrad, weights packed by fused._pack_many); the VAE's latent heads run through the module path (gin_hexconv_fwd_bf16);
  * the xyz stem through fused._stem_conv / fused._stem_bwd;
  * edge batches chosen from the plan tile counts with the dispatch rules restated below;
  * a coverage gate: the hex-conv kernels an eager training step launches must all be launched by the parity cases.

The 16-bit operand copies are [B*P + 2B][C]: pixel rows, then per sample the north and south pole-mean rows.  The five ring pixels of
each pole carry the same value, so the oracle's pole mean (and the copy's pole row) equals it exactly.  Outputs and workspaces the
wrappers allocate are filled with NaN / a garbage byte pattern first, so a row never stored or a stale partial read back fails.
"""
import contextlib
import math
import re
from collections import namedtuple

import pytest
import torch

import bench
import plan_emulator as pe
from geniconet_b200 import _lib, fused
from geniconet_b200 import models as gm
from geniconet_b200.ico_conv import IcoConvS2S, get_plan, _stream
from oracle import icocnn_ref, ico_geometry_ref as geo

SMS = 148                     # the B200's SM count: the dispatch rules below and the coverage gate assume it
EXACT = 2 ** 24               # integers up to this are exact in fp32
TARGET = 2 ** 22              # the density rule aims the largest column sum of y^2 here, a factor 4 below EXACT
GUARD = 1024                  # fp32 elements on either side of a wgrad destination slot

CONFIGS = {   # name: (model, level, batch, corner_mode)
    'ico2ico-I5': ('ico2ico', 5, 36, 'average'),
    'ico2ico_vae-I5': ('ico2ico_vae', 5, 36, 'average'),
    'ico2ico-I6': ('ico2ico', 6, 16, 'average'),
    'ico2ico-I5-zeros': ('ico2ico', 5, 36, 'zeros'),
}
BENCH_CONFIGS = ('ico2ico-I5', 'ico2ico_vae-I5', 'ico2ico-I6')

# sibling: conv00 | conv10 as one GEMM with Cout = 2 * cout and a second bias; chain: launched by the fused chain (else by the
# IcoConvS2S module: the VAE's latent heads)
Problem = namedtuple('Problem', 'name cin cout stride level cm B sibling chain')


def _P(level):
    return 10 * 4 ** level


def _cdiv(a, b):
    return -(-a // b)


def step_problems(config):
    """The distinct tensor-core hex-conv problems of one fused training step of `config`, from bench.conv_calls."""
    model_name, level, B, cm = CONFIGS[config]
    model = getattr(gm, model_name)(gm.default_params(model_name, level, cm))
    out = []
    for name, ci, co, stride, lvl, pcm, _count in bench.conv_calls(model, True):
        sibling = name.endswith('conv00|conv10')
        out.append(Problem(name, ci, co, stride, lvl, pcm, B, sibling, sibling or name.endswith('conv01')))
    return out


def stem_problem(config):
    model_name, level, B, cm = CONFIGS[config]
    model = getattr(gm, model_name)(gm.default_params(model_name, level, cm))
    conv = model.encoder[0]
    assert conv.in_features == 3 and conv.stride == 1
    return Problem('encoder.0', 3, conv.out_features, 1, conv.subdivisions, conv.corner_mode, B, False, True)


# ------------------------------------------------------------------------------------------------ the dispatch rules, restated
# gin_conv2.cuh (cv2_pick_ntile, cv2_pair_ok, cv2_dispatch, cv2::launch, cv2::launch_pair) and gin_wgrad2.cuh (wg2::launch) at the
# default settings on SMS SMs.  They choose the edge batches and the problems that also run with an fp32 y; every parity case checks
# on the device that its forward and dgrad launches run the kernel and N tile predicted here.
def plan_tiles(level, stride, cm):
    blob = _lib.plan_blob(_lib.PLAN_HEXCONV, level, stride, cm)
    h, pf = pe.parse_conv_full(blob), pe.parse_pf(blob)
    ps = h['pfwd'] if stride == 1 else pe.parse_p2(blob)           # the forward's patch side (also stride 2's in-chart dgrad)
    dg = h['pdg']['ntiles'] if stride == 1 else ps['ntiles']
    fold = pf['ntiles'] > 0 and pf['nslots'] <= 16 and pf['mask_off'] > 0      # boundary tiles folded into the dgrad launch
    return dict(group=h['group'], fwd=ps['ntiles'], U=ps['U'], Q=ps['Q'], dg=dg, pf=pf['ntiles'] if fold else 0,
                pf_all=fold and pf['all'] != 0)


# gin_conv2_pair.cuh launch_pair: four patch stages of U rows, the 64 KB weight ring and the fixed part (gin_conv2.cuh: epilogue
# staging EPI_WARPS * 32 * STAGE_PITCH, TAB_SLOTS * TAB_ROWS table words, BAR_BYTES, the plan's ntiles * Q words) must fit in
# SMEM_LIMIT; otherwise cv2_dispatch launches single tiles of the width it picked
SMEM_LIMIT = 227 * 1024
PAIR_FIXED_BYTES = 8 * 32 * 144 + 8 * 256 * 4 + ((2 * 4 + 2 * 8 + 4 + 2 * 8) * 8 + 16) + 16 + 1024


def pair_smem_bytes(t):
    return 4 * _cdiv(t['U'] * 128, 1024) * 1024 + 65536 + PAIR_FIXED_BYTES + t['fwd'] * t['Q'] * 4


def _ctas(items, n_blocks):
    c = min(items, SMS)
    c -= c % n_blocks
    return max(c, n_blocks)


def pick_ntile(tiles, N):
    best, best_cost = 0, 0.
    for nt in (256, 128, 64):
        if N % nt:
            continue
        items = tiles * (N // nt)
        cost = _cdiv(items, _ctas(items, N // nt)) * nt * (1.5 if nt == 64 else 1.0)
        if not best or cost < best_cost * 0.999:
            best, best_cost = nt, cost
    return best


def conv_dispatch(prob, which):
    """N tile, pair kernel, tile counts and persistent rounds of the forward ('fwd') or dgrad ('dgrad') launch of `prob`."""
    t = plan_tiles(prob.level, prob.stride, prob.cm)
    groups = _cdiv(prob.B, t['group'])
    if which == 'fwd':
        K, N, total, x_total = prob.cin, prob.cout, groups * t['fwd'], 0
    else:
        K, N = prob.cout, prob.cin
        total, x_total = (0 if t['pf_all'] else groups * t['dg']), groups * t['pf']
    nt = pick_ntile(total + x_total, N)
    pair = False
    if which == 'fwd' and (K // 64) * min(nt, 128) > 128:       # streamed weights (gin_conv2.cuh: cv2_pair_ok)
        ntp = min(nt, 128)
        r1 = _cdiv(total * (N // nt), _ctas(total * (N // nt), N // nt)) * nt
        pairs = _cdiv(total, 2) * (N // ntp)
        pair = _cdiv(pairs, _ctas(pairs, N // ntp)) * 2 * ntp <= r1 and pair_smem_bytes(t) <= SMEM_LIMIT
    ntile = min(nt, 128) if pair else nt
    n_blocks = N // ntile
    units = _cdiv(total, 2) if pair else total + x_total        # tile pairs or tiles, each over all n-blocks
    per_round = _ctas(units * n_blocks, n_blocks) // n_blocks
    rounds = _cdiv(units, per_round)
    return dict(ntile=ntile, pair=pair, total=total, x_total=x_total, rounds=rounds, last=units - (rounds - 1) * per_round)


def wgrad_dispatch(prob):
    t = plan_tiles(prob.level, prob.stride, prob.cm)
    total = _cdiv(prob.B, t['group']) * t['fwd']
    nblk = 128 if prob.cout % 128 == 0 else 64
    units = (prob.cin // 64) * (prob.cout // nblk)
    slices = max(1, min(SMS // units, total))
    tpc = _cdiv(total, slices)
    return dict(total=total, slices=slices, tiles_per_cta=tpc, empty_last=(slices - 1) * tpc >= total)


# stride 1 and stride 2; both reach every edge case below 16 samples
EDGE_PROBLEMS = (('ico2ico-I5', 'decoder.0.conv00|conv10'), ('ico2ico-I5', 'encoder.4.conv00|conv10'))


def edge_batches(prob, bmax=48):
    """{case: the smallest batch that gives it}: 'empty_slice' (the last wgrad slice has no tiles), 'odd_pair' (an odd tile count
    under the pair kernel: the ghost half of the last pair is live), 'single_last' (the last persistent round of the forward or the
    dgrad is one tile)."""
    found = {}
    for B in range(1, bmax + 1):
        p = prob._replace(B=B)
        f, d = conv_dispatch(p, 'fwd'), conv_dispatch(p, 'dgrad')
        if 'empty_slice' not in found and wgrad_dispatch(p)['empty_last']:
            found['empty_slice'] = B
        if 'odd_pair' not in found and f['pair'] and f['total'] % 2 == 1:
            found['odd_pair'] = B
        if 'single_last' not in found and any(not r['pair'] and r['rounds'] > 1 and r['last'] == 1 for r in (f, d)):
            found['single_last'] = B
    return found


def _edge_cases():
    out = []
    for config, name in EDGE_PROBLEMS:
        prob = next(p for p in step_problems(config) if p.name == name)
        for case, B in sorted(edge_batches(prob).items()):
            out.append(pytest.param(config, prob._replace(B=B), case, id='%s-%s-s%d-%s-B%d' % (config, name, prob.stride, case, B)))
    return out


def predicted(prob):
    """{(kernel, N tile)} of the forward and the dgrad launch of `prob` by the rules above."""
    out = set()
    for which in ('fwd', 'dgrad'):
        d = conv_dispatch(prob, which)
        out.add(('patch_conv_pair_kernel' if d['pair'] else 'patch_conv_kernel', d['ntile']))
    return out


# ------------------------------------------------------------------------------------------------ operands and the reference
def ternary(shape, p, gen):
    """float64 values in {-1, 0, +1}: nonzero with probability p, either sign equally likely."""
    r = torch.rand(shape, generator=gen, device=gen.device, dtype=torch.float64)
    return (r < p / 2).double() - ((r >= p / 2) & (r < p)).double()


def equalise_poles(m, level):
    """Give the five ring pixels of each pole, per sample and channel, the value of the first one (in place on [B, C, 5n, 2n])."""
    flat = m.view(m.shape[0], m.shape[1], -1)
    for ring in torch.from_numpy(geo.pole_rings(level).astype('int64')).to(m.device):
        flat[:, :, ring] = flat[:, :, ring[:1]]
    return m


def operand(m, level, dtype):
    """The 16-bit operand copy [B*P + 2B][C] of a pole-equalised map (row B*P + 2b + pole: the pole mean of sample b), in a
    torch.bfloat16 container as the chain keeps it."""
    B, C = m.shape[:2]
    rings = torch.from_numpy(geo.pole_rings(level)[:, 0].astype('int64')).to(m.device)
    poles = m.reshape(B, C, -1)[:, :, rings].permute(0, 2, 1).reshape(2 * B, C)
    return torch.cat((rows_of(m), poles)).to(dtype).view(torch.bfloat16).contiguous()


def rows_of(m):
    """[B * P][C] rows of a [B, C, H, W] map."""
    return m.permute(0, 2, 3, 1).reshape(-1, m.shape[1])


def density(rows, K):
    """Nonzero probability of x and W: E[y^2] = 7 K p^2 + E[b^2] per output, so the column sum of y^2 over `rows` rows stays near
    TARGET while every tap and 64-channel block keeps nonzero weights."""
    return min(1.0, math.sqrt(max(TARGET / rows - 1.0, 0.5) / (7 * K)))


def build_case(prob, gen):
    """Integer operands of `prob` and the float64 oracle's y, dx and dW, with the exactness premise asserted."""
    lvl_out = prob.level - (1 if prob.stride == 2 else 0)
    n_in, n_out = 2 ** prob.level, 2 ** lvl_out
    p = density(prob.B * _P(lvl_out), prob.cin)
    x = equalise_poles(ternary((prob.B, prob.cin, 5 * n_in, 2 * n_in), p, gen), prob.level)
    W = ternary((prob.cout, prob.cin, 7), p, gen)
    b = ternary((prob.cout,), 2. / 3., gen)
    dy = equalise_poles(ternary((prob.B, prob.cout, 5 * n_out, 2 * n_out), 0.5, gen), lvl_out)
    ref = icocnn_ref.IcoConvS2S(prob.cin, prob.cout, prob.stride, True, prob.level, prob.cm).to(device=x.device, dtype=torch.float64)
    with torch.no_grad():
        ref.weight.copy_(W)
        ref.bias.copy_(b)
    xr = x.clone().requires_grad_(True)
    y = ref(xr)
    y.backward(dy)
    y = rows_of(y.detach())
    c = dict(x=x, W=W, b=b, dy=dy, y=y, ysum=y.sum(0), ysq=(y * y).sum(0), dx=rows_of(xr.grad), dW=ref.weight.grad.detach(),
             lvl_out=lvl_out)
    # every partial of the statistics is bounded by its column's sum of |y| or y^2, every wgrad partial by the column sum of
    # |x * dy| <= sum |dy| (|x| <= 1), every dgrad partial by 7 K (|W dy| <= 1)
    c['bounds'] = dict(sum_abs_y=y.abs().sum(0).max().item(), sum_y2=c['ysq'].max().item(),
                       wgrad=rows_of(dy).abs().sum(0).max().item(), dgrad=7 * prob.cout)
    for k, v in c['bounds'].items():
        assert v < EXACT, 'exactness premise: %s = %d' % (k, v)
    assert torch.equal(c['dx'], c['dx'].round()) and torch.equal(c['dW'], c['dW'].round()) and torch.equal(y, y.round())
    return c


# ------------------------------------------------------------------------------------------------ the launches
def _poisoned(shape, dtype, dev):
    t = torch.empty(shape, dtype=dtype, device=dev)
    return t.fill_(0x7F) if dtype == torch.uint8 else t.fill_(float('nan'))     # workspaces: 0x7F7F7F7F = 3.4e38 per fp32 word


@contextlib.contextmanager
def poisoned_outputs():
    """Every buffer the fused wrappers allocate comes filled with NaN (outputs) or 0x7F bytes (workspaces)."""
    saved = fused._empty
    fused._empty = _poisoned
    try:
        yield
    finally:
        fused._empty = saved


def launch(prob, x, W, b, dy, dev):
    """The step's launches of `prob` on float64 maps x [B, cin, ...] / dy [B, cout, ...] and weights W, b.  Returns the outputs:
    y, the statistics partials (buffer, rows) or None, dx, dW and dW written into a slot of a larger buffer (with its guards)."""
    B, cin, cout = prob.B, prob.cin, prob.cout
    lvl_out = prob.level - (1 if prob.stride == 2 else 0)
    plan = get_plan(_lib.PLAN_HEXCONV, prob.level, prob.stride, prob.cm, dev)
    W32, b32 = W.float().contiguous(), b.float().contiguous()
    dyb = operand(dy, lvl_out, torch.bfloat16)
    xw = operand(x, prob.level, torch.bfloat16)
    xb = operand(x, prob.level, _lib.forward_operand_dtype())
    half = cout // 2
    if prob.chain:
        packed = fused._pack_many([(W32[:half].contiguous(), W32[half:].contiguous(), cin) if prob.sibling else (W32, None, cin)])[0]
        y, parts = fused._conv_fwd(plan, xb, packed, b32[:half] if prob.sibling else b32, B, cin, cout, _P(lvl_out),
                                   bias1=b32[half:] if prob.sibling else None)
    else:                                         # IcoConvS2S on the tensor cores (ico_conv._HexConvFn)
        packed = fused._pack(W32, cin, cout)
        y, parts = fused._empty((B * _P(lvl_out), cout), torch.float32, dev), None
        _lib.check(_lib.lib.gin_hexconv_fwd_bf16(plan.host_ptr, plan.dev_ptr, xb.data_ptr(), packed.data_ptr(), b32.data_ptr(), y.data_ptr(),
                                                 B, cin, cout, _stream()), 'gin_hexconv_fwd_bf16')
    dx = fused._conv_dgrad(plan, dyb, packed, B, cin, cout, _P(prob.level))
    dW = fused._conv_wgrad(plan, xw, dyb, B, cin, cout)
    n = 7 * cin * cout
    slot = torch.full((n + 2 * GUARD,), float('nan'), dtype=torch.float32, device=dev)
    fused._conv_wgrad(plan, xw, dyb, B, cin, cout, out=slot[GUARD:GUARD + n].view(cout, cin, 7))
    return dict(y=y, parts=parts, dx=dx, dW=dW, slot=slot)


def launch_stem(prob, x, W, b, dy, dev):
    """fused._stem_conv and fused._stem_bwd (every gradient) on fp32 copies of the integer maps."""
    conv = type('Conv', (), dict(subdivisions=prob.level, out_features=prob.cout, corner_mode=prob.cm, weight=W.float().contiguous(),
                                 bias=b.float().contiguous()))
    x32 = x.float().contiguous()                  # NCHW, as the step's xyz input (data.synthetic_batch)
    plan, packed, xs, strides, y, parts = fused._stem_conv(x32, conv)
    st = dict(plan=plan, strides=strides, C=prob.cout, level=prob.level, xs=xs, packed=packed)
    dW, db, dx = fused._stem_bwd(st, rows_of(dy).float().contiguous(), prob.B, True, True, True)
    return dict(y=y, parts=parts, dx=rows_of(dx), dW=dW, db=db)


# ------------------------------------------------------------------------------------------------ comparison
def assert_exact(what, got, want, level=None):
    """got == want element for element (NaN counts as a difference); on failure report where: (sample, chart, row, column,
    channel, 64-channel block) for [B * P][C] maps, (co, ci, tap) for weight gradients."""
    got, want = got.double(), want.double().to(got.device)
    assert got.shape == want.shape, '%s: shape %s, want %s' % (what, tuple(got.shape), tuple(want.shape))
    bad = ~(got == want)
    nbad = int(bad.sum())
    if nbad == 0:
        return
    lines = []
    for idx in bad.nonzero()[:12].tolist():
        g, w = got[tuple(idx)].item(), want[tuple(idx)].item()
        if level is not None and got.dim() == 2:
            r, c = idx
            n = 2 ** level
            s, pix = divmod(r, _P(level))
            h, j = divmod(pix, 2 * n)
            lines.append('  sample %d chart %d row %d col %d (pixel %d) channel %d (block %d): %r, want %r' % (s, h // n, h % n, j, pix, c, c // 64, g, w))
        elif got.dim() == 3:
            lines.append('  co %d ci %d tap %d: %r, want %r' % (idx[0], idx[1], idx[2], g, w))
        else:
            lines.append('  %s: %r, want %r' % (idx, g, w))
    rows = bad.reshape(bad.shape[0], -1).any(1).nonzero().flatten()
    raise AssertionError('%s: %d of %d elements differ (in %d rows, first %d, last %d)\n%s' % (
        what, nbad, bad.numel(), rows.numel(), rows[0].item(), rows[-1].item(), '\n'.join(lines)))


def check(prob, c, out):
    lvl_out = c['lvl_out']
    y = out['y']
    assert_exact('y', y, c['y'].half() if y.dtype == torch.float16 else c['y'].float(), lvl_out)
    if prob.chain:
        assert out['parts'] is not None, 'the forward of a chain convolution returns its BatchNorm statistics'
        pbuf, n = out['parts']
        s = pbuf[:n * 2 * prob.cout].view(n, 2, prob.cout).double().sum(0)
        assert_exact('column sums of y', s[0], c['ysum'])
        assert_exact('column sums of y^2', s[1], c['ysq'])
    assert_exact('dx', out['dx'], c['dx'].float(), prob.level)
    assert_exact('dW', out['dW'], c['dW'].float())
    if 'slot' in out:
        slot, n = out['slot'], 7 * prob.cin * prob.cout
        assert_exact('dW written into a bucket slot', slot[GUARD:GUARD + n].view(prob.cout, prob.cin, 7), c['dW'].float())
        assert torch.isnan(slot[:GUARD]).all() and torch.isnan(slot[GUARD + n:]).all(), 'wgrad wrote outside its destination slot'
    if out.get('db') is not None:
        assert_exact('db', out['db'], rows_of(c['dy']).sum(0).float())


def run_parity(prob, seed):
    """Launches `prob` on integer operands, checks every output against the reference and, for a tensor-core problem, that its
    forward and dgrad ran the predicted variants.  Returns the {(kernel, N tile)} of the tensor-core launches seen."""
    dev = torch.device('cuda')
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    c = build_case(prob, gen)
    out = {}
    with poisoned_outputs():
        names = _hexconv_kernels(lambda: out.update((launch_stem if prob.cin == 3 else launch)(prob, c['x'], c['W'], c['b'], c['dy'], dev)))
    try:
        check(prob, c, out)
    finally:
        del c, out
        torch.cuda.empty_cache()
    seen = variants(names)
    if prob.cin != 3:
        assert seen == predicted(prob), 'ran %s, the dispatch rules predict %s' % (sorted(seen), sorted(predicted(prob)))
    return seen


# ------------------------------------------------------------------------------------------------ parametrisation
def _parity_cases():
    """Every distinct problem once (the configurations share most of theirs), plus an fp32-y run of the first chain problem of each
    forward N tile per configuration."""
    out, seen = [], set()
    for config in CONFIGS:
        tiles_y32 = set()
        for prob in step_problems(config):
            key = prob._replace(name='')
            if key not in seen:
                seen.add(key)
                out.append(pytest.param(prob, True, id='%s-%s' % (config, prob.name)))
            nt = conv_dispatch(prob, 'fwd')['ntile']
            if prob.chain and fused._Y16 and (config, nt) not in tiles_y32:
                tiles_y32.add((config, nt))
                out.append(pytest.param(prob, False, id='%s-%s-y32' % (config, prob.name)))
    return out


PARITY_CASES = _parity_cases()
STEM_CASES = [pytest.param(stem_problem(c), id=c) for c in CONFIGS]
EDGE_CASES = _edge_cases()


@pytest.mark.gpu
@pytest.mark.parametrize('prob,y16', PARITY_CASES)
def test_conv_launch_parity(prob, y16, monkeypatch):
    if not y16:
        monkeypatch.setattr(fused, '_Y16', False)
    run_parity(prob, 1)


@pytest.mark.gpu
@pytest.mark.parametrize('prob', STEM_CASES)
def test_stem_launch_parity(prob):
    run_parity(prob, 2)


@pytest.mark.gpu
@pytest.mark.parametrize('config,prob,case', EDGE_CASES)
def test_edge_batch_parity(config, prob, case):
    seen = run_parity(prob, 3)
    if case == 'odd_pair':
        assert ('patch_conv_pair_kernel', conv_dispatch(prob, 'fwd')['ntile']) in seen, seen
    elif case == 'single_last':
        single = [d for d in (conv_dispatch(prob, w) for w in ('fwd', 'dgrad')) if not d['pair'] and d['rounds'] > 1 and d['last'] == 1]
        assert single and ('patch_conv_kernel', single[0]['ntile']) in seen, seen


# ------------------------------------------------------------------------------------------------ coverage gate
HEXCONV_KERNEL = re.compile(r'patch_conv_kernel<|patch_conv_pair_kernel<|wgrad_patch_kernel<|wgrad_reduce_kernel|narrow::|'
                            r'gather_gemm_simt_kernel|wgrad_simt_kernel|unpack_wgrad_kernel')


def _hexconv_kernels(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and HEXCONV_KERNEL.search(e.name)}


def variants(names):
    """{(kernel, N tile)} of the tensor-core forward / dgrad kernels among the kernel names `names`."""
    return {(m.group(1), int(m.group(2))) for k in names for m in [re.search(r'(patch_conv(?:_pair)?_kernel)<(\d+)', k)] if m}


def _step_kernels(config):
    from geniconet_b200 import data, losses
    model_name, level, B, cm = CONFIGS[config]
    params = gm.default_params(model_name, level, cm)
    torch.manual_seed(0)
    model = getattr(gm, model_name)(params).cuda()
    f = (params['ico']['factor_pos'], params['ico']['factor_nor'], params['ico']['factor_lap'])
    crit = losses.P2PKLD_Loss(level, *f, 1.0) if model_name == 'ico2ico_vae' else losses.P2P_Loss(level, *f)
    x, t = (v.cuda() for v in data.synthetic_batch(level, 0, B))

    def step():
        crit(model(x), t).backward()
    step()                                      # first launches: module loads, plans, packed weights
    names = _hexconv_kernels(step)
    del model, x, t
    return names


def _parity_kernels(config):
    """The kernels of the parity launches of `config`: its problems, its stem and the edge batches taken from its problems (operands
    of zeros: the values do not choose the variant, and an fp32 y is an argument of the same kernels)."""
    dev = torch.device('cuda')
    probs = step_problems(config) + [stem_problem(config)]
    probs += [p.values[1] for p in EDGE_CASES if p.values[0] == config]

    def run():
        for prob in probs:
            lvl_out = prob.level - (1 if prob.stride == 2 else 0)
            n_in, n_out = 2 ** prob.level, 2 ** lvl_out
            x = torch.zeros(prob.B, prob.cin, 5 * n_in, 2 * n_in, dtype=torch.float64, device=dev)
            dy = torch.zeros(prob.B, prob.cout, 5 * n_out, 2 * n_out, dtype=torch.float64, device=dev)
            W = torch.zeros(prob.cout, prob.cin, 7, dtype=torch.float64, device=dev)
            b = torch.zeros(prob.cout, dtype=torch.float64, device=dev)
            (launch_stem if prob.cin == 3 else launch)(prob, x, W, b, dy, dev)
    return _hexconv_kernels(run)


def predicted_variants(config):
    """{(kernel, N tile)} of the forward and dgrad launches of `config`'s problems by the dispatch rules above."""
    return set().union(*(predicted(p) for p in step_problems(config)))


@pytest.mark.gpu
@pytest.mark.parametrize('config', BENCH_CONFIGS)
def test_step_kernels_covered(config):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms != SMS:
        pytest.skip('the device has %d SMs: the default dispatch differs from the %d-SM B200 the parity cases were chosen for' % (sms, SMS))
    step = _step_kernels(config)
    parity = _parity_kernels(config)
    torch.cuda.empty_cache()
    print('\n%s: hex-conv kernels of the training step:\n  %s' % (config, '\n  '.join(sorted(step))))
    print('%s: hex-conv kernels of the parity cases:\n  %s' % (config, '\n  '.join(sorted(parity))))
    assert step, 'the profiler saw no hex-conv kernel in the training step'
    assert step <= parity, 'launched by the step but by no parity case: %s' % sorted(step - parity)
    seen = variants(step)
    assert seen == predicted_variants(config), 'the dispatch rules of this file predict %s' % sorted(predicted_variants(config))
    # the variants the small-batch layer tests never reach
    assert {('patch_conv_kernel', 128), ('patch_conv_kernel', 256)} <= seen and any(k == 'patch_conv_pair_kernel' for k, _ in seen), seen


# ------------------------------------------------------------------------------------------------ host side, no device needed
def test_problem_list():
    """One problem per distinct launch of the step, with the step's shapes: sibling GEMMs as one problem of 2 * cout outputs (the
    dgrad K), chain problems launched by the fused chain, the VAE's latent heads by the module; 'zeros' has its own plans."""
    for config, (model_name, level, B, cm) in CONFIGS.items():
        model = getattr(gm, model_name)(gm.default_params(model_name, level, cm))
        probs = step_problems(config)
        assert len({p._replace(name='') for p in probs}) == len(probs) and all(p.B == B and p.cm == cm for p in probs)
        blocks = [(n, m) for n, m in model.named_modules() if fused._is_block(m)]
        for name, blk in blocks:
            sib = next(p for p in probs if p.name == name + '.conv00|conv10')
            assert sib.sibling and sib.chain and sib.cout == 2 * blk.conv00.out_features == 2 * blk.conv10.out_features
            assert (sib.cin, sib.stride, sib.level) == (blk.conv00.in_features, blk.conv00.stride, blk.conv00.subdivisions)
            assert (sib.cout // 2) % 64 == 0                   # gin_hexconv_fwd_bf16_stats2: the bias split is a multiple of 64
        tc = {(m.in_features, m.out_features, m.stride, m.subdivisions) for n, m in model.named_modules()
              if isinstance(m, IcoConvS2S) and m.in_features % 64 == 0}
        covered = {(p.cin, p.cout // (2 if p.sibling else 1), p.stride, p.level) for p in probs}
        assert tc <= covered, tc - covered                  # every tensor-core convolution of the model is part of a problem
        modules = [p for p in probs if not p.chain]
        assert [p.name for p in modules] == (['mu.0'] if model_name == 'ico2ico_vae' else [])
        stem = stem_problem(config)
        assert (stem.cin, stem.level, stem.cm) == (3, level, cm)
    for level, stride in ((5, 1), (4, 2)):
        zeros, average = (_lib.plan_blob(_lib.PLAN_HEXCONV, level, stride, m) for m in ('zeros', 'average'))
        assert zeros.shape != average.shape or (zeros != average).any()


def test_dispatch_rules_reach_the_benchmark_variants():
    """At the benchmark batches the step runs 64-, 128- and 256-wide tiles, the pair kernel, grids of many rounds and multi-tile
    wgrad slices; the small-batch layer tests run none of these.  Every pair launch there has an even tile count (the level-3
    stride-2 plan is too large for the pair kernel's shared memory): an odd count under the pair kernel occurs in the edge batches
    only."""
    pairs = odd = rounds = tpc = 0
    widths = set()
    for config in BENCH_CONFIGS:
        for prob in step_problems(config):
            for which in ('fwd', 'dgrad'):
                d = conv_dispatch(prob, which)
                widths.add(d['ntile'])
                pairs += d['pair']
                odd += d['pair'] and d['total'] % 2 == 1
                rounds = max(rounds, d['rounds'])
            tpc = max(tpc, wgrad_dispatch(prob)['tiles_per_cta'])
    assert widths == {64, 128, 256} and pairs and not odd and rounds >= 20 and tpc >= 40, (widths, pairs, odd, rounds, tpc)
    enc5 = next(p for p in step_problems('ico2ico-I5') if p.name == 'encoder.5.conv00|conv10')
    assert pair_smem_bytes(plan_tiles(enc5.level, enc5.stride, enc5.cm)) > SMEM_LIMIT and not conv_dispatch(enc5, 'fwd')['pair']


@pytest.mark.parametrize('config,name', EDGE_PROBLEMS)
def test_edge_batch_selection(config, name):
    """The edge batches come from the plan headers through the dispatch rules, and each one is the case it is named for."""
    prob = next(p for p in step_problems(config) if p.name == name)
    found = edge_batches(prob)
    assert set(found) == {'empty_slice', 'odd_pair', 'single_last'}, found
    w = wgrad_dispatch(prob._replace(B=found['empty_slice']))
    assert w['slices'] > 1 and (w['slices'] - 1) * w['tiles_per_cta'] >= w['total']
    f = conv_dispatch(prob._replace(B=found['odd_pair']), 'fwd')
    assert f['pair'] and f['total'] % 2 == 1
    rs = [conv_dispatch(prob._replace(B=found['single_last']), w) for w in ('fwd', 'dgrad')]
    assert any(not r['pair'] and r['rounds'] > 1 and r['last'] == 1 for r in rs)
    assert len([c for c in EDGE_CASES if c.values[:2] == (config, prob._replace(B=c.values[1].B))]) == 3


@pytest.mark.parametrize('stride,cm', [(1, 'average'), (2, 'average'), (1, 'zeros')])
def test_reference_construction(stride, cm):
    """The operands and the float64 reference at a tiny batch on the CPU: equalised poles make the oracle's pole mean (and the
    operand copy's pole row) the ring value exactly, every value is an integer, and the asserted sums stay below 2^24."""
    gen = torch.Generator()
    gen.manual_seed(0)
    prob = Problem('tiny', 64, 128, stride, 3, cm, 2, True, True)
    c = build_case(prob, gen)
    rings = torch.from_numpy(geo.pole_rings(prob.level).astype('int64'))
    flat = c['x'].reshape(prob.B, prob.cin, -1)
    assert torch.equal(flat[:, :, rings].mean(-1), flat[:, :, rings[:, 0]])
    assert flat[:, :, rings].abs().sum() > 0
    xb = operand(c['x'], prob.level, torch.float16).view(torch.float16)
    P = _P(prob.level)
    assert xb.shape == (prob.B * P + 2 * prob.B, prob.cin)
    assert torch.equal(xb[:prob.B * P].double(), rows_of(c['x']))
    for s in range(prob.B):
        for pole in range(2):
            assert torch.equal(xb[prob.B * P + 2 * s + pole].double(), c['x'][s].reshape(prob.cin, -1)[:, rings[pole, 0]])
    assert set(c['W'].unique().tolist()) <= {-1., 0., 1.} and set(c['x'].unique().tolist()) <= {-1., 0., 1.}
    for t in range(7):                                    # every tap and 64-channel block carries nonzero weight
        assert (c['W'][:, :, t].reshape(2, 64, 1, 64).abs().sum((1, 3)) > 0).all()
    assert all(v < EXACT for v in c['bounds'].values())


def test_density_rule_at_the_benchmark_sizes():
    """The density rule keeps the expected column sum of y^2 (7 K p^2 + E[b^2] per row) at most TARGET = EXACT / 4 for every
    problem of the benchmark batches, so the per-case assertion of the measured sums has room to spare."""
    for config in CONFIGS:
        for prob in step_problems(config) + [stem_problem(config)]:
            rows = prob.B * _P(prob.level - (1 if prob.stride == 2 else 0))
            p = density(rows, prob.cin)
            assert rows * (7 * prob.cin * p * p + 2. / 3.) <= TARGET and 7 * prob.cin * p * p >= 1.0, (config, prob.name, p)
