"""Synchronised BatchNorm in the fused chains.

One GPU: the C ABI with "virtual ranks" (a map split by whole samples, one record per range, the records concatenated as the
all-gather would), and a converted model without a process group, which must run exactly as the unconverted one.  Two or more
GPUs: tests/diag/syncbn_worker.py under torchrun, skipped below its device count."""
import copy
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

from geniconet_b200 import _lib, data, fused, losses, models as gm
from geniconet_b200.graph import GraphedStep

pytestmark = pytest.mark.gpu
L = _lib.lib
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _s():
    return torch.cuda.current_stream().cuda_stream


def _P(level):
    return 10 * 4 ** level


def _ptr(t, off=0):
    return t.data_ptr() + t.element_size() * off if t is not None else None


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


# ---------------------------------------------------------------------------------------------------------- 1. the ABI, virtual ranks
SPLITS = {1: (6,), 2: (3, 3), 3: (1, 2, 3)}          # samples per virtual rank; three ranges are deliberately uneven


class _Bn:
    """gamma, beta and running statistics of one BatchNorm"""

    def __init__(self, C, seed):
        g = _gen(seed)
        self.w = torch.rand(C, device='cuda', generator=g) + 0.5
        self.b = torch.randn(C, device='cuda', generator=g) * 0.1
        self.rm = torch.randn(C, device='cuda', generator=g) * 0.1
        self.rv = torch.rand(C, device='cuda', generator=g) + 0.5
        self.nbt = torch.zeros((), dtype=torch.int64, device='cuda')
        self.eps, self.mom = 1e-5, 0.1

    def clone(self):
        o = copy.copy(self)
        o.rm, o.rv, o.nbt = self.rm.clone(), self.rv.clone(), self.nbt.clone()
        return o

    def args(self, stat):
        return [self.w.data_ptr(), self.b.data_ptr(), self.eps, self.mom, self.rm.data_ptr(), self.rv.data_ptr(), self.nbt.data_ptr(), stat.data_ptr()]


NULL_BN = [None, None, 0.0, 0.0, None, None, None, None]


def _ranges(B, P, k):
    first, out = 0, []
    for n in SPLITS[k]:
        out.append((first * P, (first + n) * P, first, n))
        first += n
    assert first == B
    return out


def _fp64_stats(y, bn):
    """mean, invstd and running statistics of torch's BatchNorm over the whole map, in float64"""
    yd = y.double()
    mean, var = yd.mean(0), yd.var(0, unbiased=False)
    n = yd.shape[0]
    rm = (1 - bn.mom) * bn.rm.double() + bn.mom * mean
    rv = (1 - bn.mom) * bn.rv.double() + bn.mom * var * n / (n - 1)
    return mean, 1 / torch.sqrt(var + bn.eps), rm, rv


def _close(a, b, tol):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item() <= tol


@pytest.mark.parametrize('k', [1, 2, 3])
@pytest.mark.parametrize('level,C', [(3, 64), (4, 256)])
def test_forward_records_single(level, C, k):
    B, P = 6, _P(level)
    y = torch.randn(B * P, C, device='cuda', generator=_gen(1)) * 2 + 0.5
    bn0 = _Bn(C, 2)
    rec_len = L.gin_bn_sync_record_bytes(C, 0) // 8
    ws = torch.empty(L.gin_bn_ws_bytes(C), dtype=torch.uint8, device='cuda')
    recs = torch.empty(k, rec_len, dtype=torch.float64, device='cuda')
    for r, (a, b, _, _) in enumerate(_ranges(B, P, k)):
        _lib.check(L.gin_bn_sync_stats_total(_ptr(y, a * C), C, b - a, C, _ptr(recs[r]), ws.data_ptr(), _s()), 'total')
    bn, stat = bn0.clone(), torch.empty(4 * C, device='cuda')
    _lib.check(L.gin_bn_sync_stats_final(recs.data_ptr(), k, C, *bn.args(stat), *NULL_BN, _s()), 'final')
    if k == 1:                                                   # bit for bit gin_bn_stats
        ref, sref = bn0.clone(), torch.empty(4 * C, device='cuda')
        _lib.check(L.gin_bn_stats(y.data_ptr(), C, B * P, C, ref.w.data_ptr(), ref.b.data_ptr(), ref.eps, ref.mom, ref.rm.data_ptr(), ref.rv.data_ptr(),
                                  ref.nbt.data_ptr(), sref.data_ptr(), ws.data_ptr(), _s()), 'gin_bn_stats')
        for u, v in ((stat, sref), (bn.rm, ref.rm), (bn.rv, ref.rv), (bn.nbt, ref.nbt)):
            assert torch.equal(u, v)
    mean, invstd, rm, rv = _fp64_stats(y, bn0)
    assert _close(stat[:C], mean, 1e-5) and _close(stat[C:2 * C], invstd, 1e-5)
    assert _close(bn.rm, rm, 1e-5) and _close(bn.rv, rv, 1e-5) and int(bn.nbt) == 1      # the uneven split too: the global count


@pytest.mark.parametrize('k', [1, 2, 3])
def test_forward_records_pair_from_parts(k):
    """Epilogue partials of a sibling GEMM: [nparts][2][2C], BatchNorm A in columns [0, C), B in [C, 2C)."""
    C, nparts = 128, 37
    # per part: sum y of either sign, sum y^2 large enough that every variance is positive
    parts = [torch.randn(nparts, 2, 2 * C, device='cuda', generator=_gen(10 + r)) for r in range(k)]
    for p in parts:
        p[:, 1] = p[:, 1].abs() * 50 + 20
    rows = [1000 * (r + 1) for r in range(k)]
    A0, B0 = _Bn(C, 3), _Bn(C, 4)
    recs = torch.empty(k, L.gin_bn_sync_record_bytes(C, 1) // 8, dtype=torch.float64, device='cuda')
    for r in range(k):
        _lib.check(L.gin_bn_sync_stats_total_from_parts(parts[r].data_ptr(), nparts, 2 * C, rows[r], C, 0, C, _ptr(recs[r]), _s()), 'total')
    A, Bb = A0.clone(), B0.clone()
    sA, sB = torch.empty(4 * C, device='cuda'), torch.empty(4 * C, device='cuda')
    _lib.check(L.gin_bn_sync_stats_final(recs.data_ptr(), k, C, *A.args(sA), *Bb.args(sB), _s()), 'final')
    allp = torch.cat(parts, 0)
    if k == 1:                                                   # bit for bit gin_bn_stats_from_parts2
        rA, rB = A0.clone(), B0.clone()
        tA, tB = torch.empty(4 * C, device='cuda'), torch.empty(4 * C, device='cuda')
        _lib.check(L.gin_bn_stats_from_parts2(allp.data_ptr(), nparts, 2 * C, rows[0], C, 0, *rA.args(tA)[:7], tA.data_ptr(), C, *rB.args(tB)[:7],
                                              tB.data_ptr(), _s()), 'gin_bn_stats_from_parts2')
        for u, v in ((sA, tA), (sB, tB), (A.rm, rA.rm), (A.rv, rA.rv), (Bb.rm, rB.rm), (Bb.rv, rB.rv), (A.nbt, rA.nbt), (Bb.nbt, rB.nbt)):
            assert torch.equal(u, v)
    n = sum(rows)
    for q, (bn0, bn, st) in enumerate(((A0, A, sA), (B0, Bb, sB))):
        s = allp.double().sum(0)[:, q * C:(q + 1) * C]
        mean = s[0] / n
        var = s[1] / n - mean * mean
        assert _close(st[:C], mean, 1e-6) and _close(st[C:2 * C], 1 / torch.sqrt(var + bn0.eps), 1e-6)
        assert _close(bn.rv, (1 - bn0.mom) * bn0.rv.double() + bn0.mom * var * n / (n - 1), 1e-6)


def _act_mask(y, stat, B, level, C):
    """The bf16 ReLU mask copy gin_bn_act_fwd(y, stat, relu = 1) writes, [B*P + 2B][C]"""
    out_w = torch.empty(B * _P(level) + 2 * B, C, dtype=torch.bfloat16, device='cuda')
    _lib.check(L.gin_bn_act_fwd(y.data_ptr(), C, stat.data_ptr(), None, 0, None, 0, 1, None, None, out_w.data_ptr(), B, level, C, _s()),
               'gin_bn_act_fwd')
    return out_w


def _stat_of(y, C):
    bn, stat = _Bn(C, 7), torch.empty(4 * C, device='cuda')
    ws = torch.empty(L.gin_bn_ws_bytes(C), dtype=torch.uint8, device='cuda')
    _lib.check(L.gin_bn_stats(y.data_ptr(), C, y.shape[0], C, bn.w.data_ptr(), bn.b.data_ptr(), bn.eps, bn.mom, None, None, None, stat.data_ptr(),
                              ws.data_ptr(), _s()), 'gin_bn_stats')
    return stat


def _dy_ref(dout, keep, yd, stat, C):
    """float64 dy of BatchNorm (batch statistics of the whole map, scale / mean / invstd as the forward wrote them) under g = dout * keep"""
    g = dout.double() * keep
    mean, invstd, scale = stat[:C].double(), stat[C:2 * C].double(), stat[2 * C:3 * C].double()
    yh = (yd - mean) * invstd
    return scale * (g - g.mean(0) - yh * (g * yh).mean(0)), g, yh


@pytest.mark.parametrize('k', [1, 2, 3])
@pytest.mark.parametrize('C', [64, 512])
def test_backward_records_single(C, k):
    B, level = 6, 3
    P = _P(level)
    y = torch.randn(B * P, C, device='cuda', generator=_gen(20)) + 0.3
    stat = _stat_of(y, C)
    dout = torch.randn(B * P, C, device='cuda', generator=_gen(21))
    rec_len = L.gin_bn_sync_record_bytes(C, 0) // 8
    ws = torch.empty(L.gin_bn_ws_bytes(C), dtype=torch.uint8, device='cuda')
    recs = torch.empty(k, rec_len, dtype=torch.float64, device='cuda')
    ranges = _ranges(B, P, k)
    masks = [_act_mask(y[a:b], stat, n, level, C) for a, b, _, n in ranges]
    for r, (a, b, _, n) in enumerate(ranges):
        _lib.check(L.gin_bn_sync_bwd_reduce(_ptr(dout, a * C), C, masks[r].data_ptr(), _ptr(y, a * C), C, 0, stat.data_ptr(), _ptr(recs[r]),
                                            ws.data_ptr(), n, level, C, 1, _s()), 'reduce')
    dy_f = torch.empty(B * P, C, device='cuda')
    bstats = []
    for r, (a, b, _, n) in enumerate(ranges):
        bs = torch.empty(4 * C, device='cuda')
        _lib.check(L.gin_bn_sync_bwd_final(recs.data_ptr(), k, r, C, bs.data_ptr(), None, _s()), 'bwd_final')
        _lib.check(L.gin_bn_bwd_apply(_ptr(dout, a * C), C, masks[r].data_ptr(), _ptr(y, a * C), C, 0, stat.data_ptr(), bs.data_ptr(), None, 0,
                                      _ptr(dy_f, a * C), C, n, level, C, 1, _s()), 'apply')
        bstats.append(bs)
    if k == 1:                                                   # bit for bit gin_bn_act_bwd
        bs_ref, dy_ref = torch.empty(4 * C, device='cuda'), torch.empty(B * P, C, device='cuda')
        _lib.check(L.gin_bn_act_bwd(dout.data_ptr(), C, masks[0].data_ptr(), y.data_ptr(), C, 0, stat.data_ptr(), bs_ref.data_ptr(), None, 0,
                                    dy_ref.data_ptr(), C, ws.data_ptr(), B, level, C, 1, _s()), 'gin_bn_act_bwd')
        assert torch.equal(bstats[0], bs_ref) and torch.equal(dy_f, dy_ref)
    keep = torch.cat([(m[:n * P].float() > 0).double() for m, (_, _, _, n) in zip(masks, ranges)], 0)
    ref, g, yh = _dy_ref(dout, keep, y.double(), stat, C)
    assert _close(dy_f, ref, 1e-4)
    for bs, (a, b, _, _) in zip(bstats, ranges):                  # dbeta, dgamma: this rank's sums; the means: over every rank
        assert _close(bs[:C], g[a:b].sum(0), 1e-5) and _close(bs[C:2 * C], (g[a:b] * yh[a:b]).sum(0), 1e-4)
        assert _close(bs[2 * C:3 * C], g.mean(0), 1e-5) and _close(bs[3 * C:], (g * yh).mean(0), 1e-4)


@pytest.mark.parametrize('k', [1, 2, 3])
def test_backward_records_pair(k):
    """out = relu(bnA(yA) + bnB(yB)) with yB a column slice of a wider map, as the chain's residual output; bf16 gradient copies."""
    B, level, C = 6, 3, 128
    P = _P(level)
    yA = torch.randn(B * P, C, device='cuda', generator=_gen(30)).half()
    ycat = torch.randn(B * P, 2 * C, device='cuda', generator=_gen(31)).half()
    sA, sB = _stat_of(yA.float(), C), _stat_of(ycat[:, C:].float().contiguous(), C)
    dout = torch.randn(B * P, C, device='cuda', generator=_gen(32))
    ranges = _ranges(B, P, k)
    masks = []
    for a, b, _, n in ranges:
        mw = torch.empty(n * P + 2 * n, C, dtype=torch.bfloat16, device='cuda')
        _lib.check(L.gin_bn_act_fwd(_ptr(yA, a * C), C, sA.data_ptr(), _ptr(ycat, a * 2 * C + C), 2 * C, sB.data_ptr(), 1, 1, None, None,
                                    mw.data_ptr(), n, level, C, _s()), 'gin_bn_act_fwd')
        masks.append(mw)
    ws = torch.empty(L.gin_bn_pair_ws_bytes(C), dtype=torch.uint8, device='cuda')
    recs = torch.empty(k, L.gin_bn_sync_record_bytes(C, 1) // 8, dtype=torch.float64, device='cuda')
    for r, (a, b, _, n) in enumerate(ranges):
        _lib.check(L.gin_bn_sync_bwd_reduce_pair(_ptr(dout, a * C), C, masks[r].data_ptr(), _ptr(yA, a * C), C, sA.data_ptr(), _ptr(ycat, a * 2 * C + C),
                                                 2 * C, sB.data_ptr(), 1, _ptr(recs[r]), ws.data_ptr(), n, level, C, 1, _s()), 'reduce_pair')
    outs = []
    for r, (a, b, _, n) in enumerate(ranges):
        bA, bB = torch.empty(4 * C, device='cuda'), torch.empty(4 * C, device='cuda')
        dA = torch.empty(n * P + 2 * n, C, dtype=torch.bfloat16, device='cuda')
        dcat = torch.empty(n * P + 2 * n, 2 * C, dtype=torch.bfloat16, device='cuda')
        _lib.check(L.gin_bn_sync_bwd_final(recs.data_ptr(), k, r, C, bA.data_ptr(), bB.data_ptr(), _s()), 'bwd_final')
        _lib.check(L.gin_bn_bwd_apply_pair(_ptr(dout, a * C), C, masks[r].data_ptr(), _ptr(yA, a * C), C, sA.data_ptr(), bA.data_ptr(), dA.data_ptr(), C,
                                           _ptr(ycat, a * 2 * C + C), 2 * C, sB.data_ptr(), bB.data_ptr(), _ptr(dcat, C), 2 * C, 1, n, level, C, 1, _s()),
                   'apply_pair')
        outs.append((bA, bB, dA, dcat[:, C:]))
    if k == 1:                                                   # bit for bit gin_bn_act_bwd_pair
        bA, bB = torch.empty(4 * C, device='cuda'), torch.empty(4 * C, device='cuda')
        dA = torch.empty(B * P + 2 * B, C, dtype=torch.bfloat16, device='cuda')
        dcat = torch.empty(B * P + 2 * B, 2 * C, dtype=torch.bfloat16, device='cuda')
        _lib.check(L.gin_bn_act_bwd_pair(dout.data_ptr(), C, masks[0].data_ptr(), yA.data_ptr(), C, sA.data_ptr(), bA.data_ptr(), dA.data_ptr(), C,
                                         _ptr(ycat, C), 2 * C, sB.data_ptr(), bB.data_ptr(), _ptr(dcat, C), 2 * C, 1, ws.data_ptr(), B, level, C, 1, _s()),
                   'gin_bn_act_bwd_pair')
        for u, v in zip(outs[0], (bA, bB, dA, dcat[:, C:])):
            assert torch.equal(u, v)
    keep = torch.cat([(m[:n * P].float() > 0).double() for m, (_, _, _, n) in zip(masks, ranges)], 0)
    refA, g, _ = _dy_ref(dout, keep, yA.double(), sA, C)
    refB, _, _ = _dy_ref(dout, keep, ycat[:, C:].double(), sB, C)
    gotA = torch.cat([o[2][:n * P].float() for o, (_, _, _, n) in zip(outs, ranges)], 0)
    gotB = torch.cat([o[3][:n * P].float() for o, (_, _, _, n) in zip(outs, ranges)], 0)
    assert _close(gotA, refA, 1e-2) and _close(gotB, refB, 1e-2)               # bf16 copies
    for o, (a, b, _, _) in zip(outs, ranges):
        assert _close(o[0][:C], g[a:b].sum(0), 1e-5) and torch.equal(o[0][:C], o[1][:C])
        assert _close(o[0][2 * C:3 * C], g.mean(0), 1e-5)


# ---------------------------------------------------------------------------------------------------------- 2. converted model, no process group
def _pair_of_models(name, level, seed=0):
    torch.manual_seed(seed)
    plain = getattr(gm, name)(gm.default_params(name, level)).cuda()
    conv = torch.nn.SyncBatchNorm.convert_sync_batchnorm(copy.deepcopy(plain))
    assert any(isinstance(m, torch.nn.SyncBatchNorm) for m in conv.modules())
    assert list(conv.state_dict()) == list(plain.state_dict())               # conversion keeps every key
    return plain, conv


def test_converted_model_routes_like_the_plain_one():
    plain, conv = _pair_of_models('ico2ico', 3)
    for m in (plain, conv):
        whole = list(m.encoder) + list(m.decoder)
        assert fused.chain_supported(whole) and fused.sync_group(whole) is None
    mixed = copy.deepcopy(conv)
    mixed.decoder[0].icobn01 = torch.nn.BatchNorm2d(mixed.decoder[0].icobn01.num_features).cuda()
    assert not fused.chain_supported(list(mixed.encoder) + list(mixed.decoder))   # BatchNorm2d and SyncBatchNorm in one chain
    assert fused.chain_supported(list(mixed.encoder))


def test_graphed_training_step_is_bit_identical_to_the_plain_model():
    level, B = 5, 8
    plain, conv = _pair_of_models('ico2ico', level)
    x, t = data.synthetic_batch(level, 0, B)
    x, t = x.cuda(), t.cuda()
    crit = losses.P2P_Loss(level, 1., 0., 0.)
    res = []
    for m in (plain, conv):
        m.train()

        def step(xb, tb, m=m):
            for p in m.parameters():
                p.grad = None
            out = m(xb)
            loss = crit(out, tb)
            loss.backward()
            return loss, out
        g = GraphedStep(step, (x, t))
        for _ in range(2):
            loss, out = g()
        torch.cuda.synchronize()
        res.append([loss.clone(), out.clone()] + [p.grad.clone() for p in m.parameters()] + [b.clone() for b in m.buffers()])
    assert len(res[0]) == len(res[1])
    for a, b in zip(*res):
        assert torch.equal(a, b)


def test_eval_chains_are_taken_and_bit_identical(monkeypatch):
    level, B = 5, 4
    plain, conv = _pair_of_models('ico2ico', level)
    x, _ = data.synthetic_batch(level, 0, B)
    x = x.cuda()
    old = (gm._FUSED, gm._HEAD, gm._INFER, gm._FROZEN)
    calls = []
    real = torch.nn.SyncBatchNorm.forward

    def counting(self, inp):
        calls.append(1)
        return real(self, inp)
    monkeypatch.setattr(torch.nn.SyncBatchNorm, 'forward', counting)
    try:
        gm.set_fused(True, inference=True, frozen=True)
        outs = []
        for m in (plain, conv):
            m.eval()
            with torch.no_grad():
                y_inf = m(x)
            xg = x.clone().requires_grad_(True)
            y_fr = m(xg)
            y_fr.square().sum().backward()
            outs.append((y_inf, y_fr.detach(), xg.grad))
    finally:
        gm.set_fused(*old[:1], head=old[1], inference=old[2], frozen=old[3])
    assert not calls, 'a SyncBatchNorm ran on the module path'
    for a, b in zip(*outs):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------- 3. two or more GPUs
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _torchrun(world, *args):
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world), '--master-addr', '127.0.0.1',
           '--master-port', str(_free_port()), os.path.join(ROOT, 'tests', 'diag', 'syncbn_worker.py')] + [str(a) for a in args]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('{')][-1])


def _check_split(d):
    """Against the unsynchronised step on all meshes on one device.  The bars of the first line were set before measuring; the
    same comparison of that step with itself on the reversed batch (d['noise'], measured in the same run: only the grouping of the
    fp32 per-CTA partial sums changes, the only expected difference here too) already exceeds them for the output, the running
    statistics and single small gradients (output 1.8e-3, running statistics 1.2e-5, one gradient ~1 at I5, 36 meshes on one
    B200).  So each figure must meet its bar or stay within twice that floor."""
    assert d['exchanges_per_step'] == [13, 13], d
    n = d['noise']
    for k, bar in (('loss_rel', 1e-4), ('out_rel_l2', 1e-3), ('running_max_rel', 1e-5), ('grad_rel_l2', 1e-2), ('worst_grad_rel_l2', 1e-2)):
        assert d[k] <= max(bar, 2 * n[k]), (k, d)
    assert d['ranks_agree_on_running_stats'] and d['replays_bit_identical'], d


def _check_uneven(d):
    n = d['noise']
    assert d['running_max_rel'] <= max(1e-5, 2 * n['running_max_rel']) and d['out_rel_l2'] <= max(1e-3, 2 * n['out_rel_l2']), d
    assert d['module_loss_rel'] <= 2e-3 and d['module_running_max_rel'] <= 1e-3, d
    assert d['vae_finite'] and d['vae_ranks_agree'], d


def test_two_ranks_on_one_device_through_gloo():
    """The exchanges, the split and the uneven split with two ranks sharing device 0 (gloo, eager steps): runs on one GPU."""
    _check_split(_torchrun(2, 'split', 36, 'gloo'))
    _check_uneven(_torchrun(2, 'uneven', 12, 'gloo'))


@pytest.mark.parametrize('world', [2, 4])
def test_split_batch_matches_one_device(world):
    """W ranks x 36/W meshes, converted ico2ico, graphed step with GradBuckets, against the unsynchronised fused step on all 36 meshes
    on one device from the same weights.  The only expected difference is the grouping of fp32 per-CTA partials."""
    if torch.cuda.device_count() < world:
        pytest.skip('needs %d CUDA devices' % world)
    _check_split(_torchrun(world, 'split', 36))


def test_uneven_split_and_torch_semantics():
    """5 + 7 meshes reproduce the 12-mesh running statistics and outputs; the fused synchronised step agrees with torch's own
    SyncBatchNorm on the module path; ico2ico_vae runs with its latent heads on torch's SyncBatchNorm."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 CUDA devices')
    _check_uneven(_torchrun(2, 'uneven', 12))
