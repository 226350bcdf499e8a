"""Eval-mode BatchNorm with grad enabled: the frozen chain (fused.run_frozen_chain) against the module path.

    python tools/bench_frozen.py [--out DIR] [--seconds S] [--rounds R]

Prints one JSON line per workload (and writes DIR/r04_frozen_models.json, DIR/r04_frozen_kernels.json when --out is given):
  * kind 'step': a whole graphed step, frozen chain (set_fused(True, frozen=True)) and module path (set_fused(False)), timed in
    R alternating windows each (median reported):
      - ico2ico I5 / B=36 and I6 / B=16 frozen-BatchNorm fine-tune step: eval(), every parameter trainable, P2P_Loss, optim.Adam;
      - ico2ico_vae I5 / B=36 latent fitting: decoder parameters frozen, z trainable, reconstruction loss, optim.Adam on z;
  * kind 'bn': per BatchNorm launch shape of the ico2ico I5 / B=36 chain, gin_bn_eval_bwd(_pair) (with and without the sums)
    against gin_bn_act_bwd(_pair) on the same shapes, each replayed as a CUDA graph over rotating buffer sets larger than twice
    the 126 MB L2, with GB/s from the bytes each variant has to move and the device-to-device copy rate measured in the same run.
Every line carries the GPU name and its power limit, read in the same run.
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from geniconet_b200 import _lib, data, fused, losses, models as gm  # noqa: E402
from geniconet_b200.graph import GraphedStep  # noqa: E402
from geniconet_b200.optim import Adam  # noqa: E402

L2_BYTES = 126 << 20


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit', '--format=csv,noheader,nounits'], capture_output=True,
                           text=True, timeout=30).stdout.strip()
        power = float(q) if q else None
    except (OSError, ValueError, subprocess.TimeoutExpired):
        power = None
    return {'gpu': name, 'power_limit_w': power}


def timed(fn, seconds):
    """seconds per call of fn (which enqueues work), from CUDA events over a window of at least `seconds`."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    n = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        total = a.elapsed_time(b) / 1e3
        if total >= seconds:
            return total / n
        n = max(2 * n, int(n * 1.2 * seconds / max(total, 1e-6)))


def alternate(fns, seconds, rounds):
    """{label: median seconds per call} over `rounds` windows per function, the functions taking turns."""
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            out[k].append(timed(fn, seconds))
    return {k: statistics.median(v) for k, v in out.items()}


def warmed(name, level):
    params = gm.default_params(name, level)
    torch.manual_seed(0)
    m = getattr(gm, name)(params).cuda().train()
    with torch.no_grad():                                 # non-trivial running statistics
        for k in range(2):
            x, _ = data.synthetic_batch(level, 4 * k, 4)
            m(x.cuda())
    return m.eval(), params


def fine_tune_step(m, params, level):
    crit = losses.P2P_Loss(level, params['ico']['factor_pos'], params['ico']['factor_nor'], params['ico']['factor_lap'])
    opt = Adam(m.parameters(), lr=1e-5)
    opt.prepare()

    def step(x, t):
        for p in m.parameters():
            if p.grad is not None:
                p.grad.zero_()
        loss = crit(m(x), t)
        loss.backward()
        opt.step()
        return loss
    return step


def latent_step(m, params, level, z):
    crit = losses.P2P_Loss(level, params['ico']['factor_pos'], params['ico']['factor_nor'], params['ico']['factor_lap'])
    for p in m.parameters():
        p.requires_grad_(False)
    opt = Adam([z], lr=1e-3)
    opt.prepare()

    def step(x, t):
        if z.grad is not None:
            z.grad.zero_()
        loss = crit(m.decode(z), t)
        loss.backward()
        opt.step()
        return loss
    return step


def bench_steps(seconds, rounds, info):
    rows = []
    for name, level, B, what in (('ico2ico', 5, 36, 'fine_tune'), ('ico2ico', 6, 16, 'fine_tune'), ('ico2ico_vae', 5, 36, 'latent_fit')):
        base, params = warmed(name, level)
        x, t = data.synthetic_batch(level, 0, B)
        x, t = x.cuda(), t.cuda()
        graphs = {}
        for label, on in (('frozen', True), ('module', False)):
            m = copy.deepcopy(base)
            gm.set_fused(on, frozen=on)
            if what == 'fine_tune':
                step = fine_tune_step(m, params, level)
            else:
                n = 2 ** (level - 3)
                z = torch.nn.Parameter(torch.randn(B, 512, 5 * n, 2 * n, generator=torch.Generator().manual_seed(0)).cuda())
                step = latent_step(m, params, level, z)
            graphs[label] = GraphedStep(step, (x, t))
        gm.set_fused(True, frozen=False)
        # the graphs hold their own kernels and arguments: the switch no longer matters once they are captured
        s = alternate({k: g.__call__ for k, g in graphs.items()}, seconds, rounds)
        res = dict(kind='step', model=name, level=level, B=B, what=what, rounds=rounds, **info)
        for k, v in s.items():
            res[k + '_ms'] = round(v * 1e3, 4)
        res['speedup'] = round(s['module'] / s['frozen'], 3)
        rows.append(res)
        print(json.dumps(res), flush=True)
        del graphs
        torch.cuda.empty_cache()
    return rows


def copy_rate(seconds):
    n = 1 << 28                                           # 1 GiB of fp32 each way
    a, b = torch.empty(n, device='cuda'), torch.empty(n, device='cuda')
    s = timed(lambda: b.copy_(a), seconds)
    return 2 * 4 * n / s / 1e9


def bn_shapes(level=5):
    """(name, level, C, pair) of every BatchNorm backward launch of the ico2ico chain at `level`."""
    out = [('stem.icobn', level, gm._ENC_WIDTHS['ae'][0], False)]
    enc, dec = gm._ENC_WIDTHS['ae'], gm._DEC_WIDTHS['ae']
    for d in range(len(enc) - 1):
        out += [('enc%d.icobn00' % d, level - d - 1, enc[d + 1], False), ('enc%d.icobn01+10' % d, level - d - 1, enc[d + 1], True)]
    for d in range(3):
        out += [('dec%d.icobn00' % d, level - 2 + d, dec[d + 1], False), ('dec%d.icobn01+10' % d, level - 2 + d, dec[d + 1], True)]
    return out


def bench_bn(seconds, info, B=36):
    L = _lib.lib
    dev = torch.device('cuda')
    st = lambda: torch.cuda.current_stream().cuda_stream
    gbs_copy = copy_rate(seconds)
    rows = []
    for name, lvl, C, pair in bn_shapes():
        rows_px = B * 10 * 4 ** lvl
        stem = name.startswith('stem')
        # bytes each variant must move per pixel row (fp16 y, fp32 dout, bf16 gradient copies; the stem writes fp32 dy)
        if pair:
            eval_b, train_b = C * (4 + 2 + 2 + 2 + 2), C * ((4 + 2 + 2) + (4 + 2 + 2 + 2 + 2))
        else:
            out_b = 4 if stem else 2
            eval_b, train_b = C * (4 + 2 + out_b), C * ((4 + 2) + (4 + 2 + out_b))
        per_set = rows_px * (eval_b + 16 * C)
        nsets = max(2, int(2 * L2_BYTES // per_set) + 1)
        stat = torch.stack([0.1 * torch.randn(C, device=dev), 1 + 0.1 * torch.rand(C, device=dev), 1 + 0.1 * torch.randn(C, device=dev),
                            0.1 * torch.randn(C, device=dev)]).contiguous()
        sets = []
        for _ in range(nsets):
            s = dict(d=torch.randn(rows_px, C, device=dev), ycat=torch.randn(rows_px, 2 * C, device=dev).half(),
                     y01=torch.randn(rows_px, C, device=dev).half(),
                     dycat=torch.empty(rows_px + 2 * B, 2 * C, dtype=torch.bfloat16, device=dev),
                     dy01=torch.empty(rows_px + 2 * B, C, dtype=torch.bfloat16, device=dev),
                     dyf=torch.empty(rows_px, C, device=dev) if stem else None, mask=torch.empty(rows_px + 2 * B, C, dtype=torch.bfloat16, device=dev))
            sets.append(s)
        bsA, bsB = torch.empty(4 * C, device=dev), torch.empty(4 * C, device=dev)
        ws = torch.empty(max(L.gin_bn_pair_ws_bytes(C), L.gin_bn_eval_bwd_ws_bytes(C)), dtype=torch.uint8, device=dev)
        ptr = lambda t, off=0: t.data_ptr() + off if t is not None else None

        def run(kind, sums=True):
            for s in sets:
                yB = s['ycat'].data_ptr() + 2 * C
                if pair and kind == 'eval':
                    _lib.check(L.gin_bn_eval_bwd_pair(s['d'].data_ptr(), C, None, s['y01'].data_ptr(), C, stat.data_ptr(), ptr(bsA) if sums else None,
                                                      s['dy01'].data_ptr(), C, yB, 2 * C, stat.data_ptr(), ptr(bsB) if sums else None,
                                                      s['dycat'].data_ptr() + 2 * C, 2 * C, 1, ws.data_ptr(), B, lvl, C, 1, st()), 'eval_pair')
                elif pair:
                    _lib.check(L.gin_bn_act_bwd_pair(s['d'].data_ptr(), C, s['mask'].data_ptr(), s['y01'].data_ptr(), C, stat.data_ptr(),
                                                     bsA.data_ptr(), s['dy01'].data_ptr(), C, yB, 2 * C, stat.data_ptr(), bsB.data_ptr(),
                                                     s['dycat'].data_ptr() + 2 * C, 2 * C, 1, ws.data_ptr(), B, lvl, C, 1, st()), 'train_pair')
                else:
                    y, ld = (s['y01'], C) if stem else (s['ycat'], 2 * C)
                    dyb, ldo = (None, 0) if stem else (s['dycat'].data_ptr(), 2 * C)
                    if kind == 'eval':
                        _lib.check(L.gin_bn_eval_bwd(s['d'].data_ptr(), C, None, y.data_ptr(), ld, 1, stat.data_ptr(), ptr(bsA) if sums else None,
                                                     dyb, ldo, ptr(s['dyf']), C, ws.data_ptr(), B, lvl, C, 1, st()), 'eval')
                    else:
                        _lib.check(L.gin_bn_act_bwd(s['d'].data_ptr(), C, s['mask'].data_ptr(), y.data_ptr(), ld, 1, stat.data_ptr(), bsA.data_ptr(),
                                                    dyb, ldo, ptr(s['dyf']), C, ws.data_ptr(), B, lvl, C, 1, st()), 'train')
        variants = {'eval_sums': lambda: run('eval', True), 'eval_nosums': lambda: run('eval', False), 'train': lambda: run('train')}
        res = dict(kind='bn', launch=name, level=lvl, C=C, B=B, pair=pair, sets=nsets, copy_gb_s=round(gbs_copy, 1), **info)
        for label, fn in variants.items():
            g = torch.cuda.CUDAGraph()
            fn()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                fn()
            us = timed(g.replay, seconds) / nsets * 1e6
            nbytes = rows_px * (train_b if label == 'train' else eval_b)
            res[label + '_us'] = round(us, 2)
            res[label + '_gb_s'] = round(nbytes / (us * 1e-6) / 1e9, 1)
            res[label + '_of_copy'] = round(res[label + '_gb_s'] / gbs_copy, 3)
            del g
        res['speedup_sums'] = round(res['train_us'] / res['eval_sums_us'], 3)
        rows.append(res)
        print(json.dumps(res), flush=True)
        del sets
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--seconds', type=float, default=1.0)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--only', choices=('step', 'bn'), default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_frozen.py measures on a GPU; none found')
    torch.cuda.set_device(0)
    info = gpu_info()
    out = {}
    if a.only != 'bn':
        out['models'] = bench_steps(a.seconds, a.rounds, info)
    if a.only != 'step':
        out['kernels'] = bench_bn(a.seconds, info)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        for k, rows in out.items():
            with open(os.path.join(a.out, 'r04_frozen_%s.json' % k), 'w') as f:
                json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()
