"""Chamfer distance (gin_chamfer_fwd / _bwd) on the GPU: per call against the chunked torch.cdist composition, and whole graphed steps.

    python tools/bench_chamfer.py [--out DIR] [--seconds S] [--rounds R]

Prints one JSON line per workload (and writes DIR/r05_chamfer_kernels.json, DIR/r05_chamfer_steps.json when --out is given):
  * kind 'call': (B, N, M) in (36, 10242, 10242) I5 training, (16, 40962, 40962) I6, (1, 10242, 100000) latent fitting to a dense
    scan, (36, 10242, 2562).  Forward (both directions) and backward (both cotangents, dx and dy) of the kernels, each captured as
    a CUDA graph and timed with CUDA events over windows of at least S seconds, R windows alternating with the composition a user
    would otherwise write: torch.cdist in fp32 over row chunks with the row minimum and a running column minimum (forward), and
    autograd through the gathered pair distances (backward).  The outputs of both are compared before timing.  Pair evaluations
    per second count 2*B*N*M pairs per forward; instructions per pair come from the kernel's SASS (the unrolled hot loop).
  * kind 'step': the ico2ico I5 / B=36 graphed training step (optim.Adam) with P2P_Loss against Chamfer_Loss on the data-path
    target, and one latent-fitting step (enc2ico_vae decoder frozen on the fused frozen-BatchNorm chain, B=1, z trainable, a
    one-sided Chamfer_Loss to a 100000-point scan).
Every line carries the GPU name, power limit and maximum SM clock, read in the same run.  The inputs are points near a unit sphere
(the scale of the icosahedral meshes); every working set here but the I6 one fits in the 126 MB L2, as it does in training.
"""
import argparse
import json
import os
import re
import shutil
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from geniconet_b200 import _lib, data, losses, models as gm  # noqa: E402
from geniconet_b200.graph import GraphedStep  # noqa: E402
from geniconet_b200.optim import Adam  # noqa: E402

SIZES = ((36, 10242, 10242), (16, 40962, 40962), (1, 10242, 100000), (36, 10242, 2562))


def gpu_info():
    out = {'gpu': torch.cuda.get_device_name(0), 'power_limit_w': None, 'max_sm_clock_mhz': None}
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader,nounits'],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        out['power_limit_w'], out['max_sm_clock_mhz'] = float(q[0]), float(q[1])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        pass
    return out


def timed(fn, seconds):
    """seconds per call of fn, from CUDA events over a window of at least `seconds` (after warm-up)."""
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
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            out[k].append(timed(fn, seconds))
    return {k: statistics.median(v) for k, v in out.items()}


def graphed(fn):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


def sphere_points(B, n, seed):
    g = torch.Generator().manual_seed(seed)
    p = torch.randn(B, n, 3, generator=g)
    return (p / p.norm(dim=-1, keepdim=True) * (1 + 0.05 * torch.rand(B, n, 1, generator=g))).cuda()


def instructions_per_pair():
    """Instructions of the nearest-neighbour hot loop per (query, candidate) pair, from the shipped SASS: of the loops (a backward
    branch and its target), the one densest in FFMA2, every 3 of which score 2 pairs."""
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        return None
    sass = subprocess.run([cuobjdump, '-sass', '-fun', '_ZN3gin7chamfer9nn_kernelENS0_3PtsES1_iiiPy', _lib.LIB_PATH], capture_output=True,
                          text=True).stdout
    ins = re.findall(r'/\*([0-9a-f]{4,})\*/\s+([^;]*);', sass)
    best = None
    for addr, text in ins:
        m = re.search(r'BRA(?:\.U)?\s+(?:!?U?P\d+,\s*)?0x([0-9a-f]+)', text)
        if m and int(m.group(1), 16) < int(addr, 16):
            body = [t for a, t in ins if int(m.group(1), 16) <= int(a, 16) <= int(addr, 16)]
            n2 = sum(1 for t in body if t.strip().startswith('FFMA2'))
            if n2 and (best is None or n2 / len(body) > best[1] / best[0]):
                best = (len(body), n2)
    if best is None:
        return None
    pairs = best[1] / 3 * 2
    return round(best[0] / pairs, 3)


def cdist_forward(x, y, budget=1 << 30):
    """The torch composition: squared fp32 cdist over row chunks, row minimum, running column minimum."""
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    rows = max(1, min(N, budget // (4 * M * B)))
    d_xy = torch.empty(B, N, device=x.device)
    i_xy = torch.empty(B, N, dtype=torch.long, device=x.device)
    d_yx = torch.full((B, M), float('inf'), device=x.device)
    i_yx = torch.zeros(B, M, dtype=torch.long, device=x.device)
    for s in range(0, N, rows):
        d = torch.cdist(x[:, s:s + rows], y).square_()
        d_xy[:, s:s + rows], i_xy[:, s:s + rows] = d.min(2)
        v, i = d.min(1)
        better = v < d_yx
        d_yx = torch.where(better, v, d_yx)
        i_yx = torch.where(better, i + s, i_yx)
    return d_xy, i_xy, d_yx, i_yx


def bench_calls(seconds, rounds, info, ipp):
    L = _lib.lib
    rows = []
    st = lambda: torch.cuda.current_stream().cuda_stream
    for B, N, M in SIZES:
        x, y = sphere_points(B, N, 1), sphere_points(B, M, 2)
        d_xy, d_yx = torch.empty(B, N, device='cuda'), torch.empty(B, M, device='cuda')
        i_xy, i_yx = torch.empty(B, N, dtype=torch.int32, device='cuda'), torch.empty(B, M, dtype=torch.int32, device='cuda')
        g_xy, g_yx = torch.rand(B, N, device='cuda'), torch.rand(B, M, device='cuda')
        dx, dy = torch.empty(B, N, 3, device='cuda'), torch.empty(B, M, 3, device='cuda')
        ws = torch.empty(L.gin_chamfer_ws_bytes(B, N, M), dtype=torch.uint8, device='cuda')

        def fwd():
            _lib.check(L.gin_chamfer_fwd(x.data_ptr(), *x.stride(), y.data_ptr(), *y.stride(), d_xy.data_ptr(), i_xy.data_ptr(), d_yx.data_ptr(),
                                         i_yx.data_ptr(), ws.data_ptr(), B, N, M, st()), 'gin_chamfer_fwd')

        def bwd():
            _lib.check(L.gin_chamfer_bwd(x.data_ptr(), *x.stride(), y.data_ptr(), *y.stride(), i_xy.data_ptr(), g_xy.data_ptr(), i_yx.data_ptr(),
                                         g_yx.data_ptr(), dx.data_ptr(), dy.data_ptr(), ws.data_ptr(), B, N, M, st()), 'gin_chamfer_bwd')
        fwd()
        c_xy, ci_xy, c_yx, ci_yx = cdist_forward(x, y)
        torch.cuda.synchronize()
        # same neighbours except near-ties, where the cdist composition (expanded form in a matrix product) may pick a farther point
        agree = [(i_xy.long() == ci_xy).float().mean().item(), (i_yx.long() == ci_yx).float().mean().item()]
        worse = max((d_xy - c_xy.clamp_min(0)).max().item(), (d_yx - c_yx.clamp_min(0)).max().item())
        assert min(agree) > 0.99 and worse <= 1e-5, (agree, worse)
        xg, yg = x.clone().requires_grad_(True), y.clone().requires_grad_(True)

        jxy, jyx = i_xy.long()[..., None].expand(-1, -1, 3), i_yx.long()[..., None].expand(-1, -1, 3)

        def torch_bwd():                                      # autograd through the gathered pairs, same neighbours as the kernel
            xg.grad = yg.grad = None
            pxy = (xg - yg.gather(1, jxy)).square().sum(-1)
            pyx = (yg - xg.gather(1, jyx)).square().sum(-1)
            ((pxy * g_xy).sum() + (pyx * g_yx).sum()).backward()
        bwd()
        torch_bwd()
        torch.cuda.synchronize()
        rel = max(((dx - xg.grad).norm() / xg.grad.norm()).item(), ((dy - yg.grad).norm() / yg.grad.norm()).item())
        t = alternate({'fwd': graphed(fwd), 'bwd': graphed(bwd), 'cdist_fwd': lambda: cdist_forward(x, y), 'torch_bwd': torch_bwd},
                      seconds, rounds)
        pairs = 2.0 * B * N * M
        res = dict(kind='call', B=B, N=N, M=M, rounds=rounds, pairs=pairs, **info)
        for k, v in t.items():
            res[k + '_ms'] = round(v * 1e3, 4)
        res['fwd_gpairs_s'] = round(pairs / t['fwd'] / 1e9, 1)
        res['cdist_gpairs_s'] = round(pairs / t['cdist_fwd'] / 1e9, 1)
        res['fwd_speedup_vs_cdist'] = round(t['cdist_fwd'] / t['fwd'], 2)
        res['bwd_speedup_vs_torch'] = round(t['torch_bwd'] / t['bwd'], 2)
        res['instructions_per_pair_sass'] = ipp
        res['index_agreement_vs_cdist'] = [round(a, 6) for a in agree]
        res['bwd_rel_l2_vs_torch'] = rel
        rows.append(res)
        print(json.dumps(res), flush=True)
        del x, y, ws, c_xy, c_yx, xg, yg
        torch.cuda.empty_cache()
    return rows


def training_step(m, crit):
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


def bench_steps(seconds, rounds, info):
    rows = []
    level, B = 5, 36
    params = gm.default_params('ico2ico', level)
    x, t = data.synthetic_batch(level, 0, B)
    x, t = x.cuda(), t.cuda()
    graphs = {}
    for label, crit in (('p2p', losses.P2P_Loss(level, 1., 0., 0.)), ('chamfer', losses.Chamfer_Loss(level, 1., 1.))):
        torch.manual_seed(0)
        m = gm.ico2ico(params).cuda().train()
        graphs[label] = GraphedStep(training_step(m, crit), (x, t))
    s = alternate({k: g.__call__ for k, g in graphs.items()}, seconds, rounds)
    res = dict(kind='step', model='ico2ico', level=level, B=B, what='train', rounds=rounds, **info)
    for k, v in s.items():
        res[k + '_ms'] = round(v * 1e3, 4)
    res['chamfer_cost_ms'] = round((s['chamfer'] - s['p2p']) * 1e3, 4)
    rows.append(res)
    print(json.dumps(res), flush=True)
    del graphs
    torch.cuda.empty_cache()

    # latent fitting: frozen decoder, one z, one-sided Chamfer to a dense scan
    pv = gm.default_params('ico2ico_vae', level)
    torch.manual_seed(1)
    dec = gm.enc2ico_vae(pv).cuda().eval()
    for p in dec.parameters():
        p.requires_grad_(False)
    n = 2 ** (level - 3)
    z = torch.nn.Parameter(torch.randn(1, 512, 5 * n, 2 * n, generator=torch.Generator().manual_seed(0)).cuda())
    _, tv = data.synthetic_batch(level, 3, 1)
    verts = tv[:, :3].transpose(1, 2)
    g = torch.Generator().manual_seed(5)
    pick = torch.randint(0, verts.shape[1], (100000,), generator=g)
    scan = (verts[:, pick] + 2e-3 * torch.randn(1, 100000, 3, generator=g)).cuda().contiguous()
    crit = losses.Chamfer_Loss(level, 0.0, 1.0)
    opt = Adam([z], lr=1e-3)
    opt.prepare()
    saved = gm._FUSED, gm._HEAD, gm._INFER, gm._FROZEN
    gm.set_fused(True, frozen=True)

    def step(zz, sc):
        if z.grad is not None:
            z.grad.zero_()
        loss = crit(dec.decode(z), sc)
        loss.backward()
        opt.step()
        return loss
    try:
        gstep = GraphedStep(step, (z, scan))
    finally:
        gm._FUSED, gm._HEAD, gm._INFER, gm._FROZEN = saved
    s = alternate({'latent_fit': gstep.__call__}, seconds, rounds)
    res = dict(kind='step', model='enc2ico_vae', level=level, B=1, M=100000, what='latent_fit_one_sided', rounds=rounds,
               latent_fit_ms=round(s['latent_fit'] * 1e3, 4), **info)
    rows.append(res)
    print(json.dumps(res), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--seconds', type=float, default=1.0)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--only', choices=('call', 'step'), default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_chamfer.py measures on a GPU; none found')
    torch.cuda.set_device(0)
    info = gpu_info()
    ipp = instructions_per_pair()
    out = {}
    if a.only != 'step':
        out['kernels'] = bench_calls(a.seconds, a.rounds, info, ipp)
    if a.only != 'call':
        out['steps'] = bench_steps(a.seconds, a.rounds, info)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        for k, rows in out.items():
            with open(os.path.join(a.out, 'r05_chamfer_%s.json' % k), 'w') as f:
                json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()
