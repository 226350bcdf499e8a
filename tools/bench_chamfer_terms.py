"""Normal and Laplacian terms of the Chamfer loss (gin_chamfer_terms_fwd / _bwd) on the GPU: per call against the torch composition,
and whole graphed VAE training steps.

    python tools/bench_chamfer_terms.py [--out DIR] [--seconds S] [--rounds R]

Prints one JSON line per workload (and writes DIR/r06_chamfer_terms_kernels.json, DIR/r06_chamfer_terms_steps.json with --out):
  * kind 'call': (B, N, M) = (36, 10242, 10242) I5 training and (1, 10242, 100000) latent fitting to a dense scan, both directions
    and both terms against a [B, M, 9] target.  Forward and backward of the kernels, each captured as a CUDA graph and timed with
    CUDA events over windows of at least S seconds, R windows alternating with the composition a user would otherwise write:
    mesh_utils.compute_vertex_normals / compute_laplacian_batch, a gather at the Chamfer indices and autograd (its backward
    scatters with floating-point atomics).  The outputs of both are compared before timing.  Bytes moved count what the call must
    read and write once, from the shapes: v, the target rows, the indices and the one-ring table (and dv for the backward); they
    are set against the device-to-device copy rate measured in the same run.
  * kind 'step': the graphed ico2ico_vae I5 / B=36 training step (optim.Adam) with P2PKLD_Loss (0.6 / 0.2 / 0.2), ChamferKLD_Loss
    with the position terms only (0.6 / 0.6), and ChamferKLD_Loss with the normal and Laplacian terms (0.6 / 0.6 / 0.2 / 0.2).
Every line carries the GPU name, power limit and maximum SM clock, read in the same run.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from geniconet_b200 import _lib, data, losses, mesh_utils, models as gm  # noqa: E402
from geniconet_b200.graph import GraphedStep  # noqa: E402
from geniconet_b200.ico_conv import get_plan  # noqa: E402
from bench_chamfer import alternate, gpu_info, graphed, training_step  # noqa: E402

LEVEL = 5
SIZES = ((36, 10242, 10242), (1, 10242, 100000))


def copy_rate(seconds, rounds):
    """Device-to-device copy rate in bytes/s (read + write) of a 1 GiB buffer."""
    a = torch.empty(1 << 28, device='cuda')
    b = torch.empty_like(a)
    t = alternate({'copy': lambda: b.copy_(a)}, seconds, rounds)['copy']
    return 2 * a.numel() * 4 / t


def inputs(B, M):
    """Output vertices [B,V,3] (synthetic I5 meshes with noise) and a [B,M,9] target sampled from other meshes, with noise."""
    g = torch.Generator().manual_seed(B * 7 + M)
    _, t = data.synthetic_batch(LEVEL, 0, B)
    v = t[:, :3].transpose(1, 2) + 5e-3 * torch.randn(B, t.shape[2], 3, generator=g)
    _, u = data.synthetic_batch(LEVEL, 40, B)
    rows = u.transpose(1, 2)[:, torch.randint(0, u.shape[2], (M,), generator=g)].clone()
    rows[..., :3] += 2e-3 * torch.randn(B, M, 3, generator=g)
    return v.cuda().contiguous(), rows.cuda().contiguous()


def torch_terms(v, tn, tl, jxy, jyx):
    n, lap = mesh_utils.compute_vertex_normals(v), mesh_utils.compute_laplacian_batch(v)
    cos = torch.nn.functional.cosine_similarity
    return torch.stack([(1 - cos(n, tn.gather(1, jxy), dim=-1)).mean(), (1 - cos(tn, n.gather(1, jyx), dim=-1)).mean(),
                        (lap - tl.gather(1, jxy)).square().mean(), (tl - lap.gather(1, jyx)).square().mean()])


def bench_calls(seconds, rounds, info, hbm):
    L = _lib.lib
    st = lambda: torch.cuda.current_stream().cuda_stream
    plan = get_plan(_lib.PLAN_LOSS, LEVEL, 1, 'average', torch.device('cuda'))
    rows = []
    for B, N, M in SIZES:
        v, target = inputs(B, M)
        y, tn, tl = target[..., :3], target[..., 3:6], target[..., 6:9]
        _, i_xy, _, i_yx = losses.chamfer_distance(v, y)
        out = torch.empty(4, device='cuda')
        dout = torch.tensor([0.7, 1.3, 2.1, 0.4], device='cuda')
        dv = torch.empty_like(v)
        ws = torch.empty(L.gin_chamfer_terms_ws_bytes(B, LEVEL, M), dtype=torch.uint8, device='cuda')
        common = lambda: (plan.host_ptr, plan.dev_ptr, v.data_ptr(), tn.data_ptr(), *tn.stride(), tl.data_ptr(), *tl.stride(),
                          i_xy.data_ptr(), i_yx.data_ptr())

        def fwd():
            _lib.check(L.gin_chamfer_terms_fwd(*common(), out.data_ptr(), ws.data_ptr(), B, M, st()), 'gin_chamfer_terms_fwd')

        def bwd():
            _lib.check(L.gin_chamfer_terms_bwd(*common(), dout.data_ptr(), dv.data_ptr(), ws.data_ptr(), B, M, st()),
                       'gin_chamfer_terms_bwd')
        vg = v.clone().requires_grad_(True)
        jxy, jyx = i_xy.long()[..., None].expand(-1, -1, 3), i_yx.long()[..., None].expand(-1, -1, 3)

        def torch_fwd():
            with torch.no_grad():
                return torch_terms(v, tn, tl, jxy, jyx)

        def torch_bwd():                                       # forward and backward: autograd needs its own forward
            vg.grad = None
            (torch_terms(vg, tn, tl, jxy, jyx) * dout).sum().backward()
        fwd()
        bwd()
        torch_bwd()
        ref = torch_fwd()
        torch.cuda.synchronize()
        term_rel = ((out - ref).abs() / ref.abs()).max().item()
        grad_rel = ((dv - vg.grad).norm() / vg.grad.norm()).item()
        assert term_rel <= 1e-4 and grad_rel <= 1e-4, (term_rel, grad_rel)
        t = alternate({'fwd': graphed(fwd), 'bwd': graphed(bwd), 'torch_fwd': torch_fwd, 'torch_fwd_bwd': torch_bwd}, seconds, rounds)
        V = v.shape[1]
        read = B * V * 12 + B * M * 24 + B * (V + M) * 4 + V * 24
        moved = {'fwd': read, 'bwd': read + B * V * 12}
        res = dict(kind='call', B=B, N=N, M=M, rounds=rounds, **info, copy_gb_s=round(hbm / 1e9, 1))
        for k, s in t.items():
            res[k + '_ms'] = round(s * 1e3, 4)
        for k, b in moved.items():
            res[k + '_bytes'] = b
            res[k + '_gb_s'] = round(b / t[k] / 1e9, 1)
            res[k + '_share_of_copy_rate'] = round(b / t[k] / hbm, 3)
        res['fwd_speedup_vs_torch'] = round(t['torch_fwd'] / t['fwd'], 2)
        res['fwd_bwd_speedup_vs_torch'] = round(t['torch_fwd_bwd'] / (t['fwd'] + t['bwd']), 2)
        res['terms_max_rel_vs_torch'] = term_rel
        res['grad_rel_l2_vs_torch'] = grad_rel
        rows.append(res)
        print(json.dumps(res), flush=True)
        del v, target, ws, vg
        torch.cuda.empty_cache()
    return rows


def bench_steps(seconds, rounds, info):
    B = 36
    params = gm.default_params('ico2ico_vae', LEVEL)
    x, t = data.synthetic_batch(LEVEL, 0, B)
    x, t = x.cuda(), t.cuda()
    crits = {'p2pkld': losses.P2PKLD_Loss(LEVEL, 0.6, 0.2, 0.2, 1.0),
             'chamferkld_pos': losses.ChamferKLD_Loss(LEVEL, 0.6, 0.6, 1.0),
             'chamferkld_terms': losses.ChamferKLD_Loss(LEVEL, 0.6, 0.6, 1.0, factor_nor=0.2, factor_lap=0.2)}
    graphs = {}
    for label, crit in crits.items():
        torch.manual_seed(0)
        m = gm.ico2ico_vae(params).cuda().train()
        graphs[label] = GraphedStep(training_step(m, crit), (x, t))
    s = alternate({k: g.__call__ for k, g in graphs.items()}, seconds, rounds)
    res = dict(kind='step', model='ico2ico_vae', level=LEVEL, B=B, what='train', rounds=rounds, **info)
    for k, v in s.items():
        res[k + '_ms'] = round(v * 1e3, 4)
    res['terms_cost_ms'] = round((s['chamferkld_terms'] - s['chamferkld_pos']) * 1e3, 4)
    print(json.dumps(res), flush=True)
    return [res]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--seconds', type=float, default=1.0)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--only', choices=('call', 'step'), default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_chamfer_terms.py measures on a GPU; none found')
    torch.cuda.set_device(0)
    info = gpu_info()
    out = {}
    if a.only != 'step':
        out['kernels'] = bench_calls(a.seconds, a.rounds, info, copy_rate(a.seconds, a.rounds))
    if a.only != 'call':
        out['steps'] = bench_steps(a.seconds, a.rounds, info)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        for k, rows in out.items():
            with open(os.path.join(a.out, 'r06_chamfer_terms_%s.json' % k), 'w') as f:
                json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()
