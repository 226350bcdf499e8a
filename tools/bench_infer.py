"""Forward-only inference throughput: the fused eval chain (fused.infer_chain) against the module path.

    python tools/bench_infer.py [--out DIR] [--seconds S]

Prints one JSON line per configuration (and writes them to DIR/bench_infer.jsonl when --out is given):
  * kind 'model': graphed eval forward, meshes/s, fused (set_fused(True, inference=True)) and module path (set_fused(False)),
    for ico2ico I5 / B=36 and I6 / B=16, ico2ico_vae encode (x -> mu, logvar) and decode (z -> mesh) at I5 / B=36;
  * kind 'conv': per forward conv problem of ico2ico I5 / B=36, one affine-epilogue launch (gin_hexconv_fwd_affine) against
    stats2 (fp16 y) + gin_bn_act_fwd, each replayed as a CUDA graph over rotating buffer sets larger than twice the 126 MB L2.
Times are CUDA events over windows of at least --seconds (default 1) of back-to-back replays.  Every line carries the GPU name and
its power limit, read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from geniconet_b200 import _lib, data, fused, models as gm  # noqa: E402
from geniconet_b200.graph import GraphedStep  # noqa: E402
from geniconet_b200.ico_conv import get_plan  # noqa: E402

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
    n, total = 1, 0.0
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


def eval_model(name, level):
    params = gm.default_params(name, level)
    torch.manual_seed(0)
    m = getattr(gm, name)(params).cuda().train()
    with torch.no_grad():                                 # non-trivial running statistics
        for k in range(2):
            x, _ = data.synthetic_batch(level, 4 * k, 4)
            m(x.cuda()) if name == 'ico2ico' else m.encode(x.cuda())
    return m.eval()


def bench_models(seconds, info):
    rows = []
    cases = [('ico2ico', 5, 36, 'forward'), ('ico2ico', 6, 16, 'forward'), ('ico2ico_vae', 5, 36, 'encode'), ('ico2ico_vae', 5, 36, 'decode')]
    for name, level, B, what in cases:
        m = eval_model(name, level)
        x, _ = data.synthetic_batch(level, 0, B)
        x = x.cuda()
        if what == 'decode':
            with torch.no_grad():
                mu, _ = m.encode(x)
            x = mu.contiguous()
        fn = {'forward': lambda t: m(t), 'encode': lambda t: m.encode(t), 'decode': lambda t: m.decode(t)}[what]

        def step(t):
            with torch.no_grad():
                return fn(t)
        res = dict(kind='model', model=name, level=level, B=B, what=what, **info)
        for label, on in (('fused', True), ('module', False)):
            gm.set_fused(on, inference=on)
            g = GraphedStep(step, (x,))
            s = timed(g, seconds)
            res[label + '_ms'] = round(s * 1e3, 4)
            res[label + '_meshes_per_s'] = round(B / s, 1)
            del g
        gm.set_fused(True, inference=False)
        res['speedup'] = round(res['module_ms'] / res['fused_ms'], 3)
        rows.append(res)
        print(json.dumps(res), flush=True)
    return rows


def conv_problems(level=5):
    """(name, level_in, stride, Cin, Cout, split, relu_split, residual) of every forward conv of ico2ico at `level`."""
    out = []
    enc, dec = gm._ENC_WIDTHS['ae'], gm._DEC_WIDTHS['ae']
    for d in range(len(enc) - 1):
        out.append(('enc%d.conv00|conv10' % d, level - d, 2, enc[d], 2 * enc[d + 1], enc[d + 1], enc[d + 1], False))
        out.append(('enc%d.conv01' % d, level - d - 1, 1, enc[d + 1], enc[d + 1], enc[d + 1], 0, True))
    for d in range(3):
        lvl = level - 2 + d
        out.append(('dec%d.conv00|conv10' % d, lvl, 1, dec[d], 2 * dec[d + 1], dec[d + 1], dec[d + 1], False))
        out.append(('dec%d.conv01' % d, lvl, 1, dec[d + 1], dec[d + 1], dec[d + 1], 0, True))
    return out


def bench_convs(seconds, info, B=36):
    L = _lib.lib
    rows = []
    dev = torch.device('cuda')
    st = lambda: torch.cuda.current_stream().cuda_stream
    for name, lvl_in, stride, cin, cout, split, relu_split, residual in conv_problems():
        lvl = lvl_in - 1 if stride == 2 else lvl_in
        plan = get_plan(_lib.PLAN_HEXCONV, lvl_in, stride, 'average', dev)
        P_in, P = 10 * 4 ** lvl_in, 10 * 4 ** lvl
        w0 = torch.randn(cout, cin, 7, device=dev) * (1.5 / (7 * cin)) ** 0.5
        packed = fused._pack_many([(w0, None, cin)])[0]
        bias = 0.05 * torch.randn(cout, device=dev)
        scale, shift = 1 + 0.1 * torch.randn(cout, device=dev), 0.1 * torch.randn(cout, device=dev)
        stat = torch.stack([torch.zeros(cout, device=dev), torch.ones(cout, device=dev), scale, shift]).contiguous()
        per_set = (B * P_in + 2 * B) * cin * 2 + B * P * cout * (2 + 2 + 4 + (4 if residual else 0))
        nsets = max(2, int(2 * L2_BYTES // per_set) + 1)
        sets = []
        for _ in range(nsets):
            s = dict(xb=(torch.randn((B * P_in + 2 * B) * cin, device=dev) * 0.5).to(torch.bfloat16))
            s['res'] = torch.randn(B * P, cout, device=dev) if residual else None
            s['y'] = torch.empty(B * P, cout, dtype=torch.float16, device=dev)
            s['parts'] = torch.empty(L.gin_hexconv_stats_ws_bytes(cout) // 4, device=dev)
            w = [split, cout - split]
            s['o0b'] = torch.empty((B * P + 2 * B, w[0]), dtype=torch.bfloat16, device=dev)
            s['o0f'] = torch.empty((B * P, w[0]), device=dev) if residual else None
            s['o1f'] = torch.empty((B * P, w[1]), device=dev) if w[1] else None
            s['ring'] = torch.empty(L.gin_hexconv_affine_ring_bytes(B, cout) // 4, device=dev)
            sets.append(s)
        nparts = ctypes.c_int(0)
        ptr = lambda t: t.data_ptr() if t is not None else None

        def affine():
            for s in sets:
                # the launch the chain makes: operand copy of the first destination, fp32 skip map / block output
                _lib.check(L.gin_hexconv_fwd_affine(plan.host_ptr, plan.dev_ptr, s['xb'].data_ptr(), packed.data_ptr(), scale.data_ptr(),
                                                    shift.data_ptr(), relu_split, ptr(s['res']), cout if residual else 0, 0, split,
                                                    s['o0b'].data_ptr(), ptr(s['o0f']), None, ptr(s['o1f']), s['ring'].data_ptr(), B, cin,
                                                    cout, st()), 'affine')

        def composed():
            for s in sets:
                _lib.check(L.gin_hexconv_fwd_bf16_stats2(plan.host_ptr, plan.dev_ptr, s['xb'].data_ptr(), packed.data_ptr(), bias.data_ptr(),
                                                         None, 0, s['y'].data_ptr(), 1, B, cin, cout, s['parts'].data_ptr(),
                                                         ctypes.addressof(nparts), st()), 'stats2')
                # bn_act of the first destination (the second one of a sibling GEMM is folded into the next bn_act there)
                _lib.check(L.gin_bn_act_fwd(s['y'].data_ptr(), cout, stat.data_ptr(), ptr(s['y']) if residual else None, cout,
                                            stat.data_ptr() if residual else None, 1, 1, s['o0b'].data_ptr(), ptr(s['o0f']), None, B, lvl,
                                            split, st()), 'bn_act_fwd')
        res = dict(kind='conv', problem=name, level_in=lvl_in, stride=stride, cin=cin, cout=cout, B=B, sets=nsets, **info)
        for label, fn in (('affine', affine), ('stats2_bn_act', composed)):
            g = torch.cuda.CUDAGraph()
            fn()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                fn()
            res[label + '_us'] = round(timed(g.replay, seconds) / nsets * 1e6, 2)
        res['ratio'] = round(res['stats2_bn_act_us'] / res['affine_us'], 3)
        rows.append(res)
        print(json.dumps(res), flush=True)
        del sets
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--seconds', type=float, default=1.0)
    ap.add_argument('--only', choices=('model', 'conv'), default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_infer.py measures on a GPU; none found')
    torch.cuda.set_device(0)
    info = gpu_info()
    rows = []
    if a.only != 'conv':
        rows += bench_models(a.seconds, info)
    if a.only != 'model':
        rows += bench_convs(a.seconds, info)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'bench_infer.jsonl'), 'w') as f:
            f.writelines(json.dumps(r) + '\n' for r in rows)


if __name__ == '__main__':
    main()
