"""Synchronised BatchNorm: the ico2ico I5 graphed training step at a global batch of 36 meshes, split over W GPUs.

    python tools/bench_syncbn.py [--out DIR] [--rounds R] [--steps K] [--gpus N]

starts itself under torch.distributed.run on N = min(6, device count) GPUs (--gpus overrides) and times, on one node:
  * 'single'      1 GPU, B = 36, BatchNorm2d (no exchange at all);
  * 'sync_shared' W GPUs x 36/W meshes, SyncBatchNorm on the gradient all-reduce's group (W = 2, 4 and, with >= 6 devices, 6);
  * 'sync_split'  the same with the BatchNorm exchanges on a group of their own (a second communicator);
  * 'unsync'      W GPUs x 36/W meshes, BatchNorm2d: the same per-rank work without the exchanges;
  * 'exchanges'   the 26 all-gathers of one step alone (13 forward records, 13 backward, the step's record sizes), captured as a graph.
Every step is forward + P2P_Loss + backward + dp.GradBuckets + optim.Adam, captured by graph.GraphedStep.  Each configuration is timed
with CUDA events over K replays in R windows, the configurations alternating window by window; the median window is reported, in ms
per step and meshes per second (36 / step time), from rank 0 (every rank waits for the others inside the step).  One JSON document,
with the GPU name, power limit and maximum SM clock read in the same run, is printed and written to DIR/r07_syncbn_steps.json.
"""
import argparse
import json
import os
import socket
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GLOBAL_B, LEVEL = 36, 5


def _launch(args):
    import torch
    n = args.gpus or min(6, torch.cuda.device_count())
    if n < 1:
        raise SystemExit('bench_syncbn: no CUDA device')
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n), '--master-addr', '127.0.0.1', '--master-port',
           str(port), os.path.abspath(__file__)] + sys.argv[1:]
    raise SystemExit(subprocess.run(cmd).returncode)


def gpu_info():
    q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader,nounits'], capture_output=True,
                       text=True, timeout=30).stdout.strip().split(', ')
    return {'gpu': q[0], 'power_limit_w': float(q[1]), 'max_sm_clock_mhz': float(q[2])} if len(q) == 3 else {'gpu': q}


def main(args):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from geniconet_b200 import data, fused, losses, models as gm
    from geniconet_b200.dp import GradBuckets
    from geniconet_b200.graph import GraphedStep
    from geniconet_b200.optim import Adam

    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    Ws = [w for w in (2, 4, 6) if w <= world]
    groups = {w: (dist.new_group(list(range(w))), dist.new_group(list(range(w)))) for w in Ws}    # (gradients, BatchNorm) of ranks 0..W-1
    crit = losses.P2P_Loss(LEVEL, 1., 0., 0.)
    X, T = data.synthetic_batch(LEVEL, 0, GLOBAL_B)
    cfgs = [('single', 1, None)] + [(k, w, None) for w in Ws for k in ('unsync', 'sync_shared', 'sync_split', 'exchanges')]
    steps = {}
    for name, w, _ in cfgs:
        if rank >= w:
            continue
        b = GLOBAL_B // w
        x, t = X[rank * b:(rank + 1) * b].cuda().contiguous(), T[rank * b:(rank + 1) * b].cuda().contiguous()
        if name == 'exchanges':
            # the records of one ico2ico step: stem + 2 per block forward, 2 per block + stem backward (a pair record is 2 x (2C + 1))
            widths = [64] + [c for c in (128, 256, 256, 256, 128, 64) for _ in range(2)]
            pair = [False] + [q % 2 == 0 for q in range(12)]
            recs = [torch.zeros((2 if p else 1) * (2 * c + 1), dtype=torch.float64, device='cuda') for c, p in zip(widths, pair)]
            sync = (groups[w][1], w, rank)

            def step(xb, tb, recs=recs, sync=sync):
                outs = [fused._exchange(r, sync) for r in recs + recs[::-1]]
                return outs[-1]
        else:
            torch.manual_seed(0)
            model = gm.ico2ico(gm.default_params('ico2ico', LEVEL)).cuda().train()
            if name.startswith('sync'):
                model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model, process_group=groups[w][1] if name == 'sync_split' else groups[w][0])
            buckets = GradBuckets(model.parameters(), w, process_group=groups[w][0] if w > 1 else None, adjacent=fused.weight_pairs(model))
            opt = Adam(model.parameters(), lr=1e-4)

            def step(xb, tb, model=model, buckets=buckets, opt=opt):
                buckets.reset()
                ls = crit(model(xb), tb)
                ls.backward()
                buckets.finish()
                opt.step()
                return ls
        steps[name, w] = GraphedStep(step, (x, t))
    torch.cuda.synchronize()
    dist.barrier()
    times = {k: [] for k in steps}
    for _ in range(args.rounds):
        for name, w, _ in cfgs:
            if (name, w) in steps:
                g = steps[name, w]
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.steps):
                    g()
                b.record()
                b.synchronize()
                times[name, w].append(a.elapsed_time(b) / args.steps)
            torch.cuda.synchronize()
            dist.barrier()
    if rank == 0:
        rows = []
        for name, w, _ in cfgs:
            ms = statistics.median(times[name, w])
            row = {'config': name, 'gpus': w, 'meshes_per_gpu': GLOBAL_B // w, 'step_ms': round(ms, 4),
                   'windows_ms': [round(v, 4) for v in times[name, w]]}
            if name != 'exchanges':
                row['meshes_per_s'] = round(GLOBAL_B / ms * 1e3, 1)
            rows.append(row)
        doc = dict(gpu_info(), workload='ico2ico I5 graphed training step (forward, P2P_Loss, backward, GradBuckets, Adam), 36 meshes per step',
                   rounds=args.rounds, steps_per_window=args.steps, devices=world, results=rows)
        print(json.dumps(doc), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, 'r07_syncbn_steps.json'), 'w') as f:
                json.dump(doc, f, indent=1)
    torch.cuda.synchronize()
    dist.barrier()
    sys.stdout.flush()
    os._exit(0)          # destroying communicators whose collectives live in captured graphs hung at exit (tests/diag/dp_parity_worker.py)


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--rounds', type=int, default=9)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--gpus', type=int, default=0)
    a = ap.parse_args()
    if 'RANK' in os.environ:
        main(a)
    else:
        _launch(a)
