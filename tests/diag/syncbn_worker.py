"""Synchronised-BatchNorm worker, launched by tests/test_gpu_syncbn.py or by hand:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node W --master-addr 127.0.0.1 --master-port P tests/diag/syncbn_worker.py MODE N [BACKEND]

Every rank builds the same ico2ico I5 weights and the same N synthetic meshes, and runs the unsynchronised fused step on all N of them
as the reference.  Its own share of the meshes then goes through the SyncBatchNorm-converted model.

  split  N/W meshes per rank, BatchNorm on a group of its own, a graphed step with GradBuckets: loss, outputs, running statistics,
         gradients against the reference; the exchange count; ranks agree on the running statistics; two replays agree.
  uneven (W = 2) 5 + 7 meshes, BatchNorm on the default group: running statistics and outputs against the reference; the fused step
         against torch's SyncBatchNorm on the module path; an eager ico2ico_vae step.

BACKEND 'nccl' (default): one GPU per rank.  'gloo': every rank on device 0 and the step eager instead of graphed (gloo collectives
cannot be captured), so the exchanges are tested on a machine with one GPU.  Rank 0 prints one JSON line.  The worker ends with os._exit, as dp_parity_worker.py does.
"""
import copy
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from geniconet_b200 import models as gm, losses, data, fused, reparam        # noqa: E402
from geniconet_b200.dp import GradBuckets                                     # noqa: E402
from geniconet_b200.graph import GraphedStep                                  # noqa: E402

rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ.get('LOCAL_RANK', 0))
mode = sys.argv[1] if len(sys.argv) > 1 else 'split'
N = int(sys.argv[2]) if len(sys.argv) > 2 else 36
backend = sys.argv[3] if len(sys.argv) > 3 else 'nccl'
level = 5
if backend == 'nccl':
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
else:
    torch.cuda.set_device(0)
    dist.init_process_group(backend)
params = gm.default_params('ico2ico', level)
crit = losses.P2P_Loss(level, 1., 0., 0.)
counts = [N // world + (1 if r < N % world else 0) for r in range(world)] if mode == 'split' else [5, 7]
assert sum(counts) == N and len(counts) == world
first = sum(counts[:rank])
mine = slice(first, first + counts[rank])
xs, ts = zip(*(data.synthetic_mesh(level, i) for i in range(N)))
X, T = torch.stack(xs).cuda(), torch.stack(ts).cuda()
torch.manual_seed(0)
base = gm.ico2ico(params).cuda().train()


def buffers(m):
    return [b.detach().clone() for n, b in m.named_buffers() if 'running' in n]


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def max_rel(xs, ys):
    return max(((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30)).item() for a, b in zip(xs, ys))


# the reference: the unsynchronised fused step on all N meshes, one device
ref = copy.deepcopy(base)
out_ref = ref(X)
loss_ref = crit(out_ref, T)
loss_ref.backward()
torch.cuda.synchronize()
g_ref = [p.grad.detach().clone() for p in ref.parameters()]
run_ref = buffers(ref)
res = {'mode': mode, 'world': world, 'counts': counts, 'backend': backend}


def grad_figures(gs):
    """(rel L2 of all gradients together, worst rel L2 of one non-zero parameter gradient) against the reference"""
    flat = lambda g: torch.cat([v.flatten() for v in g])
    return rel_l2(flat(gs), flat(g_ref)), max(rel_l2(a, b) for a, b in zip(gs, g_ref) if b.abs().max() > 0)


# the noise floor of the comparison: the same unsynchronised step on the same N meshes in reverse order.  Only the grouping of the
# fp32 per-CTA partial sums changes, which is also the only expected difference of the synchronised split.
perm = torch.arange(N - 1, -1, -1, device='cuda')
rev = copy.deepcopy(base)
out_rev = rev(X[perm])
loss_rev = crit(out_rev, T[perm])
loss_rev.backward()
res['noise'] = {'loss_rel': abs(loss_rev.item() - loss_ref.item()) / abs(loss_ref.item()), 'out_rel_l2': rel_l2(out_rev[perm], out_ref),
                'running_max_rel': max_rel(buffers(rev), run_ref)}
res['noise']['grad_rel_l2'], res['noise']['worst_grad_rel_l2'] = grad_figures([p.grad for p in rev.parameters()])
del rev, out_rev, loss_rev

bn_group = dist.new_group(list(range(world))) if mode == 'split' else None
model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(copy.deepcopy(base), process_group=bn_group)
scratch = torch.nn.SyncBatchNorm.convert_sync_batchnorm(copy.deepcopy(base), process_group=bn_group)
x, t = X[mine].contiguous(), T[mine].contiguous()

# exchanges per step: forward, backward (eager, one step, on a scratch copy so `model` keeps the reference's running statistics)
calls, real_exchange = [], fused._exchange


def counting(rec, sync):
    calls.append(1)
    return real_exchange(rec, sync)


fused._exchange = counting
o = scratch(x)
n_fwd = len(calls)
crit(o, t).backward()
fused._exchange = real_exchange
res['exchanges_per_step'] = [n_fwd, len(calls) - n_fwd]
del scratch, o

if mode == 'split':
    buckets = GradBuckets(model.parameters(), world, adjacent=fused.weight_pairs(model))
    state0 = {k: v.clone() for k, v in model.state_dict().items() if 'running' in k or 'num_batches' in k}

    def step(xb, tb):
        buckets.reset()
        out = model(xb)
        ls = crit(out, tb)
        ls.backward()
        buckets.finish()
        return ls, out

    graphed = GraphedStep(step, (x, t), warmup=2) if backend == 'nccl' else (lambda: step(x, t))
    with torch.no_grad():                                   # the warm-up steps moved the running statistics: start from the reference's
        for k, v in model.state_dict().items():
            if k in state0:
                v.copy_(state0[k])
    loss, out = graphed()
    torch.cuda.synchronize()
    run1, g1, l1 = buffers(model), [p.grad.detach().clone() for p in model.parameters()], loss.clone()
    gl = loss.detach().clone()
    dist.all_reduce(gl, op=dist.ReduceOp.AVG)
    res['loss_rel'] = abs(gl.item() - loss_ref.item()) / abs(loss_ref.item())
    res['out_rel_l2'] = rel_l2(out, out_ref[mine])
    res['running_max_rel'] = max_rel(run1, run_ref)
    res['grad_rel_l2'], res['worst_grad_rel_l2'] = grad_figures(g1)
    flat = torch.cat([b.flatten() for b in run1])
    flat0 = flat.clone()
    dist.broadcast(flat0, 0)
    agree = torch.tensor([float(torch.equal(flat, flat0))], device='cuda')
    loss2, _ = graphed()
    torch.cuda.synchronize()
    same = torch.equal(loss2, l1) and all(torch.equal(p.grad, g) for p, g in zip(model.parameters(), g1))
    agree = torch.cat([agree, torch.tensor([float(same)], device='cuda')])
    dist.all_reduce(agree, op=dist.ReduceOp.MIN)
    res['ranks_agree_on_running_stats'], res['replays_bit_identical'] = bool(agree[0]), bool(agree[1])
else:
    state0 = copy.deepcopy(model.state_dict())
    out = model(x)
    crit(out, t).backward()
    torch.cuda.synchronize()
    run_fused = buffers(model)
    res['running_max_rel'] = max_rel(run_fused, run_ref)
    res['out_rel_l2'] = rel_l2(out, out_ref[mine])
    # torch's SyncBatchNorm on the module path, eager, from the same state; the DP loss is the mean of the per-rank losses
    model.load_state_dict(state0)
    gm.set_fused(False)
    lm = crit(model(x), t)
    lm.backward()
    gm.set_fused(True)
    torch.cuda.synchronize()
    lf = torch.stack([crit(out, t).detach(), lm.detach()])
    dist.all_reduce(lf, op=dist.ReduceOp.AVG)
    res['module_loss_rel'] = abs(lf[0].item() - lf[1].item()) / abs(lf[1].item())
    res['module_running_max_rel'] = max_rel(run_fused, buffers(model))
    # ico2ico_vae, eager: the chains synchronise, the latent heads run torch's SyncBatchNorm
    pv = gm.default_params('ico2ico_vae', level)
    torch.manual_seed(1)
    vae = torch.nn.SyncBatchNorm.convert_sync_batchnorm(gm.ico2ico_vae(pv).cuda().train())
    f = (pv['ico']['factor_pos'], pv['ico']['factor_nor'], pv['ico']['factor_lap'])
    reparam.manual_seed(3)
    lv = losses.P2PKLD_Loss(level, *f, 1.0)(vae(x), t)
    lv.backward()
    torch.cuda.synchronize()
    vb = torch.cat([b.double().flatten() for n, b in vae.named_buffers() if 'running' in n or 'num_batches' in n])
    v0 = vb.clone()
    dist.broadcast(v0, 0)
    ok = torch.tensor([float(bool(torch.isfinite(lv)) and all(bool(torch.isfinite(p.grad).all()) for p in vae.parameters() if p.grad is not None)),
                       float(torch.equal(vb, v0))], device='cuda')
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    res['vae_finite'], res['vae_ranks_agree'] = bool(ok[0]), bool(ok[1])

KEYS = ('loss_rel', 'out_rel_l2', 'running_max_rel', 'grad_rel_l2', 'worst_grad_rel_l2', 'module_loss_rel', 'module_running_max_rel')
worst = torch.tensor([res.get(k, 0.0) for k in KEYS], device='cuda', dtype=torch.float64)
dist.all_reduce(worst, op=dist.ReduceOp.MAX)                 # every rank's figures count
for k, v in zip(KEYS, worst.tolist()):
    if k in res:
        res[k] = v
if rank == 0:
    print(json.dumps(res), flush=True)
torch.cuda.synchronize()
dist.barrier()
torch.cuda.synchronize()
sys.stdout.flush()
os._exit(0)          # destroying a communicator whose collectives live in a captured graph hung at exit (dp_parity_worker.py)
