#!/usr/bin/env python
"""Headline benchmark: ico2ico training meshes/s at I5, batch 36 per GPU (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W          # ours (one process per GPU under torchrun for N > 1)
    python bench.py --impl reference ...                   # the reference's CPU path (oracle port) on the host cores

One step = forward + P2P loss + backward + gradient all-reduce + Adam step of the reference's
ico2ico graph (models.py:219-232) on one synthetic batch.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_MESH = {('ico2ico', 5): 31.4e9, ('ico2ico_vae', 5): 35.3e9, ('ico2ico', 6): 125.5e9}   # SURVEY 8d


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--model', default='ico2ico', choices=['ico2ico', 'ico2ico_vae'])
    ap.add_argument('--level', type=int, default=5)
    ap.add_argument('--batch', type=int, default=None, help='per-GPU batch (default 36 at I5, 16 at I6)')
    ap.add_argument('--conv-impl', default='auto', choices=['auto', 'simt', 'tc'])
    ap.add_argument('--optimizer', default=os.environ.get('GIN_BENCH_OPTIMIZER', 'gin'), choices=['gin', 'torch'],
                    help="gin: geniconet_b200.optim.Adam (one launch per step); torch: torch.optim.Adam(fused=True)")
    ap.add_argument('--no-graph', action='store_true', help='issue every launch from Python instead of replaying one CUDA graph per step')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-kernel-table', action='store_true')
    ap.add_argument('--cpu-batch', type=int, default=None, help='batch of the CPU arm / cpu_baseline (default: the per-GPU batch)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step computed (loss, model output, updated parameters, '
                         'gradients) to DIR/<name>.npy in float32, for output-by-output comparison of two builds')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs dumps the GPU path; the reference arm has none')
    return args


# --------------------------------------------------------------------------------------- output dump
DUMP_BUDGET = 64 << 20          # bytes of float32 data, all files together
DUMP_MAX_ELEMS = 1 << 21        # a larger array is stored as a fixed, seeded sample of at most this many elements


def dump_outputs(dirname, arrays):
    """Write {name: tensor} as DIR/<name>.npy (float32).  An array above the per-array cap is replaced by a seeded sample of its
    flattened elements; the cap starts at DUMP_MAX_ELEMS and is halved until all arrays fit DUMP_BUDGET.  The sample indices
    depend only on the array size and the cap, so runs with the same arguments sample the same elements."""
    import numpy as np
    sizes = [t.numel() for t in arrays.values()]
    cap = DUMP_MAX_ELEMS
    while sum(min(n, cap) for n in sizes) * 4 > DUMP_BUDGET:
        cap //= 2
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(dirname, name + '.npy'), a)


# --------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        mhz, mx, reasons, pw = [], None, set(), []
        for r in self.rows:
            try:
                mhz.append(float(r[0])); mx = float(r[1]); pw.append(float(r[2]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        busy = [m for m, p in zip(mhz, pw) if p > 250] or mhz
        return {'sm_mhz': statistics.median(busy) if busy else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'power_w_max': max(pw) if pw else None, 'samples': len(mhz)}


# --------------------------------------------------------------------------------------- CPU arm
def workload_config(model, level, B):
    """The `config` object both arms print (the reference arm measures the same workload on the host cores)."""
    act_gb = 12.0 * B / 36 * (4 ** (level - 5))
    return {'workload': '%s I%d train step (fwd+loss+bwd+allreduce+Adam), batch %d/GPU' % (model, level, B),
            'l2': 'no flush: one step streams ~%.0f GB of activations, far beyond the 126 MB L2' % act_gb}


def cpu_reference_step_time(model_name, level, batch, steps, warmup, anomaly=False):
    """The reference's CPU path: the ico2ico / ico2ico_vae graph and losses restated in oracle/models_ref.py over the oracle
    icocnn port (fp32, PyTorch CPU, every host core).  Imports NOTHING from geniconet_b200 -- the product library is not
    mapped into this process.  anomaly=True wraps the loop in torch.autograd.detect_anomaly() as the reference's train() does
    (run.py:237).  Returns (median seconds per step, threads used)."""
    import contextlib
    import warnings
    import torch
    from oracle import models_ref, synth_ref
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)        # torchrun exports OMP_NUM_THREADS=1: without this the arm would run on one core
    torch.manual_seed(0)
    model = models_ref.build(model_name, level)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    x, tgt = synth_ref.synthetic_batch(level, 0, min(batch, 4))
    reps = (batch + x.shape[0] - 1) // x.shape[0]                # distinct meshes cost host time to generate, not to train on
    x, tgt = x.repeat(reps, 1, 1, 1)[:batch].contiguous(), tgt.repeat(reps, 1, 1)[:batch].contiguous()
    times = []
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        with (torch.autograd.detect_anomaly() if anomaly else contextlib.nullcontext()):
            for i in range(warmup + steps):
                t0 = time.perf_counter()
                opt.zero_grad()
                loss = models_ref.training_loss(model_name, level, model(x), tgt)
                loss.backward()
                opt.step()
                float(loss)
                if i >= warmup:
                    times.append(time.perf_counter() - t0)
    return statistics.median(times), torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    B = args.batch or (36 if args.level == 5 else 16)
    batch = args.cpu_batch or B                      # default: the arm's real per-GPU batch
    steps, warmup = args.steps, args.warmup          # a batch-36 step is seconds of CPU time: --cpu-batch / --steps keep it short
    t, threads = cpu_reference_step_time(args.model, args.level, batch, steps, warmup)
    t_anom, _ = cpu_reference_step_time(args.model, args.level, batch, 1, 0, anomaly=True)   # as run.py:237 trains
    val = batch / t
    line = {'impl': 'reference', 'metric': 'train_meshes_per_sec', 'value': val, 'unit': 'meshes/s', 'n_gpus': args.gpus,
            'steps': steps, 'warmup': warmup, 'ms_per_step': t * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args.model, args.level, B),
            'cpu_baseline': {'value': val, 'unit': 'meshes/s', 'cores': threads, 'kind': 'port',
                             'sample': 'one host process, batch %d per step, median of %d steps after %d warm-up; oracle/models_ref.py '
                                       '(reference graph + losses restated) over the oracle icocnn port, PyTorch CPU (oneDNN), fp32, '
                                       'torch.set_num_threads(os.cpu_count()=%d)' % (batch, steps, warmup, threads),
                             'with_detect_anomaly': batch / t_anom},
            'e2e': {'value': val, 'unit': 'meshes/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------- ours
def conv_calls(model, fused):
    """The distinct tcgen05 hex-conv problems one training step launches: (name, Cin, Cout, stride, level, corner_mode, count).
    On the fused path the two sibling convolutions of a residual block are ONE problem with concatenated output channels."""
    from geniconet_b200.ico_conv import IcoConvS2S
    calls = {}

    def add(name, ci, co, stride, lvl, cm):
        key = (ci, co, stride, lvl)
        if key in calls:
            calls[key][-1] += 1
        else:
            calls[key] = [name, ci, co, stride, lvl, cm, 1]
    if fused:
        for name, m in model.named_modules():
            if hasattr(m, 'conv00') and hasattr(m, 'icobn10'):
                c0, c1 = m.conv00, m.conv01
                add(name + '.conv00|conv10', c0.in_features, 2 * c0.out_features, c0.stride, c0.subdivisions, c0.corner_mode)
                add(name + '.conv01', c1.in_features, c1.out_features, 1, c1.subdivisions, c1.corner_mode)
            elif isinstance(m, IcoConvS2S) and name.split('.')[-1] not in ('conv00', 'conv01', 'conv10') and m.in_features % 64 == 0:
                add(name, m.in_features, m.out_features, m.stride, m.subdivisions, m.corner_mode)
    else:
        for name, m in model.named_modules():
            if isinstance(m, IcoConvS2S) and m.in_features % 64 == 0 and m.out_features % 64 == 0:
                add(name, m.in_features, m.out_features, m.stride, m.subdivisions, m.corner_mode)
    return list(calls.values())


def kernel_table(model, B, level, peaks, steps=5, fused=True):
    """Per-problem CUDA-event timings of the hex-conv kernels through the C ABI on activations of the real shapes (the problems
    of conv_calls).  Every problem runs on ROTATING buffer sets whose combined size exceeds twice the 126 MB L2, so a launch
    never finds the operands of an earlier launch in L2 (`sets` in each row); launches are replayed as one CUDA graph and
    timed with events on the replaying stream."""
    import torch
    from geniconet_b200 import _lib
    from geniconet_b200.ico_conv import get_plan
    L = _lib.lib
    rows = []
    for name, Ci, Co, stride, lvl, cm, count in conv_calls(model, fused):
        n = 2 ** lvl
        Pin, Pout = 10 * 4 ** lvl, 10 * 4 ** lvl // (stride ** 2)
        lvl_out = lvl - (1 if stride == 2 else 0)
        plan = get_plan(_lib.PLAN_HEXCONV, lvl, stride, cm, 'cuda')
        st = torch.cuda.current_stream().cuda_stream
        w = torch.randn(Co, Ci, 7, device='cuda') * 0.05
        bias = torch.zeros(Co, device='cuda')
        packed = torch.empty(L.gin_hexconv_packed_bytes(Ci, Co), dtype=torch.uint8, device='cuda')
        _lib.check(L.gin_hexconv_pack_weights(w.data_ptr(), packed.data_ptr(), Ci, Co, st))
        dW = torch.empty(Co, Ci, 7, device='cuda')
        ws = torch.empty(L.gin_hexconv_wgrad_ws_bytes(Ci, Co), dtype=torch.uint8, device='cuda')
        set_bytes = B * (6.0 * Ci * Pin + 6.0 * Co * Pout)           # bf16 copy + fp32 map on either side
        nsets = int(min(8, max(2, -(-2 * 126e6 // set_bytes) + 1)))
        sets = []
        for _ in range(nsets):
            x = torch.randn(B, 5 * n, 2 * n, Ci, device='cuda').permute(0, 3, 1, 2)
            dy = torch.randn(B, 5 * n // stride, 2 * n // stride, Co, device='cuda').permute(0, 3, 1, 2)
            xb = torch.empty(L.gin_cast_bf16_bytes(B, lvl, Ci) // 2, dtype=torch.bfloat16, device='cuda')
            dyb = torch.empty(L.gin_cast_bf16_bytes(B, lvl_out, Co) // 2, dtype=torch.bfloat16, device='cuda')
            _lib.check(L.gin_cast_bf16(plan.host_ptr, plan.dev_ptr, 0, x.data_ptr(), xb.data_ptr(), B, Ci, st))
            _lib.check(L.gin_cast_bf16(plan.host_ptr, plan.dev_ptr, 1, dy.data_ptr(), dyb.data_ptr(), B, Co, st))
            sets.append((xb, dyb, torch.empty_like(dy), torch.empty_like(x)))
            del x, dy

        def fwd(b, s):
            _lib.check(L.gin_hexconv_fwd_bf16(plan.host_ptr, plan.dev_ptr, b[0].data_ptr(), packed.data_ptr(), bias.data_ptr(), b[2].data_ptr(), B, Ci, Co, s))

        def dgrad(b, s):
            _lib.check(L.gin_hexconv_dgrad_bf16(plan.host_ptr, plan.dev_ptr, b[1].data_ptr(), packed.data_ptr(), b[3].data_ptr(), B, Ci, Co, s))

        def wgrad(b, s):
            _lib.check(L.gin_hexconv_wgrad_bf16(plan.host_ptr, plan.dev_ptr, b[0].data_ptr(), b[1].data_ptr(), None, dW.data_ptr(), None, ws.data_ptr(),
                                                B, Ci, Co, s))
        flops = 2.0 * 7 * Ci * Co * Pout * B
        # algorithmic bytes of one pass: bf16 operand copy read once + fp32 result written once (fwd, dgrad); both copies read (wgrad)
        by = {'fwd': B * (2.0 * Ci * Pin + 4.0 * Co * Pout), 'dgrad': B * (2.0 * Co * Pout + 4.0 * Ci * Pin),
              'wgrad': B * (2.0 * Ci * Pin + 2.0 * Co * Pout) + 28.0 * Ci * Co}
        ent = {'layer': name, 'cin': Ci, 'cout': Co, 'stride': stride, 'level': lvl, 'count': count, 'gflop': flops / 1e9,
               'sets': nsets, 'set_mbytes': set_bytes / 1e6}
        nl = max(steps, nsets) * 2
        for tag, fn in (('fwd', fwd), ('dgrad', dgrad), ('wgrad', wgrad)):
            for b in sets[:2]:
                fn(b, st)
            torch.cuda.synchronize()
            # device time only: `nl` back-to-back calls replayed as one CUDA graph (issued from Python a call costs
            # 20-30 us of host time, more than several of these kernels run)
            side = torch.cuda.Stream()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                with torch.cuda.graph(graph, stream=side):
                    for i in range(nl):
                        fn(sets[i % nsets], side.cuda_stream)
            graph.replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / nl
            ent[tag + '_us'] = ms * 1e3
            ent[tag + '_tflops'] = flops / (ms * 1e-3) / 1e12
            ent[tag + '_mbytes'] = by[tag] / 1e6
            ent[tag + '_gbs'] = by[tag] / (ms * 1e-3) / 1e9
        rows.append(ent)
        del sets
    return rows


def conv_roofline(table, peaks, args, B):
    """`roofline` object: the tcgen05 hex-conv kernel family (cv2::patch_conv_kernel [+ pair variant] forward and dgrad,
    wg2::wgrad_patch_kernel [+ reduce]) over ALL launches of one training step -- forward + dgrad + wgrad of every problem.
    achieved = sum of algorithmic FLOPs / sum of measured durations; the per-pass aggregates stay in `passes`."""
    hbm = peaks.get('hbm_gbs', 6650.0)
    tf_burst = peaks.get('bf16_tflops', 1590.0)
    ridge = tf_burst * 1e12 / (hbm * 1e9)
    tags = ('fwd', 'dgrad', 'wgrad')
    nl = 3 * sum(r['count'] for r in table)
    gflop1 = sum(r['gflop'] * r['count'] for r in table)
    gflop = 3 * gflop1
    mbytes = sum(r[t + '_mbytes'] * r['count'] for r in table for t in tags)
    us = sum(r[t + '_us'] * r['count'] for r in table for t in tags)
    ai = gflop * 1e9 / (mbytes * 1e6)
    if ai >= ridge:
        roof = {'bound': 'tensor', 'achieved': gflop / 1e3 / (us * 1e-6), 'peak': tf_burst, 'unit': 'TFLOP/s'}
    else:
        roof = {'bound': 'hbm', 'achieved': mbytes / 1e3 / (us * 1e-6), 'peak': hbm, 'unit': 'GB/s'}
    roof['frac'] = roof['achieved'] / roof['peak']
    roof['traffic'] = None
    try:          # ncu dram__bytes_read.sum + dram__bytes_write.sum of exactly this launch set (tools/measure_traffic.py)
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')))
        if tr.get('launches') == nl and args.model == 'ico2ico' and args.level == 5 and B == 36:
            roof['traffic'] = tr['dram_bytes_per_launch'] / 1e6
            roof['traffic_unit'] = 'MB per launch (dram__bytes_read.sum + dram__bytes_write.sum, L2 flushed before every launch)'
    except Exception:
        pass
    roof['kernel'] = 'tcgen05 hex-conv kernels (cv2::patch_conv*, wg2::wgrad_patch*): the %d fwd + dgrad + wgrad calls of one step' % nl
    roof['peak_source'] = ('measured' if peaks else 'fallback') + ' (MEASURED_PEAKS.json burst figure: kernels timed alone, back to back)'
    roof['timing'] = 'CUDA events around a replayed CUDA graph of back-to-back launches over rotating buffer sets > 2x L2'
    roof['algorithmic'] = {'gflop_per_launch': gflop / nl, 'mbytes_per_launch': mbytes / nl, 'us_per_launch': us / nl,
                           'arithmetic_intensity': ai, 'ridge': ridge}
    roof['passes'] = {}
    for tag in tags:
        t_us = sum(r[tag + '_us'] * r['count'] for r in table)
        roof['passes'][tag] = {'us_per_step': t_us, 'tflops': gflop1 / 1e3 / (t_us * 1e-6),
                               'frac_of_peak': gflop1 / 1e3 / (t_us * 1e-6) / tf_burst}
    allp = [(r[t + '_tflops'], t, r) for r in table for t in tags]
    lo, hi = min(allp, key=lambda v: v[0]), max(allp, key=lambda v: v[0])
    fmt = lambda v: '%s %d->%d s%d L%d: %.0f TFLOP/s' % (v[1], v[2]['cin'], v[2]['cout'], v[2]['stride'], v[2]['level'], v[0])
    roof['range'] = {'best': fmt(hi), 'worst': fmt(lo)}
    return roof


def run_ours(args):
    world_env = int(os.environ.get('WORLD_SIZE', 1))
    if world_env > 1:
        # Experiment switch (off by default): leave GIN_DP_SPARE_SMS SMs to the NCCL kernels and hold NCCL to that many CTAs.
        # Measured WORSE at every setting (2 ranks: 4.046 ms with 0, 4.064 with 4, 4.122 with 8, 4.153 with 16 spare SMs --
        # profiles/r02_dp_overhead_breakdown.md): the conv kernels lose more than the exchange gains.  Both variables must be
        # in the environment before the library / NCCL initialise.
        spare = int(os.environ.get('GIN_DP_SPARE_SMS', '0'))
        if spare > 0:
            os.environ.setdefault('GIN_SMS', str(148 - spare))
            os.environ.setdefault('NCCL_MAX_CTAS', str(spare))
    import torch
    import torch.distributed as dist
    from geniconet_b200 import _lib, models as gm, losses, data
    from geniconet_b200.dp import GradBuckets, shard_sample_ids, broadcast_parameters
    from geniconet_b200.ico_conv import set_impl

    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- geniconet_b200 has no CPU path')
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    # NCCL writes its version banner to the C-level stdout; rank 0 must print ONE JSON line there.  Everything else that goes to
    # file descriptor 1 is sent to stderr, the JSON line is written to the saved descriptor at the end.
    json_fd = os.dup(1)
    sys.stdout.flush()
    os.dup2(2, 1)
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    B = args.batch or (36 if args.level == 5 else 16)
    params = gm.default_params(args.model, args.level)
    torch.manual_seed(0)
    model = getattr(gm, args.model)(params).cuda()
    set_impl(model, args.conv_impl)
    if world > 1:
        broadcast_parameters(model)
    f = (params['ico']['factor_pos'], params['ico']['factor_nor'], params['ico']['factor_lap'])
    crit = losses.P2PKLD_Loss(args.level, *f, 1.0) if args.model == 'ico2ico_vae' else losses.P2P_Loss(args.level, *f)
    from geniconet_b200 import fused as _fused
    buckets = GradBuckets(model.parameters(), world, adjacent=_fused.weight_pairs(model))
    use_graph = not args.no_graph
    # data parallel: one optimizer per gradient bucket, stepped as soon as that bucket's all-reduce is done -- the last (smallest)
    # exchange then hides behind the update of the earlier buckets
    if args.optimizer == 'gin':
        from geniconet_b200.optim import Adam as _Adam
        make_opt = lambda ps: _Adam(ps, lr=1e-4)
    else:
        make_opt = lambda ps: torch.optim.Adam(ps, lr=1e-4, fused=True, capturable=use_graph)
    opts = [make_opt(ps) for ps in (buckets.bucket_params() if world > 1 else [list(model.parameters())])]

    # one synthetic shard per rank, staged in pinned host memory (SURVEY 8d / 8e)
    ids = shard_sample_ids(0, rank, world, B)
    xs, ts = zip(*(data.synthetic_mesh(args.level, i) for i in ids))
    x_host, t_host = torch.stack(xs).pin_memory(), torch.stack(ts).pin_memory()
    x_dev, t_dev = x_host.cuda(), t_host.cuda()

    params = list(model.named_parameters())

    def step(x, t):
        # returns the loss, the model output and the gradients: under the graph these are static tensors the replays rewrite
        buckets.reset()
        y = model(x)
        loss = crit(y, t)
        loss.backward()
        for bi, o in enumerate(opts):
            buckets.finish_bucket(bi)
            o.step()
        buckets.finish()
        return loss, y, [p.grad for _, p in params]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_rank_ms = []          # ms per step of every rank, one list per timed() call (the reported time is the maximum)

    def timed(fn, steps, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()                                      # host work that belongs to the timed steps (the last loss read-back)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device='cuda')
        if world > 1:
            every = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(every, ms)
            per_rank_ms.append([v.item() / steps for v in every])
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    W = max(args.warmup, 3)
    if use_graph:
        # the whole step (fwd + loss + bwd + bucketed all-reduce + Adam) is captured once and replayed: one launch per step
        from geniconet_b200.graph import GraphedStep
        graphed = GraphedStep(step, (x_dev, t_dev), warmup=3)
        eager_step = step

        def step(x, t):                                   # noqa: F811  (x, t are the static buffers the graph reads)
            if x is not x_dev:
                x_dev.copy_(x, non_blocking=True)
                t_dev.copy_(t, non_blocking=True)
            return graphed()
    for _ in range(W):
        last = step(x_dev, t_dev)[0]
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = _lib.launch_count()
    ms_total = timed(lambda: step(x_dev, t_dev), args.steps)
    launches = _lib.launch_count() - l0
    if use_graph:
        # replays do not pass through the library's counter: count the launches of one eagerly issued step instead
        # (the graph holds exactly these kernels) and scale by the number of timed steps
        l0 = _lib.launch_count()
        eager_step(x_dev, t_dev)
        launches = (_lib.launch_count() - l0) * args.steps
    ms_step = ms_total / args.steps

    # End to end: every step copies ITS batch from pinned host memory and reads its loss back.  As a data loader would, the
    # host->device copy of the next batch runs on a copy stream into a staging buffer while the current step computes; the
    # step then starts with a device-side copy from the staging buffer into the graph's static inputs.  The loss of step k goes
    # to a pinned two-slot ring with a non-blocking copy and is read by the host once step k+1 has been enqueued (a training
    # loop that logs its loss one step late), so the device never waits for the host; every loss, the last one included
    # (read_last), is read inside the timed region.
    copy_stream = torch.cuda.Stream()
    x_stage, t_stage = torch.empty_like(x_dev), torch.empty_like(t_dev)
    staged, consumed = torch.cuda.Event(), torch.cuda.Event()

    def prefetch():
        copy_stream.wait_event(consumed)                  # the previous contents of the staging buffers have been taken over
        with torch.cuda.stream(copy_stream):
            x_stage.copy_(x_host, non_blocking=True)
            t_stage.copy_(t_host, non_blocking=True)
            staged.record(copy_stream)

    def e2e_step():
        main = torch.cuda.current_stream()
        main.wait_event(staged)
        if use_graph:
            x_dev.copy_(x_stage, non_blocking=True)
            t_dev.copy_(t_stage, non_blocking=True)
            consumed.record(main)
            prefetch()                                    # the next batch's H2D overlaps this step
            ring['result'] = step(x_dev, t_dev)
        else:
            xd, td = x_stage.clone(), t_stage.clone()
            consumed.record(main)
            prefetch()
            ring['result'] = step(xd, td)
        loss = ring['result'][0]
        k = ring['k']
        loss_ring[k & 1:(k & 1) + 1].copy_(loss.detach().reshape(1), non_blocking=True)
        ring['event'][k & 1] = torch.cuda.Event()
        ring['event'][k & 1].record()
        ring['k'] = k + 1
        read_loss((k - 1) & 1)

    loss_ring = torch.zeros(2).pin_memory()
    ring = {'k': 0, 'event': [None, None], 'losses': []}

    def read_loss(slot):
        ev = ring['event'][slot]
        if ev is not None:
            ev.synchronize()
            ring['losses'].append(float(loss_ring[slot]))
            ring['event'][slot] = None

    def read_last():
        read_loss((ring['k'] - 1) & 1)

    consumed.record(torch.cuda.current_stream())
    prefetch()
    for _ in range(2):
        e2e_step()
    read_last()
    ring['losses'] = []
    ms_e2e = timed(e2e_step, args.steps, finish=read_last) / args.steps
    if len(ring['losses']) != args.steps:
        raise SystemExit('bench.py: %d losses read back in %d end-to-end steps' % (len(ring['losses']), args.steps))
    clk = clocks.stop() if rank == 0 else None
    final_loss = float(last.detach())
    if rank == 0 and args.dump_outputs:
        # the last end-to-end step is the last timed step
        loss, y, grads = ring['result']
        arrays = {'input.x': x_dev, 'input.target': t_dev, 'loss': loss.reshape(1)}
        arrays.update(zip(('output', 'mu', 'logvar'), y if isinstance(y, tuple) else (y,)))     # ico2ico_vae: (output, mu, logvar)
        arrays.update(('param.' + n, p) for n, p in params)
        arrays.update(('grad.' + n, g) for (n, _), g in zip(params, grads) if g is not None)
        dump_outputs(args.dump_outputs, arrays)

    table, roof = None, None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        if not args.no_kernel_table:
            from geniconet_b200 import models as _gm
            table = kernel_table(model, B, args.level, peaks, fused=_gm._FUSED)
            roof = conv_roofline(table, peaks, args, B)

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cb = args.cpu_batch or B
        t_cpu, threads = cpu_reference_step_time(args.model, args.level, cb, 2, 1)
        cpu = {'value': cb / t_cpu, 'unit': 'meshes/s', 'cores': threads, 'kind': 'port',
               'sample': 'batch %d train step (fwd+loss+bwd+Adam), median of 2 after 1 warm-up; oracle/models_ref.py over the oracle '
                         'icocnn port on PyTorch CPU fp32, torch.set_num_threads(os.cpu_count()=%d)' % (cb, threads)}
    if rank == 0:
        meshes = B * world
        line = {'metric': 'train_meshes_per_sec', 'value': meshes / (ms_step * 1e-3), 'unit': 'meshes/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': W, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': '%s forward operands, bf16 gradient operands, f32 accumulate (tcgen05 kind::f16); f32 activations, BN, loss, Adam' % ('fp16' if _lib.lib.gin_forward_operand_is_fp16() else 'bf16'),
                'data': 'synthetic',
                'config': workload_config(args.model, args.level, B),
                'details': {'conv_impl': args.conv_impl, 'parallelism': 'dp%d' % world,
                            'optimizer': 'geniconet_b200.optim.Adam (gin_adam_step, one launch)' if args.optimizer == 'gin' else 'torch.optim.Adam(fused=True)',
                            'launch': 'one CUDA graph replay per step' if use_graph else 'eager (one launch per kernel)'},
                'e2e': {'value': meshes / (ms_e2e * 1e-3), 'unit': 'meshes/s', 'ms_per_step': ms_e2e,
                        'h2d_bytes_per_step': x_host.numel() * 4 + t_host.numel() * 4, 'd2h_bytes_per_step': 4,
                        'loss_readback': 'every step, read by the host one step late (pinned ring); %d of %d read inside the timed region' % (len(ring['losses']), args.steps)},
                'gpu_launches': int(launches), 'clocks': clk, 'loss': final_loss,
                'ms_per_step_per_rank': per_rank_ms[0] if per_rank_ms else None,
                'tflops_algorithmic': FLOP_PER_MESH.get((args.model, args.level), 0) * meshes / (ms_step * 1e-3) / 1e12,
                'roofline': roof, 'kernel_table': table, 'cpu_baseline': cpu}
        os.write(json_fd, (json.dumps(line) + '\n').encode())
    if world > 1:
        # Leave without tearing the communicator down: destroying an NCCL communicator whose collectives live in a captured
        # CUDA graph hung at exit (N = 2, r01).  Every rank has finished its work once the barrier returns.
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
