#!/usr/bin/env python
"""bench.py -- RoIs/s through the BAGS head fwd+bwd (1231 classes -> 1236 logits, 5 bins).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of 4096 synthetic RoIs per GPU
(BASELINE.json configs[1]: 4096 RoIs x 1024 feat x 1231 cls, 5 bins, bf16):

    sample "others" masks -> fc_cls GEMM + grouped softmax-CE (5 bins) -> dW, db, dX
    (+ NCCL all-reduce(avg) of the fc_cls gradient bucket when N > 1, restating
     mmdet/core/utils/dist_utils.py:9-41)

`value`  : whole-job RoIs/s with inputs resident in HBM, K steps replayed from a CUDA graph
           (launch-bound inner loop), timed with CUDA events on the launching stream, max over
           ranks.  Each step uses a different member of a rotating pool of buffer sets larger than
           the 126 MB L2, so no step finds its inputs in cache.
`e2e`    : the same metric through the public autograd API (GroupSoftmaxFunction behind
           balancedgroupsoftmax_b200.bags_head_loss) with HOST (pinned) features/labels copied
           H2D and the per-bin losses read back D2H inside the timed region.
`roofline`: the dominant kernel (by measured duration) against MEASURED_PEAKS.json.
`cpu_baseline`: the oracle port of the reference's PyTorch CPU path on this box's host cores.

--impl reference: the reference's own CPU implementation of the path (its source through
oracle/ref_shim.py when a checkout is reachable, else the oracle port), same metric/config.

--dump-outputs DIR: after the timed steps, what the last timed step returned to its caller -- the five per-bin
losses, dW, db and dX of its buffer set -- as DIR/<name>.npy in float32 (see dump_outputs()).  Inputs, sampler
seeds and the step schedule depend only on the arguments, so two builds run with the same arguments can be
compared output for output.  The losses, db and dX repeat bit for bit from run to run; dW is summed split-K in
fp32 in no fixed order, so its last bits vary (measured on a B200: ~5e-8 relative).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ROIS = 4096
K_FEAT = 1024
NUM_CLASSES = 1231
RATIO = 8.0
METRIC = 'RoIs/sec through BAGS head fwd+bwd (1231 cls, 5 bins)'


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        try:
            d = json.load(open(p))
            return dict(hbm_gbs=float(d['hbm_gbs']), bf16_tflops=float(d['bf16_tflops']),
                        bf16_tflops_sustained=float(d.get('bf16_tflops_sustained', d['bf16_tflops'])),
                        source='measured')
        except Exception:
            pass
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source='fallback')


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/ncu_traffic.json)."""
    try:
        d = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
        k = d.get(kernel)
        return None if k is None else int(k['dram_read'] + k['dram_write'])
    except Exception:
        return None


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(directory, arrays, limit=DUMP_LIMIT_BYTES):
    """Write each array as <directory>/<name>.npy in float32, at most `limit` bytes in all.  When the arrays are
    larger than that together, every 2-D array keeps the same share of its rows: a sorted sample drawn with a fixed
    seed, so that runs with the same arguments write the same rows."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    budget = limit - 1024 * len(arrays)           # room for the .npy headers
    small = sum(a.nbytes for a in arrays.values() if a.ndim < 2)
    large = sum(a.nbytes for a in arrays.values() if a.ndim >= 2)
    share = 1.0 if large <= budget - small else (budget - small) / large
    for name, a in arrays.items():
        if a.ndim >= 2 and share < 1.0:
            keep = max(1, int(a.shape[0] * share))
            a = a[np.sort(np.random.RandomState(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(directory, name + '.npy'), a)
    log('wrote %s to %s' % (', '.join(sorted(arrays)), directory))


def make_labels(torch, n, num_classes, gen):
    """25 % positives first in every 512-block (RandomSampler num=512, pos_fraction=.25;
    mmdet/core/bbox/bbox_target.py:44-51), class ids uniform on 1..num_classes-1."""
    labels = torch.zeros(n, dtype=torch.int64)
    for s in range(0, n, 512):
        e = min(n, s + 512)
        npos = (e - s) // 4
        labels[s:s + npos] = torch.randint(1, num_classes, (npos,), generator=gen)
    return labels


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        while not self._halt.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(',')]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nm, v in zip(names, f[2:6]):
                    if v.lower().startswith('active'):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        s = sorted(self.samples)
        return dict(sm_mhz=(s[len(s) // 2] if s else None), sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons),
                    samples=len(s))


# ======================================================================================= reference arm
def _numa_nodes():
    """[(node id, [cpu ids])] from sysfs, restricted to the CPUs this process may run on."""
    allowed = os.sched_getaffinity(0)
    nodes = []
    base = '/sys/devices/system/node'
    try:
        for d in sorted(os.listdir(base)):
            if not (d.startswith('node') and d[4:].isdigit()):
                continue
            cpus = []
            for part in open(os.path.join(base, d, 'cpulist')).read().strip().split(','):
                if not part:
                    continue
                a, _, b_ = part.partition('-')
                cpus.extend(range(int(a), int(b_ or a) + 1))
            cpus = [c for c in cpus if c in allowed]
            if cpus:
                nodes.append((int(d[4:]), cpus))
    except Exception:
        pass
    return nodes or [(0, sorted(allowed))]


def run_reference(args):
    """The reference's CPU path on the host cores.  The 2-socket GPU hosts made an all-cores run 16-80x slower and
    noisier than a one-socket run (OpenMP threads ping-ponging 25 MB of activations across NUMA nodes), so: pin the
    process to ONE NUMA node before torch spins up its thread pool, sweep the thread count, and time the K steps with
    the best setting.  The sweep is reported in the line."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    nodes = _numa_nodes()
    node_id, node_cpus = max(nodes, key=lambda nc: len(nc[1]))
    try:
        os.sched_setaffinity(0, set(node_cpus))     # inherited by every thread torch / OpenMP creates later
    except Exception:
        pass
    os.environ.setdefault('OMP_PROC_BIND', 'close')
    import numpy as np
    import torch
    from balancedgroupsoftmax_b200.tables import synthetic_tables
    from oracle import bags_oracle as O
    from oracle import ref_shim

    tables = synthetic_tables(NUM_CLASSES, seed=0)
    gen = torch.Generator().manual_seed(0)
    n = args.rois
    x = torch.relu(torch.randn(n, K_FEAT, generator=gen))
    labels = make_labels(torch, n, NUM_CLASSES, gen)
    l2b, ps = torch.from_numpy(tables.label2binlabel), torch.from_numpy(tables.pred_slice)
    np.random.seed(0)

    if ref_shim.available():
        kind = 'reference'
        head = ref_shim.build_reference_head(tables, RATIO)
        head.init_weights()

        def step():
            xr = x.detach().requires_grad_(True)
            head.zero_grad()
            z = head.fc_cls(xr)
            losses = head.loss(z, None, labels, None, None, None)
            sum(losses.values()).backward()
    else:
        kind = 'port'
        W = torch.randn(tables.num_logits, K_FEAT, generator=gen) * 0.01
        b = torch.zeros(tables.num_logits)

        def step():
            O.head_step(x, W, b, labels, l2b, ps, RATIO, need_dx=True)

    ncpu = len(node_cpus)
    cands = sorted({t for t in (8, 16, 32, 64, ncpu) if 1 <= t <= ncpu} or {ncpu})
    sweep = {}
    for t in cands:
        torch.set_num_threads(t)
        step()
        times = []
        t_begin = time.perf_counter()
        while len(times) < 5 and time.perf_counter() - t_begin < 6.0:
            t0 = time.perf_counter()
            step()
            times.append(time.perf_counter() - t0)
        sweep[t] = sorted(times)[len(times) // 2] * 1e3   # median: a setting that is fast once but unstable loses
    best = min(sweep, key=lambda t: sweep[t])
    torch.set_num_threads(best)
    for _ in range(max(args.warmup, 1)):
        step()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    value = n / dt
    srt = sorted(times)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'RoIs/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'BAGS head fwd+loss+bwd(dW,db,dX), %d RoIs x %d feat x %d logits, 5 bins, '
                               'PyTorch CPU fp32' % (n, K_FEAT, tables.num_logits)},
        'cpu_baseline': {'value': value, 'unit': 'RoIs/s', 'cores': best, 'kind': kind,
                         'sample': '%d steps of %d RoIs' % (args.steps, n),
                         'pinned_to': 'NUMA node %d (%d of %d host CPUs)' % (node_id, ncpu, os.cpu_count() or ncpu),
                         'thread_sweep_ms_per_step': {str(t): round(v, 2) for t, v in sweep.items()},
                         'ms_per_step_median': srt[len(srt) // 2] * 1e3, 'ms_per_step_min': srt[0] * 1e3},
        'e2e': {'value': value, 'unit': 'RoIs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def cpu_baseline(n, steps=10):
    """The CPU arm (oracle port of the reference path, or the reference itself where a checkout is reachable) in a
    fresh subprocess: pinned to one NUMA node before its thread pool exists, thread count swept (see run_reference)."""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', str(steps), '--warmup', '2',
           '--rois', str(n)]
    env = dict(os.environ)
    for k in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE', 'OMP_NUM_THREADS', 'MKL_NUM_THREADS'):
        env.pop(k, None)
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
        line = json.loads([l for l in res.stdout.splitlines() if l.startswith('{')][-1])
        cb = line['cpu_baseline']
        cb['ms_per_step'] = line['ms_per_step']
        return cb
    except Exception as ex:  # pragma: no cover
        log('cpu baseline subprocess failed: %r' % (ex,))
        return None


def gpu_library_baseline(torch, tables, dev, n, iters=20):
    """The on-device bar SURVEY.md 2.2 names: the reference's own formulation through the vendor libraries on the SAME
    B200 -- F.linear (cuBLAS) + 5 x F.cross_entropy on column slices (ATen) + autograd backward (dW, db, dX).  The
    reference's host-synchronising sampler (gs_bbox_head_with0.py:63-89) is left OUT (masks are precomputed device
    tensors), which only flatters the library arm.  Timed eagerly (how the reference runs) and from a CUDA graph."""
    import torch.nn.functional as F
    gen = torch.Generator().manual_seed(5)
    x32 = torch.relu(torch.randn(n, K_FEAT, generator=gen)).to(dev)
    W32 = (torch.randn(tables.num_logits, K_FEAT, generator=gen) * 0.01).to(dev)
    b32 = torch.zeros(tables.num_logits, device=dev)
    labels = make_labels(torch, n, NUM_CLASSES, gen)
    l2b = torch.from_numpy(tables.label2binlabel)
    slices = [(int(s_), int(l_)) for s_, l_ in tables.pred_slice]
    tg = [l2b[g][labels].to(dev) for g in range(tables.num_bins)]
    wg = [torch.ones(n, device=dev) if g == 0 else (torch.rand(n, generator=gen) < 0.6).float().to(dev)
          for g in range(tables.num_bins)]
    inv_avg = [1.0 / max(float(w.sum().item()), 1.0) for w in wg]
    out = {}
    prev_tf32 = torch.backends.cuda.matmul.allow_tf32
    for name in ('fp32', 'tf32', 'bf16'):
        torch.backends.cuda.matmul.allow_tf32 = (name == 'tf32')
        dt_ = torch.bfloat16 if name == 'bf16' else torch.float32
        x = x32.to(dt_).requires_grad_(True)
        W = W32.to(dt_).requires_grad_(True)
        b = b32.to(dt_).requires_grad_(True)

        def step():
            x.grad = W.grad = b.grad = None
            z = F.linear(x, W, b)
            total = None
            for g, (s_, l_) in enumerate(slices):
                ce = F.cross_entropy(z[:, s_:s_ + l_].float(), tg[g], reduction='none')
                term = (ce * wg[g]).sum() * inv_avg[g]
                total = term if total is None else total + term
            total.backward()

        st = torch.cuda.Stream(device=dev)
        st.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(st):
            for _ in range(3):
                step()
            st.synchronize()
            a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            for _ in range(iters):
                step()
            c.record(st)
            st.synchronize()
            out[name + '_eager_us'] = a.elapsed_time(c) / iters * 1e3
            try:
                g_ = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g_, stream=st):
                    step()
                g_.replay()
                st.synchronize()
                a.record(st)
                for _ in range(iters):
                    g_.replay()
                c.record(st)
                st.synchronize()
                out[name + '_graph_us'] = a.elapsed_time(c) / iters * 1e3
                del g_
            except Exception as ex:  # pragma: no cover
                out[name + '_graph_us'] = None
                log('library baseline graph capture failed (%s): %r' % (name, ex))
        torch.cuda.current_stream(dev).wait_stream(st)
    torch.backends.cuda.matmul.allow_tf32 = prev_tf32
    best = min(v for k_, v in out.items() if v is not None)
    out['best_us'] = best
    out['value'] = n / (best * 1e-6)
    out['unit'] = 'RoIs/s'
    out['what'] = ('torch %s on the same GPU: F.linear (cuBLAS) + 5 x F.cross_entropy over column slices (ATen) + autograd '
                   'backward (dW, db, dX), %d RoIs, precomputed masks (no host-sync sampler); fp32 = allow_tf32 off, '
                   'the reference\'s setting' % (torch.__version__, n))
    return out


# ======================================================================================= our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from balancedgroupsoftmax_b200 import ops
    from balancedgroupsoftmax_b200.api import bags_head_loss
    from balancedgroupsoftmax_b200.dist import make_grad_bucket
    from balancedgroupsoftmax_b200.tables import synthetic_tables

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a B200 GPU (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        import datetime
        dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=120))

    dtype = torch.bfloat16 if args.dtype == 'bf16' else torch.float32
    tables = synthetic_tables(NUM_CLASSES, seed=0)
    dt = ops.DeviceTables.from_tables(tables, dev)
    C = tables.num_logits
    n = args.rois
    gen = torch.Generator().manual_seed(1234 + rank)

    # ---- rotating pool of buffer sets, total footprint > 2x L2 ------------------------------
    elt = 2 if dtype == torch.bfloat16 else 4
    ldd = ops.pad_cols(C)
    per_set = n * K_FEAT * elt * 2 + n * C * 4 + n * ldd * elt + C * K_FEAT * 4 + C * K_FEAT * elt * 2
    pool = max(2, int(np.ceil(2.2 * 126e6 / per_set)))
    if args.pool:
        pool = max(2, args.pool)
    elif world > 1 and args.exchange == 'overlap-next-step':
        # one CUDA graph spans the pool; its last exchange cannot hide under a following step, so a longer graph
        # amortises that tail (each set is used once per graph: no exchange ever races a later step on its bucket)
        pool = 20
    sets = []
    W_master = (torch.randn(C, K_FEAT, generator=gen) * 0.01)
    for i in range(pool):
        s = {}
        s['x'] = torch.relu(torch.randn(n, K_FEAT, generator=gen)).to(dev).to(dtype)
        s['w'] = W_master.to(dev).to(dtype)
        s['bias'] = torch.zeros(C, device=dev)
        s['labels'] = make_labels(torch, n, NUM_CLASSES, gen).to(dev)
        s['logits'] = torch.empty(n, C, device=dev)
        # flat fc_cls gradient bucket; at N > 1 it lives in NVLink peer-mapped memory (one-kernel exchange)
        if world > 1:
            s['bucket'], s['grad'], (s['dW'], s['db']), s['exchange'] = make_grad_bucket(
                [(C, K_FEAT), (C,)], dev, prefer_peer=(args.allreduce == 'peer'), max_blocks=args.ar_blocks)
            if s['bucket'] is not None and args.ar_blocks == 0 and args.exchange == 'instep-overlap-dx':
                # the product's rule for an exchange that shares the GPU with the dX GEMM (dist.exchange_overlapped)
                per_rank = (s['bucket'].count // 4 + world - 1) // world
                s['bucket'].max_blocks = max(16, min(48, (per_rank + 2047) // 2048))
        else:
            s['grad'] = torch.empty(C * K_FEAT + C, device=dev)
            s['dW'] = s['grad'][:C * K_FEAT].view(C, K_FEAT)
            s['db'] = s['grad'][C * K_FEAT:]
        s['dX'] = torch.empty(n, K_FEAT, device=dev, dtype=dtype)
        s['wscratch'] = ops.bwd_scratch(s['w'])
        s['wscratch2'] = ops.bwd_scratch(s['w'])   # the split schedule's dX launch (its W' must not race the dW launch's partials)
        sets.append(s)
    exchange_check = None
    if world > 1:
        # the exchange this run times, on RANDOM gradients, against dist.all_reduce(AVG) (dist_utils.py:9-41): same mean on
        # every rank (bit-identical across ranks; vs NCCL exact at 2 ranks, fp32 summation-order rounding beyond)
        gchk = torch.Generator(device=dev).manual_seed(99 + rank)
        worst = 0.0
        for s in sets[:2]:
            src = torch.randn(s['grad'].numel(), device=dev, generator=gchk)
            s['grad'].copy_(src)
            ref = src.clone()
            dist.all_reduce(ref, op=dist.ReduceOp.AVG)
            s['exchange']()
            torch.cuda.synchronize()
            worst = max(worst, (s['grad'] - ref).abs().max().item())
            other = s['grad'].clone()
            dist.broadcast(other, src=0)
            same = torch.tensor([1 if torch.equal(other, s['grad']) else 0], device=dev)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            tw = torch.tensor([worst], device=dev)
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
            worst = float(tw.item())
            if not bool(same.item()) or worst > (0.0 if world == 2 else 2e-6):
                raise SystemExit('gradient exchange check failed: max abs err %.3e vs NCCL AVG, ranks identical: %s'
                                 % (worst, bool(same.item())))
        exchange_check = {'max_abs_err_vs_nccl_avg': worst, 'ranks_bit_identical': True, 'data': 'randn, 2 buckets'}
    gout = torch.ones(dt.G, device=dev)
    seed_ctr = [0]
    last = {}

    def one_step(s):
        seed_ctr[0] += 1
        wmask, avg = ops.sample_others(s['labels'], dt, RATIO, seed_ctr[0])
        prez = args.prep != 'bwd' and not args.unfused
        loss, _, _, dz, colsum = ops.fused_fwd(s['x'], s['w'], s['bias'], s['labels'], dt, wmask, avg,
                                               logits=(s['logits'] if args.unfused else None),
                                               clear=(s['dW'] if prez else None),
                                               want_colsum=(args.prep == 'fwd-zero-colsum' and not args.unfused))
        if split_bwd:
            # in-step schedule with overlap (SURVEY.md 8e: "launch as soon as the dW epilogue finishes, overlap with the dX
            # GEMM"): dW + db first, then the exchange on a side stream WHILE dX runs; joined before the step ends, so the
            # reduced gradients are complete before the next forward starts
            ops.fused_bwd(dz, s['x'], s['w'], gout, dt, colsum, need_dx=False, dW=s['dW'], wscratch=s['wscratch'], db=s['db'],
                          dw_prezeroed=prez)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            side_stream.wait_event(ev)

            def do_exchange(st):
                if world > 1:
                    s['exchange']()
                elif fake is not None:
                    nat.check(nat.lib().bags_debug_spin(fake[0], fake[1], fake[2], st.cuda_stream), 'bags_debug_spin')

            def do_dx():
                ops.fused_bwd(dz, s['x'], s['w'], gout, dt, None, need_dw=False, need_db=False, dX=s['dX'],
                              wscratch=s['wscratch2'])
            if args.dx_side:    # the exchange stays on the launching stream (programmatic dependent launch after dW); dX forks
                with torch.cuda.stream(side_stream):
                    do_dx()
                do_exchange(torch.cuda.current_stream(dev))
            else:
                with torch.cuda.stream(side_stream):
                    do_exchange(side_stream)
                do_dx()
            torch.cuda.current_stream(dev).wait_stream(side_stream)
            last['loss'] = s['loss'] = loss
            return loss
        ops.fused_bwd(dz, s['x'], s['w'], gout, dt, colsum, dW=s['dW'], dX=s['dX'], wscratch=s['wscratch'],
                      db=s['db'], dw_prezeroed=prez)
        if world > 1:
            # mean over ranks of dW, db (dist_utils.py:9-41).  'overlap': on a side stream, concurrently with the next
            # step's kernels (which use another member of the buffer pool); every exchange still completes inside the
            # timed region (the side stream is joined before the closing event / at the end of the graph)
            if comm_stream is not None:
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(dev))
                comm_stream.wait_event(ev)
                with torch.cuda.stream(comm_stream):
                    s['exchange']()
            else:
                s['exchange']()
        elif fake is not None:   # scheduling probe (N = 1): a side-stream kernel that only waits
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            comm_stream.wait_event(ev)
            nat.check(nat.lib().bags_debug_spin(fake[0], fake[1], fake[2], comm_stream.cuda_stream), 'bags_debug_spin')
        last['loss'] = s['loss'] = loss
        return loss

    # sampler, fused fwd (or GEMM + grouped CE), merged backward (preparation jobs + dW + dX units in one launch)
    kernels_per_step = (4 if args.unfused else 3) + (1 if world > 1 and sets[0].get('bucket') is not None else 0) + (
        1 if args.exchange == 'instep-overlap-dx' else 0)   # split schedule: the backward is two launches (dW+db, dX)

    stream = torch.cuda.Stream(device=dev)
    comm_stream = torch.cuda.Stream(device=dev) if (world > 1 and args.exchange == 'overlap-next-step') else None
    split_bwd = args.exchange == 'instep-overlap-dx'   # (at N = 1: the split launches alone, or with --fake-exchange)
    side_stream = torch.cuda.Stream(device=dev) if split_bwd else None
    fake = None
    if world == 1 and args.fake_exchange:
        from balancedgroupsoftmax_b200 import _native as nat
        fake = [int(v) for v in args.fake_exchange.split(',')]    # blocks,threads,microseconds
        if not split_bwd:
            comm_stream = torch.cuda.Stream(device=dev)
    use_graph = not args.no_graph
    graph = None
    with torch.cuda.stream(stream):
        for s in sets[:2]:
            one_step(s)
        if comm_stream is not None:
            stream.wait_stream(comm_stream)
        stream.synchronize()
        if use_graph:
            try:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=stream):
                    for s in sets:
                        one_step(s)
                    if comm_stream is not None:
                        stream.wait_stream(comm_stream)   # join: the graph ends when its last exchange has
            except Exception as e:  # pragma: no cover
                log('graph capture failed (%s); timing eager launches' % (e,))
                graph = None
                use_graph = False
        torch.cuda.synchronize()

        def run_steps(k):
            """exactly k steps"""
            if graph is not None:
                full, rem = divmod(k, pool)
                for _ in range(full):
                    graph.replay()
                for s in sets[:rem]:
                    one_step(s)
            else:
                for i in range(k):
                    one_step(sets[i % pool])
            if comm_stream is not None:
                stream.wait_stream(comm_stream)

        run_steps(max(args.warmup, 3))
        stream.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        clocks = ClockSampler(local_rank)
        clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run_steps(args.steps)
        e1.record(stream)
        stream.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms_total = e0.elapsed_time(e1)
        ms_step = ms_total / args.steps
        if args.dump_outputs and rank == 0:
            # step i of run_steps uses sets[i % pool]; nothing has touched the last one since
            last_set = sets[(args.steps - 1) % pool]
            dump_outputs(args.dump_outputs, {name: last_set[key].detach().float().cpu().numpy() for name, key in (
                ('loss_bins', 'loss'), ('dW', 'dW'), ('db', 'db'), ('dX', 'dX'))})
        if world > 1:
            t = torch.tensor([ms_step], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_step = float(t.item())
        # the timed region is only milliseconds long: keep the SAME workload running for ~0.5 s so that the
        # clock / throttle sampler sees it under load.  The step count is derived from the all-reduced step
        # time, i.e. identical on every rank (the steps contain a collective).
        hold_steps = int(min(50000, max(pool, 500.0 / max(ms_step, 1e-3))))
        run_steps(hold_steps)
        stream.synchronize()
        clk = clocks.stop()
    value = world * n / (ms_step * 1e-3)
    if world > 1:
        # every exchange of the run completed: no bucket recorded a timed-out rank barrier
        bad = [i for i, s in enumerate(sets) if s.get('bucket') is not None and s['bucket'].status() != 0]
        if bad:
            raise SystemExit('gradient exchange timed out on buffer sets %s (rank %d)' % (bad, rank))

    # ---- e2e: public API, host buffers, H2D + D2H inside the timed region -------------------
    e2e = None
    try:
        if args.profile:
            raise RuntimeError('skipped (--profile)')
        from balancedgroupsoftmax_b200.hostmem import pinned_like
        if args.numa_pinned:   # staging buffers allocated / first-touched on the GPU's NUMA node (hostmem.py)
            x_host = pinned_like(torch.relu(torch.randn(n, K_FEAT, generator=gen)).to(dtype), local_rank)
            lab_host = pinned_like(make_labels(torch, n, NUM_CLASSES, gen), local_rank)
        else:
            x_host = torch.relu(torch.randn(n, K_FEAT, generator=gen)).to(dtype).pin_memory()
            lab_host = make_labels(torch, n, NUM_CLASSES, gen).pin_memory()
        # fp32 MASTER weight (the reference's nn.Linear parameter): its bf16 operand copy is made inside every step,
        # and dW / db come back in fp32
        w_param = torch.nn.Parameter(W_master.to(dev))
        b_param = torch.nn.Parameter(torch.zeros(C, device=dev))
        loss_host = torch.empty(dt.G, dtype=torch.float32).pin_memory()
        e2e_steps = max(10, min(args.steps, 200))

        # double-buffered pipeline: the H2D copy of step i+1 (copy stream) overlaps the compute of step i; every
        # step still pays its own H2D of features+labels and its own D2H read of the five losses.
        # Compute = the public API: GraphedHeadStep (CUDA-graph replay of bags_head_loss + backward, one instance per
        # input buffer); the eager autograd calls of the same API are timed as well (`eager_ms_per_step`).
        copy_stream = torch.cuda.Stream(device=dev)
        extra_copy_streams = [torch.cuda.Stream(device=dev) for _ in range(max(args.e2e_copy_streams, 1) - 1)]
        comp_stream = torch.cuda.current_stream(dev)
        loss_hosts = [torch.empty(dt.G, dtype=torch.float32).pin_memory() for _ in range(2)]
        ev_copied = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]
        ev_loss = [torch.cuda.Event() for _ in range(2)]
        e2e_bucket = None
        if world > 1:
            # the public data-parallel API: dW / db land in the exchange bucket, the exchange starts when they are complete
            # and overlaps the dX contraction; weight.grad / bias.grad receive the mean over ranks (dist_utils.py:9-41)
            from balancedgroupsoftmax_b200.dist import NcclGradBucket
            e2e_bucket = make_grad_bucket([(C, K_FEAT), (C,)], dev, prefer_peer=(args.allreduce == 'peer'),
                                          max_blocks=args.ar_blocks)[0]
            if e2e_bucket is None:
                e2e_bucket = NcclGradBucket([(C, K_FEAT), (C,)], dev)
        exchange = None
        graphed = []
        if not args.e2e_eager_only:
            from balancedgroupsoftmax_b200.api import GraphedHeadStep
            graphed = [GraphedHeadStep(w_param, b_param, dt, n, RATIO, compute_dtype=dtype, x_dtype=dtype,
                                       grad_bucket=e2e_bucket) for _ in range(2)]
            if world > 1:
                dist.barrier()
        xd_eager = [torch.empty(n, K_FEAT, device=dev, dtype=dtype) for _ in range(2)]
        ld_eager = [torch.empty(n, device=dev, dtype=torch.int64) for _ in range(2)]
        mode = {'graphed': bool(graphed)}

        ev_h2d0 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev_h2d1 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        h2d_in_pipe = []

        def stage(i):
            b_ = i & 1
            xdst = graphed[b_].x if mode['graphed'] else xd_eager[b_]
            ldst = graphed[b_].labels if mode['graphed'] else ld_eager[b_]
            with torch.cuda.stream(copy_stream), torch.no_grad():
                copy_stream.wait_event(ev_free[b_])
                if i >= 2 and mode.get('probe'):
                    ev_h2d1[b_].synchronize()
                    h2d_in_pipe.append(ev_h2d0[b_].elapsed_time(ev_h2d1[b_]))   # step i-2's copy (long finished)
                ev_h2d0[b_].record(copy_stream)
                if len(extra_copy_streams) == 0:
                    xdst.copy_(x_host, non_blocking=True)
                else:
                    # the feature block in row slabs over several copy streams (several copy engines share the PCIe link)
                    parts = len(extra_copy_streams) + 1
                    bounds = [n * k // parts for k in range(parts + 1)]
                    fork = torch.cuda.Event()
                    fork.record(copy_stream)
                    joins = []
                    for k, st_ in enumerate(extra_copy_streams, start=1):
                        with torch.cuda.stream(st_):
                            st_.wait_event(fork)
                            xdst[bounds[k]:bounds[k + 1]].copy_(x_host[bounds[k]:bounds[k + 1]], non_blocking=True)
                            e_ = torch.cuda.Event()
                            e_.record(st_)
                            joins.append(e_)
                    xdst[bounds[0]:bounds[1]].copy_(x_host[bounds[0]:bounds[1]], non_blocking=True)
                    for e_ in joins:
                        copy_stream.wait_event(e_)
                ldst.copy_(lab_host, non_blocking=True)
                ev_h2d1[b_].record(copy_stream)
                ev_copied[b_].record(copy_stream)

        def compute(i):
            b_ = i & 1
            comp_stream.wait_event(ev_copied[b_])
            if mode['graphed']:
                losses = graphed[b_].replay()
            else:
                xin = xd_eager[b_].detach().requires_grad_(True)
                w_param.grad = None
                b_param.grad = None
                losses = bags_head_loss(xin, w_param, b_param, ld_eager[b_], dt, RATIO, compute_dtype=dtype,
                                        grad_bucket=e2e_bucket)
                losses.sum().backward()
            ev_free[b_].record(comp_stream)
            loss_hosts[b_].copy_(losses.detach(), non_blocking=True)
            ev_loss[b_].record(comp_stream)

        def run_e2e(k):
            for b_ in range(2):
                ev_free[b_].record(comp_stream)
            stage(0)
            for i in range(k):
                if i + 1 < k:
                    stage(i + 1)
                compute(i)
                if i >= 1:
                    ev_loss[(i - 1) & 1].synchronize()   # the previous step's losses are on the host
            ev_loss[(k - 1) & 1].synchronize()

        def time_e2e(k):
            run_e2e(6)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            run_e2e(k)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) / k * 1e3
            if world > 1:
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            return ms

        eager_ms = None
        if graphed:
            mode['graphed'] = False
            eager_ms = time_e2e(max(10, min(e2e_steps, 100)))
            mode['graphed'] = True
        e2e_ms = time_e2e(e2e_steps)
        mode['probe'] = True          # untimed extra pass: how long one step's H2D takes while the pipeline runs
        run_e2e(40)
        torch.cuda.synchronize()
        mode['probe'] = False
        xd = xd_eager
        ld = ld_eager
        # what the copies alone cost (same pinned buffers, no compute): shows how much of the e2e step is PCIe
        ca, cb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(copy_stream):
            ca.record(copy_stream)
            for i in range(20):
                xd[i & 1].copy_(x_host, non_blocking=True)
                ld[i & 1].copy_(lab_host, non_blocking=True)
            cb.record(copy_stream)
        copy_stream.synchronize()
        h2d_ms = ca.elapsed_time(cb) / 20
        # the eager module-level API with device-resident inputs and a DIFFERENT RoI count every call (N is data-dependent in
        # a real detector: no graph) -- what a step costs on the host when nothing hides it
        eager_var_us = None
        if world == 1:
            try:
                sizes = [1024, 960, 1000, 896, 1024, 777, 1010, 512]
                xs = {m: torch.relu(torch.randn(m, K_FEAT, generator=gen)).to(dev).to(dtype) for m in set(sizes)}
                ls = {m: make_labels(torch, m, NUM_CLASSES, gen).to(dev) for m in set(sizes)}

                def eager_var(k):
                    for i in range(k):
                        m = sizes[i % len(sizes)]
                        xin = xs[m].detach().requires_grad_(True)
                        w_param.grad = None
                        b_param.grad = None
                        bags_head_loss(xin, w_param, b_param, ls[m], dt, RATIO, compute_dtype=dtype).sum().backward()
                eager_var(16)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                eager_var(200)
                torch.cuda.synchronize()
                eager_var_us = (time.perf_counter() - t0) / 200 * 1e6
            except Exception as ex:  # pragma: no cover
                log('eager variable-N timing failed: %r' % (ex,))
        cached_var_us = None
        if world == 1 and eager_var_us is not None:
            try:    # the same calls through api.GraphCachedHeadLoss (two CUDA graphs per recurring RoI count)
                from balancedgroupsoftmax_b200.api import GraphCachedHeadLoss
                cached = GraphCachedHeadLoss(dt, RATIO, compute_dtype=dtype, max_graphs=8, capture_after=1)

                def cached_var(k):
                    for i in range(k):
                        m = sizes[i % len(sizes)]
                        xin = xs[m].detach().requires_grad_(True)
                        w_param.grad = None
                        b_param.grad = None
                        cached(xin, w_param, b_param, ls[m]).sum().backward()
                cached_var(3 * len(sizes))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                cached_var(200)
                torch.cuda.synchronize()
                cached_var_us = (time.perf_counter() - t0) / 200 * 1e6
            except Exception as ex:  # pragma: no cover
                log('graph-cached variable-N timing failed: %r' % (ex,))
        e2e = {'value': world * n / (e2e_ms * 1e-3), 'unit': 'RoIs/s', 'h2d_only_ms_per_step': h2d_ms,
               'eager_api_us_per_step_variable_n_le_1024': eager_var_us,
               'graph_cached_api_us_per_step_variable_n_le_1024': cached_var_us,
               'h2d_bytes_per_step': int(x_host.numel() * x_host.element_size() + lab_host.numel() * 8),
               'd2h_bytes_per_step': int(loss_host.numel() * 4), 'ms_per_step': e2e_ms, 'steps': e2e_steps,
               'api': ('balancedgroupsoftmax_b200.api.GraphedHeadStep (CUDA-graph replay of bags_head_loss + backward)'
                       if graphed else 'balancedgroupsoftmax_b200.api.bags_head_loss + autograd backward (eager)'),
               'eager_ms_per_step': eager_ms,
               'h2d_ms_inside_pipeline': (sorted(h2d_in_pipe)[len(h2d_in_pipe) // 2] if h2d_in_pipe else None),
               'staging': ('pinned, GPU-local NUMA node' if args.numa_pinned else 'pinned') + (
                   '; H2D split over %d copy streams' % args.e2e_copy_streams if args.e2e_copy_streams > 1 else ''),
               'operands': ('features staged on the host in %s (the C ABI input format of this dtype mode); fp32 master '
                            'fc_cls.weight cast to the operand dtype inside every step; dW / db returned in fp32'
                            % args.dtype),
               'pipeline': 'H2D of step i+1 overlaps compute of step i (2 buffers); losses read back every step'}
    except Exception as ex:  # pragma: no cover
        log('e2e arm failed: %r' % (ex,))

    # ---- per-kernel durations (CUDA events, rotating sets) for the roofline ------------------
    roof = None
    kernel_us = {}
    if args.profile:
        if rank == 0:
            print(json.dumps({'profile_run': True, 'ms_per_step': ms_step, 'value': value}), flush=True)
        if world > 1:
            graph = None
            torch.cuda.synchronize()
            dist.barrier()
            sys.stdout.flush()
            os._exit(0)
        return 0
    if rank == 0:
        pk = peaks()

        def time_kernel(fn, reps=3):
            with torch.cuda.stream(stream):
                for s in sets:
                    fn(s)
                stream.synchronize()
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                for _ in range(reps):
                    for s in sets:
                        fn(s)
                b_.record(stream)
                stream.synchronize()
            return a.elapsed_time(b_) / (reps * pool) * 1e3

        with torch.cuda.stream(stream):
            wmask, avg = ops.sample_others(sets[0]['labels'], dt, RATIO, 1)
            _, _, _, dz0, colsum0 = ops.fused_fwd(sets[0]['x'], sets[0]['w'], sets[0]['bias'], sets[0]['labels'], dt,
                                                  wmask, avg)
            dzs = [torch.empty_like(dz0).copy_(dz0) for _ in sets]
            stream.synchronize()

        def graphed(fn):
            """time fn(s) over the pool from a CUDA graph to exclude host launch gaps"""
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(stream):
                for s in sets:
                    fn(s)
                stream.synchronize()
                with torch.cuda.graph(g, stream=stream):
                    for s in sets:
                        fn(s)
                g.replay()
                stream.synchronize()
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                for _ in range(5):
                    g.replay()
                b_.record(stream)
                stream.synchronize()
            return a.elapsed_time(b_) / (5 * pool) * 1e3

        idx = {id(s): i for i, s in enumerate(sets)}
        try:
            if args.unfused:
                kernel_us['fc_cls_gemm'] = graphed(lambda s: ops.linear_fwd(s['x'], s['w'], s['bias'], out=s['logits']))
                kernel_us['group_ce'] = graphed(lambda s: ops.group_ce(s['logits'], s['labels'], dt, wmask, avg,
                                                                       dz_dtype=dtype))
            else:
                kernel_us['fused_fwd'] = graphed(lambda s: ops.fused_fwd(s['x'], s['w'], s['bias'], s['labels'], dt,
                                                                         wmask, avg))
            kernel_us['bwd_dW_db_only'] = graphed(lambda s: ops.fused_bwd(dzs[idx[id(s)]], s['x'], s['w'], gout, dt, None,
                                                                          need_dx=False, dW=s['dW'], db=s['db'],
                                                                          wscratch=s['wscratch']))
            kernel_us['bwd_dX_only'] = graphed(lambda s: ops.fused_bwd(dzs[idx[id(s)]], s['x'], s['w'], gout, dt, None,
                                                                       need_dw=False, need_db=False, dX=s['dX'],
                                                                       wscratch=s['wscratch2']))
            kernel_us['bwd_merged(prep+dW+dX)'] = graphed(lambda s: ops.fused_bwd(dzs[idx[id(s)]], s['x'], s['w'], gout, dt,
                                                                                  None, dW=s['dW'], dX=s['dX'],
                                                                                  wscratch=s['wscratch'], db=s['db']))
            kernel_us['sample_others'] = graphed(lambda s: ops.sample_others(s['labels'], dt, RATIO, 7))
        except Exception as ex:  # pragma: no cover
            log('per-kernel timing failed: %r' % (ex,))
        TF = dtype != torch.bfloat16
        flops = {'fc_cls_gemm': 2.0 * n * K_FEAT * C, 'fused_fwd': 2.0 * n * K_FEAT * C, 'bwd_dW_db_only': 2.0 * n * K_FEAT * C,
                 'bwd_dX_only': 2.0 * n * K_FEAT * C, 'bwd_merged(prep+dW+dX)': 4.0 * n * K_FEAT * C}
        bytes_ce = n * C * 4 + n * C * elt + n * 8 + dt.G * n   # read fp32 logits, write dz, labels, masks
        # Isolated kernel timings (a few hundred microseconds of launches at full clocks) are judged against the BURST
        # cuBLAS figure of MEASURED_PEAKS.json; the whole step, timed inside a seconds-long loop, against the SUSTAINED
        # one.  Both fractions are printed for every entry.
        tfac = 1.0 if dtype == torch.bfloat16 else 0.5
        pk_burst, pk_sust = pk['bf16_tflops'] * tfac, pk['bf16_tflops_sustained'] * tfac
        psrc = pk['source'] + (' cuBLAS bf16' if dtype == torch.bfloat16 else ' cuBLAS bf16 / 2 for tf32')
        roof_worst = None
        if kernel_us:
            def tensor_roof(name):
                ach = flops[name] / (kernel_us[name] * 1e-6) / 1e12
                return {'kernel': name, 'bound': 'tensor', 'achieved': ach, 'peak': pk_burst, 'unit': 'TFLOP/s',
                        'frac': ach / pk_burst, 'frac_of_sustained_peak': ach / pk_sust, 'peak_sustained': pk_sust,
                        'kernel_us': kernel_us[name], 'algorithmic_flops': flops[name],
                        'traffic': (ncu_traffic(name) if n == N_ROIS and not TF else None),
                        'peak_source': psrc + ' (burst: the kernel is timed alone)'}
            step_kernels = [k_ for k_ in ('fused_fwd', 'fc_cls_gemm', 'group_ce', 'bwd_merged(prep+dW+dX)') if k_ in kernel_us]
            dom = max(step_kernels, key=lambda k_: kernel_us[k_])
            if dom in flops:
                roof = tensor_roof(dom)
            else:
                ach = bytes_ce / (kernel_us[dom] * 1e-6) / 1e9
                roof = {'kernel': dom, 'bound': 'hbm', 'achieved': ach, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                        'frac': ach / pk['hbm_gbs'], 'traffic': ncu_traffic(dom), 'peak_source': pk['source'],
                        'algorithmic_bytes': bytes_ce}
            cands = [tensor_roof(k_) for k_ in step_kernels if k_ in flops]
            if cands:
                roof_worst = min(cands, key=lambda r_: r_['frac'])
        step_flops = 6.0 * n * K_FEAT * C
        ach_step = step_flops / (ms_step * 1e-3) / 1e12
        step_roof = {'bound': 'tensor', 'achieved': ach_step, 'peak': pk_sust, 'unit': 'TFLOP/s',
                     'frac': ach_step / pk_sust, 'frac_of_burst_peak': ach_step / pk_burst, 'peak_burst': pk_burst,
                     'algorithmic_flops_per_step': step_flops,
                     'peak_source': psrc + ' (sustained: the step is timed inside a long loop)'}
        lib_base = None
        if world == 1 and not args.no_library_baseline:
            try:
                lib_base = gpu_library_baseline(torch, tables, dev, n)
                lib_base['ours_over_library'] = lib_base['best_us'] / (ms_step * 1e3)
            except Exception as ex:  # pragma: no cover
                log('library baseline failed: %r' % (ex,))

    if rank == 0:
        cb = cpu_baseline(n) if world == 1 else None
        line = {
            'metric': METRIC, 'value': value, 'unit': 'RoIs/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
            'config': {
                'workload': 'BASELINE.json configs[1]: fused BAGS fwd+bwd, %d RoIs/GPU x %d feat x %d cls (%d logits), '
                            '5 bins, %s operands, dW+db+dX, device sampler, %s forward' % (n, K_FEAT, NUM_CLASSES, C, args.dtype,
                                                                                    'unfused' if args.unfused else 'fused'),
                'rois_per_gpu': n, 'parallelism': 'dp%d' % world,
                'l2': 'rotating pool of %d buffer sets (%.0f MB > 126 MB L2); no step re-reads cached inputs'
                      % (pool, pool * per_set / 1e6),
                'launch': 'cuda-graph replay' if graph is not None else 'eager',
                'collective': 'none' if world == 1 else (
                    ('bags_grad_allreduce (%s over NVLink peer memory, one kernel) of %d fp32 fc_cls grads per step'
                     % (sets[0]['bucket'].transport, C * K_FEAT + C)) if sets[0].get('bucket') is not None else
                    ('nccl all_reduce(avg) of %d fp32 fc_cls grads per step' % (C * K_FEAT + C))) + (
                    '; RELAXED schedule: each exchange runs on a side stream under the NEXT step and completes inside the timed region'
                    if comm_stream is not None else (
                        '; in-step with overlap: dW+db first, the exchange runs on a side stream under the dX GEMM and is '
                        'joined before the next forward starts' if split_bwd else
                        '; in-step: stream-ordered after the backward, complete before the next forward starts')),
                'exchange_check': exchange_check,
            },
            'clocks': clk,
            'e2e': e2e,
            'gpu_launches': kernels_per_step * args.steps,
            'roofline': roof,
            'roofline_worst': roof_worst,
            'roofline_step': step_roof,
            'gpu_library_baseline': lib_base,
            'kernel_us': kernel_us,
            'loss_bins': [float(v) for v in last['loss'].detach().float().cpu().tolist()],
        }
        if cb is not None:
            line['cpu_baseline'] = cb
        print(json.dumps(line), flush=True)
    if world > 1:
        # captured graphs hold NCCL kernels: drop them before leaving, and do not tear the communicator down
        # (ncclCommDestroy with live graph references can block) -- the process exits right after the barrier
        graph = None
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=None)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--rois', type=int, default=N_ROIS)
    ap.add_argument('--dtype', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--pool', type=int, default=0, help='number of rotating buffer sets (= steps per CUDA graph)')
    ap.add_argument('--fake-exchange', default='', help='probe (N = 1): blocks,threads,microseconds of a side-stream wait kernel per step')
    ap.add_argument('--exchange', default=None, choices=['instep', 'instep-overlap-dx', 'overlap-next-step'],
                    help='N > 1: gradient exchange inside the step, stream-ordered between the backward and the next '
                         "step's forward (default: what an SGD step needs -- the optimizer reads the reduced gradients "
                         'before the next forward reads W; mmdet/core/utils/dist_utils.py:51-58), or the relaxed schedule '
                         'on a side stream under the NEXT step (not a valid training schedule; kept for comparison)')
    ap.add_argument('--prep', default=None, choices=['bwd', 'fwd-zero', 'fwd-zero-colsum'],
                    help="where the backward's preparation runs: 'bwd' = jobs inside the backward kernel (zero dW, column sums); "
                         "'fwd-zero' = dW is zeroed by the forward kernel's idle epilogue warps; 'fwd-zero-colsum' = the "
                         'bias-gradient column sums come from the forward epilogue as well (no preparation left)')
    ap.add_argument('--dx-side', action='store_true',
                    help='instep-overlap-dx: fork the dX launch to the side stream and keep the exchange on the launching stream')
    ap.add_argument('--ar-blocks', type=int, default=0, help='N > 1: grid size limit of the peer-memory exchange kernel (0 = default)')
    ap.add_argument('--allreduce', default=os.environ.get('BAGS_ALLREDUCE', 'peer'), choices=['peer', 'nccl'],
                    help='N > 1: gradient exchange by the peer-memory kernel (default) or NCCL')
    ap.add_argument('--no-numa-pinned', dest='numa_pinned', action='store_false',
                    help='e2e leg: plain pin_memory() staging buffers instead of GPU-local NUMA placement')
    ap.add_argument('--e2e-copy-streams', type=int, default=1, help='e2e leg: copy streams the H2D of the features is split over')
    ap.add_argument('--e2e-eager-only', action='store_true', help='e2e leg: eager autograd calls only (no CUDA-graph step)')
    ap.add_argument('--unfused', action='store_true', help='GEMM -> fp32 logits -> grouped CE instead of the fused kernel')
    ap.add_argument('--no-library-baseline', action='store_true', help='skip the torch/cuBLAS same-GPU baseline leg')
    ap.add_argument('--profile', action='store_true', help='timed loop only (for ncu): skip e2e / cpu / per-kernel legs')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the per-bin losses, dW, db and dX of the last timed step to DIR/<name>.npy (float32)')
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        if args.dump_outputs:
            ap.error('--dump-outputs applies to --impl ours')
        args.steps = args.steps or 20
        args.warmup = 3 if args.warmup is None else args.warmup
        return run_reference(args)
    args.steps = args.steps or 600
    args.warmup = 20 if args.warmup is None else args.warmup
    if args.exchange is None:
        # N > 1: the exchange inside the step, overlapped by the dX contraction (the product's data-parallel schedule);
        # one GPU: the merged backward (nothing to exchange)
        args.exchange = 'instep-overlap-dx' if int(os.environ.get('WORLD_SIZE', '1')) > 1 else 'instep'
    if args.prep is None:
        # split schedule: the dW + db launch sits on the critical path before the exchange -> nothing left to prepare there
        args.prep = 'fwd-zero-colsum' if args.exchange == 'instep-overlap-dx' else 'fwd-zero'
    return run_ours(args)


if __name__ == '__main__':
    sys.exit(main())
