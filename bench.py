#!/usr/bin/env python
"""Benchmark of the hot path (contract: see the task statement / DESIGN.md "Measurement").

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): CIFAR-100 ResNet-110 (`resnet-110-fc`, the variant that emits
100-d embeddings), cosine loss against embeddings/cifar100.unitsphere (fixture copy), SGD momentum
0.9 + clipnorm 10 + L2, batch 128 per GPU, synthetic N(0,1) 32x32x3 images.  One step = forward +
backward + (all-reduce) + clip + SGD.  Weak scaling: the per-GPU batch is fixed.

Printed JSON (one line, rank 0): metric/value = images/s with the batch resident in HBM; e2e = the
same through Engine.train_step with pinned-host inputs (H2D inside the timed region) and a D2H read
of the loss every step; roofline = dominant training kernel class (per-op CUDA-event times from
se_run_ops_timed); retrieval = all-pairs distance N=50000, D=100 in Gpairs/s with its HBM roofline;
cpu_baseline = the float32 CPU restatement of the Keras reference (oracle/) timed on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ARCH = 'resnet-110-fc'
PER_GPU_BATCH = 128
METRIC = 'images/sec training ResNet-110 CIFAR-100 at 1/2/4/8 B200; retrieval Gpairs/s'
# the same string on both arms (native / --impl reference): the driver compares config.workload
WORKLOAD = ('CIFAR-100 ResNet-110 (%s) cosine loss vs cifar100.unitsphere, SGD momentum 0.9 + clipnorm 10 + L2 2e-4, '
            'batch %d/GPU, synthetic 32x32x3' % (ARCH, PER_GPU_BATCH))
# the other training configurations of BASELINE.json (extra lines: `--workload config3|config4`; the driver's default
# run is configs[1] above).  arch, class matrix, per-GPU batch, input size, classifier weight, description
WORKLOADS = {
    'config2': dict(arch=ARCH, emb='cifar100', batch=PER_GPU_BATCH, size=32, cls_weight=0.0, name=WORKLOAD),
    'config3': dict(arch='wrn-28-10', emb='cifar100', batch=64, size=32, cls_weight=0.1,
                    name='CIFAR-100 WRN-28-10 cosine + softmax combined loss (cls_weight 0.1), batch 64/GPU (512 on 8 GPUs), '
                         'synthetic 32x32x3'),
    'config4': dict(arch='resnet-50', emb='nab', batch=32, size=224, cls_weight=0.0,
                    name='NABirds-shape ResNet-50 224x224x3, nab.unitsphere head (555-d), batch 32/GPU (256 on 8 GPUs), synthetic'),
}


def traffic_lookup(kernel):
    """dram bytes per launch of a kernel class from the committed ncu --set full summaries (profiles/*_traffic.json)."""
    import glob
    best = None
    for fn in sorted(glob.glob(os.path.join(ROOT, 'profiles', '*_traffic.json'))):
        try:
            with open(fn) as f:
                d = json.load(f)
        except (OSError, ValueError):
            continue
        if kernel in d:
            best = d[kernel]['dram_bytes_per_launch']
    return best


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {'hbm_gbs': d['hbm_gbs'], 'tflops_burst': d['bf16_tflops'], 'tflops_sustained': d['bf16_tflops_sustained'],
                'source': 'measured (MEASURED_PEAKS.json)'}
    return {'hbm_gbs': 6650.0, 'tflops_burst': 1590.0, 'tflops_sustained': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_arm(steps, warmup, sample_batch=None, budget_s=150.0):
    """The reference's training step restated on the CPU (oracle/, float32, all host threads).  Keras/TF are
    not installable, so this is kind='port'.  Returns (images/s, ms per step, info)."""
    import torch
    from oracle import models as omodels
    from oracle import train as otrain
    emb = np.load(os.path.join(ROOT, 'tests', 'golden', 'class_matrices.npz'))['cifar100_embedding']
    # torch.distributed.run exports OMP_NUM_THREADS=1, and "every core" (128 on the B200 host) makes the tiny convs of
    # ResNet-110 ~400x slower through OpenMP oversubscription: probe a few thread counts with one small step each and
    # keep the fastest -- the number reported as `cores`.
    ncpu = max(1, os.cpu_count() or 1)
    om = omodels.build_network(100, ARCH, input_channels=3, seed=0)
    otrain.cast_model(om, torch.float32)
    vel = otrain.make_velocity(om)
    emb_t = torch.as_tensor(emb.astype(np.float32))
    g = torch.Generator().manual_seed(1000)
    B = sample_batch or PER_GPU_BATCH

    def one(bsz):
        x = torch.randn(bsz, 32, 32, 3, generator=g)
        y = torch.randint(0, 100, (bsz,), generator=g)
        t0 = time.perf_counter()
        otrain.train_step(om, x, y, emb_t, vel, 0.1)
        return time.perf_counter() - t0

    best_t, cores = None, 1
    for nthr in sorted({1, min(8, ncpu), min(32, ncpu), min(64, ncpu)}):
        torch.set_num_threads(nthr)
        one(16)
        t = one(16)
        if best_t is None or t < best_t:
            best_t, cores = t, nthr
    torch.set_num_threads(cores)

    t_first = one(B)                                    # also the first warm-up step
    # keep the whole run inside the budget: shrink the per-step sample if a full batch is too slow
    total_steps = steps + max(warmup - 1, 0)
    if sample_batch is None and t_first * total_steps > budget_s:
        B = max(8, int(PER_GPU_BATCH * budget_s / (t_first * total_steps)) // 8 * 8)
    for _ in range(max(warmup - 1, 0)):
        one(B)
    ts = [one(B) for _ in range(steps)]
    ms = 1000.0 * float(np.mean(ts))
    return B / (ms / 1000.0), ms, {'cores': cores, 'sample_batch': B}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    ips, ms, info = cpu_reference_arm(args.steps, args.warmup)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': ips, 'unit': 'images/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'per_step_images': info['sample_batch']},
        'cpu_baseline': {'value': ips, 'unit': 'images/s', 'cores': info['cores'], 'kind': 'port',
                         'sample': '%d steps of %d images (float32 torch-CPU restatement of the Keras reference; '
                                   'Keras/TF not installable)' % (args.steps, info['sample_batch'])},
        'e2e': {'value': ips, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- GPU arm
def tc_coverage(graph, batch, mode, L):
    """How many convolutions of the network run on the tcgen05 kernels in `mode`, per direction (se_conv2d_path: the
    library's own host-side planning).  Never raises: a reporting extra must not break the bench."""
    try:
        lib = L.load()
        n, cnt = 0, [0, 0, 0]
        for node in graph.nodes:
            if node.op != 'conv':
                continue
            h, w, cin = node.inputs[0].shape
            ho, wo, cout = node.output.shape
            a = node.attrs
            d = L.ConvDesc(batch, h, w, cin, cout, a['k'], a['k'], a['stride'], a['pad_t'], a['pad_l'], ho, wo)
            n += 1
            for k in range(3):
                cnt[k] += 1 if lib.se_conv2d_path(d, mode, k) == 1 else 0
        return {'convolutions': n, 'forward': cnt[0], 'backward_data': cnt[1], 'weight_gradient': cnt[2]}
    except Exception as e:                                   # pragma: no cover
        return {'error': repr(e)}


def op_category(op, L):
    i = op.i
    names = {L.OP_CONV_FWD: 'conv_fwd', L.OP_CONV_DGRAD: 'conv_dgrad', L.OP_CONV_WGRAD: 'conv_wgrad',
             L.OP_CONV_BN_FWD: 'conv_bn_fwd'}
    if op.opcode in names:
        key = '%s %dx%d s%d %d->%d @%dx%d' % (names[op.opcode], i[5], i[6], i[7], i[3], i[4], i[1], i[2])
        flops = 2.0 * i[0] * i[10] * i[11] * i[4] * i[5] * i[6] * i[3]
        # algorithmic bytes of one launch: the input tensor, the output tensor and the filter, each once (fp32)
        byts = 4.0 * (i[0] * i[1] * i[2] * i[3] + i[0] * i[10] * i[11] * i[4] + i[5] * i[6] * i[3] * i[4])
        return key, flops, byts
    bn = {L.OP_BN_STATS: ('bn_stats', 1), L.OP_BN_FWD_TRAIN: ('bn_fwd', 2), L.OP_BN_BWD: ('bn_bwd', 7)}
    if op.opcode in bn:
        nm, passes = bn[op.opcode]
        return '%s C=%d rows=%d' % (nm, i[0], i[1]), 0.0, 4.0 * i[0] * i[1] * passes
    other = {L.OP_HEAD: 'embed_head', L.OP_SGD_PREPARE: 'sgd_prepare', L.OP_SGD_APPLY: 'sgd_apply', L.OP_MEMSET: 'memset',
             L.OP_GAP_FWD: 'gap_fwd', L.OP_GAP_BWD: 'gap_bwd', L.OP_SHORTCUT_BWD: 'shortcut_bwd', L.OP_ADD_BWD: 'add_bwd',
             L.OP_ADD_FWD: 'add_fwd', L.OP_XENT: 'softmax_xent', L.OP_TRANSPOSE_FILTERS: 'split_filters',
             L.OP_MAXPOOL_FWD: 'maxpool_fwd', L.OP_MAXPOOL_BWD: 'maxpool_bwd', L.OP_AVGPOOL_FWD: 'avgpool_fwd',
             L.OP_AVGPOOL_BWD: 'avgpool_bwd', L.OP_ALLREDUCE: 'allreduce'}
    return other.get(op.opcode, 'op%d' % op.opcode), 0.0, 0.0


def profile_step(eng, L, pk):
    """Per-op device times of one training step (eager, CUDA-event pair per op) -> dominant kernel class."""
    import ctypes
    arr = eng.plans['step']
    n = len(arr)
    ms = (ctypes.c_float * n)()
    for _ in range(2):
        L.check(eng.lib.se_run_ops_timed(arr, n, eng.mode, L.stream_ptr(), ms), 'se_run_ops_timed')
    cats = {}
    for k in range(n):
        key, flops, byts = op_category(arr[k], L)
        c = cats.setdefault(key, {'ms': 0.0, 'n': 0, 'flops': flops, 'bytes': byts})
        c['ms'] += ms[k]
        c['n'] += 1
    total = sum(c['ms'] for c in cats.values())
    top = sorted(cats.items(), key=lambda kv: -kv[1]['ms'])
    name, c = top[0]
    avg_s = c['ms'] / c['n'] / 1000.0
    # a convolution is bounded by whichever takes longer at the measured peaks: its flops on the tensor cores (TF32 =
    # half the dense bf16 rate) or its algorithmic bytes on HBM; the 16..64-channel layers of ResNet-110 (36 flop/byte
    # and less) are on the HBM side of the machine balance (~100 flop/byte)
    tf32_peak = pk['tflops_sustained'] / 2.0
    if c['flops'] > 0 and c['flops'] / (tf32_peak * 1e12) > c['bytes'] / (pk['hbm_gbs'] * 1e9):
        achieved = c['flops'] / avg_s / 1e12
        roof = {'bound': 'tensor', 'kernel': name, 'achieved': achieved, 'peak': tf32_peak, 'unit': 'TFLOP/s',
                'frac': achieved / tf32_peak, 'traffic': None}
    else:
        achieved = c['bytes'] / avg_s / 1e9 if c['bytes'] else 0.0
        roof = {'bound': 'hbm', 'kernel': name, 'achieved': achieved, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                'frac': achieved / pk['hbm_gbs'], 'traffic': None}
    roof['traffic'] = traffic_lookup(name)
    roof.update({'avg_launch_us': 1e6 * avg_s, 'launches_per_step': c['n'], 'share_of_step': c['ms'] / total,
                 'peak_source': pk['source'] + (', sustained bf16 / 2 (TF32)' if roof['bound'] == 'tensor' else ''),
                 'algorithmic_bytes_per_launch': c['bytes'], 'algorithmic_flops_per_launch': c['flops']})
    breakdown = [{'kernel': k, 'ms_per_step': v['ms'], 'launches': v['n'], 'share': v['ms'] / total} for k, v in top[:40]]
    conv_flops = sum(v['flops'] * v['n'] for v in cats.values())
    return roof, breakdown, total, conv_flops


def bench_retrieval(L, rank, world, dev, n, d, reps, mode, pk_hbm=6567.4):
    """All-pairs distance (evaluate_retrieval.py:56-63), rows sharded over ranks, no exchange step."""
    import torch
    from semantic_embeddings_b200.evaluate_retrieval import pairwise_distances
    rng = np.random.RandomState(0)
    f = rng.randn(n, d).astype(np.float32)
    f /= np.linalg.norm(f, axis=-1, keepdims=True)
    fd = torch.from_numpy(f).to(dev)
    rows = (n + world - 1) // world
    r0 = rank * rows
    rows = max(0, min(rows, n - r0))
    out = torch.empty((rows, n), dtype=torch.float32, device=dev)
    for _ in range(2):
        pairwise_distances(None, False, r0, rows, mode, out=out, feat_dev=fd)
    torch.cuda.synchronize(dev)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        a.record()
        pairwise_distances(None, False, r0, rows, mode, out=out, feat_dev=fd)
        b.record()
    torch.cuda.synchronize(dev)
    ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    chk = float(out[0, :8].sum().item())
    # ranking step (evaluate_retrieval.py:67 restricted to the clip_ahp+1 = 251 ranks the metrics read): se_row_topk
    rank_ms = None
    if rows > 0 and n <= 52000:
        from semantic_embeddings_b200.evaluate_retrieval import row_topk
        k = min(251, n)
        for _ in range(2):
            row_topk(out, k)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            row_topk(out, k)
        b.record()
        torch.cuda.synchronize(dev)
        rank_ms = a.elapsed_time(b) / 3.0
    extra = {}
    if rows > 0 and world == 1 and n <= 52000:
        from semantic_embeddings_b200.evaluate_retrieval import pairwise_topk, row_argsort
        from semantic_embeddings_b200.class_hierarchy import hierarchical_metrics
        k = min(251, n)
        # fused distance + top-251 (se_pairwise_topk): no N x N matrix
        pairwise_topk(k=k, feat_dev=fd)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            _, _, fused = pairwise_topk(k=k, feat_dev=fd)
        b.record()
        torch.cuda.synchronize(dev)
        extra['fused_topk'] = {'ms': a.elapsed_time(b) / 3.0, 'k': k, 'fused': bool(fused),
                               'gpairs_per_s': float(n) * n / (a.elapsed_time(b) / 3.0 / 1000.0) / 1e9,
                               'kernels': 'pairwise_tc_kernel<2> on a 4096-column sample (per-row thresholds in its epilogue), '
                                          'pairwise_tc_kernel<1> (candidate sweep, nothing else written), '
                                          'pairwise_topk_finish_kernel (per-row candidate sort)',
                               'note': 'includes the status read-back; the matrix-write bound of the unfused kernel at this '
                                       'size is %.2f ms' % (4.0 * n * n / pk_hbm / 1e6)}
        # full-length ranking (se_row_argsort) and P@k / AHP / AP (se_hier_metrics) for a block of 2048 query rows
        blk = min(2048, rows)
        sub = out[:blk]
        row_argsort(sub)
        a.record()
        idx = row_argsort(sub)
        b.record()
        torch.cuda.synchronize(dev)
        extra['ranking_full'] = {'rows': blk, 'ms': a.elapsed_time(b), 'ms_all_rows_extrapolated': a.elapsed_time(b) * n / blk,
                                 'kernel': 'row_argsort_kernel (bitonic network, shared-memory sub-sorts)'}
        labels = rng.randint(0, 100, n).astype(np.int32)
        hier = np.load(os.path.join(ROOT, 'tests', 'golden', 'retrieval_ref.npz'))
        t0 = time.perf_counter()
        hierarchical_metrics(idx, np.arange(blk), labels, hier['wup_lut'], hier['lcs_height_lut'], 250, -1, True)
        torch.cuda.synchronize(dev)
        extra['metrics_full'] = {'rows': blk, 'wall_ms_incl_host_setup': 1000.0 * (time.perf_counter() - t0),
                                 'kernel': 'hier_metrics_kernel (P@1..250, unclipped AHP, AP from full rankings)'}
    return ms, rows, chk, rank_ms, extra


def run_native(args):
    import torch
    import torch.distributed as dist
    from semantic_embeddings_b200 import _lib as L
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.engine import Engine

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d (launch N>1 with torch.distributed.run)' % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # stdout carries the single JSON line: NCCL's own log (the version banner at any NCCL_DEBUG level, INFO lines)
        # goes to stderr instead
        if os.environ.get('NCCL_DEBUG', '').upper() in ('VERSION', 'WARN'):
            os.environ.pop('NCCL_DEBUG')
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        dist.init_process_group('nccl', device_id=dev)
    L.load()
    pk = peaks()
    mode = {'tf32x3': L.SE_MODE_TF32X3, 'tf32': L.SE_MODE_TF32, 'f32': L.SE_MODE_F32}[args.mode]
    caps = L.load().se_tc_capabilities()
    wl = WORKLOADS[args.workload]
    emb = np.load(os.path.join(ROOT, 'tests', 'golden', 'class_matrices.npz'))[wl['emb'] + '_embedding']
    ncls, size = emb.shape[0], wl['size']
    batch = args.batch if args.batch else wl['batch']
    # weak scaling (default): the per-GPU batch is the config's; strong scaling: that many images in total
    B = batch if args.scaling == 'weak' else max(1, batch // world)
    graph = utils.build_network(emb.shape[1], wl['arch'], input_channels=3)
    eng = Engine(graph, B, emb, mode=mode, device=str(dev), world_size=world, use_cuda_graph=not args.no_graph,
                 comm=args.comm, cls_weight=wl['cls_weight'], num_classes=ncls)
    eng.set_lr(0.1)
    restore_initial_state = None
    if args.dump_outputs:
        # Training from the random initialisation is chaotic: the ordering differences of atomically accumulated sums
        # (~1e-7) grow ~100x per step, so after a few steps two runs of the same build differ by ~1e-2.  The dumped
        # step therefore starts from the seeded initial state (a ~15 MB device copy inside the timed window), which makes
        # its outputs a function of the arguments alone.
        state = (eng.P, eng.V, eng.S, eng.lr_dev)
        initial = [t.clone() for t in state]

        def restore_initial_state():
            for t, t0 in zip(state, initial):
                t.copy_(t0)

    # synthetic data: N(0,1) images, seed 1000+rank (SURVEY.md section 8d); a small pool cycled through
    gen = torch.Generator().manual_seed(1000 + rank)
    pool = 4
    xs_host = [torch.randn(B, size, size, 3, generator=gen).pin_memory() for _ in range(pool)]
    ys_host = [torch.randint(0, ncls, (B,), generator=gen, dtype=torch.int32).pin_memory() for _ in range(pool)]
    xs_dev = [x.to(dev) for x in xs_host]
    ys_dev = [y.to(dev) for y in ys_host]

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(loader, steps, read_loss, before_last=None):
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        last, pending = None, None
        for s in range(steps):
            if s == steps - 1 and before_last is not None:
                before_last()
            loader(s)
            eng.train_step()
            if read_loss:
                # every step's loss / accuracy is read back (pinned D2H); the host consumes step s-1 while step s runs
                h = eng.metrics_async()
                if pending is not None:
                    last = eng.metrics_result(pending)['loss']
                pending = h
        if pending is not None:
            last = eng.metrics_result(pending)['loss']
        t1.record()
        torch.cuda.synchronize(dev)
        ms = t0.elapsed_time(t1)
        barrier()
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, last

    resident = lambda s: eng.load_batch(xs_dev[s % pool], ys_dev[s % pool])
    from_host = lambda s: eng.load_batch(xs_host[s % pool], ys_host[s % pool])

    launches_per_step = eng.launches_per_step()
    if world > 1:
        from semantic_embeddings_b200.parallel import broadcast_parameters
        broadcast_parameters([eng.P, eng.S, eng.V])        # replicas start the timed region from identical weights
    timed(resident, args.warmup, False)                      # warm-up (also captures the CUDA graphs)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_res, _ = timed(resident, args.steps, False, restore_initial_state)
    # the headline path's last step, read before the end-to-end pass trains on
    outputs = step_outputs(eng) if (args.dump_outputs and rank == 0) else None
    ms_e2e, last_loss = timed(from_host, args.steps, True)
    clocks = sampler.stop() if rank == 0 else None

    gb = B * world
    value = gb * args.steps / (ms_res / 1000.0)
    e2e = gb * args.steps / (ms_e2e / 1000.0)

    roof, breakdown, prof_total, conv_flops = (None, None, None, None)
    if rank == 0:
        roof, breakdown, prof_total, conv_flops = profile_step(eng, L, pk)

    retrieval = None
    if not args.skip_retrieval and args.workload == 'config2':
        n, d = args.retrieval_n, 100
        ms_r, rows, chk, rank_ms, r_extra = bench_retrieval(L, rank, world, dev, n, d, 5, mode, pk['hbm_gbs'])
        if world > 1:
            t = torch.tensor([ms_r], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_r = float(t.item())
        pairs = float(n) * n
        gpairs = pairs / (ms_r / 1000.0) / 1e9
        per_gpu_bytes = 4.0 * rows * n + 4.0 * n * d        # algorithmic: write the row block once, read F once
        ach = per_gpu_bytes / (ms_r / 1000.0) / 1e9
        retrieval = {'value': gpairs, 'unit': 'Gpairs/s', 'N': n, 'D': d, 'ms': ms_r, 'rows_per_gpu': rows,
                     'roofline': {'bound': 'hbm', 'kernel': 'pairwise_dist', 'achieved': ach, 'peak': pk['hbm_gbs'],
                                  'unit': 'GB/s', 'frac': ach / pk['hbm_gbs'],
                                  'traffic': traffic_lookup('pairwise_dist') if (n == 50000 and world == 1) else None,
                                  'algorithmic_bytes_per_launch': per_gpu_bytes, 'peak_source': pk['source']},
                     'arithmetic': 'tcgen05 kind::f16, split-fp16 x3 (fp32-level accuracy)' if (mode != L.SE_MODE_F32 and caps & 8) else 'fp32 FFMA'}
        retrieval.update(r_extra)
        if rank_ms is not None:
            # per-row top-251 of this rank's row block; bound: one read of the block (4 bytes per pair)
            retrieval['ranking_top251'] = {'ms': rank_ms, 'gpairs_per_s': float(rows) * n / (rank_ms / 1000.0) / 1e9,
                                           'hbm_frac': 4.0 * rows * n / (rank_ms / 1000.0) / 1e9 / pk['hbm_gbs'],
                                           'kernel': 'row_topk_kernel (radix select + bitonic sort in shared memory)'}

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu_baseline and args.workload == 'config2':
        ips, ms_cpu, info = cpu_reference_arm(steps=3, warmup=1, budget_s=25.0)
        cpu = {'value': ips, 'unit': 'images/s', 'cores': info['cores'], 'kind': 'port',
               'sample': '3 timed steps of %d images after 1 warm-up (float32 torch-CPU restatement of the Keras '
                         'reference training step; Keras/TF not installable)' % info['sample_batch']}

    if rank == 0:
        conv_train_flops_per_img = 3 * 2 * graph.conv_macs_per_image()
        tc = bool(mode != L.SE_MODE_F32 and (caps & 7))
        line = {
            'metric': METRIC, 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_res / args.steps, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
            'dtype': (args.mode if tc else 'f32'), 'data': 'synthetic',
            'config': {'workload': wl['name'] if (args.workload != 'config2' or B != PER_GPU_BATCH) else WORKLOAD, 'per_gpu_batch': B, 'global_batch': gb, 'parallelism': 'dp%d' % world,
                       'arith_mode': args.mode, 'tc_capabilities': caps, 'tcgen05_layers': tc_coverage(eng.g, B, mode, L),
                       'cuda_graph': not args.no_graph,
                       'gradient_exchange': ('none' if world == 1 else
                                             ('NCCL inside the library: %d bucketed all-reduces overlapped with the backward '
                                              'pass, captured in the step graph' % eng.grad_buckets) if eng.comm_native
                                             else 'torch.distributed all_reduce of the flat buffer between two graphs'),
                       'l2_policy': 'activations+gradients touched per step (~%.1f GB) exceed the 126 MB L2; '
                                    'retrieval output 10 GB' % (eng_bytes(eng) / 1e9)},
            'e2e': {'value': e2e, 'unit': 'images/s', 'ms_per_step': ms_e2e / args.steps,
                    'h2d_bytes_per_step': int(xs_host[0].numel() * 4 + ys_host[0].numel() * 4),
                    'd2h_bytes_per_step': int(B * 8), 'last_loss': last_loss},
            'gpu_launches': int(launches_per_step * args.steps),
            'launches_per_step': int(launches_per_step),
            'roofline': roof, 'breakdown': breakdown,
            'conv_flop_roofline': {'train_gflop_per_image': conv_train_flops_per_img / 1e9,
                                   'achieved_tflops': value * conv_train_flops_per_img / 1e12 / world,
                                   'frac_of_bf16_sustained_peak': value * conv_train_flops_per_img / 1e12 / world / pk['tflops_sustained']},
            'retrieval': retrieval, 'cpu_baseline': cpu, 'clocks': clocks, 'peaks': pk,
        }
        print(json.dumps(line))
    if outputs is not None:
        dump_outputs(outputs, args.dump_outputs)
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_ELEMENTS = 4 << 20          # per array; a larger one is written as a fixed, seeded sample of this many elements


def step_outputs(eng):
    """What a caller of Engine.train_step receives after the step: per-sample loss / accuracy (and classifier loss /
    accuracy), the embeddings (and class probabilities), gradient norm and L2 term, and the updated weights (BatchNorm
    moving statistics included) and momentum buffers, each concatenated in weight-name order."""
    out = {k: np.asarray(v, np.float32) for k, v in eng.per_sample_metrics().items()}
    out['embeddings'] = eng.act[eng.head_node.output.name].cpu().numpy()
    if eng.xent_node is not None:
        out['class_probabilities'] = eng.act[eng.xent_node.output.name].cpu().numpy()
    out['grad_norm_and_l2'] = np.array(eng.grad_norm_and_reg(), np.float64)
    for name, d in (('weights', eng.get_weights()), ('velocity', eng.get_velocity())):
        out[name] = np.concatenate([d[k].ravel() for k in sorted(d)])
    return out


def dump_outputs(outputs, out_dir):
    """DIR/<name>.npy per array; arrays above DUMP_MAX_ELEMENTS are flattened and sampled at indices that depend only on
    their length, so that two builds given the same arguments write comparable files."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        if a.size > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.RandomState(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))
            a = a.ravel()[idx]
        np.save(os.path.join(out_dir, name + '.npy'), a)


def eng_bytes(eng):
    tot = 0
    for d in (eng.act, eng.grad):
        for t in d.values():
            tot += t.numel() * 4
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    # tf32x3 = tcgen05 tiles with error compensation (meets the 1e-4 parity gate; the mode the training CLI runs);
    # tf32 = single-pass (outside the gate, for comparison only); f32 = fp32 FFMA kernels
    ap.add_argument('--mode', default='tf32x3', choices=['tf32x3', 'tf32', 'f32'])
    ap.add_argument('--batch', type=int, default=0, help='per-GPU batch (default: the workload\'s)')
    ap.add_argument('--workload', default='config2', choices=sorted(WORKLOADS),
                    help='BASELINE.json training configuration; the driver contract is config2 (ResNet-110, batch 128)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: --batch images per GPU (the driver contract); strong: --batch images in total')
    ap.add_argument('--comm', default='torch', choices=['auto', 'native', 'torch'],
                    help='gradient exchange: torch.distributed all_reduce (default) or the library\'s NCCL-in-graph path')
    ap.add_argument('--retrieval-n', type=int, default=50000)
    ap.add_argument('--skip-retrieval', action='store_true')
    ap.add_argument('--skip-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed training step computed as DIR/<name>.npy (float32 / float64); that '
                         'step starts from the seeded initial weights, so the files depend on the arguments alone')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_native(args)


if __name__ == '__main__':
    main()
