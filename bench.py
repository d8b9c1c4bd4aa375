#!/usr/bin/env python
"""Benchmark of the RegTR correspondence-prediction hot path (BASELINE.json metric:
pairs/sec on 3DMatch-size clouds).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--pairs B] [--config C]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path (pyramid -> KPConv encoder -> cross-encoder -> regressor ->
Kabsch) over one batch of B synthetic 3DMatch-shaped pairs per GPU.  Default workload: BASELINE
config 2 (one ~20k-point pair, batch 1, 1 GPU).  N>1 (torchrun): every rank runs its own pairs
(weak scaling, no data-path collective) and the poses are all-gathered once per step.

Prints ONE JSON line on rank 0 (see the keys in `main`).  Timing: CUDA events per step on the
launching stream, W >= 3 warm-up steps, L2 flushed between timed steps, max over ranks.

--dump-outputs DIR writes the output dict of the last timed step (rank 0's pairs) as DIR/<name>.npy.  The
inputs and weights come from fixed seeds, so two builds run with the same arguments can be compared output by
output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WEIGHT_SEED = 2024
POOL = 8          # distinct synthetic pairs rotated through the steps
DUMP_BYTES = 64 * 10 ** 6     # --dump-outputs writes at most this much
# the reference's output dict; per-cloud entries are lists (one tensor per pair) with the points on this axis
OUTPUT_KEYS = ('src_feat_un', 'tgt_feat_un', 'src_feat', 'tgt_feat', 'src_kp', 'tgt_kp', 'src_kp_warped',
               'tgt_kp_warped', 'src_overlap', 'tgt_overlap', 'pose')
POINT_AXIS = {'feat_un': 0, 'kp': 0, 'feat': 1, 'kp_warped': 1, 'overlap': 1}
_T0 = time.time()


def log(msg):
    if int(os.environ.get('RANK', 0)) == 0:
        print(f'[bench {time.time() - _T0:7.1f}s] {msg}', file=sys.stderr, flush=True)


def cpu_threads():
    """Threads for the CPU legs: all host cores up to 32 (beyond that the ATen ops of this workload,
    ~1 ms each, slow down from fork/join overhead); reported as `cores`."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get('REGTR_CPU_THREADS', 32))))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', type=int, default=2, help='BASELINE.json config id (2..5)')
    ap.add_argument('--pairs', type=int, default=None, help='pairs per GPU per step (default: from config)')
    ap.add_argument('--cpu-baseline', type=int, default=1, help='time the CPU port beside the GPU run (N=1 only)')
    ap.add_argument('--checks', type=int, default=1, help='report pose error vs the oracle on one pair')
    ap.add_argument('--attention', default='fp32', choices=['fp32', 'tf32_tc', 'bf16_tc'],
                    help="fp32: parity kernel (default, pose within 1e-4); bf16_tc: tcgen05 tensor-core core")
    ap.add_argument('--inflight', type=int, default=10,
                    help='independent pairs in flight per GPU (CUDA-graph executors on private streams); 1 = serial')
    ap.add_argument('--graph', type=int, default=1, help='1: CUDA-graph executor (GraphedRegTR); 0: eager forward')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB)')
    return ap.parse_args()


def pairs_per_gpu(args):
    if args.pairs:
        return args.pairs
    return {2: 1, 3: 8, 4: 8, 5: 4}.get(args.config, 1)


def workload_name(args, B):
    n_pts = '~30k' if args.config == 5 else '~20k'
    return f'BASELINE config {args.config}: synthetic 3DMatch-like pairs, {n_pts} pts/cloud, {B} pair(s)/GPU/step'


def make_pool(config_id, n, first=0):
    from regtr_b200.synthetic import make_batch
    cid = 2 if config_id in (2, 3, 4) else config_id
    b = make_batch(cid, n, first_pair=first)
    return list(zip(b['src_xyz'], b['tgt_xyz']))


# ------------------------------------------------------------------------------ clocks

class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                                          '-i', str(index), '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self):
        """Start of the window whose samples are reported (the timed region)."""
        self.t0 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        t0 = getattr(self, 't0', 0.0)
        rows = [r for t, r in self.rows if t >= t0] or [r for _, r in self.rows[-3:]]
        for r in rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


def dump_outputs(out, folder):
    """Write one forward's output dict as <folder>/<name>.npy: per-cloud entries as <key>_<pair>, floating point as
    float32 (anything else as float64).  Above DUMP_BYTES the per-cloud arrays keep a seeded sample of their points,
    the same rows for every array of a cloud, written beside them as <side>_sample_rows_<pair>.  Returns
    (bytes written, whether the points were sampled)."""
    items = []                                  # (file name, (side, pair) or None, points axis, tensor)
    for key in OUTPUT_KEYS:
        val = out[key]
        if torch.is_tensor(val):
            items.append((key, None, None, val))
        else:
            side, kind = key.split('_', 1)
            items += [(f'{key}_{b}', (side, b), POINT_AXIS[kind], t) for b, t in enumerate(val)]
    arrays = {}
    for name, _, _, t in items:
        t = t.detach().cpu()
        arrays[name] = (t.float() if t.is_floating_point() else t.double()).numpy()
    total = sum(a.nbytes for a in arrays.values())
    fixed = sum(arrays[name].nbytes for name, cloud, _, _ in items if cloud is None)
    rows = {}
    if total > DUMP_BYTES:
        keep = 0.99 * (DUMP_BYTES - fixed) / (total - fixed)     # 1 %: room for the row lists
        for name, cloud, axis, _ in items:
            if cloud is None:
                continue
            if cloud not in rows:
                n = arrays[name].shape[axis]
                rng = np.random.default_rng([('src', 'tgt').index(cloud[0]), cloud[1]])
                rows[cloud] = np.sort(rng.choice(n, size=min(n, max(1, int(n * keep))), replace=False))
            arrays[name] = np.take(arrays[name], rows[cloud], axis=axis)
        for (side, b), r in rows.items():
            arrays[f'{side}_sample_rows_{b}'] = r.astype(np.float64)
    os.makedirs(folder, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(folder, name + '.npy'), np.ascontiguousarray(a))
    return sum(a.nbytes for a in arrays.values()), bool(rows)


# ------------------------------------------------------------------------- CPU baseline

def cpu_forward_fn(cfg, sd):
    """The reference's CPU path, restated: its own C++ pre-processing core when oracle/_ref is
    built (kind 'port' either way: the PyTorch modules are the oracle's restatement)."""
    from oracle import pre, regtr_oracle
    ref = pre.RefCpp() if pre.RefCpp.available() else None

    def run(src, tgt):
        with torch.no_grad():
            if ref is not None:
                meta = pre.preprocess_refcpp(cfg, [src, tgt], ref)
            else:
                meta = pre.preprocess(cfg, [src, tgt])
            return regtr_oracle.forward(sd, cfg, [src], [tgt], meta=meta)
    return run, ('reference C++ core (oracle/_ref: nanoflann + grid_subsampling)' if ref is not None
                 else 'oracle C restatement (brute-force first-K)')


def time_cpu(cfg, sd, pool, n_pairs, warm=1):
    cores = cpu_threads()
    torch.set_num_threads(cores)
    run, pre_kind = cpu_forward_fn(cfg, sd)
    for i in range(warm):
        run(*pool[i % len(pool)])
    ts = []
    for i in range(n_pairs):
        t0 = time.perf_counter()
        run(*pool[i % len(pool)])
        ts.append(time.perf_counter() - t0)
    return dict(value=1.0 / statistics.median(ts), unit='pairs/s', cores=cores, kind='port',
                sample=f'{n_pairs} pair(s) of the same workload, median; 1 warm-up; pre-processing = {pre_kind}; '
                       f'torch CPU fp32 with {cores} threads'), ts


# ------------------------------------------------------------------------------- main

def kpconv_algorithmic_bytes(info):
    """SURVEY.md 8d: bytes = Nq*K*4 + nnz*(12 + Cin*4) + Nq*12 + Nq*Cout*4 + 15*Cin*Cout*4 (fp32)."""
    nnz = int((info['idx'] < info['Ns']).sum().item())
    Nq, K, Cin, Cout = info['Nq'], info['K'], info['Cin'], info['Cout']
    return Nq * K * 4 + nnz * (12 + Cin * 4) + Nq * 12 + Nq * Cout * 4 + 15 * Cin * Cout * 4


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores."""
    if rank != 0:
        return
    from regtr_b200.config import get_config
    from regtr_b200.weights import random_state_dict
    cfg = get_config('3dmatch')
    sd = random_state_dict(cfg, WEIGHT_SEED)
    B = pairs_per_gpu(args)
    pool = make_pool(args.config, min(POOL, max(2, args.steps)))
    run, pre_kind = cpu_forward_fn(cfg, sd)
    cores = cpu_threads()
    torch.set_num_threads(cores)
    log(f'reference arm: {cores} threads of {os.cpu_count()} cores')
    for i in range(max(args.warmup, 1)):
        run(*pool[i % len(pool)])
    # each step = a bounded sample of the workload: ONE pair (the workload has B*N pairs/step).  All --steps steps
    # run; REGTR_REF_BUDGET_S=<seconds> opts in to stopping early (after >= 3 steps) once that much time has passed,
    # and `executed_steps` then reports how many ran
    budget = float(os.environ.get('REGTR_REF_BUDGET_S', 'inf'))
    t0 = time.perf_counter()
    done = 0
    for i in range(args.steps):
        last = run(*pool[i % len(pool)])
        done += 1
        if done >= 3 and time.perf_counter() - t0 > budget:
            break
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        log('outputs of the last step: %d bytes, points sampled: %s' % dump_outputs(last, args.dump_outputs))
    v = done / dt
    line = dict(metric='pairs/sec on 3DMatch-size clouds (~20k pts); pose err vs ref', value=v, unit='pairs/s',
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=1000 * dt / done,
                higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic',
                impl='reference', executed_steps=done,
                config=dict(workload=workload_name(args, B), sample='1 pair per step (bounded sample)'),
                cpu_baseline=dict(value=v, unit='pairs/s', cores=cores, kind='port',
                                  sample=f'{done} steps x 1 pair; pre-processing = {pre_kind}'),
                e2e=dict(value=v, unit='pairs/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line), flush=True)


def peak_table():
    """Roofline denominators: measured (MEASURED_PEAKS.json, driver-written) or the profiling guide's fallback."""
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        d = json.load(open(path))
        return dict(hbm_gbs=float(d['hbm_gbs']), bf16_tflops=float(d['bf16_tflops']),
                    bf16_tflops_sustained=float(d.get('bf16_tflops_sustained', d['bf16_tflops'])),
                    source='measured (MEASURED_PEAKS.json)')
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0,
                    source='fallback (B200_PROFILING.md: 6.65 TB/s, 1.59 PFLOP/s)')


def ncu_traffic(kernel_key, pairs):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel family (for `whole_forward`: per replay),
    read at run time from the committed ncu summary (profiles/r02_ncu_traffic.json, written by
    scripts/ncu_summary.py from one `ncu --set full` capture of a graph replay of this workload at the same number of
    pairs per forward); None when no capture at this batch size is committed.  kpconv_gather: the aggregation kernels
    only -- the [Nq, 15 Cin] intermediate they write is read back by the contraction GEMM, which the capture lists
    under gemm_tf32x3."""
    try:
        d = json.load(open(os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')))
        return d[str(pairs)][kernel_key]['dram_bytes_per_launch']
    except Exception:
        return None


def measure_stages(model, batch_at, resident, flush, W, B, reps=20):
    """Per-stage GPU time at the reference's `_TIMEIT` boundaries (regtr.py:108-216: preprocess | encoder |
    attention + decoder | pose) from CUDA events between four back-to-back graph replays of ONE serial forward
    (GraphedRegTR(stages=True)), L2 flushed before each forward, plus the single-stream latency of the
    one-graph executor.  Median over `reps` forwards."""
    from regtr_b200.regtr import GraphedRegTR
    staged, single = GraphedRegTR(model, stages=True), GraphedRegTR(model)
    per = {nm: [] for nm in GraphedRegTR.STAGES}
    lat = []
    for i in range(3):
        staged(batch_at(W + i, resident)[0]); single(batch_at(W + i, resident)[0])
    for i in range(reps):
        batch = batch_at(W + i, resident)[0]
        flush.zero_()
        ticket = staged.submit(batch)
        staged.result(ticket)
        for nm, v in staged.stage_ms(ticket[0]).items():
            per[nm].append(v)
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        single.result(single.submit(batch))
        e1.record()
        torch.cuda.synchronize()
        lat.append(e0.elapsed_time(e1))
    med = {nm: statistics.median(v) for nm, v in per.items()}
    return dict(stage_ms=med, stage_sum_ms=sum(med.values()), single_stream_latency_ms=statistics.median(lat),
                pairs_per_forward=B, note='serial forward (nothing else on the GPU), L2 flushed before each; '
                'four stage graphs replayed back to back with CUDA events between them; latency = one-graph '
                'executor incl. input copy and result D2H')


def retime(fn, flush, reps=3):
    """[L2 flush][event][launch][event], best of `reps`, and the same launch again with its inputs L2-resident."""
    best = best_w = None
    for _ in range(reps):
        flush.zero_()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record(); fn(); ev[1].record()
        ev[2].record(); fn(); ev[3].record()
        torch.cuda.synchronize()
        t, tw = ev[0].elapsed_time(ev[1]), ev[2].elapsed_time(ev[3])
        best = t if best is None else min(best, t)
        best_w = tw if best_w is None else min(best_w, tw)
    return best, best_w


def measure_rooflines(model, batch_at, resident, flush, W, K, B, ms_per_step):
    """Roofline entries of the three north-star kernel families and of the whole forward, from the REAL shapes of
    one traced eager forward: every launch is re-timed alone on the launching stream right after an L2 flush."""
    from regtr_b200 import ops
    pk = peak_table()
    tf32_peak = pk['bf16_tflops'] / 2.0                    # dense TF32 = half the measured bf16 rate (burst: kernels timed alone)
    ops.KPCONV_TRACE, ops.TRACE = [], []
    flush.zero_()
    model(batch_at(W, resident)[0])
    torch.cuda.synchronize()
    ktr, tr = ops.KPCONV_TRACE, ops.TRACE
    ops.KPCONV_TRACE = ops.TRACE = None

    # ---- KPConv neighbour gather (HBM bound, SURVEY 8d algorithmic bytes)
    gather_ms = warm_ms = 0.0
    per_launch = []
    agg_flops = 0.0
    for _, _, info in ktr:
        t, tw = retime(lambda: ops.kpconv_aggregate(*info['args'], row_flags=info.get('row_flags')), flush)
        gather_ms += t; warm_ms += tw
        nnz = int((info['idx'] < info['Ns']).sum().item())
        agg_flops += nnz * 15 * 12 + 2.0 * info['Nq'] * 15 * info['K'] * info['Cin']
        per_launch.append(dict(Nq=info['Nq'], Cin=info['Cin'], us=round(t * 1e3, 1), us_l2_warm=round(tw * 1e3, 1)))
    step_bytes = sum(kpconv_algorithmic_bytes(info) for _, _, info in ktr)
    ach = step_bytes / (gather_ms * 1e-3) / 1e9
    gather = dict(name='kpconv_gather', bound='hbm',
                  kernel='KPConv neighbour gather + kernel-point influence + aggregation (one launch per KPConv, each '
                         'timed alone right after an L2 flush); bytes = SURVEY 8d algorithmic bytes of the KPConv op',
                  achieved=ach, peak=pk['hbm_gbs'], unit='GB/s', frac=ach / pk['hbm_gbs'],
                  traffic=ncu_traffic('kpconv_gather', B), traffic_unit='bytes/launch (committed ncu capture)',
                  peak_source=pk['source'], launches=len(ktr), algorithmic_bytes_per_step=step_bytes,
                  algorithmic_bytes_per_launch=step_bytes / max(len(ktr), 1), ms_per_step=gather_ms,
                  ms_per_step_l2_warm=warm_ms, frac_l2_warm=step_bytes / (warm_ms * 1e-3) / 1e9 / pk['hbm_gbs'],
                  per_launch=per_launch)

    # ---- dense layers: 3xTF32 tcgen05 GEMM (tensor bound); MMA flops = 2*M*N*K*3
    g_ms = g_flops = 0.0
    shapes = {}
    for kind, info, fn in tr:
        if kind != 'gemm':
            continue
        t, _ = retime(fn, flush)
        fl = 2.0 * info['M'] * info['N'] * info['K']
        g_ms += t; g_flops += fl
        key = (info['M'], info['N'], info['K'])
        c = shapes.setdefault(key, [0, 0.0])
        c[0] += 1; c[1] += t
    n_gemm = sum(c[0] for c in shapes.values())
    ach = 3.0 * g_flops / (g_ms * 1e-3) / 1e12
    top = sorted(shapes.items(), key=lambda kv: -kv[1][1])[:12]
    gemm = dict(name='gemm_tf32x3', bound='tensor',
                kernel='k_gemm_tf32x3 (+ split-K reduce): every nn.Linear and the KPConv weight contraction; flops = '
                       '2*M*N*K*3 TF32 MMA flops (3xTF32 split) summed over the launches of one forward, each timed alone '
                       'after an L2 flush',
                achieved=ach, peak=tf32_peak, unit='TFLOP/s', frac=ach / tf32_peak, traffic=ncu_traffic('gemm_tf32x3', B),
                peak_source=pk['source'] + ': bf16_tflops / 2 (dense TF32)', launches=n_gemm, ms_per_step=g_ms,
                fp32_equiv_flops_per_step=g_flops, fp32_equiv_tflops=g_flops / (g_ms * 1e-3) / 1e12,
                top_shapes=[dict(M=k[0], N=k[1], K=k[2], launches=c[0], us=round(c[1] * 1e3, 1),
                                 tf32_tflops=round(3 * 2.0 * k[0] * k[1] * k[2] * c[0] / (c[1] * 1e-3) / 1e12, 1))
                            for k, c in top])

    # ---- attention core (QK^T and PV): 4*q*k*E flops per problem, x3 for the 3xTF32 split
    a_ms = a_flops = 0.0
    n_att = 0
    for kind, info, fn in tr:
        if kind != 'mha':
            continue
        t, _ = retime(fn, flush)
        a_ms += t; a_flops += 4.0 * info['pairs_qk'] * info['E']; n_att += 1
    att = None
    if n_att:
        ach = 3.0 * a_flops / (a_ms * 1e-3) / 1e12
        att = dict(name='attention_core', bound='tensor',
                   kernel='attention core (softmax(QK^T)V per head, varlen problems): 4*q*k*E flops per problem, x3 '
                          '(3xTF32 split), self and cross launches of the 6 layers',
                   achieved=ach, peak=tf32_peak, unit='TFLOP/s', frac=ach / tf32_peak, traffic=ncu_traffic('attention_core', B),
                   peak_source=pk['source'] + ': bf16_tflops / 2 (dense TF32)', launches=n_att, ms_per_step=a_ms,
                   fp32_equiv_flops_per_step=a_flops)

    # ---- whole forward: algorithmic fp32-equivalent flops and bytes of one step / the pipelined ms_per_step
    total_flops = g_flops + a_flops + agg_flops
    sus = pk['bf16_tflops_sustained'] / 2.0
    tf = total_flops / (ms_per_step * 1e-3) / 1e12
    whole = dict(name='whole_forward', bound='tensor',
                 kernel='whole forward at the benchmarked throughput: fp32-equivalent algorithmic flops of one step '
                        '(dense layers + attention core + KPConv aggregation/influence) / ms_per_step; the fp32-accurate '
                        'path issues 3 TF32 MMA flops per algorithmic flop',
                 achieved=3.0 * tf, peak=sus, unit='TFLOP/s', frac=3.0 * tf / sus, traffic=ncu_traffic('whole_forward', B),
                 traffic_unit='DRAM bytes of one forward (all kernels of a graph replay, committed ncu capture)',
                 peak_source=pk['source'] + ': bf16_tflops_sustained / 2 (dense TF32, kernel inside a long step)',
                 fp32_equiv_flops_per_step=total_flops, fp32_equiv_tflops=tf,
                 hbm_algorithmic_bytes_per_step=step_bytes,
                 hbm_frac_on_gather_bytes=step_bytes / (ms_per_step * 1e-3) / 1e9 / pk['hbm_gbs'],
                 ms_per_step=ms_per_step, pairs_per_step=B,
                 kernel_ms_alone=dict(gather=gather_ms, gemm=g_ms, attention_core=a_ms),
                 kpconv_op_ms_per_step_eager=sum(a.elapsed_time(b) for a, b, _ in ktr))
    rooflines = [r for r in (gather, gemm, att, whole) if r is not None]
    dominant = max((r for r in rooflines if r['name'] != 'whole_forward'), key=lambda r: r['ms_per_step'])
    return dominant, rooflines


def main():
    args = parse()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        return run_reference(args, rank, world)

    import torch.distributed as dist
    from regtr_b200 import ops
    from regtr_b200.config import get_config
    from regtr_b200.dist import gather_poses
    from regtr_b200.regtr import GraphedRegTR, PipelinedRegTR, RegTR
    from regtr_b200.weights import random_state_dict

    assert torch.cuda.is_available(), 'bench.py --impl b200 needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        if os.environ.get('NCCL_DEBUG', '').upper() == 'VERSION':
            os.environ['NCCL_DEBUG'] = 'WARN'   # keep stdout to the single JSON line (NCCL prints its banner there)
        dist.init_process_group('nccl', device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    B = pairs_per_gpu(args)

    cfg = get_config('3dmatch')
    cfg.attention_impl = args.attention
    sd = random_state_dict(cfg, WEIGHT_SEED)
    model = RegTR(cfg).to(dev).eval()
    model.load_state_dict(sd, strict=True)
    runner = GraphedRegTR(model) if args.graph else model      # the public call a user makes
    depth = args.inflight if args.graph else 1
    pipe = PipelinedRegTR(model, depth) if depth > 1 else None

    # rank-local pool of distinct pairs (generated rank-locally, SURVEY.md 8e)
    n_pool = max(POOL, B)
    pool = make_pool(args.config, n_pool, first=rank * n_pool)
    host = [(torch.from_numpy(s).pin_memory(), torch.from_numpy(t).pin_memory()) for s, t in pool]
    resident = [(s.to(dev), t.to(dev)) for s, t in host]

    def batch_at(step, src):
        ids = [(step * B + j) % n_pool for j in range(B)]
        return {'src_xyz': [src[i][0] for i in ids], 'tgt_xyz': [src[i][1] for i in ids]}, ids

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}                                   # output dict of the last timed step (--dump-outputs)

    def device_step(step):
        batch, _ = batch_at(step, resident)
        out = last['out'] = runner(batch)
        return gather_poses(out['pose'], B * world) if world > 1 else out['pose']

    def e2e_step(step):
        batch, ids = batch_at(step, host)
        if not args.graph:
            batch = {k: [t.to(dev, non_blocking=True) for t in v] for k, v in batch.items()}
        out = runner(batch)                     # graph executor: packs the host clouds, one H2D copy
        if world > 1:
            return gather_poses(out['pose'], B * world).cpu(), ids
        return (out['host_pose'] if 'host_pose' in out else out['pose'].cpu()), ids

    sampler = ClockSampler(local) if rank == 0 else None     # started early: nvidia-smi needs ~0.1 s to report
    log(f'pool ready ({n_pool} pairs, {sum(len(a) + len(b) for a, b in pool) // n_pool} pts/pair); warm-up')
    # ---------------- warm-up
    for i in range(W):
        device_step(i)
    if pipe is not None:                        # capture every (slot, capacity bucket) graph before timing
        pipe.warm([batch_at(i, resident)[0] for i in range(-(-n_pool // B))])
        for i in range(2 * depth):
            pipe.submit(batch_at(i, host)[0])
        pipe.drain()
    barrier()

    host_rec = {}

    def run_pipelined(src):
        """K steps with `depth` forwards in flight; returns (elapsed ms on the device, bytes in/out)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        outs = []
        t_cpu = time.perf_counter()
        for i in range(K):
            done = pipe.submit(batch_at(W + i, src)[0], pre_hook=flush.zero_)
            if done is not None:
                outs.append(done['host_pose'].clone())
        t_cpu = time.perf_counter() - t_cpu
        waited = sum(s.wait_s for s in pipe.slots)
        for s in pipe.slots:
            s.wait_s = 0.0
        host_rec['loop_ms_per_step'] = 1e3 * t_cpu / K                       # wall time of the submit loop
        host_rec['blocked_on_gpu_ms_per_step'] = 1e3 * waited / K            # of which: waiting in event.synchronize
        host_rec['host_work_ms_per_step'] = 1e3 * (t_cpu - waited) / K       # Python + CUDA API calls
        log(f'submit loop {1e3 * t_cpu / K:.3f} ms/step, of which waiting for the GPU {1e3 * waited / K:.3f}')
        drained = pipe.drain()                  # oldest first: the last one is the last step's
        outs += [o['host_pose'].clone() for o in drained]
        last['out'] = drained[-1]
        pipe.join()
        if world > 1:                           # the run's poses, gathered over the ranks (288 B / pair)
            gather_poses(torch.cat(outs, dim=1).to(dev, non_blocking=True), B * K * world)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), outs

    # ---------------- timed region: K steps, HBM-resident inputs
    if sampler:
        sampler.mark()
    launches0 = ops.LAUNCHES
    barrier()
    if pipe is None:
        evs = []
        for i in range(K):
            flush.zero_()                                   # L2 flush between timed steps (not timed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            device_step(W + i)
            e1.record()
            evs.append((e0, e1))
        barrier()
        t_dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    else:
        t_dev_ms, _ = run_pipelined(resident)               # includes the per-step L2 flush kernels
        barrier()
    launches = ops.LAUNCHES - launches0
    log(f'device-resident: {t_dev_ms / K:.3f} ms/step')
    if args.dump_outputs and rank == 0:        # before the next forwards reuse the graphs' output buffers
        log('outputs of the last timed step: %d bytes, points sampled: %s' % dump_outputs(last['out'], args.dump_outputs))

    # ---------------- end-to-end: host buffers in, pose on the host out
    h2d = sum(host[j][0].numel() * 4 + host[j][1].numel() * 4 for j in batch_at(W, host)[1])
    if pipe is None:
        for i in range(2):
            e2e_step(i)
        barrier()
        evs = []
        d2h = 0
        for i in range(K):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            pose_h, ids = e2e_step(W + i)
            e1.record()
            evs.append((e0, e1))
            d2h = pose_h.numel() * 4
        barrier()
        t_e2e_ms = sum(a.elapsed_time(b) for a, b in evs)
    else:
        run_pipelined(host)
        barrier()
        t_e2e_ms, outs = run_pipelined(host)
        d2h = next(iter(pipe.slots[0].graphs.values()))['tail_host'].numel() * 4    # level sizes + status + pose, one copy
        barrier()
    clocks = sampler.stop() if sampler else None
    log(f'e2e: {t_e2e_ms / K:.3f} ms/step; clocks {clocks}')

    # ---------------- max over ranks
    t = torch.tensor([t_dev_ms, t_e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_dev_ms, t_e2e_ms = t.tolist()

    # ---------------- where the time goes: stage times at the reference's _TIMEIT boundaries + rooflines, rank 0
    roof = rooflines = stage_rec = None
    if rank == 0:
        stage_rec = measure_stages(model, batch_at, resident, flush, W, B)
        roof, rooflines = measure_rooflines(model, batch_at, resident, flush, W, K, B, t_dev_ms / K)

    # ---------------- CPU baseline beside it (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and args.cpu_baseline:
        log('cpu baseline ...')
        cpu, _ = time_cpu(cfg, sd, pool, n_pairs=10)        # ~10 s of CPU work on the box's cores
        log(f'cpu baseline {cpu["value"]:.3f} pairs/s on {cpu["cores"]} threads')

    # ---------------- pose error vs the oracle on one pair (reported, also covered by tests/)
    pose_err = None
    if rank == 0 and args.checks:
        try:
            from oracle import pre, regtr_oracle
            s, tg = pool[0]
            out = model({'src_xyz': [resident[0][0]], 'tgt_xyz': [resident[0][1]]})
            ref = regtr_oracle.forward(sd, cfg, [s], [tg], meta=pre.preprocess(cfg, [s, tg]))
            pose_err = float((out['pose'].cpu() - ref['pose']).abs().max())
        except Exception as exc:  # pragma: no cover
            pose_err = f'unavailable: {exc}'

    if rank == 0:
        pairs = B * world * K
        line = dict(
            metric='pairs/sec on 3DMatch-size clouds (~20k pts); pose err vs ref',
            value=pairs / (t_dev_ms * 1e-3), unit='pairs/s', n_gpus=world, steps=K, warmup=W,
            ms_per_step=t_dev_ms / K, higher_is_better=True, scaling='weak', vs_baseline=None,
            dtype='f32', data='synthetic',
            config=dict(workload=workload_name(args, B), pairs_per_gpu_per_step=B,
                        parallelism=f'pair-level data parallel x{world}', l2_flush_between_steps=True,
                        weights='seeded random init (no pretrained weights offline)', precision_mode='fp32 parity (3xTF32 tcgen05 GEMMs, 3xTF32 mma.sync attention + KPConv aggregation)' if args.attention == 'fp32'
                        else 'fast (3xTF32 GEMMs, bf16 tcgen05 attention core)',
                        executor=(f'cuda-graph, {depth} pairs in flight (PipelinedRegTR)' if depth > 1 else
                                  'cuda-graph (GraphedRegTR)') if args.graph else 'eager',
                        timed_region='K steps incl. one 256 MB L2-flush kernel per step' if depth > 1 else
                                     'per-step CUDA events, L2 flush between steps not timed'),
            e2e=dict(value=pairs / (t_e2e_ms * 1e-3), unit='pairs/s', h2d_bytes_per_step=h2d,
                     d2h_bytes_per_step=d2h, ms_per_step=t_e2e_ms / K),
            gpu_launches=launches, host=host_rec or None, clocks=clocks, roofline=roof, rooflines=rooflines, stages=stage_rec,
            cpu_baseline=cpu,
            pose_err_vs_oracle=pose_err, impl='b200')
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
