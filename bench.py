#!/usr/bin/env python
"""bench.py -- BPR triples/sec at d=64 on the synthetic 1M x 100K x 50M set (BASELINE.json
configs[1]), one process per GPU.

A "step" is one epoch of the hot path over the rank's shard of the 50M interactions, in the
reference's own iteration order (model/ranking/BPR.py:31-33: users in id order, each user's positives):
  K0+K1  qrec_bpr_epoch_usermajor_f32: Philox negative sampling (rejection against the user's rated
         row) fused into gather -> dots -> sigmoid -> SGD step -> scatter-add; P[u] register-resident
         inside a user, item rows REDG-added, j never written to HBM
  +   regU*|P|^2 + regI*|Q|^2 for the epoch loss                  (qrec_sumsq_f32, BPR.py:40)
with the (u,i) pairs, the rated-item CSR and both tables already resident in HBM.  `e2e` is the
same epoch entered through the host-buffer C-ABI call (qrec_bpr_epoch_usermajor_host): the step's
positives (CSR: rowptr + item ids) start in pinned HOST memory and are copied to the device chunk by
chunk inside the timed region, overlapped with the kernel; the loss comes back to the host.

Multi-GPU (strong scaling of the fixed 50M set): users are range-partitioned, so P rows and each
user's triples live on one rank; Q (25.6 MB) is replicated and the ranks exchange the sum of their
item-row deltas after each of `--q-syncs` launches per step -- asynchronously, hidden behind the next
launch (parallel.OverlappedTableSync: peer-memory reduce-scatter / all-gather kernels, NCCL fallback).

Further objects on the same JSON line (N=1 unless noted; each can be switched off, none can cost the headline):
  parity_check       (any N) epoch 0 of this very path from the initial tables, negatives exported, against the
                     sequential float64 oracle on the same stream -- also the CPU baseline (whole epoch, 1 core)
  roofline           contract fields + row_op_peak (measured L2 / HBM row gather + scatter-add rates,
                     csrc/microbench.cu) + hbm_bound_config (1M-item table: Q does not fit the L2)
  shuffled_order     the same epoch with shuffled pairs through the order-agnostic kernel
  lightgcn           (any N) LightGCN 3-layer minibatch steps, users sharded / items replicated; epoch time
  neumf              BASELINE config 4: NeuMF steps, reference and [256,128,64] MLP widths, tcgen05 TF32
  config1_filmtrust  BASELINE config 1: the recorded reference run replayed through the drop-in class
  zipf_contended     the fused epoch on Zipf-distributed items

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the timed path computed, as of its last timed step, to DIR/<name>.npy: the tables P and Q
and the step's loss terms.  A table larger than DUMP_TABLE_BYTES is cut to a fixed, seeded sample of its rows.  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NUM_USERS, NUM_ITEMS, DEGREE, D = 1_000_000, 100_000, 50, 64
LR, REG_U, REG_I = 0.01, 0.001, 0.001
ALGO_BYTES_PER_TRIPLE = 24 * D + 12          # SURVEY.md 8(d): 3 rows read + 3 rows written + 3 int32
METRIC = 'BPR triples/sec at d=64'
# Multi-GPU code paths that are on by default.  'blocking' = the round-1 delta all-reduce; 'auto' = the overlapped exchange
# (peer-memory kernels, NCCL fallback).  Flipped to the new paths only once they have been validated on >= 2 GPUs.
LIGHTGCN_MULTI_SCHEME = 'user'        # 'cols' once its N>1 numbers are in (QREC_LGCN_SCHEME overrides)
MULTI_GPU_DEFAULTS = {'qsync': 'auto', 'lightgcn_multi': True, 'parity_multi': True}     # validated at N=2 (profiles/r2/multi_n2)
WORKLOAD = 'BPR synthetic 1M users x 100K items x 50M interactions, d=64, fp32, user-major (reference) order'
DUMP_TABLE_BYTES = 28 << 20          # per table: P and Q together stay under 64 MB in float32 and in float64


def measured_hbm_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(p) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def recorded_traffic():
    """dram bytes per K1 launch from the committed ncu --set full capture, if one exists."""
    p = os.path.join(ROOT, 'profiles', 'k1_traffic.json')
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


def dump_rows(n, row_bytes):
    """Rows of an n-row table that --dump-outputs writes: all of them, or, above DUMP_TABLE_BYTES, the same seeded
    sample on every run."""
    if n * row_bytes <= DUMP_TABLE_BYTES:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_TABLE_BYTES // row_bytes, replace=False))


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + '.npy'), np.ascontiguousarray(a))


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's numpy loop on host cores
# ---------------------------------------------------------------------------------------------
def host_workload(n_triples, seed=7):
    """A user-major sample of the bench workload for the host-side legs: the first n_triples/DEGREE
    users (sample users, DEGREE triples each, in the reference's iteration order BPR.py:31-33), items and
    negatives uniform over the 100K items (the rejection of rated negatives changes 0.05 % of them)."""
    rng = np.random.default_rng(seed)
    users = n_triples // DEGREE
    P = rng.random((users, D)) / 3                # float64, like base/iterativeRecommender.py:37-38
    Q = rng.random((NUM_ITEMS, D)) / 3
    u = np.repeat(np.arange(users, dtype=np.int32), DEGREE)
    i = rng.integers(0, NUM_ITEMS, users * DEGREE).astype(np.int32)
    j = ((i + 1 + rng.integers(0, NUM_ITEMS - 1, users * DEGREE)) % NUM_ITEMS).astype(np.int32)
    return P, Q, u, i, j


def cpu_baseline(sample_triples):
    """Times oracle/bpr_ref.c (float64 restatement of model/ranking/BPR.py:45-53) on one host core on a
    user-major sample (used when the full-epoch parity check, which times the whole epoch, is off)."""
    from oracle import c_oracle
    P, Q, u, i, j = host_workload(sample_triples)
    n = len(u)
    c_oracle.bpr_sgd_sequential(P, Q, u[:100000], i[:100000], j[:100000], LR, REG_U, REG_I)  # warm
    t0 = time.perf_counter()
    c_oracle.bpr_sgd_sequential(P, Q, u, i, j, LR, REG_U, REG_I)
    dt = time.perf_counter() - t0
    return {'value': n / dt, 'unit': 'triples/s', 'cores': 1, 'kind': 'port',
            'sample': '%d user-major triples (%d users x %d) of the same 1M x 100K d=64 workload, float64 C port of the '
                      'reference numpy loop (oracle/bpr_ref.c); the loop is a serial dependency chain, '
                      'so 1 thread (host has %d cores)' % (n, n // DEGREE, DEGREE, os.cpu_count() or 0),
            'seconds': dt, 'host_cores': os.cpu_count()}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import c_oracle
    sample = args.ref_sample
    P, Q, u, i, j = host_workload(sample * (args.steps + args.warmup))
    for w in range(args.warmup):
        s = slice(w * sample, (w + 1) * sample)
        c_oracle.bpr_sgd_sequential(P, Q, u[s], i[s], j[s], LR, REG_U, REG_I)
    t0 = time.perf_counter()
    for k in range(args.steps):
        s = slice((args.warmup + k) * sample, (args.warmup + k + 1) * sample)
        loss = c_oracle.bpr_sgd_sequential(P, Q, u[s], i[s], j[s], LR, REG_U, REG_I)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'P': P[dump_rows(len(P), P[0].nbytes)], 'Q': Q[dump_rows(len(Q), Q[0].nbytes)],
                                         'loss': np.array([loss])})
    desc = ('%d user-major triples per step (fresh users each step) of the same workload; float64 C port (oracle/bpr_ref.c) of '
            'model/ranking/BPR.py:45-53; the Python reference itself cannot travel to the GPU box '
            '(measured here: ~95 K triples/s); serial dependency chain => 1 thread of %d' % (sample, os.cpu_count() or 0))
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'triples/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic', 'config': {'workload': WORKLOAD, 'sample_triples_per_step': sample},
        'cpu_baseline': {'value': value, 'unit': 'triples/s', 'cores': 1, 'kind': 'port', 'sample': desc},
        'e2e': {'value': value, 'unit': 'triples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }))


# ---------------------------------------------------------------------------------------------
# parity of the BENCHMARKED path at the benchmarked size: the fused user-major epoch (all ranks)
# against the reference's sequential loop on the same (u, i, j) stream
# ---------------------------------------------------------------------------------------------
def table_errors(X, Xref, X0):
    """max-norm relative error of the table (the metric of the fp32 parity tests) and the error
    relative to what the epoch moved: ||X - Xref||_F / ||Xref - X0||_F."""
    X = np.asarray(X, np.float64)
    diff = X - Xref
    mv = Xref - X0
    return {'max_abs_err': float(np.abs(diff).max()), 'max_norm_rel': float(np.abs(diff).max() / np.abs(Xref).max()),
            'rms_err_over_rms_update': float(np.sqrt((diff * diff).mean()) / max(1e-300, np.sqrt((mv * mv).mean())))}


def oracle_epoch(P0, Q0, u, i, j, dtype, user_block_perm=None):
    """model/ranking/BPR.py:29-53 through the C port on one host thread; returns P, Q, sum(-ln s), seconds.
    user_block_perm: visit blocks of 1024 users in a permuted order (still user-major inside a block) -- the
    reference's own sensitivity to the iteration order, as a yardstick for the parallel kernel's error."""
    from oracle import c_oracle
    P, Q = P0.astype(dtype), Q0.astype(dtype)
    t0 = time.perf_counter()
    if user_block_perm is None:
        l = c_oracle.bpr_sgd_sequential(P, Q, u, i, j, LR, REG_U, REG_I)
    else:
        l = 0.0
        blk = 1024 * DEGREE
        for b in user_block_perm:
            sl = slice(b * blk, min(len(u), (b + 1) * blk))
            l += c_oracle.bpr_sgd_sequential(P, Q, u[sl], i[sl], j[sl], LR, REG_U, REG_I)
    return P, Q, float(l), time.perf_counter() - t0


def parity_against_sequential(P0, Q0, u, i, j, P_gpu, Q_gpu, loss_gpu, full=True):
    """Compares one GPU epoch from (P0, Q0) on the stream (u, i, j) with the sequential reference loop.
    full: also run the fp32 sequential port (rounding yardstick) and a block-permuted float64 run
    (iteration-order yardstick), the three on separate host threads."""
    from concurrent.futures import ThreadPoolExecutor
    P0d, Q0d = P0.astype(np.float64), Q0.astype(np.float64)
    ex = ThreadPoolExecutor(3)
    try:
        main = ex.submit(oracle_epoch, P0d, Q0d, u, i, j, np.float64)         # this run is also the CPU timing
        if full:                                                             # the two yardsticks on two more host threads
            nblk = -(-(len(u) // DEGREE) // 1024)
            perm = np.random.default_rng(3).permutation(nblk)
            f32 = ex.submit(oracle_epoch, P0d, Q0d, u, i, j, np.float32)
            prm = ex.submit(oracle_epoch, P0d, Q0d, u, i, j, np.float64, perm)
        Pr, Qr, lr_, secs = main.result()
        if full:
            P32, Q32, l32, _ = f32.result()
            Pp, Qp, lp, _ = prm.result()
    finally:
        ex.shutdown()
    out = {'oracle': 'oracle/bpr_ref.c float64, sequential, the same (u,i,j) stream in the same user-major order '
                     '(model/ranking/BPR.py:29-53)',
           'triples': int(len(u)), 'oracle_seconds': secs, 'oracle_triples_per_s': len(u) / secs,
           'oracle_threads_running_concurrently': 3 if full else 1,
           'loss_sum_neg_log_sigmoid': {'gpu': float(loss_gpu), 'oracle_f64': lr_, 'rel_err': abs(loss_gpu - lr_) / lr_},
           'P': table_errors(P_gpu, Pr, P0d), 'Q': table_errors(Q_gpu, Qr, Q0d)}
    if full:
        out['yardstick_f32_sequential_vs_f64'] = {'loss_rel_err': abs(l32 - lr_) / lr_, 'P': table_errors(P32, Pr, P0d),
                                                  'Q': table_errors(Q32, Qr, Q0d)}
        out['yardstick_f64_user_blocks_permuted_vs_in_order'] = {
            'note': 'same sequential float64 loop, blocks of 1024 users visited in a random order',
            'loss_rel_err': abs(lp - lr_) / lr_, 'P': table_errors(Pp, Pr, P0d), 'Q': table_errors(Qp, Qr, Q0d)}
        out['gpu_vs_f32_sequential'] = {'loss_rel_err': abs(loss_gpu - l32) / l32,
                                        'P': table_errors(P_gpu, P32.astype(np.float64), P0d),
                                        'Q': table_errors(Q_gpu, Q32.astype(np.float64), Q0d)}
    return out


# ---------------------------------------------------------------------------------------------
# the roofs K1 is compared with, measured on this box in this run
# ---------------------------------------------------------------------------------------------
def _time_ms(torch, fn, reps):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def row_op_peaks(torch, E, dev):
    """csrc/microbench.cu: random 256-byte row gathers (LDG.E.128 x16 lanes) and scatter-adds (REDG.E.ADD.F32x4
    x16 lanes) with nothing else in the loop -- K1's item-table instructions -- on a table that fits the L2
    (the benchmark's 100K x 64 item table) and on one that does not (4M rows = 1 GB)."""
    out = {}
    for name, rows, n_ops in (('item_table_100K_rows_25.6MB_L2_resident', NUM_ITEMS, 200_000_000),
                              ('table_4M_rows_1GB_HBM', 4_000_000, 100_000_000)):
        T = torch.rand(rows, 64, device=dev)
        sec = {}
        for mode, label, rows_per_op in ((0, 'gather', 1), (1, 'scatter_add', 1), (2, 'gather_plus_scatter_add', 2)):
            E.ubench_row_ops(T, n_ops // 10, mode)
            ms = _time_ms(torch, lambda: E.ubench_row_ops(T, n_ops, mode), 3)
            sec[label] = {'ops_per_s': n_ops / (ms * 1e-3), 'GBs': n_ops * rows_per_op * 256 / (ms * 1e-3) / 1e9, 'ms': ms}
        out[name] = sec
        del T
    return out


def hbm_bound_config(torch, E, synthetic, dev, peak, steps=5):
    """The same fused epoch on an item table that does NOT fit the 126 MB L2: 1M users x 1M items (256 MB, config 5's
    item-table shape) x 50M interactions -- the regime in which the HBM roofline of SURVEY 8(d) is the binding one."""
    items = 1_000_000
    data = synthetic.make_interactions(NUM_USERS, items, DEGREE, device=dev, seed=31337)
    P, Q = synthetic.init_tables(NUM_USERS, items, D, seed=11, device=dev)
    loss = torch.zeros(1, dtype=torch.float64, device=dev)
    ep = [0]

    def one():
        ep[0] += 1
        E.bpr_epoch_usermajor(P, Q, data['sorted_rowptr'], data['i'], data['sorted_rowptr'], data['sorted_cols'], items, 77, ep[0],
                              LR, REG_U, REG_I, loss)
    one(); one()
    ms = _time_ms(torch, one, steps)
    n = NUM_USERS * DEGREE
    achieved = n * ALGO_BYTES_PER_TRIPLE / (ms * 1e-3) / 1e9
    assert np.isfinite(float(loss.item()))
    return {'workload': 'BPR synthetic 1M users x 1M items x 50M interactions, d=64 (item table 256 MB > 126 MB L2)',
            'ms_per_epoch': ms, 'triples_per_s': n / (ms * 1e-3), 'achieved_GBs_algorithmic': achieved, 'peak_GBs': peak,
            'frac': achieved / peak, 'algorithmic_bytes_per_triple': ALGO_BYTES_PER_TRIPLE,
            'dram_traffic_note': 'ncu dram bytes for this configuration: profiles/ (k1_hbm_bound_r2*)'}


# ---------------------------------------------------------------------------------------------
# BASELINE config 4: NeuMF (GMF + MLP) minibatch steps, tensor-core MLP path
# ---------------------------------------------------------------------------------------------
def neumf_section(torch, E, data, dev, peak_hbm, steps=10, warmup=3, batch=2048):
    """One minibatch = `batch` interactions x (1 positive + 4 sampled negatives) = 5*batch samples through the
    drop-in NeuMF class (model/ranking/NeuMF.py:12-100 of the reference): gathers, 3-layer MLP forward/backward on
    tcgen05 (TF32), fused head + BCE, scatter-add of the row gradients and TF1's dense Adam over every reached
    table.  Both the reference's widths (2d -> 5d -> 2d -> d) and BASELINE.json's [256,128,64]; phases 0/1/2 =
    GMF / MLP / fused NeuMF.  FLOPs: 3 products forward, 2x that backward (dX and dW)."""
    from qrec_b200.model.ranking.NeuMF import NeuMF

    class FakeData(object):
        user, item = range(NUM_USERS), range(NUM_ITEMS)

    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            tc_peak = float(json.load(f)['bf16_tflops_sustained']) / 2      # TF32 dense = half the bf16 rate
        tc_src = 'MEASURED_PEAKS.json bf16_tflops_sustained / 2 (TF32)'
    except Exception:                                                      # noqa: BLE001
        tc_peak, tc_src = 2250.0 / 2, 'nominal 2.25 PF bf16 / 2'
    g = torch.Generator(device=dev); g.manual_seed(17)
    B = 5 * batch
    batches = []
    n = NUM_USERS * DEGREE
    for t in range(steps + warmup):
        idx = torch.randint(0, n, (batch,), device=dev, generator=g)
        pu = data['u'][idx].repeat_interleave(5).contiguous()
        pi = torch.randint(0, NUM_ITEMS, (B,), device=dev, generator=g, dtype=torch.int32)
        pi[::5] = data['i'][idx]
        pr = torch.zeros(B, device=dev); pr[::5] = 1.0
        batches.append((pu, pi, pr))
    out = {'samples_per_step': B, 'batch_interactions': batch, 'tensor_peak_TFLOPs': tc_peak, 'tensor_peak_source': tc_src,
           'dtype': 'tf32 MMA (tcgen05, fp32 accumulate in TMEM), fp32 everywhere else'}
    for name, widths in (('reference_2d_5d_2d_d', None), ('baseline_256_128_64', (256, 128, 64))):
        m = NeuMF.__new__(NeuMF)
        m.data = FakeData()
        m.num_users, m.num_items, m.emb_size, m.batch_size = NUM_USERS, NUM_ITEMS, D, batch
        m.lRate, m.regU, m.regI, m.engine_device, m.engine_seed, m.device = 0.001, 0.001, 0.001, dev.index or 0, 0, dev
        if widths:
            m.mlp_widths = widths
        _neumf_init(m)
        w1, w2, w3 = m.mlp_widths
        fwd = 2 * (2 * D * w1 + w1 * w2 + w2 * w3)
        sec = {'mlp_widths': [2 * D, w1, w2, w3], 'mlp_flop_per_sample_fwd_bwd': 3 * fwd}
        for mode, label in ((0, 'gmf'), (1, 'mlp'), (2, 'neumf')):
            for t in range(warmup):
                m.train_step(mode, *batches[t])
            it = iter(range(warmup, warmup + steps))
            ms = _time_ms(torch, lambda: m.train_step(mode, *batches[next(it)]), steps)
            tables = (2 if mode != 2 else 4) * (NUM_USERS + NUM_ITEMS) * D
            sec[label] = {'ms_per_step': ms, 'samples_per_s': B / (ms * 1e-3),
                          'mlp_TFLOPs': (3 * fwd * B / (ms * 1e-3) / 1e12) if mode else 0.0,
                          'dense_adam_GB_per_step': tables * 28 / 1e9,
                          'dense_adam_floor_ms': tables * 28 / 1e9 / peak_hbm * 1e3, 'loss': float(m._loss.item())}
        out[name] = sec
        del m
        torch.cuda.empty_cache()
    return out


def _neumf_init(m):
    """NeuMF.initModel without the DeepRecommender/IterativeRecommender data plumbing (synthetic ids)."""
    from qrec_b200.base.deepRecommender import DeepRecommender
    orig = DeepRecommender.initModel
    DeepRecommender.initModel = lambda self: None
    try:
        type(m).initModel(m)
    finally:
        DeepRecommender.initModel = orig


# ---------------------------------------------------------------------------------------------
# BASELINE config 1: the reference's own FilmTrust run through the drop-in class (parity mode)
# ---------------------------------------------------------------------------------------------
def filmtrust_section():
    """configs[0]: BPR on FilmTrust, d=64, the seeded 3-epoch run recorded from the UNMODIFIED reference
    (tests/golden/bpr_filmtrust_seed0.npz: split, MT19937 states, epoch losses, learning rates, metrics), replayed
    through qrec_b200.model.ranking.BPR in parity mode (sequential semantics on the GPU, float64): the epoch losses
    and the ranking measures must equal the reference's; trainModel() is timed.  The reference class itself
    (pure-Python loop, measured in the build container, BASELINE.md section 2) does ~95 K triples/s on one core;
    it cannot be run on this box (no reference checkout, no network)."""
    import contextlib
    import io
    import random
    import tempfile
    from qrec_b200.util.config import ModelConf
    from qrec_b200.model.ranking.BPR import BPR
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'bpr_filmtrust_seed0.npz'))
    train = [[u, i, r] for u, i, r in zip(g['train_users'].tolist(), g['train_items'].tolist(), g['train_rating'].tolist())]
    test = [[u, i, r] for u, i, r in zip(g['test_users'].tolist(), g['test_items'].tolist(), g['test_rating'].tolist())]
    out = {'workload': 'BPR on FilmTrust (ratings.txt, -ap 0.2 -b 1, d=64, lr 0.01, 3 epochs, seeds 0/0): %d training pairs'
                       % len(train), 'reference_python_triples_per_s_build_container': 95_500.0}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            for mode, extra in (('parity_f64', ''), ('fast_f32', 'engine=-mode fast\n')):
                random.setstate((3, tuple(int(x) for x in g['mt_state_after_split']), None))
                np.random.seed(0)
                losses = []
                with contextlib.redirect_stdout(io.StringIO()):       # the bench prints ONE line: keep the class quiet
                    model = BPR(ModelConf.from_string(str(g['conf']) + extra), train, test)
                    orig = model.isConverged
                    model.isConverged = lambda epoch, m=model, o=orig: (losses.append(m.loss), o(epoch))[1]
                    model.readConfiguration(); model.initializing_log(); model.initModel()
                    t0 = time.perf_counter()
                    model.trainModel()
                    dt = time.perf_counter() - t0
                    model.evalRanking()
                ref_loss = g['loss'].tolist()
                out[mode] = {'train_seconds': dt, 'epochs': len(losses), 'triples_per_s': len(losses) * len(g['triples_epoch'][0]) / dt,
                             'epoch_losses': losses, 'reference_epoch_losses': ref_loss,
                             'max_loss_rel_err': max(abs(a - b) / b for a, b in zip(losses, ref_loss)),
                             'measure': [m.strip() for m in model.measure], 'reference_measure': g['measure'].tolist(),
                             'measure_equal': [m.strip() for m in model.measure] == g['measure'].tolist()}
        finally:
            os.chdir(cwd)
    return out


def zipf_section(torch, E, synthetic, dev, steps=5):
    """SURVEY 8(d) contention stress: the same 1M x 100K x 50M shape with Zipf-like item popularity
    (item = floor(I x^2): the hottest item takes ~0.3 % of all positives), fused user-major epoch."""
    data = synthetic.make_interactions(NUM_USERS, NUM_ITEMS, DEGREE, device=dev, zipf=True, seed=424242)
    P, Q = synthetic.init_tables(NUM_USERS, NUM_ITEMS, D, seed=12, device=dev)
    loss = torch.zeros(1, dtype=torch.float64, device=dev)
    ep = [0]

    def one():
        ep[0] += 1
        E.bpr_epoch_usermajor(P, Q, data['sorted_rowptr'], data['i'], data['sorted_rowptr'], data['sorted_cols'], NUM_ITEMS, 99, ep[0],
                              LR, REG_U, REG_I, loss)
    one(); one()
    ms = _time_ms(torch, one, steps)
    hot = int(torch.bincount(data['i'].long(), minlength=NUM_ITEMS).max().item())
    assert np.isfinite(float(loss.item()))
    return {'workload': 'BPR synthetic 1M x 100K x 50M, Zipf-like items (item = floor(I x^2)), d=64, fused user-major epoch',
            'ms_per_epoch': ms, 'triples_per_s': NUM_USERS * DEGREE / (ms * 1e-3), 'hottest_item_positives': hot,
            'parity': 'tests/test_gpu_parity_config2.py::test_fused_epoch_vs_sequential_reference_zipf_contended'}


# ---------------------------------------------------------------------------------------------
# second half of the headline metric: LightGCN epoch time on the same synthetic graph
# ---------------------------------------------------------------------------------------------
def local_bipartite_blocks(torch, dist, data, users_local, num_items, world):
    """The rank's blocks of D^-1/2 (R (+) R^T) D^-1/2 (base/graphRecommender.py:10-29) from ITS users'
    interactions: A_ui [users_local, I] (CSR over local users, global item columns) and its transpose A_iu
    [I, users_local]; item degrees are global (one all-reduce of the histogram).  Setup code (torch ops)."""
    dev = data['sorted_cols'].device
    cols = data['sorted_cols']
    deg_i = torch.bincount(cols.long(), minlength=num_items).double()
    if world > 1:
        dist.all_reduce(deg_i)
    rowptr = data['sorted_rowptr']
    lens = rowptr[1:] - rowptr[:-1]
    users = torch.repeat_interleave(torch.arange(users_local, device=dev), lens)
    vals = (1.0 / torch.sqrt(lens.double()[users] * deg_i[cols.long()])).float().contiguous()
    order = torch.argsort(cols.long() * users_local + users)
    iu_rowptr = torch.zeros(num_items + 1, dtype=torch.int64, device=dev)
    iu_rowptr[1:] = torch.cumsum(torch.bincount(cols.long(), minlength=num_items), 0)
    A_ui = (rowptr.contiguous(), cols.contiguous(), vals)
    A_iu = (iu_rowptr, users[order].int().contiguous(), vals[order].contiguous())
    return A_ui, A_iu


def lightgcn_section(torch, dist, E, synthetic, data, dev, peak, rank, world, layers=3, steps=6, warmup=2):
    """LightGCN (3 layers, d=64) minibatch steps with the reference's semantics -- the whole propagation,
    its backward pass and a dense Adam update for EVERY minibatch (model/ranking/LightGCN.py:35-39) -- on the
    1M x 100K x 50M-edge graph, users partitioned over the ranks and the item rows replicated
    (parallel.UserShardedLightGCN; one all-reduce of the [I, d] item block per layer).  Every timed step is a
    DIFFERENT minibatch.  Step time does not depend on the batch size B (SpMM bound), so the epoch time is
    step x ceil(50M / B); the reference-style B=2048 and a large batch are both reported."""
    from qrec_b200 import parallel
    users_local = NUM_USERS // world
    U, I, N = NUM_USERS, NUM_ITEMS, NUM_USERS + NUM_ITEMS
    nnz = 2 * NUM_USERS * DEGREE
    g = torch.Generator(device=dev); g.manual_seed(5)
    # N > 1: 'user' = users partitioned over the ranks, items replicated (all-reduces of the item block);
    #        'cols' = embedding columns partitioned, adjacency replicated (one [B] all-reduce per step)
    scheme = os.environ.get('QREC_LGCN_SCHEME', LIGHTGCN_MULTI_SCHEME) if world > 1 else 'user'
    if scheme == 'cols' and D % (4 * world):
        scheme = 'user'
    item_blocks = 1
    if scheme == 'cols':
        from qrec_b200.base.graphRecommender import DeviceCSR
        # every rank needs the whole graph: the ranks' user ranges are consecutive, so the all-gathered column lists
        # are the global user-major CSR (setup code)
        parts = [torch.empty_like(data['sorted_cols']) for _ in range(world)]
        dist.all_gather(parts, data['sorted_cols'].contiguous())
        full = {'sorted_cols': torch.cat(parts), 'u': torch.arange(U, device=dev, dtype=torch.int32).repeat_interleave(DEGREE)}
        del parts
        rowptr, cols, vals = synthetic.build_norm_adj(full, U, I, dev)
        del full
        torch.cuda.empty_cache()
        dw = D // world
        ego_cols = (torch.randn(N, D, device=dev, generator=g) * 0.005)[:, rank * dw:(rank + 1) * dw].contiguous()   # same seed: one table
        m = parallel.ColumnShardedLightGCN(DeviceCSR.from_tensors((N, N), rowptr, cols, vals), ego_cols, U, layers, 0.001, 0.001)
        g.manual_seed(50 + rank)                       # the ranks draw different parts of the (all-gathered) minibatch
    else:
        A_ui, A_iu = local_bipartite_blocks(torch, dist, data, users_local, I, world)
        Ei = torch.randn(I, D, device=dev, generator=g) * 0.005               # same seed on every rank: replicated items
        g.manual_seed(50 + rank)
        Eu = torch.randn(users_local, D, device=dev, generator=g) * 0.005
        # experiment switch (default 1 = the measured path): column-blocked item-side SpMM, DESIGN.md section 10
        item_blocks = int(os.environ.get('QREC_LGCN_ITEM_BLOCKS', '1'))
        m = parallel.UserShardedLightGCN(A_ui, A_iu, Eu, Ei, layers, 0.001, 0.001, rank * users_local, item_side_blocks=item_blocks)
    spmm_algo = nnz * (8 + 4 * D) + N * (4 + 4 * D)                 # SURVEY 8(d) no-reuse gather model
    res = {'layers': layers, 'rows': N, 'nnz': nnz, 'n_gpus': world,
           'semantics': 'the reference step: n-layer propagation + loss + its backward pass + dense Adam on every row, once per '
                        'minibatch; every timed step a different minibatch.  At B <= 8192 the two layers that touch only the '
                        "batch's rows -- the last forward layer (the loss reads nothing else of its output) and the first backward "
                        'layer (the loss gradient is zero elsewhere) -- run over those rows\' edges only; the parameter update '
                        'equals the all-rows computation (tests/test_lightgcn_model_cpu.py, test_gpu_models.py vs autograd)',
           'scheme': scheme,
           'impl': ('parallel.ColumnShardedLightGCN: the %d embedding columns partitioned over %d ranks (every rank runs the '
                    'single-GPU step at width %d on the whole, replicated adjacency); the only data-path collective of a step is '
                    'the all-reduce of the [B] partial scores' % (D, world, D // world)) if scheme == 'cols' else
                   'parallel.UserShardedLightGCN: users partitioned over %d rank(s), items replicated, bipartite blocks '
                   'A_ui/A_iu, row-restricted last forward / first backward layer, %s' % (world, 'one all-reduce of the item block per layer '
                                                                   '(overlapped with the user-side SpMM)' if world > 1 else 'no collective'),
           'item_side_blocks': item_blocks}
    n_local = users_local * DEGREE
    for B in (2048, 65536):
        per_rank = B // world
        batches = []
        for t in range(warmup + steps):                                    # distinct minibatches, built outside the timed region
            idx = torch.randint(0, n_local, (per_rank,), device=dev, generator=g)
            bu_l, bi = data['u'][idx].contiguous(), data['i'][idx].contiguous()
            bj = E.sample_neg_philox(bu_l, data['sorted_rowptr'], data['sorted_cols'], I, 1, t)
            bu = (bu_l + rank * users_local).int()
            if world > 1:
                parts = [torch.empty(3, per_rank, dtype=torch.int32, device=dev) for _ in range(world)]
                dist.all_gather(parts, torch.stack([bu, bi, bj]))
                allb = torch.cat(parts, dim=1)
                bu, bi, bj = allb[0].contiguous(), allb[1].contiguous(), allb[2].contiguous()
            batches.append((bu, bi, bj))
        def timed(step_fn, first):
            for t in range(warmup):
                step_fn(*batches[(first + t) % len(batches)])
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for t in range(steps):
                step_fn(*batches[(first + warmup + t) % len(batches)])
            b.record()
            torch.cuda.synchronize()
            tms = torch.tensor([a.elapsed_time(b) / steps], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            return float(tms.item())
        ms_eager = timed(m.train_step, 0)
        # the same steps replayed from a CUDA graph (parallel.UserShardedLightGCN.train_step_graphed: one capture per batch
        # size, three small device copies + one replay per minibatch); a failed capture falls back to the eager step
        # run on hardware at N = 1, 2 and 4 (profiles/r2/s2); beyond that it is opt-in (QREC_LGCN_GRAPH=1): a capture that
        # goes wrong at an untested size must not cost the whole line
        g_env = os.environ.get('QREC_LGCN_GRAPH', 'auto')
        graphed = hasattr(m, 'train_step_graphed') and g_env != '0' and (world <= 4 or g_env == '1')
        ms_graph = timed(m.train_step_graphed, 0) if graphed else None
        graph_ok = bool(graphed and getattr(m, 'graph_error', None) is None)
        # the step API is chosen by measurement: the replayed graph wins where the host cannot issue ~80 launches per step
        # fast enough (N > 1, a rank's share of a step is ~1 ms of device work); at N = 1 the step is device-bound either way
        graph_used = bool(graph_ok and ms_graph <= ms_eager)
        ms = ms_graph if graph_used else ms_eager
        n_steps = -(-U * DEGREE // B)
        full_products = 2 * layers - (2 if (B <= 8192 and layers > 1) else 0)       # whole-graph SpMMs actually executed
        rest_bytes = (layers + 2) * N * D * 8 + B * (3 * 4 * D * 2 + 12) + 7 * N * D * 4
        executed_bytes = full_products * spmm_algo + rest_bytes
        step_bytes = 2 * layers * spmm_algo + (layers + 2) * N * D * 8 + B * (3 * 4 * D * 2 + 12) + 7 * N * D * 4
        res['batch_%d' % B] = {'ms_per_step': ms, 'steps_per_epoch': n_steps, 'epoch_s': ms * n_steps / 1e3,
                               'epoch_extrapolated_from_steps': steps, 'ms_per_step_eager_launches': ms_eager,
                               'ms_per_step_graph_replay': ms_graph if graph_ok else None,
                               'cuda_graph': graph_used, 'graph_error': getattr(m, 'graph_error', None),
                               'algorithmic_GB_per_step': step_bytes / 1e9,
                               'whole_graph_products_per_step': full_products, 'executed_GB_per_step': executed_bytes / 1e9,
                               'frac_of_hbm_peak_executed': executed_bytes / ms / 1e6 / (peak * world),
                               'frac_of_hbm_peak_whole_job': step_bytes / ms / 1e6 / (peak * world), 'loss': float(m.loss.item())}
        del batches
    if world == 1:
        # one whole-graph SpMM (the joint (U+I)^2 operator) for the K2 roofline
        rowptr, cols, vals = synthetic.build_norm_adj(data, U, I, dev)
        X = torch.cat([Eu, Ei]); Y = torch.empty_like(X)
        for _ in range(warmup):
            E.spmm_csr(rowptr, cols, vals, X, Y, rowsplit=True)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            E.spmm_csr(rowptr, cols, vals, X, Y, rowsplit=True)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        res['spmm'] = {'kernel': 'spmm_csr_kernel<16,1>', 'ms': ms, 'algorithmic_GB': spmm_algo / 1e9,
                       'achieved_GBs': spmm_algo / ms / 1e6, 'frac_of_hbm_peak': spmm_algo / ms / 1e6 / peak}
        del rowptr, cols, vals, X, Y
        # K2 as the step runs it: the two bipartite halves, one launch each.  Their bound is the rate at which the SMs can
        # gather 256-byte rows out of the L2 (main() relates them to roofline.row_op_peak's measured gather rate): cutting the
        # item side into column blocks of users that fit the L2 changes nothing (profiles/r2/s2/bench_spmm_blocks.jsonl)
        Yu, Yi = torch.empty_like(Eu), torch.empty_like(Ei)
        halves = {}
        for name, A, X_, Y_ in (('user_side_A_ui_E_i', A_ui, Ei, Yu), ('item_side_A_iu_E_u', A_iu, Eu, Yi)):
            for _ in range(warmup):
                E.spmm_csr(A[0], A[1], A[2], X_, Y_, rowsplit=True)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                E.spmm_csr(A[0], A[1], A[2], X_, Y_, rowsplit=True)
            b.record()
            torch.cuda.synchronize()
            hms = a.elapsed_time(b) / steps
            halves[name] = {'ms': hms, 'gathered_rows': int(A[1].numel()), 'gathers_per_s': int(A[1].numel()) / (hms * 1e-3)}
        try:                                               # DRAM bytes per launch from the committed ncu --set full capture
            with open(os.path.join(ROOT, 'profiles', 'k2_traffic.json')) as f:
                k2t = json.load(f)
            for name in halves:
                t = k2t.get(name)
                if t:
                    halves[name]['traffic'] = t['dram_bytes_read'] + t['dram_bytes_write']
                    halves[name]['algorithmic_bytes'] = k2t['algorithmic_bytes_per_half']
                    halves[name]['traffic_source'] = k2t['source']
        except Exception:                                  # noqa: BLE001
            pass
        res['spmm_halves'] = halves
        del Yu, Yi
        if rank == 0:
            res['cpu_baseline'] = lightgcn_cpu_baseline(torch, synthetic, dev, layers, res['batch_2048']['steps_per_epoch'])
            res['cpu_baseline']['gpu_speedup_epoch_batch_2048'] = res['cpu_baseline']['epoch_s_batch_2048_best'] / res['batch_2048']['epoch_s']
    return res


def lightgcn_cpu_baseline(torch, synthetic, dev, layers, steps_per_epoch, scale=10):
    """CPU restatement of the reference's TF step cost (TensorFlow 1.14 is not installed): one SpMM
    of the normalised adjacency on a 1/`scale` graph of the same degree structure -- the C port
    (oracle/bpr_ref.c, index-order accumulation like TF's CPU kernel, 1 thread) and torch's CPU CSR
    SpMM on all host cores -- scaled by `scale` (SpMM cost is linear in nnz) and by the 2*layers
    products per minibatch (forward + backward); dense Adam and the O(B) terms are left out (they
    only make the CPU slower)."""
    from oracle import c_oracle
    U, I = NUM_USERS // scale, NUM_ITEMS // scale
    small = synthetic.make_interactions(U, I, DEGREE, device=dev, seed=777)
    rp, co, va = (t.cpu() for t in synthetic.build_norm_adj(small, U, I, dev))
    X = (torch.randn(U + I, D) * 0.005).contiguous()
    t0 = time.perf_counter()
    c_oracle.spmm_csr(rp.numpy(), co.numpy(), va.numpy(), X.numpy())
    t_c = time.perf_counter() - t0
    A = torch.sparse_csr_tensor(rp, co.long(), va, size=(U + I, U + I))
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    A @ X
    t0 = time.perf_counter()
    for _ in range(3):
        A @ X
    t_t = (time.perf_counter() - t0) / 3
    per_step = lambda t: t * scale * 2 * layers                           # noqa: E731
    best = min(t_c, t_t)
    return {'kind': 'port', 'sample': '1/%d-scale graph (%d x %d, %d nnz), one SpMM, extrapolated x%d and x%d products/step'
            % (scale, U, I, int(co.numel()), scale, 2 * layers),
            'spmm_s_c_port_1_thread': t_c, 'spmm_s_torch_cpu_all_cores': t_t, 'cores': os.cpu_count(),
            'step_s_c_port': per_step(t_c), 'step_s_torch_cpu': per_step(t_t),
            'epoch_s_batch_2048_best': per_step(best) * steps_per_epoch}


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from qrec_b200 import engine as E
    from qrec_b200 import synthetic, parallel

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)   # the exchange must not queue behind K1
        dist.init_process_group('nccl', device_id=dev, pg_options=opts)

    users_local = NUM_USERS // world
    n_local = users_local * DEGREE
    data = synthetic.make_interactions(users_local, NUM_ITEMS, DEGREE, device=dev,
                                       user_offset=rank * users_local)
    P, Q = synthetic.init_tables(users_local, NUM_ITEMS, D, seed=1 + rank, device=dev)
    if world > 1:
        dist.broadcast(Q, 0)
    g = torch.Generator(device=dev); g.manual_seed(99 + rank)
    u, i = data['u'], data['i']                  # CSR order: user-major, random item order inside a user
    j = torch.empty(n_local, dtype=torch.int32, device=dev)
    rowptr, cols = data['sorted_rowptr'], data['sorted_cols']
    csr_rowptr = rowptr                          # every user has DEGREE positives: same offsets
    loss = torch.zeros(3, dtype=torch.float64, device=dev)
    q_syncs = max(1, args.q_syncs) if world > 1 else 1
    # N>1: asynchronous exchange of the item-table deltas, hidden behind the next launch
    # (parallel.OverlappedTableSync: peer-memory reduce-scatter / all-gather kernels, NCCL as a fallback)
    make_sync = (lambda t: parallel.OverlappedTableSync(t, backend=args.qsync)) if args.qsync != 'blocking' \
        else (lambda t: parallel.ReplicatedTableSync(t))
    qsync = make_sync(Q)
    drain = getattr(qsync, 'finalize', lambda: None)
    loss_hist = torch.zeros(args.steps + args.warmup + 8, 3, dtype=torch.float64, device=dev)
    # sync points at user boundaries (multiples of DEGREE triples)
    ub = parallel.sync_points(users_local, q_syncs)
    k1_events = []

    # the sampler's rejection test: 512-bit rated-set signature per user before the bisection (identical negatives,
    # tests/test_gpu_k1_sig.py; 6.27 vs 6.59 ms per 50 M triples) unless --sampler bisect
    rated_sig = E.rated_signature(rowptr, cols) if args.sampler == 'sig' else None

    def fused(Pt, Qt, pos_rowptr, pos_i, rated_rowptr, rated_cols, sig, seed, epoch, loss1, j_out):
        if sig is not None:
            E.bpr_epoch_usermajor_sig(Pt, Qt, pos_rowptr, pos_i, rated_rowptr, rated_cols, sig, NUM_ITEMS, seed, epoch, LR, REG_U,
                                      REG_I, loss1, j_out=j_out)
        else:
            E.bpr_epoch_usermajor(Pt, Qt, pos_rowptr, pos_i, rated_rowptr, rated_cols, NUM_ITEMS, seed, epoch, LR, REG_U, REG_I,
                                  loss1, j_out=j_out)

    def epoch_on(Pt, Qt, sync, epoch, loss_t, j_out=None, events=None):
        """One epoch of the rank's shard on tables (Pt, Qt): q_syncs fused launches, each followed by the
        item-table delta all-reduce when N>1.  j_out (int32[n_local]) receives the sampled negatives."""
        for s in range(q_syncs):
            ua, ub_ = ub[s], ub[s + 1]
            a, b = ua * DEGREE, ub_ * DEGREE
            if events is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            if q_syncs == 1:
                fused(Pt, Qt, csr_rowptr, i, rowptr, cols, rated_sig, 2024, epoch, loss_t[0:1], j_out)
            else:
                rp = (csr_rowptr[ua:ub_ + 1] - a).contiguous()
                fused(Pt[ua:ub_], Qt, rp, i[a:b], rowptr[ua:ub_ + 1].contiguous(), cols,
                      None if rated_sig is None else rated_sig[ua:ub_], 2024 + s, epoch, loss_t[0:1],
                      None if j_out is None else j_out[a:b])
            if events is not None:
                e1.record()
                events.append((e0, e1, b - a))
            sync.sync()           # N>1: NCCL all-reduce of this rank's item-row deltas (no-op at N=1)

    def step(epoch, timed):
        l = loss_hist[epoch]                 # one slot per epoch: the Q term is written from the exchange's stream
        epoch_on(P, Q, qsync, epoch, l, events=k1_events if timed else None)
        E.sumsq(P, l[1:2])
        if world > 1 and hasattr(qsync, 'after_merge'):
            qsync.after_merge(lambda: E.sumsq(qsync.base, l[2:3]))       # |Q|^2 of the table all ranks agree on
        else:
            E.sumsq(Q, l[2:3])

    launches_before = None
    for w in range(args.warmup):
        step(w, False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    launches_before = E.launch_count()
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_beg.record()
    for k in range(args.steps):
        step(args.warmup + k, True)
    drain()                                   # N>1: the last exchange + merge are inside the timed region
    t_end.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches = E.launch_count() - launches_before
    clocks = sampler.stop() if sampler else None
    elapsed_ms = t_beg.elapsed_time(t_end)
    k1_ms = sum(a.elapsed_time(b) for a, b, _ in k1_events)
    k1_triples = sum(c for _, _, c in k1_events)
    final = loss_hist[args.warmup + args.steps - 1].cpu().numpy()
    loss = loss_hist[-1]                    # scratch slot for the secondary sections
    t = torch.tensor([elapsed_ms, k1_ms], dtype=torch.float64, device=dev)
    lsum = torch.tensor([float(final[0] + REG_U * final[1])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lsum)
    elapsed_ms, k1_ms = float(t[0].item()), float(t[1].item())
    epoch_loss = float(lsum.item()) + REG_I * float(final[2])
    assert np.isfinite(epoch_loss), 'loss is not finite'
    total_triples = n_local * world * args.steps
    value = total_triples / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:       # N>1: rank 0's user shard of P; Q is the same on every rank after drain()
        p_rows = torch.from_numpy(dump_rows(users_local, P[0].nbytes)).to(dev)
        dump_outputs(args.dump_outputs, {'P': P[p_rows].cpu().numpy(), 'Q': Q.cpu().numpy()[dump_rows(NUM_ITEMS, Q[0].nbytes)],
                                         'loss': final})       # sum(-ln sigmoid), |P|^2, |Q|^2 of the last timed epoch

    # ------------------------------------------------------------------ the same epoch, shuffled order
    perm = torch.randperm(n_local, device=dev, generator=g)
    su, si = u[perm].contiguous(), i[perm].contiguous()
    sj = torch.empty_like(su)
    del perm

    def shuffled_step(epoch):
        E.sample_neg_philox(su, rowptr, cols, NUM_ITEMS, 4048, epoch, out=sj)
        E.bpr_sgd_batch(P, Q, su, si, sj, LR, REG_U, REG_I, loss[0:1])
        qsync.sync()
        E.sumsq(P, loss[1:2]); E.sumsq(Q, loss[2:3])
    for w in range(2):
        shuffled_step(w)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    s_beg, s_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s_beg.record()
    for k in range(max(3, args.steps // 2)):
        shuffled_step(2 + k)
    drain()
    s_end.record()
    torch.cuda.synchronize()
    ts = torch.tensor([s_beg.elapsed_time(s_end) / max(3, args.steps // 2)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
    shuffled_ms = float(ts.item())

    # ------------------------------------------------------------------ e2e: host buffers
    hu, hj = None, None
    hi = i.cpu().pin_memory()                                  # this epoch's positives, CSR order
    hrp = csr_rowptr.cpu().pin_memory()
    pipe = E.HostPipeline(local, chunk_triples=1 << 22)
    pipe.set_rated_signature(rated_sig)                       # same sampler as the device-resident path
    e2e_epoch = [1000]

    def e2e_step():
        e2e_epoch[0] += 1
        l = pipe.bpr_epoch_usermajor(P, Q, hrp, hi, rowptr, cols, NUM_ITEMS, 2024, e2e_epoch[0], LR, REG_U, REG_I)
        qsync.sync()
        if not hasattr(qsync, 'finalize'):
            torch.cuda.synchronize()      # blocking exchange rewrites Q: the next epoch's kernels (own streams) must wait
        # overlapped exchange: delta is taken on this stream, the sum and the atomic merge run beside the next epoch
        return l

    for w in range(max(1, args.warmup // 2)):
        e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        e2e_loss = e2e_step()
    drain()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    assert np.isfinite(e2e_loss)
    pipe.close()
    e2e_value = total_triples / e2e_s

    # ------------------------------------------------------------------ parity of this very path at this size
    parity = None
    if not args.no_parity and (world == 1 or args.parity_multi):
        try:
            P1, Q1 = synthetic.init_tables(users_local, NUM_ITEMS, D, seed=1 + rank, device=dev)
            if world > 1:
                dist.broadcast(Q1, 0)
            Q0_host = Q1.cpu().numpy() if rank == 0 else None
            sync1 = make_sync(Q1)
            jx = torch.empty(n_local, dtype=torch.int32, device=dev)
            l1 = torch.zeros(3, dtype=torch.float64, device=dev)
            epoch_on(P1, Q1, sync1, 0, l1, j_out=jx)
            getattr(sync1, 'finalize', lambda: None)()
            torch.cuda.synchronize()
            replicas_equal = None
            if world > 1:
                qs = [torch.empty_like(Q1) for _ in range(world)]
                dist.all_gather(qs, Q1)
                replicas_equal = all(torch.equal(qs[0], t) for t in qs)       # after the drain every rank holds the same item table
                del qs
                dist.all_reduce(l1)
                gi = torch.empty(n_local * world, dtype=torch.int32, device=dev)
                gj = torch.empty(n_local * world, dtype=torch.int32, device=dev)
                gP = torch.empty(users_local * world, D, dtype=torch.float32, device=dev)
                dist.all_gather_into_tensor(gi, i.contiguous())
                dist.all_gather_into_tensor(gj, jx)
                dist.all_gather_into_tensor(gP, P1)
            else:
                gi, gj, gP = i, jx, P1
            if rank == 0:
                P0_host = np.concatenate([synthetic.init_tables(users_local, NUM_ITEMS, D, seed=1 + r, device=dev)[0].cpu().numpy()
                                          for r in range(world)])
                hu_all = np.repeat(np.arange(users_local * world, dtype=np.int32), DEGREE)
                try:
                    parity = parity_against_sequential(P0_host, Q0_host, hu_all, gi.cpu().numpy(), gj.cpu().numpy(),
                                                       gP.cpu().numpy(), Q1.cpu().numpy(), float(l1[0].item()), full=(world == 1))
                except Exception as exc:                 # noqa: BLE001  (never costs the headline line)
                    parity = {'error': '%s: %s' % (type(exc).__name__, exc)}
                parity['what'] = ('epoch 0 of the benchmarked path (qrec_bpr_epoch_usermajor_f32, fused Philox sampling, %d GPU(s), '
                                  '%d item-table syncs) from the initial tables, negatives exported through j_out, against the '
                                  'sequential reference loop on the same stream' % (world, q_syncs))
                parity['bound_held_in_tests'] = 'loss rel_err <= 1e-3 (tests/test_gpu_parity_config2.py)'
                if replicas_equal is not None:
                    parity['item_table_replicas_bit_identical_after_drain'] = bool(replicas_equal)
                del P0_host, hu_all
            del P1, Q1, jx, gi, gj, gP, sync1
            torch.cuda.empty_cache()
            if world > 1:
                dist.barrier()
        except Exception as exc:                         # noqa: BLE001
            if world > 1:
                raise                                    # a rank that drops out would hang the others' collectives
            parity = {'error': '%s: %s' % (type(exc).__name__, exc)}

    # ------------------------------------------------------------------ second half of the metric: LightGCN
    # (all ranks; the secondary sections must never cost the headline line: report their failure instead)
    lightgcn = None
    if not args.no_lightgcn and (world == 1 or args.lightgcn_multi):
        del u, i, j, hu, hi, hj, su, si, sj
        torch.cuda.empty_cache()
        try:
            lightgcn = lightgcn_section(torch, dist, E, synthetic, data, dev, measured_hbm_peak()[0], rank, world)
        except Exception as exc:                     # noqa: BLE001
            if world > 1:
                raise                                # a rank that drops out would hang the others' collectives
            lightgcn = {'error': '%s: %s' % (type(exc).__name__, exc)}

    neumf = None
    if world == 1 and not args.no_neumf:
        try:
            neumf = neumf_section(torch, E, data, dev, measured_hbm_peak()[0])
        except Exception as exc:                     # noqa: BLE001
            neumf = {'error': '%s: %s' % (type(exc).__name__, exc)}
        torch.cuda.empty_cache()

    filmtrust, zipf = None, None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            filmtrust = filmtrust_section()
        except Exception as exc:                     # noqa: BLE001
            filmtrust = {'error': '%s: %s' % (type(exc).__name__, exc)}
        try:
            zipf = zipf_section(torch, E, synthetic, dev)
        except Exception as exc:                     # noqa: BLE001
            zipf = {'error': '%s: %s' % (type(exc).__name__, exc)}
        torch.cuda.empty_cache()

    roofs, hbm_cfg = None, None
    if rank == 0 and world == 1 and not args.no_roofs:
        try:
            roofs = row_op_peaks(torch, E, dev)
            hbm_cfg = hbm_bound_config(torch, E, synthetic, dev, measured_hbm_peak()[0])
        except Exception as exc:                     # noqa: BLE001
            roofs = roofs or {'error': '%s: %s' % (type(exc).__name__, exc)}
            hbm_cfg = hbm_cfg or {'error': '%s: %s' % (type(exc).__name__, exc)}
        torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        per_launch_triples = k1_triples / max(1, len(k1_events))
        per_launch_ms = k1_ms / max(1, len(k1_events))
        achieved = per_launch_triples * ALGO_BYTES_PER_TRIPLE / (per_launch_ms * 1e-3) / 1e9
        tr = recorded_traffic()
        if tr and not str(tr.get('kernel', '')).startswith('bpr_sgd_usermajor'):
            tr = None                    # a capture of another kernel says nothing about this one
        # what this kernel itself must move per triple: 2 item rows read + 2 RED-added, 2 ids, and the
        # P row once per user segment of a 32-triple chunk (about 1.64 segments per chunk at degree 50)
        kernel_model_bytes = 4 * 4 * D + 8 + (1.0 + 32.0 / DEGREE) * (2 * 4 * D + 8) / 32.0
        out = {
            'metric': METRIC, 'value': value, 'unit': 'triples/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': elapsed_ms / args.steps, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {
                'workload': WORKLOAD, 'users': NUM_USERS, 'items': NUM_ITEMS, 'interactions': NUM_USERS * DEGREE,
                'd': D, 'lr': LR, 'reg': REG_U, 'triples_per_step': n_local * world,
                'order': 'user-major CSR order (the reference loop, BPR.py:31-33), random item order inside a user, '
                         'negatives re-sampled on device every step (Philox)',
                'l2_policy': 'inputs larger than L2: P 256 MB + 600 MB of indices per step vs 126 MB L2',
                'parallelism': ('users range-partitioned over %d ranks, Q replicated; %d launches (waves) per step, the item-table '
                                'deltas exchanged after each (%s, backend %s%s) while the next wave runs'
                                % (world, q_syncs, type(qsync).__name__, getattr(qsync, 'backend', 'nccl-blocking'),
                                   ('; p2p unavailable: ' + qsync.p2p_error) if hasattr(qsync, 'p2p_error') else ''))
                if world > 1 else 'single GPU',
                'epoch_loss': epoch_loss,
            },
            'roofline': {
                'bound': 'hbm', 'kernel': 'bpr_sgd_usermajor_kernel<16,4,32,true,true%s> (fused Philox sampling%s)' % ((',3,true', ', signature pre-test') if rated_sig is not None else ('', '')), 'achieved': achieved, 'peak': peak,
                'unit': 'GB/s', 'frac': achieved / peak, 'peak_source': peak_src,
                'algorithmic_bytes_per_triple': ALGO_BYTES_PER_TRIPLE,
                'kernel_model_bytes_per_triple': kernel_model_bytes,
                'achieved_kernel_model': per_launch_triples * kernel_model_bytes / (per_launch_ms * 1e-3) / 1e9,
                'launch_ms': per_launch_ms, 'launch_triples': per_launch_triples,
                'traffic': (int(tr['dram_bytes_per_launch'] * per_launch_triples / tr['launch_triples'])
                            if tr and tr.get('launch_triples') else None),
                'traffic_note': (tr or {}).get('note', 'no ncu --set full capture recorded yet'),
            },
            'e2e': {'value': e2e_value, 'unit': 'triples/s',
                    'h2d_bytes_per_step': (4 * n_local + 8 * (users_local + 1)) * world,
                    'd2h_bytes_per_step': 8 * world, 'ms_per_step': 1e3 * e2e_s / args.steps,
                    'api': 'qrec_bpr_epoch_usermajor_host: pinned host CSR positives (rowptr, i) -> chunked H2D overlapped '
                           'with the fused sampling+SGD kernel -> loss D2H; negatives are drawn on the device'},
            'shuffled_order': {'value': n_local * world / (shuffled_ms * 1e-3), 'unit': 'triples/s', 'ms_per_step': shuffled_ms,
                               'kernel': 'bpr_sgd_batch_kernel<16,1,4> (order-agnostic: every triple loads and RED-adds all 3 rows)',
                               'note': 'same epoch with the (u,i) pairs shuffled once (stand-alone Philox sampler + order-agnostic kernel)'},
            'gpu_launches': int(launches),
            'clocks': clocks,
        }
        # What actually bounds the fused kernel is the LSU's REDG issue rate, not HBM (DESIGN.md §4 K1): every
        # triple retires 2 item rows x 16 lanes of red.global.add.v4.f32 (+ the amortised P row), and
        # /opt/skills/guides/B300_MICROARCH.md measures 0.854 (single address) .. 1.29 (spread) cycles per
        # REDG lane per SM.  Reported beside the HBM roofline; never allowed to cost the headline line.
        try:
            mhz = float((clocks or {}).get('sm_mhz') or 0.0)
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            lanes = 2 * (D // 4) + (1.0 + 32.0 / DEGREE) * (D // 4) / 32.0
            if mhz > 0:
                lo, hi = (sms * mhz * 1e6 / (lanes * c) for c in (1.29, 0.854))
                rate = per_launch_triples / (per_launch_ms * 1e-3)
                out['roofline']['redg_issue_floor'] = {
                    'redg_lanes_per_triple': lanes, 'cycles_per_lane': [1.29, 0.854], 'sms': sms, 'sm_mhz': mhz,
                    'triples_per_s': [lo, hi], 'kernel_triples_per_s': rate, 'frac_of_spread_floor': rate / lo,
                    'source': 'B300_MICROARCH.md atomics table (REDG spread / single address), measured on B300'}
        except Exception as exc:                         # noqa: BLE001
            out['roofline']['redg_issue_floor'] = {'error': '%s: %s' % (type(exc).__name__, exc)}
        if roofs is not None and 'error' not in roofs:
            # K1 per triple: 2 item-row gathers + 2 item-row scatter-adds = 2 (gather + scatter-add) pairs on the L2-resident
            # item table (the P row, the ids and the sampler come on top) -> the memory-system ceiling of this formulation
            pair = roofs['item_table_100K_rows_25.6MB_L2_resident']['gather_plus_scatter_add']
            rate = per_launch_triples / (per_launch_ms * 1e-3)
            out['roofline']['row_op_peak'] = {
                'measured': roofs, 'pairs_per_triple': 2, 'ceiling_triples_per_s': pair['ops_per_s'] / 2,
                'frac_of_row_op_ceiling': rate / (pair['ops_per_s'] / 2),
                'note': 'the item table (25.6 MB) lives in the L2, so HBM is not what bounds this kernel: `frac` above follows the '
                        'contract (algorithmic bytes / time / measured HBM copy bandwidth) and exceeds 1; this entry is the '
                        'fraction of the measured L2 gather + RED row-operation rate (csrc/microbench.cu, same instructions, no math)'}
        elif roofs is not None:
            out['roofline']['row_op_peak'] = roofs
        if hbm_cfg is not None:
            out['roofline']['hbm_bound_config'] = hbm_cfg
        if lightgcn is not None:
            if 'spmm_halves' in lightgcn and roofs is not None and 'error' not in roofs:
                g_peak = roofs['item_table_100K_rows_25.6MB_L2_resident']['gather']['ops_per_s']
                for h in lightgcn['spmm_halves'].values():
                    h['frac_of_measured_l2_gather_rate'] = h['gathers_per_s'] / g_peak
                both = sum(h['gathered_rows'] for h in lightgcn['spmm_halves'].values()) / sum(h['ms'] for h in lightgcn['spmm_halves'].values()) * 1e3
                lightgcn['spmm_halves']['both'] = {'gathers_per_s': both, 'frac_of_measured_l2_gather_rate': both / g_peak,
                                                   'l2_gather_peak_rows_per_s': g_peak}
            out['lightgcn'] = lightgcn
        if neumf is not None:
            out['neumf'] = neumf
        if filmtrust is not None:
            out['config1_filmtrust'] = filmtrust
        if zipf is not None:
            out['zipf_contended'] = zipf
        if parity is not None:
            out['parity_check'] = parity
        if world == 1 and parity is not None and 'error' not in parity:
            out['cpu_baseline'] = {
                'value': parity['oracle_triples_per_s'], 'unit': 'triples/s', 'cores': 1, 'kind': 'port',
                'seconds': parity['oracle_seconds'], 'host_cores': os.cpu_count(),
                'sample': 'the WHOLE 50M-triple user-major epoch of this workload (the stream the GPU epoch sampled), float64 '
                          'C port of the reference numpy loop (oracle/bpr_ref.c) -- a serial dependency chain, so 1 thread '
                          'of the %d host cores (two more single-thread oracle runs, the parity yardsticks, were active on '
                          'other cores meanwhile); the same run is the parity oracle' % (os.cpu_count() or 0)}
        elif world == 1 and not args.no_cpu_baseline:
            try:
                out['cpu_baseline'] = cpu_baseline(args.cpu_sample)
            except Exception as exc:                     # noqa: BLE001
                out['cpu_baseline'] = {'value': None, 'unit': 'triples/s', 'cores': 1, 'kind': 'port',
                                       'sample': 'failed: %s: %s' % (type(exc).__name__, exc)}
        print(json.dumps(out), flush=True)
    if world > 1:
        from qrec_b200 import parallel
        if parallel.any_rank_captured_graphs():
            parallel.finish_process(0)      # a live CUDA graph with NCCL work inside blocks the communicator teardown
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--q-syncs', type=int, default=1, help='launches (waves) per step when N>1; the item-table deltas are exchanged after each (overlapped with the next '
                         'launch).  1 = one exchange per epoch: 53 G triples/s at N=8, epoch loss after 25 epochs 1.7 %% above one GPU; '
                         '2: 45 G, 0.9 %%; 4: 35 G (profiles/README.md)')
    ap.add_argument('--qsync', default=MULTI_GPU_DEFAULTS['qsync'], choices=['auto', 'p2p', 'nccl', 'blocking'],
                    help='N>1 item-table exchange: overlapped peer-memory kernels (p2p), overlapped ncclAllReduce (nccl), auto = p2p with nccl fallback, blocking = round-1 path')
    ap.add_argument('--cpu-sample', type=int, default=20_000_000)
    ap.add_argument('--ref-sample', type=int, default=4_000_000)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-lightgcn', action='store_true')
    ap.add_argument('--no-neumf', action='store_true')
    ap.add_argument('--sampler', default='sig', choices=['sig', 'bisect'],
                    help='in-kernel rejection test: rated-set signature before the bisection (default) or bisection only')
    ap.add_argument('--parity-multi', action=argparse.BooleanOptionalAction, default=MULTI_GPU_DEFAULTS['parity_multi'],
                    help='run the full-epoch parity check at N>1 too (rank 0 runs the 50M-triple oracle, ~20 s)')
    ap.add_argument('--lightgcn-multi', action=argparse.BooleanOptionalAction, default=MULTI_GPU_DEFAULTS['lightgcn_multi'],
                    help='run the LightGCN section at N>1 too (users sharded, items replicated)')
    ap.add_argument('--no-extras', action='store_true', help='skip the FilmTrust (config 1) and Zipf sections')
    ap.add_argument('--no-roofs', action='store_true', help='skip the row-op microbenchmark and the HBM-bound configuration')
    ap.add_argument('--no-parity', action='store_true', help='skip the full-epoch parity check against the sequential oracle')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the tables and the loss of the last timed step to DIR/<name>.npy '
                    '(tables above %d MiB: a fixed seeded sample of their rows)' % (DUMP_TABLE_BYTES >> 20))
    args = ap.parse_args()
    assert args.warmup >= 0 and args.steps >= 1
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
