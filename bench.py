#!/usr/bin/env python
"""Benchmark of TIGER's per-batch temporal memory path on B200 (see DESIGN.md, "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload reddit|wikipedia|mooc|lastfm|scaled]
    python bench.py --impl reference ...      # the CPU restatement of the reference path (oracle/), host cores
    python bench.py --dump-outputs DIR ...    # + the last timed step's results as DIR/<name>.npy (float32)

One step = one batch of 200 events through the whole fused path: temporal neighbor finder ->
involved/outdated compaction -> lazy restart -> pending-message gather + GRU -> temporal
attention embedding -> argmax-by-timestamp selection -> right write-back -> message build +
store -> left write-back (fused into the last attention product) -> link scorer + loss.  `value` is
measured with the batch inputs already resident in HBM (CUDA-graph replay, CUDA events); `e2e` goes
through pinned HOST buffers (H2D of the batch, the graphs, D2H of scores + loss inside the timed region).
Both use the batch pipeline of www2023tiger_b200/engine.py:StreamRunner (csrc/pipe.cu): the model kernels of
consecutive batches run strictly in order on one stream (the memory is state), while the upload + neighbor
finder of batch i+1 and the link scorer + download of batch i-1 run beside them on copy streams; every
batch still pays its own H2D and D2H, and every result is read on the host before the clock stops.

Only the `cpu_baseline` leg and `--impl reference` import oracle/ (the CPU checker); the product
path never does.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'events/sec (memory update + embedding, batch 200)'
METRIC_TRAIN = 'events/sec (full training step: memory update + embedding + restarter + backward + Adam, batch 200)'
UNIT = 'events/s'
HIST_LEN = 40
BATCH = 200
K_NEIGH = 10
N_HEAD = 2


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=1000)
    p.add_argument('--warmup', type=int, default=20)
    p.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    p.add_argument('--mode', default='infer', choices=['infer', 'train'],
                   help='infer: the no-grad memory path (BASELINE metric); train: the full training step')
    p.add_argument('--workload', default='reddit', choices=['wikipedia', 'reddit', 'mooc', 'lastfm', 'scaled'])
    p.add_argument('--events', type=int, default=0, help='override the number of events of the stream')
    p.add_argument('--skip-batches', type=int, default=1000, help='batches skipped so that histories are populated')
    p.add_argument('--cpu-batches', type=int, default=400, help='bounded sample of the cpu_baseline leg (0 = off)')
    p.add_argument('--profile-steps', type=int, default=100, help='eager steps with per-kernel CUDA events')
    p.add_argument('--no-e2e', action='store_true')
    p.add_argument('--micro', action='store_true',
                   help='feed each gather/scatter kernel >= 256k rows (tables >> L2) and report HBM GB/s vs peak')
    p.add_argument('--micro-rows', type=int, default=1 << 18)
    p.add_argument('--seed', type=int, default=0)
    p.add_argument('--restarter', default='auto', choices=['auto', 'seq', 'static'],
                   help="auto = the restarter BASELINE.json's config line names for the workload")
    p.add_argument('--cpu-seconds', type=float, default=25.0, help='time budget of the cpu_baseline leg')
    p.add_argument('--parity-batches', type=int, default=3,
                   help='batches replayed after a reset and compared with the CPU arm (0 = off)')
    p.add_argument('--cpu-kind', default='auto', choices=['auto', 'reference', 'port'])
    p.add_argument('--api', default='engine', choices=['engine', 'dropin'],
                   help="engine: the fused per-batch engine (the benchmarked path); dropin: the reference's own evaluation "
                        "loop (eval_edge_prediction) on the tiger/ mirror classes, host collation and host restart sets included")
    p.add_argument('--train-steps', type=int, default=100,
                   help='infer mode: also time this many training steps (fwd + bwd + all-reduce + Adam) of the same '
                        'configuration and report them under "train_step" (0 = off)')
    p.add_argument('--dump-outputs', metavar='DIR', default=None,
                   help='write what the last timed step computed (scores, loss, embeddings, memories) to '
                        'DIR/<name>.npy as float32, so that two builds can be compared output for output')
    args = p.parse_args()
    if args.dump_outputs and (args.micro or args.impl != 'b200' or args.mode != 'infer' or args.api != 'engine'):
        p.error('--dump-outputs covers the default path (--impl b200 --mode infer --api engine) only')
    if args.steps < 1:
        p.error('--steps must be at least 1')
    if args.dump_outputs:
        # the engine runs with the CPU arm's parameters when there is one: random_weights(seed) for the oracle port
        # (the same as without an arm), but the reference's own init_model where oracle/_ref is vendored - pinned to
        # the port, so that a dump depends on the arguments only
        if args.cpu_kind == 'reference':
            p.error('--dump-outputs runs with the seeded random_weights: --cpu-kind reference does not apply')
        args.cpu_kind = 'port'
    return args


def pick_restarter(args, shape):
    return shape.restarter if args.restarter == 'auto' else args.restarter


def dist_env():
    return int(os.environ.get('RANK', 0)), int(os.environ.get('LOCAL_RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))


# ------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------
def load_workload(args, with_efeats=True, cpu_only=False):
    from www2023tiger_b200.synthetic import SHAPES, NegativeSampler, make_stream
    shape = SHAPES[args.workload]
    n_events = args.events or shape.n_events
    if cpu_only:
        with_efeats = with_efeats and st_fits_host(args)    # scaled: CpuArm draws the rows of its event prefix
    st = make_stream(shape, seed=args.seed, n_events=n_events, with_efeats=with_efeats)
    neg = NegativeSampler(st.src, st.dst, seed=args.seed).pre_sample_neg_dsts(st.n_events, BATCH)
    return shape, st, neg


def chunk_bounds(n, rank, world, bs, seed=0):
    """The reference's ChunkSampler partition (tiger/data/data_loader.py:27-37)."""
    import torch
    g = torch.Generator()
    g.manual_seed(seed)
    residual = n % (world * bs)
    shift = int(torch.randint(0, residual + 1, size=(), generator=g))
    length = n // (world * bs) * bs
    return shift + length * rank, shift + length * (rank + 1)


def max_over_ranks(value: float, world: int, device=None) -> float:
    """Timing of a multi-rank run = the slowest rank (all-reduce MAX; identity at world 1)."""
    if world <= 1:
        return float(value)
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def batch_window(args, n_events, rank, world):
    """[first batch start, number of whole batches available] for this rank."""
    if world > 1:
        lo, hi = chunk_bounds(n_events, rank, world, BATCH, args.seed)
    else:
        lo = min(args.skip_batches, (n_events // BATCH) // 2) * BATCH   # histories populated, at least half the stream left
        hi = n_events
    return lo, (hi - lo) // BATCH


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML from a thread of this process while the timed regions
    run (a timed region of the driver's default 20 steps lasts ~2 ms: a `nvidia-smi -lms 100` child never sees
    it).  Samples are taken every ~0.5 ms between start() and stop()."""

    def __init__(self, gpu_index=0):
        import threading
        self.samples, self.reasons_seen = [], 0
        self.max_mhz, self.h, self.nv = None, None, None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = gpu_index
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            if vis:
                try:
                    idx = int(vis.split(',')[gpu_index])
                except (ValueError, IndexError):
                    pass
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None
        if self.h is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.reasons_seen |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                break
            time.sleep(0.0005)

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': []}
        if self._t is None:
            return out
        self._stop.set()
        self._t.join(timeout=2)
        nv = self.nv
        names = {'hw_slowdown': nv.nvmlClocksEventReasonHwSlowdown,
                 'hw_thermal_slowdown': nv.nvmlClocksEventReasonHwThermalSlowdown,
                 'sw_thermal_slowdown': nv.nvmlClocksEventReasonSwThermalSlowdown,
                 'sw_power_cap': nv.nvmlClocksEventReasonSwPowerCap}
        out['reasons'] = sorted(n for n, bit in names.items() if self.reasons_seen & bit)
        if self.samples:
            out['sm_mhz'] = float(np.median(self.samples))
            out['samples'] = len(self.samples)
        return out


# ------------------------------------------------------------------------------------------
# CPU arm: the reference itself (oracle/_ref, vendored by tools/vendor_ref.py) on the host cores; the oracle
# restatement (oracle/tiger_oracle.py) as the second reported number and as the fallback
# ------------------------------------------------------------------------------------------
class CpuArm:
    """step(i) runs batch i of the window that starts at event `lo` (collate + lazy restart + contrast step; in
    train mode the whole training step: + restarter targets, backward, Adam) on the CPU."""

    def __init__(self, args, shape, st, neg, lo, n_batches, *, kind='auto', mode='infer', efeats_prefix=None):
        import torch
        self.kind, self.mode, self.lo, self.args = None, mode, lo, args
        self.restarter = pick_restarter(args, shape)
        self.cores = os.cpu_count() or 1
        n_graph = min(st.n_events, lo + (n_batches + 2) * BATCH)
        if st.efeats is None and shape.efeat_dim > 0:
            # scaled stream: the 34 GB edge table lives on the device only; the CPU arm replays a window of an event
            # prefix and needs the rows of that prefix (efeats_prefix: the device rows when parity is checked)
            if efeats_prefix is None:
                efeats_prefix = np.random.RandomState(args.seed).standard_normal(
                    (n_graph + 1, shape.efeat_dim)).astype(np.float32)
                efeats_prefix[0] = 0
            import copy
            st = copy.copy(st)
            st.efeats = efeats_prefix
        if kind in ('auto', 'reference'):
            from oracle import ref_harness
            why = ref_harness.available()
            if why is None:
                self.ref = ref_harness.ReferenceRunner(
                    st, neg, restarter=self.restarter, msg_src=shape.msg_src, upd_src=shape.upd_src,
                    n_graph_events=n_graph, n_neighbors=K_NEIGH, n_heads=N_HEAD, hist_len=HIST_LEN, batch=BATCH,
                    seed=args.seed, threads=self.cores)
                self.ref.reset(train=(mode == 'train'))
                self.kind = 'reference'
                self.what = ('the unmodified reference (oracle/_ref: GraphCollator + TIGER.restart + '
                             + ('contrast_and_mutual_learning + backward + Adam' if mode == 'train'
                                else 'contrast_learning') + f'), torch {torch.__version__} CPU')
            elif kind == 'reference':
                raise SystemExit(f'--cpu-kind reference: {why}')
        if self.kind is None:
            if mode == 'train':
                raise SystemExit('the training step has no oracle port; vendor the reference (tools/vendor_ref.py)')
            from oracle import tiger_oracle as O
            from www2023tiger_b200.init import random_weights
            torch.set_num_threads(self.cores)
            N, d = st.n_nodes, st.dim
            de = st.efeats.shape[1] if st.efeats is not None else d
            self.W = random_weights(d, de, n_nodes=N, restarter=self.restarter, hist_len=HIST_LEN, seed=args.seed)
            self.O, self.st, self.neg = O, st, neg
            E = n_graph
            self.graph = O.OracleGraph(st.src[:E], st.dst[:E], st.ts[:E], st.eids[:E], n_nodes=N)
            self.model = O.OracleTIGER(self.W, self.graph, N, d, st.efeats, None, n_neighbors=K_NEIGH, n_head=N_HEAD,
                                       msg_src=shape.msg_src, upd_src=shape.upd_src, restarter=self.restarter,
                                       hist_len=HIST_LEN)
            self.uptodate = np.zeros(N, dtype=bool)
            self.kind = 'port'
            self.what = 'oracle/tiger_oracle.py (collate + lazy restart + contrast step), ' \
                        f'torch {torch.__version__} CPU'

    def weights(self):
        return self.ref.state_dict() if self.kind == 'reference' else self.W

    def step(self, i):
        """-> dict(neigh_nids, winner_index, pos_scores, neg_scores, loss) as numpy (eval mode)."""
        lo = self.lo + i * BATCH
        if self.kind == 'reference':
            if self.mode == 'train':
                return self.ref.train_step(lo)
            (loss, _, ps, ns, _, _), cg = self.ref.eval_step(lo)
            return {'neigh_nids': cg.layers[1][0].numpy(), 'winner_index': cg.restart_data.index.numpy(),
                    'pos_scores': ps.numpy(), 'neg_scores': ns.numpy(), 'loss': float(loss)}
        import torch
        O, st, neg = self.O, self.st, self.neg
        s = slice(lo, lo + BATCH)
        b = O.collate(self.graph, st.src[s], st.dst[s], neg[s], st.ts[s], st.eids[s], K_NEIGH)
        rn = O.lazy_restart_nodes(b.involved, self.uptodate)
        with torch.no_grad():
            self.model.restart(rn, np.full(len(rn), b.ts.min(), dtype=np.float32))
            r = self.model.contrast_step(b)
        _, idx = O.select_latest(np.concatenate([b.src, b.dst]), np.tile(b.ts64, 2))
        return {'neigh_nids': b.neigh_nids, 'winner_index': idx, 'pos_scores': r['pos_scores'].numpy(),
                'neg_scores': r['neg_scores'].numpy(), 'loss': float(r['loss'])}

    def time(self, first, max_batches, budget_s, warmup=2):
        """Times consecutive batches first+warmup .. until `max_batches` or the time budget; -> (n, seconds)."""
        for i in range(first, first + warmup):
            self.step(i)
        n, t0 = 0, time.perf_counter()
        while n < max_batches:
            self.step(first + warmup + n)
            n += 1
            if time.perf_counter() - t0 > budget_s and n >= 3:
                break
        return n, time.perf_counter() - t0

    def describe(self, n, lo_batch):
        return (f'{n} consecutive batches of {BATCH} events from event {self.lo + lo_batch * BATCH} of the '
                f'{self.args.workload}-shaped stream: {self.what}, {self.cores} threads')


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    shape, st, neg = load_workload(args, with_efeats=True, cpu_only=True)
    lo, avail = batch_window(args, st.n_events, 0, max(world, 1))
    W, K = args.warmup, args.steps
    if W + K > avail:
        raise SystemExit(f'--warmup {W} + --steps {K} exceed the {avail} batches of the stream window')
    arm = CpuArm(args, shape, st, neg, lo, W + K, kind=args.cpu_kind, mode=args.mode)
    for i in range(W):
        arm.step(i)
    t0 = time.perf_counter()
    for i in range(W, W + K):
        arm.step(i)
    dt = time.perf_counter() - t0
    value = K * BATCH / dt
    line = {
        'impl': 'reference', 'metric': metric_name(args), 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': K,
        'warmup': W, 'ms_per_step': dt / K * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(args, shape, st, world),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': arm.cores, 'kind': arm.kind,
                         'sample': arm.describe(K, W)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def metric_name(args):
    return METRIC_TRAIN if args.mode == 'train' else METRIC


CONFIG_LINES = {   # BASELINE.json:configs, verbatim
    'wikipedia': 'TIGER seq restarter on synthetic Wikipedia-shaped stream (9,227 nodes, 157,474 events, 172-d edge '
                 'feats, dim 172, batch 200)',
    'reddit': 'Synthetic Reddit-shaped stream (10,984 nodes, 672,447 events, 172-d feats), static restarter, 1xB200',
    'mooc': 'Synthetic MOOC-shaped stream (7,144 nodes, 411,749 events, 4-d feats, --dim 100), msg_src/upd_src right',
    'lastfm': 'Synthetic LastFM-shaped stream (1,980 nodes, 1,293,103 events, no edge feats, --dim 100), restart_prob '
              '0.001',
    'scaled': 'Scaled synthetic stream (1M nodes, 50M events, 172-d feats) via train_self_supervised_ddp at 2/4/8xB200',
}


def workload_config(args, shape, st, world):
    rst = pick_restarter(args, shape)
    return {'workload': f'{CONFIG_LINES[args.workload]} :: {st.n_nodes - 1} nodes, {st.n_events} events, '
                        f'd={st.dim}, de={shape.efeat_dim or st.dim}, {rst} restarter'
                        f'{" (hist_len %d)" % HIST_LEN if rst == "seq" else ""}, lazy restart, '
                        f'msg_src={shape.msg_src}, upd_src={shape.upd_src}',
            'mode': args.mode, 'restarter': rst,
            'batch': BATCH, 'n_neighbors': K_NEIGH, 'n_heads': N_HEAD, 'n_layers': 1,
            'partition': 'ChunkSampler time chunks, rank-local memory replicas'
                         + (', gradient all-reduce (NCCL) every step' if args.mode == 'train' else
                            ', no data-path collective') if world > 1 else 'single stream',
            'l2': 'tables read per step (edge features + message store + memories) exceed the 126 MB L2 for '
                  'reddit/scaled; no flush between steps: consecutive batches are state-dependent and run '
                  'back to back exactly as in the real workload'}


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def algorithmic_bytes(kernel, c, d, de, M, B, K):
    """Bytes each kernel must move per launch (SURVEY.md §8(d)); c = mean device counters."""
    U, O, R, P, Po, deg = c['U'], c['O'], c['R'], c['P'], c['Po'], c['log_deg']
    f = 4
    return {
        'tiger_find_recent': 3 * B * (deg * 8 + K * 16 + K * 20) + 3 * B * 16,
        'tiger_compact_involved': c['bitmap_words'] * 4 * 2 + U * (8 + 4 + 1) + O * 8 + R * 8,
        'tiger_static_restart': R * (2 * 2 * d * f + deg * 8 + 16),
        'tiger_gru_update': O * (M + 1) * f + O * d * f + O * d * f,
        'tiger_temporal_attention': 3 * B * K * (d + de) * f + 3 * B * K * 20 + 3 * B * d * f * 2,
        'tiger_select_latest': 2 * B * (8 + 4 + 1),
        'tiger_right_writeback': Po * (2 * d + 2) * f + 2 * B * 9,
        'tiger_store_messages': P * ((2 * d + de) * f + M * f + 8) + 2 * B * 13,
        'tiger_left_writeback': P * (2 * d + 2) * f + 2 * B * 9,
        'tiger_link_score': 3 * B * d * f + 3 * B * K * 8 + 2 * B * f,
    }.get(kernel, 0)


class DeviceWorkload:
    """Stream, features, device CSR, the rank's window of batch records resident in HBM, and (rank 0 at N = 1) the CPU
    arm, whose parameters - the reference's own init_model under torch.manual_seed(seed) - the B200 arm runs with so
    that the two can be compared batch by batch."""

    def __init__(self, args, mode='infer'):
        import torch
        import torch.distributed as dist
        from www2023tiger_b200 import _lib, ops
        rank, local_rank, world = dist_env()
        if not torch.cuda.is_available():
            raise SystemExit('bench.py needs a CUDA device: the TIGER B200 path has no CPU fallback')
        torch.cuda.set_device(local_rank)
        dev = torch.device('cuda', local_rank)
        if world > 1:
            dist.init_process_group('nccl', device_id=dev)
        _lib.load()
        self.rank, self.local_rank, self.world, self.dev = rank, local_rank, world, dev
        shape, st, neg = load_workload(args, with_efeats=st_fits_host(args))
        self.shape, self.st, self.neg = shape, st, neg
        self.N, self.d = st.n_nodes, st.dim
        self.de = shape.efeat_dim or self.d
        if shape.efeat_dim > 0:
            if st.efeats is not None:
                efeats = torch.from_numpy(st.efeats).to(dev)
            else:
                efeats = torch.empty(st.n_events + 1, self.de, device=dev)
                g = torch.Generator(device=dev).manual_seed(args.seed)
                chunk = 1 << 22
                for i in range(0, st.n_events + 1, chunk):
                    efeats[i:i + chunk].normal_(generator=g)
                efeats[0] = 0
        else:
            efeats = None
        self.efeats = efeats
        to = lambda x, dt: torch.as_tensor(x).to(dt).to(dev).contiguous()
        self.csr = ops.csr_build(to(st.src, torch.int64), to(st.dst, torch.int64), to(st.ts, torch.float64),
                                 to(st.eids, torch.int64), self.N)
        self.rst = pick_restarter(args, shape)
        lo, avail = batch_window(args, st.n_events, rank, world)
        if avail < 8:
            raise SystemExit('stream too short for this rank')
        avail = min(avail, max(args.warmup + args.steps + args.profile_steps + 8, 64))   # records actually replayed
        self.lo, self.avail = lo, avail
        B = BATCH
        self.arm = None
        if rank == 0 and world == 1 and args.cpu_batches > 0:
            n_cpu = min(args.cpu_batches + args.parity_batches + 4, avail - 2)
            prefix = None
            if st.efeats is None and efeats is not None:
                prefix = efeats[:min(st.n_events, lo + (n_cpu + 2) * B) + 1].cpu().numpy()
            self.arm = CpuArm(args, shape, st, neg, lo, n_cpu, kind=args.cpu_kind, efeats_prefix=prefix, mode=mode)
        # all batch inputs of this rank's window, resident in HBM: [avail, 5B] int64 (ts as float64 bits)
        host_in = np.empty((avail, 5 * B), dtype=np.int64)
        s = slice(lo, lo + avail * B)
        host_in[:, :B] = st.src[s].reshape(avail, B)
        host_in[:, B:2 * B] = st.dst[s].reshape(avail, B)
        host_in[:, 2 * B:3 * B] = neg[s].reshape(avail, B)
        host_in[:, 3 * B:4 * B] = st.eids[s].reshape(avail, B)
        host_in[:, 4 * B:] = st.ts[s].reshape(avail, B).view(np.int64)
        self.host_in = host_in
        self.dev_in = torch.from_numpy(host_in).to(dev)

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()


DUMP_BYTES = 60 << 20      # --dump-outputs: array bytes, leaves room for the .npy headers under 64 MB


def dump_outputs(out_dir, eng, out_buf):
    """Writes one step's results as float32 .npy files: the link scores and loss (`out_buf`, the step's [pos | neg |
    loss] buffer), the [src | dst | neg] embeddings, and the left / right memories with their update times after the
    step.  Memories larger than the DUMP_BYTES budget keep a fixed sample of rows (RandomState(0), ascending node
    ids), the same rows in every run."""
    import torch
    B, N, d = eng.B, eng.N, eng.d
    res = out_buf.cpu().numpy()
    arrays = {'pos_scores': res[:B], 'neg_scores': res[B:2 * B], 'loss': res[2 * B:], 'embeddings': eng.emb.cpu().numpy()}
    per_row = 2 * (d + 1) * 4
    n_rows = min(N, (DUMP_BYTES - sum(a.nbytes for a in arrays.values())) // per_row)
    rows = None if n_rows == N else torch.from_numpy(
        np.sort(np.random.RandomState(0).choice(N, n_rows, replace=False))).to(eng.device)
    for name, t in (('left_memory', eng.left_vals), ('left_memory_ts', eng.left_ts),
                    ('right_memory', eng.right_vals), ('right_memory_ts', eng.right_ts)):
        arrays[name] = (t if rows is None else t[rows]).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a.astype(np.float32))


def run_b200(args):
    import torch
    import torch.distributed as dist
    from www2023tiger_b200.engine import StreamRunner, TigerEngine
    from www2023tiger_b200.init import random_weights

    wl = DeviceWorkload(args)
    rank, local_rank, world, dev = wl.rank, wl.local_rank, wl.world, wl.dev
    shape, st, neg, efeats, csr, rst = wl.shape, wl.st, wl.neg, wl.efeats, wl.csr, wl.rst
    N, d, de, lo, avail, arm = wl.N, wl.d, wl.de, wl.lo, wl.avail, wl.arm
    host_in, dev_in = wl.host_in, wl.dev_in
    B = BATCH
    if arm is not None:
        W = arm.weights()
    else:
        W = random_weights(d, de, n_nodes=N, restarter=rst, hist_len=HIST_LEN, seed=args.seed)
    eng = TigerEngine(W, csr, n_nodes=N, dim=d, efeats=efeats, n_neighbors=K_NEIGH, n_head=N_HEAD,
                      batch_size=BATCH, msg_src=shape.msg_src, upd_src=shape.upd_src, restarter=rst,
                      hist_len=HIST_LEN, lazy_restart=True, device=dev)

    runner = StreamRunner(eng)
    eng.inp.copy_(dev_in[0])
    runner.capture(warmup=2)
    eng.reset()

    def device_step(i):
        j = i % avail
        if j == 0 and i > 0:
            eng.reset()           # epoch boundary (train_self_supervised.py:127-128): the window wraps
        return runner.submit_device(dev_in[j])

    barrier = wl.barrier
    Wm, K = args.warmup, args.steps
    for i in range(Wm):
        device_step(i)
    barrier()
    clocks = ClockSampler(local_rank) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(Wm, Wm + K):
        slot = device_step(i)
    runner.join()             # the last batch's link scorer runs on the copy-out stream
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    eng.check_errors()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, runner.d_out[slot])
    ms = max_over_ranks(ms, world, dev)
    value = world * K * B / (ms * 1e-3)

    # ---- e2e: pinned host buffers -> H2D -> graph -> D2H of scores + loss, every step ----
    e2e = None
    if not args.no_e2e:
        eng.reset()
        cols = lambda j: (host_in[j, :B], host_in[j, B:2 * B], host_in[j, 2 * B:3 * B],
                          host_in[j, 4 * B:].view(np.float64), host_in[j, 3 * B:4 * B])
        slots = []
        for i in range(Wm):
            slots.append(runner.submit_host(*cols(i % avail)))
            if len(slots) >= runner.n_slots:
                runner.wait(slots.pop(0))
        while slots:
            runner.wait(slots.pop(0))
        barrier()
        checksum = 0.0
        t0 = time.perf_counter()
        pending = []
        for i in range(Wm, Wm + K):
            j = i % avail
            if j == 0:
                eng.reset()
            pending.append(runner.submit_host(*cols(j)))
            if len(pending) >= runner.n_slots:
                checksum += float(runner.wait(pending.pop(0))[2])   # the step's loss, read on the host
        while pending:
            checksum += float(runner.wait(pending.pop(0))[2])
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dt = max_over_ranks(dt, world, dev)
        eng.check_errors()
        e2e = {'value': world * K * B / dt, 'unit': UNIT, 'h2d_bytes_per_step': runner.h2d_bytes_per_step,
               'd2h_bytes_per_step': runner.d2h_bytes_per_step, 'ms_per_step': dt / K * 1e3,
               'mean_loss': checksum / K}
    clk = clocks.stop() if clocks is not None else None

    # ---- per-kernel CUDA-event breakdown (eager launches, same stream, same state progression) ----
    roofline, kernels = None, None
    if rank == 0 and args.profile_steps > 0:
        kernels, counters = profile_kernels(args, eng, dev_in, avail, csr)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except OSError:
            pass
        peak = float(peaks.get('hbm_gbs', 6650.0))
        top = max(kernels, key=lambda k: kernels[k]['us'])
        for k, v in kernels.items():
            v['bytes'] = int(algorithmic_bytes(k, counters, d, de, eng.M, B, K_NEIGH))
            v['gbs'] = v['bytes'] / (v['us'] * 1e-6) / 1e9 if v['us'] > 0 else 0.0
        traffic = None
        tf = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tf):
            traffic = json.load(open(tf)).get(args.workload, {}).get(top)
        roofline = {'bound': 'hbm', 'kernel': top, 'achieved': kernels[top]['gbs'], 'peak': peak, 'unit': 'GB/s',
                    'frac': kernels[top]['gbs'] / peak, 'traffic': traffic,
                    'peak_source': 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback',
                    'launch_us': kernels[top]['us'], 'bytes_per_launch': kernels[top]['bytes'],
                    'counters': counters,
                    'note': 'entry-point granularity (CUDA events around the C-ABI call, eager launches); at batch 200 '
                            'every kernel is latency bound - see bench.py --micro for the HBM fractions at 256k rows'}
        # K7: the seq restarter's dense products (q/k in-projection of R x L tokens, value / out / out_fn / merger
        # products of R rows) - the dominant entry point of the seq-restarter configurations
        sg = kernels.get('tiger_sgemm_nt')
        if rst == 'seq' and sg:
            dm, L = 4 * d + de, HIST_LEN
            flops = counters['R'] * 2.0 * (L * dm * 2 * dm + 2 * dm * dm + dm * d + 2 * d * d)
            tf32_peak = float(peaks.get('bf16_tflops', 1590.0)) / 2.0
            sg['tensor'] = {'bound': 'tensor', 'useful_tflops': flops / (sg['us'] * 1e-6) / 1e12,
                            'issued_tflops': 3.0 * flops / (sg['us'] * 1e-6) / 1e12, 'peak': tf32_peak, 'unit': 'TFLOP/s',
                            'frac': 3.0 * flops / (sg['us'] * 1e-6) / 1e12 / tf32_peak, 'restarted_nodes_per_batch': counters['R'],
                            'note': 'seq restarter (K7): 7 launches per batch on ~R x 40 tokens; latency bound at this '
                                    'size (54 dependent k-steps per product), see profiles/r02_launches_wikipedia_infer.md'}
            if top == 'tiger_sgemm_nt':
                roofline = {'bound': 'tensor', 'kernel': top, 'achieved': sg['tensor']['issued_tflops'], 'peak': tf32_peak,
                            'unit': 'TFLOP/s', 'frac': sg['tensor']['frac'], 'traffic': None,
                            'peak_source': 'half of the measured bf16 GEMM peak (tf32 runs at half the bf16 rate)',
                            'launch_us': sg['us'], 'launches_per_step': sg['launches_per_step'], 'flops_per_step': flops,
                            'counters': counters,
                            'note': 'entry-point granularity (CUDA events around the eager C-ABI calls); issued = 3 x useful '
                                    'flops (tf32x3)'}
        # the dense kernel of the path: GRU gate GEMM on the tensor cores (tf32x3: 3 MMAs per useful product)
        g = kernels.get('tiger_gru_update')
        if g:
            flops = 2.0 * counters['O'] * (eng.M + d) * 3 * d
            tf32_peak = float(peaks.get('bf16_tflops', 1590.0)) / 2.0
            g['tensor'] = {'bound': 'tensor', 'useful_tflops': flops / (g['us'] * 1e-6) / 1e12,
                           'issued_tflops': 3.0 * flops / (g['us'] * 1e-6) / 1e12, 'peak': tf32_peak, 'unit': 'TFLOP/s',
                           'frac': 3.0 * flops / (g['us'] * 1e-6) / 1e12 / tf32_peak,
                           'peak_source': 'half of the measured bf16 GEMM peak (tf32 runs at half the bf16 rate)'}

    # ---- parity inside the bench: the first batches after a reset, engine vs the CPU arm on the same inputs ----
    parity = None
    if arm is not None and args.parity_batches > 0:
        parity = check_parity(eng, arm, dev_in, args.parity_batches)

    # ---- CPU baseline: the reference on the host cores, bounded sample, rank 0 at N=1 (+ the oracle port) ----
    cpu = None
    if arm is not None:
        first = args.parity_batches if parity is not None else 0
        n, dt = arm.time(first, min(args.cpu_batches, avail - first - 4), args.cpu_seconds)
        cpu = {'value': n * B / dt, 'unit': UNIT, 'cores': arm.cores, 'kind': arm.kind,
               'sample': arm.describe(n, first + 2), 'ms_per_step': dt / n * 1e3}
        if arm.kind == 'reference' and st.efeats is not None:
            port = CpuArm(args, shape, st, neg, lo, first + n + 4, kind='port')
            n2, dt2 = port.time(first, n, args.cpu_seconds)
            cpu['port'] = {'value': n2 * B / dt2, 'unit': UNIT, 'cores': port.cores, 'kind': 'port',
                           'sample': port.describe(n2, first + 2), 'ms_per_step': dt2 / n2 * 1e3}

    # ---- the training step of the same configuration (DDP at N > 1: gradient all-reduce inside the timed region) ----
    train_step = None
    if args.train_steps > 0:
        del runner
        t = measure_train(args, wl, args.train_steps, min(Wm, 10), parity=False, cpu=False, e2e=False, profile_steps=0)
        train_step = {'metric': METRIC_TRAIN, 'value': t['value'], 'unit': UNIT, 'ms_per_step': t['ms_per_step'],
                      'n_gpus': world, **t['train']}

    if rank == 0:
        line = {
            'metric': metric_name(args), 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': Wm,
            'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(args, shape, st, world),
            'e2e': e2e, 'gpu_launches': eng.launches_per_step() * K, 'clocks': clk, 'roofline': roofline,
            'cpu_baseline': cpu, 'parity_checked': bool(parity), 'parity': parity, 'train_step': train_step,
            'kernels': kernels,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
# B200 arm, training step (--mode train): forward + hand-written backward + [gradient all-reduce] + Adam
# ------------------------------------------------------------------------------------------
def train_flops(c, d, de, B, K, L, seq):
    """Algorithmic flops of the dense products of one training step (forward; backward = 2x for layers whose input
    needs a gradient, 1x for the GRU whose inputs are buffers); c = mean device counters."""
    M, E, C, dm = 3 * d + de, 2 * d, 2 * d + de, 4 * d + de
    gru = 2.0 * c['O'] * 3 * d * (M + d)
    attn = 2.0 * 3 * B * (E * E + K * C * 2 * E + E * E + (E + d) * d + d * d)
    score = 2.0 * 2 * B * (2 * d * d)
    fwd_bwd = 2 * gru + 3 * attn + 3 * score
    if seq:
        per_node = 2.0 * (L * dm * 2 * dm + 2 * dm * dm + dm * d + 2 * d * d)
        fwd_bwd += 3 * c['P'] * per_node + c['R'] * per_node
    return fwd_bwd


def run_train(args):
    """One step = the loop body of train_self_supervised_ddp.py:186-214 for one batch of 200 events: neighbor finder,
    lazy restart of not-yet-seen nodes, contrast_and_mutual_learning forward, backward, gradient all-reduce over NCCL
    (N > 1; one bucket = the flat gradient buffer, 1/N folded into the optimizer), Adam.  lr = 1e-4 * sqrt(N) (:146)."""
    import torch.distributed as dist
    wl = DeviceWorkload(args, mode='train')
    r = measure_train(args, wl, args.steps, args.warmup, parity=True, cpu=True, e2e=not args.no_e2e,
                      profile_steps=args.profile_steps)
    if wl.rank == 0:
        line = {
            'metric': metric_name(args), 'value': r['value'], 'unit': UNIT, 'n_gpus': wl.world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args, wl.shape, wl.st, wl.world),
            'e2e': r['e2e'], 'gpu_launches': r['gpu_launches'], 'clocks': r['clocks'], 'roofline': r['roofline'],
            'cpu_baseline': r['cpu_baseline'], 'parity_checked': bool(r['parity']), 'parity': r['parity'],
            'train': r['train'], 'kernels': r['kernels'],
        }
        print(json.dumps(line))
    if wl.world > 1:
        dist.destroy_process_group()


def measure_train(args, wl, steps, warmup, *, parity, cpu, e2e, profile_steps):
    import torch
    import torch.distributed as dist
    from www2023tiger_b200 import train as T, train_seq as TS, ops
    from www2023tiger_b200.init import build_model
    from www2023tiger_b200.tiger.data.graph import Graph

    rank, world, dev = wl.rank, wl.world, wl.dev
    shape, st, rst, arm, dev_in, host_in, avail, lo = wl.shape, wl.st, wl.rst, wl.arm, wl.dev_in, wl.host_in, wl.avail, wl.lo
    B, d, de = BATCH, wl.d, wl.de
    torch.manual_seed(args.seed)
    graph = Graph.from_csr(wl.csr)
    model = build_model(None, wl.efeats, graph, wl.N, st.n_events, dev, dim=shape.dim, n_layers=1, n_heads=N_HEAD,
                        n_neighbors=K_NEIGH, hit_type='bin', dropout=0.1, restarter_type=rst, hist_len=HIST_LEN,
                        msg_src=shape.msg_src, upd_src=shape.upd_src)
    if arm is not None and arm.kind == 'reference':
        res = model.load_state_dict(arm.weights(), strict=False)
        assert not res.unexpected_keys, res.unexpected_keys
    if world > 1:                                  # DDP broadcasts rank 0's parameters at construction (:145)
        for p in model.parameters():
            dist.broadcast(p.data, 0)
    model.train()
    lr = 1e-4 * math.sqrt(world)
    tr = model.native_trainer(B, lr=lr, seed=args.seed)
    tr.attach_stream(wl.csr, HIST_LEN)
    losses = torch.zeros(2, device=dev)
    comm_bytes = tr.fp.grad_all.numel() * 4 if world > 1 else 0

    allreduce = (lambda t: dist.all_reduce(t, async_op=True)) if world > 1 else None

    def device_step(i):
        j = i % avail
        if j == 0 and i > 0:
            tr.reset_stream()                      # epoch boundary: the window wraps (model.reset(), :176)
        closs, mloss = tr.step_stream(dev_in[j], mutual_coef=1.0, grad_scale=1.0 / world, allreduce=allreduce)
        losses[0:1].add_(closs)
        losses[1:2].add_(mloss)

    # ---- parity: the first training steps from a reset, dropout off on both sides, against the reference's loop body
    par = None
    if parity and arm is not None and args.parity_batches > 0 and arm.kind == 'reference':
        par = check_train_parity(args, wl, model, tr)
    # The step is replayed as one CUDA graph (the eager step is bound by the host's ~80-140 Python -> C calls); at N > 1 the
    # three gradient all-reduce slices are captured with it (NCCL through torch.distributed is capturable).
    # TIGER_TRAIN_EAGER=1 keeps eager launches.  A capture that fails on any rank puts every rank back on eager launches.
    graphed = os.environ.get('TIGER_TRAIN_EAGER') != '1'
    graph_error = None
    if graphed:
        tr.reset_stream()
        tr.capture_stream(mutual_coef=1.0, grad_scale=1.0 / world, allreduce=allreduce)
        try:
            for i in range(3):                     # two eager steps + the capture, off the clock
                device_step(i)
            torch.cuda.synchronize()
        except Exception as e:                     # noqa: BLE001 - reported in the JSON line, eager launches take over
            graph_error = f'{type(e).__name__}: {e}'[:300]
        ok = torch.tensor([0.0 if graph_error else 1.0], device=dev)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if float(ok) < 1.0:
            graphed = False
            graph_error = graph_error or 'capture failed on another rank'
            tr.release_graph()
            print(f'[bench] CUDA-graph capture of the training step failed ({graph_error}); eager launches', file=sys.stderr)
    tr.reset_stream()
    Wm, K = warmup, steps
    for i in range(Wm):
        device_step(i)
    wl.barrier()
    clocks = ClockSampler(wl.local_rank) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    losses.zero_()
    ev0.record()
    t_host = time.perf_counter()
    for i in range(Wm, Wm + K):
        device_step(i)
    host_ms = (time.perf_counter() - t_host) / K * 1e3      # host time to ISSUE one step (launches are asynchronous)
    ev1.record()
    wl.barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1), world, dev)
    tr.check_errors()
    value = world * K * B / (ms * 1e-3)
    if world > 1 and os.environ.get('TIGER_BENCH_DDP_EXP') == '1':
        # experiment (stderr only): where the multi-rank step time goes - no collective / one bucket / three slices
        for name, ar, sliced in (('no all-reduce', None, True), ('one bucket after backward', allreduce, False),
                                 ('three slices (default)', allreduce, True)):
            tr.reset_stream()
            for i in range(Wm + K):
                if i == Wm:
                    wl.barrier()
                    ev0.record()
                tr.step_stream(dev_in[i % avail], mutual_coef=1.0, grad_scale=1.0 / world, allreduce=ar, sliced=sliced)
            ev1.record()
            wl.barrier()
            own = ev0.elapsed_time(ev1) / K
            worst = max_over_ranks(ev0.elapsed_time(ev1), world, dev) / K
            print(f'[ddp-exp] rank {rank} {name}: own {own:.3f} ms/step, slowest rank {worst:.3f}', file=sys.stderr, flush=True)
    if world > 1:
        dist.all_reduce(losses)                    # the reference all-reduces its loss scalars (:209-211)
    mean_losses = (losses / (K * world)).cpu().tolist()

    # ---- e2e: the batch record comes from pinned host memory every step, the two losses go back to the host ----
    e2e_out = None
    if e2e:
        tr.reset_stream()
        pin = [torch.empty(5 * B, dtype=torch.int64).pin_memory() for _ in range(4)]
        d_in = [torch.empty(5 * B, dtype=torch.int64, device=dev) for _ in range(4)]
        h_out = torch.empty(K + Wm, 2).pin_memory()
        copied = [None] * 4
        wl.barrier()
        t0 = None
        for i in range(Wm + K):
            if i == Wm:
                wl.barrier()
                t0 = time.perf_counter()
            sl = i % 4
            if copied[sl] is not None:
                copied[sl].synchronize()            # the slot's previous upload has left the pinned buffer
            pin[sl].numpy()[:] = host_in[i % avail]
            d_in[sl].copy_(pin[sl], non_blocking=True)
            copied[sl] = torch.cuda.Event()
            copied[sl].record()
            j = i % avail
            if j == 0 and i > 0:
                tr.reset_stream()
            closs, mloss = tr.step_stream(d_in[sl], mutual_coef=1.0, grad_scale=1.0 / world, allreduce=allreduce)
            h_out[i, 0:1].copy_(closs, non_blocking=True)
            h_out[i, 1:2].copy_(mloss, non_blocking=True)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0, world, dev)
        tr.check_errors()
        e2e_out = {'value': world * K * B / dt, 'unit': UNIT, 'h2d_bytes_per_step': 5 * B * 8, 'd2h_bytes_per_step': 8,
                   'ms_per_step': dt / K * 1e3, 'mean_loss': float(h_out[Wm:].sum(1).mean())}
    clk = clocks.stop() if clocks is not None else None

    # ---- per-entry-point CUDA-event breakdown + launch count ----
    kernels, roofline, launches = None, None, None
    tr.release_graph()
    if rank == 0 and profile_steps > 0:
        from www2023tiger_b200 import _lib
        tr.reset_stream()
        records = []
        orig = _lib.call

        def timed_call(name, *a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            orig(name, *a)
            e1.record()
            records.append((name, e0, e1))
        n_steps = min(profile_steps, avail)
        warm = min(10, n_steps // 2)
        counts = []
        ops.call = T.call = TS.call = timed_call
        try:
            for i in range(n_steps):
                if i == warm:
                    torch.cuda.synchronize()
                    records.clear()
                    counts.clear()
                # rank 0 alone runs this breakdown: no collective here (the other ranks have left the loop)
                tr.step_stream(dev_in[i], mutual_coef=1.0, grad_scale=1.0 / world, allreduce=None)
                counts.append(torch.cat([tr.counts[:3].long(), tr.t_count.long()]))
        finally:
            ops.call = T.call = TS.call = orig
        torch.cuda.synchronize()
        agg = {}
        for name, e0, e1 in records:
            agg.setdefault(name, []).append(e0.elapsed_time(e1) * 1e3)
        n = n_steps - warm
        kernels = {k: {'us': float(np.sum(v)) / n, 'launches_per_step': len(v) / n} for k, v in agg.items()}
        launches = sum(v['launches_per_step'] for v in kernels.values())
        U, O_, R, P = (float(x) for x in torch.stack(counts).double().mean(0).cpu())
        counters = {'U': U, 'O': O_, 'R': R, 'P': P}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except OSError:
            pass
        flops = train_flops(counters, d, de, B, K_NEIGH, HIST_LEN, rst == 'seq')
        dense = [kernels[k] for k in ('tiger_sgemm_ex', 'tiger_sgemm_pp', 'tiger_gemm_pp_pack') if k in kernels]
        g = {'us': sum(x['us'] for x in dense), 'launches_per_step': sum(x['launches_per_step'] for x in dense)} if dense else None
        tf32_peak = float(peaks.get('bf16_tflops', 1590.0)) / 2.0
        if g:
            ach = 3.0 * flops / (g['us'] * 1e-6) / 1e12
            roofline = {'bound': 'tensor', 'kernel': 'tiger_sgemm_ex + tiger_sgemm_pp (+ tiger_gemm_pp_pack)', 'achieved': ach, 'peak': tf32_peak, 'unit': 'TFLOP/s',
                        'frac': ach / tf32_peak, 'traffic': None, 'useful_tflops': ach / 3.0, 'launch_us': g['us'],
                        'launches_per_step': g['launches_per_step'], 'flops_per_step': flops, 'counters': counters,
                        'peak_source': 'half of the measured bf16 GEMM peak (tf32 runs at half the bf16 rate)'
                        if peaks else 'fallback',
                        'note': 'all tensor-core products of the step (forward, input and weight gradients) together: '
                                'issued = 3 x useful flops (tf32x3); entry-point granularity: CUDA events around the '
                                'eager C-ABI calls include the launch gaps between them - profiles/ holds the ncu launch '
                                'list with the kernel durations'}

    # ---- CPU baseline: the reference's training loop body on the host cores ----
    cpu_out = None
    if cpu and arm is not None:
        if arm.kind == 'reference':
            arm.ref.reset(train=True)
        n, dt = arm.time(0, min(args.cpu_batches, avail - 4), args.cpu_seconds, warmup=1)
        cpu_out = {'value': n * B / dt, 'unit': UNIT, 'cores': arm.cores, 'kind': arm.kind, 'sample': arm.describe(n, 1),
                   'ms_per_step': dt / n * 1e3}
    return {'value': value, 'ms_per_step': ms / K, 'e2e': e2e_out, 'gpu_launches': int(round((launches or 0) * K)),
            'clocks': clk, 'roofline': roofline, 'cpu_baseline': cpu_out, 'parity': par, 'kernels': kernels,
            'train': {'lr': lr, 'optimizer': 'Adam (flat buffer, per-tensor step counters)', 'params': tr.fp.numel,
                      'allreduce_bytes_per_step': comm_bytes, 'host_issue_ms_per_step': host_ms, 'cuda_graph': graphed, 'cuda_graph_error': graph_error, 'mean_contrast_loss': mean_losses[0],
                      'mean_mutual_loss': mean_losses[1], 'dropout': 0.1, 'steps': K}}


def check_train_parity(args, wl, model, tr):
    """First training steps after a reset, dropout off on both sides (masks are not reproducible across
    implementations): losses of every step must agree with the reference's loop body within 1e-5 / 2e-5, and because
    step k + 1 runs on the parameters Adam produced from step k's gradients, backward and optimizer are covered too."""
    import torch
    from oracle import ref_harness
    n = args.parity_batches
    ref = ref_harness.ReferenceRunner(wl.st if wl.st.efeats is not None else wl.arm.ref.st, wl.neg,
                                      restarter=wl.rst, msg_src=wl.shape.msg_src, upd_src=wl.shape.upd_src,
                                      n_graph_events=wl.lo + (n + 1) * BATCH, n_neighbors=K_NEIGH, n_heads=N_HEAD,
                                      hist_len=HIST_LEN, batch=BATCH, seed=args.seed, dropout=0.0)
    ref.reset(train=True)
    saved = {k: v.clone() for k, v in tr.fp.p.items()}
    keep = (tr.p_attn, tr.p_score)
    tr.p_attn = tr.p_score = 0.0
    if tr.rkind == 'seq':
        p_seq, tr.seq.p = tr.seq.p, 0.0
    tr.reset_stream()
    worst = [0.0, 0.0]
    for j in range(n):
        c, m = tr.step_stream(wl.dev_in[j], mutual_coef=1.0)
        rc, rm = ref.train_step(wl.lo + j * BATCH, lr=tr.lr)
        torch.cuda.synchronize()
        tr.check_errors()
        e_c = abs(float(c) - rc) / max(abs(rc), 1e-30)
        e_m = abs(float(m) - rm) / max(abs(rm), 1e-30)
        if os.environ.get('TIGER_DEBUG_PARITY') == '1':
            sd = ref.model.state_dict()
            rows = []
            for k, v in tr.fp.p.items():
                dv = (v.detach().cpu() - sd[k]).abs()
                rows.append((float(dv.max()) / tr.lr, k, float(dv.mean()) / tr.lr))
            rows.sort(reverse=True)
            print(f'[parity debug] step {j}: contrast {float(c):.7f} vs {rc:.7f}, mutual {float(m):.7f} vs {rm:.7f}; '
                  f'parameter deviation in units of lr (max, mean):', file=sys.stderr)
            for r in rows[:8]:
                print(f'    {r[1]:60s} {r[0]:10.4f} {r[2]:10.6f}', file=sys.stderr)
        worst = [max(worst[0], e_c), max(worst[1], e_m)]
        # steps 0-1 pin the forward and the first update; from then on Adam's normalisation (update ~ lr * sign(g)
        # for a tensor's first gradients) amplifies fp32 round-off in near-zero gradient entries: single weights move
        # by +-lr instead of ~0 and the trajectories separate slowly (torch on a GPU does the same against itself)
        tol_c, tol_m = (1e-5, 5e-5) if j < 2 else (1e-3, 1e-3)
        if e_c > tol_c or e_m > tol_m:
            raise SystemExit(f'train parity: step {j} contrast {float(c):.7f} vs {rc:.7f} ({e_c:.1e}), '
                             f'mutual {float(m):.7f} vs {rm:.7f} ({e_m:.1e})')
    # back to the initial parameters / optimizer state for the timed run
    for k, v in saved.items():
        tr.fp.p[k].copy_(v)
    tr.fp.reset_optimizer()
    tr.p_attn, tr.p_score = keep
    if tr.rkind == 'seq':
        tr.seq.p = p_seq
    return {'against': 'reference', 'steps': n, 'what': 'contrast and mutual loss of consecutive optimisation steps '
            '(forward + backward + Adam), dropout 0 on both sides', 'contrast_rel': worst[0], 'mutual_rel': worst[1],
            'tol': 'steps 0-1: 1e-5 / 5e-5; later steps: 1e-3 (Adam amplifies fp32 round-off of near-zero gradients)'}


def check_parity(eng, arm, dev_in, n_batches):
    """Replays the first `n_batches` batches of the window from a reset state through the engine (eager launches)
    and through the CPU arm, which runs with the same parameters: neighbor tables and argmax-by-timestamp winners
    must be bit-identical, scores and loss within 1e-5 (max-norm, the tolerance BASELINE.json states).  Raises on
    a mismatch - a fast wrong kernel must not produce a bench line."""
    import torch
    eng.reset()
    B = eng.B
    worst = {'scores': 0.0, 'loss': 0.0}
    for j in range(n_batches):
        eng.inp.copy_(dev_in[j])
        eng.step()
        torch.cuda.synchronize()
        eng.check_errors()
        ref = arm.step(j)
        if not np.array_equal(eng.neigh_nids.cpu().numpy(), ref['neigh_nids']):
            raise SystemExit(f'parity: neighbor table of batch {j} differs from the {arm.kind}')
        got = np.flatnonzero(eng.winner.cpu().numpy())
        if not np.array_equal(got, np.sort(ref['winner_index'])):
            raise SystemExit(f'parity: argmax-by-timestamp winners of batch {j} differ from the {arm.kind}')
        out = eng.out_buf.cpu().numpy()
        want = np.concatenate([ref['pos_scores'], ref['neg_scores']])
        e_s = float(np.abs(out[:2 * B] - want).max() / max(np.abs(want).max(), 1e-30))
        e_l = abs(float(out[2 * B]) - ref['loss']) / max(abs(ref['loss']), 1e-30)
        worst['scores'], worst['loss'] = max(worst['scores'], e_s), max(worst['loss'], e_l)
        if e_s > 1e-5 or e_l > 1e-5:
            raise SystemExit(f'parity: batch {j} scores {e_s:.2e} / loss {e_l:.2e} exceed 1e-5 vs the {arm.kind}')
    eng.reset()
    return {'against': arm.kind, 'batches': n_batches, 'neighbor_tables': 'bit-identical',
            'winners': 'bit-identical', 'scores_max_rel': worst['scores'], 'loss_rel': worst['loss'], 'tol': 1e-5}


def st_fits_host(args):
    return args.workload != 'scaled'


def profile_kernels(args, eng, dev_in, avail, csr):
    """Eager pass with a CUDA-event pair around every C-ABI launch; returns mean us per entry point and
    the mean device counters the algorithmic-byte formulas need."""
    import torch
    from www2023tiger_b200 import _lib
    eng.reset()
    records = []
    orig_call = _lib.call

    def timed_call(name, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_call(name, *a)
        e1.record()
        records.append((name, e0, e1))

    from www2023tiger_b200 import ops
    n_steps = min(args.profile_steps, avail)
    warm = min(20, n_steps // 2)
    counts = []
    ops.call = timed_call
    try:
        for i in range(n_steps):
            if i == warm:
                torch.cuda.synchronize()
                records.clear()
                counts.clear()
            eng.inp.copy_(dev_in[i], non_blocking=True)
            eng.step()
            persisted = (eng.winner.bool() & (eng.gru_row[eng.pos] >= 0)).sum()
            counts.append(torch.cat([eng.counts[:3].long(), eng.winner.sum().reshape(1), persisted.reshape(1)]))
    finally:
        ops.call = orig_call
    torch.cuda.synchronize()
    agg = {}
    for name, e0, e1 in records:
        agg.setdefault(name, []).append(e0.elapsed_time(e1) * 1e3)
    n = n_steps - warm
    kernels = {k: {'us': float(np.sum(v)) / n, 'launches_per_step': len(v) / n} for k, v in agg.items()}
    U, O_, R, P, Po = (float(x) for x in torch.stack(counts).double().mean(0).cpu())
    deg = float(csr.indptr[1:].sub(csr.indptr[:-1]).float().mean().item())
    counters = {'U': U, 'O': O_, 'R': R, 'P': P, 'Po': Po,
                'log_deg': max(1.0, math.log2(max(deg, 2.0))), 'bitmap_words': (eng.N + 31) // 32}
    return kernels, counters


# ------------------------------------------------------------------------------------------
# micro mode: HBM fraction of the gather / scatter / search kernels at sizes that leave the L2
# ------------------------------------------------------------------------------------------
def run_micro(args):
    """At batch 200 the whole path moves ~17 MB per step, so every kernel is launch / latency bound in
    situ.  What the gather/scatter kernels can do is measured here: each one is fed `--micro-rows` rows out
    of tables far larger than the 126 MB L2 (scaled-config shapes: 1M-node tables, d = de = 172), timed
    with CUDA events over 20 launches after 3 warm-ups, against the measured HBM peak."""
    import torch
    from www2023tiger_b200 import _lib, ops
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --micro needs a CUDA device')
    torch.cuda.set_device(0)
    dev = torch.device('cuda', 0)
    _lib.load()
    try:
        peak = float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['hbm_gbs'])
        peak_src = 'measured (MEASURED_PEAKS.json)'
    except (OSError, KeyError):
        peak, peak_src = 6650.0, 'fallback'
    g = torch.Generator(device=dev).manual_seed(args.seed)
    N, d, de, R, K = 1_000_001, 172, 172, args.micro_rows, K_NEIGH
    M = 3 * d + de
    f32, i64 = torch.float32, torch.int64
    table = torch.randn(N, d, device=dev, generator=g)
    table2 = torch.randn(N, d, device=dev, generator=g)
    ts_table = torch.zeros(N, device=dev)
    active = torch.zeros(N, dtype=torch.uint8, device=dev)
    perm = torch.randperm(N - 1, device=dev, generator=g)[:2 * R] + 1          # distinct node ids, no padding id
    ids = perm[:R].contiguous()
    vals = torch.randn(R, d, device=dev, generator=g)
    ts_r = torch.rand(R, device=dev, generator=g) * 1e6 + 1.0
    results = {}

    def timed(name, fn, nbytes, n=20, warm=3, note=''):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / n * 1e3
        gbs = nbytes / (us * 1e-6) / 1e9
        results[name] = {'us': us, 'bytes': int(nbytes), 'gbs': gbs, 'frac_of_peak': gbs / peak, 'rows': R, 'note': note}

    # Memory.get / Memory.set (memory.py:36-52): row gather / scatter of d floats (+ update_ts)
    timed('tiger_gather_rows', lambda: ops.gather_rows(table, ids, ts_table), R * (2 * d * 4 + 8 + 8),
          note='Memory.get: R random rows of a 688 MB table -> dense [R, d]')
    timed('tiger_scatter_rows', lambda: ops.scatter_rows(table, ids, vals, ts_table=ts_table, ts=ts_r, active=active),
          R * (2 * d * 4 + 8 + 9), note='Memory.set: dense [R, d] -> R random rows')
    # store_events (tiger.py:422-442, memory.py:77-106): 2R message rows of M floats, all positions winners
    B = R // 2
    src, dst = perm[:B].contiguous(), perm[B:2 * B].contiguous()
    n_e = 4_000_000
    efeats = torch.randn(n_e + 1, de, device=dev, generator=g)
    eids = torch.randint(1, n_e + 1, (B,), device=dev, generator=g)
    ev_ts = torch.rand(B, device=dev, generator=g) * 1e6 + 2e6
    winner = torch.ones(2 * B, dtype=torch.uint8, device=dev)
    msg_vals = torch.empty(N, M, device=dev)
    msg_ts = torch.zeros(N, device=dev)
    has_msg = torch.zeros(N, dtype=torch.uint8, device=dev)
    time_w = torch.from_numpy((1 / 10 ** np.linspace(0, 9, d)).astype(np.float32)).to(dev)
    time_b = torch.zeros(d, device=dev)

    def store():
        has_msg.zero_()
        ops.store_messages(src, dst, eids, ev_ts, winner, table, ts_table, None, efeats, d, de, time_w, time_b,
                           msg_vals, msg_ts, has_msg)
    timed('tiger_store_messages', store, 2 * B * ((2 * d + de) * 4 + M * 4 + 8 + 13) + N,
          note='2R message rows [mem(self) | mem(other) | efeat | time code] built in the table (incl. the has_msg clear)')
    # write-backs (tiger.py:396-420)
    pos = torch.cat([src, dst])
    gru_row = torch.full((N,), -1, dtype=torch.int32, device=dev)
    gru_row[pos] = torch.arange(2 * B, dtype=torch.int32, device=dev)
    h_new = torch.randn(2 * B, d, device=dev, generator=g)

    def right():
        has_msg.fill_(1)
        ops.right_writeback(pos, winner, gru_row, h_new, d, table2, ts_table, active, msg_ts, has_msg)
    timed('tiger_right_writeback', right, 2 * B * (2 * d * 4 + 8 + 4 + 10) + N,
          note='2R GRU rows persisted into the right memory (incl. the has_msg fill)')
    h_left = torch.randn(3 * B, d, device=dev, generator=g)
    left_ts = torch.zeros(N, device=dev)
    timed('tiger_left_writeback',
          lambda: ops.left_writeback(pos, B, winner, h_left, d, ev_ts, table, left_ts, active),
          2 * B * (2 * d * 4 + 8 + 4 + 6), note='2R embedding rows persisted into the left memory')
    # GRU update (update_modules.py:30-37 behind tiger.py:331-345): R outdated nodes, message + memory rows gathered
    # from the 1M-row tables.  688 + 172 -> 516 gate pre-activations per row: at this size the kernel is bound by the
    # tensor pipe (tf32x3), reported beside the HBM figure.
    from www2023tiger_b200.init import random_weights
    try:
        tpeak = float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['bf16_tflops']) / 2
    except (OSError, KeyError):
        tpeak = 1100.0
    W = {k: v.to(dev) for k, v in random_weights(d, de, seed=args.seed).items()}
    c = 'right_mem_updater.cell.'
    gpack = ops.GruPack(W[c + 'weight_ih'], W[c + 'weight_hh'], W[c + 'bias_ih'], W[c + 'bias_hh'])
    gru_out = torch.empty(R, d, device=dev)
    timed('tiger_gru_update', lambda: ops.gru_update(gpack, node_ids=ids, x_table=msg_vals, h_table=table, n_rows=R,
                                                    out=gru_out),
          R * ((M + 2 * d) * 4 + 8), note='R rows: message row (M floats) + memory row gathered by node id, h_new written')
    fl = 2.0 * R * 3 * d * (M + d)
    t = results['tiger_gru_update']
    t['tensor'] = {'useful_tflops': fl / (t['us'] * 1e-6) / 1e12, 'issued_tflops': 3 * fl / (t['us'] * 1e-6) / 1e12,
                   'peak': tpeak, 'frac': 3 * fl / (t['us'] * 1e-6) / 1e12 / tpeak,
                   'peak_source': 'half of the measured bf16 GEMM peak (tf32 runs at half the bf16 rate); tf32x3 issues 3 MMAs per product'}
    # temporal attention (temporal_agg_modules.py:29-83,210-235): Q queries x K neighbors gathered from the 1M-row
    # memory and the 4M-row edge-feature table, folded projections, softmax pooling, merger
    Q = max(R // 4, 1024)
    apack = ops.AttnPack(d, de, dev, 2)
    a = 'temporal_embedding_fn.fns.0.'
    apack.refresh(W[a + 'mha_fn.q_proj_weight'], W[a + 'mha_fn.k_proj_weight'], W[a + 'mha_fn.v_proj_weight'],
                  W[a + 'mha_fn.in_proj_bias'], W[a + 'mha_fn.out_proj.weight'], W[a + 'mha_fn.out_proj.bias'],
                  W[a + 'merger.fc1.weight'], W[a + 'merger.fc1.bias'], W[a + 'merger.fc2.weight'], W[a + 'merger.fc2.bias'],
                  W['time_encoder.basis_freq'], W['time_encoder.phase'])
    centers = torch.randint(1, N, (Q,), device=dev, generator=g)
    q_ts = torch.rand(Q, device=dev, generator=g) * 1e6 + 2e6
    nn_ids = torch.randint(1, N, (Q, K), device=dev, generator=g)
    nn_eids = torch.randint(1, n_e + 1, (Q, K), device=dev, generator=g)
    nn_ts = q_ts[:, None] - torch.rand(Q, K, device=dev, generator=g) * 1e5
    att_out = torch.empty(Q, d, device=dev)
    timed('tiger_temporal_attention',
          lambda: ops.temporal_attention(apack, 2, centers, q_ts, nn_ids, nn_eids, nn_ts, rows_a=table2, rows_b=h_new,
                                         sel=gru_row, nfeats=None, efeats=efeats, out=att_out),
          Q * (d * 4 + 12 + K * ((d + de) * 4 + 20 + 4) + d * 4), n=10,
          note=f'{Q} queries x {K} neighbors: center row + K (memory row + edge-feature row + ids/ts + sel) gathered, [Q, d] written')
    results['tiger_temporal_attention']['rows'] = Q
    del apack, gpack
    del msg_vals, efeats
    # neighbor finder (graph.py:44-53,117-127): R queries over a 1M-node / 8M-event CSR
    from www2023tiger_b200.synthetic import StreamShape, make_stream
    st = make_stream(StreamShape('micro', 900000, 100000, 8_000_000, 0, d), seed=args.seed, n_events=8_000_000,
                     with_efeats=False)
    csr = ops.csr_build(torch.from_numpy(st.src).to(dev), torch.from_numpy(st.dst).to(dev),
                        torch.from_numpy(st.ts).to(dev), torch.from_numpy(st.eids).to(dev), N)
    q_n = torch.from_numpy(np.concatenate([st.src[-R // 2:], st.dst[-R // 2:]])).to(dev)
    q_t = torch.from_numpy(np.concatenate([st.ts[-R // 2:], st.ts[-R // 2:]])).to(dev)
    out = (torch.empty(R, K, dtype=i64, device=dev), torch.empty(R, K, dtype=i64, device=dev),
           torch.empty(R, K, dtype=f32, device=dev), None)
    deg = (csr.indptr[q_n + 1] - csr.indptr[q_n]).double().clamp(min=1)
    # timestamps probed by the 8-ary lower bound: 8 per round, never more than the segment itself
    rounds = (deg / 8).clamp(min=1).log2().div(3).ceil() + 1
    search = float(torch.minimum(deg, rounds * 8).mul(8).mean())
    kk = float(deg.clamp(max=K).mean())
    timed('tiger_find_recent', lambda: ops.find_recent(csr, q_n, q_t, K, out=out),
          R * (16 + 16 + search + kk * 17 + K * 20),
          note=f'R queries, mean degree {float(deg.mean()):.0f}: query + indptr + 8-ary lower bound + gather of the last K '
               f'entries (4+4+8+1 B) + [K] outputs (8+8+4 B)')
    src_d, dst_d = torch.from_numpy(st.src).to(dev), torch.from_numpy(st.dst).to(dev)
    ts_d, eid_d = torch.from_numpy(st.ts).to(dev), torch.from_numpy(st.eids).to(dev)
    E = st.n_events
    timed('tiger_csr_build', lambda: ops.csr_build(src_d, dst_d, ts_d, eid_d, N), 2 * E * (4 * 3 * 2 * 2 + 21) + E * 32,
          n=5, warm=1, note='8M events -> 16M CSR entries: LSD radix sort by owner (3 passes of key+value) + entry fill')
    line = {'metric': 'HBM GB/s of the gather/scatter/search kernels at >= 256k rows (micro mode)', 'unit': 'GB/s',
            'peak': peak, 'peak_source': peak_src, 'rows': R,
            'tables': f'{N} nodes x d={d} (688 MB per memory), message store {N} x {M}, 4M x {de} edge features',
            'micro': results}
    print(json.dumps(line))


def run_dropin(args):
    """`--api dropin`: what a user of the reference gets WITHOUT changing a line of their script - the mirror classes of
    www2023tiger_b200/tiger behind the reference's own loop `eval_edge_prediction(model, dl, device, restart_mode=True)`
    (eval_utils.py:15-68): per batch a DataLoader item list -> GraphCollator (device finder, host copy of the involved
    ids: the signature hands them to the driver) -> Python-set restart bookkeeping (`ts.min().item()`) -> TIGER.restart ->
    contrast_learning on the kernel route -> scores; AP / AUC with sklearn at the end.  Timed with the wall clock around
    the call (synchronised on both sides): there is no device-resident variant of this loop, so `value` repeats `e2e`."""
    import torch
    from torch.utils.data import DataLoader
    from www2023tiger_b200 import ops
    from www2023tiger_b200.init import build_model
    from www2023tiger_b200.tiger.data.data_loader import GraphCollator, InteractionData
    from www2023tiger_b200.tiger.data.graph import Graph
    from www2023tiger_b200.tiger.eval_utils import eval_edge_prediction

    wl = DeviceWorkload(args)
    if wl.world > 1:
        raise SystemExit('--api dropin is a single-process loop')
    st, neg, shape, rst, dev, lo, B = wl.st, wl.neg, wl.shape, wl.rst, wl.dev, wl.lo, BATCH
    Wm, K = args.warmup, args.steps
    if Wm + K > wl.avail:
        raise SystemExit(f'--warmup {Wm} + --steps {K} exceed the {wl.avail} batches of the stream window')
    graph = Graph.from_csr(wl.csr)
    torch.manual_seed(args.seed)
    model = build_model(None, wl.efeats, graph, wl.N, st.n_events, dev, dim=shape.dim, n_layers=1, n_heads=N_HEAD,
                        n_neighbors=K_NEIGH, hit_type='bin', dropout=0.1, restarter_type=rst, hist_len=HIST_LEN,
                        msg_src=shape.msg_src, upd_src=shape.upd_src)
    if wl.arm is not None and wl.arm.kind == 'reference':
        res = model.load_state_dict(wl.arm.weights(), strict=False)
        assert not res.unexpected_keys, res.unexpected_keys
    coll = GraphCollator(graph, K_NEIGH, 1, restarter=rst, hist_len=HIST_LEN)

    def loader(first, n):
        s = slice(lo + first * B, lo + (first + n) * B)
        data = InteractionData(st.src[s], st.dst[s], st.ts[s], st.eids[s], np.zeros(n * B, dtype=np.int64), seed=0,
                               eval=True, neg_dst=neg[s])
        return DataLoader(data, batch_size=B, collate_fn=coll)

    calls = [0]
    orig = ops.call

    def counted(name, *a):
        calls[0] += 1
        orig(name, *a)
    model.reset()
    seen = set()
    eval_edge_prediction(model, loader(0, Wm), dev, restart_mode=True, uptodate_nodes=seen)
    torch.cuda.synchronize()
    clocks = ClockSampler(wl.local_rank)
    ops.call = counted
    t0 = time.perf_counter()
    try:
        ap, auc = eval_edge_prediction(model, loader(Wm, K), dev, restart_mode=True, uptodate_nodes=seen)
        torch.cuda.synchronize()
    finally:
        ops.call = orig
    dt = time.perf_counter() - t0
    clk = clocks.stop()
    cpu = None
    if wl.arm is not None:
        n, dtc = wl.arm.time(0, min(args.cpu_batches, K), args.cpu_seconds)
        cpu = {'value': n * B / dtc, 'unit': UNIT, 'cores': wl.arm.cores, 'kind': wl.arm.kind,
               'sample': wl.arm.describe(n, 2), 'ms_per_step': dtc / n * 1e3}
    value = K * B / dt
    cfg = workload_config(args, shape, st, 1)
    cfg['api'] = "dropin: eval_edge_prediction(model, DataLoader(InteractionData, collate_fn=GraphCollator), restart_mode=True) on the tiger/ mirror"
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': 1, 'steps': K, 'warmup': Wm, 'ms_per_step': dt / K * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': cfg,
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 5 * B * 8, 'd2h_bytes_per_step': 2 * B * 4,
                    'note': 'wall clock around the reference-facing call; host collation, restart sets and AP / AUC included'},
            'gpu_launches': calls[0], 'clocks': clk, 'roofline': None, 'cpu_baseline': cpu, 'ap': ap, 'auc': auc}
    print(json.dumps(line))


def main():
    args = parse_args()
    if args.micro:
        run_micro(args)
    elif args.impl == 'reference':
        run_reference(args)
    elif args.mode == 'train':
        run_train(args)
    elif args.api == 'dropin':
        run_dropin(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
