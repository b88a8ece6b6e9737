#!/usr/bin/env python
"""Throughput of TigerEngine(n_chunks=M): M time chunks of the stream as one batched step on one GPU.

    python tools/bench_chunks.py [--workloads reddit,wikipedia] [--chunks 1,2,4,8,16] [--repeats 2]
                                 [--parent-tree DIR] [--out profiles/r07_chunks.json]

Every leg (workload, M) runs in its own process with bench.py's settings: the first 1000 batches skipped (at most half the stream), the rest of
the stream split into M contiguous chunks by the reference's ChunkSampler rule (engine.chunk_bounds), B = 200 events
per chunk and step, K = 10, the workload's restarter with lazy restart, every batch record resident in HBM,
StreamRunner graph replay fed by submit_device, CUDA events around enough timed steps for a window of at least
--min-window seconds (each chunk wraps to its start with a reset, as bench.py's window does).  A leg records events/s,
ms per step, the peak of torch's device allocator, and CUDA-event times per C-ABI entry point over eager steps.  The
largest M of each workload also replays its first --parity-batches steps against M independent engines (neighbor
tables bit-identical, scores and state slices within 1e-5).  With --parent-tree the default bench.py line runs on both
trees, alternated, with --dump-outputs, and the dumped arrays are compared.  The GPU's name and power limit are read
before and after.
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tools')]
from bench_layers import bench_args, gpu_info  # noqa: E402

STATE = ('left_vals', 'left_ts', 'left_active', 'right_vals', 'right_ts', 'right_active', 'msg_vals', 'msg_ts',
         'has_msg', 'uptodate')


def leg(workload, M, min_window, parity_batches):
    import torch
    from www2023tiger_b200 import _lib, ops
    from www2023tiger_b200.engine import StreamRunner, TigerEngine, chunk_bounds
    from www2023tiger_b200.init import random_weights
    bench, args = bench_args(ROOT, workload, 100, 20)
    wl = bench.DeviceWorkload(args)
    B, K, st = bench.BATCH, bench.K_NEIGH, wl.st
    skip = min(args.skip_batches, (st.n_events // B) // 2) * B      # bench.py's rule: at least half the stream left
    bounds = [(lo + skip, hi + skip) for lo, hi in chunk_bounds(st.n_events - skip, M, B, seed=args.seed)]
    n_rec = (bounds[0][1] - bounds[0][0]) // B
    idx = np.stack([np.arange(lo, lo + n_rec * B).reshape(n_rec, B) for lo, _ in bounds], 1)   # [step, chunk, event]
    W = random_weights(wl.d, wl.de, n_nodes=wl.N, restarter=wl.rst, hist_len=bench.HIST_LEN, seed=args.seed)
    kw = dict(n_nodes=wl.N, dim=wl.d, efeats=wl.efeats, n_neighbors=K, n_head=bench.N_HEAD, batch_size=B,
              msg_src=wl.shape.msg_src, upd_src=wl.shape.upd_src, restarter=wl.rst, hist_len=bench.HIST_LEN,
              lazy_restart=True, device=wl.dev)
    eng = TigerEngine(W, wl.csr, n_chunks=M, **kw)
    records = eng.device_records(st.src[idx], st.dst[idx], wl.neg[idx], st.ts[idx], st.eids[idx])
    runner = StreamRunner(eng)
    eng.inp.copy_(records[0])
    runner.capture(warmup=2)
    eng.reset()

    def step(i):
        j = i % n_rec
        if j == 0 and i > 0:
            eng.reset()                 # every chunk wraps to its start
        return runner.submit_device(records[j])

    def timed(first, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(first, first + n):
            step(i)
        runner.join()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3

    for i in range(20):
        step(i)
    probe = timed(20, 200)
    steps = max(1000, int(math.ceil(min_window * 1.2 / (probe / 200))))
    torch.cuda.reset_peak_memory_stats()
    sec = timed(220, steps)
    eng.check_errors()
    out = {'workload': workload, 'restarter': wl.rst, 'n_chunks': M, 'B_per_chunk': B, 'events_per_step': M * B,
           'batches_per_chunk': n_rec, 'steps': steps, 'window_s': sec, 'ms_per_step': sec / steps * 1e3,
           'events_per_s': M * B * steps / sec, 'peak_alloc_bytes': torch.cuda.max_memory_allocated(),
           'launches_per_step': eng.launches_per_step(), 'involved_capacity': eng.cap}

    # CUDA-event time per entry point, eager launches on one stream (separate from the timed window)
    records_t, orig = [], _lib.call

    def timed_call(name, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig(name, *a)
        e1.record()
        records_t.append((name, e0, e1))

    eng.reset()
    n_prof, warm = min(60, n_rec), 10
    ops.call = timed_call
    try:
        for i in range(n_prof):
            if i == warm:
                torch.cuda.synchronize()
                records_t.clear()
            eng.inp.copy_(records[i])
            eng.step()
    finally:
        ops.call = orig
    torch.cuda.synchronize()
    agg = {}
    for name, e0, e1 in records_t:
        agg[name] = agg.get(name, 0.0) + e0.elapsed_time(e1) * 1e3
    out['entry_point_us_per_step'] = {k: v / (n_prof - warm) for k, v in sorted(agg.items(), key=lambda x: -x[1])}

    if parity_batches > 0:
        out['parity'] = parity(eng, [TigerEngine(W, wl.csr, **kw) for _ in range(M)], records, idx, st, wl.neg,
                               parity_batches)
    return out


def parity(eng, refs, records, idx, st, neg, n_batches):
    """The chunked engine against M independent engines, each fed its own chunk, from reset."""
    import torch
    M, N, B = eng.n_chunks, eng.N, eng.chunk_batch
    worst = {}
    for e in [eng] + refs:
        e.reset()
    for i in range(n_batches):
        eng.inp.copy_(records[i])
        eng.step()
        for c, r in enumerate(refs):
            s = idx[i, c]
            r.set_batch(st.src[s], st.dst[s], neg[s], st.ts[s], st.eids[s])
            r.step()
        torch.cuda.synchronize()
        nn = eng.neigh_nids.view(3, M, B, -1)
        pos, negs = eng.chunk_scores()
        for c, r in enumerate(refs):
            got = nn[:, c].reshape(3 * B, -1)
            if not torch.equal(torch.where(got == 0, got, got - c * N), r.neigh_nids):
                raise SystemExit(f'parity: chunk {c} neighbor table of step {i} differs')
            if not torch.equal(eng.winner.view(2, M, B)[:, c].reshape(-1), r.winner):
                raise SystemExit(f'parity: chunk {c} winners of step {i} differ')
            pairs = [('scores', torch.cat([pos[c], negs[c]]), r.scores)]
            pairs += [(n, getattr(eng, n)[c * N:(c + 1) * N], getattr(r, n)) for n in STATE]
            # message rows without a pending message are dead (reset() keeps them; the chunked engine was timed first)
            live = r.has_msg.bool()
            pairs = [(n, a[live], b[live]) if n in ('msg_vals', 'msg_ts') else (n, a, b) for n, a, b in pairs]
            for name, a, b in pairs:
                a, b = a.double(), b.double()
                err = float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)) if b.numel() else 0.0
                worst[name] = max(worst.get(name, 0.0), err)
        loss = float(np.mean([float(r.loss) for r in refs]))
        worst['loss_abs'] = max(worst.get('loss_abs', 0.0), abs(float(eng.loss) - loss))
    bad = {k: v for k, v in worst.items() if v > 1e-5}
    if bad:
        raise SystemExit(f'parity: {bad} exceed 1e-5')
    return {'steps': n_batches, 'neighbor_tables': 'bit-identical', 'winners': 'bit-identical', 'max_rel': worst,
            'tol': 1e-5}


def run_leg(workload, M, a):
    cmd = [sys.executable, os.path.abspath(__file__), '--leg', workload, '--chunks', str(M), '--min-window',
           str(a.min_window), '--parity-batches', str(a.parity_batches if M == max(a.chunk_list) else 0)]
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith('{')]
    if res.returncode != 0 or not lines:
        return {'workload': workload, 'n_chunks': M, 'error': (res.stdout + res.stderr)[-2000:]}
    return json.loads(lines[-1])


def run_bench_py(tree, dump):
    res = subprocess.run([sys.executable, 'bench.py', '--gpus', '1', '--steps', '1000', '--warmup', '20',
                          '--cpu-batches', '0', '--profile-steps', '0', '--parity-batches', '0', '--train-steps', '0',
                          '--dump-outputs', dump], capture_output=True, text=True, cwd=tree)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith('{')]
    if res.returncode != 0 or not lines:
        return {'error': (res.stdout + res.stderr)[-2000:]}
    r = json.loads(lines[-1])
    return {k: r[k] for k in ('metric', 'value', 'unit', 'ms_per_step', 'gpu_launches') if k in r}


def same_dumps(a, b):
    names = sorted(f for f in os.listdir(b) if f.endswith('.npy'))
    if sorted(f for f in os.listdir(a) if f.endswith('.npy')) != names or not names:
        return False
    return all(np.array_equal(np.load(os.path.join(a, f)), np.load(os.path.join(b, f)), equal_nan=True) for f in names)


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--workloads', default='reddit,wikipedia')
    p.add_argument('--chunks', default='1,2,4,8,16')
    p.add_argument('--repeats', type=int, default=2, help='runs of every leg (the spread)')
    p.add_argument('--min-window', type=float, default=1.0, help='seconds of the timed window of a leg')
    p.add_argument('--parity-batches', type=int, default=5, help='parity steps of the largest M (0: skip)')
    p.add_argument('--parent-tree', default=None, help='built source tree of the bench.py comparison (parent commit)')
    p.add_argument('--rounds', type=int, default=2, help='alternations of the bench.py legs of the two trees')
    p.add_argument('--out', default=None)
    p.add_argument('--leg', default=None)
    a = p.parse_args()
    a.chunk_list = [int(x) for x in a.chunks.split(',')]
    if a.leg is not None:
        print(json.dumps(leg(a.leg, a.chunk_list[0], a.min_window, a.parity_batches)))
        return
    report = {'gpu_before': gpu_info(), 'settings': {k: v for k, v in vars(a).items() if k not in ('leg', 'out')},
              'legs': []}
    for r in range(a.repeats):
        for w in a.workloads.split(','):
            for M in a.chunk_list:
                t0 = time.time()
                res = run_leg(w, M, a)
                res['repeat'] = r
                report['legs'].append(res)
                print(f'{w} M={M} repeat {r}: ' + (f"{res['events_per_s']:.0f} events/s, {res['ms_per_step']:.3f} "
                      f"ms/step" if 'events_per_s' in res else res['error'][-400:]) + f' ({time.time() - t0:.0f} s)',
                      flush=True)
    if a.parent_tree:
        runs = {'tree': [], 'parent': []}
        tmp = tempfile.mkdtemp(prefix='bench_chunks_')
        for r in range(a.rounds):
            for name, tree in (('parent', os.path.abspath(a.parent_tree)), ('tree', ROOT)):
                runs[name].append(run_bench_py(tree, os.path.join(tmp, f'{name}{r}')))
                print(f'bench.py {name} round {r}: {runs[name][-1]}', flush=True)
        report['bench_py'] = runs
        report['bench_py_dumps_identical'] = all(same_dumps(os.path.join(tmp, f'tree{r}'), os.path.join(tmp, f'parent{r}'))
                                                 for r in range(a.rounds))
        print(f"bench.py --dump-outputs identical on both trees: {report['bench_py_dumps_identical']}", flush=True)
    report['gpu_after'] = gpu_info()
    text = json.dumps(report, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
