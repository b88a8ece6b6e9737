#!/usr/bin/env python
"""Cost of the second attention layer (n_layers=2) on the BASELINE workloads.

    python tools/bench_layers.py [--workloads wikipedia,reddit] [--steps 1000] [--parent-tree DIR] [--out FILE]

Every leg runs in its own process (own peak-memory counter) with bench.py's settings: 1000 skipped batches, batch
inputs resident in HBM, the workload's restarter and lazy restart, CUDA events around >= --steps timed steps.
  engine L1 / L2   TigerEngine(n_layers=1 | 2), StreamRunner graph replay (bench.py's `value` loop)
  dropin L2        eval_edge_prediction over the drop-in TIGER(n_layers=2), wall clock around the synchronised loop
                   (bench.py --api dropin); with --parent-tree also the same loop on that source tree, the legs of
                   the two trees alternated
The drop-in loop cannot wrap around the stream window (collation carries the host restart set), so on a short
stream it times fewer steps; the JSON records how many.  Also reports the seq restarter's device buffers at the
capacity of each depth on the scaled stream, and the GPU's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench_args(tree, workload, steps, warmup):
    sys.path.insert(0, tree)
    import bench
    sys.argv = ['bench.py', '--workload', workload, '--steps', str(steps), '--warmup', str(warmup), '--cpu-batches',
                '0', '--profile-steps', '0', '--parity-batches', '0', '--train-steps', '0']
    return bench, bench.parse_args()


def leg_engine(tree, workload, steps, warmup, n_layers):
    import torch
    bench, args = bench_args(tree, workload, steps, warmup)
    from www2023tiger_b200.engine import StreamRunner, TigerEngine
    from www2023tiger_b200.init import random_weights
    wl = bench.DeviceWorkload(args)
    W = random_weights(wl.d, wl.de, n_nodes=wl.N, restarter=wl.rst, hist_len=bench.HIST_LEN, seed=args.seed,
                       n_layers=n_layers)
    eng = TigerEngine(W, wl.csr, n_nodes=wl.N, dim=wl.d, efeats=wl.efeats, n_neighbors=bench.K_NEIGH,
                      n_head=bench.N_HEAD, batch_size=bench.BATCH, msg_src=wl.shape.msg_src, upd_src=wl.shape.upd_src,
                      restarter=wl.rst, hist_len=bench.HIST_LEN, lazy_restart=True, n_layers=n_layers, device=wl.dev)
    runner = StreamRunner(eng)
    eng.inp.copy_(wl.dev_in[0])
    runner.capture(warmup=2)
    eng.reset()

    def device_step(i):
        j = i % wl.avail
        if j == 0 and i > 0:
            eng.reset()
        return runner.submit_device(wl.dev_in[j])
    for i in range(warmup):
        device_step(i)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(warmup, warmup + steps):
        slot = device_step(i)
    runner.join()
    ev1.record()
    torch.cuda.synchronize()
    eng.check_errors()
    ms = ev0.elapsed_time(ev1)
    loss = float(runner.d_out[slot][-1])
    return {'ms_per_step': ms / steps, 'events_per_s': steps * bench.BATCH / (ms * 1e-3), 'steps': steps,
            'launches_per_step': eng.launches_per_step(), 'cap': eng.cap, 'last_loss': loss,
            'peak_mem_bytes': torch.cuda.max_memory_allocated()}


def leg_dropin(tree, workload, steps, warmup):
    import numpy as np
    import torch
    from torch.utils.data import DataLoader
    bench, args = bench_args(tree, workload, steps, warmup)
    from www2023tiger_b200.init import build_model
    from www2023tiger_b200.tiger.data.data_loader import GraphCollator, InteractionData
    from www2023tiger_b200.tiger.data.graph import Graph
    from www2023tiger_b200.tiger.eval_utils import eval_edge_prediction
    wl = bench.DeviceWorkload(args)
    st, neg, lo, B = wl.st, wl.neg, wl.lo, bench.BATCH
    steps = min(steps, wl.avail - warmup)
    graph = Graph.from_csr(wl.csr)
    torch.manual_seed(args.seed)
    model = build_model(None, wl.efeats, graph, wl.N, st.n_events, wl.dev, dim=wl.shape.dim, n_layers=2,
                        n_heads=bench.N_HEAD, n_neighbors=bench.K_NEIGH, hit_type='bin', dropout=0.1,
                        restarter_type=wl.rst, hist_len=bench.HIST_LEN, msg_src=wl.shape.msg_src,
                        upd_src=wl.shape.upd_src)
    model.eval()
    coll = GraphCollator(graph, bench.K_NEIGH, 2, restarter=wl.rst, hist_len=bench.HIST_LEN)

    def loader(first, n):
        s = slice(lo + first * B, lo + (first + n) * B)
        data = InteractionData(st.src[s], st.dst[s], st.ts[s], st.eids[s], np.zeros(n * B, dtype=np.int64), seed=0,
                               eval=True, neg_dst=neg[s])
        return DataLoader(data, batch_size=B, collate_fn=coll)
    model.reset()
    seen = set()
    eval_edge_prediction(model, loader(0, warmup), wl.dev, restart_mode=True, uptodate_nodes=seen)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ap, auc = eval_edge_prediction(model, loader(warmup, steps), wl.dev, restart_mode=True, uptodate_nodes=seen)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {'ms_per_step': dt / steps * 1e3, 'events_per_s': steps * B / dt, 'steps': steps, 'ap': ap, 'auc': auc,
            'peak_mem_bytes': torch.cuda.max_memory_allocated()}


def seq_restarter_bytes():
    """Device bytes of SeqRestarterOp at the involved-node capacity of each depth on the scaled stream (B = 200,
    K = 10, d = d_e = 172, hist_len 40), counted on the meta device (nothing is allocated)."""
    import torch
    sys.path.insert(0, ROOT)
    from www2023tiger_b200 import ops
    from www2023tiger_b200.synthetic import SHAPES
    sh = SHAPES['scaled']
    N, B, K, d = sh.n_users + sh.n_items + 1, 200, 10, 172
    out = {'n_nodes': N}
    for L, cap in ((1, 3 * B * (K + 1)), (2, min((3 * B + 3 * B * K) * (K + 1), N))):
        op = ops.SeqRestarterOp(d, d, 40, 2, cap, torch.device('meta'))
        out[f'n_layers_{L}'] = {'cap': cap, 'bytes': sum(t.numel() * t.element_size() for t in vars(op).values()
                                                         if isinstance(t, torch.Tensor))}
    return out


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def run_leg(kind, tree, workload, steps, warmup):
    cmd = [sys.executable, os.path.abspath(__file__), '--leg', kind, '--tree', tree, '--workloads', workload,
           '--steps', str(steps), '--warmup', str(warmup)]
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=tree)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith('{')]
    if res.returncode != 0 or not lines:
        return {'error': (res.stdout + res.stderr)[-2000:]}
    return json.loads(lines[-1])


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--workloads', default='wikipedia,reddit')
    p.add_argument('--steps', type=int, default=1000)
    p.add_argument('--warmup', type=int, default=20)
    p.add_argument('--rounds', type=int, default=2, help='alternations of the drop-in legs of the two trees')
    p.add_argument('--parent-tree', default=None, help='source tree of the comparison (built), e.g. the parent commit')
    p.add_argument('--out', default=None)
    p.add_argument('--leg', default=None, choices=['engine1', 'engine2', 'dropin'])
    p.add_argument('--tree', default=ROOT)
    a = p.parse_args()
    if a.leg is not None:
        os.chdir(a.tree)
        if a.leg == 'dropin':
            r = leg_dropin(a.tree, a.workloads, a.steps, a.warmup)
        else:
            r = leg_engine(a.tree, a.workloads, a.steps, a.warmup, int(a.leg[-1]))
        print(json.dumps(r))
        return
    report = {'gpu': gpu_info(), 'steps': a.steps, 'warmup': a.warmup, 'seq_restarter_scaled': seq_restarter_bytes(),
              'workloads': {}}
    trees = [('branch', ROOT)] + ([('parent', os.path.abspath(a.parent_tree))] if a.parent_tree else [])
    for w in a.workloads.split(','):
        r = {}
        for L in (1, 2):
            r[f'engine_n_layers_{L}'] = run_leg(f'engine{L}', ROOT, w, a.steps, a.warmup)
        for rnd in range(a.rounds):
            for name, tree in (trees if rnd % 2 == 0 else trees[::-1]):
                r.setdefault(f'dropin_n_layers_2_{name}', []).append(run_leg('dropin', tree, w, a.steps, a.warmup))
        report['workloads'][w] = r
        print(json.dumps({w: r}), flush=True)
    report['gpu_after'] = gpu_info()
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == '__main__':
    main()
