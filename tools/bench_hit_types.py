#!/usr/bin/env python
"""Cost of the scorer's hit types (--hit_type vec | count) on the fused inference path, on the BASELINE workloads.

    python tools/bench_hit_types.py [--workloads wikipedia,reddit] [--steps 1000] [--parent-tree DIR] [--out FILE]

Every leg runs in its own process with bench.py's settings: 1000 skipped batches, batch inputs resident in HBM, the
workload's restarter and lazy restart, B = 200, K = 10, CUDA events around >= --steps timed steps.
  engine <hit>   TigerEngine, StreamRunner graph replay (bench.py's `value` loop), for bin (the default), vec, count
  dropin vec     eval_edge_prediction over the drop-in TIGER(hit_type='vec') - the TIGER class's own default -, wall
                 clock around the synchronised loop; with --parent-tree also the same loop on that tree (the
                 step-by-step torch-op route there), the legs of the two trees alternated, AP / AUC of both recorded
  bench.py       `python bench.py --gpus 1` (its timed loop) on this tree and on --parent-tree, alternated: the default
                 model's line
Also records the GPU's name and power limit before and after.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_layers import bench_args, gpu_info  # noqa: E402
from bench_variants import run_bench_py  # noqa: E402

ENGINE_HITS = ('bin', 'vec', 'count')
DROPIN_HITS = ('vec',)


def leg_engine(tree, workload, steps, warmup, hit_type):
    import torch
    bench, args = bench_args(tree, workload, steps, warmup)
    from www2023tiger_b200.engine import StreamRunner, TigerEngine
    from www2023tiger_b200.init import random_weights
    wl = bench.DeviceWorkload(args)
    W = random_weights(wl.d, wl.de, n_nodes=wl.N, restarter=wl.rst, hist_len=bench.HIST_LEN, seed=args.seed,
                       hit_type=hit_type, n_neighbors=bench.K_NEIGH)
    eng = TigerEngine(W, wl.csr, n_nodes=wl.N, dim=wl.d, efeats=wl.efeats, n_neighbors=bench.K_NEIGH,
                      n_head=bench.N_HEAD, batch_size=bench.BATCH, msg_src=wl.shape.msg_src, upd_src=wl.shape.upd_src,
                      restarter=wl.rst, hist_len=bench.HIST_LEN, lazy_restart=True, hit_type=hit_type, device=wl.dev)
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
    return {'ms_per_step': ms / steps, 'events_per_s': steps * bench.BATCH / (ms * 1e-3), 'steps': steps,
            'launches_per_step': eng.launches_per_step(), 'last_loss': float(runner.d_out[slot][-1])}


def leg_dropin(tree, workload, steps, warmup, hit_type):
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
    model = build_model(None, wl.efeats, graph, wl.N, st.n_events, wl.dev, dim=wl.shape.dim, n_layers=1,
                        n_heads=bench.N_HEAD, n_neighbors=bench.K_NEIGH, hit_type=hit_type, dropout=0.1,
                        restarter_type=wl.rst, hist_len=bench.HIST_LEN, msg_src=wl.shape.msg_src,
                        upd_src=wl.shape.upd_src)
    model.eval()
    coll = GraphCollator(graph, bench.K_NEIGH, 1, restarter=wl.rst, hist_len=bench.HIST_LEN)

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
    return {'ms_per_step': dt / steps * 1e3, 'events_per_s': steps * B / dt, 'steps': steps, 'ap': ap, 'auc': auc}


def run_leg(kind, tree, workload, steps, warmup, hit_type):
    cmd = [sys.executable, os.path.abspath(__file__), '--leg', kind, '--tree', tree, '--workloads', workload,
           '--steps', str(steps), '--warmup', str(warmup), '--hit-type', hit_type]
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
    p.add_argument('--rounds', type=int, default=2, help='alternations of the legs of the two trees')
    p.add_argument('--parent-tree', default=None, help='source tree of the comparison (built), e.g. the parent commit')
    p.add_argument('--bench-steps', type=int, default=1000, help='--steps of the bench.py legs (0: skip them)')
    p.add_argument('--out', default=None)
    p.add_argument('--leg', default=None, choices=['engine', 'dropin'])
    p.add_argument('--hit-type', default='bin')
    p.add_argument('--tree', default=ROOT)
    a = p.parse_args()
    if a.leg is not None:
        os.chdir(a.tree)
        fn = leg_dropin if a.leg == 'dropin' else leg_engine
        print(json.dumps(fn(a.tree, a.workloads, a.steps, a.warmup, a.hit_type)))
        return
    report = {'gpu': gpu_info(), 'steps': a.steps, 'warmup': a.warmup, 'workloads': {}}
    trees = [('branch', ROOT)] + ([('parent', os.path.abspath(a.parent_tree))] if a.parent_tree else [])
    for w in a.workloads.split(','):
        r = {}
        for hit in ENGINE_HITS:
            r[f'engine {hit}'] = run_leg('engine', ROOT, w, a.steps, a.warmup, hit)
            print(json.dumps({w: {hit: r[f'engine {hit}']}}), flush=True)
        for hit in DROPIN_HITS:
            for rnd in range(a.rounds):
                for name, tree in (trees if rnd % 2 == 0 else trees[::-1]):
                    r.setdefault(f'dropin {hit} {name}', []).append(run_leg('dropin', tree, w, a.steps, a.warmup, hit))
        report['workloads'][w] = r
        print(json.dumps({w: r}), flush=True)
    if a.bench_steps > 0:
        bp = {}
        for rnd in range(a.rounds):
            for name, tree in (trees if rnd % 2 == 0 else trees[::-1]):
                bp.setdefault(name, []).append(run_bench_py(tree, a.bench_steps, a.warmup))
        report['bench_py'] = bp
    report['gpu_after'] = gpu_info()
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == '__main__':
    main()
