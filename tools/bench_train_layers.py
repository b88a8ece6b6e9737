#!/usr/bin/env python
"""Cost of training the second attention layer (n_layers=2) on the BASELINE workloads.

    python tools/bench_train_layers.py [--workloads wikipedia,reddit] [--steps 300] [--parent-tree DIR] [--out FILE]

Every leg runs in its own process (own peak-memory counter) with bench.py's train settings: 1000 skipped batches, batch
inputs resident in HBM, the workload's restarter, B = 200, K = 10, dropout 0.1, lr 1e-4.
  native L1 graph     NativeTrainer.step_stream at n_layers=1, CUDA-graph replay (bench.py --mode train's loop)
  native L2 graph     the same at n_layers=2
  native L2 eager     the same at n_layers=2, eager launches
  autograd L2         today's route for a two-layer model without the native step: the loop body of
                      train_self_supervised.py:143-171 over the drop-in TIGER(n_layers=2) on its torch-op route
                      (TIGER_AUTOGRAD_ROUTE=1) - GraphCollator, host restart set, contrast_and_mutual_learning,
                      loss.backward(), torch.optim.Adam - wall clock around the synchronised loop
The native legs time --steps steps with CUDA events; the autograd leg times --autograd-steps steps.  With
--parent-tree, `bench.py --mode train --cpu-batches 0` (one layer) also runs on this tree and on that one, alternated
--rounds times.
The GPU's name and power limit are read before and after.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def workload(tree, name, steps, warmup):
    sys.path.insert(0, tree)
    import bench
    sys.argv = ['bench.py', '--workload', name, '--mode', 'train', '--steps', str(steps), '--warmup', str(warmup),
                '--cpu-batches', '0', '--profile-steps', '0', '--parity-batches', '0']
    args = bench.parse_args()
    return bench, args, bench.DeviceWorkload(args, mode='train')


def make_model(bench, args, wl, n_layers):
    import torch
    from www2023tiger_b200.init import build_model
    from www2023tiger_b200.tiger.data.graph import Graph
    torch.manual_seed(args.seed)
    graph = Graph.from_csr(wl.csr)
    model = build_model(None, wl.efeats, graph, wl.N, wl.st.n_events, wl.dev, dim=wl.shape.dim, n_layers=n_layers,
                        n_heads=bench.N_HEAD, n_neighbors=bench.K_NEIGH, hit_type='bin', dropout=0.1,
                        restarter_type=wl.rst, hist_len=bench.HIST_LEN, msg_src=wl.shape.msg_src,
                        upd_src=wl.shape.upd_src)
    model.train()
    return model, graph


def leg_native(tree, name, steps, warmup, n_layers, graphed):
    import torch
    bench, args, wl = workload(tree, name, steps, warmup)
    model, _ = make_model(bench, args, wl, n_layers)
    tr = model.native_trainer(bench.BATCH, lr=1e-4, seed=args.seed)
    tr.attach_stream(wl.csr, bench.HIST_LEN)
    losses = torch.zeros(2, device=wl.dev)

    def device_step(i):
        j = i % wl.avail
        if j == 0 and i > 0:
            tr.reset_stream()
        closs, mloss = tr.step_stream(wl.dev_in[j], mutual_coef=1.0, grad_scale=1.0)
        losses[0:1].add_(closs)
        losses[1:2].add_(mloss)
    tr.reset_stream()
    if graphed:
        tr.capture_stream(mutual_coef=1.0, grad_scale=1.0)
    for i in range(warmup):
        device_step(i)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    losses.zero_()
    ev0.record()
    for i in range(warmup, warmup + steps):
        device_step(i)
    ev1.record()
    torch.cuda.synchronize()
    tr.check_errors()
    ms = ev0.elapsed_time(ev1)
    assert not graphed or tr._graph is not None
    return {'ms_per_step': ms / steps, 'events_per_s': steps * bench.BATCH / (ms * 1e-3), 'steps': steps,
            'cap': tr.cap, 'mean_contrast_loss': float(losses[0]) / steps, 'mean_mutual_loss': float(losses[1]) / steps,
            'peak_mem_bytes': torch.cuda.max_memory_allocated()}


def leg_autograd(tree, name, steps, warmup):
    import numpy as np
    import torch
    os.environ['TIGER_AUTOGRAD_ROUTE'] = '1'
    bench, args, wl = workload(tree, name, steps, warmup)
    model, graph = make_model(bench, args, wl, 2)
    from www2023tiger_b200.tiger.data.data_loader import GraphCollator, InteractionData
    st, neg, lo, B, dev = wl.st, wl.neg, wl.lo, bench.BATCH, wl.dev
    steps = min(steps, wl.avail - warmup)
    coll = GraphCollator(graph, bench.K_NEIGH, 2, restarter=wl.rst, hist_len=bench.HIST_LEN)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    data = InteractionData(st.src, st.dst, st.ts, st.eids, np.zeros(len(st.src), dtype=np.int64), seed=0, eval=True,
                           neg_dst=neg)
    uptodate = set()

    def step(i):                        # train_self_supervised.py:143-171 (restart_mode: :151-160)
        first = lo + i * B
        src, dst, ng, ts, eids, _, cg = coll([data[k] for k in range(first, first + B)])
        src, dst, ng, eids = (x.long().to(dev) for x in (src, dst, ng, eids))
        ts, cg = ts.float().to(dev), cg.to(dev)
        fresh = sorted(set(cg.np_computation_graph_nodes.tolist()) - uptodate)
        if fresh:
            model.restart(torch.tensor(fresh, dtype=torch.long, device=dev),
                          torch.full((len(fresh),), ts.min().item(), device=dev))
            uptodate.update(fresh)
        opt.zero_grad()
        c, m = model.contrast_and_mutual_learning(src, dst, ng, ts, eids, cg)
        assert not type(c.grad_fn).__name__.startswith('_NativeStep')
        (c + m).backward()
        opt.step()
        return c, m
    model.reset()
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    acc = torch.zeros(2, device=dev)
    for i in range(warmup, warmup + steps):
        c, m = step(i)
        acc[0:1].add_(c.detach())
        acc[1:2].add_(m.detach())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    c_sum, m_sum = float(acc[0]), float(acc[1])
    return {'ms_per_step': dt / steps * 1e3, 'events_per_s': steps * B / dt, 'steps': steps,
            'mean_contrast_loss': c_sum / steps, 'mean_mutual_loss': m_sum / steps,
            'peak_mem_bytes': torch.cuda.max_memory_allocated()}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def run(cmd, cwd):
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=cwd)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith('{')]
    if res.returncode != 0 or not lines:
        return {'error': (res.stdout + res.stderr)[-2000:]}
    return json.loads(lines[-1])


def run_leg(kind, tree, name, steps, warmup):
    return run([sys.executable, os.path.abspath(__file__), '--leg', kind, '--tree', tree, '--workloads', name,
                '--steps', str(steps), '--warmup', str(warmup)], tree)


def bench_train(tree, steps, warmup):
    r = run([sys.executable, 'bench.py', '--gpus', '1', '--mode', 'train', '--steps', str(steps), '--warmup',
             str(warmup), '--cpu-batches', '0'], tree)
    keep = ('metric', 'value', 'ms_per_step', 'steps', 'warmup', 'parity_checked', 'error')
    return {k: r[k] for k in keep if k in r}


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--workloads', default='wikipedia,reddit')
    p.add_argument('--steps', type=int, default=300)
    p.add_argument('--autograd-steps', type=int, default=40)
    p.add_argument('--warmup', type=int, default=10)
    p.add_argument('--rounds', type=int, default=2, help='alternations of bench.py --mode train on the two trees')
    p.add_argument('--bench-steps', type=int, default=500)
    p.add_argument('--parent-tree', default=None, help='source tree of the comparison (built), e.g. the parent commit')
    p.add_argument('--out', default=None)
    p.add_argument('--leg', default=None, choices=['native1_graph', 'native2_graph', 'native2_eager', 'autograd2'])
    p.add_argument('--tree', default=ROOT)
    a = p.parse_args()
    if a.leg is not None:
        os.chdir(a.tree)
        if a.leg == 'autograd2':
            r = leg_autograd(a.tree, a.workloads, a.steps, a.warmup)
        else:
            r = leg_native(a.tree, a.workloads, a.steps, a.warmup, int(a.leg[6]), a.leg.endswith('graph'))
        print(json.dumps(r))
        return
    report = {'gpu': gpu_info(), 'batch': 200, 'n_neighbors': 10, 'steps': a.steps, 'autograd_steps': a.autograd_steps,
              'warmup': a.warmup, 'workloads': {}}
    for w in filter(None, a.workloads.split(',')):
        r = {}
        for leg in ('native1_graph', 'native2_graph', 'native2_eager'):
            r[leg] = run_leg(leg, ROOT, w, a.steps, a.warmup)
        r['autograd2'] = run_leg('autograd2', ROOT, w, a.autograd_steps, a.warmup)
        report['workloads'][w] = r
        print(json.dumps({w: r}), flush=True)
    if a.parent_tree:
        trees = [('branch', ROOT), ('parent', os.path.abspath(a.parent_tree))]
        one = report['bench_train_n_layers_1'] = {}
        for rnd in range(a.rounds):
            for name, tree in (trees if rnd % 2 == 0 else trees[::-1]):
                one.setdefault(name, []).append(bench_train(tree, a.bench_steps, 20))
        print(json.dumps(one), flush=True)
    report['gpu_after'] = gpu_info()
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == '__main__':
    main()
