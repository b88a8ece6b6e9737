#!/usr/bin/env python
"""Cost of one-vs-many candidate queries (TigerEngine.candidate_query) on the BASELINE workloads.

    python tools/bench_candidates.py [--workloads wikipedia,reddit] [--reps 200] [--parent-tree DIR] [--out FILE]

Per workload (its own process, bench.py's settings: the workload's restarter with lazy restart, B = 200, K = 10): the
engine ingests bench.py's skipped batches (the first 1000) through its captured step, so that memories, messages and
histories are those of the state bench.py times; then, for (Q, C) in QC, a captured query with seeded random
candidates (column 0 the true destination, ts the next batch's times) is timed with CUDA events over --reps calls:
  replay  the captured graph alone (inputs already in the query's buffer): device time per query call
  score   CandidateQuery.score with device inputs (input checks, copy into the buffer, replay)
with candidate pairs/s and the peak device memory of the process.  With --parent-tree, `bench.py --gpus 1` is run on
both trees, alternated, to show the ingest step unchanged.  The GPU's name, power limit and max SM clock are read in
the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_layers import bench_args, gpu_info  # noqa: E402
from bench_variants import run_bench_py  # noqa: E402

QC = ((200, 2), (200, 20), (200, 100))


def leg(workload, reps, warmup):
    import numpy as np
    import torch
    bench, args = bench_args(ROOT, workload, 1, 1)
    from www2023tiger_b200.engine import StreamRunner, TigerEngine
    from www2023tiger_b200.init import random_weights
    wl = bench.DeviceWorkload(args)
    st, B = wl.st, bench.BATCH
    W = random_weights(wl.d, wl.de, n_nodes=wl.N, restarter=wl.rst, hist_len=bench.HIST_LEN, seed=args.seed)
    eng = TigerEngine(W, wl.csr, n_nodes=wl.N, dim=wl.d, efeats=wl.efeats, n_neighbors=bench.K_NEIGH,
                      n_head=bench.N_HEAD, batch_size=B, msg_src=wl.shape.msg_src, upd_src=wl.shape.upd_src,
                      restarter=wl.rst, hist_len=bench.HIST_LEN, lazy_restart=True, device=wl.dev)
    runner = StreamRunner(eng)
    eng.inp.copy_(wl.dev_in[0])
    runner.capture(warmup=2)
    eng.reset()
    n_skip = wl.lo // B
    neg = wl.neg
    for i in range(n_skip):
        s = slice(i * B, (i + 1) * B)
        runner.wait(runner.submit_host(st.src[s], st.dst[s], neg[s], st.ts[s], st.eids[s]))
    runner.join()
    torch.cuda.synchronize()
    eng.check_errors()
    s = slice(wl.lo, wl.lo + B)
    out = {'ingested_batches': n_skip, 'queries': {}}
    for Q, C in QC:
        rng = np.random.default_rng(args.seed + C)
        cands = rng.integers(1, wl.N, (Q, C)).astype(np.int64)
        cands[:, 0] = st.dst[s][:Q]
        src, ts = torch.from_numpy(st.src[s][:Q].copy()).to(wl.dev), torch.from_numpy(st.ts[s][:Q].copy()).to(wl.dev)
        cands = torch.from_numpy(cands).to(wl.dev)
        torch.cuda.reset_peak_memory_stats()
        q = eng.candidate_query(Q, C)
        q.capture(Q)
        scores, ranks = q.score(src, cands, ts)
        torch.cuda.synchronize()
        q.check_errors()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        res = {}
        for name, call in (('replay', q.graph.replay), ('score', lambda: q.score(src, cands, ts))):
            for _ in range(warmup):
                call()
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(reps):
                call()
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / reps
            res[name] = {'ms_per_call': ms, 'pairs_per_s': Q * C / (ms * 1e-3)}
        r = ranks.cpu().numpy()
        res.update(reps=reps, cap=q.cap, peak_mem_mb=torch.cuda.max_memory_allocated() / 2**20,
                   mrr=float(np.mean(1.0 / r)), hits_at_10=float(np.mean(r <= 10)),
                   scores_finite=bool(torch.isfinite(scores).all()))
        out['queries'][f'Q={Q} C={C}'] = res
        print(json.dumps({workload: {f'Q={Q} C={C}': res}}), file=sys.stderr, flush=True)
        del q
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--workloads', default='wikipedia,reddit')
    p.add_argument('--reps', type=int, default=200)
    p.add_argument('--warmup', type=int, default=10)
    p.add_argument('--parent-tree', default=None, help='built source tree of the comparison, e.g. the parent commit')
    p.add_argument('--rounds', type=int, default=2, help='alternations of the bench.py legs of the two trees')
    p.add_argument('--bench-steps', type=int, default=1000)
    p.add_argument('--out', default=None)
    p.add_argument('--leg', default=None)
    a = p.parse_args()
    if a.leg is not None:
        print(json.dumps(leg(a.leg, a.reps, a.warmup)))
        return
    report = {'gpu': gpu_info(), 'reps': a.reps, 'workloads': {}}
    for w in a.workloads.split(','):
        res = subprocess.run([sys.executable, os.path.abspath(__file__), '--leg', w, '--reps', str(a.reps),
                              '--warmup', str(a.warmup)], capture_output=True, text=True, cwd=ROOT)
        lines = [ln for ln in res.stdout.splitlines() if ln.startswith('{')]
        report['workloads'][w] = json.loads(lines[-1]) if res.returncode == 0 and lines else \
            {'error': (res.stdout + res.stderr)[-3000:]}
        print(json.dumps({w: report['workloads'][w]}), flush=True)
    if a.parent_tree and a.bench_steps > 0:
        trees = [('branch', ROOT), ('parent', os.path.abspath(a.parent_tree))]
        bp = {}
        for rnd in range(a.rounds):
            for name, tree in (trees if rnd % 2 == 0 else trees[::-1]):
                bp.setdefault(name, []).append(run_bench_py(tree, a.bench_steps, 20))
        report['bench_py'] = bp
    report['gpu_after'] = gpu_info()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == '__main__':
    main()
