"""A tiny dataset in the on-disk format the reference reads (TGN / JODIE preprocessing: `data/ml_<name>.csv` with
columns [index, u, i, ts, label, idx], `data/ml_<name>.npy` edge features with a zero row 0,
`data/ml_<name>_node.npy` node features; reference loader tiger/data/data_loader.py:316-404)."""
import json
import os
import subprocess
import sys

import numpy as np
import pandas as pd

from www2023tiger_b200.synthetic import StreamShape, make_stream


def write_toy_dataset(root, name='toy', n_users=60, n_items=20, n_events=3000, efeat_dim=6, seed=3, node_feats=True):
    st = make_stream(StreamShape(name, n_users, n_items, n_events, efeat_dim, None, horizon=50000.), seed=seed)
    os.makedirs(os.path.join(root, 'data'), exist_ok=True)
    df = pd.DataFrame({'u': st.src, 'i': st.dst, 'ts': st.ts, 'label': st.labels.astype(np.float64), 'idx': st.eids})
    df.to_csv(os.path.join(root, 'data', f'ml_{name}.csv'))
    np.save(os.path.join(root, 'data', f'ml_{name}.npy'), st.efeats)
    if node_feats:                       # TGN writes an all-zero node table of the edge-feature width
        np.save(os.path.join(root, 'data', f'ml_{name}_node.npy'), np.zeros((st.n_nodes, efeat_dim), dtype=np.float32))
    return st


SPLITS = ['full', 'train', 'val', 'test', 'ind_val', 'ind_test']
SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', '_shim')

# The reference's own load_jodie_data in a subprocess, with exactly one call made Python >= 3.11 safe
# (random.sample over the SORTED set, which is what the drop-in does); prints summarize_splits() of its result.
REFERENCE_LOADER = r'''
import random, sys, json
import numpy as np
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[2])           # torch_scatter shim
_orig = random.sample
random.sample = lambda pop, k: _orig(sorted(pop), k)      # the only change: sets are rejected by Python >= 3.11
from tiger.data.data_loader import load_jodie_data
out = load_jodie_data('toy', train_seed=5, root=sys.argv[3])
names = ['full', 'train', 'val', 'test', 'ind_val', 'ind_test']
res = {'nfeats_shape': list(out[0].shape) if out[0] is not None else None, 'efeats_sum': float(out[1].sum())}
for n, d in zip(names, out[2:]):
    res[n] = {'eids': d.eids.tolist(), 'neg': (d.neg_dst.tolist() if d.neg_dst is not None else None), 'eval': bool(d.eval),
              'seed': d.seed}
print(json.dumps(res))
'''


def reference_splits(ref_dir, root):
    """summarize_splits() of the reference's loader (sources in `ref_dir`) on the toy dataset written under `root`."""
    res = subprocess.run([sys.executable, '-c', REFERENCE_LOADER, ref_dir, SHIM, root], capture_output=True, text=True,
                         timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def summarize_splits(out):
    """What a `load_jodie_data` result is compared on: feature shapes / sums, and per split the events, the
    pre-sampled negatives, the eval flag and the sampling seed (JSON-serialisable)."""
    res = {'nfeats_shape': list(out[0].shape) if out[0] is not None else None, 'efeats_sum': float(out[1].sum())}
    for n, d in zip(SPLITS, out[2:]):
        res[n] = {'eids': d.eids.tolist(), 'neg': (d.neg_dst.tolist() if d.neg_dst is not None else None),
                  'eval': bool(d.eval), 'seed': d.seed}
    return res
