"""f4: the on-disk format.  `load_jodie_data` of the drop-in package (rewritten for Python >= 3.11, where the
reference's own `random.sample(set, k)` raises) against the reference's loader with exactly that one call made
3.11-safe (tests/jodie_utils.py:REFERENCE_LOADER), run live where the reference's sources are vendored in
oracle/_ref, and against the splits stored in tests/golden/jodie_toy_splits.json, whose `source` field says which
loader recorded them (tests/golden/make_golden_jodie.py)."""
import json
import os

import numpy as np
import pytest

from jodie_utils import SPLITS, reference_splits, write_toy_dataset
from www2023tiger_b200.tiger.data.data_loader import load_jodie_data

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'jodie_toy_splits.json')
REF = os.path.join(ROOT, 'oracle', '_ref')


def test_load_jodie_data_properties(tmp_path):
    st = write_toy_dataset(str(tmp_path))
    nfeats, efeats, full, train, val, test, ind_val, ind_test = load_jodie_data('toy', train_seed=5, root=str(tmp_path))
    assert nfeats.shape == (st.n_nodes, 6) and np.array_equal(efeats, st.efeats)
    assert len(full) == st.n_events and np.array_equal(full.src, st.src) and np.array_equal(full.ts, st.ts)
    val_time, test_time = np.quantile(st.ts, [0.7, 0.85])
    assert train.ts.max() <= val_time and val.ts.min() > val_time and val.ts.max() <= test_time and test.ts.min() > test_time
    # chronological 70 / 15 / 15 split; the training set additionally loses the edges of the hidden (inductive) nodes
    assert len(val) + len(test) + int((st.ts <= val_time).sum()) == st.n_events and 0 < len(train) < (st.ts <= val_time).sum()
    train_nodes = set(train.src) | set(train.dst)
    for ind in (ind_val, ind_test):
        assert len(ind) > 0
        assert all((s not in train_nodes) or (d not in train_nodes) for s, d in zip(ind.src, ind.dst))
    # evaluation sets carry pre-sampled negatives (seeds 0, 2, 1, 3), the training set samples on the fly
    assert not train.eval and train.neg_dst is None and train.seed == 5
    for d, seed in ((val, 0), (test, 2), (ind_val, 1), (ind_test, 3)):
        assert d.eval and d.seed == seed and len(d.neg_dst) == len(d)
    src, dst, neg, ts, eid, label = train[0]
    assert neg in set(train.dst)


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'tiger')), reason='no reference sources (vendor with tools/vendor_ref.py)')
def test_load_jodie_data_equals_reference_loader(tmp_path):
    write_toy_dataset(str(tmp_path))
    ref = reference_splits(REF, str(tmp_path))
    assert_same_splits(load_jodie_data('toy', train_seed=5, root=str(tmp_path)), ref)


def test_load_jodie_data_equals_recorded_splits(tmp_path):
    """Against the stored splits.  Recorded from the reference's loader they are the comparison above without its
    sources; recorded from this package's loader (`source` says so) they only catch changes to it."""
    write_toy_dataset(str(tmp_path))
    with open(GOLDEN) as f:
        ref = json.load(f)
    out = load_jodie_data('toy', train_seed=5, root=str(tmp_path))
    assert_same_splits(out, ref, 'splits recorded by ' + ref['source'])


def assert_same_splits(out, ref, what='reference loader'):
    assert list(out[0].shape) == ref['nfeats_shape'] and abs(float(out[1].sum()) - ref['efeats_sum']) < 1e-3, what
    for n, d in zip(SPLITS, out[2:]):
        r, w = ref[n], f'{n} vs {what}'
        assert d.eids.tolist() == r['eids'], w                       # the same events in every split
        assert bool(d.eval) == r['eval'] and d.seed == r['seed'], w
        assert (d.neg_dst.tolist() if d.neg_dst is not None else None) == r['neg'], w   # the same pre-sampled negatives
