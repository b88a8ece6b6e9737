"""CPU checks of the message transform / memory updater keywords: unknown values are refused before any device work,
and random_weights draws the default model's parameters exactly as before the keywords existed."""
import hashlib

import pytest
import torch

from www2023tiger_b200.engine import TigerEngine
from www2023tiger_b200.init import random_weights


def digest(W):
    h = hashlib.sha256()
    for k in sorted(W):
        h.update(k.encode())
        h.update(W[k].contiguous().numpy().tobytes())
    return h.hexdigest()[:16]


@pytest.mark.parametrize('kw', [{'msg_tsfm_type': 'attn'}, {'mem_update_type': 'rnn'}, {'msg_tsfm_type': 'Linear'}])
def test_engine_rejects_unknown_variants(kw):
    with pytest.raises(NotImplementedError):
        TigerEngine({}, None, n_nodes=10, dim=8, efeats=None, device='cpu', **kw)


def test_random_weights_rejects_unknown_variants():
    with pytest.raises(NotImplementedError):
        random_weights(8, 4, mem_update_type='rnn')


@pytest.mark.parametrize('kw,want', [
    (dict(d=8, de=4), '90a786501dce9cd8'),
    (dict(d=12, de=12, n_nodes=30, restarter='seq', hist_len=6, seed=3, n_layers=2), '3febd5252c7b731c'),
    (dict(d=10, de=10, n_nodes=40, restarter='static', nonzero_static=True, seed=1), '3fedb072c5639e66'),
])
def test_random_weights_defaults_unchanged(kw, want):
    """Digests of the parameters random_weights drew before the variant keywords were added."""
    kw = dict(kw)
    d, de = kw.pop('d'), kw.pop('de')
    assert digest(random_weights(d, de, **kw)) == want
    assert digest(random_weights(d, de, msg_tsfm_type='id', mem_update_type='gru', **kw)) == want


@pytest.mark.parametrize('tsfm,upd', [('linear', 'gru'), ('mlp', 'gru'), ('id', 'merge'), ('mlp', 'merge')])
def test_random_weights_variants(tsfm, upd):
    """The variants add their modules under the reference's state_dict names (a merge model has no GRU cell) and
    leave every other parameter as the default model draws it."""
    d, de = 10, 4
    M = 3 * d + de
    base = random_weights(d, de, seed=2)
    W = random_weights(d, de, seed=2, msg_tsfm_type=tsfm, mem_update_type=upd)
    shapes = {'linear': {'msg_transform_fn.fn.1.weight': (M, M), 'msg_transform_fn.fn.1.bias': (M,)},
              'mlp': {'msg_transform_fn.fn.1.weight': (M // 2, M), 'msg_transform_fn.fn.1.bias': (M // 2,),
                      'msg_transform_fn.fn.4.weight': (M, M // 2), 'msg_transform_fn.fn.4.bias': (M,)},
              'id': {}}[tsfm]
    if upd == 'merge':
        shapes.update({'right_mem_updater.fn.fc1.weight': (d, M + d), 'right_mem_updater.fn.fc1.bias': (d,),
                       'right_mem_updater.fn.fc2.weight': (d, d), 'right_mem_updater.fn.fc2.bias': (d,)})
    cell = {k for k in base if k.startswith('right_mem_updater.cell.')}
    assert set(W) == (set(base) - (cell if upd == 'merge' else set())) | set(shapes)
    for k, s in shapes.items():
        assert tuple(W[k].shape) == s, k
    for k in set(W) & set(base):
        assert torch.equal(W[k], base[k]), k
