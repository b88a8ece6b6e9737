"""CPU checks of the drop-in class surface: the modules construct with the reference's keywords and
expose exactly the reference's state_dict keys / shapes (golden fixtures hold the reference model's
state_dict); host-side samplers behave like the reference's."""
import numpy as np
import pytest
import torch

from golden_utils import CASES, Golden
import dropin_utils as D
from tiger.data.data_loader import ChunkSampler, InteractionData, RandEdgeSampler
from oracle import tiger_oracle as O


@pytest.mark.parametrize('name', CASES)
def test_state_dict_keys_and_shapes_match_reference(name):
    g = Golden(name)
    model = D.model_from_golden(g, graph=None, device=None)
    sd = model.state_dict()
    ours = {k: tuple(v.shape) for k, v in sd.items() if not k.endswith(D.STATE_BUFFER_SUFFIXES)}
    ref = {k: tuple(v.shape) for k, v in g.W.items()}
    assert ours == ref
    for side in ('left', 'right', 'msg', 'upd'):
        assert tuple(sd[f'{side}_memory.vals'].shape) == (g.N, g.dim)
        assert sd[f'{side}_memory.active_mask'].dtype == torch.bool
    assert 'msg_store.node_msg_vals' not in sd                       # non-persistent, as in the reference
    D.load_golden_weights(model, g)


def test_invalid_sources_raise_value_error():
    g = Golden(CASES[0])
    with pytest.raises(ValueError):
        D.init_model(g.nfeats, g.efeats, None, g.N, len(g.src), None, dim=g.dim, n_layers=1, n_heads=2,
                     n_neighbors=5, hit_type='bin', dropout=0.1, restarter_type='seq', hist_len=4, msg_src='up',
                     upd_src='right')
    with pytest.raises(NotImplementedError):
        D.init_model(g.nfeats, g.efeats, None, g.N, len(g.src), None, dim=g.dim, n_layers=1, n_heads=2,
                     n_neighbors=5, hit_type='bin', dropout=0.1, restarter_type='seq', hist_len=4, msg_src='left',
                     upd_src='right', mem_update_type='lstm')


def test_chunk_sampler_partition():
    n, world, bs = 10_000, 4, 200
    ranges = [ChunkSampler(n, r, world, bs, seed=3).bounds() for r in range(world)]
    assert all(hi - lo == n // (world * bs) * bs for lo, hi in ranges)
    assert all(ranges[r][1] == ranges[r + 1][0] for r in range(world - 1))
    assert 0 <= ranges[0][0] <= n % (world * bs)
    assert ranges == [O.chunk_range(n, r, world, bs, seed=3) for r in range(world)]
    s = ChunkSampler(n, 1, world, bs, seed=3)
    assert list(s) == list(range(*ranges[1])) and len(s) == ranges[1][1] - ranges[1][0]


def test_interaction_data_negatives_follow_reference_rng():
    g = Golden(CASES[0])
    data = InteractionData(g.src, g.dst, g.ts, g.eids, np.zeros_like(g.src), seed=0, eval=True)
    assert np.array_equal(data.neg_dst, g.neg)                        # pre-sampled exactly like RandEdgeSampler
    sub = data.get_subset(10, 40)
    # like the reference, a subset keeps the parent's un-sliced negatives (data_loader.py:239)
    assert len(sub) == 30 and sub[0][0] == g.src[10] and sub[0][2] == g.neg[0]
    s = RandEdgeSampler(g.src, g.dst, seed=5)
    a = s.sample(7)
    s.reset_random_state()
    assert np.array_equal(a[1], s.sample(7)[1])


def test_ap_and_auc_equal_sklearn():
    """The chunk metrics of eval_edge_prediction (reference eval_utils.py:55-62 calls sklearn) restated in numpy."""
    from sklearn import metrics
    from tiger.eval_utils import average_precision_score, roc_auc_score
    rng = np.random.RandomState(0)
    for trial in range(40):
        n = int(rng.randint(2, 400))
        label = np.r_[np.ones(n), np.zeros(n)]
        score = rng.rand(2 * n)
        if trial % 3 == 0:
            score = np.round(score, 1)                 # many ties
        if trial % 7 == 0:
            score[:] = 0.5                             # all tied
        if trial % 5 == 0:
            keep = rng.rand(2 * n) > 0.3               # unbalanced, as after dropping non-finite scores
            keep[0] = keep[-1] = True
            label, score = label[keep], score[keep]
        assert abs(average_precision_score(label, score) - metrics.average_precision_score(label, score)) < 1e-12
        assert abs(roc_auc_score(label, score) - metrics.roc_auc_score(label, score)) < 1e-12


@pytest.mark.parametrize('K,restarter,hist_len,match', [(40, 'static', 8, 'at most 32 neighbors'),
                                                        (10, 'seq', 70, 'at most 64 events'),
                                                        (33, 'seq', 8, 'n_neighbors=33')])
def test_native_trainer_refuses_sizes_past_its_kernels(K, restarter, hist_len, match):
    """The attention core keeps one dropout bit per slot in 32 bits and the seq pool stages at most 64 positions:
    NativeTrainer refuses such models at construction (before it allocates anything), and the drop-in's route
    choice sends them to the torch-op route."""
    from www2023tiger_b200.init import build_model
    from www2023tiger_b200.train import NativeTrainer, native_limit_error
    model = build_model(None, torch.zeros(50, 6), None, 40, 49, torch.device('cpu'), dim=None, n_neighbors=K,
                        restarter_type=restarter, hist_len=hist_len)
    assert match in native_limit_error(model)
    with pytest.raises(NotImplementedError, match=match):
        NativeTrainer(model, 10)
    ok = build_model(None, torch.zeros(50, 6), None, 40, 49, torch.device('cpu'), dim=None, n_neighbors=32,
                     restarter_type=restarter, hist_len=64)
    assert native_limit_error(ok) is None
