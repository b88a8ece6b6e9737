"""CPU checks of the scorer's hit types (--hit_type vec | count): the engine refuses unknown hit types and hit weights
sized for another K before any device work, random_weights draws build_model's shapes, and the native training step
still refuses these models."""
import pytest
import torch

import dropin_utils as D
from www2023tiger_b200.engine import TigerEngine
from www2023tiger_b200.init import build_model, random_weights


@pytest.mark.parametrize('hit_type', ['Vec', 'counts', 'onehot'])
def test_engine_rejects_unknown_hit_type(hit_type):
    with pytest.raises(NotImplementedError):
        TigerEngine({}, None, n_nodes=10, dim=8, efeats=None, device='cpu', hit_type=hit_type)


@pytest.mark.parametrize('hit_type,weights_k,engine_k', [('count', 4, 5), ('count', 6, 5), ('vec', 4, 5),
                                                         ('vec', 40, 10)])
def test_engine_rejects_hit_weights_of_another_k(hit_type, weights_k, engine_k):
    W = random_weights(8, 8, hit_type=hit_type, n_neighbors=weights_k)
    with pytest.raises(ValueError, match='n_neighbors'):
        TigerEngine(W, None, n_nodes=10, dim=8, efeats=None, device='cpu', hit_type=hit_type, n_neighbors=engine_k)


@pytest.mark.parametrize('hit_type', ['count', 'vec'])
def test_engine_rejects_bin_weights_for_count_and_vec(hit_type):
    W = random_weights(8, 8, hit_type='bin')
    with pytest.raises(ValueError, match=hit_type):
        TigerEngine(W, None, n_nodes=10, dim=8, efeats=None, device='cpu', hit_type=hit_type, n_neighbors=10)


@pytest.mark.parametrize('hit_type', ['bin', 'none', 'vec', 'count'])
@pytest.mark.parametrize('K', [5, 33])
def test_random_weights_have_build_model_shapes(hit_type, K):
    """Every parameter of build_model's state_dict, under the same name and shape (the time encoders that other
    modules share with the model's own appear once, as time_encoder.*)."""
    d, N = 6, 40
    model = build_model(None, torch.zeros(50, d), None, N, 49, torch.device('cpu'), dim=None, n_neighbors=K,
                        restarter_type='static', hit_type=hit_type)
    want = {k: tuple(v.shape) for k, v in model.state_dict().items()
            if not k.endswith(D.STATE_BUFFER_SUFFIXES) and '.time_encoder.' not in k}
    W = random_weights(d, d, n_nodes=N, restarter='static', hit_type=hit_type, n_neighbors=K)
    assert {k: tuple(v.shape) for k, v in W.items()} == want
    model.load_state_dict(W, strict=False)


@pytest.mark.parametrize('hit_type', ['count', 'vec'])
def test_random_weights_hit_types_keep_the_other_draws(hit_type):
    """The hit tensors are drawn last: every other parameter is the default model's."""
    base = random_weights(10, 4, seed=2)
    W = random_weights(10, 4, seed=2, hit_type=hit_type, n_neighbors=7)
    changed = {'count': {'hit_embedding.weight'}, 'vec': {'score_fn.fc1.weight'}}[hit_type]
    for k in set(W) & set(base) - changed:
        assert torch.equal(W[k], base[k]), k
    assert ('hit_embedding.weight' in W) == (hit_type == 'count')


@pytest.mark.parametrize('hit_type', ['vec', 'count'])
def test_native_trainer_refuses_vec_and_count(hit_type):
    from www2023tiger_b200.train import NativeTrainer
    model = build_model(None, torch.zeros(50, 6), None, 40, 49, torch.device('cpu'), dim=None, n_neighbors=10,
                        n_layers=1, restarter_type='static', hit_type=hit_type)
    with pytest.raises(NotImplementedError, match='hit_type'):
        NativeTrainer(model, 10)
