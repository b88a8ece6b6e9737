"""Host side of TigerEngine(n_chunks=M): the chunk-bounds helper against the reference's ChunkSampler, the chunk-major
input records (virtual-id offsets), and the construction checks that run before anything touches a device."""
import numpy as np
import pytest
import torch

from www2023tiger_b200.engine import TigerEngine, chunk_bounds
from www2023tiger_b200.tiger.data.data_loader import ChunkSampler


@pytest.mark.parametrize('n,M,B', [(157474, 4, 200), (672447, 16, 200), (10000, 3, 7), (4000, 2, 2000),
                                   (999, 1, 100)])
@pytest.mark.parametrize('seed', [0, 1, 17])
@pytest.mark.parametrize('epoch', [0, 3])
def test_chunk_bounds_equal_chunk_sampler(n, M, B, seed, epoch):
    got = chunk_bounds(n, M, B, seed=seed, epoch=epoch)
    want = []
    for rank in range(M):
        s = ChunkSampler(n, rank, M, B, seed=seed)
        s.set_epoch(epoch)
        want.append(s.bounds())
    assert got == want


def host_engine(M, N, B):
    """The attributes fill_record / device_records read, without device state."""
    e = TigerEngine.__new__(TigerEngine)
    e.n_chunks, e.chunk_batch, e.N, e.B, e.device = M, B, N, M * B, torch.device('cpu')
    return e


@pytest.mark.parametrize('M,N,B', [(1, 50, 4), (3, 97, 5), (16, 13, 2)])
def test_records_carry_virtual_ids(M, N, B):
    rng = np.random.RandomState(M)
    n = 3
    src, dst, neg = (rng.randint(1 if M > 1 else 0, N, (n, M, B)) for _ in range(3))
    src[0, -1, -1] = N - 1
    eids = rng.randint(1, 10 ** 6, (n, M, B))
    ts = rng.uniform(0, 1e6, (n, M, B))
    e = host_engine(M, N, B)
    rec = e.device_records(src, dst, neg, ts, eids).numpy()
    assert rec.shape == (n, 5 * M * B)
    off = (np.arange(M) * N)[None, :, None]
    r = rec.reshape(n, 5, M, B)
    for i, x in enumerate((src, dst, neg)):
        assert np.array_equal(r[:, i], x + off)
    assert np.array_equal(r[:, 3], eids)
    assert np.array_equal(r[:, 4].view(np.float64), ts)
    one = e.device_records(src[1], dst[1], neg[1], ts[1], eids[1]).numpy()
    assert np.array_equal(one, rec[1])
    h = np.zeros(5 * M * B, dtype=np.int64)
    e.fill_record(h, torch.from_numpy(src[2]), dst[2], neg[2], ts[2], eids[2])
    assert np.array_equal(h, rec[2])


def test_records_reject_ids_outside_the_node_range():
    e = host_engine(2, 10, 3)
    ok = np.ones((2, 3), dtype=np.int64)
    h = np.zeros(30, dtype=np.int64)
    for bad in (10, -1, 0):                 # 0: the padding node of a chunked engine
        src = ok.copy()
        src[1, 2] = bad
        with pytest.raises(ValueError, match='node ids'):
            e.fill_record(h, src, ok, ok, ok.astype(np.float64), ok)
    one = host_engine(1, 10, 3)                                     # an unchunked engine takes node 0
    one.fill_record(np.zeros(15, dtype=np.int64), np.zeros((1, 3), dtype=np.int64), ok[:1], ok[:1],
                    ok[:1].astype(np.float64), ok[:1])


@pytest.mark.parametrize('M', [0, -2, 1.5, True, '2'])
def test_construction_rejects_a_bad_chunk_count(M):
    with pytest.raises(ValueError, match='n_chunks'):
        TigerEngine({}, None, n_nodes=100, dim=8, efeats=None, n_chunks=M)


def test_construction_rejects_virtual_ids_past_int32():
    with pytest.raises(ValueError, match='int32'):
        TigerEngine({}, None, n_nodes=1_000_001, dim=8, efeats=None, n_chunks=2148)
    with pytest.raises(ValueError, match='int32'):
        TigerEngine({}, None, n_nodes=2 ** 30, dim=8, efeats=None, n_chunks=2)


def test_construction_refuses_training_targets_on_chunks():
    with pytest.raises(NotImplementedError):
        TigerEngine({}, None, n_nodes=100, dim=8, efeats=None, n_chunks=2, want_restarter_targets=True)
