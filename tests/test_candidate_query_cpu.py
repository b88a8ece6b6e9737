"""Refusals of the candidate query that need no device: the input checks CandidateQuery.score runs before it launches
anything, and the argument checks of the new entry points, which return TIGER_EINVAL before any CUDA call."""
import ctypes

import numpy as np
import pytest
import torch

from www2023tiger_b200 import _lib, ops
from www2023tiger_b200.build import build
from www2023tiger_b200.engine import check_query_inputs

KW = dict(max_queries=8, n_candidates=3, n_nodes=100, device='cuda:0')


def ok(Q=4, C=3):
    return dict(src=np.arange(1, Q + 1, dtype=np.int64), cands=np.ones((Q, C), np.int64), ts=np.linspace(1.0, 2.0, Q))


def test_valid_inputs_pass():
    assert check_query_inputs(**ok(), **KW) == 4
    t = {k: torch.from_numpy(v) for k, v in ok(8).items()}
    assert check_query_inputs(**t, **KW) == 8


@pytest.mark.parametrize('what, change', [
    ('too many queries', ok(9)),
    ('no queries', ok(0)),
    ('cands width', dict(cands=np.ones((4, 2), np.int64))),
    ('cands rows', dict(cands=np.ones((5, 3), np.int64))),
    ('ts length', dict(ts=np.ones(3))),
    ('src dtype', dict(src=np.arange(4, dtype=np.int32))),
    ('cands dtype', dict(cands=np.ones((4, 3), np.float64))),
    ('ts dtype', dict(ts=np.ones(4, np.float32))),
    ('ts tensor dtype', dict(ts=torch.ones(4))),
    ('src rank', dict(src=np.ones((4, 1), np.int64))),
    ('cands rank', dict(cands=np.ones(12, np.int64))),
    ('negative id', dict(src=np.array([1, 2, -1, 3], np.int64))),
    ('id past n_nodes', dict(cands=np.full((4, 3), 100, np.int64))),
    ('tensor id past n_nodes', dict(cands=torch.full((4, 3), 100, dtype=torch.int64))),
    ('list input', dict(src=[1, 2, 3, 4])),
])
def test_refusals(what, change):
    with pytest.raises(ValueError):
        check_query_inputs(**{**ok(), **change}, **KW)


@pytest.fixture(scope='module')
def lib():
    build()
    return _lib.load()


def test_entry_points_refuse_bad_arguments_before_any_launch(lib):
    x = ctypes.c_void_p(16)            # never dereferenced: every call below is refused on its arguments
    # scorer: no candidate column, negative query count, no second-column pointer, unknown hit type
    sc = lambda q, c, negs, hit: lib.tiger_link_score_cands(x, q, c, 8, x, x, negs, x, 4, hit, x, x, x, x, None, None,
                                                            None, None)
    assert sc(10, 0, x, 1) == -1 and sc(-1, 2, x, 1) == -1 and sc(10, 3, None, 1) == -1 and sc(10, 2, x, 7) == -1
    assert sc(0, 2, x, 1) == 0         # nothing to score
    # read-only compaction: negative restart base, restart base + capacity past int32
    cp = lambda base, cap: lib.tiger_compact_involved_ex(x, 100, x, x, x, cap, None, x, x, x, x, None, 1, base, None)
    assert cp(-1, 10) == -1 and cp(2**31 - 5, 10) == -1
    # surrogate rows: no output
    assert lib.tiger_static_restart_rows(x, None, 4, x, 8, None, None) == -1
    # the query's attention takes the score fold without a left write-back only
    p = ops.AttnParamsC()
    p.folded, p.score_folded, p.pq_out = 16, 16, 16
    att = lambda: lib.tiger_temporal_attention_query(x, x, 4, 4, 1, x, x, x, 4, x, x, None, x, 0, None, None, 8, 8, 2,
                                                     ctypes.addressof(p), x, x, None)
    p.left_wb = 16
    assert att() == -1
    p.left_wb, p.pq_out = None, None
    assert att() == -1
