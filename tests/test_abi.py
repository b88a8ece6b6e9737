"""CPU checks of the C-ABI boundary: the library loads, exports every symbol the header
declares, and the ctypes signatures in www2023tiger_b200/_lib.py match the header."""
import os
import re

import pytest

from www2023tiger_b200 import _lib
from www2023tiger_b200.build import INCLUDE, build


def header_decls():
    text = open(os.path.join(INCLUDE, 'tiger_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    decls = {}
    for m in re.finditer(r'\b(?:int|int64_t)\s+(tiger_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;', text, flags=re.S):
        name, params = m.group(1), m.group(2).strip()
        kinds = ''
        if params and params != 'void':
            for p in params.split(','):
                p = p.strip()
                if '*' in p:
                    kinds += 'p'
                elif p.startswith('int64_t'):
                    kinds += 'l'
                elif p.startswith('int '):
                    kinds += 'i'
                elif p.startswith('float '):
                    kinds += 'f'
                else:
                    raise AssertionError(f'unparsed parameter {p!r} in {name}')
        decls[name] = kinds
    return decls


@pytest.fixture(scope='module')
def lib():
    build()
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    names = _lib.header_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f'{n} declared in the header but not exported'
    assert lib.tiger_abi_version() == 1


def test_ctypes_signatures_match_header():
    decls = header_decls()
    assert set(decls) == set(_lib._SIGNATURES), set(decls) ^ set(_lib._SIGNATURES)
    for name, kinds in decls.items():
        sig = _lib._SIGNATURES[name]
        # every stream-ordered entry point takes the stream as its last pointer argument,
        # which _lib.call appends
        assert sig == kinds, f'{name}: header {kinds} vs binding {sig}'


def test_work_size_query_runs_without_gpu(lib):
    assert lib.tiger_csr_build_work_bytes(1000, 50) >= (4000 + 256 + 51) * 4


def test_attention_limits_at_each_boundary(lib):
    """tiger_temporal_attention_work_bytes refuses what the attention kernel refuses (K > 64, more than 8 heads, a
    score-pool footprint over 200 KiB) and ops.attention_limit_error names the limit."""
    from www2023tiger_b200.ops import attention_limit_error as err
    ru4 = lambda x: (x + 3) // 4 * 4
    pool_bytes = lambda d, de, k, h: 4 * (k * ru4(2 * d + de) + ru4(h * k) + h * ru4(2 * d + de + 1))
    assert err(16, 8, 64, 2) is None and lib.tiger_temporal_attention_work_bytes(10, 64, 16, 8, 2) > 0
    assert 'at most 64 neighbors' in err(16, 8, 65, 2) and lib.tiger_temporal_attention_work_bytes(10, 65, 16, 8, 2) == -1
    assert err(18, 6, 10, 8) is None
    assert 'at most 8 heads' in err(18, 6, 10, 9) and lib.tiger_temporal_attention_work_bytes(10, 10, 18, 6, 9) == -1
    # the footprint on both sides of 200 KiB at K = 64, two heads: d = d_e = 257 fits, 258 does not
    assert pool_bytes(257, 257, 64, 2) <= 200 * 1024 < pool_bytes(258, 258, 64, 2)
    assert err(257, 257, 64, 2) is None
    assert 'shared memory' in err(258, 258, 64, 2) and lib.tiger_temporal_attention_work_bytes(10, 64, 258, 258, 2) == -1
    assert err(258, 258, 10, 2) is None                      # the same widths at fewer slots
    assert err(172, 172, 64, 2) is None                      # the baseline width at the largest K
    assert 'invalid' in err(16, 8, 0, 2)
