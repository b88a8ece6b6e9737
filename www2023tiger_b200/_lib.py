"""ctypes binding of libtiger_b200.so (the C ABI declared in include/tiger_b200.h).

There is no CPU or PyTorch fallback: if the shared library is missing or a call fails,
the operators raise.  PyTorch is used for device memory and streams only.
"""
import ctypes
import os
import re
from typing import Dict, List

import torch

from .build import INCLUDE, LIB_PATH

P, L, I, F = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_float

# argument kinds per entry point: p = device/host pointer, l = int64, i = int
_SIGNATURES: Dict[str, str] = {
    'tiger_abi_version': '',
    'tiger_csr_build_work_bytes': 'll',
    'tiger_csr_build': 'ppppll' + 'ppppp' + 'p' + 'p',
    'tiger_find_recent': 'ppppp' + 'pp' + 'lli' + 'pppp' + 'pp' + 'p' + 'p',
    'tiger_find_recent_ex': 'ppppp' + 'pp' + 'lli' + 'pppp' + 'pp' + 'p' + 'li' + 'p',
    'tiger_hit_window': 'ppli' + 'p' + 'p',
    'tiger_mark_nodes': 'plpl' + 'p',
    'tiger_compact_involved': 'plpp' + 'plp' + 'ppp' + 'pp' + 'p',
    'tiger_compact_involved_ex': 'plpp' + 'plp' + 'ppp' + 'pp' + 'ii' + 'p',
    'tiger_select_latest': 'ppil' + 'llppp' + 'pppp' + 'p',
    'tiger_anonymized_reindex': 'plip' + 'p' + 'p',
    'tiger_gather_rows': 'plplp' + 'pp' + 'p',
    'tiger_scatter_rows': 'plplp' + 'ppp' + 'pip' + 'p',
    'tiger_time_encode': 'plppip' + 'p',
    'tiger_store_messages': 'ppppl' + 'ppp' + 'ppii' + 'pppp' + 'pp' + 'p',
    'tiger_store_messages_dense': 'ppppl' + 'p' + 'pppp' + 'ppii' + 'pppp' + 'pp' + 'p',
    'tiger_right_writeback': 'plp' + 'ppi' + 'pppp' + 'pppp' + 'p' + 'p',
    'tiger_left_writeback': 'pllp' + 'pip' + 'ppp' + 'p' + 'p',
    'tiger_gru_pack_bytes': 'ii',
    'tiger_gru_pack': 'ppiip' + 'p',
    'tiger_gru_update': 'ppl' + 'plpl' + 'ii' + 'p' + 'ppp' + 'ppi' + 'p' + 'p',
    'tiger_gru_update_rows': 'ppl' + 'plpl' + 'ii' + 'p' + 'ppp' + 'ppi' + 'p' + 'p',
    'tiger_merge_pack': 'piipp',
    'tiger_merge_update': 'ppl' + 'plipl' + 'ii' + 'ppp' + 'ppi' + 'p' + 'p',
    'tiger_attn_fold_bytes': 'iii',
    'tiger_attn_fold': 'piii' + 'p',
    'tiger_temporal_attention_work_bytes': 'liiii',
    'tiger_temporal_attention_ex': 'pplll' + 'pppi' + 'ppppi' + 'pp' + 'iii' + 'ppp' + 'p',
    'tiger_temporal_attention_query': 'pplll' + 'pppi' + 'ppppi' + 'pp' + 'iii' + 'ppp' + 'p',
    'tiger_temporal_attention_dense': 'pppppp' + 'li' + 'iii' + 'ppp' + 'p',
    'tiger_score_fold_bytes': 'i',
    'tiger_score_fold_cab_offset': 'i',
    'tiger_score_fold': 'pppppip' + 'p',
    'tiger_link_score_folded': 'pli' + 'pppp' + 'i' + 'ppp' + 'ppp' + 'p',
    'tiger_score_fold_hit_bytes': 'iii',
    'tiger_score_fold_hit_offset': 'iii',
    'tiger_score_fold_hit': 'pppppiii' + 'p' + 'p',
    'tiger_link_score_folded_hit': 'pli' + 'pppp' + 'ii' + 'ppp' + 'ppp' + 'p',
    'tiger_link_score_cands': 'plii' + 'ppp' + 'pii' + 'ppp' + 'pppp' + 'p',
    'tiger_sgemm_nt_packed_gather': 'ppi' + 'pplp' + 'pi' + 'ppl' + 'lpl' + 'iifi' + 'p',
    'tiger_sgemm_nt_packed_splitk_fused': 'plpi' + 'ppl' + 'i' + 'lpl' + 'iifi' + 'p',
    'tiger_pipe_capture_begin': 'p',
    'tiger_pipe_capture_end': 'ppii',
    'tiger_pipe_submit': 'pipplpplp',
    'tiger_pipe_wait': 'pii',
    'tiger_pipe_join': 'pp',
    'tiger_sgemm_nt_packed_scatter': 'plpippli' + 'pliil' + 'ip' + 'p',
    'tiger_min_time': 'plp' + 'p',
    'tiger_min_time_ex': 'pllp' + 'p',
    'tiger_seq_tokens': 'ppli' + 'ppppp' + 'ppii' + 'ppp' + 'ppp' + 'p',
    'tiger_sgemm_nt': 'plplp' + 'pl' + 'lpl' + 'iii' + 'p',
    'tiger_train_gather_pending': 'pplpippipipppppp',
    'tiger_train_gru_gates': 'pppplippppp',
    'tiger_train_gru_gates_bwd': 'ppppppplippp',
    'tiger_train_attn_build_ex': 'plpll' + 'pppi' + 'ppppp' + 'p' + 'ii' + 'pp' + 'ppp' + 'li' + 'p',
    'tiger_train_attn_core': 'plpplpliiifiplpppp',
    'tiger_train_attn_core_bwd': 'plplpplppliiifpppp',
    'tiger_train_attn_build_bwd_ex': 'pppli' + 'plpll' + 'ppi' + 'pii' + 'pp' + 'pppp' + 'p',
    'tiger_train_zero_rows': 'plilpp',
    'tiger_train_relu_bwd': 'plplilplfp',
    'tiger_train_colsum': 'pllplifpp',
    'tiger_train_scatter_add_rows': 'pplplplifp',
    'tiger_train_score_build': 'ppppiplippp',
    'tiger_train_score_head': 'ppplifipppp',
    'tiger_train_score_head_bwd': 'pfpplifpppp',
    'tiger_train_score_build_bwd': 'pplippp',
    'tiger_train_seed_step': 'p',
    'tiger_train_mse': 'pppppplipppppp',
    'tiger_train_adam': 'ppppppppiplfffffip',
    'tiger_train_seq_pool': 'plpppliiifippppp',
    'tiger_train_seq_pool_bwd': 'pppplpppliiifippp',
    'tiger_train_seq_vbias': 'ppppliip',
    'tiger_train_seq_vbias_bwd': 'ppppliippp',
    'tiger_train_seq_tokens_bwd': 'pplippiipppppp',
    'tiger_train_dropout': 'ppllfiip',
    'tiger_train_axpy': 'pppllfp',
    'tiger_gemm_pp_pack_bytes': 'll',
    'tiger_gemm_pp_pack': 'plillpplpp',
    'tiger_sgemm_pp': 'ppppllilpplfiiip',
    'tiger_seq_gate_count': 'pipp' + 'p',
    'tiger_seq_tail': 'ppliii' + 'pppppp' + 'plp' + 'pp' + 'pfi' + 'ppppp' + 'p',
    'tiger_sgemm_ex': 'pli' + 'pli' + 'ppl' + 'lil' + 'ppl' + 'fiii' + 'p',
    'tiger_gemm_pick_bn': 'lii',
    'tiger_gemm_pack_bytes': 'iii',
    'tiger_gemm_pack_weight': 'plpiiiip' + 'p',
    'tiger_sgemm_nt_packed': 'plpippllpliifi' + 'p',
    'tiger_static_restart': 'ppl' + 'plp' + 'pp' + 'ppi' + 'ppp' + 'ppp' + 'pp' + 'p',
    'tiger_static_restart_ex': 'ppl' + 'plp' + 'pp' + 'ppi' + 'ppp' + 'ppp' + 'pp' + 'lp' + 'p',
    'tiger_static_restart_rows': 'pplpi' + 'p' + 'p',
}
_KIND = {'p': P, 'l': L, 'i': I, 'f': F}

ERR_BITS = {
    1: 'You are not allowed to modify past memory.',
    2: 'Node has unused messages.',
    4: 'Messages happened later than memory updating.',
    8: "Messages' ts should be equal to last update ts when using left memory as msg source.",
    16: 'Events occur before the udpated memory.',
    32: 'involved-node capacity exceeded',
}


class TigerLibraryError(RuntimeError):
    pass


def header_symbols() -> List[str]:
    """Every function name include/tiger_b200.h declares."""
    text = open(os.path.join(INCLUDE, 'tiger_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(tiger_[a-z0-9_]+)\s*\(', text)))


_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (built in-tree by www2023tiger_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TigerLibraryError(
            f'{LIB_PATH} is missing: run `python -m www2023tiger_b200.build` (or __graft_entry__.build()). '
            'There is no CPU fallback for the TIGER memory path.')
    lib = ctypes.CDLL(LIB_PATH)
    for name, sig in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = [_KIND[c] for c in sig]
        fn.restype = L if (name.endswith('_bytes') or name.endswith('_offset')) else I
    # the two entry points that do not return a status / size
    lib.tiger_pipe_create.argtypes, lib.tiger_pipe_create.restype = [I], ctypes.c_void_p
    lib.tiger_pipe_destroy.argtypes, lib.tiger_pipe_destroy.restype = [ctypes.c_void_p], None
    _lib = lib
    return lib


def ptr(t):
    """Device (or pinned host) pointer of a tensor; None -> NULL."""
    if t is None:
        return None
    return t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def call(name: str, *args):
    """Invoke an entry point on the current CUDA stream (appended as the last argument)."""
    lib = load()
    rc = getattr(lib, name)(*args, stream_ptr())
    if rc != 0:
        raise TigerLibraryError(f'{name} failed with code {rc} '
                                f'({"invalid argument" if rc == -1 else "CUDA launch error"})')


def check_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise TigerLibraryError('TIGER B200 operators need CUDA tensors; there is no CPU fallback.')
        if t is not None and not t.is_contiguous():
            raise TigerLibraryError('TIGER B200 operators need contiguous tensors.')


def raise_on_err_flags(flags: int):
    """Translate the device error word into the reference's ValueError messages."""
    if flags:
        msgs = [m for b, m in ERR_BITS.items() if flags & b]
        raise ValueError('; '.join(msgs))
