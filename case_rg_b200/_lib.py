"""ctypes binding of libcase_b200.so (the C ABI declared in include/case_b200.h).

There is no CPU fallback: if the library is missing the import fails loudly, and every call that
returns non-zero raises ``RuntimeError`` with the library's message.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libcase_b200.so')

H, NH, HD = 256, 8, 32
MAX_W, MAX_T, MAX_SPLIT = 8, 128, 16
F32, BF16 = 0, 1
MODE_MODULE_GREEDY, MODE_PROTO_GREEDY, MODE_BEAM = 0, 1, 2
XATTN_TILE = AATTN_TILE = 128
# option bits of StepArgs.opt / GttpStepArgs.opt (include/case_b200.h: a set bit switches one feature OFF)
OPT_NO_PDL, OPT_NO_CHAIN, OPT_NO_STACK, OPT_NO_FORK, OPT_NO_POST, OPT_NO_GATE = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20
OPT_NO_EVICT_FIRST, OPT_DENSE_TAIL, OPT_UNFUSED_TAIL, OPT_NO_FUSED_SELECT, OPT_NO_COPY_PLAN = 0x40, 0x80, 0x100, 0x200, 0x400

vp, i32, f32p = C.c_void_p, C.c_int32, C.c_void_p
MAX_BAN_SEQ, MAX_BAN_LEN = 256, 16     # CASE_MAX_BAN_SEQ / CASE_MAX_BAN_LEN: banned sequences (length >= 2), their length


def _pad(block, full_type):
    """Give an argument block built as an earlier (shorter) form the storage of the complete one, zeroed: the launchers
    read every block as the complete struct."""
    size, full = C.sizeof(type(block)), C.sizeof(full_type)
    if size < full:
        C.resize(block, full)
        C.memset(C.addressof(block) + size, 0, full - size)


class Seg(C.Structure):
    _fields_ = [('p', vp), ('ld', i32), ('width', i32), ('div', i32), ('gather', i32)]


class RowLinArgs(C.Structure):
    _fields_ = [('seg', Seg * 4), ('nseg', i32), ('K', i32), ('Wt', vp), ('bias', vp), ('N', i32), ('act', i32),
                ('res', vp), ('ldres', i32), ('out', vp), ('ldo', i32), ('gather_idx', vp), ('R', i32),
                ('dtype', i32)]


class LayerWeights(C.Structure):
    _fields_ = [(n, vp) for n in ('Wqkv_t', 'bqkv', 'Wo_t', 'bo', 'Wq2_t', 'bq2', 'Wo2_t', 'bo2', 'W1_t', 'b1',
                                  'W2_t', 'b2', 'ln1_g', 'ln1_b', 'ln2_g', 'ln2_b', 'ln3_g', 'ln3_b', 'Wc')]


class Attr(C.Structure):
    """case_attr_t: the attribution record of one answer token (16 bytes)."""
    _fields_ = [('part', C.c_float * 3), ('source', i32)]


# The attribution pointers trail the argument blocks (ABI version 2 unchanged).  They are appended the ctypes way, by
# subclassing: SelectArgs / StepArgs / GttpStepArgs keep the fields up to nbest, and the *AttrArgs subclasses add the
# attribution pointers - the complete blocks the launchers read, and what the engines pass.


class SelectArgs(C.Structure):
    _fields_ = [(n, i32) for n in ('mode', 'B', 'W', 't', 'max_len', 'Tmax', 'BOS', 'EOS', 'UNK', 'PAD')] + \
               [(n, vp) for n in ('top_vals', 'top_idx', 'live', 'cum', 'length', 'tok', 'anc_in', 'anc_out',
                                  'parent', 'ended', 'best_key', 'best_len', 'out_tokens', 'n_live')] + \
               [('V_in', i32), ('tok_ext', vp), ('nbest', i32)]


class SelectAttrArgs(SelectArgs):
    _fields_ = [('attr_cand', vp), ('attr_hist', vp), ('out_attr', vp)]


class PostLinear(C.Structure):
    _fields_ = [('Wc', vp), ('bias', vp), ('out', vp), ('nchunk', i32), ('seg', i32 * 3)]


class ChainPost(C.Structure):
    _fields_ = [('npost', i32), ('W', i32), ('lin', PostLinear * 2), ('feat', vp), ('x_in', vp), ('ln_g', vp),
                ('ln_b', vp), ('ln_out', vp)]


class TailArgs(C.Structure):
    _fields_ = [(n, i32) for n in ('R', 'V', 'W', 'K', 'ldl', 'ldd', 'mask_col0', 'nmem', 'do_finalize', 'fac_ld',
                                   'map_ld')] + \
               [('ns', i32 * 2), ('fac_off', i32 * 2), ('map_off', i32 * 2), ('S', i32 * 2),
                ('logits', vp), ('hN', vp), ('stats', vp * 2), ('ctxp', vp * 2), ('Wm', vp), ('bm', vp),
                ('ctx', vp * 2), ('gates', vp), ('fac', vp), ('map', vp), ('prior', vp * 2), ('attn_un', vp * 2),
                ('top_vals', vp), ('top_idx', vp), ('dist', vp), ('gate_ctx', i32), ('cp_ld', i32),
                ('cp_n', vp), ('cp_uid', vp), ('cp_first', vp), ('cp_start', vp), ('cp_perm', vp), ('Vext', i32),
                ('attr', vp)]

    def __init__(self, *args, **kw):
        # the launchers read every block as the complete case_tail_args_t: a block built as TailArgs gets the storage of
        # the trailing constraint and ban fields too (zero: no constraints, no bans)
        super().__init__(*args, **kw)
        _pad(self, TailBanArgs)


# The search constraints trail the argument blocks (ABI version 2 unchanged), appended by subclassing like the attribution
# pointers: TailConstrArgs / StepConstrArgs / GttpStepConstrArgs.
class TailConstrArgs(TailArgs):
    _fields_ = [('hist_tok', vp), ('hist_anc', vp)] + \
               [(n, i32) for n in ('hist_ld', 't', 'eos', 'no_repeat_ngram', 'min_len')]


# The banned words trail them in turn: TailBanArgs / StepBanArgs / GttpStepBanArgs are the complete blocks the launchers
# read.  ban_mask uint32 [ceil(V / 32)], ban_tok int32 [MAX_BAN_SEQ][MAX_BAN_LEN], ban_len int32 [MAX_BAN_SEQ], ban_n
# int32 [1], all in device memory (NULL = no bans).
_BAN_FIELDS = [('ban_mask', vp), ('ban_tok', vp), ('ban_len', vp), ('ban_n', vp)]


class TailBanArgs(TailConstrArgs):
    _fields_ = _BAN_FIELDS


class StepArgs(C.Structure):
    def __init__(self, *args, **kw):
        # as TailArgs: the storage of every trailing field, zeroed (no attribution, constraints or bans)
        super().__init__(*args, **kw)
        _pad(self, StepBanArgs)

    _fields_ = [(n, i32) for n in ('B', 'W', 'R', 'V', 'ldv', 'Tmax', 'dtype', 'fast_tanh', 'vocab_impl', 'mode')] + \
               [('S', i32 * 2), ('nsplit_x', i32 * 2), ('nsplit_a', i32 * 2), ('map_off', i32 * 2)] + \
               [(n, i32) for n in ('max_len', 'BOS', 'EOS', 'UNK', 'PAD', 'materialize_only')] + \
               [('E', vp), ('pe', vp), ('layers', LayerWeights * 8), ('lnN_g', vp), ('lnN_b', vp),
                ('Wqa_t', vp * 2), ('bqa', vp * 2), ('va', vp * 2), ('Wg_t', vp), ('bg', vp), ('Wv', vp), ('Wm', vp),
                ('bm', vp), ('feat', vp), ('Kx', vp * 8), ('Vx', vp * 8), ('U', vp * 2), ('Mv', vp * 2),
                ('mask', vp * 2), ('prior', vp * 2), ('map', vp), ('map_ld', i32),
                ('kcache', vp * 8), ('vcache', vp * 8), ('anc', vp * 2), ('tok', vp), ('live', vp), ('cum', vp),
                ('length', vp), ('parent', vp), ('ended', vp), ('best_key', vp), ('best_len', vp),
                ('out_tokens', vp), ('n_live', vp),
                ('x_in', vp), ('h', vp), ('bbuf', vp), ('q2', vp), ('part_ml', vp), ('part_acc', vp), ('qa', vp),
                ('attn_un', vp * 2), ('stats', vp * 2), ('ctxp', vp * 2), ('hN', vp), ('ctx', vp * 2), ('gates', vp),
                ('fac', vp), ('gfeat', vp), ('logits', vp), ('dist', vp), ('top_vals', vp), ('top_idx', vp), ('vocab_ws', vp), ('prow', vp), ('h0', vp), ('qa1', vp), ('base_ms', vp), ('base_e', vp), ('base_i', vp), ('xcount', vp), ('xprefix', vp), ('xslots', i32), ('xidx', vp), ('xorder', vp), ('qcount', vp), ('Wqa_c', vp * 2), ('Wg_c', vp), ('xns', vp), ('cp_n', vp), ('cp_uid', vp), ('cp_first', vp), ('cp_start', vp), ('cp_perm', vp), ('cp_ld', i32), ('Gv', vp * 2), ('opt', i32), ('fork', vp), ('n_oov', i32), ('tok_ext', vp), ('nbest', i32)]


class StepAttrArgs(StepArgs):
    _fields_ = [('attr_cand', vp), ('attr_hist', vp), ('out_attr', vp)]


class StepConstrArgs(StepAttrArgs):
    _fields_ = [('no_repeat_ngram', i32), ('min_len', i32)]


class StepBanArgs(StepConstrArgs):
    _fields_ = _BAN_FIELDS


class GttpStepArgs(C.Structure):
    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        _pad(self, GttpStepBanArgs)

    _fields_ = [(n, i32) for n in ('B', 'W', 'R', 'V', 'ldv', 'dtype', 'fast_tanh', 'vocab_impl', 'mode', 'Lc', 'Lb',
                                   'nsplit_c', 'nsplit_b', 'max_len', 'BOS', 'EOS', 'UNK', 'PAD',
                                   'materialize_only', 'Tmax')] + \
               [(n, vp) for n in ('E', 'Wqs_t', 'bqs', 'vs', 'Wqb_t', 'bqb', 'vb', 'Wih_t', 'bih', 'Whh_t', 'bhh',
                                  'Wr_t', 'br', 'Wv', 'bv', 'wc', 'bc', 'Us', 'Ms', 'Ub', 'Mb', 'mask_c', 'mask_b',
                                  'map')] + \
               [('map_ld', i32), ('state', vp * 2), ('anc', vp * 2)] + \
               [(n, vp) for n in ('tok', 'live', 'cum', 'length', 'parent', 'ended', 'best_key', 'best_len',
                                  'out_tokens', 'n_live', 'emb', 'qa')] + \
               [('attn_un', vp * 2), ('stats', vp * 2), ('ctxp', vp * 2), ('ctx', vp * 2)] + \
               [(n, vp) for n in ('gi', 'gh', 'feat', 'gates', 'fac', 'logits', 'dist', 'top_vals', 'top_idx', 'vocab_ws')] + \
               [('opt', i32)] + [(n, vp) for n in ('base_ms', 'base_e', 'base_i', 'fork', 'qa1')] + [('nbest', i32)]


class GttpStepAttrArgs(GttpStepArgs):
    _fields_ = [('attr_cand', vp), ('attr_hist', vp), ('out_attr', vp)]


class GttpStepConstrArgs(GttpStepAttrArgs):
    _fields_ = [('no_repeat_ngram', i32), ('min_len', i32)]


class GttpStepBanArgs(GttpStepConstrArgs):
    _fields_ = _BAN_FIELDS


# name -> argtypes (return type is int for all but the three listed below)
_PROTOS = {
    'case_embed_rows': [vp, vp, vp, i32, i32, C.c_float, vp, i32, vp],
    'case_layernorm_rows': [vp, vp, vp, vp, i32, vp],
    'case_row_linear': [C.POINTER(RowLinArgs), vp],
    'case_layer_front': [vp, C.POINTER(LayerWeights), vp, vp, vp, i32, vp, i32, i32, i32, vp, vp, i32, i32, vp],
    'case_cross_attn_partial': [vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, i32, vp],
    'case_cross_attn_partial_tc': [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp],
    'case_pack_kv_tiles': [vp, i32, i32, i32, i32, i32, vp, vp],
    'case_pack_kv_tiles_gather': [vp, i32, i32, i32, vp, vp, i32, vp, vp],
    'case_cross_attn_part': [vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp],
    'case_cross_attn_part_slots': [i32],
    'case_layer_back': [vp, vp, vp, i32, C.POINTER(LayerWeights), vp, i32, i32, vp],
    'case_layer_chain': [C.POINTER(LayerWeights), C.POINTER(LayerWeights), vp, vp, vp, C.c_float, vp, vp, vp, vp, i32,
                         vp, vp, vp, vp, i32, vp, i32, vp, i32, i32, vp, vp, i32, i32, C.POINTER(ChainPost), vp],
    'case_layer_chain_max_tmax': [],
    'case_layer_stack': [C.POINTER(LayerWeights), i32, vp, vp, vp, vp, i32, i32, vp, vp, vp, C.c_float, vp, vp, vp, i32, vp,
                         i32, vp, i32, i32, vp, vp, i32, i32, C.POINTER(ChainPost), vp],
    'case_layer_chain_max_s0': [],
    'case_additive_attn': [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, i32, i32, vp],
    'case_additive_attn_compact': [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, vp,
                                   vp, vp],
    'case_finalize_rows': [vp, vp, vp, vp, vp, i32, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, i32, vp],
    'case_vocab_gemm': [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp],
    'case_vocab_gemm_tc': [vp, vp, vp, vp, i32, i32, i32, vp, vp],
    'case_softmax_mix': [vp, i32, vp, vp, i32, i32, i32, i32, vp],
    'case_copy_scatter': [vp, i32, i32, vp, vp, vp, i32, vp, i32, i32, i32, i32, i32, vp],
    'case_topk_rows': [vp, i32, i32, i32, i32, vp, vp, vp],
    'case_oov_fold': [vp, i32, i32, i32, i32, vp, vp, i32, vp],
    'case_row_tail': [C.POINTER(TailArgs), vp],
    'case_row_tail_max_vocab': [],
    'case_vocab_base': [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp],
    'case_sparse_tail': [C.POINTER(TailArgs), vp, vp, vp, i32, C.POINTER(SelectArgs), vp, vp],
    'case_sparse_tail_max_sources': [],
    'case_beam_select': [C.POINTER(SelectArgs), vp],
    'case_gru_cell': [vp, vp, vp, vp, vp, i32, vp],
    'case_attn_merge': [vp, vp, i32, i32, vp, vp, i32, i32, vp],
    'case_gttp_gates': [vp, vp, vp, vp, vp, i32, i32, i32, vp],
    'case_additive_attn_gate': [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, vp, vp, vp, vp],
    'case_gate_project': [vp, vp, vp, C.c_longlong, vp],
    'case_split_plan': [vp, i32, i32, i32, vp, vp],
    'case_prefill_project_tc': [vp, vp, vp, i32, i32, vp, vp, i32, vp, vp, vp],
    'case_enc_embed': [vp, vp, vp, C.c_longlong, i32, C.c_float, vp, vp],
    'case_ln_rows_wide': [vp, vp, i32, vp, vp, vp, vp, C.c_longlong, i32, vp],
    'case_enc_attention': [vp, vp, i32, i32, i32, i32, vp, vp],
    'case_interaction': [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp],
    'case_rows_dot': [vp, vp, vp, C.c_longlong, C.c_longlong, vp, vp],
    'case_prior_answer': [vp, vp, vp, vp, i32, i32, i32, vp, vp, vp],
    'case_gemm_rows_tc': [vp, vp, vp, C.c_longlong, i32, i32, i32, vp, i32, vp, vp, i32, vp],
    'case_ffn_rows_tc': [vp, vp, vp, i32, i32, vp, vp, C.c_longlong, vp, i32, vp, vp, i32, vp],
    'case_thread_options': [i32],
    'case_fork_create': [C.POINTER(vp)],
    'case_fork_destroy': [vp],
    'case_decode_step': [C.POINTER(StepArgs), i32, vp],
    'gttp_decode_step': [C.POINTER(GttpStepArgs), i32, vp],
}
_SIZE_FNS = ['case_vocab_tc_workspace_bytes', 'case_vocab_tc_packed_weight_bytes']
_SIZE_FNS2 = ['case_interaction_smem_bytes', 'case_gemm_rows_packed_weight_bytes']      # (int, int) -> size_t
EXPORTS = sorted(list(_PROTOS) + ['case_abi_version', 'case_last_error', 'case_struct_size'] + _SIZE_FNS + _SIZE_FNS2)
_STRUCTS = [Seg, RowLinArgs, LayerWeights, SelectAttrArgs, StepBanArgs, GttpStepBanArgs, TailBanArgs, ChainPost]

_lib = None


def load():
    """dlopen the library (building nothing): raises if it is absent or its ABI does not match."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} not found: run `python -c "import __graft_entry__ as g; g.build()"` '
                           '(there is no CPU fallback for the decode path)')
    lib = C.CDLL(LIB_PATH)
    lib.case_abi_version.restype = C.c_int
    lib.case_last_error.restype = C.c_char_p
    lib.case_struct_size.restype = C.c_size_t
    lib.case_struct_size.argtypes = [C.c_int]
    if lib.case_abi_version() != 2:
        raise RuntimeError('libcase_b200.so: unexpected ABI version')
    for i, st in enumerate(_STRUCTS):
        if lib.case_struct_size(i) != C.sizeof(st):
            raise RuntimeError(f'ABI mismatch for {st.__name__}: C {lib.case_struct_size(i)} != ctypes {C.sizeof(st)}')
    for name in _SIZE_FNS:
        getattr(lib, name).restype = C.c_size_t
        getattr(lib, name).argtypes = [C.c_int]
    for name in _SIZE_FNS2:
        getattr(lib, name).restype = C.c_size_t
        getattr(lib, name).argtypes = [C.c_int, C.c_int]
    for name, argtypes in _PROTOS.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    _lib = lib
    return lib


TORCH_LIB_PATH = os.path.join(HERE, 'libcase_b200_torch.so')
_torch_ops = None


def load_torch_ops():
    """Register the torch custom-op layer (TORCH_LIBRARY(case_b200, ...), csrc/torch_ops.cpp) and return
    ``torch.ops.case_b200``.  The ops validate their tensors at the dispatcher boundary and call the same C ABI; only
    CUDA kernels are registered (a CPU tensor fails in the dispatcher: no CPU fallback)."""
    global _torch_ops
    if _torch_ops is None:
        import torch
        load()
        if not os.path.exists(TORCH_LIB_PATH):
            raise RuntimeError(f'{TORCH_LIB_PATH} not found: run `python -c "import __graft_entry__ as g; g.build()"`')
        torch.ops.load_library(TORCH_LIB_PATH)
        _torch_ops = torch.ops.case_b200
    return _torch_ops


def check(rc, what=''):
    if rc != 0:
        msg = load().case_last_error().decode()
        raise RuntimeError(f'libcase_b200 {what} failed (code {rc}): {msg}')


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def call(name, *args):
    check(getattr(load(), name)(*args), name)
