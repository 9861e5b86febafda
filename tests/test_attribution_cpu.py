"""Attribution records, CPU side: the C ABI refuses an attribution request it cannot serve before it launches anything
(and the n-best refusals still come first with every pointer set), the oracle's teacher-forced records - what the
device records are compared with on the GPU - add up to the oracle's distribution and point at positions that map to
the token, and ``results.source_location`` decodes a source position."""
import ctypes

import pytest
import torch

from case_rg_b200 import _lib
from case_rg_b200.results import source_location
from helpers import build_case, build_gttp
from attribution_tools import teacher_forced_attribution

DUMMY = 0x1000          # a non-null pointer that is never dereferenced: the checks run before any launch


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    return _lib.load()


def _filled(struct_type, **ints):
    """An argument block with every pointer field (inherited ones included) set to DUMMY and the given int fields."""
    a = struct_type()
    for cls in reversed(struct_type.__mro__):
        for name, ctype in cls.__dict__.get('_fields_', []):
            if ctype is ctypes.c_void_p:
                setattr(a, name, DUMMY)
            elif isinstance(ctype, type) and issubclass(ctype, ctypes.Array) and ctype._type_ is ctypes.c_void_p:
                for i in range(ctype._length_):
                    getattr(a, name)[i] = DUMMY
    for k, v in ints.items():
        setattr(a, k, v)
    return a


def _refused(lib, rc, word):
    return rc == 100001 and word in lib.case_last_error()


def _step_blocks(opt, nbest=1, mode=_lib.MODE_BEAM, **kw):
    ints = dict(dict(B=2, W=2, R=4, V=1000, ldv=1000, Tmax=8, max_len=8, mode=mode, nbest=nbest, opt=opt), **kw)
    lb = ints.pop('Lb', 10)
    a = _filled(_lib.StepAttrArgs, **ints)
    a.fork = None
    g = _filled(_lib.GttpStepAttrArgs, Lb=lb, **ints)
    g.fork = None
    return a, g


@pytest.mark.parametrize('opt', [_lib.OPT_DENSE_TAIL, _lib.OPT_UNFUSED_TAIL, _lib.OPT_DENSE_TAIL | _lib.OPT_UNFUSED_TAIL])
def test_steps_refuse_attribution_without_the_sparse_tail(lib, opt):
    a, g = _step_blocks(opt)
    a.S[0], a.S[1] = 10, 20
    assert _refused(lib, lib.case_decode_step(ctypes.byref(a), 0, None), b'sparse tail'), lib.case_last_error()
    assert _refused(lib, lib.gttp_decode_step(ctypes.byref(g), 0, None), b'sparse tail'), lib.case_last_error()


def test_steps_refuse_attribution_on_other_unservable_steps(lib):
    a, g = _step_blocks(0, materialize_only=1)                       # the `generate` face: no top-k, no records
    a.S[0], a.S[1] = 10, 20
    assert _refused(lib, lib.case_decode_step(ctypes.byref(a), 0, None), b'sparse tail'), lib.case_last_error()
    assert _refused(lib, lib.gttp_decode_step(ctypes.byref(g), 0, None), b'sparse tail'), lib.case_last_error()
    a, g = _step_blocks(0, V=3)                                      # V < 2W
    a.S[0], a.S[1] = 10, 20
    assert _refused(lib, lib.case_decode_step(ctypes.byref(a), 0, None), b'sparse tail'), lib.case_last_error()
    assert _refused(lib, lib.gttp_decode_step(ctypes.byref(g), 0, None), b'sparse tail'), lib.case_last_error()
    big = lib.case_sparse_tail_max_sources() + 1                     # too many source positions for the tail's table
    a, g = _step_blocks(0, Lb=big)
    a.S[0], a.S[1] = 10, big
    assert _refused(lib, lib.case_decode_step(ctypes.byref(a), 0, None), b'sparse tail'), lib.case_last_error()
    assert _refused(lib, lib.gttp_decode_step(ctypes.byref(g), 0, None), b'sparse tail'), lib.case_last_error()


def test_steps_refuse_a_partial_attribution_request(lib):
    a, g = _step_blocks(_lib.OPT_DENSE_TAIL)
    a.S[0], a.S[1] = 10, 20
    a.attr_hist = g.attr_hist = None
    assert _refused(lib, lib.case_decode_step(ctypes.byref(a), 0, None), b'attr_hist'), lib.case_last_error()
    assert _refused(lib, lib.gttp_decode_step(ctypes.byref(g), 0, None), b'attr_hist'), lib.case_last_error()


@pytest.mark.parametrize('mode,nbest', [(_lib.MODE_BEAM, 3), (_lib.MODE_PROTO_GREEDY, 2)])
def test_bad_nbest_is_refused_first_with_every_pointer_set(lib, mode, nbest):
    """Every pointer set is a valid attribution request, so the n-best refusal still wins - also with a dense tail."""
    for opt in (0, _lib.OPT_DENSE_TAIL):
        a, g = _step_blocks(opt, nbest=nbest, mode=mode)
        assert _refused(lib, lib.case_decode_step(ctypes.byref(a), 0, None), b'nbest'), lib.case_last_error()
        assert _refused(lib, lib.gttp_decode_step(ctypes.byref(g), 0, None), b'nbest'), lib.case_last_error()
    sel = _filled(_lib.SelectAttrArgs, mode=mode, B=2, W=2, t=0, max_len=4, Tmax=4, BOS=1, EOS=2, UNK=100, PAD=0,
                  nbest=nbest)
    assert _refused(lib, lib.case_beam_select(ctypes.byref(sel), None), b'nbest'), lib.case_last_error()


def test_select_refuses_a_partial_attribution_request(lib):
    sel = _filled(_lib.SelectAttrArgs, mode=_lib.MODE_BEAM, B=2, W=2, t=0, max_len=4, Tmax=4, BOS=1, EOS=2, UNK=100,
                  PAD=0, nbest=2)
    sel.attr_cand = None
    assert _refused(lib, lib.case_beam_select(ctypes.byref(sel), None), b'attr_cand'), lib.case_last_error()


def test_fused_select_needs_the_tail_records(lib):
    ta = _filled(_lib.TailArgs, R=4, V=1000, W=2, K=2, ldl=1000, ldd=1000, nmem=1, do_finalize=0, fac_ld=16,
                 map_ld=10, gate_ctx=0, cp_ld=0, Vext=0)
    ta.S[0] = 10
    ta.cp_n = ta.cp_uid = ta.cp_first = ta.cp_start = ta.cp_perm = None
    ta.attr = None                                                   # the select asks for records the tail does not write
    sel = _filled(_lib.SelectAttrArgs, mode=_lib.MODE_BEAM, B=2, W=2, t=0, max_len=4, Tmax=4, BOS=1, EOS=2, UNK=100,
                  PAD=0, nbest=2)
    rc = lib.case_sparse_tail(ctypes.byref(ta), DUMMY, DUMMY, DUMMY, 4, ctypes.byref(sel), DUMMY, None)
    assert _refused(lib, rc, b'attr_cand'), lib.case_last_error()


def test_attribution_fields_trail_the_blocks():
    """ABI version 2 unchanged: the record is 16 bytes and the attribution pointers come after every earlier field."""
    assert ctypes.sizeof(_lib.Attr) == 16
    for base, ext in ((_lib.SelectArgs, _lib.SelectAttrArgs), (_lib.StepArgs, _lib.StepAttrArgs),
                      (_lib.GttpStepArgs, _lib.GttpStepAttrArgs)):
        assert issubclass(ext, base)
        assert [n for n, _ in ext._fields_] == ['attr_cand', 'attr_hist', 'out_attr']
        assert ext.attr_cand.offset >= ctypes.sizeof(base)
    assert _lib.TailArgs._fields_[-1] == ('attr', ctypes.c_void_p)


# ------------------------------------------------------------------------------------------------ the oracle's records
def _check_records(rec, tokens, smap_rows, P):
    """Parts are >= 0 and sum to dist[y]; a source maps to the token; source -1 exactly when no copy part."""
    parts, src, valid = rec['parts'], rec['source'], rec['valid']
    assert parts.shape[-1] == P
    assert bool((parts >= 0).all())
    gap = (parts.sum(-1) - rec['p']).abs()[valid]
    assert float(gap.max()) <= 1e-6, float(gap.max())
    N, L = src.shape
    for i in range(N):
        for j in range(L):
            s = int(src[i, j])
            if s >= 0:
                assert int(smap_rows[i, s]) == int(tokens[i, j]), (i, j, s)
            assert (s == -1) == bool((parts[i, j, 1:] == 0).all()) or not valid[i, j], (i, j)
    assert bool((src >= 0).any()), 'the golden problems copy tokens'


@pytest.mark.parametrize('family', ['case', 'gttp'])
def test_oracle_records_on_golden_problems(family):
    import numpy as np
    from oracle import generations as OG
    if family == 'case':
        from oracle.case_decoder import CaseOracle
        z, cfg, sd, inp = build_case('case_generations')
        factory = lambda: CaseOracle(sd).incremental(inp)
        smap, P = inp.source_map, 3
    else:
        from oracle.gttp import GttpOracle
        z, cfg, sd, inp = build_gttp()
        factory = lambda: GttpOracle(sd).stepper(inp)
        smap, P = inp.background_map, 2
    B, T = int(cfg['B']), int(cfg['T'])
    greedy = torch.from_numpy(z['greedy']).long()
    rec = teacher_forced_attribution(factory(), greedy, proto_greedy=True, parts=P)
    _check_records(rec, greedy, smap, P)
    W = 4
    _, _, results = OG.beam(factory(), T, W, return_all=True)
    L = max(len(h.tokens) - 1 for q in range(B) for h in results[q][:W])
    toks = torch.zeros(B * W, L, dtype=torch.long)
    lens = torch.zeros(B * W, dtype=torch.long)
    keys = []
    for q in range(B):
        for i, h in enumerate(results[q][:W]):
            toks[q * W + i, :len(h.tokens) - 1] = torch.tensor(h.tokens[1:])
            lens[q * W + i] = len(h.tokens) - 1
            keys.append(h.cum / h.length)
    rec = teacher_forced_attribution(factory(), toks, n=W, lengths=lens, parts=P)
    _check_records(rec, toks, smap.repeat_interleave(W, 0), P)
    # the records reproduce the search's own costs: sum_j -log(p_j + 1e-10) / (len + 1)
    cost = [float(sum(-np.log(float(p) + 1e-10) for p in rec['parts'][i, :int(lens[i])].sum(-1))) / (int(lens[i]) + 1)
            for i in range(B * W)]
    assert max(abs(a - b) for a, b in zip(cost, keys)) < 1e-5


# ------------------------------------------------------------------------------------------------ source_location
def test_source_location():
    S0, Lp = 10, 12
    assert source_location(-1, S0, Lp) == (-1, -1, -1)
    assert source_location(0, S0, Lp) == (0, -1, 0)
    assert source_location(9, S0, Lp) == (0, -1, 9)
    assert source_location(10, S0, Lp) == (1, 0, 0)
    assert source_location(10 + 12 * 2 + 5, S0, Lp) == (1, 2, 5)
    src = torch.tensor([[-1, 3, 10], [21, 22, 45]])
    m, p, o = source_location(src, S0, Lp)
    assert torch.equal(m, torch.tensor([[-1, 0, 1], [1, 1, 1]]))
    assert torch.equal(p, torch.tensor([[-1, -1, 0], [0, 1, 2]]))
    assert torch.equal(o, torch.tensor([[-1, 3, 0], [11, 0, 11]]))
    for s in range(-1, S0 + 3 * Lp):
        assert tuple(int(x) for x in (t[0] for t in source_location(torch.tensor([s]), S0, Lp))) == \
            source_location(s, S0, Lp)
