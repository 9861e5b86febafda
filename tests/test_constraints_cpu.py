"""Search constraints, CPU side: the C ABI refuses a constraint request it cannot serve before it launches anything (the
n-best and attribution refusals still come first), the new fields trail the argument blocks, and the oracle's
constrained searches (tests/constraint_tools.py, on top of the unchanged oracle) - what the device is compared with on
the GPU - take the best allowed ids and never repeat an
n-gram or end early."""
import ctypes

import pytest
import torch

from case_rg_b200 import _lib
from helpers import build_case, build_gttp
from oracle import generations as OG
import constraint_tools as CT

DUMMY = 0x1000          # a non-null pointer that is never dereferenced: the checks run before any launch
EOS = OG.EOS


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


def _step_blocks(opt=0, mode=_lib.MODE_BEAM, attribution=False, **kw):
    """Constrained step blocks that would pass every other check (attribution pointers NULL unless asked for)."""
    ints = dict(dict(B=2, W=2, R=4, V=1000, ldv=1000, Tmax=8, max_len=8, mode=mode, nbest=1, opt=opt), **kw)
    lb = ints.pop('Lb', 10)
    a = _filled(_lib.StepConstrArgs, **ints)
    g = _filled(_lib.GttpStepConstrArgs, Lb=lb, **ints)
    for x in (a, g):
        x.fork = None
        if not attribution:
            x.attr_cand = x.attr_hist = x.out_attr = None
    a.S[0], a.S[1] = 10, 20
    return a, g


def _both_refused(lib, a, g, word):
    assert _refused(lib, lib.case_decode_step(ctypes.byref(a), 0, None), word), lib.case_last_error()
    assert _refused(lib, lib.gttp_decode_step(ctypes.byref(g), 0, None), word), lib.case_last_error()


@pytest.mark.parametrize('n,m', [(-1, 0), (9, 0), (0, 8), (0, -1), (2, 9)])
def test_steps_refuse_out_of_range_constraints(lib, n, m):
    a, g = _step_blocks(no_repeat_ngram=n, min_len=m)
    _both_refused(lib, a, g, b'out of range')


@pytest.mark.parametrize('opt', [_lib.OPT_DENSE_TAIL, _lib.OPT_UNFUSED_TAIL])
def test_steps_refuse_constraints_without_the_sparse_tail(lib, opt):
    a, g = _step_blocks(opt, no_repeat_ngram=2)
    _both_refused(lib, a, g, b'sparse tail')
    a, g = _step_blocks(0, min_len=2, materialize_only=1)            # the `generate` face
    _both_refused(lib, a, g, b'sparse tail')
    big = lib.case_sparse_tail_max_sources() + 1
    a, g = _step_blocks(0, no_repeat_ngram=1, Lb=big)
    a.S[1] = big
    _both_refused(lib, a, g, b'sparse tail')


def test_steps_refuse_constraints_in_module_greedy_and_small_vocabularies(lib):
    a, g = _step_blocks(0, mode=_lib.MODE_MODULE_GREEDY, W=1, R=2, no_repeat_ngram=2)
    _both_refused(lib, a, g, b'CASE_MODE_BEAM')
    a, g = _step_blocks(0, V=12, ldv=16, no_repeat_ngram=2)          # V >= 2W, but V < 2W + Tmax + 1
    _both_refused(lib, a, g, b'2W + Tmax + 1')


def test_nbest_and_attribution_refusals_come_first(lib):
    a, g = _step_blocks(_lib.OPT_DENSE_TAIL, nbest=3, no_repeat_ngram=-1)
    _both_refused(lib, a, g, b'nbest')
    a, g = _step_blocks(_lib.OPT_DENSE_TAIL, attribution=True, no_repeat_ngram=-1)
    _both_refused(lib, a, g, b'attribution')


def _tail(**kw):
    ints = dict(R=4, V=1000, W=2, K=2, ldl=1000, ldd=1000, nmem=1, do_finalize=0, fac_ld=16, map_ld=10, gate_ctx=0,
                cp_ld=0, Vext=0, hist_ld=9, t=3, eos=EOS)
    ta = _filled(_lib.TailConstrArgs, **dict(ints, **kw))
    ta.S[0] = 10
    ta.cp_n = ta.cp_uid = ta.cp_first = ta.cp_start = ta.cp_perm = ta.attr = None
    return ta


@pytest.mark.parametrize('kw,word', [(dict(no_repeat_ngram=-1), b'no_repeat_ngram'),
                                     (dict(min_len=_lib.MAX_T), b'min_len'),
                                     (dict(no_repeat_ngram=2, t=9), b'history'),
                                     (dict(min_len=2, V=12), b'V >= 2K')])
def test_sparse_tail_refuses_bad_constraints(lib, kw, word):
    ta = _tail(**kw)
    rc = lib.case_sparse_tail(ctypes.byref(ta), DUMMY, DUMMY, DUMMY, 4, None, None, None)
    assert _refused(lib, rc, word), lib.case_last_error()
    ta = _tail(no_repeat_ngram=2)
    ta.hist_anc = None
    rc = lib.case_sparse_tail(ctypes.byref(ta), DUMMY, DUMMY, DUMMY, 4, None, None, None)
    assert _refused(lib, rc, b'history'), lib.case_last_error()


def test_constraint_fields_trail_the_blocks():
    """ABI version 2 unchanged: the constraint fields come after every earlier field of the tail and step blocks, and a
    block built as TailArgs carries them zeroed (no constraints)."""
    for base, ext, names in ((_lib.TailArgs, _lib.TailConstrArgs,
                              ['hist_tok', 'hist_anc', 'hist_ld', 't', 'eos', 'no_repeat_ngram', 'min_len']),
                             (_lib.StepAttrArgs, _lib.StepConstrArgs, ['no_repeat_ngram', 'min_len']),
                             (_lib.GttpStepAttrArgs, _lib.GttpStepConstrArgs, ['no_repeat_ngram', 'min_len'])):
        assert issubclass(ext, base)
        assert [n for n, _ in ext._fields_] == names
        assert getattr(ext, names[0]).offset >= ctypes.sizeof(base)
    a = _lib.TailArgs()
    full = _lib.TailConstrArgs.from_address(ctypes.addressof(a))
    assert (full.hist_tok, full.hist_anc, full.no_repeat_ngram, full.min_len) == (None, None, 0, 0)


def test_python_faces_refuse_before_building(lib):
    from case_rg_b200.engine import check_constraints
    check_constraints(0, 1000, 4, 100, 10, 0, 0)                    # off: always servable
    check_constraints(0, 1000, 4, 100, 10, 3, 5, 10, _lib.MODE_BEAM)
    for args in ((0, 1000, 4, 100, 10, -1, 0), (0, 1000, 4, 100, 10, 11, 0), (0, 1000, 4, 100, 10, 0, 10),
                 (_lib.OPT_DENSE_TAIL, 1000, 4, 100, 10, 2, 0), (0, 18, 4, 100, 10, 2, 0),
                 (0, 1000, 4, lib.case_sparse_tail_max_sources() + 1, 10, 2, 0)):
        with pytest.raises(ValueError):
            check_constraints(*args)
    with pytest.raises(ValueError):
        check_constraints(0, 1000, 1, 100, 10, 2, 0, 10, _lib.MODE_MODULE_GREEDY)


# ------------------------------------------------------------------------------------------------ the oracle
def test_banned_ids():
    b = CT.banned_ids
    assert b([5, 6, 5], 3, 1) == [5, 6]
    assert b([5, 6, 5], 3, 2) == [6]                              # (5, 6) is in the answer, the answer ends in 5
    assert b([5, 6, 7, 5, 6], 5, 3) == [7]
    assert b([5, 6, 7], 3, 3) == []
    assert b([5, 6], 2, 3) == []                                  # fewer than n tokens: no complete n-gram
    assert b([], 0, 2, min_len=1) == [EOS]
    assert b([5], 1, 0, min_len=1) == []


def _problems():
    from oracle.case_decoder import CaseOracle
    from oracle.gttp import GttpOracle
    z, cfg, sd, inp = build_case('case_generations')
    yield 'case', (lambda: CaseOracle(sd).incremental(inp)), int(cfg['B']), int(cfg['T'])
    z, cfg, sd, inp = build_gttp()
    yield 'gttp', (lambda: GttpOracle(sd).stepper(inp)), int(cfg['B']), int(cfg['T'])


def _answer(row):
    out = []
    for tk in row:
        if tk == 0:
            break
        out.append(tk)
        if tk == EOS:
            break
    return out


def _repeats_ngram(ys, n):
    grams = [tuple(ys[j:j + n]) for j in range(len(ys) - n + 1)]
    return len(grams) != len(set(grams))


@pytest.mark.parametrize('n,m', [(1, 0), (2, 3), (3, 0), (0, 3)])
def test_oracle_constrained_greedy_is_the_best_allowed_id(n, m):
    """Brute-force restatement: step by step, the best id of the stepper's dist that banned_ids allows for the tokens
    emitted so far (EOS at t = 0 becomes UNK, PAD after the end)."""
    for name, factory, B, T in _problems():
        got = CT.greedy(factory(), T, no_repeat_ngram=n, min_len=m)
        st = factory()
        inp, ended, rows = torch.full((B,), OG.BOS), [False] * B, [[] for _ in range(B)]
        for t in range(T):
            dist = st.advance(torch.arange(B), inp).cpu()
            nxt = []
            for b in range(B):
                ban = set(CT.banned_ids(rows[b], t, n, m))
                order = sorted(range(dist.size(1)), key=lambda v: (-float(dist[b, v]), v))
                tk = next(v for v in order if v not in ban)
                end = tk == EOS
                if t == 0 and end:
                    tk = OG.UNK
                elif ended[b]:
                    tk = OG.PAD
                ended[b] = ended[b] or end
                rows[b].append(tk)
                nxt.append(tk)
            inp = torch.tensor(nxt)
        assert torch.equal(got, torch.tensor(rows)), name
        if n:
            for b in range(B):
                ys = [v for v in rows[b] if v != OG.PAD]
                assert not _repeats_ngram(ys, n), (name, ys)


def test_oracle_constrained_beams_satisfy_the_constraints_and_bite():
    bites = 0
    for name, factory, B, T in _problems():
        for W in (2, 4, 8):
            plain = OG.beam(factory(), T, W)
            for b in range(B):
                bites += _repeats_ngram(_answer(plain[b].tolist()), 2)
            for n in (1, 2, 3):
                for m in (0, 3):
                    out, best, results = CT.beam(factory(), T, W, return_all=True, no_repeat_ngram=n, min_len=m)
                    for q in range(B):
                        for h in results[q]:
                            ys = h.tokens[1:]
                            assert not _repeats_ngram(ys, n), (name, W, n, m, ys)
                            if EOS in ys:
                                assert ys.index(EOS) >= m, (name, W, n, m, ys)
                        # the costs are the unconstrained mixture's: cum is a sum of -log(p + 1e-10) >= 0
                        assert results[q][0].cum >= 0
    assert bites >= 1, 'on the golden problems some unconstrained answer repeats a bigram'


def test_restated_search_is_the_oracle_when_nothing_is_banned():
    """With an n longer than any answer nothing is ever banned, so the restated loops of constraint_tools must give the
    oracle's own answers and costs; both values 0 call the oracle itself."""
    for name, factory, B, T in _problems():
        assert torch.equal(CT.greedy(factory(), T, no_repeat_ngram=T + 1), OG.greedy(factory(), T)), name
        assert torch.equal(CT.greedy(factory(), T), OG.greedy(factory(), T)), name
        for W in (2, 4):
            got, gbest, _ = CT.beam(factory(), T, W, return_all=True, no_repeat_ngram=T + 1)
            want, wbest, _ = OG.beam(factory(), T, W, return_all=True)
            assert torch.equal(got, want), (name, W)
            assert [h.cum for h in gbest] == [h.cum for h in wbest], (name, W)
