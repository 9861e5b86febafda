"""Banned words, CPU side: the new fields trail the argument blocks, the C ABI refuses a ban it cannot serve before it
launches anything (after the n-best, attribution and constraint refusals), every public face raises ValueError for an
unservable list before any engine is built, and the oracle's banned searches (tests/bad_words_tools.py, on top of the
unchanged oracle) - what the device is compared with on the GPU - take the best allowed ids and never produce a banned
id or sequence."""
import collections
import ctypes
import types

import pytest
import torch

from case_rg_b200 import _lib
from helpers import build_case, build_gttp
from oracle import generations as OG
import bad_words_tools as BT

DUMMY = 0x1000          # a non-null pointer that is never dereferenced: the checks run before any launch
EOS = OG.EOS
BANS = ('ban_mask', 'ban_tok', 'ban_len', 'ban_n')


# ------------------------------------------------------------------------------------------------ shared helpers
def answer_of(row):
    """Answer tokens of a returned row: up to and including EOS; PAD (0) ends it."""
    out = []
    for tk in row:
        if tk == 0:
            break
        out.append(tk)
        if tk == EOS:
            break
    return out


def contains_banned(ys, bad_words):
    """Does the token list ys contain one of the banned sequences contiguously?"""
    for w in bad_words:
        w = [int(v) for v in w]
        if any(ys[i:i + len(w)] == w for i in range(len(ys) - len(w) + 1)):
            return True
    return False


def bans_from_answers(rows, extra=()):
    """A ban list that changes answers: the most frequent answer token (EOS excluded), the first 2- and 3-token window
    of the longest answers, and ``extra``."""
    answers = [answer_of(r) for r in rows]
    freq = collections.Counter(t for ys in answers for t in ys if t != EOS)
    out = [[freq.most_common(1)[0][0]]] if freq else []
    for ys in sorted(answers, key=len, reverse=True)[:3]:
        body = [t for t in ys if t != EOS]
        if len(body) >= 3:
            out += [body[1:3], body[:3]]
    return out + [list(w) for w in extra]


# ------------------------------------------------------------------------------------------------ the C ABI
@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    return _lib.load()


def test_ban_structs_match_the_library(lib):
    for i, st in ((4, _lib.StepBanArgs), (5, _lib.GttpStepBanArgs), (6, _lib.TailBanArgs)):
        assert lib.case_struct_size(i) == ctypes.sizeof(st), st.__name__


def test_ban_fields_trail_the_blocks():
    """ABI version 2 unchanged: the four pointers come after every earlier field, and a block built as an earlier form
    carries them zeroed (no bans)."""
    for base, ext in ((_lib.TailConstrArgs, _lib.TailBanArgs), (_lib.StepConstrArgs, _lib.StepBanArgs),
                      (_lib.GttpStepConstrArgs, _lib.GttpStepBanArgs)):
        assert issubclass(ext, base)
        assert [n for n, _ in ext._fields_] == list(BANS)
        assert ext.ban_mask.offset >= ctypes.sizeof(base)
    for short, full in ((_lib.TailArgs, _lib.TailBanArgs), (_lib.TailConstrArgs, _lib.TailBanArgs),
                        (_lib.StepArgs, _lib.StepBanArgs), (_lib.StepConstrArgs, _lib.StepBanArgs),
                        (_lib.GttpStepArgs, _lib.GttpStepBanArgs), (_lib.GttpStepAttrArgs, _lib.GttpStepBanArgs)):
        a = short()
        assert ctypes.sizeof(a) == ctypes.sizeof(full)
        view = full.from_address(ctypes.addressof(a))
        assert all(getattr(view, n) is None for n in BANS), short.__name__


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


def _step_blocks(opt=0, mode=_lib.MODE_BEAM, attribution=False, bans=BANS, **kw):
    """Step blocks with the given ban pointers set that would pass every other check."""
    ints = dict(dict(B=2, W=2, R=4, V=1000, ldv=1000, Tmax=8, max_len=8, mode=mode, nbest=1, opt=opt), **kw)
    lb = ints.pop('Lb', 10)
    a = _filled(_lib.StepBanArgs, **ints)
    g = _filled(_lib.GttpStepBanArgs, Lb=lb, **ints)
    for x in (a, g):
        x.fork = None
        if not attribution:
            x.attr_cand = x.attr_hist = x.out_attr = None
        for n in BANS:
            if n not in bans:
                setattr(x, n, None)
    a.S[0], a.S[1] = 10, 20
    return a, g


def _both_refused(lib, a, g, word):
    for fn, blk in ((lib.case_decode_step, a), (lib.gttp_decode_step, g)):
        rc = fn(ctypes.byref(blk), 0, None)
        assert rc == 100001 and word in lib.case_last_error(), (rc, lib.case_last_error())


@pytest.mark.parametrize('some', [('ban_mask',), ('ban_tok', 'ban_len', 'ban_n'), ('ban_mask', 'ban_n')])
def test_steps_refuse_partial_ban_pointers(lib, some):
    a, g = _step_blocks(bans=some)
    _both_refused(lib, a, g, b'ban_mask / ban_tok / ban_len / ban_n')


@pytest.mark.parametrize('opt', [_lib.OPT_DENSE_TAIL, _lib.OPT_UNFUSED_TAIL])
def test_steps_refuse_bans_without_the_sparse_tail(lib, opt):
    a, g = _step_blocks(opt)
    _both_refused(lib, a, g, b'banned words need the sparse tail')
    a, g = _step_blocks(0, materialize_only=1)                         # the `generate` face
    _both_refused(lib, a, g, b'banned words need the sparse tail')
    big = lib.case_sparse_tail_max_sources() + 1
    a, g = _step_blocks(0, Lb=big)
    a.S[1] = big
    _both_refused(lib, a, g, b'banned words need the sparse tail')


def test_steps_refuse_bans_in_module_greedy_and_small_vocabularies(lib):
    a, g = _step_blocks(0, mode=_lib.MODE_MODULE_GREEDY, W=1, R=2)
    _both_refused(lib, a, g, b'banned words need CASE_MODE_BEAM')
    a, g = _step_blocks(0, V=12, ldv=16)                               # V >= 2W, but V < 2W + Tmax + 1
    _both_refused(lib, a, g, b'2W + Tmax + 1')


def test_nbest_attribution_and_constraint_refusals_come_first(lib):
    a, g = _step_blocks(_lib.OPT_DENSE_TAIL, bans=('ban_mask',), nbest=3)
    _both_refused(lib, a, g, b'nbest')
    a, g = _step_blocks(_lib.OPT_DENSE_TAIL, bans=('ban_mask',), attribution=True)
    _both_refused(lib, a, g, b'attribution')
    a, g = _step_blocks(_lib.OPT_DENSE_TAIL, bans=('ban_mask',), no_repeat_ngram=-1)
    _both_refused(lib, a, g, b'out of range')


def test_sparse_tail_refuses_partial_ban_pointers(lib):
    ints = dict(R=4, V=1000, W=2, K=2, ldl=1000, ldd=1000, nmem=1, do_finalize=0, fac_ld=16, map_ld=10, gate_ctx=0,
                cp_ld=0, Vext=0, hist_ld=9, t=3, eos=EOS)
    ta = _filled(_lib.TailBanArgs, **ints)
    ta.S[0] = 10
    ta.cp_n = ta.cp_uid = ta.cp_first = ta.cp_start = ta.cp_perm = ta.attr = None
    ta.ban_len = None
    rc = lib.case_sparse_tail(ctypes.byref(ta), DUMMY, DUMMY, DUMMY, 4, None, None, None)
    assert rc == 100001 and b'ban_mask / ban_tok / ban_len / ban_n' in lib.case_last_error(), lib.case_last_error()
    ta.ban_len, ta.hist_anc = DUMMY, None                              # bans need the answer history too
    rc = lib.case_sparse_tail(ctypes.byref(ta), DUMMY, DUMMY, DUMMY, 4, None, None, None)
    assert rc == 100001 and b'history' in lib.case_last_error(), lib.case_last_error()


# ------------------------------------------------------------------------------------------------ the Python faces
def test_check_bad_words_limits(lib):
    from case_rg_b200.engine import BadWords, check_bad_words
    ok = (0, 1000, 4, 100, 20)
    assert check_bad_words(*ok, None) is None and check_bad_words(*ok, []) is None
    bw = check_bad_words(*ok, [[7], torch.tensor([5, 6]), [5, 6], [7], (1, 2, 3)])
    assert bw == BadWords((7,), ((5, 6), (1, 2, 3)))                   # duplicates dropped, tensors taken
    assert check_bad_words(*ok, bw) == bw
    assert check_bad_words(*ok, [list(range(16))] + [[i, i] for i in range(255)]) is not None
    nmax = 1000 - (2 * 4 + 20 + 1)                                     # the most single ids V allows
    assert check_bad_words(*ok, [[i] for i in range(nmax)]) is not None
    bad = [[[1000]], [[-1]], [[]], [[2.0]], [list(range(17))], [[i, i] for i in range(257)],
           [[i] for i in range(nmax + 1)], [[i] for i in range(nmax)] + [[1, 2]], torch.tensor([[1, 2]])]
    for b in bad:
        with pytest.raises(ValueError):
            check_bad_words(*ok, b)
    for args in ((_lib.OPT_DENSE_TAIL, 1000, 4, 100, 20), (_lib.OPT_UNFUSED_TAIL, 1000, 4, 100, 20),
                 (0, 1000, 4, lib.case_sparse_tail_max_sources() + 1, 20), (0, 28, 4, 100, 20)):
        with pytest.raises(ValueError):
            check_bad_words(*args, [[3]])
    with pytest.raises(ValueError):
        check_bad_words(0, 1000, 1, 100, 20, [[3]], _lib.MODE_MODULE_GREEDY)


def _unbuilt(cls, V, opt=0):
    """A model of cls without device state: every face must refuse before it reaches engine_for / the producers."""
    m = cls.__new__(cls)
    m.weights = types.SimpleNamespace(V=V, device='cpu')
    m.opt, m.n_oov, m.use_graph, m._engines = opt, 0, True, {}

    def no_engine(*a, **k):
        raise AssertionError('an engine was built')
    m.engine_for = no_engine
    m.producers = types.SimpleNamespace(__call__=no_engine)
    return m


@pytest.mark.parametrize('family', ['case', 'gttp'])
def test_every_face_refuses_before_building(lib, family):
    from case_rg_b200 import generations as FG
    cls = FG.FastCaSE if family == 'case' else FG.FastGTTP
    V, T = 1000, 10
    lists = [[[V]], [[-1]], [[]], [list(range(17))], [[i, i] for i in range(257)], [[i] for i in range(V - 12)]]
    faces = [lambda m, b: FG.greedy(m, {}, None, T, bad_words=b),
             lambda m, b: FG.beam(m, {}, None, T, 4, bad_words=b),
             lambda m, b: FG.beam_nbest(m, {}, None, T, 4, 2, bad_words=b),
             lambda m, b: FG.beam_attributed(m, {}, None, T, 4, 2, bad_words=b),
             lambda m, b: FG.greedy_attributed(m, {}, None, T, bad_words=b),
             lambda m, b: FG.beam_batches(m, iter([]), None, T, 4, bad_words=b),
             lambda m, b: FG.greedy_batches(m, iter([]), None, T, bad_words=b),
             lambda m, b: m.fast_search({}, T, 4, _lib.MODE_BEAM, bad_words=b)]
    if family == 'case':
        faces.append(lambda m, b: m.search_ids({}, T, 4, mode='beam', bad_words=b))
    for b in lists:
        for face in faces:
            with pytest.raises(ValueError):
                face(_unbuilt(cls, V), b)
    for opt in (_lib.OPT_DENSE_TAIL, _lib.OPT_UNFUSED_TAIL):
        for face in faces:
            with pytest.raises(ValueError):
                face(_unbuilt(cls, V, opt), [[5]])
    with pytest.raises(ValueError):
        _unbuilt(cls, V).fast_search({}, T, 1, _lib.MODE_MODULE_GREEDY, bad_words=[[5]])
    if family == 'case':
        with pytest.raises(ValueError):
            _unbuilt(cls, V).search_ids({}, T, 1, mode='module_greedy', bad_words=[[5]])


# ------------------------------------------------------------------------------------------------ the oracle
def test_banned_ids_with_bad_words():
    b = BT.banned_ids
    assert b([5, 6, 7], 3, bad_words=[[9]]) == [9]
    assert b([5, 6, 7], 3, bad_words=[[7, 8]]) == [8]                  # the answer ends with w_1
    assert b([5, 6, 7], 3, bad_words=[[6, 8]]) == []
    assert b([5, 6, 7], 3, bad_words=[[6, 7, 4], [5, 6, 7, 3], [4, 5, 6, 7, 2]]) == [3, 4]   # L - 1 > t: no match
    assert b([], 0, bad_words=[[9], [1, 2]]) == [9]
    assert b([5, 6], 2, 1, bad_words=[[6, 5], [3]]) == [3, 5, 6]       # the union with the n-gram rule
    assert b([5], 1, 0, 3, bad_words=[[5, 4]]) == [EOS, 4]             # and with min_len


def _problems():
    from oracle.case_decoder import CaseOracle
    from oracle.gttp import GttpOracle
    z, cfg, sd, inp = build_case('case_generations')
    yield 'case', (lambda: CaseOracle(sd).incremental(inp)), int(cfg['B']), int(cfg['T'])
    z, cfg, sd, inp = build_gttp()
    yield 'gttp', (lambda: GttpOracle(sd).stepper(inp)), int(cfg['B']), int(cfg['T'])


@pytest.mark.parametrize('n,m', [(0, 0), (2, 1)])
def test_oracle_banned_greedy_is_the_best_allowed_id(n, m):
    """Brute-force restatement: step by step, the best id of the stepper's dist that no rule bans for the tokens emitted
    so far (EOS at t = 0 becomes UNK, PAD after the end)."""
    for name, factory, B, T in _problems():
        plain = OG.greedy(factory(), T).tolist()
        bans = bans_from_answers(plain)
        got = BT.greedy(factory(), T, no_repeat_ngram=n, min_len=m, bad_words=bans)
        st = factory()
        inp, ended, rows = torch.full((B,), OG.BOS), [False] * B, [[] for _ in range(B)]
        for t in range(T):
            dist = st.advance(torch.arange(B), inp).cpu()
            nxt = []
            for q in range(B):
                ys = rows[q]
                ban = set(BT.banned_ids(ys, t, n, m))
                for w in bans:
                    if len(w) == 1 or (t >= len(w) - 1 and ys[t - len(w) + 1:t] == list(w[:-1])):
                        ban.add(w[-1])
                order = sorted(range(dist.size(1)), key=lambda v: (-float(dist[q, v]), v))
                tk = next(v for v in order if v not in ban)
                end = tk == EOS
                if t == 0 and end:
                    tk = OG.UNK
                elif ended[q]:
                    tk = OG.PAD
                ended[q] = ended[q] or end
                rows[q].append(tk)
                nxt.append(tk)
            inp = torch.tensor(nxt)
        assert torch.equal(got, torch.tensor(rows)), name
        assert got.tolist() != plain, (name, 'the bans must change an answer')
        for q in range(B):
            assert not contains_banned(answer_of(rows[q]), bans), (name, rows[q])


def test_oracle_banned_beams_avoid_every_ban_and_bite():
    changed = 0
    for name, factory, B, T in _problems():
        for W in (2, 4, 8):
            plain = OG.beam(factory(), T, W)
            bans = bans_from_answers(plain.tolist())
            for n, m in ((0, 0), (2, 0), (0, 3), (3, 2)):
                out, best, results = BT.beam(factory(), T, W, return_all=True, no_repeat_ngram=n, min_len=m,
                                             bad_words=bans)
                for q in range(B):
                    for h in results[q]:                                 # every finished hypothesis, not only the best
                        assert not contains_banned(h.tokens[1:], bans), (name, W, n, m, h.tokens)
                        if EOS in h.tokens[1:]:
                            assert h.tokens[1:].index(EOS) >= m
                    assert results[q][0].cum >= 0
                if (n, m) == (0, 0):
                    changed += not torch.equal(out, plain)
    assert changed >= 6, 'the bans taken from the answers must change answers at every width'


def test_a_ban_that_never_matches_is_the_oracle():
    """Sequences longer than an answer can grow ban nothing: the restated loops give the oracle's answers and costs."""
    for name, factory, B, T in _problems():
        never = [[5] * (T + 2), list(range(3, 3 + T + 3))]             # need t >= L - 1 > T - 1
        assert torch.equal(BT.greedy(factory(), T, bad_words=never), OG.greedy(factory(), T)), name
        for W in (2, 4, 8):
            got, gbest, _ = BT.beam(factory(), T, W, return_all=True, bad_words=never)
            want, wbest, _ = OG.beam(factory(), T, W, return_all=True)
            assert torch.equal(got, want), (name, W)
            assert [h.cum for h in gbest] == [h.cum for h in wbest], (name, W)
            got, gbest, _ = BT.beam(factory(), T, W, return_all=True, no_repeat_ngram=T + 1, min_len=0,
                                    bad_words=never)
            assert torch.equal(got, want), (name, W)
