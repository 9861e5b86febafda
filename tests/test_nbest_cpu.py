"""n-best lists of the beam search, CPU side: the C ABI refuses an n-best request it cannot serve before it launches
anything, and the oracle's sorted ``results[q]`` list - what the device n-best list is compared with on the GPU - has
at least ``width`` entries for every query, with element 0 the reference's answer."""
import ctypes

import numpy as np
import pytest

from case_rg_b200 import _lib
from helpers import build_case, build_gttp

DUMMY = 0x1000          # a non-null pointer that is never dereferenced: the checks run before any launch


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    return _lib.load()


def _filled(struct_type, **ints):
    """An argument block with every pointer field set to DUMMY and the given int fields."""
    a = struct_type()
    for name, ctype in struct_type._fields_:
        if ctype is ctypes.c_void_p:
            setattr(a, name, DUMMY)
        elif isinstance(ctype, type) and issubclass(ctype, ctypes.Array) and ctype._type_ is ctypes.c_void_p:
            for i in range(ctype._length_):
                getattr(a, name)[i] = DUMMY
    for k, v in ints.items():
        setattr(a, k, v)
    return a


def _select_args(mode, W, nbest):
    return _filled(_lib.SelectArgs, mode=mode, B=2, W=W, t=0, max_len=4, Tmax=4, BOS=1, EOS=2, UNK=100, PAD=0,
                   nbest=nbest)


def _refused(lib, rc):
    return rc == 100001 and b'nbest' in lib.case_last_error()


@pytest.mark.parametrize('mode,W,nbest', [(_lib.MODE_BEAM, 2, 3), (_lib.MODE_BEAM, 4, 5), (_lib.MODE_BEAM, 8, 9),
                                          (_lib.MODE_BEAM, 4, -1), (_lib.MODE_PROTO_GREEDY, 1, 2),
                                          (_lib.MODE_MODULE_GREEDY, 1, 2), (_lib.MODE_PROTO_GREEDY, 2, 2)])
def test_beam_select_refuses_bad_nbest_without_touching_the_gpu(lib, mode, W, nbest):
    a = _select_args(mode, W, nbest)
    assert _refused(lib, lib.case_beam_select(ctypes.byref(a), None)), lib.case_last_error()


def test_fused_select_refuses_bad_nbest_without_touching_the_gpu(lib):
    ta = _filled(_lib.TailArgs, R=4, V=1000, W=2, K=2, ldl=1000, ldd=1000, nmem=1, do_finalize=0, fac_ld=16,
                 map_ld=10, gate_ctx=0, cp_ld=0, Vext=0)
    ta.S[0] = 10
    ta.cp_n = ta.cp_uid = ta.cp_first = ta.cp_start = ta.cp_perm = None
    sel = _select_args(_lib.MODE_BEAM, 2, 3)
    rc = lib.case_sparse_tail(ctypes.byref(ta), DUMMY, DUMMY, DUMMY, 4, ctypes.byref(sel), DUMMY, None)
    assert _refused(lib, rc), lib.case_last_error()


@pytest.mark.parametrize('mode,nbest', [(_lib.MODE_BEAM, 3), (_lib.MODE_PROTO_GREEDY, 2)])
def test_step_orchestrators_refuse_bad_nbest_before_the_first_launch(lib, mode, nbest):
    a = _filled(_lib.StepArgs, B=2, W=2, R=4, V=1000, ldv=1000, Tmax=8, max_len=8, mode=mode, nbest=nbest)
    a.fork = None
    assert _refused(lib, lib.case_decode_step(ctypes.byref(a), 0, None)), lib.case_last_error()
    g = _filled(_lib.GttpStepArgs, B=2, W=2, R=4, V=1000, ldv=1000, Tmax=8, max_len=8, mode=mode, nbest=nbest)
    g.fork = None
    assert _refused(lib, lib.gttp_decode_step(ctypes.byref(g), 0, None)), lib.case_last_error()


def test_nbest_mirrors_are_the_last_fields():
    """nbest is appended (ABI version 2 unchanged): every earlier field keeps its offset."""
    for st in (_lib.SelectArgs, _lib.StepArgs, _lib.GttpStepArgs):
        assert st._fields_[-1] == ('nbest', ctypes.c_int32), st.__name__


# ------------------------------------------------------------------------------------------------ the oracle's lists
def _check_results(results, want, width, B):
    for q in range(B):
        res = results[q]
        assert len(res) >= width, (q, len(res))
        keys = [h.cum / h.length for h in res]
        assert keys == sorted(keys)
        first = res[0].tokens[1:]
        assert np.array_equal(np.asarray(first), want[q, :len(first)]) and not want[q, len(first):].any(), (q, first)


@pytest.mark.parametrize('width', [2, 4, 8])
def test_oracle_results_fill_nbest_case(width):
    from oracle import generations as G
    from oracle.case_decoder import CaseOracle
    z, cfg, sd, inp = build_case('case_generations')
    B, T = int(cfg['B']), int(cfg['T'])
    out, best, results = G.beam(CaseOracle(sd).incremental(inp), T, width, return_all=True)
    assert np.array_equal(out.numpy(), z[f'beam{width}'])
    _check_results(results, z[f'beam{width}'], width, B)


@pytest.mark.parametrize('width', [2, 4, 8])
def test_oracle_results_fill_nbest_gttp(width):
    from oracle import generations as G
    from oracle.gttp import GttpOracle
    z, cfg, sd, inp = build_gttp()
    B, T = int(cfg['B']), int(cfg['T'])
    out, best, results = G.beam(GttpOracle(sd).stepper(inp), T, width, return_all=True)
    want = z[f'beam{width}'] if f'beam{width}' in z else out.numpy()    # the golden has widths 1, 4 and 8
    assert np.array_equal(out.numpy(), want)
    _check_results(results, want, width, B)
