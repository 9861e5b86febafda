"""n-best lists of the device beam search against the oracle's sorted ``results[q]`` lists (Generations.py:183-185).

fp32 storage: every entry of every list - tokens, lengths - is identical to the oracle's, costs within 1e-4 nats of
its keys, on the golden problems (widths 2 / 4 / 8, every n), at full C2 / C4 and over the extended vocabulary.
bf16 storage: entry 0 is ``beam``'s answer bit for bit, the lists are well formed and every entry's cost agrees with
the oracle's key of the same sequence within the band of the beam parity tests (largest gap recorded as
nbest_<case>.json next to the search parity records).  The public faces (beam_batches, search_ids, the torch ops)
carry the same lists.
"""
import json
import os

import numpy as np
import pytest
import torch

from case_rg_b200 import synthetic as syn
from helpers import build_case, build_gttp, producers_case, H
import parity_tools as PT
from test_gpu_search_parity import OUT, _case_problem

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = {'fp32': 1e-4, 'bf16': 2e-2}


def _record(name, payload):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, f'nbest_{name}.json'), 'w') as f:
        json.dump(payload, f, indent=1, default=float)
    print(f'\nNBEST {name}: ' + json.dumps(payload, default=float))


def _case_data(inp):
    d = inp.to(DEV)
    return dict(mem_q=d.mem_q, mem_p=d.mem_p, query=d.query, passage=d.passage, prior_q=d.prior_q,
                prior_p=d.prior_p, answer_rep=d.answer_rep, source_map=d.source_map)


def _gttp_data(inp):
    d = inp.to(DEV)
    return dict(context=d.context, background=d.background, background_map=d.background_map,
                src_output=d.src_output, bg_output=d.bg_output, init_state=d.init_state)


def _oracle_lists(results, n):
    """results[q][:n] of the oracle's beam -> (tokens int64 [B, n, L], lengths int64 [B, n], keys fp64 [B, n])."""
    B = len(results)
    ents = [results[q][:n] for q in range(B)]
    assert all(len(e) == n for e in ents)
    L = max(len(h.tokens) - 1 for e in ents for h in e)
    toks = torch.zeros(B, n, L, dtype=torch.long)
    lens = torch.zeros(B, n, dtype=torch.long)
    keys = torch.zeros(B, n, dtype=torch.float64)
    for q, e in enumerate(ents):
        for i, h in enumerate(e):
            toks[q, i, :len(h.tokens) - 1] = torch.tensor(h.tokens[1:])
            lens[q, i] = len(h.tokens) - 1
            keys[q, i] = h.cum / h.length
    return toks, lens, keys


def _assert_lists_equal(got, results, n, what):
    """-> largest |cost - oracle key|; tokens and lengths identical, costs within the fp32 gate."""
    toks, lens, keys = _oracle_lists(results, n)
    assert torch.equal(got.tokens.cpu(), toks), (what, got.tokens.cpu(), toks)
    assert torch.equal(got.lengths.cpu(), lens), (what, got.lengths.cpu(), lens)
    gap = float((got.costs.cpu() - keys).abs().max())
    assert gap <= TOL['fp32'], (what, gap)
    return gap


def _same_padded(a, b):
    a, b = a.cpu(), b.cpu()
    L = max(a.size(1), b.size(1))
    return torch.equal(PT._pad(a, L), PT._pad(b, L))


# ------------------------------------------------------------------------------------ 1. golden problems, fp32
@pytest.mark.parametrize('family', ['case', 'gttp'])
def test_fp32_nbest_equals_oracle_results_on_golden_problems(family):
    from case_rg_b200 import generations as FG
    from oracle import generations as OG
    if family == 'case':
        from oracle.case_decoder import CaseOracle
        z, cfg, sd, inp = build_case('case_generations')
        stepper = lambda: CaseOracle(sd).incremental(inp)
        model = FG.FastCaSE(sd, device=DEV, dtype='fp32')
        data = _case_data(inp)
    else:
        from oracle.gttp import GttpOracle
        z, cfg, sd, inp = build_gttp()
        stepper = lambda: GttpOracle(sd).stepper(inp)
        model = FG.FastGTTP(sd, device=DEV, dtype='fp32')
        data = _gttp_data(inp)
    T = int(cfg['T'])
    gaps = {}
    for W in (2, 4, 8):
        _, _, results = OG.beam(stepper(), T, W, return_all=True)
        for n in range(1, W + 1):
            got = FG.beam_nbest(model, data, None, T, W, n)
            gaps[f'w{W}n{n}'] = _assert_lists_equal(got, results, n, (family, W, n))
            if f'beam{W}' in z:                  # the golden has widths 1, 2, 4, 8 (CaSE) and 1, 4, 8 (GTTP)
                assert _same_padded(got.tokens[:, 0], torch.from_numpy(z[f'beam{W}'])), (family, W, n)
    _record(f'golden_{family}_fp32', dict(max_cost_gap_nats=max(gaps.values())))


# ------------------------------------------------------------------------------------ 2./3./4. C2 and C4
def _check_bf16_lists(name, got, ref, factory, B, T, W):
    """bf16: entry 0 == beam, well-formed lists, costs against the oracle's keys of the same sequences."""
    assert _same_padded(got.tokens[:, 0], ref), name
    toks, lens, costs = got.tokens.cpu(), got.lengths.cpu(), got.costs.cpu()
    assert toks.shape[:2] == (B, W) and bool(torch.isfinite(costs).all())
    assert bool((costs[:, 1:] >= costs[:, :-1]).all()), costs
    for q in range(B):
        seqs = {tuple(toks[q, i, :lens[q, i]].tolist()) for i in range(W)}
        assert len(seqs) == W, (q, toks[q])
        for i in range(W):
            n = int(lens[q, i])
            assert 1 <= n <= T and (int(toks[q, i, n - 1]) == syn.EOS or n == T), (q, i, toks[q, i])
            assert not toks[q, i, n:].any()
    _, _, scale = PT.oracle_greedy(factory, B, T)
    tol = TOL['bf16'] * scale
    gap = 0.0
    for i in range(W):
        keys, _, length = PT.oracle_keys(factory, toks[:, i], T)
        assert length == (lens[:, i] + 1).tolist()
        gap = max(gap, float((costs[:, i] - torch.tensor(keys, dtype=torch.float64)).abs().max()))
    _record(name, dict(max_cost_gap_nats=gap, tol_nats=tol, logit_scale=scale))
    assert gap <= tol, (gap, tol)


def _check_n1_and_reuse(FG, model, data, T, W, before):
    """n = 1 through beam_nbest is beam; beam after an n-best call is unchanged."""
    one = FG.beam_nbest(model, data, None, T, W, 1)
    assert one.tokens.shape[1] == 1 and _same_padded(one.tokens[:, 0], before)
    assert torch.equal(FG.beam(model, data, None, T, W).cpu(), before)


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_c2_nbest(dtype):
    """C2 (B=64, beam 4, 10 x 256 passages, V=30522, T=40) on the peaked problem of the search parity tests, n = 4."""
    from case_rg_b200 import generations as FG
    from oracle import generations as OG
    from oracle.case_decoder import CaseOracle
    B, W, T = 64, 4, 40
    sd, inp = _case_problem(B, 60, 10, 256, 51, 61)
    orc = CaseOracle(sd, device=DEV)
    factory = lambda: orc.incremental(inp)
    data = _case_data(inp)
    model = FG.FastCaSE(sd, device=DEV, dtype=dtype)
    before = FG.beam(model, data, None, T, W).cpu()
    got = FG.beam_nbest(model, data, None, T, W, W)
    if dtype == 'fp32':
        _, _, results = OG.beam(factory(), T, W, return_all=True)
        gap = _assert_lists_equal(got, results, W, 'c2')
        _record('c2_fp32', dict(max_cost_gap_nats=gap))
    else:
        _check_bf16_lists('c2_bf16', got, before, factory, B, T, W)
        again = FG.beam_nbest(model, data, None, T, W, W)
        assert all(torch.equal(x, y) for x, y in zip(got, again)), 'the n-best lists are not reproducible run to run'
    _check_n1_and_reuse(FG, model, data, T, W, before)


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_c4_gttp_nbest(dtype):
    """C4: GTTP pointer-generator, B=128, beam 4, V=50,000, Lc=60, Lb=10 x 100, T=40, n = 4."""
    from case_rg_b200 import generations as FG
    from oracle import generations as OG
    from oracle.gttp import GttpOracle
    V, B, W, T = 50000, 128, 4, 40
    sd = syn.make_gttp_state(54, V, H, H, peaked=0.3, boost={syn.EOS: 6.0})
    inp = syn.make_gttp_inputs(64, B, 60, 10, 100, V, H)
    orc = GttpOracle(sd, device=DEV)
    factory = lambda: orc.stepper(inp)
    data = _gttp_data(inp)
    model = FG.FastGTTP(sd, device=DEV, dtype=dtype)
    before = FG.beam(model, data, None, T, W).cpu()
    got = FG.beam_nbest(model, data, None, T, W, W)
    if dtype == 'fp32':
        _, _, results = OG.beam(factory(), T, W, return_all=True)
        gap = _assert_lists_equal(got, results, W, 'c4')
        _record('c4_fp32', dict(max_cost_gap_nats=gap))
    else:
        _check_bf16_lists('c4_bf16', got, before, factory, B, T, W)
    _check_n1_and_reuse(FG, model, data, T, W, before)


# ------------------------------------------------------------------------------------ 5./6./8. the public faces
def _small_case(seed, B, V=3000):
    return syn.make_case_inputs(seed, B, 24, 3, 50, V, H)


def _small_model(FG, **kw):
    sd = syn.make_case_decoder_state(61, 3000, H, peaked=0.3, boost={syn.EOS: 8.0}, gen_gate_bias=2.0)
    return FG.FastCaSE(sd, device=DEV, dtype='bf16', **kw)


def test_beam_batches_nbest_equals_beam_nbest_per_batch():
    """Three host batches, the last a smaller tail batch: the streamed lists equal beam_nbest batch by batch."""
    from case_rg_b200 import generations as FG
    T, W = 10, 4
    model = _small_model(FG)
    inps = [_small_case(71, 6), _small_case(72, 6), _small_case(73, 3)]
    host = [{k: getattr(i, k) for k in FG.FastCaSE._KEYS} for i in inps]
    streamed = list(FG.beam_batches(model, iter(host), None, T, W, n_best=4))
    assert len(streamed) == 3
    for inp, got in zip(inps, streamed):
        want = FG.beam_nbest(model, _case_data(inp), None, T, W, 4)
        assert isinstance(got, FG.NBest) and got.tokens.device.type == 'cpu'
        assert all(torch.equal(x, y.cpu()) for x, y in zip(got, want))
    plain = list(FG.beam_batches(model, iter(host), None, T, W))        # the answers-only stream is unchanged
    for inp, got in zip(inps, plain):
        assert torch.equal(got, FG.beam(model, _case_data(inp), None, T, W).cpu())


def test_search_ids_nbest_entry0_is_the_answer():
    from case_rg_b200 import generations as FG
    cfg, sd_prod, sd_dec, data, _ = producers_case()
    model = FG.FastCaSE(sd_dec, device=DEV, dtype='bf16', producers=sd_prod)
    d = {k: v.to(DEV) for k, v in data.items()}
    out = model.search_ids(d, cfg['T'], 4, mode='beam', n_best=4)
    plain = model.search_ids(d, cfg['T'], 4, mode='beam')
    assert set(out) == {'answer', 'rank', 'nbest'} and set(plain) == {'answer', 'rank'}
    assert torch.equal(out['answer'], plain['answer'])
    assert out['nbest'].tokens.shape[:2] == (cfg['B'], 4)
    assert _same_padded(out['nbest'].tokens[:, 0], out['answer'])
    with pytest.raises(ValueError):
        model.search_ids(d, cfg['T'], 1, mode='greedy', n_best=1)


@pytest.mark.parametrize('graph', [False, True])
def test_torch_op_path_gives_the_same_lists(graph):
    from case_rg_b200 import generations as FG
    from case_rg_b200.engine import CaseDecodeEngine
    T, W = 10, 4
    data = _case_data(_small_case(62, 6))
    want = FG.beam_nbest(_small_model(FG, use_graph=graph), data, None, T, W, W)
    CaseDecodeEngine.use_torch_ops = True
    try:
        got = FG.beam_nbest(_small_model(FG, use_graph=graph), data, None, T, W, W)
    finally:
        CaseDecodeEngine.use_torch_ops = False
    assert all(torch.equal(x, y) for x, y in zip(got, want))


# ------------------------------------------------------------------------------------ 7. extended vocabulary
@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_nbest_over_extended_vocabulary(dtype):
    """The n_oov problem of the GLKS / OOV tests: dynamic ids >= V come back in the lists (tok_ext rows)."""
    from case_rg_b200 import generations as FG
    from oracle import generations as OG
    from oracle.case_decoder import CaseOracle
    V, B, T, W, NO = 3000, 6, 8, 4, 50
    sd = syn.make_case_decoder_state(41, V, H, peaked=0.3, boost={syn.EOS: 6.0}, gen_gate_bias=0.5)
    inp = syn.make_case_inputs(42, B, 24, 4, 40, V, H)
    g = torch.Generator().manual_seed(43)
    oov = torch.rand(inp.source_map.shape, generator=g) < 0.2
    oov &= inp.source_map > 102
    inp.source_map = torch.where(oov, V + torch.randint(0, NO, inp.source_map.shape, generator=g), inp.source_map)
    data = _case_data(inp)
    model = FG.FastCaSE(sd, device=DEV, dtype=dtype, n_oov=NO)
    got = FG.beam_nbest(model, data, None, T, W, W)
    if dtype == 'fp32':
        _, _, results = OG.beam(CaseOracle(sd).incremental(inp, n_oov=NO), T, W, return_all=True)
        assert int(_oracle_lists(results, W)[0].max()) >= V, 'the lists must contain dynamic words'
        _assert_lists_equal(got, results, W, 'oov')
    else:
        assert _same_padded(got.tokens[:, 0], FG.beam(model, data, None, T, W))
        assert int(got.tokens.max()) < V + NO


# ------------------------------------------------------------------------------------ 9. errors
def test_bad_n_raises_before_launch():
    from case_rg_b200 import generations as FG
    from case_rg_b200.engine import CaseDecodeEngine
    model = _small_model(FG)
    data = _case_data(_small_case(62, 2))
    for n, width in ((0, 4), (5, 4), (2, 1), (-1, 4)):
        with pytest.raises(ValueError):
            FG.beam_nbest(model, data, None, 10, width, n)
        with pytest.raises(ValueError):
            FG.beam_batches(model, iter([]), None, 10, width, n_best=n)
    assert not model._engines, 'nothing was built, so nothing was launched'
    with pytest.raises(ValueError):                    # a greedy engine (W = 1) has no n-best list
        CaseDecodeEngine(model.weights, 2, 1, 24, 150, 10, nbest=2)
