"""Attribution records of the device search against the oracle's teacher-forced records (tests/attribution_tools.py).

1. Attribution does not perturb the search: tokens, lengths and costs are bit-identical to ``beam_nbest`` / ``greedy``.
2. Every record is well formed: parts >= 0, ``source_map[source] == token``, source -1 exactly when no copy part, and
   for beam entries sum_j -log(sum parts_j + 1e-10) / (len + 1) is the entry's cost within 1e-5 nats.
3. fp32: every part within 1e-4 * p(y) of the oracle's, sources identical except oracle-scored near-ties, on the golden
   problems (greedy and beam widths 2 / 4 / 8 with n = width), at full C2 and C4 and over the extended vocabulary.
4. bf16: the bf16 search's p(y) is not the oracle's - that gap belongs to the search, and every part inherits it (the
   largest part gap equals the largest gap of p(y) itself).  So bf16 compares what attribution adds: the split of p(y),
   every part / p(y) within 5e-2 of the oracle's part / p(y), and sources identical or oracle-scored near-ties; p(y)
   itself is held to the band of the n-best cost checks (per answer, the mean of log p_device - log p_oracle within
   2e-2 x the oracle's max|logit| nats, tests/parity_tools.py).  The largest gaps are recorded as
   attribution_<case>.json next to the search parity records.
5. The public faces (beam_batches / greedy_batches, search_ids, the torch ops) carry the same records; unservable
   requests raise before anything is built.
"""
import json
import math
import os

import pytest
import torch

from case_rg_b200 import _lib as L, synthetic as syn
from helpers import build_case, build_gttp, producers_case, H
from attribution_tools import teacher_forced_attribution
from test_gpu_nbest import _case_data, _gttp_data, _small_case, _small_model
from test_gpu_search_parity import OUT, _case_problem

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
PARTS_TOL = {'fp32': 1e-4}                      # |device part - oracle part| / p(y)
SOURCE_TIE = {'fp32': 1e-5}                     # a differing source must contribute >= (1 - this) x the oracle's largest
BF16_LOGIT_BAND = 2e-2                          # bf16: tol = this x the oracle's max|logit| nats (tests/parity_tools.py)
BF16_SPLIT_TOL = 5e-2                           # bf16: |device part / p(y) - oracle part / p(y)|
NAMES = ('max_part_gap_rel_p', 'max_p_gap_rel_p', 'max_split_gap', 'max_row_logp_gap_nats', 'sources_differing',
         'max_source_shortfall_rel', 'tol_nats')


def _record(name, payload):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, f'attribution_{name}.json'), 'w') as f:
        json.dump(payload, f, indent=1, default=float)
    print(f'\nATTRIBUTION {name}: ' + json.dumps(payload, default=float))


def _beam_rows(att):
    """beam Attributed -> (tokens [B*n, L], lengths [B*n], costs [B*n], parts [B*n, L, P], source [B*n, L]) on the CPU."""
    nb = att.answer
    B, n, Lm = nb.tokens.shape
    return (nb.tokens.cpu().reshape(B * n, Lm), nb.lengths.cpu().reshape(-1), nb.costs.cpu().reshape(-1),
            att.parts.cpu().reshape(B * n, Lm, -1), att.source.cpu().reshape(B * n, Lm))


def _check_invariants(tokens, parts, source, smap_rows, lengths=None, costs=None):
    assert parts.shape[:2] == tokens.shape and source.shape == tokens.shape
    assert bool((parts >= 0).all()) and bool(torch.isfinite(parts).all())
    has = source >= 0
    got = smap_rows.cpu().long().gather(1, source.clamp(min=0))
    assert torch.equal(got[has], tokens[has]), 'a source position does not map to its token'
    assert torch.equal(~has, (parts[..., 1:] == 0).all(-1)), 'source -1 must mean no copy part'
    if lengths is not None:
        pos = torch.arange(tokens.size(1))[None, :]
        assert bool((parts[pos >= lengths[:, None]] == 0).all()) and bool((source[pos >= lengths[:, None]] == -1).all())
        p = parts.double().sum(-1)
        nll = torch.where(pos < lengths[:, None], -torch.log(p + 1e-10), torch.zeros_like(p)).sum(1)
        gap = float((nll / (lengths.double() + 1) - costs).abs().max())
        assert gap <= 1e-5, gap
        return gap
    return 0.0


def _vs_oracle(dtype, stepper, tokens, parts, source, n=1, lengths=None, proto_greedy=False):
    """-> NAMES: largest part gap / p(y), largest gap of p(y) itself / p(y), largest gap of part / p(y) (the split),
    largest per-row |mean log p_device - log p_oracle|, differing sources, largest relative shortfall of a differing
    source, tol_nats; asserts the dtype's gates.  fp32: parts within 1e-4 p(y), a differing source only where the
    oracle's two largest contributions agree within 1e-5.  bf16: the split within 5e-2, the row's mean log p(y) within
    tol = 2e-2 x logit scale nats, a differing source contributing at least e^-tol x the oracle's largest."""
    P = parts.size(-1)
    rec = teacher_forced_attribution(stepper, tokens, n=n, lengths=lengths, proto_greedy=proto_greedy, parts=P,
                                     probe=source)
    v = rec['valid']
    po = rec['p'].clamp(min=1e-30)
    gap = ((parts.double() - rec['parts']).abs().amax(-1) / po)[v]
    gap = float(gap.max()) if gap.numel() else 0.0
    pd = parts.double().sum(-1)
    pgap = ((pd - rec['p']).abs() / po)[v]
    pgap = float(pgap.max()) if pgap.numel() else 0.0
    split = ((parts.double() / pd.clamp(min=1e-30)[..., None] - rec['parts'] / po[..., None]).abs().amax(-1))[v]
    split = float(split.max()) if split.numel() else 0.0
    dlog = torch.where(v, torch.log(pd.clamp(min=1e-30)) - torch.log(po), torch.zeros_like(po))
    rowgap = float((dlog.sum(1) / v.sum(1).clamp(min=1)).abs().max())
    diff = (source != rec['source']) & v
    top = rec['top2'][..., 0]
    short = ((top - rec['at_probe']) / top.clamp(min=1e-30))[diff]
    short = float(short.max()) if short.numel() else 0.0
    if dtype == 'fp32':
        tol = 0.0
        assert gap <= PARTS_TOL['fp32'], (dtype, gap)
        t2 = rec['top2'][diff]   # a differing source: the oracle's two largest contributions agree within 1e-5
        assert bool(((t2[:, 0] - t2[:, 1]) <= SOURCE_TIE['fp32'] * t2[:, 0]).all()), t2
    else:
        tol = BF16_LOGIT_BAND * rec['logit_scale']
        assert split <= BF16_SPLIT_TOL, (dtype, split, gap, pgap)
        assert rowgap <= tol, (dtype, rowgap, tol)
        assert short <= -math.expm1(-tol), (dtype, int(diff.sum()), short, tol)
    return gap, pgap, split, rowgap, int(diff.sum()), short, tol


def _greedy_check(dtype, att, plain, stepper, smap):
    assert torch.equal(att.answer.cpu(), plain.cpu())
    toks, parts, src = att.answer.cpu(), att.parts.cpu(), att.source.cpu()
    _check_invariants(toks, parts, src, smap)
    return _vs_oracle(dtype, stepper, toks, parts, src, proto_greedy=True)


# ------------------------------------------------------------------------------------ 3. golden problems, fp32
@pytest.mark.parametrize('family', ['case', 'gttp'])
def test_fp32_records_equal_oracle_on_golden_problems(family):
    from case_rg_b200 import generations as FG
    if family == 'case':
        from oracle.case_decoder import CaseOracle
        z, cfg, sd, inp = build_case('case_generations')
        stepper = lambda: CaseOracle(sd).incremental(inp)
        model, data, smap = FG.FastCaSE(sd, device=DEV, dtype='fp32'), _case_data(inp), inp.source_map
    else:
        from oracle.gttp import GttpOracle
        z, cfg, sd, inp = build_gttp()
        stepper = lambda: GttpOracle(sd).stepper(inp)
        model, data, smap = FG.FastGTTP(sd, device=DEV, dtype='fp32'), _gttp_data(inp), inp.background_map
    T = int(cfg['T'])
    gaps = {'greedy': _greedy_check('fp32', FG.greedy_attributed(model, data, None, T), FG.greedy(model, data, None, T),
                                    stepper(), smap)}
    for W in (2, 4, 8):
        att = FG.beam_attributed(model, data, None, T, W, W)
        ref = FG.beam_nbest(model, data, None, T, W, W)
        assert all(torch.equal(x, y) for x, y in zip(att.answer, ref))
        toks, lens, costs, parts, src = _beam_rows(att)
        _check_invariants(toks, parts, src, smap.repeat_interleave(W, 0), lens, costs)
        gaps[f'beam{W}'] = _vs_oracle('fp32', stepper(), toks, parts, src, n=W, lengths=lens)
    _record(f'golden_{family}_fp32', gaps)


# ------------------------------------------------------------------------------------ 1./2./3./4. C2 and C4
def _c2():
    sd, inp = _case_problem(64, 60, 10, 256, 51, 61)
    return sd, inp, _case_data(inp), inp.source_map, 3


def _c4():
    V, B = 50000, 128
    sd = syn.make_gttp_state(54, V, H, H, peaked=0.3, boost={syn.EOS: 6.0})
    inp = syn.make_gttp_inputs(64, B, 60, 10, 100, V, H)
    return sd, inp, _gttp_data(inp), inp.background_map, 2


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
@pytest.mark.parametrize('case', ['c2', 'c4'])
def test_attribution_search_is_the_plain_search_and_matches_the_oracle(case, dtype):
    """C2: CaSE, B=64, beam 4, 10 x 256 passages, V=30522, T=40; C4: GTTP, B=128, beam 4, V=50,000, Lb=10 x 100, T=40;
    beam with n = 4 and greedy, with and without the CUDA graph."""
    from case_rg_b200 import generations as FG
    W, T = 4, 40
    sd, inp, data, smap, P = (_c2 if case == 'c2' else _c4)()
    if case == 'c2':
        from oracle.case_decoder import CaseOracle
        orc = CaseOracle(sd, device=DEV)
        stepper = lambda: orc.incremental(inp)
        make = lambda g: FG.FastCaSE(sd, device=DEV, dtype=dtype, use_graph=g)
    else:
        from oracle.gttp import GttpOracle
        orc = GttpOracle(sd, device=DEV)
        stepper = lambda: orc.stepper(inp)
        make = lambda g: FG.FastGTTP(sd, device=DEV, dtype=dtype, use_graph=g)
    atts = {}
    for graph in (False, True):
        model = make(graph)
        ref = FG.beam_nbest(model, data, None, T, W, W)
        att = FG.beam_attributed(model, data, None, T, W, W)
        assert all(torch.equal(x, y) for x, y in zip(att.answer, ref)), (case, dtype, graph)
        g_att, g_ref = FG.greedy_attributed(model, data, None, T), FG.greedy(model, data, None, T)
        assert torch.equal(g_att.answer, g_ref), (case, dtype, graph)
        assert torch.equal(FG.beam_nbest(model, data, None, T, W, W).costs, ref.costs)   # the plain engine is unchanged
        atts[graph] = (att, g_att)
    for x, y in zip(atts[False], atts[True]):                      # graph replay and eager steps give the same records
        assert torch.equal(x.parts, y.parts) and torch.equal(x.source, y.source)
    att, g_att = atts[True]
    toks, lens, costs, parts, src = _beam_rows(att)
    cost_gap = _check_invariants(toks, parts, src, smap.repeat_interleave(W, 0), lens, costs)
    _check_invariants(g_att.answer.cpu(), g_att.parts.cpu(), g_att.source.cpu(), smap)
    beam = _vs_oracle(dtype, stepper(), toks, parts, src, n=W, lengths=lens)
    greedy = _vs_oracle(dtype, stepper(), g_att.answer.cpu(), g_att.parts.cpu(), g_att.source.cpu(), proto_greedy=True)
    _record(f'{case}_{dtype}', dict(beam=dict(zip(NAMES, beam)), greedy=dict(zip(NAMES, greedy)),
                                    max_cost_gap_nats=cost_gap, copied=int((src >= 0).sum() + (g_att.source >= 0).sum())))


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_records_over_extended_vocabulary(dtype):
    """The n_oov problem of the n-best tests: dynamic ids >= V have no generation part and are copied only."""
    from case_rg_b200 import generations as FG
    from oracle.case_decoder import CaseOracle
    V, B, T, W, NO = 3000, 6, 8, 4, 50
    sd = syn.make_case_decoder_state(41, V, H, peaked=0.3, boost={syn.EOS: 6.0}, gen_gate_bias=0.5)
    inp = syn.make_case_inputs(42, B, 24, 4, 40, V, H)
    g = torch.Generator().manual_seed(43)
    oov = torch.rand(inp.source_map.shape, generator=g) < 0.2
    oov &= inp.source_map > 102
    inp.source_map = torch.where(oov, V + torch.randint(0, NO, inp.source_map.shape, generator=g), inp.source_map)
    model = FG.FastCaSE(sd, device=DEV, dtype=dtype, n_oov=NO)
    data = _case_data(inp)
    att = FG.beam_attributed(model, data, None, T, W, W)
    assert all(torch.equal(x, y) for x, y in zip(att.answer, FG.beam_nbest(model, data, None, T, W, W)))
    toks, lens, costs, parts, src = _beam_rows(att)
    _check_invariants(toks, parts, src, inp.source_map.repeat_interleave(W, 0), lens, costs)
    dyn = toks >= V
    assert bool(dyn.any()), 'the answers must contain dynamic words'
    assert bool((parts[..., 0][dyn] == 0).all()) and bool((src[dyn] >= 0).all())
    gap = _vs_oracle(dtype, CaseOracle(sd).incremental(inp, n_oov=NO), toks, parts, src, n=W, lengths=lens)
    _record(f'oov_{dtype}', dict(zip(NAMES, gap)))


# ------------------------------------------------------------------------------------ 5. the public faces
def test_streamed_batches_carry_the_records():
    """Three host batches, the last a smaller tail batch: the streamed Attributed equal the per-batch calls."""
    from case_rg_b200 import generations as FG
    T, W = 10, 4
    model = _small_model(FG)
    inps = [_small_case(71, 6), _small_case(72, 6), _small_case(73, 3)]
    host = [{k: getattr(i, k) for k in FG.FastCaSE._KEYS} for i in inps]

    def same(got, want):
        assert isinstance(got, FG.Attributed) and got.parts.device.type == 'cpu'
        a, b = got.answer, want.answer
        assert all(torch.equal(x, y.cpu()) for x, y in zip(a, b)) if isinstance(a, FG.NBest) else torch.equal(a, b.cpu())
        assert torch.equal(got.parts, want.parts.cpu()) and torch.equal(got.source, want.source.cpu())

    for n in (2, None):
        streamed = list(FG.beam_batches(model, iter(host), None, T, W, n_best=n, attribution=True))
        assert len(streamed) == 3
        for inp, got in zip(inps, streamed):
            same(got, FG.beam_attributed(model, _case_data(inp), None, T, W, n))
    gmodel = _small_model(FG)
    streamed = list(FG.greedy_batches(gmodel, iter(host), None, T, attribution=True))
    for inp, got in zip(inps, streamed):
        same(got, FG.greedy_attributed(gmodel, _case_data(inp), None, T))
    plain = list(FG.beam_batches(model, iter(host), None, T, W))       # the answers-only stream is unchanged
    for inp, got in zip(inps, plain):
        assert torch.equal(got, FG.beam(model, _case_data(inp), None, T, W).cpu())


def test_search_ids_attribution_in_every_mode():
    from case_rg_b200 import generations as FG
    cfg, sd_prod, sd_dec, data, _ = producers_case()
    model = FG.FastCaSE(sd_dec, device=DEV, dtype='bf16', producers=sd_prod)
    d = {k: v.to(DEV) for k, v in data.items()}
    T, B = cfg['T'], cfg['B']
    for mode, width in (('beam', 4), ('greedy', 1), ('module_greedy', 1)):
        plain = model.search_ids(d, T, width, mode=mode)
        out = model.search_ids(d, T, width, mode=mode, attribution=True)
        assert set(out) == {'answer', 'rank', 'attribution'}
        assert torch.equal(out['answer'], plain['answer']) and torch.equal(out['attribution'].answer, out['answer'])
        att = out['attribution']
        assert att.parts.shape == (*out['answer'].shape, 3) and att.source.shape == out['answer'].shape
        toks = out['answer'].cpu()
        _check_invariants(toks, att.parts.cpu(), att.source.cpu(), data['source_map'])
        if mode == 'module_greedy':          # no end rule: every position holds the record of its argmax
            assert bool((att.parts.sum(-1) > 0).all())
    out = model.search_ids(d, T, 4, mode='beam', n_best=4, attribution=True)
    assert set(out) == {'answer', 'rank', 'nbest', 'attribution'}
    assert out['attribution'].answer is out['nbest'] and out['attribution'].parts.shape[:2] == (B, 4)
    with pytest.raises(ValueError):
        model.search_ids(d, T, 1, mode='greedy', n_best=1, attribution=True)


@pytest.mark.parametrize('graph', [False, True])
def test_torch_op_path_gives_the_same_records(graph):
    from case_rg_b200 import generations as FG
    from case_rg_b200.engine import CaseDecodeEngine
    T, W = 10, 4
    data = _case_data(_small_case(62, 6))
    want = FG.beam_attributed(_small_model(FG, use_graph=graph), data, None, T, W, W)
    CaseDecodeEngine.use_torch_ops = True
    try:
        got = FG.beam_attributed(_small_model(FG, use_graph=graph), data, None, T, W, W)
    finally:
        CaseDecodeEngine.use_torch_ops = False
    assert all(torch.equal(x, y) for x, y in zip(got.answer, want.answer))
    assert torch.equal(got.parts, want.parts) and torch.equal(got.source, want.source)


def test_unservable_requests_raise_before_launch():
    from case_rg_b200 import generations as FG
    from case_rg_b200.engine import CaseDecodeEngine, GttpDecodeEngine
    data = _case_data(_small_case(62, 2))
    for opt in (L.OPT_DENSE_TAIL, L.OPT_UNFUSED_TAIL):
        model = _small_model(FG, opt=opt)
        with pytest.raises(ValueError):
            FG.beam_attributed(model, data, None, 10, 4)
        with pytest.raises(ValueError):
            FG.greedy_attributed(model, data, None, 10)
        with pytest.raises(ValueError):
            next(FG.beam_batches(model, iter([]), None, 10, 4, attribution=True), None)
        assert not model._engines, 'nothing was built, so nothing was launched'
    model = _small_model(FG)
    for n, width in ((0, 4), (5, 4), (-1, 4)):
        with pytest.raises(ValueError):
            FG.beam_attributed(model, data, None, 10, width, n)
    assert not model._engines
    with pytest.raises(ValueError):                     # more source positions than the sparse tail's table holds
        CaseDecodeEngine(model.weights, 2, 4, 24, L.load().case_sparse_tail_max_sources(), 10, attribution=True)
    _, _, sd, _ = build_gttp()
    gw = FG.FastGTTP(sd, device=DEV, dtype='bf16').weights
    with pytest.raises(ValueError):
        GttpDecodeEngine(gw, 2, 4, 10, 16, 10, opt=L.OPT_DENSE_TAIL, attribution=True)
