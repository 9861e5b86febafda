"""Banned words on the device against the banned oracle search of tests/bad_words_tools.py (the oracle's own searches with
each row's banned ids masked).  The ban lists are taken from the unbanned answers, so every list changes answers.

1. Kernel: case_vocab_base + the constrained case_sparse_tail with a ban mask and a sequence table give the exact top-k
   of the dense mixture (case_row_tail) with the banned ids masked - banned copy targets and base top entries, matching
   and non-matching sequences, hash and plan mode, with and without the finaliser, and rows whose whole global top-16 is
   banned (the exact pass, counted by case_debug_sparse_tail_fallbacks).
2. fp32: tokens identical to the banned oracle and costs within 1e-4 nats, with and without the CUDA graph, on the golden
   problems (CaSE and GTTP; greedy, beam 2 / 4 / 8, alone and with no_repeat_ngram / min_len), at full C2 and C4 and
   over the extended vocabulary.
3. bf16 at C2 and C4: no answer or n-best entry contains a banned id or sequence, and the oracle-scored tie criterion of
   tests/parity_tools.py gives no miss.
4. Composition with n-best and attribution, one captured graph serving two lists, and the streamed faces.
"""
import ctypes as C
import json
import os

import pytest
import torch

from case_rg_b200 import _lib as L, synthetic as syn
from helpers import build_case, build_gttp, H
import parity_tools as PT
import bad_words_tools as BT
from test_bad_words_cpu import answer_of, bans_from_answers, contains_banned
from test_gpu_nbest import _case_data, _gttp_data, _oracle_lists, _small_case, _small_model
from test_gpu_search_parity import OUT, _case_problem

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
EOS, UNK = syn.EOS, 100
SPECIALS = [UNK, 101, 102, 103]                         # [UNK] [CLS] [SEP] [MASK] of the BERT-uncased ids


def _record(name, payload):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, f'bad_words_{name}.json'), 'w') as f:
        json.dump(payload, f, indent=1, default=float)
    print(f'\nBAD_WORDS {name}: ' + json.dumps(payload, default=float))


def _clean(rows, bans):
    """Rows (lists of ids) that contain a banned id or sequence."""
    return [r for r in rows if contains_banned(answer_of(r), bans)]


# ------------------------------------------------------------------------------------------------ 1. the kernel
@pytest.mark.timeout(120)
@pytest.mark.parametrize('finalize,plan', [(1, 0), (1, 1), (0, 0)])
@pytest.mark.parametrize('mode', ['mix', 'fallback'])
def test_banned_sparse_tail_matches_masked_dense_tail(finalize, plan, mode):
    """History Tmax = 20, t = 14 reached through a shuffled ancestry.  'mix': the mask bans copy targets and base top
    entries, and the table holds sequences that match some rows (ending in a copy target and in a base top entry) and
    one that matches none; 'fallback': the mask bans every row's global top-16 base ids, so every row takes the exact
    pass."""
    from case_rg_b200.engine import BadWords, _BanBuffers, build_copy_plan
    torch.manual_seed(17 + finalize * 3 + plan)
    dev, f32 = 'cuda', dict(dtype=torch.float32, device='cuda')
    R, W, K, V, S0, S1 = 8, 4, 4, 30522, 60, 2560
    B, MS, Tmax, t = R // W, L.MAX_SPLIT, 20, 14
    TL, ldv = Tmax + 1, -(-V // 8) * 8
    ns, S, nmem = (1, 3), (S0, S1), (2 if finalize else 1)
    logits = torch.randn(R, ldv, **f32) * 3
    hN = torch.randn(R, H, **f32)
    Wm, bm = torch.randn(3, 3 * H, **f32) * 0.05, torch.randn(3, **f32)
    stats = [torch.rand(R, n, 4, **f32) + 0.1 for n in ns]
    ctxp = [torch.randn(R, n, H, **f32) for n in ns]
    attn = [torch.randn(R, s, **f32) for s in S]
    attn[1][:, ::5] = float('-inf')
    prior = [torch.rand(B, s, **f32) for s in S]
    smap = torch.randint(3, V, (B, S0 + S1), device=dev, dtype=torch.int32)
    lgv = logits[:, :V].clone()
    if not finalize:
        lgv[:, 0] = float('-inf')
    top16 = lgv.topk(16, dim=1).indices.int()
    smap[:, S0 + 3] = top16[::W, 1]                          # a base top entry that is also a copy target
    gates, fac = torch.rand(R, 4, **f32), torch.rand(R, 2, MS, **f32)
    fac[:, :, 1] = 0.5
    hist = torch.randint(3, V, (R, TL), device=dev, dtype=torch.int32)
    rows = torch.arange(R, device=dev)
    anc = torch.stack([(rows // W) * W + (rows % W + j) % W for j in range(TL)], 1).int()
    ans = torch.randint(3, V, (R, t), device=dev, dtype=torch.int32)
    for r in range(R):
        for j in range(1, t + 1):
            hist[r if j == t else int(anc[r, j]), j] = ans[r, j - 1]
    st = torch.cuda.current_stream().cuda_stream

    def args(cp=None):
        a = L.TailBanArgs()
        a.R, a.V, a.W, a.K, a.ldl, a.ldd, a.mask_col0, a.nmem, a.do_finalize = R, V, W, K, ldv, ldv, 1 - finalize, nmem, finalize
        a.fac_ld, a.map_ld = 2 * MS, S0 + S1
        keep = dict(ctx=[torch.zeros(R, H, **f32) for _ in range(2)], gates=gates.clone(), fac=fac.clone(),
                    tv=torch.zeros(R, K, **f32), ti=torch.zeros(R, K, dtype=torch.int32, device=dev),
                    dist=torch.zeros(R, ldv, **f32))
        for i in range(nmem):
            j = i if finalize else 1
            a.ns[i], a.fac_off[i], a.map_off[i], a.S[i] = ns[j], i * MS, (0, S0)[j], S[j]
            a.stats[i], a.ctxp[i], a.ctx[i] = stats[j].data_ptr(), ctxp[j].data_ptr(), keep['ctx'][i].data_ptr()
            a.prior[i], a.attn_un[i] = (prior[j].data_ptr() if finalize else None), attn[j].data_ptr()
        a.logits, a.hN, a.Wm, a.bm = logits.data_ptr(), hN.data_ptr(), Wm.data_ptr(), bm.data_ptr()
        a.gates, a.fac, a.map = keep['gates'].data_ptr(), keep['fac'].data_ptr(), smap.data_ptr()
        a.top_vals, a.top_idx = keep['tv'].data_ptr(), keep['ti'].data_ptr()
        if cp is not None:
            a.cp_n, a.cp_uid, a.cp_first = cp['n'].data_ptr(), cp['uid'].data_ptr(), cp['first'].data_ptr()
            a.cp_start, a.cp_perm, a.cp_ld = cp['start'].data_ptr(), cp['perm'].data_ptr(), S0 + S1 + 1
        return a, keep

    lib = L.load()
    cp = None
    if plan:
        valid = torch.ones(B, S0 + S1, dtype=torch.bool, device=dev)
        valid[:, S0::5] = False
        cp = dict(n=torch.zeros(B, dtype=torch.int32, device=dev),
                  **{k: torch.zeros(B, S0 + S1 + 1, dtype=torch.int32, device=dev) for k in ('uid', 'first', 'start', 'perm')})
        build_copy_plan(smap, valid, V, cp['n'], cp['uid'], cp['first'], cp['start'], cp['perm'])
    a, dense = args()
    a.dist = dense['dist'].data_ptr()
    L.check(lib.case_row_tail(C.byref(a), st), 'case_row_tail')
    torch.cuda.synchronize()
    d = dense['dist'][:, :V].double().cpu()
    ref_top = torch.argsort(-d, dim=1, stable=True)[:, :K]     # the unbanned top-k
    A = ans.cpu().tolist()
    if mode == 'mix':
        # copy targets, base top entries, and the unbanned winners of rows 0 and 2
        singles = {int(smap[0, 5]), int(smap[1, S0 + 7]), int(top16[0, 0]), int(top16[5, 0]), int(smap[1, S0 + 3]),
                   int(ref_top[0, 0])}
        seqs = [(A[0][-2], A[0][-1], int(top16[0, 1])),       # row 0: its second base entry
                (A[2][-1], int(ref_top[2, 1])),               # row 2: its second unbanned winner
                (A[6][-1], int(smap[1, 9])),                  # row 6: a copy target of its query
                (A[3][-1], int(smap[0, S0 + 11])),            # row 3
                (V - 1, V - 2, int(top16[2, 0]))]             # matches no row
    else:
        singles = {int(v) for v in top16.reshape(-1).tolist()}
        seqs = [(A[1][-1], int(smap[0, 4]))]
    bw = BadWords(tuple(sorted(singles)), tuple(seqs))
    bans = _BanBuffers(torch.device(dev), V)
    bans.write(bw)
    k2 = 2 * L.MAX_W
    base_ms, base_e = torch.zeros(R, 4, 2, **f32), torch.zeros(R, 4, k2, **f32)
    base_i = torch.zeros(R, 4, k2, dtype=torch.int32, device=dev)
    L.call('case_vocab_base', logits.data_ptr(), ldv, R, V, 1 - finalize, k2, base_ms.data_ptr(), base_e.data_ptr(),
           base_i.data_ptr(), st)
    counter = torch.zeros(1, dtype=torch.int32, device=dev)
    lib.case_debug_sparse_tail_fallbacks.argtypes = [C.c_void_p]
    a2, sparse = args(cp)
    a2.hist_tok, a2.hist_anc, a2.hist_ld, a2.t, a2.eos = hist.data_ptr(), anc.data_ptr(), TL, t, EOS
    bans.bind(a2)
    lib.case_debug_sparse_tail_fallbacks(counter.data_ptr())
    try:
        L.check(lib.case_sparse_tail(C.byref(a2), base_ms.data_ptr(), base_e.data_ptr(), base_i.data_ptr(), k2, None, None,
                                     st), 'case_sparse_tail(bans)')
    finally:
        lib.case_debug_sparse_tail_fallbacks(None)
    torch.cuda.synchronize()
    banned = torch.zeros(R, V, dtype=torch.bool)
    matched = 0
    for r in range(R):
        ids = BT.banned_ids(A[r], t, bad_words=[[v] for v in bw.singles] + [list(s) for s in bw.seqs])
        banned[r, ids] = True
        matched += len(set(ids) - set(bw.singles))
    if mode == 'mix':
        assert matched >= 4, 'four sequences match their rows'
        assert bool(banned.gather(1, ref_top).any()), 'the bans must hit the unbanned top-k'
    dm = d.masked_fill(banned, float('-inf'))
    want = torch.argsort(-dm, dim=1, stable=True)[:, :K]
    got_i, got_v = sparse['ti'].cpu().long(), sparse['tv'].cpu()
    assert not bool(banned.gather(1, got_i.clamp(max=V - 1)).any()), 'a banned id was chosen'
    ref_v = torch.gather(dense['dist'][:, :V].cpu(), 1, got_i)
    assert torch.allclose(got_v, ref_v, rtol=1e-5, atol=0), (got_v, ref_v)
    same = got_i == want
    if not bool(same.all()):
        wv = torch.gather(dense['dist'][:, :V].cpu(), 1, want)
        assert torch.allclose(wv[~same], ref_v[~same], rtol=1e-5, atol=0), (got_i, want)
    nfb = int(counter.item())
    if mode == 'fallback':
        assert nfb == R, nfb
    _record(f'kernel_{mode}_fin{finalize}_plan{plan}', dict(fallback_rows=nfb, rows=R, matched_sequences=matched))


# ------------------------------------------------------------------------------------------------ 2. fp32 vs the oracle
def _golden(family, graph):
    from case_rg_b200 import generations as FG
    if family == 'case':
        from oracle.case_decoder import CaseOracle
        z, cfg, sd, inp = build_case('case_generations')
        return (lambda: CaseOracle(sd).incremental(inp), FG.FastCaSE(sd, device=DEV, dtype='fp32', use_graph=graph),
                _case_data(inp), int(cfg['T']))
    from oracle.gttp import GttpOracle
    z, cfg, sd, inp = build_gttp()
    return (lambda: GttpOracle(sd).stepper(inp), FG.FastGTTP(sd, device=DEV, dtype='fp32', use_graph=graph),
            _gttp_data(inp), int(cfg['T']))


@pytest.mark.parametrize('family', ['case', 'gttp'])
def test_fp32_golden_problems_equal_banned_oracle(family):
    from case_rg_b200 import generations as FG
    from oracle import generations as OG
    gaps, changed = {}, 0
    for graph in (False, True):
        stepper, model, data, T = _golden(family, graph)
        g_bans = bans_from_answers(OG.greedy(stepper(), T).tolist())
        for n, m in ((0, 0), (2, 1)):
            want = BT.greedy(stepper(), T, no_repeat_ngram=n, min_len=m, bad_words=g_bans)
            got = FG.greedy(model, data, None, T, no_repeat_ngram=n, min_len=m, bad_words=g_bans).cpu()
            assert torch.equal(got, want), (family, graph, n, m)
            for W in (2, 4, 8):
                plain = OG.beam(stepper(), T, W)
                bans = bans_from_answers(plain.tolist())
                out, _, results = BT.beam(stepper(), T, W, return_all=True, no_repeat_ngram=n, min_len=m,
                                          bad_words=bans)
                toks, lens, keys = _oracle_lists(results, W)
                nb = FG.beam_nbest(model, data, None, T, W, W, no_repeat_ngram=n, min_len=m, bad_words=bans)
                Lm = max(nb.tokens.size(2), toks.size(2))
                pad = lambda x: torch.nn.functional.pad(x, (0, Lm - x.size(2)))
                assert torch.equal(pad(nb.tokens.cpu()), pad(toks)), (family, graph, n, m, W)
                assert torch.equal(nb.lengths.cpu(), lens)
                gap = float((nb.costs.cpu() - keys).abs().max())
                assert gap <= 1e-4, gap
                gaps[f'{n}_{m}_beam{W}'] = max(gaps.get(f'{n}_{m}_beam{W}', 0.0), gap)
                assert not _clean(nb.tokens.reshape(-1, nb.tokens.size(2)).cpu().tolist(), bans)
                if (n, m) == (0, 0):
                    changed += not torch.equal(PT._pad(nb.tokens[:, 0].cpu(), Lm), PT._pad(plain, Lm))
    assert changed >= 3, changed
    _record(f'golden_{family}_fp32', dict(max_cost_gap_nats=gaps, changed_answer_sets=changed))


def _c4():
    V, B = 50000, 128
    sd = syn.make_gttp_state(54, V, H, H, peaked=0.3, boost={syn.EOS: 6.0})
    inp = syn.make_gttp_inputs(64, B, 60, 10, 100, V, H)
    return sd, inp, _gttp_data(inp)


class _Rec:
    def __init__(self, st):
        self.st, self.B, self.scale = st, st.B, 0.0

    def advance(self, parents, tokens):
        d = self.st.advance(parents, tokens)
        self.scale = max(self.scale, PT.logit_scale(self.st))
        return d


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
@pytest.mark.parametrize('case', ['c2', 'c4'])
def test_full_size_search_vs_banned_oracle(case, dtype):
    """C2 (CaSE, B=64, beam 4, V=30522, T=40) and C4 (GTTP, B=128, beam 4, V=50,000, T=40), the ban list taken from the
    unbanned answers plus the special ids: fp32 identical to the oracle (costs within 1e-4 nats), bf16 with no miss under
    the oracle-scored tie criterion; no answer or n-best entry holds a ban; no list is the plain search."""
    from case_rg_b200 import generations as FG
    W, T = 4, 40
    if case == 'c2':
        from oracle.case_decoder import CaseOracle
        sd, inp = _case_problem(64, 60, 10, 256, 51, 61)
        data = _case_data(inp)
        orc = CaseOracle(sd, device=DEV)
        factory = lambda: orc.incremental(inp)
        make = lambda g: FG.FastCaSE(sd, device=DEV, dtype=dtype, use_graph=g)
    else:
        from oracle.gttp import GttpOracle
        sd, inp, data = _c4()
        orc = GttpOracle(sd, device=DEV)
        factory = lambda: orc.stepper(inp)
        make = lambda g: FG.FastGTTP(sd, device=DEV, dtype=dtype, use_graph=g)
    out = {}
    for graph in (False, True):
        model = make(graph)
        plain = FG.beam_nbest(model, data, None, T, W, W)
        B = plain.tokens.size(0)
        if not graph:
            bans = bans_from_answers(plain.tokens[:, 0].cpu().tolist(), [[v] for v in SPECIALS])
            rec = _Rec(factory())
            want_b, _, results = BT.beam(rec, T, W, return_all=True, bad_words=bans)
            keys = torch.tensor([results[q][0].cum / results[q][0].length for q in range(B)], dtype=torch.float64)
            want_g = BT.greedy(factory(), T, min_len=1, bad_words=bans)      # min_len 1: no t = 0 EOS -> UNK
            tol = {'fp32': 1e-4, 'bf16': 2e-2}[dtype] * rec.scale
            out['unbanned_answers_with_a_ban'] = len(_clean(plain.tokens[:, 0].cpu().tolist(), bans))
            assert out['unbanned_answers_with_a_ban'] >= 1
        none = FG.beam_nbest(model, data, None, T, W, W, bad_words=[])
        assert all(torch.equal(x, y) for x, y in zip(plain, none)), 'an empty list must be the plain search'
        nb = FG.beam_nbest(model, data, None, T, W, W, bad_words=bans)
        got_b = nb.tokens[:, 0].cpu()
        got_g = FG.greedy(model, data, None, T, min_len=1, bad_words=bans).cpu()
        assert not _clean(nb.tokens.reshape(B * W, -1).cpu().tolist(), bans)
        assert not _clean(got_g.tolist(), bans)
        if dtype == 'fp32':
            Lm = max(got_b.size(1), want_b.size(1))
            assert torch.equal(PT._pad(got_b, Lm), PT._pad(want_b, Lm)), (case, graph)
            gap = float((nb.costs[:, 0].cpu() - keys).abs().max())
            assert gap <= 1e-4, gap
            assert torch.equal(got_g, want_g), (case, graph)
            out[f'graph{int(graph)}'] = dict(max_cost_gap_nats=gap)
        else:
            res = PT.compare_beam(factory, got_b, want_b, T, tol)
            res.pop('details')
            assert res['miss'] == 0, res
            out[f'graph{int(graph)}'] = dict(beam=res, greedy_identical_rows=int((got_g == want_g).all(1).sum()), rows=B)
    out['bans'] = len(bans)
    _record(f'{case}_{dtype}', out)


def test_extended_vocabulary_fp32():
    """n_oov problem: fixed ids banned, the sequences compared on the returned (extended) ids."""
    from case_rg_b200 import generations as FG
    from oracle.case_decoder import CaseOracle
    V, B, T, W, NO = 3000, 6, 12, 4, 50
    sd = syn.make_case_decoder_state(41, V, H, peaked=0.3, boost={syn.EOS: 6.0}, gen_gate_bias=0.5)
    inp = syn.make_case_inputs(42, B, 24, 4, 40, V, H)
    g = torch.Generator().manual_seed(43)
    oov = torch.rand(inp.source_map.shape, generator=g) < 0.2
    oov &= inp.source_map > 102
    inp.source_map = torch.where(oov, V + torch.randint(0, NO, inp.source_map.shape, generator=g), inp.source_map)
    model = FG.FastCaSE(sd, device=DEV, dtype='fp32', n_oov=NO)
    data = _case_data(inp)
    plain = FG.beam(model, data, None, T, W).cpu()
    bans = [w for w in bans_from_answers(plain.tolist()) if all(v < V for v in w)]
    assert bans
    nb = FG.beam_nbest(model, data, None, T, W, W, bad_words=bans)
    assert not _clean(nb.tokens.reshape(B * W, -1).cpu().tolist(), bans)
    out, _, results = BT.beam(CaseOracle(sd).incremental(inp, n_oov=NO), T, W, return_all=True, bad_words=bans)
    toks, lens, keys = _oracle_lists(results, W)
    Lm = max(nb.tokens.size(2), toks.size(2))
    pad = lambda x: torch.nn.functional.pad(x, (0, Lm - x.size(2)))
    assert torch.equal(pad(nb.tokens.cpu()), pad(toks))
    assert float((nb.costs.cpu() - keys).abs().max()) <= 1e-4
    g_tok = FG.greedy(model, data, None, T, bad_words=bans).cpu()
    assert torch.equal(g_tok, BT.greedy(CaseOracle(sd).incremental(inp, n_oov=NO), T, bad_words=bans))
    with pytest.raises(ValueError):                              # dynamic ids cannot be banned by value
        FG.beam(model, data, None, T, W, bad_words=[[V + 1]])


# ------------------------------------------------------------------------------------------------ 4. composition, reuse
def test_attribution_and_nbest_compose():
    """Attribution on and off give bit-identical tokens, lengths and costs; the parts still sum to p(y)."""
    from case_rg_b200 import generations as FG
    T, W = 12, 4
    model = _small_model(FG)
    data = _case_data(_small_case(81, 6))
    bans = bans_from_answers(FG.beam(model, data, None, T, W).cpu().tolist(), [[UNK]])
    for n, m in ((0, 0), (2, 3)):
        att = FG.beam_attributed(model, data, None, T, W, W, no_repeat_ngram=n, min_len=m, bad_words=bans)
        nb = FG.beam_nbest(model, data, None, T, W, W, no_repeat_ngram=n, min_len=m, bad_words=bans)
        assert all(torch.equal(x, y) for x, y in zip(att.answer, nb))
        B = nb.tokens.size(0)
        assert not _clean(nb.tokens.reshape(B * W, -1).cpu().tolist(), bans)
        lens = nb.lengths.reshape(-1).cpu()
        parts = att.parts.reshape(B * W, -1, 3).cpu().double()
        pos = torch.arange(parts.size(1))[None, :]
        p = parts.sum(-1)
        nll = torch.where(pos < lens[:, None], -torch.log(p + 1e-10), torch.zeros_like(p)).sum(1)
        gap = float((nll / (lens.double() + 1) - nb.costs.reshape(-1).cpu()).abs().max())
        assert gap <= 1e-5, gap
        g = FG.greedy_attributed(model, data, None, T, no_repeat_ngram=n, min_len=m, bad_words=bans)
        assert torch.equal(g.answer, FG.greedy(model, data, None, T, no_repeat_ngram=n, min_len=m, bad_words=bans))
    _record('compose', dict(max_cost_gap_nats=gap))


def test_one_graph_serves_every_list():
    """Two lists back to back through one engine and its one captured graph: each answer equals its own oracle, so the
    list content is not frozen into the capture; the streamed faces equal single calls."""
    from case_rg_b200 import generations as FG
    stepper, model, data, T = _golden('case', True)
    W = 4
    from oracle import generations as OG
    plain = OG.beam(stepper(), T, W).tolist()
    first = bans_from_answers(plain)
    second = [[w[0]] for w in first[1:]] + [[EOS]]
    answers = []
    for bans in (first, second, first):
        got = FG.beam(model, data, None, T, W, bad_words=bans).cpu()
        want = BT.beam(stepper(), T, W, bad_words=bans)
        Lm = max(got.size(1), want.size(1))
        assert torch.equal(PT._pad(got, Lm), PT._pad(want, Lm))
        answers.append(PT._pad(got, T))
    assert not torch.equal(answers[0], answers[1]) and torch.equal(answers[0], answers[2])
    engines = [e for k, e in model._engines.items() if k[-1] is True]
    assert len(engines) == 1 and len(engines[0]._graphs) == 1
    # the streamed faces: the list is written once per call, the answers equal single calls
    bmodel = _small_model(FG)
    inps = [_small_case(71, 6), _small_case(72, 6), _small_case(73, 3)]
    host = [{k: getattr(i, k) for k in FG.FastCaSE._KEYS} for i in inps]
    bans = bans_from_answers(FG.beam(bmodel, _case_data(inps[0]), None, 10, W).cpu().tolist(), [[UNK]])
    streamed = list(FG.beam_batches(bmodel, iter(host), None, 10, W, bad_words=bans))
    for inp, got in zip(inps, streamed):
        assert torch.equal(got, FG.beam(bmodel, _case_data(inp), None, 10, W, bad_words=bans).cpu())
        assert not _clean(got.tolist(), bans)
    streamed = list(FG.greedy_batches(bmodel, iter(host), None, 10, bad_words=bans))
    for inp, got in zip(inps, streamed):
        assert torch.equal(got, FG.greedy(bmodel, _case_data(inp), None, 10, bad_words=bans).cpu())


def test_unservable_requests_raise_before_launch():
    from case_rg_b200 import generations as FG
    from case_rg_b200.engine import CaseDecodeEngine
    data = _case_data(_small_case(62, 2))
    for opt in (L.OPT_DENSE_TAIL, L.OPT_UNFUSED_TAIL):
        model = _small_model(FG, opt=opt)
        with pytest.raises(ValueError):
            FG.beam(model, data, None, 10, 4, bad_words=[[5]])
        assert not model._engines
    model = _small_model(FG)
    with pytest.raises(ValueError):
        model.fast_search(data, 10, 1, L.MODE_MODULE_GREEDY, bad_words=[[5]])
    with pytest.raises(ValueError):
        FG.beam(model, data, None, 10, 4, bad_words=[[3000]])
    assert not model._engines
    eng = CaseDecodeEngine(model.weights, 2, 1, 72, 150, 10, bans=True)
    with pytest.raises(ValueError):
        eng.launch(10, L.MODE_MODULE_GREEDY, use_graph=False)
    with pytest.raises(ValueError):
        eng.step_distribution(0)
    with pytest.raises(ValueError):
        CaseDecodeEngine(model.weights, 2, 1, 72, 150, 10).set_bad_words([[5]])
