"""Search constraints on the device (no_repeat_ngram / min_len) against the constrained oracle search of
tests/constraint_tools.py (the oracle's own searches with the banned ids masked).

1. Kernel: case_vocab_base + the constrained case_sparse_tail give the exact top-k of the dense mixture (case_row_tail)
   with the banned ids masked - banned copy targets, banned base top entries, the EOS ban, hash and plan mode, a row
   whose base top-k2 is mostly banned (the exact pass over the logits) and a banned dynamic id (Vext).
2. fp32: tokens identical to the constrained oracle and costs within 1e-4 nats, with and without the CUDA graph, on the
   golden problems (greedy; beam 2 / 4 / 8), at full C2 and C4 and over the extended vocabulary.
3. bf16: every answer satisfies the constraints; against the constrained oracle the oracle-scored tie criterion of
   tests/parity_tools.py gives no miss at C2 and C4.
4. Off is unchanged, the constraints compose with n-best and attribution, the public faces carry them, unservable
   requests raise before anything is built, and at C2 the unconstrained beam repeats trigrams the constrained one
   does not.
"""
import ctypes as C
import json
import os

import pytest
import torch

from case_rg_b200 import _lib as L, synthetic as syn
from helpers import build_case, build_gttp, producers_case, H
import parity_tools as PT
import constraint_tools as CT
from test_gpu_nbest import _case_data, _gttp_data, _small_case, _small_model
from test_gpu_search_parity import OUT, _case_problem

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
EOS = syn.EOS


def _record(name, payload):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, f'constraints_{name}.json'), 'w') as f:
        json.dump(payload, f, indent=1, default=float)
    print(f'\nCONSTRAINTS {name}: ' + json.dumps(payload, default=float))


def _answer(row):
    """Answer tokens of a row: up to and including EOS, PAD (0) ends it."""
    out = []
    for tk in row:
        if tk == 0:
            break
        out.append(tk)
        if tk == EOS:
            break
    return out


def _violations(rows, n, m, greedy=False):
    """Rows (lists of ids) that repeat an n-gram or end before min_len (greedy: the t = 0 EOS -> UNK rewrite ends a row
    too, but with m >= 1 it cannot happen)."""
    bad = []
    for i, row in enumerate(rows):
        ys = _answer(row) if not greedy else [t for t in row if t != 0]
        if n:
            grams = [tuple(ys[j:j + n]) for j in range(len(ys) - n + 1)]
            if len(grams) != len(set(grams)):
                bad.append((i, 'ngram', ys))
        if m and EOS in ys and ys.index(EOS) < m:
            bad.append((i, 'min_len', ys))
    return bad


def _repeats(rows, n):
    return sum(1 for row in rows if len({tuple(_answer(row)[j:j + n]) for j in range(len(_answer(row)) - n + 1)})
               != max(0, len(_answer(row)) - n + 1))


# ------------------------------------------------------------------------------------------------ 1. the kernel
@pytest.mark.timeout(120)
@pytest.mark.parametrize('R,W,V,S0,S1,K,finalize,plan,mode', [
    (8, 4, 30522, 60, 2560, 4, 1, 0, 'copy'), (8, 4, 30522, 60, 2560, 4, 1, 1, 'copy'),
    (8, 4, 30522, 60, 2560, 4, 1, 0, 'fallback'), (8, 4, 30522, 60, 2560, 4, 1, 1, 'fallback'),
    (6, 2, 4000, 1, 500, 2, 0, 0, 'copy'), (6, 2, 4000, 1, 500, 2, 0, 0, 'fallback'),
    (8, 8, 5003, 16, 100, 8, 1, 0, 'eos')])
def test_constrained_sparse_tail_matches_masked_dense_tail(R, W, V, S0, S1, K, finalize, plan, mode):
    """History (Tmax = 20, t = 14, rows reached through a shuffled ancestry) with n = 1: every answer token is banned.
    'copy': the answers hold copy targets and base top entries; 'fallback': the answers hold 13 of the row's 16 best base
    ids, so fewer than 2K allowed ids remain among them; 'eos': EOS is the row's best id and min_len bans it."""
    from case_rg_b200.engine import build_copy_plan
    torch.manual_seed(R * 131 + V + S1 + plan)
    dev, f32 = 'cuda', dict(dtype=torch.float32, device='cuda')
    B, MS, Tmax, t = R // W, L.MAX_SPLIT, 20, 14
    TL = Tmax + 1
    ldv = -(-V // 8) * 8
    ns, S, nmem = (1, 3), (S0, S1), (2 if finalize else 1)
    logits = torch.randn(R, ldv, **f32) * 3
    logits[:, 7] = logits[:, 3]
    if mode == 'eos':
        logits[:, EOS] = logits[:, :V].max(1).values + 3.0
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
    st = torch.cuda.current_stream().cuda_stream
    gates, fac = torch.rand(R, 4, **f32), torch.rand(R, 2, MS, **f32)
    fac[:, :, 1] = 0.5
    # answers: rows of the query in the history table, reached through anc (row r's position j lives in row anc[r][j])
    hist = torch.randint(3, V, (R, TL), device=dev, dtype=torch.int32)
    # position j < t of row r lives in another row of its query (a permutation of the query's rows per position)
    rows = torch.arange(R, device=dev)
    anc = torch.stack([(rows // W) * W + (rows % W + j) % W for j in range(TL)], 1).int()
    ans = torch.zeros(R, t, dtype=torch.int32, device=dev)       # the answer each row sees
    for r in range(R):
        b = r // W
        if mode == 'copy':
            ans[r] = torch.cat([smap[b, S0 + 3:S0 + 4], smap[b, :3], smap[b, S0 + 10:S0 + 14], top16[r, :2],
                                hist[r, :t - 10]])
        elif mode == 'fallback':                             # 13 of the row's 16 best base ids
            ans[r] = torch.cat([top16[r, :13], smap[b, S0:S0 + 1]])
        else:
            ans[r] = hist[r, :t]
    for r in range(R):
        for j in range(1, t + 1):
            hist[r if j == t else int(anc[r, j]), j] = ans[r, j - 1]
    min_len = t + 1 if mode == 'eos' else 0

    def args(cp=None):
        a = L.TailConstrArgs()
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
    k2 = 2 * L.MAX_W
    base_ms, base_e = torch.zeros(R, 4, 2, **f32), torch.zeros(R, 4, k2, **f32)
    base_i = torch.zeros(R, 4, k2, dtype=torch.int32, device=dev)
    L.call('case_vocab_base', logits.data_ptr(), ldv, R, V, 1 - finalize, k2, base_ms.data_ptr(), base_e.data_ptr(),
           base_i.data_ptr(), st)
    counter = torch.zeros(1, dtype=torch.int32, device=dev)
    lib.case_debug_sparse_tail_fallbacks.argtypes = [C.c_void_p]
    a2, sparse = args(cp)
    a2.hist_tok, a2.hist_anc, a2.hist_ld, a2.t, a2.eos = hist.data_ptr(), anc.data_ptr(), TL, t, EOS
    a2.no_repeat_ngram, a2.min_len = (0 if mode == 'eos' else 1), min_len
    lib.case_debug_sparse_tail_fallbacks(counter.data_ptr())
    try:
        L.check(lib.case_sparse_tail(C.byref(a2), base_ms.data_ptr(), base_e.data_ptr(), base_i.data_ptr(), k2, None, None,
                                     st), 'case_sparse_tail(constrained)')
    finally:
        lib.case_debug_sparse_tail_fallbacks(None)
    torch.cuda.synchronize()
    # reference: the dense mixture with each row's banned ids at -inf, exact top-k (value desc, index asc)
    d = dense['dist'][:, :V].double().cpu()
    banned = torch.zeros(R, V, dtype=torch.bool)
    for r in range(R):
        if mode != 'eos':
            banned[r, ans[r].long().cpu()] = True
        else:
            banned[r, EOS] = True
    dm = d.masked_fill(banned, float('-inf'))
    want = torch.argsort(torch.argsort(torch.argsort(-dm, dim=1, stable=True), dim=1), dim=1)[:, :K]
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
    if mode == 'eos':
        assert not bool((got_i == EOS).any())
    _record(f'kernel_{mode}_V{V}_K{K}_plan{plan}', dict(fallback_rows=nfb, rows=R))


def test_constrained_sparse_tail_bans_a_dynamic_id():
    """Extended vocabulary (Vext > V, hash mode): the top-8 of the unconstrained tail is the reference - the banned
    dynamic id, the row's best, leaves it and everything else keeps its order."""
    torch.manual_seed(5)
    dev, f32 = 'cuda', dict(dtype=torch.float32, device='cuda')
    R, W, V, NO, S1, K, Tmax, t = 4, 2, 3000, 40, 300, 2, 10, 3
    B, TL, Vx = R // W, Tmax + 1, V + NO
    ldv = -(-Vx // 8) * 8
    logits = torch.randn(R, ldv, **f32)
    attn = torch.randn(R, S1, **f32)
    smap = torch.randint(3, V, (B, S1), device=dev, dtype=torch.int32)
    smap[:, :40] = V + 7                                      # one dynamic id with most of the copy mass
    gates = torch.tensor([[0.3, 0.7, 0.0, 0.0]], **f32).repeat(R, 1)
    fac = torch.zeros(R, L.MAX_SPLIT, **f32)
    fac[:, 0] = 0.7 / attn.exp().sum(1)
    hist = torch.zeros(R, TL, dtype=torch.int32, device=dev)
    anc = torch.arange(R, device=dev, dtype=torch.int32)[:, None].repeat(1, TL)
    hist[:, 1], hist[:, 2], hist[:, 3] = 5, V + 7, 6          # n = 1: the answer holds the dynamic id
    lib = L.load()
    k2 = 16
    base_ms, base_e = torch.zeros(R, 4, 2, **f32), torch.zeros(R, 4, k2, **f32)
    base_i = torch.zeros(R, 4, k2, dtype=torch.int32, device=dev)
    L.call('case_vocab_base', logits.data_ptr(), ldv, R, V, 1, k2, base_ms.data_ptr(), base_e.data_ptr(),
           base_i.data_ptr(), torch.cuda.current_stream().cuda_stream)

    def run(k, constrained):
        a = L.TailConstrArgs()
        a.R, a.V, a.W, a.K, a.ldl, a.ldd, a.mask_col0, a.nmem, a.do_finalize = R, V, W, k, ldv, ldv, 1, 1, 0
        a.fac_ld, a.map_ld, a.Vext = L.MAX_SPLIT, S1, Vx
        a.S[0], a.attn_un[0] = S1, attn.data_ptr()
        tv, ti = torch.zeros(R, k, **f32), torch.zeros(R, k, dtype=torch.int32, device=dev)
        a.logits, a.gates, a.fac, a.map, a.top_vals, a.top_idx = (logits.data_ptr(), gates.data_ptr(), fac.data_ptr(),
                                                                  smap.data_ptr(), tv.data_ptr(), ti.data_ptr())
        if constrained:
            a.hist_tok, a.hist_anc, a.hist_ld, a.t, a.eos, a.no_repeat_ngram = (hist.data_ptr(), anc.data_ptr(), TL, t, EOS,
                                                                                1)
        L.check(lib.case_sparse_tail(C.byref(a), base_ms.data_ptr(), base_e.data_ptr(), base_i.data_ptr(), k2, None, None,
                                     torch.cuda.current_stream().cuda_stream), 'case_sparse_tail')
        torch.cuda.synchronize()
        return tv.cpu(), ti.cpu()

    fv, fi = run(L.MAX_W, False)
    assert bool((fi[:, 0] == V + 7).all()), fi[:, 0]
    cv, ci = run(K, True)
    for r in range(R):
        keep = [j for j in range(L.MAX_W) if int(fi[r, j]) not in (5, V + 7, 6)][:K]
        assert ci[r].tolist() == [int(fi[r, j]) for j in keep]
        assert torch.equal(cv[r], fv[r, keep])


# ------------------------------------------------------------------------------------------------ 2./3. vs the oracle
def _oracle_nbest(stepper, T, W, n, m):
    out, best, results = CT.beam(stepper, T, W, return_all=True, no_repeat_ngram=n, min_len=m)
    return out, [h.cum / h.length for h in best]


CONS = [(3, 0), (2, 3), (1, 0), (0, 4)]


@pytest.mark.parametrize('family', ['case', 'gttp'])
def test_fp32_golden_problems_equal_constrained_oracle(family):
    from case_rg_b200 import generations as FG
    if family == 'case':
        from oracle.case_decoder import CaseOracle
        z, cfg, sd, inp = build_case('case_generations')
        stepper = lambda: CaseOracle(sd).incremental(inp)
        make, data = (lambda g: FG.FastCaSE(sd, device=DEV, dtype='fp32', use_graph=g)), _case_data(inp)
    else:
        from oracle.gttp import GttpOracle
        z, cfg, sd, inp = build_gttp()
        stepper = lambda: GttpOracle(sd).stepper(inp)
        make, data = (lambda g: FG.FastGTTP(sd, device=DEV, dtype='fp32', use_graph=g)), _gttp_data(inp)
    T = int(cfg['T'])
    gaps = {}
    for graph in (False, True):
        model = make(graph)
        for n, m in CONS:
            want = CT.greedy(stepper(), T, no_repeat_ngram=n, min_len=m)
            got = FG.greedy(model, data, None, T, no_repeat_ngram=n, min_len=m).cpu()
            assert torch.equal(got, want), (family, graph, n, m)
            assert not _violations(got.tolist(), n, m, greedy=True)
            for W in (2, 4, 8):
                want_b, keys = _oracle_nbest(stepper(), T, W, n, m)
                nb = FG.beam_nbest(model, data, None, T, W, 1, no_repeat_ngram=n, min_len=m)
                got_b = nb.tokens[:, 0].cpu()
                Lm = max(got_b.size(1), want_b.size(1))
                assert torch.equal(PT._pad(got_b, Lm), PT._pad(want_b, Lm)), (family, graph, n, m, W)
                gap = float((nb.costs[:, 0].cpu() - torch.tensor(keys, dtype=torch.float64)).abs().max())
                assert gap <= 1e-4, gap
                gaps[f'{n}_{m}_beam{W}'] = max(gaps.get(f'{n}_{m}_beam{W}', 0.0), gap)
                assert not _violations(got_b.tolist(), n, m)
    _record(f'golden_{family}_fp32', dict(max_cost_gap_nats=gaps))


def _c2():
    sd, inp = _case_problem(64, 60, 10, 256, 51, 61)
    return sd, inp, _case_data(inp)


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
def test_full_size_search_vs_constrained_oracle(case, dtype):
    """C2 (CaSE, B=64, beam 4, V=30522, T=40) and C4 (GTTP, B=128, beam 4, V=50,000, T=40) with n = 3, min_len = 5:
    fp32 identical to the oracle (costs within 1e-4), bf16 with no miss under the oracle-scored tie criterion; every
    answer satisfies the constraints; off is bit-identical to the plain call."""
    from case_rg_b200 import generations as FG
    W, T, n, m = 4, 40, 3, 5
    sd, inp, data = (_c2 if case == 'c2' else _c4)()
    if case == 'c2':
        from oracle.case_decoder import CaseOracle
        orc = CaseOracle(sd, device=DEV)
        factory = lambda: orc.incremental(inp)
        make = lambda g: FG.FastCaSE(sd, device=DEV, dtype=dtype, use_graph=g)
    else:
        from oracle.gttp import GttpOracle
        orc = GttpOracle(sd, device=DEV)
        factory = lambda: orc.stepper(inp)
        make = lambda g: FG.FastGTTP(sd, device=DEV, dtype=dtype, use_graph=g)
    B = data['source_map' if case == 'c2' else 'background_map'].size(0)
    rec = _Rec(factory())
    want_b, _, results = CT.beam(rec, T, W, return_all=True, no_repeat_ngram=n, min_len=m)
    keys = torch.tensor([results[q][0].cum / results[q][0].length for q in range(B)], dtype=torch.float64)
    want_g = CT.greedy(factory(), T, no_repeat_ngram=n, min_len=m)
    tol = {'fp32': 1e-4, 'bf16': 2e-2}[dtype] * rec.scale          # the logit band of tests/parity_tools.py in nats
    out = {}
    for graph in (False, True):
        model = make(graph)
        plain = FG.beam_nbest(model, data, None, T, W, 1)
        off = FG.beam_nbest(model, data, None, T, W, 1, no_repeat_ngram=0, min_len=0)
        assert all(torch.equal(x, y) for x, y in zip(plain, off)), 'constraints off must be the plain search'
        nb = FG.beam_nbest(model, data, None, T, W, 1, no_repeat_ngram=n, min_len=m)
        got_b = nb.tokens[:, 0].cpu()
        got_g = FG.greedy(model, data, None, T, no_repeat_ngram=n, min_len=m).cpu()
        assert not _violations(got_b.tolist(), n, m), _violations(got_b.tolist(), n, m)[:3]
        assert not _violations(got_g.tolist(), n, m, greedy=True)
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
            g_same = int((got_g == want_g).all(1).sum())
            out[f'graph{int(graph)}'] = dict(beam=res, greedy_identical_rows=g_same, rows=B)
        if case == 'c2' and not graph:
            out['unconstrained_trigram_repeats'] = _repeats(plain.tokens[:, 0].cpu().tolist(), 3)
            out['constrained_trigram_repeats'] = _repeats(got_b.tolist(), 3)
            assert out['unconstrained_trigram_repeats'] >= 1, 'the constraint must bite at C2'
    _record(f'{case}_{dtype}', out)


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_extended_vocabulary(dtype):
    """n_oov problem: the ids compared are the returned (extended) ids; fp32 equals the constrained oracle."""
    from case_rg_b200 import generations as FG
    from oracle.case_decoder import CaseOracle
    V, B, T, W, NO = 3000, 6, 12, 4, 50
    sd = syn.make_case_decoder_state(41, V, H, peaked=0.3, boost={syn.EOS: 6.0}, gen_gate_bias=0.5)
    inp = syn.make_case_inputs(42, B, 24, 4, 40, V, H)
    g = torch.Generator().manual_seed(43)
    oov = torch.rand(inp.source_map.shape, generator=g) < 0.2
    oov &= inp.source_map > 102
    inp.source_map = torch.where(oov, V + torch.randint(0, NO, inp.source_map.shape, generator=g), inp.source_map)
    model = FG.FastCaSE(sd, device=DEV, dtype=dtype, n_oov=NO)
    data = _case_data(inp)
    for n, m in ((1, 0), (2, 3)):
        nb = FG.beam_nbest(model, data, None, T, W, W, no_repeat_ngram=n, min_len=m)
        rows = nb.tokens.reshape(B * W, -1).cpu().tolist()
        assert not _violations(rows, n, m)
        g_tok = FG.greedy(model, data, None, T, no_repeat_ngram=n, min_len=m).cpu()
        assert not _violations(g_tok.tolist(), n, m, greedy=True)
        if dtype == 'fp32':
            want, keys = _oracle_nbest(CaseOracle(sd).incremental(inp, n_oov=NO), T, W, n, m)
            got = nb.tokens[:, 0].cpu()
            Lm = max(got.size(1), want.size(1))
            assert torch.equal(PT._pad(got, Lm), PT._pad(want, Lm)), (n, m)
            assert float((nb.costs[:, 0].cpu() - torch.tensor(keys, dtype=torch.float64)).abs().max()) <= 1e-4
            assert torch.equal(g_tok, CT.greedy(CaseOracle(sd).incremental(inp, n_oov=NO), T, n, m))


# ------------------------------------------------------------------------------------------------ 4. composition, faces
def test_nbest_and_attribution_compose():
    from case_rg_b200 import generations as FG
    T, W, n, m = 12, 4, 2, 3
    model = _small_model(FG)
    inp = _small_case(81, 6)
    data = _case_data(inp)
    att = FG.beam_attributed(model, data, None, T, W, W, no_repeat_ngram=n, min_len=m)
    nb = FG.beam_nbest(model, data, None, T, W, W, no_repeat_ngram=n, min_len=m)
    assert all(torch.equal(x, y) for x, y in zip(att.answer, nb))
    B = nb.tokens.size(0)
    rows = nb.tokens.reshape(B * W, -1).cpu().tolist()
    assert not _violations(rows, n, m), _violations(rows, n, m)[:3]
    lens = nb.lengths.reshape(-1).cpu()
    parts = att.parts.reshape(B * W, -1, 3).cpu().double()
    pos = torch.arange(parts.size(1))[None, :]
    p = parts.sum(-1)
    nll = torch.where(pos < lens[:, None], -torch.log(p + 1e-10), torch.zeros_like(p)).sum(1)
    gap = float((nll / (lens.double() + 1) - nb.costs.reshape(-1).cpu()).abs().max())
    assert gap <= 1e-5, gap
    g = FG.greedy_attributed(model, data, None, T, no_repeat_ngram=n, min_len=m)
    assert torch.equal(g.answer, FG.greedy(model, data, None, T, no_repeat_ngram=n, min_len=m))
    _record('compose', dict(max_cost_gap_nats=gap))


def test_faces_carry_the_constraints():
    from case_rg_b200 import generations as FG
    T, W, n, m = 10, 4, 2, 3
    model = _small_model(FG)
    inps = [_small_case(71, 6), _small_case(72, 6), _small_case(73, 3)]
    host = [{k: getattr(i, k) for k in FG.FastCaSE._KEYS} for i in inps]
    streamed = list(FG.beam_batches(model, iter(host), None, T, W, no_repeat_ngram=n, min_len=m))
    for inp, got in zip(inps, streamed):
        assert torch.equal(got, FG.beam(model, _case_data(inp), None, T, W, no_repeat_ngram=n, min_len=m).cpu())
    streamed = list(FG.beam_batches(model, iter(host), None, T, W, n_best=2, no_repeat_ngram=n, min_len=m))
    for inp, got in zip(inps, streamed):
        want = FG.beam_nbest(model, _case_data(inp), None, T, W, 2, no_repeat_ngram=n, min_len=m)
        assert all(torch.equal(x, y.cpu()) for x, y in zip(got, want))
    gmodel = _small_model(FG)
    streamed = list(FG.greedy_batches(gmodel, iter(host), None, T, no_repeat_ngram=n, min_len=m))
    for inp, got in zip(inps, streamed):
        assert torch.equal(got, FG.greedy(gmodel, _case_data(inp), None, T, no_repeat_ngram=n, min_len=m).cpu())
    cfg, sd_prod, sd_dec, data, _ = producers_case()
    pm = FG.FastCaSE(sd_dec, device=DEV, dtype='bf16', producers=sd_prod)
    d = {k: v.to(DEV) for k, v in data.items()}
    for mode, width in (('beam', 4), ('greedy', 1)):
        out = pm.search_ids(d, cfg['T'], width, mode=mode, no_repeat_ngram=1, min_len=2)
        rows = out['answer'].cpu().tolist()
        assert not _violations(rows, 1, 2, greedy=mode == 'greedy'), rows
    with pytest.raises(ValueError):
        pm.search_ids(d, cfg['T'], 1, mode='module_greedy', no_repeat_ngram=1)


def test_unservable_requests_raise_before_launch():
    from case_rg_b200 import generations as FG
    from case_rg_b200.engine import CaseDecodeEngine, GttpDecodeEngine, check_constraints
    data = _case_data(_small_case(62, 2))
    for opt in (L.OPT_DENSE_TAIL, L.OPT_UNFUSED_TAIL):
        model = _small_model(FG, opt=opt)
        with pytest.raises(ValueError):
            FG.beam(model, data, None, 10, 4, no_repeat_ngram=2)
        with pytest.raises(ValueError):
            FG.greedy(model, data, None, 10, min_len=2)
        with pytest.raises(ValueError):
            FG.beam_batches(model, iter([]), None, 10, 4, no_repeat_ngram=2)
        assert not model._engines
    model = _small_model(FG)
    for n, m in ((-1, 0), (11, 0), (0, 10), (0, -1)):
        with pytest.raises(ValueError):
            FG.beam(model, data, None, 10, 4, no_repeat_ngram=n, min_len=m)
        with pytest.raises(ValueError):
            FG.greedy_batches(model, iter([]), None, 10, no_repeat_ngram=n, min_len=m)
    with pytest.raises(ValueError):
        model.fast_search(data, 10, 1, L.MODE_MODULE_GREEDY, no_repeat_ngram=2)
    assert not model._engines
    with pytest.raises(ValueError):                     # V < 2W + Tmax + 1
        check_constraints(0, 40, 4, 10, 35, 2, 0)
    _, _, sd, _ = build_gttp()
    gw = FG.FastGTTP(sd, device=DEV, dtype='bf16').weights
    with pytest.raises(ValueError):
        GttpDecodeEngine(gw, 2, 4, 10, 16, 10, opt=L.OPT_DENSE_TAIL, min_len=3)
    eng = CaseDecodeEngine(model.weights, 2, 1, 72, 150, 10, no_repeat_ngram=2)
    with pytest.raises(ValueError):
        eng.launch(10, L.MODE_MODULE_GREEDY, use_graph=False)
    with pytest.raises(ValueError):
        eng.step_distribution(0)
