"""Protocol face: ``greedy`` / ``beam`` with the signatures of common/Generations.py:66,112, and the
models they drive.

The reference drives an ``EncDecModel`` (GTTP/EncDecModel.py:11-42) from Python, one ``.item()``
per hypothesis per step.  Here the whole search runs on the device; the functions below only hand
the model's encoder outputs to an engine and return the same LongTensor the reference returns
(``[B, max_len]`` for greedy; for beam the best hypothesis per query without BOS, EOS kept,
zero-padded to the longest answer - ``merge1D``, common/Utils.py:366-377).

``beam_nbest`` returns more than the reference's single answer: the n best finished hypotheses of every query with
their costs, the sorted ``results[q]`` list that Generations.beam builds and reads element 0 of (Generations.py:183-185).
``beam_attributed`` / ``greedy_attributed`` also report where every answer token came from: the split of its
probability into generation and copy from each memory, and the source position it was most copied from.

Every search face takes two constraints, applied inside the device search (0 = off, the reference's search):
``no_repeat_ngram = n`` - no answer contains the same n-gram twice (a token that would complete an n-gram already in
the answer is not a candidate; n = 1: no token repeats) - and ``min_len = m`` - EOS is not a candidate before step m,
so every answer has at least m tokens before its EOS.  Banned ids leave the candidate set and nothing is renormalised:
a chosen token still costs -log(p + 1e-10) under the model's mixture, so costs stay comparable with unconstrained
searches.  The ids compared are the returned ones (extended-vocabulary ids; greedy: the emitted token).

Every search face also takes ``bad_words``: a list of token-id sequences (lists of ints or 1-D integer tensors) that no
answer may contain.  A single id is never a candidate; a sequence (w_1 .. w_L) bans w_L wherever the answer so far ends
with w_1 .. w_{L-1}, so no answer and no n-best entry contains it contiguously.  The same rule as the constraints:
nothing is renormalised, costs stay those of the model's mixture.  Unlike GTTP's fixed mask of id 0 (removed from the
softmax itself), a banned id keeps its share of the distribution.  In ``greedy`` an EOS chosen at t = 0 is still
rewritten to UNK (Generations.py:99-100), even when UNK is banned; ``min_len >= 1`` prevents that.  None or empty (the
default) is the unbanned search.  Ids must lie in [0, V); at most 256 sequences of two or more ids, each at most 16
long (_lib.MAX_BAN_SEQ / MAX_BAN_LEN), and V - (single ids) >= 2 * width + max_len + 1 + (sequences).

``FastCaSE`` gives the unchanged CaSE decoder the protocol the reference never implemented for it
(SURVEY.md §8c adapter); ``FastGTTP`` replaces ``GTTP.decode/generate/to_word`` + the search
(GTTP/Model.py:176-193).  Both take the *encoder-side outputs* as inputs: the encoders are outside
the hot path and stay on the reference's own code.
"""
from typing import Dict, Optional

import torch

from . import _lib as L
from .engine import (Attributed, CaseDecodeEngine, CaseWeights, GttpDecodeEngine, GttpWeights, NBest, attributed_from,
                     check_bad_words, check_constraints, nbest_from)

PAD_WORD, BOS_WORD, UNK_WORD, EOS_WORD = '[PAD]', '[unused0]', '[UNK]', '[unused1]'


def _check_vocab(vocab2id):
    if vocab2id is None:
        return
    want = {PAD_WORD: 0, BOS_WORD: 1, EOS_WORD: 2, UNK_WORD: 100}
    for w, i in want.items():
        if vocab2id.get(w, i) != i:
            raise ValueError(f'special token {w} must have id {i} (BERT-uncased ids, common/Constants.py:1-7)')


def greedy(model, data, vocab2id=None, max_len=20, encode_outputs=None, init_decoder_states=None, no_repeat_ngram=0,
           min_len=0, bad_words=None):
    """Generations.greedy (Generations.py:66-110) on the device; no_repeat_ngram / min_len / bad_words: see the module
    docstring."""
    _check_vocab(vocab2id)
    return model.fast_search(data, max_len, 1, L.MODE_PROTO_GREEDY, encode_outputs, init_decoder_states,
                             no_repeat_ngram=no_repeat_ngram, min_len=min_len, bad_words=bad_words)


def beam(model, data, vocab2id=None, max_len=20, width=5, encode_outputs=None, init_decoder_states=None,
         no_repeat_ngram=0, min_len=0, bad_words=None):
    """Generations.beam (Generations.py:112-190) on the device; no_repeat_ngram / min_len / bad_words: see the module
    docstring."""
    _check_vocab(vocab2id)
    return model.fast_search(data, max_len, width, L.MODE_BEAM, encode_outputs, init_decoder_states,
                             no_repeat_ngram=no_repeat_ngram, min_len=min_len, bad_words=bad_words)


def _nbest_count(n, width):
    n = width if n is None else int(n)
    if not 1 <= n <= width:
        raise ValueError(f'n must be 1..width ({width}), got {n}')
    return n


def beam_nbest(model, data, vocab2id=None, max_len=20, width=5, n=None, encode_outputs=None, init_decoder_states=None,
               no_repeat_ngram=0, min_len=0, bad_words=None):
    """The n best answers of ``beam`` per query with their costs: ``NBest(tokens, lengths, costs)`` on the model's
    device, entry [:, i] the i-th of sorted(results[q], key=cum_cost/length)[:n] (Generations.py:183-185).  tokens int64
    [B, n, L] (BOS dropped, EOS kept, zero padded to the longest entry), lengths int64 [B, n], costs fp64 [B, n] = the
    ranking key cum_cost / length in nats per position (lower is better).  Entry 0 is what ``beam`` returns.  n defaults
    to the width; 1 <= n <= width.  With no_repeat_ngram / min_len / bad_words every entry satisfies the constraints and
    contains no banned word."""
    _check_vocab(vocab2id)
    n = _nbest_count(n, width)
    return model.fast_search(data, max_len, width, L.MODE_BEAM, encode_outputs, init_decoder_states, nbest=n,
                             no_repeat_ngram=no_repeat_ngram, min_len=min_len, bad_words=bad_words)


def beam_attributed(model, data, vocab2id=None, max_len=20, width=5, n=None, encode_outputs=None,
                    init_decoder_states=None, no_repeat_ngram=0, min_len=0, bad_words=None):
    """``beam_nbest`` with the attribution record of every answer token: ``Attributed(answer, parts, source)`` on the
    model's device, ``answer`` the NBest of ``beam_nbest`` (the same search, bit for bit), ``parts`` fp32 [B, n, L, P] and
    ``source`` int64 [B, n, L], trimmed like the tokens (see engine.Attributed).  n defaults to the width."""
    _check_vocab(vocab2id)
    n = _nbest_count(n, width)
    return model.fast_search(data, max_len, width, L.MODE_BEAM, encode_outputs, init_decoder_states, nbest=n,
                             attribution=True, no_repeat_ngram=no_repeat_ngram, min_len=min_len, bad_words=bad_words)


def greedy_attributed(model, data, vocab2id=None, max_len=20, encode_outputs=None, init_decoder_states=None,
                      no_repeat_ngram=0, min_len=0, bad_words=None):
    """``greedy`` with the attribution record of every answer token: ``Attributed(answer, parts, source)``, ``answer`` the
    LongTensor [B, max_len] of ``greedy``, ``parts`` fp32 [B, max_len, P], ``source`` int64 [B, max_len].  At t = 0 an
    EOS rewritten to UNK keeps the record of the EOS the distribution chose; PAD positions after the end have zero parts
    and source -1."""
    _check_vocab(vocab2id)
    return model.fast_search(data, max_len, 1, L.MODE_PROTO_GREEDY, encode_outputs, init_decoder_states,
                             attribution=True, no_repeat_ngram=no_repeat_ngram, min_len=min_len, bad_words=bad_words)


def beam_batches(model, batches, vocab2id=None, max_len=20, width=5, n_best=None, attribution=False, no_repeat_ngram=0,
                 min_len=0, bad_words=None):
    """``beam`` over an iterable of HOST batches, the way the predict loop feeds a model one batch after
    another (common/CumulativeTrainer.py:141-156): yields the answers of every batch, in order, as host
    LongTensors.  The host-to-device copy of batch i+1 runs on a copy stream while batch i is decoding
    (double-buffered staging, pinned host tensors copy asynchronously), so the PCIe time of the encoder
    outputs (175 MB per batch at the BASELINE shape) is hidden behind the decode.  n_best: yields the ``beam_nbest``
    lists of every batch instead (NBest of host tensors).  attribution: yields what ``beam_attributed(..., n=n_best)``
    returns for every batch (host Attributed; n_best None = the width).  no_repeat_ngram / min_len / bad_words: the
    constraints and bans of ``beam`` (checked here, before the first batch is read; the ban list is written to the
    engine once, before the first prefill)."""
    _check_vocab(vocab2id)
    if n_best is not None or attribution:
        n_best = _nbest_count(n_best, width)
    bw = model._check_constraints(max_len, width, L.MODE_BEAM, no_repeat_ngram, min_len, bad_words)
    return model.search_batches(batches, max_len, width, L.MODE_BEAM, n_best, attribution, no_repeat_ngram, min_len, bw)


def greedy_batches(model, batches, vocab2id=None, max_len=20, attribution=False, no_repeat_ngram=0, min_len=0,
                   bad_words=None):
    """``greedy`` over an iterable of host batches with the copy of the next batch overlapped (see beam_batches).
    attribution: yields what ``greedy_attributed`` returns for every batch (host Attributed).  no_repeat_ngram /
    min_len / bad_words: the constraints and bans of ``greedy``."""
    _check_vocab(vocab2id)
    bw = model._check_constraints(max_len, 1, L.MODE_PROTO_GREEDY, no_repeat_ngram, min_len, bad_words)
    return model.search_batches(batches, max_len, 1, L.MODE_PROTO_GREEDY, None, attribution, no_repeat_ngram, min_len,
                                bw)


def _to_host(att: Attributed) -> Attributed:
    ans = NBest(*(x.cpu() for x in att.answer)) if isinstance(att.answer, NBest) else att.answer.cpu()
    return Attributed(ans, att.parts.cpu(), att.source.cpu())


class _FastModel:
    beam_width = 1
    max_dec_len = 40

    def greedy(self, data):                       # EncDecModel.greedy / .beam (EncDecModel.py:38-42)
        return greedy(self, data, None, self.max_dec_len)

    def beam(self, data):
        return beam(self, data, None, self.max_dec_len, self.beam_width)

    def forward(self, data, method='test'):       # GTTP.forward test branch (GTTP/Model.py:204-212)
        if method != 'test':
            raise NotImplementedError('only the test-mode decode path is implemented on the device')
        return {'answer': self.greedy(data) if self.beam_width == 1 else self.beam(data)}

    __call__ = forward

    id2vocab = None

    def to_sentence(self, data, batch_indices):    # CaSE.to_sentence (CaSE/Model.py:270-271); needs self.id2vocab
        from .results import to_sentence
        if self.id2vocab is None:
            raise ValueError('set model.id2vocab before calling to_sentence')
        return to_sentence(batch_indices, self.id2vocab)

    # ---- streamed batches (beam_batches / greedy_batches)
    def search_batches(self, batches, max_len, width, mode, n_best=None, attribution=False, no_repeat_ngram=0,
                       min_len=0, bad_words=None):
        """Generator behind beam_batches / greedy_batches (n_best: beam mode, yields NBest per batch; attribution: yields
        Attributed per batch; no_repeat_ngram / min_len / bad_words: the search constraints and bans)."""
        dev = self.weights.device
        if attribution:
            self._check_attribution_opt()
        bw = self._check_constraints(max_len, width, mode, no_repeat_ngram, min_len, bad_words)
        main = torch.cuda.current_stream(dev)
        # the copy stream and the two staging sets live as long as the model: allocating 2 x 175 MB on a
        # fresh stream per call costs tens of milliseconds of cudaMalloc
        if getattr(self, '_copy_stream', None) is None:
            self._copy_stream, self._staging = torch.cuda.Stream(dev), [None, None]
        copy, staging = self._copy_stream, self._staging
        copy.wait_stream(main)              # earlier readers of the staging sets (previous call) are done
        prefilled = [None, None]            # event: the prefill that last read staging set k has finished

        def stage(k, host):
            shapes = {n: (tuple(host[n].shape), host[n].dtype) for n in self._KEYS}
            with torch.cuda.stream(copy):
                if staging[k] is None or staging[k][0] != shapes:
                    # allocated ON the copy stream: a block the allocator recycles from the main stream's pool
                    # (e.g. a prefill temporary that was freed on the host but is still being read on the
                    # device) must never be handed to a buffer the copy stream writes
                    staging[k] = (shapes, {n: torch.empty(host[n].shape, dtype=host[n].dtype, device=dev)
                                           for n in self._KEYS})
                if prefilled[k] is not None:
                    copy.wait_event(prefilled[k])
                for n in self._KEYS:
                    staging[k][1][n].copy_(host[n], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
            return ev

        it = iter(batches)
        nxt = next(it, None)
        k = 0
        ready = stage(0, nxt) if nxt is not None else None
        pending = None                      # engine whose decode is in flight
        while nxt is not None:
            d = staging[k][1]
            # stream order: decode(i-1) -> prefill(i); the host enqueues prefill(i) while decode(i-1) runs.
            # (prefill never touches the search state the pending answers are read from; an engine that is still
            # decoding is never prefilled: engine_for returns the SAME engine for equal shapes, and its decode is
            # ahead of this prefill on the main stream)
            main.wait_event(ready)
            eng = self._prefill_staged(d, width, max_len, n_best or 1, attribution, no_repeat_ngram, min_len, bw)
            prefilled[k] = torch.cuda.Event()
            prefilled[k].record(main)
            nxt = next(it, None)
            if nxt is not None:             # the next batch starts crossing PCIe before this one decodes
                ready = stage(k ^ 1, nxt)
            if mode != L.MODE_BEAM and eng.W != 1:
                raise ValueError('greedy modes need an engine built with W == 1')
            if pending is not None:
                # answers of the previous batch: snapshot them on the device (stream-ordered after its decode), put
                # THIS batch's decode behind the snapshot right away, and only then wait for the snapshot on a side
                # stream - the device never idles while the host reads answers
                st = pending.state
                snap = (st.out_tokens[..., :max_len].clone(), st.best_len.clone()) + \
                    ((st.best_key.clone(),) if n_best or attribution else ()) + \
                    ((st.out_attr[..., :max_len, :].clone(),) if attribution else ())
                ev = torch.cuda.Event()
                ev.record(main)
                eng.launch(max_len, mode, use_graph=self.use_graph)
                yield self._read_snapshot(snap, ev, mode, (pending.nparts, max_len, n_best) if attribution else None)
            else:
                eng.launch(max_len, mode, use_graph=self.use_graph)
            self.last_engine = pending = eng
            k ^= 1
        if pending is not None:
            if attribution:
                yield _to_host(pending._finish_attribution(max_len, mode, mode == L.MODE_BEAM))
            elif n_best:
                yield NBest(*(x.cpu() for x in pending._finish_nbest()))
            else:
                yield pending._finish_tokens(max_len, mode).cpu()

    def _read_snapshot(self, snap, ev, mode, attr=None):
        """Device snapshot (tokens [B, T] int32, best_len [B], or with best_key [B, n] the n-best buffers, with out_attr
        the attribution records too) -> host int64 tokens trimmed like _finish_tokens, the host NBest, or with attr =
        (parts, max_len, n_best) the host Attributed."""
        dev = self.weights.device
        if getattr(self, '_d2h_stream', None) is None:
            self._d2h_stream = torch.cuda.Stream(dev)
        d2h = self._d2h_stream
        d2h.wait_event(ev)
        with torch.cuda.stream(d2h):
            host = [x.to('cpu', non_blocking=True) for x in snap]
        d2h.synchronize()
        if attr is not None:
            P, max_len, n_best = attr
            return attributed_from(*host, P, mode, max_len, mode == L.MODE_BEAM)
        if len(host) == 3:
            return nbest_from(*host)
        toks, blen = host
        out = toks.to(torch.int64)
        if mode == L.MODE_BEAM:             # merge1D (Utils.py:366-377): pad to the longest answer of the batch
            out = out[:, :max(int(blen.max()), 1)]
        return out

    def _check_attribution_opt(self):
        """Attribution needs the sparse tail: refuse the option bits that switch it off before anything is built."""
        if self.opt & (L.OPT_DENSE_TAIL | L.OPT_UNFUSED_TAIL):
            raise ValueError('attribution needs the sparse tail: not with OPT_DENSE_TAIL / OPT_UNFUSED_TAIL')

    def _check_constraints(self, max_len, width, mode, no_repeat_ngram, min_len, bad_words=None):
        """no_repeat_ngram / min_len / bad_words: ValueError for a request the device search cannot serve, before anything
        is built (the engines of a search are sized Tmax = max_len; the source count is checked when the engine is
        built).  -> the checked ban list (engine.BadWords), None when there is none."""
        check_constraints(self.opt, self.weights.V, width, 0, max_len, no_repeat_ngram, min_len, max_len, mode)
        return check_bad_words(self.opt, self.weights.V, width, 0, max_len, bad_words, mode)

    def _finish(self, eng, max_len, mode, nbest, attribution):
        """Answers of the decode just launched on ``eng``: tokens, the NBest list (nbest), or Attributed (attribution)."""
        if attribution:
            return eng._finish_attribution(max_len, mode, nbest is not None)
        if nbest is None:
            return eng._finish_tokens(max_len, mode)
        return eng._finish_nbest()


class FastCaSE(_FastModel):
    """EncDecModel-protocol driver for the CaSE decoder.

    ``data`` carries what ``ResponseGeneration.action`` hands the decoder (CaSE/Model.py:247-251):
    'mem_q' [B,1,Lq,H], 'mem_p' [B,NP,Lp,H], 'query' / 'passage' ids (masks = ids != 0),
    'prior_q', 'prior_p', 'answer_rep' [B,H], 'source_map' int64 [B,S]."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device=None, dtype='bf16', max_dec_len=40,
                 beam_width=1, vocab_impl: Optional[int] = None, use_graph=True, prefix='', opt: int = 0,
                 n_oov: int = 0, producers: Optional[Dict[str, torch.Tensor]] = None):
        """opt: CASE_OPT_* bits for every engine of this model (0 = the default fast path; A/B and fallback tests).
        n_oov: size of the per-query dynamic vocabulary behind the V fixed ids (``source_map`` may point into
        [V, V + n_oov); returned ids then range over the extended vocabulary)."""
        self.weights = CaseWeights(state_dict, device=device, dtype=dtype, prefix=prefix)
        self.max_dec_len, self.beam_width, self.vocab_impl, self.use_graph = max_dec_len, beam_width, vocab_impl, use_graph
        self.opt, self.n_oov = int(opt), int(n_oov)
        self._engines = {}
        # producers: state_dict of the pre-decode modules (reference key names 'query_encoder.*', 'passage_selection.*',
        # 'span_extraction.*') -> search_ids decodes from token ids, the encoder outputs never leave the device
        self.producers = None
        if producers is not None:
            from .producers import CaseProducers
            self.producers = CaseProducers(producers, device=self.weights.device)

    def search_ids(self, data, max_len=None, width=None, mode='beam', n_best=None, attribution=False, no_repeat_ngram=0,
                   min_len=0, bad_words=None):
        """CaSE.do_test from token ids (CaSE/Model.py:313-331): ``data`` = {'query' int [B,1,Lq], 'passage' int [B,NP,Lp],
        'source_map' int [B,S]} -> {'answer': LongTensor, 'rank': [B,NP]} like the reference's forward(data, 'test').
        n_best (beam mode): also 'nbest', the ``beam_nbest`` list of the same search (its entry 0 is 'answer').
        attribution (every mode): also 'attribution', the Attributed of the same search - its answer is the NBest with
        n_best, else 'answer'.  no_repeat_ngram / min_len / bad_words (beam and greedy modes): the search constraints and
        bans of ``beam``."""
        if self.producers is None:
            raise RuntimeError('FastCaSE was built without producers=...')
        max_len = self.max_dec_len if max_len is None else max_len
        width = self.beam_width if width is None else width
        if n_best is not None:
            if mode != 'beam':
                raise ValueError('n_best needs mode="beam"')
            n_best = _nbest_count(n_best, width)
        if attribution:
            self._check_attribution_opt()
        m = {'beam': L.MODE_BEAM, 'greedy': L.MODE_PROTO_GREEDY, 'module_greedy': L.MODE_MODULE_GREEDY}[mode]
        bw = self._check_constraints(max_len, width, m, no_repeat_ngram, min_len, bad_words)
        p = self.producers(data['query'], data['passage'])
        d = dict(mem_q=p['mem_q'], mem_p=p['mem_p'], query=data['query'].to(self.weights.device),
                 passage=data['passage'].to(self.weights.device), prior_q=p['prior_q'], prior_p=p['prior_p'],
                 answer_rep=p['answer_rep'], source_map=data['source_map'].to(self.weights.device))
        cons = dict(no_repeat_ngram=no_repeat_ngram, min_len=min_len, bad_words=bw)
        if n_best is None and not attribution:
            return {'answer': self.fast_search(d, max_len, width, m, **cons), 'rank': p['rank']}
        got = self.fast_search(d, max_len, width, m, nbest=n_best, attribution=attribution, **cons)
        out = {'answer': self.last_engine._finish_tokens(max_len, m), 'rank': p['rank']}
        if n_best is not None:
            out['nbest'] = got.answer if attribution else got
        if attribution:
            out['attribution'] = got
        return out

    def engine_for(self, B, W, S0, S1, T, nbest=1, attribution=False, no_repeat_ngram=0, min_len=0, bans=False):
        # the constraints are captured in the engine's CUDA graphs: part of the key.  The ban list is not (an engine built
        # with bans reads it from its buffers at every launch), only whether there is one
        key = (B, W, S0, S1, T, self.opt, self.n_oov, nbest, bool(attribution), int(no_repeat_ngram), int(min_len)) + \
            ((True,) if bans else ())
        if key not in self._engines:
            if len(self._engines) >= 4:
                self._engines.clear()
            self._engines[key] = CaseDecodeEngine(self.weights, B, W, S0, S1, T, vocab_impl=self.vocab_impl,
                                                  opt=self.opt, n_oov=self.n_oov, nbest=nbest, attribution=attribution,
                                                  no_repeat_ngram=no_repeat_ngram, min_len=min_len, bans=bans)
        return self._engines[key]

    def encode(self, data):
        return data

    def fast_search(self, data, max_len, width, mode, encode_outputs=None, init_decoder_states=None, nbest=None,
                    attribution=False, no_repeat_ngram=0, min_len=0, bad_words=None):
        """-> the answers (LongTensor), with nbest the NBest list of a beam search, with attribution an Attributed."""
        if attribution:
            self._check_attribution_opt()
        bw = self._check_constraints(max_len, width, mode, no_repeat_ngram, min_len, bad_words)
        d = encode_outputs if encode_outputs is not None else data
        eng = self._prefill_staged(d, width, max_len, nbest or 1, attribution, no_repeat_ngram, min_len, bw)
        self.last_engine = eng
        if nbest is None and not attribution:
            return eng.decode(max_len, mode, use_graph=self.use_graph)
        if mode != L.MODE_BEAM and eng.W != 1:
            raise ValueError('greedy modes need an engine built with W == 1')
        eng.launch(max_len, mode, use_graph=self.use_graph)
        return self._finish(eng, max_len, mode, nbest, attribution)

    _KEYS = ('mem_q', 'mem_p', 'query', 'passage', 'prior_q', 'prior_p', 'answer_rep', 'source_map')

    def _prefill_staged(self, d, width, max_len, nbest=1, attribution=False, no_repeat_ngram=0, min_len=0,
                        bad_words=None):
        """Engine of the batch d, prefilled; bad_words (a checked BadWords or None) is written to its ban buffers first."""
        B = d['source_map'].size(0)
        S0 = d['mem_q'].reshape(B, -1, L.H).size(1)
        S1 = d['mem_p'].reshape(B, -1, L.H).size(1)
        eng = self.engine_for(B, width, S0, S1, max_len, nbest, attribution, no_repeat_ngram, min_len,
                              bad_words is not None)
        eng.set_bad_words(bad_words)
        eng.prefill(d['mem_q'], d['mem_p'], d['query'].ne(0), d['passage'].ne(0), d['prior_q'], d['prior_p'],
                    d['answer_rep'], d['source_map'])
        return eng

    def module_greedy(self, data, max_len):
        """The in-module loop of CaSETransformerSeqDecoder.forward (no EOS handling, Model.py:91-123)."""
        return self.fast_search(data, max_len, 1, L.MODE_MODULE_GREEDY)


class FastGTTP(_FastModel):
    """Step side of GTTP on the device.  ``data``: 'context' [B,Lc], 'background' [B,Lb],
    'background_map' int64 [B,Lb] (index form, never one-hot), and the encoder outputs
    'src_output' [B,Lc,2H], 'bg_output' [B,Lb,2H], 'init_state' [B,1,H] (GTTP/Model.py:156-174)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device=None, dtype='bf16', max_dec_len=40,
                 beam_width=1, vocab_impl: Optional[int] = None, use_graph=True, prefix='', opt: int = 0):
        self.weights = GttpWeights(state_dict, device=device, dtype=dtype, prefix=prefix)
        self.max_dec_len, self.beam_width, self.vocab_impl, self.use_graph = max_dec_len, beam_width, vocab_impl, use_graph
        self.opt = int(opt)
        self._engines = {}

    def engine_for(self, B, W, Lc, Lb, T, nbest=1, attribution=False, no_repeat_ngram=0, min_len=0, bans=False):
        key = (B, W, Lc, Lb, T, nbest, bool(attribution), int(no_repeat_ngram), int(min_len)) + ((True,) if bans else ())
        if key not in self._engines:
            if len(self._engines) >= 4:
                self._engines.clear()
            self._engines[key] = GttpDecodeEngine(self.weights, B, W, Lc, Lb, T, vocab_impl=self.vocab_impl,
                                                  opt=self.opt, nbest=nbest, attribution=attribution,
                                                  no_repeat_ngram=no_repeat_ngram, min_len=min_len, bans=bans)
        return self._engines[key]

    def fast_search(self, data, max_len, width, mode, encode_outputs=None, init_decoder_states=None, nbest=None,
                    attribution=False, no_repeat_ngram=0, min_len=0, bad_words=None):
        """-> the answers (LongTensor), with nbest the NBest list of a beam search, with attribution an Attributed."""
        if attribution:
            self._check_attribution_opt()
        bw = self._check_constraints(max_len, width, mode, no_repeat_ngram, min_len, bad_words)
        d = dict(data)
        if encode_outputs is not None:
            d.update(encode_outputs)
        if init_decoder_states is not None:
            d['init_state'] = init_decoder_states
        eng = self._prefill_staged(d, width, max_len, nbest or 1, attribution, no_repeat_ngram, min_len, bw)
        self.last_engine = eng
        if nbest is None and not attribution:
            return eng.decode(max_len, mode, use_graph=self.use_graph)
        eng.launch(max_len, mode, use_graph=self.use_graph)
        return self._finish(eng, max_len, mode, nbest, attribution)

    _KEYS = ('context', 'background', 'background_map', 'src_output', 'bg_output', 'init_state')

    def _prefill_staged(self, d, width, max_len, nbest=1, attribution=False, no_repeat_ngram=0, min_len=0,
                        bad_words=None):
        B, Lc = d['context'].shape
        Lb = d['background'].size(1)
        eng = self.engine_for(B, width, Lc, Lb, max_len, nbest, attribution, no_repeat_ngram, min_len,
                              bad_words is not None)
        eng.set_bad_words(bad_words)
        eng.prefill(d['src_output'], d['bg_output'], d['context'], d['background'], d['background_map'],
                    d['init_state'])
        return eng
