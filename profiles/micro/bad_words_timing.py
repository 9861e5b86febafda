#!/usr/bin/env python
"""Cost of the banned words: the C2 bf16 beam decode (bench.py's seeds and weights: B=64, beam 4, 10 x 256 passages,
V=30522, T=40) in three arms, alternated in one process, CUDA events around
  call    the public function: ban-list write + prefill + 40 decode steps (CUDA graph) + reading the result
  decode  the graph replay of the 40 steps alone
The arms: off (``beam``); constrained (no_repeat_ngram=3, min_len=5); banned (the same plus a realistic list: every
[unusedN] id except BOS / EOS, [UNK], [CLS], [SEP], [MASK] - 996 single ids - and 64 sequences of 2-4 tokens taken from
the off arm's answers).  Also: the rows that took the exact pass over their logits (case_debug_sparse_tail_fallbacks)
per decode, and the answers that contain a banned id or sequence in each arm.
usage: python profiles/micro/bad_words_timing.py [reps]"""
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..')
sys.path.insert(0, ROOT)
import bench                                                      # noqa: E402
from case_rg_b200 import _lib as L, synthetic as syn             # noqa: E402
from case_rg_b200 import generations as FG                       # noqa: E402

N, MIN_LEN, NSEQ = 3, 5, 64
# BERT-uncased: [unused0..98] = 1..99, [UNK] [CLS] [SEP] [MASK] = 100..103, [unused99..993] = 104..998;
# [unused0] / [unused1] are BOS / EOS
SINGLES = [[i] for i in range(3, 999)]


def _events(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def _answers(tokens):
    out = []
    for row in tokens.tolist():
        ys = []
        for tk in row:
            if tk == 0:
                break
            ys.append(tk)
            if tk == syn.EOS:
                break
        out.append(ys)
    return out


def _sequences(answers):
    """NSEQ distinct windows of 2-4 tokens of the answers (EOS excluded), spread over the answers."""
    seqs, k = [], 0
    while len(seqs) < NSEQ and k < 4 * NSEQ:
        ys = [t for t in answers[k % len(answers)] if t != syn.EOS]
        L_ = 2 + k % 3
        j = (k // len(answers)) % max(1, len(ys) - L_ + 1)
        w = ys[j:j + L_]
        if len(w) == L_ and w not in seqs:
            seqs.append(w)
        k += 1
    return seqs


def _with_ban(answers, bans):
    n = 0
    for ys in answers:
        n += any(ys[i:i + len(w)] == w for w in bans for i in range(len(ys) - len(w) + 1))
    return n


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    c = bench.CONFIGS['c2']
    B, W, T, V = c['B'], c['W'], c['T'], c['V']
    sd = syn.make_case_decoder_state(bench.WSEED, V, bench.H)
    inp = syn.make_case_inputs(bench.ISEED, B, c['Lq'], c['NP'], c['Lp'], V, bench.H, id_base=0).to('cuda')
    data = {k: getattr(inp, k) for k in FG.FastCaSE._KEYS}
    model = FG.FastCaSE(sd, device='cuda', dtype='bf16', max_dec_len=T, beam_width=W)
    off_answers = _answers(FG.beam(model, data, None, T, W).cpu())
    bans = SINGLES + _sequences(off_answers)
    lib = L.load()
    lib.case_debug_sparse_tail_fallbacks.argtypes = [C.c_void_p]
    counter = torch.zeros(1, dtype=torch.int32, device='cuda')
    lib.case_debug_sparse_tail_fallbacks(counter.data_ptr())     # read at launch: the graphs captured below keep it
    arms = {'off': lambda: FG.beam(model, data, None, T, W),
            'constrained': lambda: FG.beam(model, data, None, T, W, no_repeat_ngram=N, min_len=MIN_LEN),
            'banned': lambda: FG.beam(model, data, None, T, W, no_repeat_ngram=N, min_len=MIN_LEN, bad_words=bans)}
    engines, answers = {}, {}
    for k, fn in arms.items():                                   # warm-up: engines, graphs, allocator
        for _ in range(3):
            answers[k] = fn().cpu()
        engines[k] = model.last_engine
    assert len({id(e) for e in engines.values()}) == 3, 'one engine per arm'
    fallbacks = {}
    for k in arms:
        torch.cuda.synchronize()
        counter.zero_()
        engines[k].launch(T, L.MODE_BEAM)
        torch.cuda.synchronize()
        fallbacks[k] = int(counter.item())
    call = {k: [] for k in arms}
    decode = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            call[k].append(_events(fn))
            decode[k].append(_events(lambda: engines[k].launch(T, L.MODE_BEAM)))
    lib.case_debug_sparse_tail_fallbacks(None)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                            str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        q = 'nvidia-smi unavailable'
    print(f'device: {torch.cuda.get_device_name()}  power limit, max SM clock: {q}')
    print(f'C2 bf16: B={B}, beam {W}, T={T}, V={V}; constrained = no_repeat_ngram {N}, min_len {MIN_LEN}; banned = '
          f'constrained + {len(SINGLES)} single ids + {len(bans) - len(SINGLES)} sequences of 2-4 tokens; '
          f'{reps} alternating reps per arm, ms')
    for what, d in (('call', call), ('decode', decode)):
        for k in arms:
            x = d[k]
            print(f'  {what:6s} {k:11s}: median {statistics.median(x):8.3f}  min {min(x):8.3f}'
                  f'  mean {statistics.mean(x):8.3f}  max {max(x):8.3f}')
        m0 = statistics.median(d['off'])
        for k in ('constrained', 'banned'):
            m1 = statistics.median(d[k])
            print(f'  {what:6s} {k} / off (medians): {m1 / m0:.4f}  ({(m1 - m0) / T * 1000:+.1f} us per step)')
    for k in arms:
        print(f'exact-pass rows per decode, {k:11s}: {fallbacks[k]} of {B * W * T} row-steps')
    for k in arms:
        print(f'answers containing a banned id or sequence, {k:11s}: {_with_ban(_answers(answers[k]), bans)} / {B}')


if __name__ == '__main__':
    main()
