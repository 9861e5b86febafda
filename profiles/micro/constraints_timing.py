#!/usr/bin/env python
"""Cost of the search constraints: the C2 bf16 beam decode (bench.py's seeds and weights: B=64, beam 4, 10 x 256
passages, V=30522, T=40) with the constraints off (``beam``) and on (``beam(..., no_repeat_ngram=3, min_len=5)``), the
two arms alternated in one process, CUDA events around
  call    the public function: prefill + 40 decode steps (CUDA graph) + reading the result
  decode  the graph replay of the 40 steps alone
and the number of constrained rows that took the exact pass over their logits (case_debug_sparse_tail_fallbacks), per
decode, with the answers' repeated trigrams in each arm.
usage: python profiles/micro/constraints_timing.py [reps]"""
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

N, MIN_LEN = 3, 5


def _events(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def _trigram_repeats(tokens):
    out = 0
    for row in tokens.tolist():
        ys = []
        for tk in row:
            if tk == 0:
                break
            ys.append(tk)
            if tk == syn.EOS:
                break
        grams = [tuple(ys[j:j + 3]) for j in range(len(ys) - 2)]
        out += len(grams) != len(set(grams))
    return out


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    c = bench.CONFIGS['c2']
    B, W, T, V = c['B'], c['W'], c['T'], c['V']
    sd = syn.make_case_decoder_state(bench.WSEED, V, bench.H)
    inp = syn.make_case_inputs(bench.ISEED, B, c['Lq'], c['NP'], c['Lp'], V, bench.H, id_base=0).to('cuda')
    data = {k: getattr(inp, k) for k in FG.FastCaSE._KEYS}
    model = FG.FastCaSE(sd, device='cuda', dtype='bf16', max_dec_len=T, beam_width=W)
    lib = L.load()
    lib.case_debug_sparse_tail_fallbacks.argtypes = [C.c_void_p]
    counter = torch.zeros(1, dtype=torch.int32, device='cuda')
    lib.case_debug_sparse_tail_fallbacks(counter.data_ptr())     # read at launch: the graphs captured below keep it
    arms = {'off': lambda: FG.beam(model, data, None, T, W),
            'on': lambda: FG.beam(model, data, None, T, W, no_repeat_ngram=N, min_len=MIN_LEN)}
    engines, answers = {}, {}
    for k, fn in arms.items():                                   # warm-up: engines, graphs, allocator
        for _ in range(3):
            answers[k] = fn().cpu()
        engines[k] = model.last_engine
    assert len({id(e) for e in engines.values()}) == 2, 'one engine per arm'
    torch.cuda.synchronize()
    counter.zero_()
    engines['on'].launch(T, L.MODE_BEAM)
    torch.cuda.synchronize()
    fallbacks = int(counter.item())
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
    print(f'C2 bf16: B={B}, beam {W}, T={T}, V={V}; constraints on = no_repeat_ngram {N}, min_len {MIN_LEN}; '
          f'{reps} alternating reps per arm, ms')
    for what, d in (('call', call), ('decode', decode)):
        for k in arms:
            x = d[k]
            print(f'  {what:6s} constraints {k:3s}: median {statistics.median(x):8.3f}  min {min(x):8.3f}'
                  f'  mean {statistics.mean(x):8.3f}  max {max(x):8.3f}')
        m0, m1 = statistics.median(d['off']), statistics.median(d['on'])
        print(f'  {what:6s} on / off (medians): {m1 / m0:.4f}  ({(m1 - m0) / T * 1000:+.1f} us per step)')
    print(f'exact-pass rows per constrained decode: {fallbacks} of {B * W * T} row-steps')
    print(f'answers repeating a trigram: off {_trigram_repeats(answers["off"])} / {B}, '
          f'on {_trigram_repeats(answers["on"])} / {B}')


if __name__ == '__main__':
    main()
