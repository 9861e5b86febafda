#!/usr/bin/env python
"""Cost of the attribution records: the C2 bf16 beam decode (bench.py's seeds and weights: B=64, beam 4, 10 x 256
passages, V=30522, T=40) with attribution off (``beam`` / ``beam_nbest``) and on (``beam_attributed``), with n = 1 and
n = 4, the four arms alternated in one process, CUDA events around
  call    the public function: prefill + 40 decode steps (CUDA graph) + reading the result
  decode  the graph replay of the 40 steps alone
usage: python profiles/micro/attribution_timing.py [reps]"""
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


def _events(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    c = bench.CONFIGS['c2']
    B, W, T, V = c['B'], c['W'], c['T'], c['V']
    sd = syn.make_case_decoder_state(bench.WSEED, V, bench.H)
    inp = syn.make_case_inputs(bench.ISEED, B, c['Lq'], c['NP'], c['Lp'], V, bench.H, id_base=0).to('cuda')
    data = {k: getattr(inp, k) for k in FG.FastCaSE._KEYS}
    model = FG.FastCaSE(sd, device='cuda', dtype='bf16', max_dec_len=T, beam_width=W)
    arms = {('off', 1): lambda: FG.beam(model, data, None, T, W),
            ('on', 1): lambda: FG.beam_attributed(model, data, None, T, W, 1),
            ('off', 4): lambda: FG.beam_nbest(model, data, None, T, W, 4),
            ('on', 4): lambda: FG.beam_attributed(model, data, None, T, W, 4)}
    engines = {}
    for k, fn in arms.items():                                   # warm-up: engines, graphs, allocator
        for _ in range(3):
            fn()
        engines[k] = model.last_engine
    assert len({id(e) for e in engines.values()}) == 4, 'one engine per arm'
    call = {k: [] for k in arms}
    decode = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            call[k].append(_events(fn))
            decode[k].append(_events(lambda: engines[k].launch(T, L.MODE_BEAM)))
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                            str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        q = 'nvidia-smi unavailable'
    print(f'device: {torch.cuda.get_device_name()}  power limit, max SM clock: {q}')
    print(f'C2 bf16: B={B}, beam {W}, T={T}, V={V}; {reps} alternating reps per arm, ms')
    for what, d in (('call', call), ('decode', decode)):
        for k in arms:
            x = d[k]
            print(f'  {what:6s} attribution {k[0]:3s} n={k[1]}: median {statistics.median(x):8.3f}  min {min(x):8.3f}'
                  f'  mean {statistics.mean(x):8.3f}  max {max(x):8.3f}')
        for n in (1, 4):
            m0, m1 = statistics.median(d[('off', n)]), statistics.median(d[('on', n)])
            print(f'  {what:6s} n={n} on / off (medians): {m1 / m0:.4f}  (+{(m1 - m0) / T * 1000:.1f} us per step)')


if __name__ == '__main__':
    main()
