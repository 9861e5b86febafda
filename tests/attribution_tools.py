"""Oracle attribution records (test infrastructure; drives the steppers of ``oracle``).

Teacher-forces token sequences through the oracle's steppers (CaseOracle.incremental, GttpOracle.stepper) and splits
the probability of every token ``y`` at position ``j`` - taken from the distribution of its prefix at step ``j`` - into
the parts of the reference's mixture, read from the stepper's ``last``:

* CaSE (CaSE/Model.py:38-48, 110-111): ``gates[0] * gen[y]`` (0 for dynamic ids >= V), then per memory i the copy mass
  ``sum over s with source_map[s] == y of copy_w[s]``, ``copy_w = gates[i + 1] * p_i`` (query positions, then passages);
* GTTP (GTTP/Model.py:25-43): ``(1 - p_copy) * gen[y]`` (gen[0] = 0: logit 0 is masked), then
  ``p_copy * sum over s with background_map[s] == y of bg_attn[s]``.

``source`` is the position with the largest single contribution (ties to the lowest position), -1 when none
contributes.  The two largest contributions are returned too, so that a caller can tell an exact source from a tie.
"""
import torch

PAD, BOS, EOS, UNK = 0, 1, 2, 100


def _contributions(stepper, y):
    """-> (generation part [R], copy contributions [R, S] (zero where the map is not y), S0 = positions of memory 0,
    dist[y] [R]) of the stepper's last step, in float64."""
    last = stepper.last
    y = y.to(last['dist'].device)
    ar = torch.arange(y.numel(), device=y.device)
    if 'gates' in last:                                              # CaSE
        gen, g0 = last['gen'].double(), last['gates'][:, 0].double()
        V = gen.size(1)
        gpart = torch.where(y < V, g0 * gen[ar, y.clamp(max=V - 1)], torch.zeros_like(g0))
        smap = stepper.ctx['source_map'][stepper.row2q]
        cw = last['copy_w'].double()
        S0 = last['p'][0].size(1)
    else:                                                            # GTTP
        gen, pc = last['gen'].double(), last['p_copy'][:, 0].double()
        gpart = (1 - pc) * gen[ar, y]
        smap = stepper.inp.background_map[stepper.row2q]
        cw = pc[:, None] * last['bg_attn'].double()
        S0 = cw.size(1)
    contrib = torch.where(smap.to(y.device) == y[:, None], cw, torch.zeros_like(cw))
    return gpart, contrib, S0, last['dist'][ar, y].double()


def teacher_forced_attribution(stepper, tokens, n=1, lengths=None, proto_greedy=False, parts=3, probe=None):
    """Records of ``tokens`` int64 [N, L] (BOS dropped; row i belongs to query i // n; token j is fed at step j + 1).

    Which positions hold a real record: ``lengths`` [N] (beam entries: positions < length), or ``proto_greedy``
    (Generations.py:96-107: PAD after the row's end gets the zero record, and at t = 0 a UNK that replaced the EOS the
    distribution chose gets EOS's record), else every position (module greedy).

    probe (int64 [N, L], may be None): source positions (e.g. the device's) whose oracle contribution to the token is
    returned as ``at_probe`` (0 where the probe is -1).

    -> dict(parts float64 [N, L, parts], source int64 [N, L], top2 float64 [N, L, 2] the two largest single
    contributions, p float64 [N, L] the oracle's dist[y], valid bool [N, L], at_probe float64 [N, L], logit_scale the
    largest finite |logit| of all steps - the scale the relative logit band of tests/parity_tools.py refers to), on the
    CPU."""
    N, L = tokens.shape
    B = N // n
    tokens = tokens.cpu()
    par = torch.repeat_interleave(torch.arange(B), n)
    feed = torch.full((N,), BOS, dtype=torch.long)
    out_parts = torch.zeros(N, L, parts, dtype=torch.float64)
    out_src = torch.full((N, L), -1, dtype=torch.long)
    out_top2 = torch.zeros(N, L, 2, dtype=torch.float64)
    out_p = torch.zeros(N, L, dtype=torch.float64)
    at_probe = torch.zeros(N, L, dtype=torch.float64)
    valid = torch.ones(N, L, dtype=torch.bool)
    if lengths is not None:
        valid = torch.arange(L)[None, :] < lengths.cpu()[:, None]
    ended = torch.zeros(N, dtype=torch.bool)
    scale = 0.0
    for t in range(L):
        dist = stepper.advance(par, feed)
        lg = stepper.last['logits']
        scale = max(scale, float(lg.masked_fill(~torch.isfinite(lg), 0).abs().max()))
        y = tokens[:, t].clone()
        if proto_greedy:
            if t == 0:
                y = torch.where((y == UNK) & (dist.argmax(1).cpu() == EOS), torch.full_like(y, EOS), y)
            else:
                valid[:, t] = ~ended
            ended |= y == EOS
        gpart, contrib, S0, p = _contributions(stepper, y)
        contrib = contrib.cpu()
        out_parts[:, t, 0] = gpart.cpu()
        out_parts[:, t, 1] = contrib[:, :S0].sum(1)
        if parts > 2:
            out_parts[:, t, 2] = contrib[:, S0:].sum(1)
        top = torch.topk(contrib, min(2, contrib.size(1)), dim=1).values
        out_top2[:, t, :top.size(1)] = top
        best = contrib.argmax(1)                                     # first maximal value: the lowest position
        out_src[:, t] = torch.where(top[:, 0] > 0, best, torch.full_like(best, -1))
        out_p[:, t] = p.cpu()
        if probe is not None:
            pr = probe[:, t].cpu()
            at_probe[:, t] = torch.where(pr >= 0, contrib.gather(1, pr.clamp(min=0)[:, None])[:, 0],
                                         torch.zeros_like(at_probe[:, t]))
        par = torch.arange(N)
        feed = tokens[:, t]
    out_parts[~valid] = 0
    out_src[~valid] = -1
    out_top2[~valid] = 0
    return dict(parts=out_parts, source=out_src, top2=out_top2, p=out_p, valid=valid, at_probe=at_probe,
                logit_scale=scale)
