"""Banned-word restatement of the oracle's searches (test infrastructure; imports ``oracle``).

``greedy`` / ``beam`` are the constrained searches of tests/constraint_tools.py (no_repeat_ngram / min_len) with the
banned words of the device (bad_words, INTEGRATION.md §3) added to each fringe row's banned ids: the row's distribution
is masked to -inf at every id ``banned_ids`` returns before the top-k, and the costs use the UNMASKED probabilities of
the chosen ids, so they stay the costs of the unbanned mixture.  Without bad_words the calls are those of
constraint_tools (and with both constraints 0, the oracle's own searches).
"""
import math
from typing import List

import torch

import constraint_tools as CT
from oracle import generations as OG
from oracle.generations import BOS, EOS, PAD, UNK, topk


def banned_ids(answer, t: int, no_repeat_ngram: int = 0, min_len: int = 0, eos: int = EOS,
               bad_words=None) -> List[int]:
    """Ids a hypothesis with answer tokens ``answer`` (y_1 .. y_t, BOS excluded) may not choose at step t: those of
    constraint_tools.banned_ids, and for every banned sequence (w_1 .. w_L) of bad_words its w_L when L == 1 or when the
    answer ends with w_1 .. w_{L-1}."""
    ys = list(answer)
    out = set(CT.banned_ids(ys, t, no_repeat_ngram, min_len, eos))
    for w in bad_words or ():
        w = [int(v) for v in w]
        if len(w) == 1 or (t >= len(w) - 1 and ys[len(ys) - len(w) + 1:] == w[:-1]):
            out.add(w[-1])
    return sorted(out)


def _masked(dist, answers, t, no_repeat_ngram, min_len, bad_words):
    """A copy of dist with every row's banned ids at -inf: the candidates of a banned search."""
    dist = dist.clone()
    for i, ys in enumerate(answers):
        ban = banned_ids(ys, t, no_repeat_ngram, min_len, bad_words=bad_words)
        if ban:
            dist[i, torch.tensor(ban, device=dist.device)] = -math.inf
    return dist


def greedy(stepper, max_len: int, no_repeat_ngram: int = 0, min_len: int = 0, bad_words=None) -> torch.Tensor:
    """oracle.generations.greedy whose step top-1 is taken over the ids ``banned_ids`` allows for the tokens emitted so
    far (an EOS rewritten to UNK at t = 0 counts as UNK, PAD after the end as PAD)."""
    if not bad_words:
        return CT.greedy(stepper, max_len, no_repeat_ngram, min_len)
    B = stepper.B
    parents = torch.arange(B)
    inp = torch.full((B,), BOS, dtype=torch.long)
    ended = torch.zeros(B, dtype=torch.bool)
    out = []
    for t in range(max_len):
        dist = stepper.advance(parents, inp)
        emitted = torch.cat(out, dim=1).tolist() if out else [[] for _ in range(B)]
        _, ids = topk(_masked(dist, emitted, t, no_repeat_ngram, min_len, bad_words), 1)
        tok = ids[:, 0].clone().cpu()
        this_end = tok == EOS
        if t == 0:
            tok[this_end] = UNK
        else:
            tok[ended] = PAD
        out.append(tok.unsqueeze(1))
        ended = ended | this_end
        inp = tok
    return torch.cat(out, dim=1)


def beam(stepper, max_len: int, width: int, return_all: bool = False, no_repeat_ngram: int = 0, min_len: int = 0,
         bad_words=None):
    """oracle.generations.beam (same fringe, ranking, finishing and tie rules) whose per-row top-k is taken over the ids
    ``banned_ids`` allows for the row's answer so far; costs -log(p + 1e-10) with p the unmasked probability."""
    if not bad_words:
        return CT.beam(stepper, max_len, width, return_all, no_repeat_ngram, min_len)
    B = stepper.B
    nxt = [OG._Hyp([BOS], 0.0, 1, q, q) for q in range(B)]
    results = {q: [] for q in range(B)}
    for l in range(max_len + 1):
        fringe = []
        for h in nxt:
            if h.tokens[-1] == EOS or l == max_len:
                results[h.q].append(h)
            else:
                fringe.append(h)
        if not fringe:
            break
        parents = torch.tensor([h.row for h in fringe], dtype=torch.long)
        toks = torch.tensor([h.tokens[-1] for h in fringe], dtype=torch.long)
        dist = stepper.advance(parents, toks)
        _, ids = topk(_masked(dist, [h.tokens[1:] for h in fringe], l, no_repeat_ngram, min_len, bad_words), width)
        probs = torch.gather(dist, 1, ids)                    # costs under the unbanned mixture
        probs, ids = probs.cpu(), ids.cpu()
        children = {q: [] for q in range(B)}
        for i, h in enumerate(fringe):
            for j in range(width):
                cost = -math.log(probs[i, j].item() + 1e-10)
                children[h.q].append(OG._Hyp(h.tokens + [ids[i, j].item()], h.cum + cost, h.length + 1, h.q, i))
        nxt = []
        for q in range(B):
            nxt += sorted(children[q], key=lambda n: n.cum / n.length)[:width]
    best = []
    for q in range(B):
        results[q].sort(key=lambda n: n.cum / n.length)
        best.append(results[q][0])
    L = max(len(h.tokens) - 1 for h in best)
    out = torch.zeros(B, L, dtype=torch.long)
    for q, h in enumerate(best):
        out[q, :len(h.tokens) - 1] = torch.tensor(h.tokens[1:], dtype=torch.long)
    if return_all:
        return out, best, results
    return out
