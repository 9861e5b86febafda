"""Output side of test mode (SURVEY.md §8f N3): decoded token ids -> words -> de-duplicated, detokenised
answers -> the ``.answer`` / ``.run`` files that ``Run_Evaluation.py`` reads.

Reference behaviour restated here (same names, arguments and file formats):
  * ``to_sentence``       common/Utils.py:193-210  (CaSE.to_sentence, CaSE/Model.py:270-271)
  * ``remove_duplicate``  common/Utils.py:170-191
  * ``bert_detokenizer``  common/Utils.py:38-41
  * ``save_result``       Utils.py:5-49 (called from CaSE/Run.py:58-62)

What is different is the cost: the reference pulls every token id to the host on its own
(``index.item()``, one device synchronisation per token: 2,560 per batch at B=64, T=40) and re-scans the
sentence prefix for every candidate cut of ``remove_duplicate`` (cubic in the sentence length); here a batch
is one device->host copy and every cut test is a suffix maximum over first-occurrence positions (linear).
"""
import codecs
import os
from typing import Callable, Dict, List, Sequence

import torch

PAD_WORD, BOS_WORD, UNK_WORD, EOS_WORD = '[PAD]', '[unused0]', '[UNK]', '[unused1]'   # common/Constants.py:1-4


def to_sentence(batch_indices, id2vocab: Dict[int, str]) -> List[List[str]]:
    """Token ids [B, T] (tensor or nested lists) -> words per row: BOS / PAD words are dropped, the row ends at
    the first EOS word, an empty row becomes [UNK]  (common/Utils.py:193-210)."""
    if isinstance(batch_indices, torch.Tensor):
        rows = batch_indices.detach().to('cpu').tolist()        # ONE copy for the whole batch
    else:
        rows = [[int(x) for x in r] for r in batch_indices]
    out = []
    for ids in rows:
        words = []
        for i in ids:
            w = id2vocab[i]
            if w == BOS_WORD or w == PAD_WORD:
                continue
            if w == EOS_WORD:
                break
            words.append(w)
        out.append(words if words else [UNK_WORD])
    return out


def source_location(source, S0: int, Lp: int):
    """Attribution source position (``Attributed.source``: an index of CaSE's ``source_map``, the query's S0 positions
    followed by the passages flattened [NP][Lp], CaSEDataset.py:98-104) -> (memory, passage, offset): (0, -1, s) for a
    query position, (1, p, o) for offset o of passage p, (-1, -1, -1) for source -1 (pure generation).  Works on an int
    or elementwise on an integer tensor (then three int64 tensors of its shape)."""
    if isinstance(source, torch.Tensor):
        s = source.to(torch.int64)
        none, query = s < 0, s < S0
        q = s - S0
        neg = torch.full_like(s, -1)
        memory = torch.where(none, neg, torch.where(query, torch.zeros_like(s), torch.ones_like(s)))
        passage = torch.where(none | query, neg, torch.div(q, Lp, rounding_mode='floor'))
        offset = torch.where(none, neg, torch.where(query, s, q % Lp))
        return memory, passage, offset
    s = int(source)
    if s < 0:
        return -1, -1, -1
    if s < S0:
        return 0, -1, s
    return 1, (s - S0) // Lp, (s - S0) % Lp


def _cut_point(sent: Sequence, n: int) -> int:
    """The cut ``remove_duplicate_once`` takes for one sentence, or -1: the LARGEST index in [1, len - n] such
    that every element of sent[index:] also occurs in sent[:index]  (common/Utils.py:176-186).
    An element at position p >= index occurs in the prefix iff its first occurrence is < index, so the test
    is max(first_occurrence over the suffix) < index."""
    L = len(sent)
    if L <= n:
        return -1
    first = {}
    fo = [0] * L
    for p, w in enumerate(sent):
        fo[p] = first.setdefault(w, p)
    suffix_max = -1
    for p in range(L - 1, L - n, -1):          # positions that belong to every candidate suffix
        suffix_max = max(suffix_max, fo[p])
    for index in range(L - n, 0, -1):
        suffix_max = max(suffix_max, fo[index])
        if suffix_max < index:
            return index
    return -1


def remove_duplicate_once(sents: List[List], n: int = 3) -> bool:
    changed = False
    for b in range(len(sents)):
        cut = _cut_point(sents[b], n)
        if cut >= 0:
            sents[b] = sents[b][:cut]
            changed = True
    return changed


def remove_duplicate(sents: List[List], n: int = 3) -> None:
    """In place: while some sentence ends in a tail (>= n tokens) made only of tokens seen before it, drop that
    tail  (common/Utils.py:188-191)."""
    while remove_duplicate_once(sents, n):
        pass


def bert_detokenizer() -> Callable[[Sequence[str]], str]:
    def detokenizer(tokens):
        return ' '.join(tokens).replace(' ##', '').strip()
    return detokenizer


def nltk_detokenizer() -> Callable[[Sequence[str]], str]:
    def detokenizer(tokens):
        return ' '.join(tokens)
    return detokenizer


def answers_from_tokens(tokens, id2vocab, detokenizer=None) -> List[str]:
    """tokens [B, T] -> final answer strings: to_sentence -> remove_duplicate -> detokenise (Utils.py:17-24)."""
    sents = to_sentence(tokens, id2vocab)
    remove_duplicate(sents)
    detok = detokenizer or bert_detokenizer()
    return [detok(s) for s in sents]


def save_result(predictions, dataset, to_sentence, detokenizer, output_path, local_rank, epoch, eval_type):
    """Drop-in for Utils.save_result (Utils.py:5-49): ``predictions`` is the list of ``[data, output]`` pairs
    CumulativeTrainer.predict returns; writes ``result/<eval_type>_<epoch>.<local_rank>.answer`` (context ids ;
    query id ; passage ids ; answer, tab separated) and ``.run`` (TREC run lines, one ranking per query sorted
    by score, ties in pool order).  ``to_sentence(data, indices)`` is the model's method (CaSE/Model.py:270).
    Returns (answer_path or None, run_path or None)."""
    system_answers, system_ranks = [], []
    for data, output in predictions:
        sents = None
        if 'answer' in output:
            sents = to_sentence(data, output['answer'])
            remove_duplicate(sents)
        ids = data['id'].detach().to('cpu').tolist() if isinstance(data['id'], torch.Tensor) else list(data['id'])
        scores = None
        if 'rank' in output:
            r = output['rank']
            scores = r.detach().to('cpu').tolist() if isinstance(r, torch.Tensor) else r
        for i, qid in enumerate(ids):
            if sents is not None:
                system_answers.append([';'.join(dataset.context_id(qid)), dataset.query_id(qid),
                                       ';'.join(dataset.passage_id(qid)), detokenizer(sents[i])])
            if scores is not None:
                pool = dataset.pool(qid)
                run = [[dataset.query_id(qid), 'Q0', pool[j], 0, scores[i][j], 'system'] for j in range(len(pool))]
                run.sort(key=lambda r_: r_[4], reverse=True)            # stable, like sorted() in the reference
                for k, r_ in enumerate(run):
                    r_[3], r_[4] = str(k + 1), str(r_[4])
                system_ranks.append(run)
    out_dir = os.path.join(output_path, 'result/')
    os.makedirs(out_dir, exist_ok=True)
    answer_path = run_path = None
    stem = os.path.join(out_dir, eval_type + '_' + str(epoch) + '.' + str(local_rank))
    if system_answers:
        answer_path = stem + '.answer'
        with codecs.open(answer_path, 'w', 'utf-8') as f:
            for row in system_answers:
                f.write('\t'.join(row) + os.linesep)
    if system_ranks:
        run_path = stem + '.run'
        with codecs.open(run_path, 'w', 'utf-8') as f:
            for run in system_ranks:
                for row in run:
                    f.write(' '.join(row) + os.linesep)
    return answer_path, run_path
