"""Device-side engines for the CaSE and GTTP answer decoders.

An engine owns every device buffer of one (B, W, S, Tmax, V) problem shape, fills the C argument
struct once, and then a decode is: ``prefill(inputs)`` (once per batch: project the memories,
build masks / priors / copy map) followed by ``max_len`` calls of ``case_decode_step`` /
``gttp_decode_step`` - optionally replayed from a captured CUDA graph.  torch is used for device
memory, streams and the per-batch prefill GEMMs only; every per-step op is a kernel of
libcase_b200.so.  There is no CPU path.

Reference being replaced: the eval loop of CaSETransformerSeqDecoder.forward (CaSE/Model.py:91-123),
Generations.greedy/beam (common/Generations.py:66-190) and the GTTP step (GTTP/Model.py:113-131,
14-43, 176-193).
"""
import ctypes as C
import math
import operator
import os
from typing import Dict, NamedTuple, Optional, Tuple

import numpy as np
import torch

from . import _lib as L

PAD, BOS, EOS, UNK = 0, 1, 2, 100


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise RuntimeError('case_rg_b200 needs a CUDA device: the decode path has no CPU fallback')
    dev = torch.device(device if device is not None else 'cuda')
    if dev.type != 'cuda':
        raise RuntimeError(f'case_rg_b200 needs a CUDA device, got {dev}: the decode path has no CPU fallback')
    if dev.index is None:
        dev = torch.device('cuda', torch.cuda.current_device())
    return dev


class _on_device:
    """The C launchers work on the calling thread's CURRENT device (include/case_b200.h): every engine entry point
    runs under its own device, so an engine built for cuda:1 is usable whatever the caller's current device is."""

    def __init__(self, dev):
        self.guard = torch.cuda.device(dev)

    def __enter__(self):
        return self.guard.__enter__()

    def __exit__(self, *a):
        return self.guard.__exit__(*a)


class _Fork:
    """Owner of a case_fork_t (side stream + events of the step's fork/join) on one device."""

    def __init__(self, dev):
        self.h = C.c_void_p()
        with torch.cuda.device(dev):
            L.check(L.load().case_fork_create(C.byref(self.h)), 'case_fork_create')

    def __del__(self):
        try:
            if self.h:
                L.load().case_fork_destroy(self.h)
                self.h = C.c_void_p()
        except Exception:
            pass


def _storage(dtype: str):
    if dtype in ('bf16', 'bfloat16'):
        return torch.bfloat16, L.BF16
    if dtype in ('fp32', 'float32', 'f32'):
        return torch.float32, L.F32
    raise ValueError(f'dtype must be "bf16" or "fp32", got {dtype!r}')


def _nsplit(units_per_split_group: int, S: int, tile: int, target_ctas: int) -> int:
    """splits so that units*nsplit >= target CTAs, bounded by the tile count and the ABI limit"""
    n = max(1, -(-target_ctas // max(1, units_per_split_group)))
    return int(max(1, min(n, L.MAX_SPLIT, -(-S // tile))))


def _nsplit_additive(B: int, S: int, bf16: bool, target_ctas: int = 296) -> int:
    """Key splits of the additive attention (CTAs = B * nsplit).  bf16 kernel: splits are whole 32-key
    tiles and 2 CTAs are resident per SM, so pick the split count that minimises
    (rounds of 296 resident CTAs) x (tiles per split) - at B = 64, S = 2560 that is 9 splits (576 CTAs,
    two full rounds of 9 tiles) instead of 10 (640 CTAs: a third, mostly empty round).  fp32 kernel:
    the older rule on 128-key tiles."""
    if not bf16:
        return _nsplit(B, S, L.AATTN_TILE, 2 * target_ctas)
    best, best_cost = 1, None
    for ns in range(1, L.MAX_SPLIT + 1):
        chunk = -(-(-(-S // ns)) // 32) * 32
        if (ns - 1) * chunk >= S:          # the last split would be empty
            continue
        cost = -(-(B * ns) // target_ctas) * (chunk // 32)
        if best_cost is None or cost < best_cost or (cost == best_cost and ns < best):
            best, best_cost = ns, cost
    return best


def build_copy_plan(smap, valid, V, cp_n, cp_uid, cp_first, cp_start, cp_perm):
    """Copy plan of a batch for case_sparse_tail (case_tail_args_t.cp_*): per query the VALID source positions
    (valid [B, St] bool over the concatenation [memory 0 ; memory 1], ids smap [B, St] inside [0, V)) sorted by
    vocabulary id - stable, so position order inside an id - and the list of unique ids with, per id, its first
    position | (occurrences - 1) << 16 and the start of its run.  Outputs int32 [B] / [B, St + 1] (a spare column
    takes the writes of the non-heads).  Device-side torch ops only, no synchronisation."""
    B, St = valid.shape
    ids = smap.to(torch.int64)
    BIG = 1 << 40
    key = torch.where(valid & (ids >= 0) & (ids < V), ids, torch.full_like(ids, BIG))
    sid, perm = torch.sort(key, dim=1, stable=True)
    live = sid < BIG
    head = live.clone()
    head[:, 1:] &= sid[:, 1:] != sid[:, :-1]
    uidx = head.cumsum(1) - 1                          # list index of every sorted position
    spare = torch.full_like(uidx, St)
    tgt = torch.where(head, uidx, spare)               # non-heads write the spare column
    ar = torch.arange(St, device=valid.device, dtype=torch.int32).expand(B, St)
    cp_uid.scatter_(1, tgt, sid.to(torch.int32))
    cp_start.scatter_(1, tgt, ar)
    cnt = torch.zeros_like(cp_first)
    cnt.scatter_add_(1, torch.where(live, uidx, spare), torch.ones_like(ar))
    cp_first.scatter_(1, tgt, perm.to(torch.int32))
    cp_first.bitwise_or_((cnt - 1).clamp_(min=0) << 16)
    cp_perm[:, :St].copy_(perm)
    cp_n.copy_(head.sum(1))


def pack_tiled(w: torch.Tensor, dtype) -> torch.Tensor:
    """nn.Linear weight [N, K] -> the kernels' streaming layout (one contiguous run of 16 KB tiles per
    256 output columns).  fp32: [N/256][K][256] for the CUDA-core kernels.  bf16: [N/256][K/32] slabs
    of [256 n][32 k] for the mma.sync kernels, the four 16-byte k-chunks of every row XOR-swizzled
    with ((n >> 1) & 3) so ldmatrix reads are bank-conflict free (layout: csrc/rowops_tc.cu)."""
    N, K = w.shape
    if N % 256 or K % 32:
        raise ValueError(f'weight {tuple(w.shape)}: N must be a multiple of 256 and K of 32')
    if dtype == torch.bfloat16:
        t = w.to(torch.bfloat16).reshape(N // 256, 256, K // 32, 4, 8).permute(0, 2, 1, 3, 4)   # [nt][slab][n][chunk][8]
        n = torch.arange(256, device=w.device)
        src = torch.arange(4, device=w.device)[None, :] ^ ((n >> 1) & 3)[:, None]                # [n][chunk'] -> chunk
        return t[:, :, n[:, None], src].contiguous()
    return w.t().reshape(K, N // 256, 256).permute(1, 0, 2).contiguous().to(dtype)


def unpack_tiled(wp: torch.Tensor, N: int, K: int) -> torch.Tensor:
    """Inverse of pack_tiled -> fp32 [N, K] (used by tests to share the storage rounding)."""
    if wp.dtype == torch.bfloat16:
        n = torch.arange(256, device=wp.device)
        src = torch.arange(4, device=wp.device)[None, :] ^ ((n >> 1) & 3)[:, None]               # the XOR is an involution
        t = wp.view(N // 256, K // 32, 256, 4, 8)[:, :, n[:, None], src]
        return t.permute(0, 2, 1, 3, 4).reshape(N, K).float()
    return wp.float().permute(0, 2, 1).reshape(N, K)


def pack_cluster(mats) -> torch.Tensor:
    """Eight nn.Linear weights [256 out][256 in] (Wq, Wk, Wv, Wo, Wq2, Wo2, W1, W2) -> the layout of
    case_layer_chain: bf16 [4 ranks][8 matrices][64 n][256 k], rank c = output rows 64c..64c+63, the
    16-byte chunk kc of row n stored at chunk position kc ^ (n & 7) (csrc/layer_cluster.cu)."""
    w = torch.stack([m.to(torch.bfloat16) for m in mats])              # [m][256 n][256 k]
    if tuple(w.shape) != (8, 256, 256):
        raise ValueError(f'pack_cluster needs eight 256x256 matrices, got {tuple(w.shape)}')
    w = w.view(8, 4, 64, 32, 8)                                          # [m][rank][n][kc][8]
    n = torch.arange(64, device=w.device)
    src = torch.arange(32, device=w.device)[None, :] ^ (n & 7)[:, None]  # stored position p holds chunk p ^ (n & 7)
    return w[:, :, n[:, None], src].permute(1, 0, 2, 3, 4).contiguous()


def pack_post(w: torch.Tensor) -> torch.Tensor:
    """nn.Linear weight [256 out][256 * nchunk in] -> the post-linear layout of the cluster kernels: bf16
    [4 ranks][nchunk][64 n][256 k], chunk kc of row n stored at kc ^ (n & 7) (csrc/layer_cluster.cu)."""
    N, K = w.shape
    if N != 256 or K % 256:
        raise ValueError(f'pack_post needs a [256, 256*n] weight, got {tuple(w.shape)}')
    t = w.to(torch.bfloat16).view(4, 64, K // 256, 32, 8)               # [rank][n][chunk][kc][8]
    n = torch.arange(64, device=w.device)
    src = torch.arange(32, device=w.device)[None, :] ^ (n & 7)[:, None]
    return t.permute(0, 2, 1, 3, 4)[:, :, n[:, None], src].contiguous()  # [rank][chunk][n][p][8]: position p holds chunk p ^ (n & 7)


def pack_vocab_tc(w: torch.Tensor, rows: int = 128) -> torch.Tensor:
    """[V, 256] output-projection weight -> bf16 tiles of ``rows`` rows in the UMMA K-major no-swizzle
    canonical layout the tcgen05 kernels bulk-copy straight into shared memory (case_b200.h)."""
    V, K = w.shape
    VT = -(-V // rows)
    wp = torch.zeros(VT * rows, K, dtype=torch.bfloat16, device=w.device)
    wp[:V] = w.to(torch.bfloat16)
    return wp.view(VT, rows // 8, 8, K // 8, 8).permute(0, 3, 1, 2, 4).contiguous()   # [tile][k/8][row/8][row%8][k%8]


_SWZ = {}


def _swizzle_index(device):
    """[64 keys][4 chunks] source chunk for each stored chunk position: c ^ ((key >> 1) & 3) (an involution)."""
    if device not in _SWZ:
        key = torch.arange(64, device=device)
        _SWZ[device] = (key[:, None], torch.arange(4, device=device)[None, :] ^ ((key >> 1) & 3)[:, None])
    return _SWZ[device]


def pack_kv_tiles(k: torch.Tensor, v: torch.Tensor, out: torch.Tensor = None) -> torch.Tensor:
    """K, V [B, NH, S, 32] -> the tensor-core cross-attention layout (case_b200.h): bf16
    [B][NH][ceil(S/64)][2][64][32], keys >= S zero, 16-byte chunks of each key row XOR-swizzled."""
    B, NH, S, HD = k.shape
    nt = -(-S // 64)
    if out is None:
        out = torch.zeros(B, NH, nt, 2, 64, HD, dtype=torch.bfloat16, device=k.device)
    kidx, cidx = _swizzle_index(k.device)
    for j, src in enumerate((k, v)):
        pad = torch.zeros(B, NH, nt * 64, HD, dtype=torch.bfloat16, device=k.device)
        pad[:, :, :S] = src
        out[:, :, :, j] = pad.view(B, NH, nt, 64, 4, 8)[:, :, :, kidx, cidx].reshape(B, NH, nt, 64, HD)
    return out


def split_chunk(S, nsplit, tile=128):
    c = -(-S // nsplit)
    return -(-c // tile) * tile


class CaseWeights:
    """Weights of CaSETransformerSeqDecoder re-laid-out for the kernels (CaSE/Model.py:14-36 names).

    Matrices are re-tiled to [N/256][K][256] in the storage dtype; the 1/sqrt(hd) attention scale is
    folded into the query projections; cross-attention K/V and attns.*.linear_key weights are kept
    fp32 [K][N] for the per-batch prefill GEMMs."""

    def __init__(self, sd: Dict[str, torch.Tensor], device=None, dtype: str = 'bf16', prefix: str = ''):
        dev = _require_cuda(device)
        self.device, self.dtype_name = dev, dtype
        self.tdtype, self.cdtype = _storage(dtype)
        g = lambda k: sd[prefix + k].detach().to(dev, torch.float32)
        self.H = H = g('embedding.0.weight').size(1)
        if H != L.H:
            raise ValueError(f'hidden_size must be {L.H} (got {H})')
        self.V = g('gen.2.weight').size(0)
        self.M = len({k[len(prefix):].split('.')[1] for k in sd if k.startswith(prefix + 'decs.')})
        self.Ln = len({k[len(prefix):].split('.')[3] for k in sd if k.startswith(prefix + 'decs.0.layers.')})
        if self.M != 2 or self.Ln != 4:
            raise ValueError('the fused step is built for num_memories=2, num_layers=4 (CaSE/Model.py:265)')
        scale = math.sqrt(1.0 / L.HD)
        mat = lambda w: pack_tiled(w, self.tdtype)
        vec = lambda b: b.contiguous()
        self.keep = []            # keeps every tensor alive
        self.layers = (L.LayerWeights * 8)()
        self.kv_w, self.kv_b = [], []                              # per stack: [H][Ln*2*H], [Ln*2*H]
        self._kv_rows, self.pf_bias = [], []
        for i in range(2):
            kvw, kvb = [], []
            for l in range(4):
                p = f'decs.{i}.layers.{l}.'
                Wi, bi = g(p + 'self_attn.in_proj_weight').clone(), g(p + 'self_attn.in_proj_bias').clone()
                Wi[:H] *= scale
                bi[:H] *= scale
                Wx, bx = g(p + 'multihead_attn.in_proj_weight'), g(p + 'multihead_attn.in_proj_bias')
                t = dict(Wqkv_t=mat(Wi), bqkv=vec(bi),
                         Wo_t=mat(g(p + 'self_attn.out_proj.weight')), bo=vec(g(p + 'self_attn.out_proj.bias')),
                         Wq2_t=mat(Wx[:H] * scale), bq2=vec(bx[:H] * scale),
                         Wo2_t=mat(g(p + 'multihead_attn.out_proj.weight')),
                         bo2=vec(g(p + 'multihead_attn.out_proj.bias')),
                         W1_t=mat(g(p + 'linear1.weight')), b1=vec(g(p + 'linear1.bias')),
                         W2_t=mat(g(p + 'linear2.weight')), b2=vec(g(p + 'linear2.bias')),
                         ln1_g=vec(g(p + 'norm1.weight')), ln1_b=vec(g(p + 'norm1.bias')),
                         ln2_g=vec(g(p + 'norm2.weight')), ln2_b=vec(g(p + 'norm2.bias')),
                         ln3_g=vec(g(p + 'norm3.weight')), ln3_b=vec(g(p + 'norm3.bias')))
                if self.cdtype == L.BF16:
                    t['Wc'] = pack_cluster([Wi[:H], Wi[H:2 * H], Wi[2 * H:], g(p + 'self_attn.out_proj.weight'),
                                            Wx[:H] * scale, g(p + 'multihead_attn.out_proj.weight'),
                                            g(p + 'linear1.weight'), g(p + 'linear2.weight')])
                self.keep.append(t)
                lw = self.layers[i * 4 + l]
                for k, v in t.items():
                    setattr(lw, k, v.data_ptr())
                kvw.append(Wx[H:].t())                            # [H][2H]: K cols then V cols
                kvb.append(bx[H:])
            self.kv_w.append(torch.cat(kvw, dim=1).contiguous().to(self.tdtype))  # [H][Ln*2H]
            self._kv_rows.append(torch.cat([k.t() for k in kvw], dim=0))             # [Ln*2H][H] fp32
            self.pf_bias.append(torch.cat(kvb).float().contiguous())
            self.kv_b.append(torch.cat(kvb).contiguous().to(self.tdtype))
        self.E = g('embedding.0.weight').contiguous()
        self.pe = g('embedding.1.pe').contiguous()
        self.lnN_g, self.lnN_b = vec(g('norm1.weight')), vec(g('norm1.bias'))
        self.ln2_g, self.ln2_b = vec(g('norm2.weight')), vec(g('norm2.bias'))
        self.Wqa_t = [mat(g(f'attns.{i}.linear_query.weight')) for i in range(2)]
        self.bqa = [vec(g(f'attns.{i}.linear_query.bias')) for i in range(2)]
        self.va = [g(f'attns.{i}.v.weight').reshape(-1).contiguous() for i in range(2)]
        self.Uk_t = [g(f'attns.{i}.linear_key.weight').t().contiguous().to(self.tdtype) for i in range(2)]   # [H][H]
        self.Wg_t, self.bg = mat(g('gen.0.weight')), vec(g('gen.0.bias'))
        bf = self.cdtype == L.BF16
        # prefill GEMM of case_prefill_project_tc: rows (layer, K|V, head, dim) of the stack ++ the rows of Uk, 128-row blocks
        self.Wpf = [pack_vocab_tc(torch.cat([self._kv_rows[i], g(f'attns.{i}.linear_key.weight')], 0)) if bf else None
                    for i in range(2)]
        del self._kv_rows
        self.Wqa_c = [pack_post(g(f'attns.{i}.linear_query.weight')) if bf else None for i in range(2)]
        self.Wg_c = pack_post(g('gen.0.weight')) if bf else None
        self.Wv = g('gen.2.weight').contiguous().to(self.tdtype)                               # [V][H]
        self.Wv_tc = pack_vocab_tc(g('gen.2.weight')) if self.cdtype == L.BF16 else None
        self.Wm, self.bm = g('mix.weight').contiguous(), vec(g('mix.bias'))
        # gate form (CaSE/Model.py:39,117): W_m's slice for context i as a [H][4] projection of the memory keys
        self.Wm_g = [self.Wm[:, H * (1 + i):H * (2 + i)].contiguous() for i in range(2)]          # [3][H] each


class NBest(NamedTuple):
    """The n best finished hypotheses of every query, in rank order (sorted(results[q], key=cum_cost/length)[:n],
    Generations.py:183-185): ``tokens`` int64 [B, n, L] (BOS dropped, EOS kept, zero padded to the longest entry of the
    batch), ``lengths`` int64 [B, n] answer tokens, ``costs`` fp64 [B, n] the ranking key cum_cost / length in nats per
    position (BOS counted in the length; lower is better)."""
    tokens: torch.Tensor
    lengths: torch.Tensor
    costs: torch.Tensor


def nbest_from(out_tokens, best_len, best_key) -> NBest:
    """n-best buffers of a search state (out_tokens [B, (n,) Tmax], best_len / best_key [B, (n)]) -> NBest on their
    device, trimmed like merge1D (Utils.py:366-377) to the longest entry."""
    B = best_len.size(0)
    lengths = best_len.reshape(B, -1).to(torch.int64)
    n = lengths.size(1)
    L = max(int(lengths.max()), 1)
    return NBest(out_tokens.reshape(B, n, -1)[:, :, :L].to(torch.int64), lengths,
                 best_key.reshape(B, n).clone())


class Attributed(NamedTuple):
    """Answers with the attribution record of every token: where its probability came from in the mixture of its parent
    prefix (CaSE/Model.py:38-48, GTTP/Model.py:25-43).  ``answer``: the search's own result (the ``beam_nbest`` NBest,
    or the LongTensor of ``greedy`` / ``beam``).  ``parts`` fp32 [..., L, P]: the split of the chosen token's probability
    p(y) - the ``p`` whose -log(p + 1e-10) entered the cost - into P parts that sum to it: CaSE (P = 3) generation, copy
    from the query, copy from the passages; GTTP (P = 2) generation, copy from the background.  ``source`` int64
    [..., L]: the source position with the largest single copy contribution to the token (an index of ``source_map`` /
    ``background_map``, ties to the lowest position; see ``results.source_location``), -1 for pure generation.
    Positions past an answer's end (and greedy PAD positions) have zero parts and source -1."""
    answer: object
    parts: torch.Tensor
    source: torch.Tensor


def attributed_from(out_tokens, best_len, best_key, out_attr, P, mode, max_len, nbest) -> Attributed:
    """Search-state buffers (out_tokens [B, (n,) T], best_len / best_key [B, (n)], out_attr [B, (n,) T, 4] fp32 records)
    -> Attributed on their device.  nbest: the answer is the NBest list and the records are [B, n, L, ...]; otherwise the
    answer is entry 0's token rows ([B, max_len] greedy; beam trimmed to the longest answer) and the records [B, L, ...]."""
    B = best_len.size(0)
    rec = out_attr.reshape(B, -1, out_attr.size(-2), 4)[:, :, :max_len]
    if mode == L.MODE_BEAM:
        rec = rec[:, :, :max(int(best_len.max()), 1)]         # merge1D, like the token rows
    parts = rec[..., :P].clone()
    source = rec[..., 3].contiguous().view(torch.int32).to(torch.int64)
    if nbest:
        return Attributed(nbest_from(out_tokens, best_len, best_key), parts, source)
    toks = out_tokens.reshape(B, -1, out_tokens.size(-1))[:, 0, :rec.size(2)].to(torch.int64)
    return Attributed(toks, parts[:, 0], source[:, 0])


def check_attribution(opt: int, V: int, W: int, nsources: int) -> None:
    """Attribution records come from the sparse tail only: ValueError for a request the step would refuse."""
    if opt & (L.OPT_DENSE_TAIL | L.OPT_UNFUSED_TAIL):
        raise ValueError('attribution needs the sparse tail: not with OPT_DENSE_TAIL / OPT_UNFUSED_TAIL')
    if V < 2 * W:
        raise ValueError(f'attribution needs the sparse tail, which needs V >= 2 * width (V = {V}, width = {W})')
    if nsources > L.load().case_sparse_tail_max_sources():
        raise ValueError(f'attribution needs the sparse tail: {nsources} source positions exceed its '
                         f'{L.load().case_sparse_tail_max_sources()}')


def check_constraints(opt: int, V: int, W: int, nsources: int, Tmax: int, no_repeat_ngram: int, min_len: int,
                      max_len: Optional[int] = None, mode: Optional[int] = None) -> None:
    """Search constraints (no_repeat_ngram / min_len, 0 = off) are applied by the sparse tail only: ValueError for a
    request the step would refuse.  max_len / mode: also check them against one decode."""
    n, m = int(no_repeat_ngram), int(min_len)
    if n == 0 and m == 0:
        return
    lim = Tmax if max_len is None else max_len
    if not 0 <= n <= lim:
        raise ValueError(f'no_repeat_ngram must be 0..max_len ({lim}), got {n}')
    if not 0 <= m < lim:
        raise ValueError(f'min_len must be 0..max_len - 1 ({lim - 1}), got {m}')
    if mode is not None and mode not in (L.MODE_BEAM, L.MODE_PROTO_GREEDY):
        raise ValueError('no_repeat_ngram / min_len apply to the beam and greedy searches (not module_greedy)')
    if opt & (L.OPT_DENSE_TAIL | L.OPT_UNFUSED_TAIL):
        raise ValueError('no_repeat_ngram / min_len need the sparse tail: not with OPT_DENSE_TAIL / OPT_UNFUSED_TAIL')
    if V < 2 * W + Tmax + 1:
        raise ValueError(f'no_repeat_ngram / min_len need V >= 2 * width + max_target_length + 1 (V = {V}, width = {W}, '
                         f'max_target_length = {Tmax})')
    if nsources > L.load().case_sparse_tail_max_sources():
        raise ValueError(f'no_repeat_ngram / min_len need the sparse tail: {nsources} source positions exceed its '
                         f'{L.load().case_sparse_tail_max_sources()}')


class BadWords(NamedTuple):
    """A checked ban list (see check_bad_words): the distinct single ids (ascending) and the distinct sequences of two or
    more ids (in the caller's order)."""
    singles: Tuple[int, ...]
    seqs: Tuple[Tuple[int, ...], ...]


def _ban_ids(seq) -> Tuple[int, ...]:
    if isinstance(seq, torch.Tensor):
        if seq.dim() != 1 or seq.dtype.is_floating_point or seq.dtype.is_complex or seq.dtype == torch.bool:
            raise ValueError(f'a banned sequence must be a 1-D integer tensor or a list of ints, got {seq.dtype} '
                             f'{tuple(seq.shape)}')
        return tuple(seq.tolist())
    if isinstance(seq, (str, bytes)) or not hasattr(seq, '__iter__'):
        raise ValueError(f'a banned sequence must be a 1-D integer tensor or a list of ints, got {seq!r}')
    ids = tuple(seq)
    if all(type(v) is int for v in ids):                 # the common case, without the per-id checks below
        return ids
    for v in ids:
        if isinstance(v, bool) or not hasattr(v, '__index__'):
            raise ValueError(f'banned ids must be ints, got {v!r}')
    return tuple(operator.index(v) for v in ids)


def _check_bans_servable(opt: int, V: int, W: int, nsources: int, Tmax: int, mode: Optional[int] = None) -> None:
    """Bans run in the sparse tail's constrained instance: ValueError where a search cannot take it."""
    if mode is not None and mode not in (L.MODE_BEAM, L.MODE_PROTO_GREEDY):
        raise ValueError('bad_words apply to the beam and greedy searches (not module_greedy)')
    if opt & (L.OPT_DENSE_TAIL | L.OPT_UNFUSED_TAIL):
        raise ValueError('bad_words need the sparse tail: not with OPT_DENSE_TAIL / OPT_UNFUSED_TAIL')
    if nsources > L.load().case_sparse_tail_max_sources():
        raise ValueError(f'bad_words need the sparse tail: {nsources} source positions exceed its '
                         f'{L.load().case_sparse_tail_max_sources()}')
    if V < 2 * W + Tmax + 1:
        raise ValueError(f'bad_words need V >= 2 * width + max_target_length + 1 (V = {V}, width = {W}, '
                         f'max_target_length = {Tmax})')


def check_bad_words(opt: int, V: int, W: int, nsources: int, Tmax: int, bad_words,
                    mode: Optional[int] = None) -> Optional[BadWords]:
    """Banned words (a list of token-id sequences, each a list of ints or a 1-D integer tensor; None or empty = off) ->
    the checked BadWords, or None when off.  ValueError for a list or a search the device cannot serve: ids outside
    [0, V) (dynamic OOV ids differ per query), an empty sequence, more than MAX_BAN_SEQ sequences of two or more ids, a
    sequence longer than MAX_BAN_LEN, no sparse tail (OPT_DENSE_TAIL / OPT_UNFUSED_TAIL, too many source positions),
    module_greedy (mode), or fewer than 2 * width + max_target_length + 1 + (sequences) ids left allowed.  Duplicates are
    dropped; a BadWords is checked against the search only."""
    if bad_words is None:
        return None
    if isinstance(bad_words, torch.Tensor) or isinstance(bad_words, (str, bytes)):
        raise ValueError('bad_words must be a list of token-id sequences (lists of ints or 1-D integer tensors)')
    if isinstance(bad_words, BadWords):                   # checked already: only the search-dependent limits
        singles, seqs = bad_words.singles, bad_words.seqs
        if not 0 <= len(seqs) <= L.MAX_BAN_SEQ or (singles and not 0 <= min(singles) <= max(singles) < V):
            raise ValueError('bad_words: a BadWords outside the limits')
        return _check_ban_counts(opt, V, W, nsources, Tmax, bad_words, mode)
    singles, seqs = set(), {}                             # seqs: an insertion-ordered set
    for seq in bad_words:
        ids = _ban_ids(seq)
        if not ids:
            raise ValueError('bad_words: a banned sequence is empty')
        if len(ids) > L.MAX_BAN_LEN:
            raise ValueError(f'bad_words: a sequence of {len(ids)} ids exceeds MAX_BAN_LEN = {L.MAX_BAN_LEN}')
        if not (0 <= min(ids) and max(ids) < V):
            bad = next(v for v in ids if not 0 <= v < V)
            raise ValueError(f'bad_words: id {bad} outside [0, V = {V}) (dynamic OOV ids cannot be banned by value)')
        if len(ids) == 1:
            singles.add(ids[0])
        else:
            seqs[ids] = None
    if not singles and not seqs:
        return None
    if len(seqs) > L.MAX_BAN_SEQ:
        raise ValueError(f'bad_words: {len(seqs)} sequences of two or more ids exceed MAX_BAN_SEQ = {L.MAX_BAN_SEQ}')
    return _check_ban_counts(opt, V, W, nsources, Tmax, BadWords(tuple(sorted(singles)), tuple(seqs)), mode)


def _check_ban_counts(opt, V, W, nsources, Tmax, bw: BadWords, mode) -> Optional[BadWords]:
    if not bw.singles and not bw.seqs:
        return None
    _check_bans_servable(opt, V, W, nsources, Tmax, mode)
    if V - len(bw.singles) < 2 * W + Tmax + 1 + len(bw.seqs):
        raise ValueError(f'bad_words leave too few ids: need V - (single ids) >= 2 * width + max_target_length + 1 + '
                         f'(sequences) (V = {V}, {len(bw.singles)} single ids, width = {W}, max_target_length = {Tmax}, '
                         f'{len(bw.seqs)} sequences)')
    return bw


class _BanBuffers:
    """Fixed-capacity device copy of a ban list, the layout of case_tail_args_t.ban_*: one int32 buffer holding the
    single-id bit mask [ceil(V / 32)], the sequence table [MAX_BAN_SEQ][MAX_BAN_LEN], the lengths [MAX_BAN_SEQ] and the
    count.  ``write`` replaces the content with a stream-ordered copy on the current stream, so a decode (or a captured
    graph) enqueued after it reads the new list and the ones enqueued before it read the old one."""

    def __init__(self, dev, V):
        self.nw = (V + 31) // 32
        nt = L.MAX_BAN_SEQ * L.MAX_BAN_LEN
        self.buf = torch.zeros(self.nw + nt + L.MAX_BAN_SEQ + 1, dtype=torch.int32, device=dev)
        self.mask = self.buf[:self.nw]
        self.tok = self.buf[self.nw:self.nw + nt]
        self.len = self.buf[self.nw + nt:self.nw + nt + L.MAX_BAN_SEQ]
        self.n = self.buf[self.nw + nt + L.MAX_BAN_SEQ:]
        self.current = BadWords((), ())                      # what the buffer holds (the zeros: nothing banned)

    def bind(self, a):
        a.ban_mask, a.ban_tok, a.ban_len, a.ban_n = (self.mask.data_ptr(), self.tok.data_ptr(), self.len.data_ptr(),
                                                     self.n.data_ptr())

    def write(self, bw: BadWords):
        if bw == self.current:
            return
        nt = L.MAX_BAN_SEQ * L.MAX_BAN_LEN
        host = np.zeros(self.buf.numel(), dtype=np.uint32)
        ids = np.asarray(bw.singles, dtype=np.int64)
        np.bitwise_or.at(host, ids >> 5, (np.ones_like(ids) << (ids & 31)).astype(np.uint32))
        for i, seq in enumerate(bw.seqs):
            host[self.nw + i * L.MAX_BAN_LEN:self.nw + i * L.MAX_BAN_LEN + len(seq)] = seq
            host[self.nw + nt + i] = len(seq)
        host[-1] = len(bw.seqs)
        # pinned: the copy is asynchronous on the current stream; the caching host allocator keeps the block until it
        # has been read
        self.buf.copy_(torch.from_numpy(host.view(np.int32)).pin_memory(), non_blocking=True)
        self.current = bw


class _SearchState:
    """Buffers shared by both engines for the on-device greedy / beam bookkeeping.  nbest > 1: the beam search keeps
    the nbest best finished hypotheses of every query (best_key / best_len [B, nbest], out_tokens [B, nbest, Tmax]).
    attribution: the records of the search (case_attr_t as fp32 [..., 4], the source bits in the last lane) - of the
    top-k candidates attr_cand [R, W], of every (physical row, position) attr_hist [R, Tmax + 1], and of the returned
    tokens out_attr (the layout of out_tokens)."""

    def __init__(self, dev, B, W, Tmax, ext=False, nbest=1, attribution=False):
        if not 1 <= nbest <= W:
            raise ValueError(f'nbest must be 1..{W} (the beam width), got {nbest}')
        R, TL = B * W, Tmax + 1
        nb = () if nbest == 1 else (nbest,)
        i32 = dict(dtype=torch.int32, device=dev)
        self.tok = torch.zeros(R, TL, **i32)
        # extended vocabulary: tok feeds the decoder (OOV ids become UNK), tok_ext keeps the ids of the returned sequences
        self.tok_ext = torch.zeros(R, TL, **i32) if ext else None
        self.anc = [torch.zeros(R, TL, **i32), torch.zeros(R, TL, **i32)]
        self.live = torch.zeros(R, **i32)
        self.cum = torch.zeros(R, dtype=torch.float64, device=dev)
        self.length = torch.zeros(R, **i32)
        self.parent = torch.zeros(R, **i32)
        self.ended = torch.zeros(B, **i32)
        self.best_key = torch.zeros(B, *nb, dtype=torch.float64, device=dev)
        self.best_len = torch.zeros(B, *nb, **i32)
        self.out_tokens = torch.zeros(B, *nb, Tmax, **i32)
        self.n_live = torch.zeros(B, **i32)
        self.attribution = bool(attribution)
        if self.attribution:
            f32 = dict(dtype=torch.float32, device=dev)
            self.attr_cand = torch.zeros(R, W, 4, **f32)
            self.attr_hist = torch.zeros(R, TL, 4, **f32)
            self.out_attr = torch.zeros(B, *nb, Tmax, 4, **f32)
        self.B, self.W, self.R, self.Tmax, self.nbest = B, W, R, Tmax, nbest
        self._arange = torch.arange(R, **i32)
        self._slot0 = (self._arange % W == 0).to(torch.int32)

    def reset(self, bos=BOS):
        self.tok.zero_()
        self.tok[:, 0] = bos
        if self.tok_ext is not None:
            self.tok_ext.copy_(self.tok)
        self.anc[0].copy_(self._arange[:, None].expand_as(self.anc[0]))   # every row is its own history
        self.anc[1].copy_(self.anc[0])
        self.live.copy_(self._slot0)            # one root hypothesis per query (Generations.py:132-134)
        self.cum.zero_()
        self.length.fill_(1)
        self.parent.copy_(self._arange)
        self.ended.zero_()
        self.best_key.fill_(float('inf'))
        self.best_len.zero_()
        self.out_tokens.zero_()
        self.n_live.zero_()
        if self.attribution:                    # zero records: parts 0, source -1
            for r in (self.attr_hist, self.out_attr):
                r.zero_()
                r[..., 3].view(torch.int32).fill_(-1)

    def bind(self, a):
        a.anc[0], a.anc[1] = self.anc[0].data_ptr(), self.anc[1].data_ptr()
        for n in ('tok', 'live', 'cum', 'length', 'parent', 'ended', 'best_key', 'best_len', 'out_tokens', 'n_live'):
            setattr(a, n, getattr(self, n).data_ptr())
        a.nbest = self.nbest
        if self.attribution:
            a.attr_cand, a.attr_hist, a.out_attr = (self.attr_cand.data_ptr(), self.attr_hist.data_ptr(),
                                                    self.out_attr.data_ptr())


class _EngineBase:
    def set_options(self, opt: int):
        """CASE_OPT_* bits of this engine's step calls (0 = the default fast path); drops captured graphs."""
        if int(opt) != int(self.args.opt):
            self.args.opt = int(opt)
            self._graphs.clear()

    # The step orchestrator is reached either through ctypes (default) or through the torch custom op
    # case_b200::decode_step / gttp_step (use_torch_ops = True): the same C entry point, the same argument block - the op
    # takes it as a uint8 view of the ctypes struct - and the stream is torch's current stream either way.
    use_torch_ops = False

    def _check_launch_constraints(self, max_len: int, mode: int) -> None:
        n, m = self.constraints
        if n or m:
            check_constraints(int(self.args.opt), self.V, self.W, 0, self.Tmax, n, m, max_len, mode)
        if self.bans is not None:
            _check_bans_servable(int(self.args.opt), self.V, self.W, 0, self.Tmax, mode)

    def set_bad_words(self, bad_words) -> None:
        """The ban list of the decodes launched after this call (an engine built with bans=True; see check_bad_words; a
        checked BadWords is taken as it is).  None or empty: nothing banned.  The list is copied into the engine's
        buffers on the current stream - no new graph capture, no host synchronisation."""
        if self.bans is None:
            if bad_words:
                raise ValueError('this engine was built without bans=True')
            return
        bw = check_bad_words(int(self.args.opt), self.V, self.W, 0, self.Tmax, bad_words)
        self.bans.write(bw if bw is not None else BadWords((), ()))

    def _step(self, t: int, cuda_stream: int):
        if self.use_torch_ops:
            ops = L.load_torch_ops()
            if getattr(self, '_args_blob', None) is None:
                self._args_blob = torch.frombuffer(self.args, dtype=torch.uint8)
            (ops.gttp_step if self._step_name == 'gttp_decode_step' else ops.decode_step)(self._args_blob, t)
        else:
            L.check(self._step_fn(C.byref(self.args), t, cuda_stream), self._step_name)

    def _run_steps(self, max_len: int):
        with _on_device(self.device):
            stream = torch.cuda.current_stream(self.device)
            for t in range(max_len):
                self._step(t, stream.cuda_stream)

    def _capture(self, max_len, mode):
        """Capture all ``max_len`` steps into one CUDA graph (t is a by-value kernel argument)."""
        with _on_device(self.device):
            stream = torch.cuda.current_stream(self.device)
            self._step(0, stream.cuda_stream)                                                  # warm-up, not captured
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                cs = torch.cuda.current_stream(self.device)
                for t in range(max_len):
                    self._step(t, cs.cuda_stream)
        self._graphs[(max_len, mode)] = g

    def _finish_tokens(self, max_len: int, mode: int) -> torch.Tensor:
        st = self.state
        out = st.out_tokens.view(st.B, -1, st.Tmax)[:, 0, :max_len].to(torch.int64)   # entry 0 of an n-best list
        if mode == L.MODE_BEAM:
            # merge1D (Utils.py:366-377): pad to the longest answer of the batch
            Lmax = int(st.best_len.view(st.B, -1)[:, 0].max().item())
            out = out[:, :max(Lmax, 1)]
        return out

    def _finish_nbest(self) -> NBest:
        """The n-best list of the last beam decode (see NBest), on the engine's device."""
        st = self.state
        return nbest_from(st.out_tokens, st.best_len, st.best_key)

    def _finish_attribution(self, max_len: int, mode: int, nbest: bool = False) -> Attributed:
        """The answers and attribution records of the last decode of an engine built with attribution=True (see
        Attributed); nbest: the answer is the NBest list and the records carry its n axis."""
        st = self.state
        if not st.attribution:
            raise ValueError('this engine was built without attribution=True')
        return attributed_from(st.out_tokens, st.best_len, st.best_key, st.out_attr, self.nparts, mode, max_len, nbest)


class CaseDecodeEngine(_EngineBase):
    """All buffers + the step argument block for one CaSE problem shape."""

    def __init__(self, weights: CaseWeights, B: int, W: int, S0: int, S1: int, Tmax: int = 40,
                 fast_tanh: Optional[bool] = None, vocab_impl: Optional[int] = None, target_ctas: int = 296,
                 opt: int = 0, n_oov: int = 0, nbest: int = 1, attribution: bool = False, no_repeat_ngram: int = 0,
                 min_len: int = 0, bans: bool = False):
        """n_oov > 0: extended vocabulary - ``source_map`` entries in [V, V + n_oov) are per-query dynamic (OOV) words,
        the mixture and its top-k range over V + n_oov ids (pointer-generator extension; an OOV id is fed back as UNK).
        nbest (1..W): a beam decode keeps the nbest best finished hypotheses per query (read with ``_finish_nbest``).
        attribution: every decode also records where each answer token came from (read with ``_finish_attribution``).
        no_repeat_ngram / min_len: search constraints of every beam / greedy decode (0 = off; see
        generations.beam): no answer repeats an n-gram, EOS is banned before step min_len.
        bans: the engine owns ban-list buffers and every decode applies the list last given to ``set_bad_words``."""
        self.opt, self.n_oov = int(opt), int(n_oov)
        if not (1 <= W <= L.MAX_W):
            raise ValueError(f'beam width must be 1..{L.MAX_W}')
        if attribution:
            check_attribution(self.opt, weights.V, W, S0 + S1)
        check_constraints(self.opt, weights.V, W, S0 + S1, Tmax, no_repeat_ngram, min_len)
        self.constraints = (int(no_repeat_ngram), int(min_len))
        if bans:
            _check_bans_servable(self.opt, weights.V, W, S0 + S1, Tmax)
        self.bans = _BanBuffers(weights.device, weights.V) if bans else None
        self.nparts = 3
        if not (1 <= Tmax <= L.MAX_T):
            raise ValueError(f'max_target_length must be 1..{L.MAX_T}')
        self.w = weights
        self.device = dev = weights.device
        self.B, self.W, self.R, self.S, self.Tmax, self.V = B, W, B * W, (S0, S1), Tmax, weights.V
        R, V, H = self.R, self.V, L.H
        self.ldv = -(-(V + self.n_oov) // 8) * 8
        td = weights.tdtype
        self.fast_tanh = int(weights.cdtype == L.BF16 if fast_tanh is None else fast_tanh)
        self.vocab_impl = int((1 if weights.cdtype == L.BF16 else 0) if vocab_impl is None else vocab_impl)
        if self.vocab_impl == 1 and weights.cdtype != L.BF16:
            raise ValueError('the tcgen05 vocabulary GEMM needs bf16 storage')
        self.vocab_ws = torch.zeros(max(16, L.load().case_vocab_tc_workspace_bytes(self.R)), dtype=torch.uint8,
                                    device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        z = lambda *s: torch.zeros(*s, **f32)
        if weights.cdtype == L.BF16:   # tensor-core kernel: CTA = (query, split), one warp per head, 1 CTA per SM
            self.nsx = [_nsplit(B, s, 2 * 64, 128) for s in self.S]
        else:                          # SIMT kernel: CTA = (query, head, split)
            self.nsx = [_nsplit(B * L.NH, s, L.XATTN_TILE, 6 * 148) for s in self.S]
        target_ctas = int(os.environ.get('CASE_ADD_CTAS', target_ctas))
        self.nsa = [_nsplit_additive(B, s, weights.cdtype == L.BF16, target_ctas) for s in self.S]
        # per-batch tensors
        self.feat = z(B, H)
        if weights.cdtype == L.BF16:      # interleaved, swizzled K|V tiles for the tensor-core kernel
            self.Kx = [torch.zeros(B, L.NH, -(-self.S[l // 4] // 64), 2, 64, L.HD, dtype=td, device=dev)
                       for l in range(8)]
            self.Vx = [None] * 8
        else:
            self.Kx = [torch.zeros(B, L.NH, self.S[l // 4], L.HD, dtype=td, device=dev) for l in range(8)]
            self.Vx = [torch.zeros(B, L.NH, self.S[l // 4], L.HD, dtype=td, device=dev) for l in range(8)]
        self.U = [torch.zeros(B, s, H, dtype=td, device=dev) for s in self.S]
        self.Mv = [torch.zeros(B, s, H, dtype=td, device=dev) for s in self.S]
        # gate-projected keys for the search path (case_additive_attn_gate): 3 gate logits' worth per key
        self.Gv = [z(B, s, 4) for s in self.S] if weights.cdtype == L.BF16 else None
        self.mask = [torch.zeros(B, s, dtype=torch.uint8, device=dev) for s in self.S]
        self.prior = [z(B, s) for s in self.S]
        self.map = torch.zeros(B, S0 + S1, dtype=torch.int32, device=dev)
        # state
        self.kcache = [torch.zeros(R, Tmax, H, dtype=td, device=dev) for _ in range(8)]
        self.vcache = [torch.zeros(R, Tmax, H, dtype=td, device=dev) for _ in range(8)]
        self.state = _SearchState(dev, B, W, Tmax, ext=self.n_oov > 0, nbest=nbest, attribution=attribution)
        # scratch
        # second memory: only valid keys are packed (case_cross_attn_part); CASE_NO_COMPACT=1 keeps the masked form (A/B)
        self.compact = weights.cdtype == L.BF16 and os.environ.get('CASE_NO_COMPACT', '0') != '1'
        # prefill projections on the own tcgen05 GEMM (K|V tiles + U written from its epilogue); CASE_PREFILL_TC=0: cuBLAS + pack (A/B)
        self.prefill_tc = weights.cdtype == L.BF16 and os.environ.get('CASE_PREFILL_TC', '1') != '0'
        self.xslots = L.load().case_cross_attn_part_slots(S1) if self.compact else 0
        nsx = max(max(self.nsx), self.xslots)
        self.xcount = torch.zeros(B, dtype=torch.int32, device=dev)
        self.xprefix = torch.zeros(B + 1, dtype=torch.int32, device=dev)
        self.xidx = torch.zeros(B, S1, dtype=torch.int32, device=dev) if self.compact else None
        self.xorder = torch.zeros(B, dtype=torch.int32, device=dev)
        self.qcount = torch.zeros(B, dtype=torch.int32, device=dev)
        # work-proportional key splits of the second memory's additive attention (gate form): query b uses
        # xns[b] of the MAX_SPLIT slots so that every CTA walks about the same number of valid keys and the
        # whole launch is one resident wave (add_slots CTAs).  Two CTAs per SM, not the three that fit: alone the
        # launch is slower that way (64 against 47 us), but three CTAs fill the register file, and with two the
        # vocabulary GEMM and vocab_base of the main stream get onto the SMs beside it - measured per step at C2:
        # 0.3357 / 0.3317 / 0.3295 / 0.3294 / 0.3327 ms for 222 / 259 / 296 / 333 / 444 slots
        self.prop_split = self.compact and self.Gv is not None and os.environ.get('CASE_PROP_SPLIT', '1') != '0'
        self.add_slots = int(os.environ.get('CASE_ADD_SLOTS', 2 * 148))
        self.xns = torch.zeros(B, dtype=torch.int32, device=dev)
        self._mv_src = [None, None]
        # copy plan of the batch (sparse tail from a sorted unique-id list instead of the hash table: no atomics, so
        # bit-reproducible copy mass).  Opt-in (CASE_COPY_PLAN=1): measured neutral per step at C2 (0.3387 against
        # 0.3380 ms) and +0.25 ms of prefill for the sort
        St = S0 + S1
        self.use_plan = St < 65536 and os.environ.get('CASE_COPY_PLAN', '0') == '1'
        if self.use_plan:
            i32z = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
            self.cp_n = i32z(B)
            self.cp_uid, self.cp_first, self.cp_start, self.cp_perm = (i32z(B, St + 1) for _ in range(4))
        if self.prop_split:
            self.nsa[1] = L.MAX_SPLIT
        self.x_in, self.h, self.bbuf, self.q2 = z(R, H), z(R, H), z(R, H), z(R, H)
        self.part_ml, self.part_acc = z(R, L.NH, nsx, 2), z(R, L.NH, nsx, L.HD)
        self.qa = z(R, H)
        self.attn_un = [z(R, s) for s in self.S]
        self.stats = [z(R, n, 4) for n in self.nsa]
        self.ctxp = [z(R, n, H) for n in self.nsa]
        self.hN, self.ctx = z(R, H), [z(R, H), z(R, H)]
        self.gates, self.fac, self.gfeat = z(R, 4), z(R, 2, L.MAX_SPLIT), z(R, H)
        self.logits, self.dist = z(R, self.ldv), z(R, self.ldv)
        self.top_vals = z(R, W)
        self.top_idx = torch.zeros(R, W, dtype=torch.int32, device=dev)
        self.prow = torch.zeros(R, Tmax, dtype=torch.int32, device=dev)
        self.h0, self.qa1 = z(R, H), z(R, H)
        self.base_ms, self.base_e = z(R, 4, 2), z(R, 4, 16)
        self.base_i = torch.zeros(R, 4, 16, dtype=torch.int32, device=dev)
        self._graphs = {}
        self._step_fn = L.load().case_decode_step
        self._step_name = 'case_decode_step'
        self._fork = _Fork(dev)               # side stream + events of this engine's fork/join (per engine, per device)
        self._fill_args()

    def _fill_args(self):
        a = self.args = L.StepBanArgs()
        a.no_repeat_ngram, a.min_len = self.constraints
        if self.bans is not None:
            self.bans.bind(a)
        w = self.w
        a.opt, a.fork = self.opt, self._fork.h
        if self.n_oov:
            a.n_oov, a.tok_ext = self.n_oov, self.state.tok_ext.data_ptr()
        a.B, a.W, a.R, a.V, a.ldv, a.Tmax = self.B, self.W, self.R, self.V, self.ldv, self.Tmax
        a.dtype, a.fast_tanh, a.vocab_impl, a.mode = w.cdtype, self.fast_tanh, self.vocab_impl, L.MODE_MODULE_GREEDY
        for i in range(2):
            a.S[i], a.nsplit_x[i], a.nsplit_a[i] = self.S[i], self.nsx[i], self.nsa[i]
            a.Wqa_t[i], a.bqa[i], a.va[i] = w.Wqa_t[i].data_ptr(), w.bqa[i].data_ptr(), w.va[i].data_ptr()
            a.U[i], a.Mv[i] = self.U[i].data_ptr(), self.Mv[i].data_ptr()
            a.mask[i], a.prior[i] = self.mask[i].data_ptr(), self.prior[i].data_ptr()
            a.attn_un[i], a.stats[i], a.ctxp[i] = (self.attn_un[i].data_ptr(), self.stats[i].data_ptr(),
                                                   self.ctxp[i].data_ptr())
            a.ctx[i] = self.ctx[i].data_ptr()
            if self.Gv is not None:
                a.Gv[i] = self.Gv[i].data_ptr()
        a.map_off[0], a.map_off[1] = 0, self.S[0]
        a.max_len, a.BOS, a.EOS, a.UNK, a.PAD, a.materialize_only = self.Tmax, BOS, EOS, UNK, PAD, 0
        a.E, a.pe = w.E.data_ptr(), w.pe.data_ptr()
        for l in range(8):
            C.memmove(C.byref(a.layers[l]), C.byref(w.layers[l]), C.sizeof(L.LayerWeights))
            a.Kx[l], a.Vx[l] = self.Kx[l].data_ptr(), (self.Vx[l].data_ptr() if self.Vx[l] is not None else None)
            a.kcache[l], a.vcache[l] = self.kcache[l].data_ptr(), self.vcache[l].data_ptr()
        a.lnN_g, a.lnN_b = w.lnN_g.data_ptr(), w.lnN_b.data_ptr()
        wv = w.Wv_tc if self.vocab_impl == 1 else w.Wv
        a.Wg_t, a.bg, a.Wv, a.Wm, a.bm = (w.Wg_t.data_ptr(), w.bg.data_ptr(), wv.data_ptr(), w.Wm.data_ptr(),
                                          w.bm.data_ptr())
        a.vocab_ws = self.vocab_ws.data_ptr()
        a.feat = self.feat.data_ptr()
        a.map, a.map_ld = self.map.data_ptr(), self.map.size(1)
        if self.compact:
            a.xcount, a.xprefix, a.xslots = self.xcount.data_ptr(), self.xprefix.data_ptr(), self.xslots
            a.xidx, a.xorder = self.xidx.data_ptr(), self.xorder.data_ptr()
            if self.prop_split:
                a.xns = self.xns.data_ptr()
        a.qcount = self.qcount.data_ptr()
        if self.use_plan:
            a.cp_n, a.cp_uid, a.cp_first = self.cp_n.data_ptr(), self.cp_uid.data_ptr(), self.cp_first.data_ptr()
            a.cp_start, a.cp_perm, a.cp_ld = self.cp_start.data_ptr(), self.cp_perm.data_ptr(), self.cp_uid.size(1)
        if w.Wg_c is not None:
            a.Wqa_c[0], a.Wqa_c[1], a.Wg_c = w.Wqa_c[0].data_ptr(), w.Wqa_c[1].data_ptr(), w.Wg_c.data_ptr()
        self.state.bind(a)
        for n in ('x_in', 'h', 'bbuf', 'q2', 'part_ml', 'part_acc', 'qa', 'hN', 'gates', 'fac', 'gfeat', 'logits',
                  'dist', 'top_vals', 'top_idx', 'prow', 'h0', 'qa1', 'base_ms', 'base_e', 'base_i'):
            setattr(a, n, getattr(self, n).data_ptr())

    # ------------------------------------------------------------------ per batch
    @torch.no_grad()
    def prefill(self, *tensors):
        with _on_device(self.device):
            return self._prefill(*tensors)

    def _prefill(self, mem_q, mem_p, mask_q, mask_p, prior_q, prior_p, answer_rep, source_map):
        """Once per batch: flatten (Model.py:56-58), norm2(answer_rep) (:98), and everything the
        reference recomputes every step although it never changes - the cross-attention K/V
        projections of both memories for all 8 layers (TransformerDecoder.py:81) and Uk.mem
        (BilinearAttention.py:34)."""
        B, H, w, dev = self.B, L.H, self.w, self.device
        mems = [mem_q.reshape(B, -1, H), mem_p.reshape(B, -1, H)]
        masks = [mask_q.reshape(B, -1), mask_p.reshape(B, -1)]
        priors = [prior_q.reshape(B, -1), prior_p.reshape(B, -1)]
        stream = torch.cuda.current_stream(dev).cuda_stream
        ar = answer_rep.to(dev, torch.float32).contiguous()
        L.call('case_layernorm_rows', ar.data_ptr(), w.ln2_g.data_ptr(), w.ln2_b.data_ptr(), self.feat.data_ptr(),
               B, stream)
        for i in range(2):
            S = self.S[i]
            m = mems[i].to(dev, w.tdtype)         # bf16 storage: the prefill GEMMs run on bf16 tensor cores
            if m.size(1) != S:
                raise ValueError(f'memory {i} has {m.size(1)} positions, engine was built for {S}')
            flat = m.reshape(B * S, H).contiguous()
            fused = self.prefill_tc and w.cdtype == L.BF16      # own tcgen05 GEMM writes K|V tiles and U directly
            kv = None if fused else torch.addmm(w.kv_b[i], flat, w.kv_w[i])    # [B*S, 4*2*H]
            cidx = ncount = None
            if w.cdtype == L.BF16:        # one pass: GEMM rows -> swizzled bf16 K|V tiles of all 4 layers
                outs = (C.c_void_p * 4)(*[self.Kx[i * 4 + l].data_ptr() for l in range(4)])
                if i == 1 and self.compact:
                    # padding keys are dropped here, once: valid positions first (ascending), counts, tile prefix
                    valid = masks[i].to(dev).bool()
                    self.xidx.copy_(torch.argsort(~valid, dim=1, stable=True))
                    cnt = valid.sum(1)
                    self.xcount.copy_(cnt)
                    self.xprefix[1:].copy_(torch.cumsum((cnt + 63) // 64, 0))
                    self.xorder.copy_(torch.argsort(cnt, descending=True, stable=True))
                    if self.prop_split:     # keys per CTA: the launch fits add_slots CTAs, no query needs > MAX_SPLIT
                        L.call('case_split_plan', self.xcount.data_ptr(), B, max(self.add_slots - B // 2, 1), L.MAX_SPLIT,
                               self.xns.data_ptr(), stream)
                    # the additive attention visits valid keys only: padding scores are -inf once and for all
                    self.attn_un[i].masked_fill_(~valid.repeat_interleave(self.W, 0), float('-inf'))
                    cidx, ncount = self.xidx.data_ptr(), self.xcount.data_ptr()
                    if not fused:
                        L.call('case_pack_kv_tiles_gather', kv.data_ptr(), kv.size(1), B, S, cidx, ncount, 4, outs, stream)
                elif not fused:
                    L.call('case_pack_kv_tiles', kv.data_ptr(), L.BF16, kv.size(1), B, S, 4, outs, stream)
            else:
                kv = kv.view(B, S, 4, 2, L.NH, L.HD).permute(2, 3, 0, 4, 1, 5)     # [l][k/v][B][NH][S][HD]
                for l in range(4):
                    self.Kx[i * 4 + l].copy_(kv[l, 0])
                    self.Vx[i * 4 + l].copy_(kv[l, 1])
            lazy = self.Gv is not None and not (self.args.opt & L.OPT_NO_GATE)   # the search path reads G only
            if fused:       # K|V tiles of the 4 layers + U in one launch
                L.call('case_prefill_project_tc', flat.data_ptr(), w.Wpf[i].data_ptr(), w.pf_bias[i].data_ptr(), B, S,
                       cidx, ncount, 4, outs, self.U[i].data_ptr(), stream)
            else:
                torch.mm(flat, w.Uk_t[i], out=self.U[i].view(B * S, H))
            if not lazy:
                self.Mv[i].copy_(m)
                self._mv_src[i] = None
            else:                   # the search path reads G instead; the value rows are filled when the `generate` face asks
                self._mv_src[i] = m
                L.call('case_gate_project', flat.data_ptr(), w.Wm_g[i].data_ptr(), self.Gv[i].data_ptr(), B * S, stream)
            self.mask[i].copy_(masks[i].to(dev).to(torch.uint8))
            self.prior[i].copy_(priors[i].to(dev, torch.float32))
        self.map.copy_(source_map.to(dev).to(torch.int32))
        if self.use_plan:
            self._copy_plan(torch.cat([masks[0].to(dev), masks[1].to(dev)], 1).bool())

    def _copy_plan(self, valid):
        build_copy_plan(self.map, valid, self.V, self.cp_n, self.cp_uid, self.cp_first, self.cp_start, self.cp_perm)

    @torch.no_grad()
    def decode(self, max_len: int, mode: int = L.MODE_MODULE_GREEDY, use_graph: bool = True) -> torch.Tensor:
        """Run ``max_len`` steps; returns int64 tokens [B, max_len] (beam: trimmed to the longest answer)."""
        if max_len > self.Tmax:
            raise ValueError('max_len exceeds the engine Tmax')
        if mode != L.MODE_BEAM and self.W != 1:
            raise ValueError('greedy modes need an engine built with W == 1')
        self.launch(max_len, mode, use_graph)
        return self._finish_tokens(max_len, mode)

    @torch.no_grad()
    def launch(self, max_len: int, mode: int = L.MODE_MODULE_GREEDY, use_graph: bool = True) -> None:
        """Enqueue a whole decode on the current stream without any host synchronisation (the result is
        read later with ``_finish_tokens``); lets several engines decode concurrently on several streams."""
        if max_len > self.Tmax:
            raise ValueError('max_len exceeds the engine Tmax')
        self._check_launch_constraints(max_len, mode)
        self.args.mode, self.args.max_len, self.args.materialize_only = mode, max_len, 0
        self.ensure_graph(max_len, mode, use_graph)
        self.state.reset()
        if use_graph:
            self._graphs[(max_len, mode)].replay()
        else:
            self._run_steps(max_len)

    def ensure_graph(self, max_len, mode, use_graph=True):
        if use_graph and (max_len, mode) not in self._graphs:
            self.args.mode, self.args.max_len, self.args.materialize_only = mode, max_len, 0
            self.state.reset()
            self._capture(max_len, mode)

    @torch.no_grad()
    def step_distribution(self, t: int) -> torch.Tensor:
        """Protocol ``generate`` face: run step t up to the finished distribution and return a view
        [R, V] of it (no top-k / select); the caller drives tok/anc through ``state``."""
        if any(self.constraints):
            raise ValueError('no_repeat_ngram / min_len apply to the beam and greedy searches, not to the `generate` face')
        if self.bans is not None:
            raise ValueError('bad_words apply to the beam and greedy searches, not to the `generate` face')
        for i in range(2):
            if self._mv_src[i] is not None:
                self.Mv[i].copy_(self._mv_src[i].view_as(self.Mv[i]))
                self._mv_src[i] = None
        self.args.materialize_only = 1
        with _on_device(self.device):
            self._step(t, torch.cuda.current_stream(self.device).cuda_stream)
        self.args.materialize_only = 0
        return self.dist[:, :self.V + self.n_oov]

    def answer_tokens(self) -> int:
        st = self.state
        return int(st.best_len.view(st.B, -1)[:, 0].sum().item())      # entry 0 of an n-best list

    def kernel_launches_per_step(self) -> int:
        # (+1 in bench.py: the activation re-pack inside the vocabulary GEMM call)
        lib = L.load()
        tail = 2                       # vocab_base + sparse_tail (search bookkeeping fused into it)
        if self.w.cdtype == L.BF16 and self.Tmax <= lib.case_layer_chain_max_tmax() and not (self.args.opt & L.OPT_NO_CHAIN):
            # attention queries, norm1 and gen.0 ride on the cluster launches (post linears): no row_linear launches
            if self.S[0] <= lib.case_layer_chain_max_s0():
                # layer_stack (first stack + front 4) + 4 x cross + 4 x layer_chain + 2 x additive + vocab + tail
                return 1 + 4 + 4 + 2 + 1 + tail
            # 9 x layer_chain + 8 x cross + 2 x additive + vocab + tail
            return 9 + 8 + 2 + 1 + tail
        # embed + 8 x (front, cross, back) + 2 x (row_linear, additive) + norm1 + gen.0 + vocab + tail
        return 1 + 24 + 4 + 1 + 1 + 1 + tail


class GttpWeights:
    """Step-side GTTP weights (dec.*, gen.*; GTTP/Model.py:96-111, 8-9) laid out for the kernels."""

    def __init__(self, sd: Dict[str, torch.Tensor], device=None, dtype: str = 'bf16', prefix: str = ''):
        dev = _require_cuda(device)
        self.device, self.dtype_name = dev, dtype
        self.tdtype, self.cdtype = _storage(dtype)
        g = lambda k: sd[prefix + k].detach().to(dev, torch.float32)
        H = g('dec.gru.weight_hh_l0').size(1)
        if H != L.H or g('dec.embedding.weight').size(1) != L.H:
            raise ValueError(f'hidden and embedding size must be {L.H}')
        self.V = g('gen.linear.weight').size(0)
        mat = lambda w: pack_tiled(w, self.tdtype)
        self.E = g('dec.embedding.weight').contiguous()
        self.Wq_t = [mat(g(f'dec.{a}.linear_query.weight')) for a in ('src_attn', 'bg_attn')]
        self.bq = [g(f'dec.{a}.linear_query.bias').contiguous() for a in ('src_attn', 'bg_attn')]
        self.v = [g(f'dec.{a}.v.weight').reshape(-1).contiguous() for a in ('src_attn', 'bg_attn')]
        self.Uk_t = [g(f'dec.{a}.linear_key.weight').t().contiguous().to(self.tdtype) for a in ('src_attn', 'bg_attn')]  # [2H][H]
        self.Wih_t, self.bih = mat(g('dec.gru.weight_ih_l0')), g('dec.gru.bias_ih_l0').contiguous()
        self.Whh_t, self.bhh = mat(g('dec.gru.weight_hh_l0')), g('dec.gru.bias_hh_l0').contiguous()
        self.Wr_t, self.br = mat(g('dec.readout.weight')), g('dec.readout.bias').contiguous()
        self.Wv, self.bv = g('gen.linear.weight').contiguous().to(self.tdtype), g('gen.linear.bias').contiguous()
        self.Wv_tc = pack_vocab_tc(g('gen.linear.weight')) if self.cdtype == L.BF16 else None
        self.wc = g('gen.linear_copy.weight').reshape(-1).contiguous()
        self.bc = g('gen.linear_copy.bias').reshape(-1).contiguous()


class GttpDecodeEngine(_EngineBase):
    def __init__(self, weights: GttpWeights, B: int, W: int, Lc: int, Lb: int, Tmax: int = 40,
                 fast_tanh: Optional[bool] = None, vocab_impl: Optional[int] = None, target_ctas: int = 296,
                 opt: int = 0, nbest: int = 1, attribution: bool = False, no_repeat_ngram: int = 0, min_len: int = 0,
                 bans: bool = False):
        if not (1 <= W <= L.MAX_W):
            raise ValueError(f'beam width must be 1..{L.MAX_W}')
        if attribution:
            check_attribution(int(opt), weights.V, W, Lb)
        check_constraints(int(opt), weights.V, W, Lb, Tmax, no_repeat_ngram, min_len)
        self.constraints = (int(no_repeat_ngram), int(min_len))
        if bans:
            _check_bans_servable(int(opt), weights.V, W, Lb, Tmax)
        self.bans = _BanBuffers(weights.device, weights.V) if bans else None
        self.nparts = 2
        self.w = weights
        self.device = dev = weights.device
        self.B, self.W, self.R, self.Lc, self.Lb, self.Tmax, self.V = B, W, B * W, Lc, Lb, Tmax, weights.V
        R, V, H = self.R, self.V, L.H
        self.ldv = -(-V // 8) * 8
        td = weights.tdtype
        self.fast_tanh = int(weights.cdtype == L.BF16 if fast_tanh is None else fast_tanh)
        self.vocab_impl = int((1 if weights.cdtype == L.BF16 else 0) if vocab_impl is None else vocab_impl)
        if self.vocab_impl == 1 and weights.cdtype != L.BF16:
            raise ValueError('the tcgen05 vocabulary GEMM needs bf16 storage')
        self.vocab_ws = torch.zeros(max(16, L.load().case_vocab_tc_workspace_bytes(self.R)), dtype=torch.uint8,
                                    device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        z = lambda *s: torch.zeros(*s, **f32)
        self.ns = [_nsplit_additive(B, s, weights.cdtype == L.BF16, target_ctas) for s in (Lc, Lb)]
        self.U = [torch.zeros(B, s, H, dtype=td, device=dev) for s in (Lc, Lb)]
        self.Mv = [torch.zeros(B, s, 2 * H, dtype=td, device=dev) for s in (Lc, Lb)]
        self.mask = [torch.zeros(B, s, dtype=torch.uint8, device=dev) for s in (Lc, Lb)]
        self.map = torch.zeros(B, Lb, dtype=torch.int32, device=dev)
        self.gstate = [z(R, H), z(R, H)]
        self.state = _SearchState(dev, B, W, Tmax, nbest=nbest, attribution=attribution)
        self.emb, self.qa = z(R, H), z(R, H)
        self.attn_un = [z(R, Lc), z(R, Lb)]
        self.stats = [z(R, n, 4) for n in self.ns]
        self.ctxp = [z(R, n, 2 * H) for n in self.ns]
        self.ctx = [z(R, 2 * H), z(R, 2 * H)]
        self.gi, self.gh, self.feat = z(R, 3 * H), z(R, 3 * H), z(R, H)
        self.gates, self.fac = z(R, 4), z(R, L.MAX_SPLIT)
        self.logits, self.dist = z(R, self.ldv), z(R, self.ldv)
        self.top_vals = z(R, W)
        self.top_idx = torch.zeros(R, W, dtype=torch.int32, device=dev)
        self.qa1 = z(R, H)                                            # query of the context attention when it runs on the side stream
        self._fork = _Fork(dev)
        self.base_ms, self.base_e = z(R, 4, 2), z(R, 4, 16)          # case_vocab_base statistics (sparse tail)
        self.base_i = torch.zeros(R, 4, 16, dtype=torch.int32, device=dev)
        self._graphs = {}
        self._step_fn = L.load().gttp_decode_step
        self._step_name = 'gttp_decode_step'
        a = self.args = L.GttpStepBanArgs()
        a.no_repeat_ngram, a.min_len = self.constraints
        if self.bans is not None:
            self.bans.bind(a)
        w = weights
        a.B, a.W, a.R, a.V, a.ldv, a.dtype = B, W, R, V, self.ldv, w.cdtype
        a.opt = int(opt)
        a.fast_tanh, a.vocab_impl, a.mode = self.fast_tanh, self.vocab_impl, L.MODE_PROTO_GREEDY
        a.Lc, a.Lb, a.nsplit_c, a.nsplit_b = Lc, Lb, self.ns[0], self.ns[1]
        a.max_len, a.BOS, a.EOS, a.UNK, a.PAD, a.materialize_only, a.Tmax = Tmax, BOS, EOS, UNK, PAD, 0, Tmax
        a.E = w.E.data_ptr()
        a.Wqs_t, a.bqs, a.vs = w.Wq_t[0].data_ptr(), w.bq[0].data_ptr(), w.v[0].data_ptr()
        a.Wqb_t, a.bqb, a.vb = w.Wq_t[1].data_ptr(), w.bq[1].data_ptr(), w.v[1].data_ptr()
        a.Wih_t, a.bih, a.Whh_t, a.bhh = w.Wih_t.data_ptr(), w.bih.data_ptr(), w.Whh_t.data_ptr(), w.bhh.data_ptr()
        a.Wr_t, a.br = w.Wr_t.data_ptr(), w.br.data_ptr()
        wv = w.Wv_tc if self.vocab_impl == 1 else w.Wv
        a.Wv, a.bv, a.wc, a.bc = wv.data_ptr(), w.bv.data_ptr(), w.wc.data_ptr(), w.bc.data_ptr()
        a.vocab_ws = self.vocab_ws.data_ptr()
        a.Us, a.Ms, a.Ub, a.Mb = self.U[0].data_ptr(), self.Mv[0].data_ptr(), self.U[1].data_ptr(), self.Mv[1].data_ptr()
        a.mask_c, a.mask_b = self.mask[0].data_ptr(), self.mask[1].data_ptr()
        a.map, a.map_ld = self.map.data_ptr(), Lb
        a.state[0], a.state[1] = self.gstate[0].data_ptr(), self.gstate[1].data_ptr()
        self.state.bind(a)
        for i in range(2):
            a.attn_un[i], a.stats[i], a.ctxp[i], a.ctx[i] = (self.attn_un[i].data_ptr(), self.stats[i].data_ptr(),
                                                             self.ctxp[i].data_ptr(), self.ctx[i].data_ptr())
        a.fork = self._fork.h
        for n in ('emb', 'qa', 'qa1', 'gi', 'gh', 'feat', 'gates', 'fac', 'logits', 'dist', 'top_vals', 'top_idx', 'base_ms', 'base_e',
                  'base_i'):
            setattr(a, n, getattr(self, n).data_ptr())

    @torch.no_grad()
    def prefill(self, src_output, bg_output, context, background, background_map, init_state):
        """Once per batch: Uk.memory for both attentions (BilinearAttention.py:34), value copies,
        masks (GTTP/Model.py:177-178) and the initial GRU state (:170-174), replicated per beam slot."""
        B, H, w, dev = self.B, L.H, self.w, self.device
        for i, (m, ids) in enumerate(((src_output, context), (bg_output, background))):
            m = m.to(dev, w.tdtype)
            S = m.size(1)
            torch.mm(m.reshape(B * S, 2 * H), w.Uk_t[i], out=self.U[i].view(B * S, H))
            self.Mv[i].copy_(m)
            self.mask[i].copy_(ids.to(dev).ne(0).to(torch.uint8))
        self.map.copy_(background_map.to(dev).to(torch.int32))
        st = init_state.to(dev, torch.float32).reshape(B, 1, H).expand(B, self.W, H).reshape(self.R, H)
        self._init_state = st.contiguous()

    @torch.no_grad()
    def decode(self, max_len: int, mode: int = L.MODE_PROTO_GREEDY, use_graph: bool = True) -> torch.Tensor:
        self.launch(max_len, mode, use_graph)
        return self._finish_tokens(max_len, mode)

    @torch.no_grad()
    def launch(self, max_len: int, mode: int = L.MODE_PROTO_GREEDY, use_graph: bool = True) -> None:
        """Enqueue a whole decode on the current stream without any host synchronisation (see CaseDecodeEngine.launch)."""
        if max_len > self.Tmax:
            raise ValueError('max_len exceeds the engine Tmax')
        if mode != L.MODE_BEAM and self.W != 1:
            raise ValueError('greedy modes need an engine built with W == 1')
        self._check_launch_constraints(max_len, mode)
        self.args.mode, self.args.max_len, self.args.materialize_only = mode, max_len, 0
        self._reset()
        if use_graph and (max_len, mode) not in self._graphs:
            self._capture(max_len, mode)
            self._reset()
        if use_graph:
            self._graphs[(max_len, mode)].replay()
        else:
            self._run_steps(max_len)

    def _reset(self):
        self.state.reset()
        self.gstate[0].copy_(self._init_state)
        self.gstate[1].zero_()

    def kernel_launches_per_step(self) -> int:
        # embed, 2 x (query linear, additive, merge), gi, gh, gru, readout, vocab, gates, vocab_base + sparse_tail (or the
        # dense row_tail), select
        sparse = not (self.args.opt & (L.OPT_DENSE_TAIL | L.OPT_UNFUSED_TAIL)) and self.Lb <= L.load().case_sparse_tail_max_sources()
        return 1 + 2 * 3 + 3 + 1 + 1 + 1 + (2 if sparse else 1) + 1
