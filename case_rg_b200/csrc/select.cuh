// Search bookkeeping on the device: greedy token hand-off and the beam step of
// common/Generations.py:136-185, with no host round trips (shared by the standalone kernel of select.cu
// and the fused form at the end of sparse_tail.cu).
#pragma once
#include "common.cuh"

namespace cb {

// The n-best list (case_select_args_t.nbest) holds at most W <= CASE_MAX_W entries and exists in beam mode only; every
// launcher that can run the select checks it before its first launch.
static inline int check_nbest(int nbest, int W, int mode) {
  CB_REQUIRE(nbest >= 0 && nbest <= W && nbest <= CASE_MAX_W, "nbest out of range: 0 <= nbest <= W <= CASE_MAX_W");
  CB_REQUIRE(nbest <= 1 || mode == CASE_MODE_BEAM, "nbest > 1 needs CASE_MODE_BEAM");
  return 0;
}

// Attribution (case_select_args_t.attr_*) is all three pointers or none; the caller picks the instance of the select
static inline int check_attr_select(const case_select_args_t& a) {
  const int n = (a.attr_cand != nullptr) + (a.attr_hist != nullptr) + (a.out_attr != nullptr);
  CB_REQUIRE(n == 0 || n == 3, "attribution needs attr_cand, attr_hist and out_attr (or none of them)");
  return 0;
}

__device__ __forceinline__ case_attr_t attr_zero() {
  case_attr_t z;
  z.part[0] = z.part[1] = z.part[2] = 0.f;
  z.source = -1;
  return z;
}

// a record written by another CTA of the same launch (fused form): L2 load, as top_vals
__device__ __forceinline__ case_attr_t attr_ldcg(const case_attr_t* p) {
  const float4 v = __ldcg(reinterpret_cast<const float4*>(p));
  case_attr_t r;
  r.part[0] = v.x; r.part[1] = v.y; r.part[2] = v.z; r.source = __float_as_int(v.w);
  return r;
}

// One warp runs the bookkeeping of query b (all 32 lanes must call).  top_vals / top_idx may have been
// written by other CTAs of the same launch (fused form: the last CTA of the query's W rows calls this
// after a fence + atomic), hence the L2 (.cg) loads.  ATTR: the attribution records (case_select_args_t.attr_*) travel
// with the tokens - candidate c of the query is attr_cand[r0 * W + c], kept children write attr_hist next to tok, the
// finished rows copy it along the anc path like out_tokens.
template <bool ATTR = false>
__device__ __forceinline__ void beam_select_query(const case_select_args_t& a, int b, int lane) {
  const int W = a.W, t = a.t, TL = a.Tmax + 1;
  const int r0 = b * W;
  // extended vocabulary: ids >= V_in are dynamic (OOV) entries - the decoder is fed UNK, tok_ext keeps the id
  const bool ext = a.V_in > 0 && a.tok_ext != nullptr;
  int32_t* tok_o = ext ? a.tok_ext : a.tok;
  auto feed = [&](int id) { return (ext && id >= a.V_in) ? a.UNK : id; };

  if (a.mode != CASE_MODE_BEAM) {   // W == 1
    if (lane == 0) {
      int tk = __ldcg(a.top_idx + r0);
      bool padded = false;
      if (a.mode == CASE_MODE_PROTO_GREEDY) {
        const int was_ended = a.ended[b];
        const int this_end = tk == a.EOS;
        if (t == 0) { if (this_end) tk = a.UNK; }          // Generations.py:99-100
        else if (was_ended) { tk = a.PAD; padded = true; } // Generations.py:101-102
        a.ended[b] = was_ended | this_end;
      }
      a.out_tokens[(size_t)b * a.Tmax + t] = tk;
      // the record of the id the distribution chose (an EOS rewritten to UNK keeps it); PAD after the end: zero record
      if constexpr (ATTR) a.out_attr[(size_t)b * a.Tmax + t] = padded ? attr_zero() : attr_ldcg(a.attr_cand + r0);
      a.tok[(size_t)r0 * TL + t + 1] = feed(tk);
      if (ext) tok_o[(size_t)r0 * TL + t + 1] = tk;
      a.parent[r0] = r0;
      a.live[r0] = 1;
      a.n_live[b] = 1;
    }
    for (int j = lane; j <= t; j += 32) a.anc_out[(size_t)r0 * TL + j] = r0;
    return;
  }

  // n-best list of the query, in rank order: keys bkey, lengths blen, token rows out[i] ([nb][Tmax])
  const int nb = a.nbest > 1 ? a.nbest : 1;
  double* bkey = a.best_key + (size_t)b * nb;
  int32_t* blen = a.best_len + (size_t)b * nb;
  int* out = a.out_tokens + (size_t)b * nb * a.Tmax;
  __shared__ double key[64], ccum[64], s_bkey[CASE_MAX_W];
  __shared__ int ctok[64], cpar[64], clen[64], order[CASE_MAX_W], dst[CASE_MAX_W], ins[CASE_MAX_W], s_blen[CASE_MAX_W];
  __shared__ int s_nlive;
  if (lane < nb) { s_bkey[lane] = bkey[lane]; s_blen[lane] = blen[lane]; }
  int nl = 0;
  for (int w = 0; w < W; ++w) nl += a.live[r0 + w] != 0;
  const int ncand = nl * W;
  for (int c = lane; c < ncand; c += 32) {
    const int w = c / W, j = c % W, r = r0 + w;
    const double p = (double)__ldcg(a.top_vals + (size_t)r * W + j);
    const double cm = a.cum[r] + (-log(p + 1e-10));         // Generations.py:170, Node.cum_cost :198
    const int ln = a.length[r] + 1;                         // Node.length :199
    key[c] = cm / (double)ln;
    ccum[c] = cm;
    ctok[c] = __ldcg(a.top_idx + (size_t)r * W + j);
    cpar[c] = r;
    clen[c] = ln;
  }
  __syncwarp();
  // stable ascending rank (sorted(..., key=cum_cost/length)[:width], Generations.py:180)
  for (int c = lane; c < ncand; c += 32) {
    const double k = key[c];
    int rank = 0;
    for (int o = 0; o < ncand; ++o) rank += (key[o] < k) || (key[o] == k && o < c);
    if (rank < W) order[rank] = c;
  }
  __syncwarp();
  const int nsel = min(W, ncand);
  if (lane == 0) {
    int nn = 0;
    for (int k = 0; k < nsel; ++k) {
      const int c = order[k];
      const bool fin = (ctok[c] == a.EOS) || (t == a.max_len - 1);   // Generations.py:139
      ins[k] = -1;
      if (fin) {
        // stable sort of the finished list (:183-185): after every entry whose key is <= this one, so equal keys stay
        // in finishing order; a position >= nb drops it (nb = 1: the first finisher wins ties)
        int pos = 0;
        while (pos < nb && s_bkey[pos] <= key[c]) ++pos;
        if (pos < nb) {
          for (int i = nb - 1; i > pos; --i) { s_bkey[i] = s_bkey[i - 1]; s_blen[i] = s_blen[i - 1]; }
          s_bkey[pos] = key[c];
          s_blen[pos] = t + 1;
          ins[k] = pos;
        }
        dst[k] = -1;
      } else {
        dst[k] = nn++;
      }
    }
    s_nlive = nn;
    a.n_live[b] = nn;
  }
  __syncwarp();
  if (lane < nb) { bkey[lane] = s_bkey[lane]; blen[lane] = s_blen[lane]; }
  // read everything the new slots need from the old state before any slot is overwritten
  // (anc is double-buffered; cum/length/live were staged in shared memory above)
  for (int k = 0; k < nsel; ++k) {
    if (dst[k] < 0) continue;
    const int c = order[k], rn = r0 + dst[k], pr = cpar[c];
    for (int j = lane; j < t; j += 32) a.anc_out[(size_t)rn * TL + j] = a.anc_in[(size_t)pr * TL + j];
    if (lane == 0) {
      a.anc_out[(size_t)rn * TL + t] = pr;
      a.tok[(size_t)rn * TL + t + 1] = feed(ctok[c]);
      if (ext) tok_o[(size_t)rn * TL + t + 1] = ctok[c];
      a.cum[rn] = ccum[c];
      a.length[rn] = clen[c];
      a.live[rn] = 1;
      a.parent[rn] = pr;
      if constexpr (ATTR) a.attr_hist[(size_t)rn * TL + t + 1] = attr_ldcg(a.attr_cand + (size_t)r0 * W + c);
    }
  }
  for (int w = s_nlive + lane; w < W; w += 32) {     // dead slots: harmless, in-range contents
    const int rn = r0 + w;
    a.live[rn] = 0;
    a.parent[rn] = rn;
    a.tok[(size_t)rn * TL + t + 1] = a.PAD;
    if (ext) tok_o[(size_t)rn * TL + t + 1] = a.PAD;
    if constexpr (ATTR) a.attr_hist[(size_t)rn * TL + t + 1] = attr_zero();
    for (int j = 0; j <= t; ++j) a.anc_out[(size_t)rn * TL + j] = rn;
  }
  // record the inserted finished sequences in insertion order: BOS dropped, EOS kept (:188).  Lane j owns column j of
  // every row, so the shift of the lower rows and the new row need no synchronisation between insertions.
  for (int k = 0; k < nsel; ++k) {
    const int pos = ins[k];
    if (pos < 0) continue;
    const int c = order[k], pr = cpar[c];
    for (int j = lane; j < a.max_len; j += 32) {
      for (int i = nb - 1; i > pos; --i) out[(size_t)i * a.Tmax + j] = out[(size_t)(i - 1) * a.Tmax + j];
      int v = a.PAD;
      if (j < t) {
        const int src = (j + 1 == t) ? pr : a.anc_in[(size_t)pr * TL + j + 1];
        v = tok_o[(size_t)src * TL + j + 1];
      } else if (j == t) {
        v = ctok[c];
      }
      out[(size_t)pos * a.Tmax + j] = v;
      if constexpr (ATTR) {                              // the records ride the same path
        case_attr_t* oa = a.out_attr + (size_t)b * nb * a.Tmax;
        for (int i = nb - 1; i > pos; --i) oa[(size_t)i * a.Tmax + j] = oa[(size_t)(i - 1) * a.Tmax + j];
        case_attr_t e = attr_zero();
        if (j < t) {
          const int src = (j + 1 == t) ? pr : a.anc_in[(size_t)pr * TL + j + 1];
          e = a.attr_hist[(size_t)src * TL + j + 1];
        } else if (j == t) {
          e = attr_ldcg(a.attr_cand + (size_t)r0 * W + c);
        }
        oa[(size_t)pos * a.Tmax + j] = e;
      }
    }
  }
}

}  // namespace cb
