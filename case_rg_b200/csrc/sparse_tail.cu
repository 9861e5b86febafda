// Sparse form of the vocabulary tail for the search path (the [R, V] mixture is never built).
//
//   dist[r, v] = g0[r] * softmax(logits[r])[v] + sum over source positions s with map[b, s] == v of
//                gate_i[r] * p_i[r, s]                          (Model.py:34-43, Utils.build_map)
//   followed by top-k per row                                   (Utils.topk, Utils.py:156-168)
//
// Every id of the final top-k is either one of the (at most S0 + S1) copy targets of the row or one of
// the top-k ids of the base softmax: an id that receives no copy mass keeps the order it has in the
// base distribution.  So the step splits into
//   case_vocab_base  - per row: max, sum of exp and the 2k largest base entries (k extra entries
//                      absorb ties created when the gate scale rounds two neighbouring values onto
//                      one float).  Needs only the logits, so it runs beside the additive attention;
//   case_sparse_tail - after the attentions: [CaSE gates] -> a shared-memory hash table keyed by
//                      vocabulary id accumulates the copy mass of both memories -> every touched id
//                      gets g0 * exp(logit - max) / sum + mass (one gather from the logits) -> top-k
//                      over touched ids + base candidates.
// Work after the attentions drops from three passes over the 31 MB tile to ~2.7 k entries per row.
#include <string.h>

#include "common.cuh"
#include "topk.cuh"
#include "select.cuh"

namespace cb {

constexpr int ST = 256;          // vocab_base threads
constexpr int SW = ST / 32;
constexpr int TS = 512;          // sparse_tail threads
constexpr int TSW = TS / 32;

// ------------------------------------------------------------------------------------------ base statistics
// grid = R x SP_PARTS: CTA (r, c) reduces the quarter [c*Vq, (c+1)*Vq) of row r in ONE read, with all of a
// thread's 16-byte loads of a batch in flight together: local (max, sum exp(l - max)) and the k2 largest
// logits of the quarter (value desc, index asc).  The consumer merges the four partials.
constexpr int SP_PARTS = 4;
constexpr int SP_BATCH = 8;      // float4 loads in flight per thread

// fast exp for the softmax terms: one ex2.approx (results below 2^-126 flush to zero, which no top-k sees)
__device__ __forceinline__ float sp_exp(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}

__device__ __forceinline__ float4 vb_load(const float* x, int q, int nf4, int nv, bool mask0) {
  float4 v = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  if (q < nf4) {
    v = *reinterpret_cast<const float4*>(x + q * 4);
    const int i = q * 4;
    if (i + 3 >= nv) {                                   // tail chunk: slots past the quarter do not exist
      if (i + 1 >= nv) v.y = -INFINITY;
      if (i + 2 >= nv) v.z = -INFINITY;
      if (i + 3 >= nv) v.w = -INFINITY;
    }
    if (mask0 && q == 0) v.x = -INFINITY;
  }
  return v;
}

__global__ __launch_bounds__(ST) void vocab_base_kernel(const float* __restrict__ logits, int ldl, int V, int Vq,
                                                        int mask_col0, int k2, float* __restrict__ base_ms,
                                                        float* __restrict__ base_l, int32_t* __restrict__ base_i) {
  __shared__ float shm[SW], shs[SW];
  __shared__ TopKScratch<SW, 256> sc;
  pdl_wait();
  const int r = blockIdx.x / SP_PARTS, c = blockIdx.x % SP_PARTS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int v0 = c * Vq, nv = max(0, min(V, v0 + Vq) - v0);
  const float* x = logits + (size_t)r * ldl + v0;       // 16-byte aligned: Vq % 4 == 0
  const int nf4 = (nv + 3) / 4;                          // the row is padded to a multiple of 4 (ldl)
  const bool mask0 = mask_col0 && c == 0;
  // ---- pass A: per-thread max and sum of exp (online), all loads of a batch in flight together
  float m = -INFINITY, s = 0.f;
  for (int base = 0; base < nf4; base += SP_BATCH * ST) {
    float4 v[SP_BATCH];
#pragma unroll
    for (int u = 0; u < SP_BATCH; ++u) v[u] = vb_load(x, base + u * ST + tid, nf4, nv, mask0);
    float bm = -INFINITY;
#pragma unroll
    for (int u = 0; u < SP_BATCH; ++u) bm = fmaxf(bm, fmaxf(fmaxf(v[u].x, v[u].y), fmaxf(v[u].z, v[u].w)));
    if (bm > m) { s *= sp_exp(m - bm); m = bm; }         // m = -inf: s was 0 and exp(-inf) = 0
    const float mm = (m > -INFINITY) ? m : 0.f;
#pragma unroll
    for (int u = 0; u < SP_BATCH; ++u)
      s += (sp_exp(v[u].x - mm) + sp_exp(v[u].y - mm)) + (sp_exp(v[u].z - mm) + sp_exp(v[u].w - mm));
  }
  {
    const float Mw = warp_max(m);
    float sw = (m > -INFINITY) ? s * sp_exp(m - Mw) : 0.f;
    sw = warp_sum(sw);
    if (lane == 0) { shm[warp] = Mw; shs[warp] = sw; }
  }
  // ---- the k2-th largest thread maximum bounds the top-k2 from below; collect everything >= it
  const float T = block_kth_max(sc, k2, m);
  if (tid == 0) {
    float MM = shm[0];
#pragma unroll
    for (int w = 1; w < SW; ++w) MM = fmaxf(MM, shm[w]);
    float t2 = 0.f;
#pragma unroll
    for (int w = 0; w < SW; ++w) t2 += (shm[w] > -INFINITY) ? shs[w] * sp_exp(shm[w] - MM) : 0.f;
    base_ms[((size_t)r * SP_PARTS + c) * 2] = MM;
    base_ms[((size_t)r * SP_PARTS + c) * 2 + 1] = t2;
  }
  if (m >= T && m > -INFINITY) {                        // only threads that own a candidate look again
    for (int q = tid; q < nf4; q += ST) {
      const float4 v = vb_load(x, q, nf4, nv, mask0);
      const int i = v0 + q * 4;
      if (v.x >= T) topk_append(sc, v.x, i);
      if (v.y >= T) topk_append(sc, v.y, i + 1);
      if (v.z >= T) topk_append(sc, v.z, i + 2);
      if (v.w >= T) topk_append(sc, v.w, i + 3);
    }
  }
  __syncthreads();
  float ov = -INFINITY;
  int oi = 0x7fffffff;
  if (!block_select(sc, k2, ov, oi)) {                   // massive ties: offer every element
    WarpTopK wl;
    wl.init();
    for (int q0 = 0; q0 < nf4; q0 += ST) {
      const int q = q0 + tid;
      const float4 v = vb_load(x, q, nf4, nv, mask0);
      const int i = v0 + q * 4;
      wl.offer(k2, v.x, i); wl.offer(k2, v.y, i + 1); wl.offer(k2, v.z, i + 2); wl.offer(k2, v.w, i + 3);
    }
    block_merge_lists(sc, wl, k2);
    ov = wl.ev; oi = wl.ei;
  }
  if (warp == 0 && lane < k2) {
    base_l[((size_t)r * SP_PARTS + c) * k2 + lane] = ov;
    base_i[((size_t)r * SP_PARTS + c) * k2 + lane] = oi;
  }
}

// ------------------------------------------------------------------------------------------ sparse tail
// double hashing over a power-of-two table: start = high bits of a multiplicative hash, odd step
__device__ __forceinline__ uint32_t sp_hash(int id, int shift) { return ((uint32_t)id * 2654435761u) >> shift; }
__device__ __forceinline__ uint32_t sp_step(int id) { return (((uint32_t)id * 40503u) >> 4) | 1u; }

// slot of id in the row's touched-id table, -1 if untouched: binary search of the sorted list (plan mode) or the probe
// sequence of the hash table
__device__ __forceinline__ int sp_find(const int* hkeys, int nent, bool plan, int id, int hshift, uint32_t hmask) {
  if (plan) {
    int lo = 0, hi = nent;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (hkeys[mid] < id) lo = mid + 1; else hi = mid;
    }
    return lo < nent && hkeys[lo] == id ? lo : -1;
  }
  uint32_t slot = sp_hash(id, hshift);
  const uint32_t step = sp_step(id);
  while (true) {
    const int key = hkeys[slot];
    if (key == id) return (int)slot;
    if (key == -1) return -1;
    slot = (slot + step) & hmask;
  }
}

// Constrained launches (case_tail_args_t.no_repeat_ngram / min_len / ban_*) append these int arrays to the dynamic shared
// memory, after the table: the row's answer so far, the ban candidates (t n-gram continuations, the EOS of min_len, one
// per banned sequence; -1 = none), the banned ids (the distinct candidates, compacted), the row's base entries and the
// length of the banned list
constexpr int CS_NCAND = CASE_MAX_T + 1 + CASE_MAX_BAN_SEQ;
constexpr int CS_HIST = 0, CS_CAND = CS_HIST + CASE_MAX_T, CS_BAN = CS_CAND + CS_NCAND, CS_BASE = CS_BAN + CS_NCAND,
              CS_NBAN = CS_BASE + 2 * SP_PARTS * 2 * CASE_MAX_W, CS_INTS = CS_NBAN + 1;
static_assert(CS_NCAND <= TS, "one ban candidate per thread");

__device__ __forceinline__ bool sp_banned(const int* ban, int nban, int id) {
  bool hit = false;
  for (int i = 0; i < nban; ++i) hit |= ban[i] == id;
  return hit;
}

// single-id bans (case_tail_args_t.ban_mask, NULL = none): bit id of the mask, read through L1 (the few words a row
// tests are shared by every row of the step, so they stay cached; no shared-memory staging per CTA)
__device__ __forceinline__ bool sp_masked(const uint32_t* mask, int id, int V) {
  return mask != nullptr && (unsigned)id < (unsigned)V && ((__ldg(mask + (id >> 5)) >> (id & 31)) & 1u);
}

// ATTR (case_tail_args_t.attr != NULL): after the top-k, an attribution pass writes the record of every winner (see
// below); the fused select then carries the records with the tokens.
// CONSTR (no_repeat_ngram or min_len set): the row's banned ids leave the candidate set.  A banned touched id is looked
// up once and its value set to -inf; a banned base entry is not offered.  Exactness: an untouched id enters the top-K
// through the base entries only, and the unconstrained argument needs 2K of them (K for the result, K of slack for the
// ties of the gate scale's rounding).  A banned base entry uses up one of them, so with a = the allowed ids among the
// row's global top-k2 base entries the row keeps the usual path while a >= 2K and otherwise takes an exact pass over
// all V logits (offering every allowed untouched id; fbcount counts these rows).  Banned words (ban_*) run in the same
// instance: a banned sequence whose first L - 1 tokens end the answer adds its last token to the banned list, and the
// single-id mask is tested wherever the list is (touched ids, base entries, the exact pass).
template <bool ATTR, bool CONSTR>
__global__ __launch_bounds__(TS) void sparse_tail_kernel(const case_tail_args_t a, const float* __restrict__ base_ms,
                                                         const float* __restrict__ base_e,
                                                         const int32_t* __restrict__ base_i, int k2, int nslots,
                                                         long long* dbg, const case_select_args_t sel, int do_select,
                                                         int32_t* __restrict__ qcount, int* fbcount) {
  // [nslots] ids (-1 = empty), then [nslots] low words of the masses (later: the final float values), then - hash
  // mode only - [nslots] high words.  The copy mass of an id is accumulated as a 64-bit FIXED-POINT integer (2^-48
  // units, two native 32-bit shared-memory atomics with an explicit carry): integer addition is associative, so the
  // mass - and with it every top-k value, cost and token - is bit-identical from run to run whatever order the
  // threads arrive in, and it is the exactly rounded sum of the fp32 contributions.
  extern __shared__ __align__(16) int hkeys[];
  float* hvals = reinterpret_cast<float*>(hkeys + nslots);
  uint32_t* hlo = reinterpret_cast<uint32_t*>(hkeys + nslots);
  uint32_t* hhi = reinterpret_cast<uint32_t*>(hkeys + 2 * nslots);
  __shared__ float sh[TSW * 3];
  __shared__ TopKScratch<TSW, 256> sc;
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = r / a.W, V = a.V;
  const int Vx = a.Vext > V ? a.Vext : V;                  // extended vocabulary: ids in [V, Vx) are dynamic entries without a logit
  const uint32_t hmask = (uint32_t)nslots - 1;
  const int hshift = 32 - (31 - __clz(nslots));            // nslots is a power of two
  // plan mode (a.cp_n != NULL): the prefill sorted the valid source positions of the query by vocabulary id, so
  // the touched ids are a ready list (ascending, unique) with their positions - no hash table, no atomics, the
  // mass of a repeated id is summed in a fixed order, the logit gathers of neighbouring threads share lines.
  // hkeys / hvals then hold (id, final value) of the list entries, nent of them.
  const bool plan = a.cp_n != nullptr;
  const int nent = plan ? a.cp_n[b] : nslots;
  int dbg_n = 0;
  auto stamp = [&]() { if (dbg != nullptr && blockIdx.x == 0 && tid == 0) dbg[dbg_n++] = clock64(); };
  stamp();
  if (!plan)
    for (int i = tid; i < nslots; i += TS) { hkeys[i] = -1; hlo[i] = 0u; hhi[i] = 0u; }
  // weights of the mixture gate (the h part) are requested before the dependency wait
  float wmh[3] = {0.f, 0.f, 0.f}, bmv[3] = {0.f, 0.f, 0.f};
  if (a.do_finalize) {
    const int colw = tid < H ? tid : 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) { wmh[k] = __ldg(a.Wm + (size_t)k * 3 * H + colw); bmv[k] = __ldg(a.bm + k); }
  }
  pdl_wait();
  stamp();
  // constrained: the row's answer y_1 .. y_t, gathered along its ancestry like the select writes a finished path (the
  // previous step's select wrote it)
  int* const cs = hkeys + (plan ? 2 : 3) * nslots;
  if constexpr (CONSTR) {
    if (tid == 0) cs[CS_NBAN] = 0;
    for (int j = tid; j < a.t; j += TS) {
      const int p = j + 1;
      const int src = p == a.t ? r : a.hist_anc[(size_t)r * a.hist_ld + p];
      cs[CS_HIST + j] = a.hist_tok[(size_t)src * a.hist_ld + p];
    }
  }
  float g0, F[2] = {0.f, 0.f}, M[2] = {0.f, 0.f};
  if (a.do_finalize) {
    // every thread merges the split statistics itself (a few broadcast loads), column tid of the contexts
    int wn = 0;
    auto wstamp = [&]() { if (dbg != nullptr && blockIdx.x == 0 && lane == 0) dbg[32 + warp * 8 + wn++] = clock64(); };
    wstamp();
    const int col = tid < H ? tid : 0;                     // threads past H repeat column 0 and contribute nothing
    const float y = a.hN[(size_t)r * H + col];
    float Z[2], Q[2], cx[2] = {0.f, 0.f};
    float gsum[3] = {0.f, 0.f, 0.f};                       // gate form: W_m,i . m_i summed over both memories
    if (a.gate_ctx) {
      // gate form: one load round for everything - lane (half = memory, slot) fetches the statistics and the gate
      // partials of its slot, the merge is a segmented (16-lane) shuffle reduction (ns <= CASE_MAX_SPLIT = 16)
      const int half = lane >> 4, sl = lane & 15;
      const int nsh = half ? a.ns[1] : a.ns[0];
      const float4* stp = reinterpret_cast<const float4*>(half ? a.stats[1] : a.stats[0]);
      const float4* gpp = reinterpret_cast<const float4*>(half ? a.ctxp[1] : a.ctxp[0]);
      float4 sj = make_float4(-INFINITY, 0.f, 0.f, 0.f), gj = make_float4(0.f, 0.f, 0.f, 0.f);
      if (sl < nsh) {
        sj = __ldg(stp + (size_t)r * nsh + sl);
        gj = gpp[(size_t)r * nsh + sl];
      }
      float Mx = sj.x;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) Mx = fmaxf(Mx, __shfl_xor_sync(0xffffffffu, Mx, o));
      const float e = (sj.x == -INFINITY) ? 0.f : fexp(sj.x - Mx);
      float z = sj.y * e, q = sj.z * e, a0 = gj.x * e, a1 = gj.y * e, a2 = gj.z * e;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
        z += __shfl_xor_sync(0xffffffffu, z, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        a1 += __shfl_xor_sync(0xffffffffu, a1, o);
        a2 += __shfl_xor_sync(0xffffffffu, a2, o);
      }
      const float g0h = z > 0.f ? a0 / z : 0.f, g1h = z > 0.f ? a1 / z : 0.f, g2h = z > 0.f ? a2 / z : 0.f;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        M[i] = __shfl_sync(0xffffffffu, Mx, 16 * i);
        Z[i] = __shfl_sync(0xffffffffu, z, 16 * i);
        Q[i] = __shfl_sync(0xffffffffu, q, 16 * i);
        gsum[0] += __shfl_sync(0xffffffffu, g0h, 16 * i);
        gsum[1] += __shfl_sync(0xffffffffu, g1h, 16 * i);
        gsum[2] += __shfl_sync(0xffffffffu, g2h, 16 * i);
      }
      wstamp();
      wstamp();
    } else {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int ns = a.ns[i];
      const float4* st = reinterpret_cast<const float4*>(a.stats[i]) + (size_t)r * ns;
      float Mx = -INFINITY;
#pragma unroll 4
      for (int j = 0; j < ns; ++j) Mx = fmaxf(Mx, __ldg(st + j).x);
      float z = 0.f, q = 0.f;
      {
        const float* cp = a.ctxp[i] + (size_t)r * ns * H + col;
        float acc = 0.f;
#pragma unroll 4
        for (int j = 0; j < ns; ++j) {
          const float4 sj = __ldg(st + j);
          const float cj = cp[(size_t)j * H];
          const float e = (sj.x == -INFINITY) ? 0.f : fexp(sj.x - Mx);
          z = fmaf(sj.y, e, z);
          q = fmaf(sj.z, e, q);
          acc = fmaf(cj, e, acc);
        }
        cx[i] = z > 0.f ? acc / z : 0.f;
        if (tid < H) a.ctx[i][(size_t)r * H + tid] = cx[i];
      }
      M[i] = Mx; Z[i] = z; Q[i] = q;
      wstamp();
    }
    }
    float part[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      float pk = wmh[k] * y;
      if (!a.gate_ctx) {
        const float* wr = a.Wm + (size_t)k * 3 * H;
        pk = fmaf(__ldg(wr + H + col), cx[0], fmaf(__ldg(wr + 2 * H + col), cx[1], pk));
      }
      part[k] = warp_sum(tid < H ? pk : 0.f);
    }
    if (lane == 0) { sh[warp * 3] = part[0]; sh[warp * 3 + 1] = part[1]; sh[warp * 3 + 2] = part[2]; }
    wstamp();
    __syncthreads();
    wstamp();
    float lg[3] = {bmv[0] + gsum[0], bmv[1] + gsum[1], bmv[2] + gsum[2]};
#pragma unroll
    for (int w = 0; w < TSW; ++w) { lg[0] += sh[w * 3]; lg[1] += sh[w * 3 + 1]; lg[2] += sh[w * 3 + 2]; }
    const float mx = fmaxf(lg[0], fmaxf(lg[1], lg[2]));
    const float e0 = expf(lg[0] - mx), e1 = expf(lg[1] - mx), e2 = expf(lg[2] - mx);
    const float inv = 1.f / (e0 + e1 + e2);
    g0 = e0 * inv;
    const float gi[2] = {e1 * inv, e2 * inv};
    // copy weight(r,i,s) = F_i * prior_i[s] * exp(e_i[s] - M_i) == gate_{i+1} * (w a) / (1e-8 + sum w a)
    // (Model.py:110-111, 42) with a = softmax(e): F_i = gate_{i+1} / (Z_i * (1e-8 + Q_i / Z_i))
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      F[i] = Z[i] > 0.f ? gi[i] / (Z[i] * (1e-8f + Q[i] / Z[i])) : 0.f;
      M[i] = Z[i] > 0.f ? M[i] : 0.f;
    }
    if (tid == 0) {
      float* gt = a.gates + (size_t)r * 4;
      gt[0] = g0; gt[1] = gi[0]; gt[2] = gi[1]; gt[3] = 0.f;
      float* f = a.fac + (size_t)r * a.fac_ld;
      f[a.fac_off[0]] = F[0]; f[a.fac_off[0] + 1] = M[0];
      f[a.fac_off[1]] = F[1]; f[a.fac_off[1] + 1] = M[1];
    }
    wstamp();
  } else {
    g0 = a.gates[(size_t)r * 4];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      if (i < a.nmem) {
        F[i] = a.fac[(size_t)r * a.fac_ld + a.fac_off[i]];
        M[i] = a.fac[(size_t)r * a.fac_ld + a.fac_off[i] + 1];
      }
    }
    __syncthreads();       // the table is initialised
  }
  if constexpr (CONSTR) {
    // (both branches above end with a barrier: the history is visible.)  Candidate j < t: the n-gram y_{j+1} ..
    // y_{j+n} lies in the answer and its first n - 1 tokens are the answer's last n - 1, so y_{j+n} is banned;
    // candidate t: the EOS of an answer shorter than min_len; candidate t + 1 + i: banned sequence i = (w_1 .. w_L)
    // bans w_L when the answer ends with w_1 .. w_{L-1}.  An id is kept at its first candidate only, and the kept ids
    // are compacted into the banned list (its order does not matter)
    const int t = a.t, n = a.no_repeat_ngram;
    const int nseq = a.ban_n != nullptr ? min(max(*a.ban_n, 0), CASE_MAX_BAN_SEQ) : 0;
    const int ncand = t + 1 + nseq;
    if (tid < ncand) {
      int c = -1;
      if (tid < t) {
        if (n > 0 && tid + n <= t) {
          bool eq = true;
          for (int k = 0; k < n - 1; ++k) eq &= cs[CS_HIST + tid + k] == cs[CS_HIST + t - n + 1 + k];
          if (eq) c = cs[CS_HIST + tid + n - 1];
        }
      } else if (tid == t) {
        if (t < a.min_len) c = a.eos;
      } else {
        const int i = tid - t - 1, L = a.ban_len[i];
        const int32_t* w = a.ban_tok + (size_t)i * CASE_MAX_BAN_LEN;
        if (L >= 2 && L <= CASE_MAX_BAN_LEN && t >= L - 1) {
          bool eq = true;
          for (int k = 0; k < L - 1; ++k) eq &= cs[CS_HIST + t - L + 1 + k] == w[k];
          if (eq) c = w[L - 1];
        }
      }
      cs[CS_CAND + tid] = c;
    }
    __syncthreads();
    if (tid < ncand) {
      const int c = cs[CS_CAND + tid];
      bool first = c >= 0;
      if (first)
        for (int j = 0; j < tid; ++j) first &= cs[CS_CAND + j] != c;
      if (first) cs[CS_BAN + atomicAdd(cs + CS_NBAN, 1)] = c;
    }
    // (visible after the barrier that ends the copy-mass pass)
  }
  stamp();
  // ---- copy mass of both memories into the hash table (double hashing, ids are exact).  The source positions of
  // both memories are one index space, so all loads of a thread (ids, scores, priors: <= 6 positions at S = 2620)
  // are in flight in ONE round
  if (!plan) {
    const int S0n = a.S[0], S1n = a.nmem > 1 ? a.S[1] : 0, Stot = S0n + S1n;
    const float* at0 = a.attn_un[0] + (size_t)r * S0n;
    const float* at1 = a.nmem > 1 ? a.attn_un[1] + (size_t)r * S1n : nullptr;
    const float* pr0 = a.prior[0] ? a.prior[0] + (size_t)b * S0n : nullptr;
    const float* pr1 = (a.nmem > 1 && a.prior[1]) ? a.prior[1] + (size_t)b * S1n : nullptr;
    const int32_t* mp0 = a.map + (size_t)b * a.map_ld + a.map_off[0];
    const int32_t* mp1 = a.map + (size_t)b * a.map_ld + a.map_off[1];
    constexpr int HU = 8;                                  // positions per thread per round
    for (int s0 = tid; s0 < Stot; s0 += HU * TS) {
      int id[HU];
      float ev[HU], pv[HU];
#pragma unroll
      for (int u = 0; u < HU; ++u) {
        const int sidx = s0 + u * TS;
        const bool in = sidx < Stot, m1 = sidx >= S0n;
        const int sl = m1 ? sidx - S0n : sidx;
        const float* pr = m1 ? pr1 : pr0;
        id[u] = in ? __ldg((m1 ? mp1 : mp0) + sl) : -1;
        ev[u] = in ? (m1 ? at1 : at0)[sl] : -INFINITY;
        pv[u] = (in && pr) ? __ldg(pr + sl) : 1.f;
      }
#pragma unroll
      for (int u = 0; u < HU; ++u) {
        if (ev[u] == -INFINITY || (unsigned)id[u] >= (unsigned)Vx) continue;   // masked source position
        const bool m1 = s0 + u * TS >= S0n;
        const float cw = (m1 ? F[1] : F[0]) * pv[u] * fexp(ev[u] - (m1 ? M[1] : M[0]));
        if (cw == 0.f) continue;
        uint32_t slot = sp_hash(id[u], hshift);
        const uint32_t step = sp_step(id[u]);
        while (true) {
          const int old = atomicCAS(hkeys + slot, -1, id[u]);
          if (old == -1 || old == id[u]) {
            // units of 2^-48 (3.6e-15: below fp32 resolution for every mass >= 6e-8, exact conversion for cw >= 2^-24);
            // probability masses are <= 1, the 16 integer bits are headroom for un-normalised callers (saturating)
            const unsigned long long q = __float2ull_rn(fminf(cw, 32768.f) * 281474976710656.f);
            const uint32_t lo = (uint32_t)q;
            const uint32_t prev = atomicAdd(hlo + slot, lo);
            const uint32_t hi = (uint32_t)(q >> 32) + ((uint32_t)(prev + lo) < prev ? 1u : 0u);   // carry out of the low word
            if (hi) atomicAdd(hhi + slot, hi);
            break;
          }
          slot = (slot + step) & hmask;
        }
      }
    }
  }
  __syncthreads();
  stamp();
  // ---- candidates: every touched id (base value gathered from the logits) and the base top entries
  float mrow = -INFINITY;
#pragma unroll
  for (int k = 0; k < SP_PARTS; ++k) mrow = fmaxf(mrow, base_ms[((size_t)r * SP_PARTS + k) * 2]);
  float srow = 0.f;
#pragma unroll
  for (int k = 0; k < SP_PARTS; ++k) {
    const float mk = base_ms[((size_t)r * SP_PARTS + k) * 2];
    srow += (mk > -INFINITY) ? base_ms[((size_t)r * SP_PARTS + k) * 2 + 1] * sp_exp(mk - mrow) : 0.f;
  }
  const float mm = (mrow > -INFINITY) ? mrow : 0.f;
  const float scl = g0 / srow;
  const float* x = a.logits + (size_t)r * a.ldl;
  const int K = a.K;
  // pass A: the final value of every touched id replaces its mass in the table; thread maximum
  float tmax = -INFINITY;
  if (plan) {
    const int S0n = a.S[0], S1n = a.S[1];
    const float* at0 = a.attn_un[0] + (size_t)r * S0n;
    const float* at1 = a.attn_un[1] + (size_t)r * S1n;
    const float* pr0 = a.prior[0] ? a.prior[0] + (size_t)b * S0n : nullptr;
    const float* pr1 = a.prior[1] ? a.prior[1] + (size_t)b * S1n : nullptr;
    const size_t pb = (size_t)b * a.cp_ld;
    auto copy_w = [&](int pos) -> float {                // gate_i * p_i[pos] of the reference (Model.py:41-42, 110-111)
      const bool m1 = pos >= S0n;
      const int sl = m1 ? pos - S0n : pos;
      const float ev = (m1 ? at1 : at0)[sl];
      const float* pr = m1 ? pr1 : pr0;
      const float pv = pr ? __ldg(pr + sl) : 1.f;
      return ev == -INFINITY ? 0.f : (m1 ? F[1] : F[0]) * pv * fexp(ev - (m1 ? M[1] : M[0]));
    };
    constexpr int PU = 4;                                  // list entries per thread per round
    for (int u0 = tid; u0 < nent; u0 += PU * TS) {
      int id[PU], fp[PU];
      float lv[PU], ev[PU], pv[PU];
#pragma unroll
      for (int j = 0; j < PU; ++j) {
        const int u = u0 + j * TS;
        id[j] = u < nent ? __ldg(a.cp_uid + pb + u) : -1;
        fp[j] = u < nent ? __ldg(a.cp_first + pb + u) : 0;      // first position | (occurrences - 1) << 16
      }
#pragma unroll
      for (int j = 0; j < PU; ++j) {
        lv[j] = 0.f; ev[j] = -INFINITY; pv[j] = 1.f;
        if (id[j] >= 0) {
          const int pos = fp[j] & 0xffff;
          const bool m1 = pos >= S0n;
          const int sl = m1 ? pos - S0n : pos;
          const float* pr = m1 ? pr1 : pr0;
          lv[j] = x[id[j]];
          ev[j] = (m1 ? at1 : at0)[sl];
          if (pr) pv[j] = __ldg(pr + sl);
        }
      }
#pragma unroll
      for (int j = 0; j < PU; ++j) {
        if (id[j] < 0) continue;
        const int u = u0 + j * TS, pos = fp[j] & 0xffff;
        const bool m1 = pos >= S0n;
        float mass = ev[j] == -INFINITY ? 0.f : (m1 ? F[1] : F[0]) * pv[j] * fexp(ev[j] - (m1 ? M[1] : M[0]));
        const int extra = (int)((uint32_t)fp[j] >> 16);
        if (extra > 0) {                                   // repeated id: the other occurrences, in position order
          const int k0 = __ldg(a.cp_start + pb + u);
          for (int k = 1; k <= extra; ++k) mass += copy_w(__ldg(a.cp_perm + pb + k0 + k));
        }
        const float e = (a.mask_col0 && id[j] == 0) ? 0.f : sp_exp(lv[j] - mm);
        const float f = fmaf(scl, e, mass);
        hkeys[u] = id[j];
        hvals[u] = f;
        tmax = fmaxf(tmax, f);
      }
    }
    __syncthreads();                                       // the list is read by other threads below
  } else
  for (int s0 = tid; s0 < nslots; s0 += 4 * TS) {        // nslots is a multiple of 4 * TS
    int id[4];
    float lv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      id[u] = hkeys[s0 + u * TS];
      lv[u] = (id[u] >= 0 && id[u] < V) ? x[id[u]] : -INFINITY;     // dynamic entries: no base term
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (id[u] < 0) continue;
      const float e = ((a.mask_col0 && id[u] == 0) || id[u] >= V) ? 0.f : sp_exp(lv[u] - mm);
      const unsigned long long q = ((unsigned long long)hhi[s0 + u * TS] << 32) | hlo[s0 + u * TS];
      const float f = fmaf(scl, e, __ull2float_rn(q) * 3.552713678800501e-15f);   // 2^-48
      hvals[s0 + u * TS] = f;
      tmax = fmaxf(tmax, f);
    }
  }
  stamp();
  const int nban = CONSTR ? cs[CS_NBAN] : 0;             // constrained: entries of the banned list
  // constrained: is id banned (the row's list or the single-id mask)?
  auto banned = [&](int id) { return sp_banned(cs + CS_BAN, nban, id) || sp_masked(a.ban_mask, id, V); };
  if constexpr (CONSTR) {
    // banned touched ids: one lookup each, the value becomes -inf; then the thread maxima again without them, every
    // touched id tested against the mask on the way
    __syncthreads();
    if (tid < nban) {
      const int id = cs[CS_BAN + tid];
      const int sl = sp_find(hkeys, nent, plan, id, hshift, hmask);
      if (sl >= 0) hvals[sl] = -INFINITY;
    }
    __syncthreads();
    tmax = -INFINITY;
    for (int sl = tid; sl < nent; sl += TS) {
      const int id = hkeys[sl];
      if (id < 0) continue;
      if (sp_masked(a.ban_mask, id, V)) hvals[sl] = -INFINITY;
      else tmax = fmaxf(tmax, hvals[sl]);
    }
  }
  float fb = -INFINITY;                                  // base candidates that received no copy mass
  int idb = 0x7fffffff;
  if (tid < SP_PARTS * k2) {
    const int id = base_i[(size_t)r * SP_PARTS * k2 + tid];
    const float l = base_e[(size_t)r * SP_PARTS * k2 + tid];
    if ((unsigned)id < (unsigned)V && l > -INFINITY) {
      bool found = false;
      if (plan) {                                          // the list is sorted: binary search
        int lo = 0, hi = nent;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (hkeys[mid] < id) lo = mid + 1; else hi = mid;
        }
        found = lo < nent && hkeys[lo] == id;
      } else {
        uint32_t slot = sp_hash(id, hshift);
        const uint32_t step = sp_step(id);
        while (true) {
          const int key = hkeys[slot];
          if (key == id) { found = true; break; }
          if (key == -1) break;
          slot = (slot + step) & hmask;
        }
      }
      if (!found && !(CONSTR && banned(id))) { fb = scl * sp_exp(l - mm); idb = id; }
    }
  }
  bool exact = false;
  if constexpr (CONSTR) {
    // a = allowed ids among the row's global top-k2 base entries (rank over the SP_PARTS * k2 partial entries)
    int* bi = cs + CS_BASE;
    float* bl = reinterpret_cast<float*>(bi + SP_PARTS * k2);
    int id = 0x7fffffff;
    float l = -INFINITY;
    if (tid < SP_PARTS * k2) {
      id = base_i[(size_t)r * SP_PARTS * k2 + tid];
      l = base_e[(size_t)r * SP_PARTS * k2 + tid];
      if (!((unsigned)id < (unsigned)V && l > -INFINITY)) { id = 0x7fffffff; l = -INFINITY; }
      bi[tid] = id;
      bl[tid] = l;
    }
    __syncthreads();
    bool allowed = false;
    if (tid < SP_PARTS * k2 && l > -INFINITY) {
      int rank = 0;
      for (int j = 0; j < SP_PARTS * k2; ++j) rank += tk_better(bl[j], bi[j], l, id);
      allowed = rank < k2 && !banned(id);
    }
    exact = __syncthreads_count(allowed) < 2 * K;
  }
  float ov = -INFINITY;
  int oi = 0x7fffffff;
  if (CONSTR && exact) {
    // exact pass: every allowed touched id (banned ones hold -inf) and every allowed untouched id of the row
    if (fbcount != nullptr && tid == 0) atomicAdd(fbcount, 1);
    WarpTopK wl;
    wl.init();
    for (int s0 = 0; s0 < nent; s0 += TS) {
      const int id = s0 + tid < nent ? hkeys[s0 + tid] : -1;
      const float v = id >= 0 ? hvals[s0 + tid] : -INFINITY;
      wl.offer(K, v, v > -INFINITY ? id : 0x7fffffff);
    }
    for (int v0 = 0; v0 < V; v0 += TS) {
      const int id = v0 + tid;
      float f = -INFINITY;
      if (id < V && !(a.mask_col0 && id == 0) && sp_find(hkeys, nent, plan, id, hshift, hmask) < 0 &&
          !banned(id)) {
        const float l = x[id];
        if (l > -INFINITY) f = scl * sp_exp(l - mm);
      }
      wl.offer(K, f, f > -INFINITY ? id : 0x7fffffff);
    }
    block_merge_lists(sc, wl, K);
    ov = wl.ev; oi = wl.ei;
    stamp();
  } else {
  tmax = fmaxf(tmax, fb);
  const float T = block_kth_max(sc, K, tmax);
  if (tmax >= T && tmax > -INFINITY) {
    for (int sl = tid; sl < nent; sl += TS) {
      const int id = hkeys[sl];
      if (id >= 0 && hvals[sl] >= T) topk_append(sc, hvals[sl], id);
    }
    if (fb >= T) topk_append(sc, fb, idb);
  }
  __syncthreads();
  stamp();
  if (!block_select(sc, K, ov, oi)) {                    // massive ties: offer every candidate
    WarpTopK wl;
    wl.init();
    for (int s0 = 0; s0 < nent; s0 += TS) {
      const int id = s0 + tid < nent ? hkeys[s0 + tid] : -1;
      wl.offer(K, id >= 0 ? hvals[s0 + tid] : -INFINITY, id >= 0 ? id : 0x7fffffff);
    }
    wl.offer(K, fb, idb);
    block_merge_lists(sc, wl, K);
    ov = wl.ev; oi = wl.ei;
  }
  }
  if (warp == 0 && lane < K) {
    a.top_vals[(size_t)r * K + lane] = ov;
    a.top_idx[(size_t)r * K + lane] = oi;
  }
  stamp();
  if constexpr (ATTR) {
    // ---- attribution of the K winners: the source positions are walked again (the same map / score / prior loads as
    // the hash pass, which just read them, so they come from L2) and a position whose id is a winner adds its
    // contribution to the (winner, memory) accumulator - in the fixed point and with the split-word atomics of the hash
    // table, so in hash mode the two copy parts add up, as integers, to exactly the mass the ranking used - and offers
    // (float bits of the contribution, ~position) to one 64-bit maximum: contributions are positive, so the bit order
    // is the value order, and ties go to the lowest position.  Independent of the copy plan.
    __shared__ int s_aid[CASE_MAX_W];
    __shared__ uint32_t s_alo[CASE_MAX_W][2], s_ahi[CASE_MAX_W][2];
    __shared__ unsigned long long s_asrc[CASE_MAX_W];
    if (tid < CASE_MAX_W) {                                // warp 0: lane k < K holds winner k
      s_aid[tid] = tid < K ? oi : -1;
      s_alo[tid][0] = s_alo[tid][1] = s_ahi[tid][0] = s_ahi[tid][1] = 0u;
      s_asrc[tid] = 0ull;
    }
    __syncthreads();
    const int S0n = a.S[0], S1n = a.nmem > 1 ? a.S[1] : 0, Stot = S0n + S1n;
    const float* at0 = a.attn_un[0] + (size_t)r * S0n;
    const float* at1 = a.nmem > 1 ? a.attn_un[1] + (size_t)r * S1n : nullptr;
    const float* pr0 = a.prior[0] ? a.prior[0] + (size_t)b * S0n : nullptr;
    const float* pr1 = (a.nmem > 1 && a.prior[1]) ? a.prior[1] + (size_t)b * S1n : nullptr;
    const int32_t* mp0 = a.map + (size_t)b * a.map_ld + a.map_off[0];
    const int32_t* mp1 = a.map + (size_t)b * a.map_ld + a.map_off[1];
    constexpr int HU = 4;                                  // positions per thread per round (loads from L2)
    for (int s0 = tid; s0 < Stot; s0 += HU * TS) {
      int id[HU];
      float ev[HU], pv[HU];
#pragma unroll
      for (int u = 0; u < HU; ++u) {
        const int sidx = s0 + u * TS;
        const bool in = sidx < Stot, m1 = sidx >= S0n;
        const int sl = m1 ? sidx - S0n : sidx;
        const float* pr = m1 ? pr1 : pr0;
        id[u] = in ? __ldg((m1 ? mp1 : mp0) + sl) : -1;
        ev[u] = in ? (m1 ? at1 : at0)[sl] : -INFINITY;
        pv[u] = (in && pr) ? __ldg(pr + sl) : 1.f;
      }
#pragma unroll
      for (int u = 0; u < HU; ++u) {
        if (ev[u] == -INFINITY || (unsigned)id[u] >= (unsigned)Vx) continue;
        int k = -1;
        for (int j = 0; j < K; ++j) k = id[u] == s_aid[j] ? j : k;
        if (k < 0) continue;
        const int sidx = s0 + u * TS;
        const bool m1 = sidx >= S0n;
        const float cw = (m1 ? F[1] : F[0]) * pv[u] * fexp(ev[u] - (m1 ? M[1] : M[0]));   // as in the hash pass
        const unsigned long long q = __float2ull_rn(fminf(cw, 32768.f) * 281474976710656.f);
        if (q == 0ull) continue;                           // below the fixed point's resolution: no contribution
        const uint32_t lo = (uint32_t)q;
        const uint32_t prev = atomicAdd(&s_alo[k][m1], lo);
        const uint32_t hi = (uint32_t)(q >> 32) + ((uint32_t)(prev + lo) < prev ? 1u : 0u);
        if (hi) atomicAdd(&s_ahi[k][m1], hi);
        atomicMax(&s_asrc[k], ((unsigned long long)__float_as_uint(cw) << 32) | (0xFFFFFFFFu - (uint32_t)sidx));
      }
    }
    __syncthreads();
    if (tid < K) {
      const int y = s_aid[tid];
      case_attr_t rec;
      rec.part[0] = rec.part[1] = rec.part[2] = 0.f;
      rec.source = -1;
      if ((unsigned)y < (unsigned)Vx) {
        // generation part: the expression the value was built from
        const float e = ((a.mask_col0 && y == 0) || y >= V) ? 0.f : sp_exp(x[y] - mm);
        rec.part[0] = scl * e;
#pragma unroll
        for (int i = 0; i < 2; ++i)
          rec.part[1 + i] = __ull2float_rn(((unsigned long long)s_ahi[tid][i] << 32) | s_alo[tid][i]) * 3.552713678800501e-15f;
        const unsigned long long key = s_asrc[tid];
        if (key) rec.source = (int)(0xFFFFFFFFu - (uint32_t)key);
      }
      a.attr[(size_t)r * K + tid] = rec;
    }
  }
  // ---- fused search bookkeeping: the last CTA of a query's W rows runs Generations.beam / greedy for it
  if (do_select) {
    __shared__ int s_last;
    __syncthreads();                                      // this row's top-k is written (CTA scope) ...
    if (tid == 0) {
      // ... and published by ONE release at device scope (cumulative over the barrier) instead of a
      // sequentially-consistent fence by all 512 threads; the same operation acquires the other rows' top-k
      int old;
      asm volatile("atom.acq_rel.gpu.global.add.s32 %0, [%1], 1;" : "=r"(old) : "l"(qcount + b) : "memory");
      s_last = old == a.W - 1;
      if (s_last) qcount[b] = 0;                          // ready for the next step
    }
    __syncthreads();
    if (s_last && warp == 0) beam_select_query<ATTR>(sel, b, lane);
  }
}

}  // namespace cb

using namespace cb;

extern "C" int case_vocab_base(const float* logits, int ldl, int R, int V, int mask_col0, int k2, float* base_ms,
                               float* base_l, int32_t* base_i, case_stream_t stream) {
  CB_REQUIRE(logits && base_ms && base_l && base_i && R > 0 && V > 0, "case_vocab_base: bad arguments");
  CB_REQUIRE(k2 >= 1 && k2 <= 2 * CASE_MAX_W, "case_vocab_base: k2 out of range (1..16)");
  CB_REQUIRE(ldl % 4 == 0 && ldl >= ((V + 3) / 4) * 4 && (uintptr_t)logits % 16 == 0, "case_vocab_base: logits rows must be 16-byte aligned and padded to a multiple of 4");
  cudaStream_t st = (cudaStream_t)stream;
  const int Vq = (((V + SP_PARTS - 1) / SP_PARTS) + 3) / 4 * 4;
  const int grid = R * SP_PARTS;
  launch_k(vocab_base_kernel, grid, ST, 0, st, logits, ldl, V, Vq, mask_col0, k2, base_ms, base_l, base_i);
  return check_launch("case_vocab_base");
}

static thread_local long long* g_sp_dbg = nullptr;   // debugging aid of the calling thread
extern "C" int case_debug_sparse_tail_timing(void* buf) { g_sp_dbg = (long long*)buf; return 0; }
// debugging aid: every constrained row that takes the exact pass over its logits adds 1 to *counter (int32 on the
// device; NULL = off).  Read at launch, so a CUDA graph keeps the pointer it was captured with
static thread_local int* g_sp_fallbacks = nullptr;
extern "C" int case_debug_sparse_tail_fallbacks(void* counter) { g_sp_fallbacks = (int*)counter; return 0; }

extern "C" int case_sparse_tail_max_sources(void) { return 10900; }   // 16384 slots at load factor <= 2/3

extern "C" int case_sparse_tail(const case_tail_args_t* a, const float* base_ms, const float* base_e,
                                const int32_t* base_i, int k2, const case_select_args_t* sel, int32_t* qcount,
                                case_stream_t stream) {
  CB_REQUIRE(a && a->logits && a->gates && a->fac && a->map && base_ms && base_e && base_i, "case_sparse_tail: null pointer");
  CB_REQUIRE(a->R > 0 && a->W >= 1 && a->V > 0 && a->top_vals && a->top_idx, "case_sparse_tail: bad sizes / outputs");
  CB_REQUIRE(a->K >= 1 && a->K <= CASE_MAX_W && k2 >= a->K && k2 <= 2 * CASE_MAX_W, "case_sparse_tail: need K <= k2 <= 16");
  CB_REQUIRE(a->nmem >= 1 && a->nmem <= 2, "case_sparse_tail: nmem must be 1 or 2");
  CB_REQUIRE(!a->do_finalize || (a->nmem == 2 && a->hN && a->stats[0] && a->stats[1] && a->ctxp[0] && a->ctxp[1] && a->Wm && a->bm && (a->gate_ctx || (a->ctx[0] && a->ctx[1])) && a->ns[0] >= 1 && a->ns[1] >= 1 && a->ns[0] <= CASE_MAX_SPLIT && a->ns[1] <= CASE_MAX_SPLIT),
             "case_sparse_tail: the CaSE finaliser needs hN, stats, ctxp, Wm, bm, ctx for both memories");
  int total = 0;
  for (int i = 0; i < a->nmem; ++i) {
    CB_REQUIRE(a->attn_un[i] && a->S[i] > 0, "case_sparse_tail: attn_un / S missing");
    total += a->S[i];
  }
  CB_REQUIRE(total <= case_sparse_tail_max_sources(), "case_sparse_tail: too many source positions for the shared-memory table");
  int nslots = 4 * TS;
  while (nslots < 3 * total && nslots < 16384) nslots *= 2;  // load factor ~1/3 (<= 2/3 at the size limit)
  const bool plan = a->cp_n != nullptr;
  CB_REQUIRE(a->Vext == 0 || (a->Vext >= a->V && !plan), "case_sparse_tail: Vext must be >= V (hash-table mode)");
  CB_REQUIRE(!plan || (a->nmem == 2 && a->cp_uid && a->cp_first && a->cp_start && a->cp_perm && a->cp_ld >= total && total < 65536),
             "case_sparse_tail: the copy plan needs cp_uid / cp_first / cp_start / cp_perm with cp_ld >= S0 + S1 (two memories, < 65536 positions)");
  // plan mode: (id, value) per list entry, at most one per source position; the hash layout otherwise
  size_t smem = plan ? (size_t)((total + 3) / 4 * 4) * 8 : (size_t)nslots * 12;
  if (plan) nslots = (total + 3) / 4 * 4;
  if (sel) {
    int rc = check_nbest(sel->nbest, sel->W, sel->mode);
    if (rc) return rc;
    rc = check_attr_select(*sel);
    if (rc) return rc;
    CB_REQUIRE((sel->out_attr != nullptr) == (a->attr != nullptr) && (sel->attr_cand == nullptr || sel->attr_cand == a->attr),
               "case_sparse_tail: a fused select with attribution needs attr_cand == the tail's attr (both on or both off)");
  }
  const int nbanp = (a->ban_mask != nullptr) + (a->ban_tok != nullptr) + (a->ban_len != nullptr) + (a->ban_n != nullptr);
  CB_REQUIRE(nbanp == 0 || nbanp == 4, "case_sparse_tail: banned words need all of ban_mask / ban_tok / ban_len / ban_n (or none)");
  const bool constr = a->no_repeat_ngram != 0 || a->min_len != 0 || nbanp == 4;
  if (constr) {
    CB_REQUIRE(a->no_repeat_ngram >= 0 && a->no_repeat_ngram <= CASE_MAX_T && a->min_len >= 0 && a->min_len < CASE_MAX_T,
               "case_sparse_tail: no_repeat_ngram must be 0..CASE_MAX_T and min_len 0..CASE_MAX_T-1");
    CB_REQUIRE(a->hist_tok && a->hist_anc && a->t >= 0 && a->t < CASE_MAX_T && a->hist_ld > a->t,
               "case_sparse_tail: constraints need the answer history (hist_tok, hist_anc, 0 <= t < hist_ld)");
    CB_REQUIRE(a->V >= 2 * a->K + a->hist_ld, "case_sparse_tail: constraints need V >= 2K + Tmax + 1 (hist_ld = Tmax + 1)");
    smem += (size_t)CS_INTS * 4;
  }
  const bool attr = a->attr != nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  constexpr int cx = CS_INTS * 4;
  if (constr) {
    if (attr) ensure_smem<sparse_tail_kernel<true, true>>(16384 * 12 + cx);
    else ensure_smem<sparse_tail_kernel<false, true>>(16384 * 12 + cx);
  } else {
    if (attr) ensure_smem<sparse_tail_kernel<true, false>>(16384 * 12);
    else ensure_smem<sparse_tail_kernel<false, false>>(16384 * 12);
  }
  CB_REQUIRE(sel == nullptr || (qcount != nullptr && sel->B * sel->W == a->R && sel->W == a->W && a->K == a->W),
             "case_sparse_tail: fused select needs qcount and matching B / W (k = W)");
  case_select_args_t sv;
  memset(&sv, 0, sizeof(sv));
  if (sel) sv = *sel;
  auto kern = constr ? (attr ? sparse_tail_kernel<true, true> : sparse_tail_kernel<false, true>)
                     : (attr ? sparse_tail_kernel<true, false> : sparse_tail_kernel<false, false>);
  launch_k(kern, a->R, TS, smem, st, *a, base_ms, base_e, base_i, k2, nslots, g_sp_dbg, sv, sel ? 1 : 0, qcount,
           g_sp_fallbacks);
  return check_launch("case_sparse_tail");
}
