// Error plumbing and the whole-step orchestrators: one C call enqueues every kernel of a decode
// step on the caller's stream (so a step, or a whole decode, can be captured in a CUDA graph).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "select.cuh"

namespace cb {

// Nothing here is process-global: the error text, the pending launch error and the launch options belong to the
// calling thread; the side stream and events of the fork/join live in a caller-owned case_fork_t.
static thread_local char g_err[512] = "ok";
static thread_local cudaError_t g_launch_err = cudaSuccess;
static thread_local LaunchOpts g_opts = {1, 1};

LaunchOpts& launch_opts() { return g_opts; }
cudaError_t& launch_err() { return g_launch_err; }

void set_error(const char* msg) {
  strncpy(g_err, msg, sizeof(g_err) - 1);
  g_err[sizeof(g_err) - 1] = 0;
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = g_launch_err;
  g_launch_err = cudaSuccess;
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

// the orchestrators run with the options of THEIR argument block and put the thread's own back on every exit path
struct OptScope {
  LaunchOpts saved;
  explicit OptScope(int opt) : saved(g_opts) {
    g_opts.pdl = (opt & CASE_OPT_NO_PDL) ? 0 : 1;
    g_opts.evict_first = (opt & CASE_OPT_NO_EVICT_FIRST) ? 0 : 1;
  }
  ~OptScope() { g_opts = saved; }
};

}  // namespace cb

// side stream + events of the fork/join inside a step, owned by the caller (one per engine, on the engine's device)
struct case_fork_s {
  cudaStream_t aux;
  cudaEvent_t ev_fork[2], ev_join[2];
  int device;
};

using namespace cb;

extern "C" int case_fork_create(case_fork_t** out) {
  CB_REQUIRE(out, "case_fork_create: null pointer");
  case_fork_s* f = (case_fork_s*)calloc(1, sizeof(case_fork_s));
  CB_REQUIRE(f, "case_fork_create: out of host memory");
  cudaError_t e = cudaGetDevice(&f->device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&f->aux, cudaStreamNonBlocking);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&f->ev_fork[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->ev_join[i], cudaEventDisableTiming);
  }
  if (e != cudaSuccess) {
    set_error(cudaGetErrorString(e));
    case_fork_destroy(f);
    return (int)e;
  }
  *out = f;
  return 0;
}

extern "C" int case_fork_destroy(case_fork_t* f) {
  if (!f) return 0;
  for (int i = 0; i < 2; ++i) {
    if (f->ev_fork[i]) cudaEventDestroy(f->ev_fork[i]);
    if (f->ev_join[i]) cudaEventDestroy(f->ev_join[i]);
  }
  if (f->aux) cudaStreamDestroy(f->aux);
  free(f);
  return 0;
}

extern "C" int case_abi_version(void) { return 2; }
extern "C" int case_thread_options(int opt) {
  const int old = (g_opts.pdl ? 0 : CASE_OPT_NO_PDL) | (g_opts.evict_first ? 0 : CASE_OPT_NO_EVICT_FIRST);
  if (opt >= 0) {
    g_opts.pdl = (opt & CASE_OPT_NO_PDL) ? 0 : 1;
    g_opts.evict_first = (opt & CASE_OPT_NO_EVICT_FIRST) ? 0 : 1;
  }
  return old;
}
extern "C" const char* case_last_error(void) { return g_err; }

#define TRY(x)            \
  do {                    \
    int _e = (x);         \
    if (_e) return _e;    \
  } while (0)

static case_seg_t seg(const float* p, int ld, int width, int div, int gather = 0) {
  case_seg_t s;
  s.p = p; s.ld = ld; s.width = width; s.div = div; s.gather = gather;
  return s;
}

static case_select_args_t select_args(int mode, int B, int W, int t, int max_len, int Tmax, int BOS, int EOS, int UNK,
                                      int PAD, const float* top_vals, const int32_t* top_idx, int32_t* live, double* cum,
                                      int32_t* length, int32_t* tok, int32_t* const anc[2], int32_t* parent,
                                      int32_t* ended, double* best_key, int32_t* best_len, int32_t* out_tokens,
                                      int32_t* n_live, int nbest) {
  case_select_args_t s;
  memset(&s, 0, sizeof(s));
  s.mode = mode; s.B = B; s.W = W; s.t = t; s.max_len = max_len; s.Tmax = Tmax;
  s.BOS = BOS; s.EOS = EOS; s.UNK = UNK; s.PAD = PAD;
  s.top_vals = top_vals; s.top_idx = top_idx; s.live = live; s.cum = cum; s.length = length; s.tok = tok;
  s.anc_in = anc[t & 1]; s.anc_out = anc[(t + 1) & 1]; s.parent = parent; s.ended = ended;
  s.best_key = best_key; s.best_len = best_len; s.out_tokens = out_tokens; s.n_live = n_live; s.nbest = nbest;
  return s;
}

// Attribution records of a step (the attr_* fields of the step blocks): all three or none, and only where the step takes
// the sparse tail - the only tail with an attribution pass.  Checked before the first launch of the step.
static int check_step_attr(const case_attr_t* cand, const case_attr_t* hist, const case_attr_t* out, bool sparse,
                           const char* what) {
  const int n = (cand != nullptr) + (hist != nullptr) + (out != nullptr);
  if (n == 0) return 0;
  if (n != 3) {
    char msg[160];
    snprintf(msg, sizeof(msg), "%s: attribution needs attr_cand, attr_hist and out_attr (or none of them)", what);
    set_error(msg);
    return CASE_EINVAL;
  }
  if (!sparse) {
    char msg[256];
    snprintf(msg, sizeof(msg), "%s: attribution needs the sparse tail (not with CASE_OPT_DENSE_TAIL / UNFUSED_TAIL, "
             "materialize_only, missing base_* buffers, V < 2W or too many source positions)", what);
    set_error(msg);
    return CASE_EINVAL;
  }
  return 0;
}

// Search constraints of a step (no_repeat_ngram / min_len of the step blocks; both 0 = off): in range, in a search mode
// that has them, and only where the step takes the sparse tail - the only tail that applies them.  Checked before the
// first launch of the step, after the n-best and attribution checks.
static int check_step_constr(int n, int min_len, int mode, int max_len, int V, int W, int Tmax, bool sparse,
                             const char* what) {
  if (n == 0 && min_len == 0) return 0;
  char msg[256];
  const char* why = nullptr;
  if (n < 0 || n > max_len || min_len < 0 || min_len >= max_len)
    why = "constraints out of range: 0 <= no_repeat_ngram <= max_len, 0 <= min_len < max_len";
  else if (mode != CASE_MODE_BEAM && mode != CASE_MODE_PROTO_GREEDY)
    why = "constraints need CASE_MODE_BEAM or CASE_MODE_PROTO_GREEDY";
  else if (!sparse)
    why = "constraints need the sparse tail (not with CASE_OPT_DENSE_TAIL / UNFUSED_TAIL, materialize_only, missing "
          "base_* buffers, V < 2W or too many source positions)";
  else if (V < 2 * W + Tmax + 1)
    why = "constraints need V >= 2W + Tmax + 1";
  if (why == nullptr) return 0;
  snprintf(msg, sizeof(msg), "%s: %s", what, why);
  set_error(msg);
  return CASE_EINVAL;
}

// Banned words of a step (ban_mask / ban_tok / ban_len / ban_n of the step blocks; all four or none, NULL = off): in a
// search mode that has them and only where the step takes the sparse tail, like the constraints.  The list itself lives
// in device memory and the launchers never synchronise, so only the pointers are checked here (the kernel bounds what it
// reads of the content).  Checked before the first launch of the step, after the constraint check.
static int check_step_bans(const void* mask, const void* tok, const void* len, const void* n, int mode, int V, int W,
                           int Tmax, bool sparse, const char* what) {
  const int set = (mask != nullptr) + (tok != nullptr) + (len != nullptr) + (n != nullptr);
  if (set == 0) return 0;
  char msg[256];
  const char* why = nullptr;
  if (set != 4)
    why = "banned words need all of ban_mask / ban_tok / ban_len / ban_n (or none)";
  else if (mode != CASE_MODE_BEAM && mode != CASE_MODE_PROTO_GREEDY)
    why = "banned words need CASE_MODE_BEAM or CASE_MODE_PROTO_GREEDY";
  else if (!sparse)
    why = "banned words need the sparse tail (not with CASE_OPT_DENSE_TAIL / UNFUSED_TAIL, materialize_only, missing "
          "base_* buffers, V < 2W or too many source positions)";
  else if (V < 2 * W + Tmax + 1)
    why = "banned words need V >= 2W + Tmax + 1";
  if (why == nullptr) return 0;
  snprintf(msg, sizeof(msg), "%s: %s", what, why);
  set_error(msg);
  return CASE_EINVAL;
}

// the tail's view of the search state: row r's answer tokens along anc_in (the returned ids: tok_ext when present);
// needed by the constraints and the banned words alike
static void set_tail_constr(case_tail_args_t& ta, const int32_t* tok, const int32_t* anc_in, int TL, int t, int EOS,
                            int n, int min_len, const uint32_t* ban_mask, const int32_t* ban_tok, const int32_t* ban_len,
                            const int32_t* ban_n) {
  if (n == 0 && min_len == 0 && ban_mask == nullptr) return;
  ta.hist_tok = tok; ta.hist_anc = anc_in; ta.hist_ld = TL; ta.t = t; ta.eos = EOS;
  ta.no_repeat_ngram = n; ta.min_len = min_len;
  ta.ban_mask = ban_mask; ta.ban_tok = ban_tok; ta.ban_len = ban_len; ta.ban_n = ban_n;
}

static void set_select_attr(case_select_args_t& s, case_attr_t* cand, case_attr_t* hist, case_attr_t* out) {
  if (out == nullptr) return;
  s.attr_cand = cand; s.attr_hist = hist; s.out_attr = out;
}

extern "C" int case_decode_step(const case_step_args_t* a, int t, case_stream_t stream) {
  CB_REQUIRE(a, "case_decode_step: null args");
  CB_REQUIRE(a->R == a->B * a->W && a->W >= 1 && a->W <= CASE_MAX_W, "case_decode_step: R != B*W or W out of range");
  CB_REQUIRE(t >= 0 && t < a->Tmax && a->Tmax <= CASE_MAX_T, "case_decode_step: t out of range");
  CB_REQUIRE(a->materialize_only || t < a->max_len, "case_decode_step: t >= max_len");
  TRY(check_nbest(a->nbest, a->W, a->mode));
  cudaStream_t st = (cudaStream_t)stream;
  const int R = a->R, B = a->B, W = a->W, TL = a->Tmax + 1, dt = a->dtype;
  const int32_t* anc = a->anc[t & 1];
  const int opt = a->opt;
  OptScope scope(opt);
  // extended vocabulary (n_oov dynamic ids behind the V fixed ones): the sparse tail handles it on the search path, the
  // dense forms fall to the unfused kernels, which are generic in the row width
  const int n_oov = a->n_oov > 0 ? a->n_oov : 0, Vx = a->V + n_oov;
  CB_REQUIRE(n_oov == 0 || (a->tok_ext != nullptr && a->ldv >= Vx), "case_decode_step: n_oov needs tok_ext and ldv >= V + n_oov");
  const int use_tail = (opt & CASE_OPT_UNFUSED_TAIL) ? 0 : ((opt & CASE_OPT_DENSE_TAIL) ? 1 : 2);
  if (a->fork != nullptr) {
    int dev = -1;
    cudaGetDevice(&dev);
    CB_REQUIRE(dev == a->fork->device, "case_decode_step: the fork handle was created on another device");
  }

  // search path: the sparse tail (touched ids + base candidates); `generate` face: the dense fused tail
  const int k2 = 2 * W;
  const bool sparse = use_tail == 2 && !a->materialize_only && a->base_ms && a->base_e && a->base_i && a->V >= k2 &&
                      a->S[0] + a->S[1] <= case_sparse_tail_max_sources();
  TRY(check_step_attr(a->attr_cand, a->attr_hist, a->out_attr, sparse, "case_decode_step"));
  TRY(check_step_constr(a->no_repeat_ngram, a->min_len, a->mode, a->max_len, a->V, W, a->Tmax, sparse, "case_decode_step"));
  TRY(check_step_bans(a->ban_mask, a->ban_tok, a->ban_len, a->ban_n, a->mode, a->V, W, a->Tmax, sparse, "case_decode_step"));
  const bool attr = a->out_attr != nullptr;
  // constrained steps ask vocab_base for the most base entries the buffers hold (see sparse_tail.cu: exactness)
  const int k2b = (a->no_repeat_ngram || a->min_len || a->ban_mask) ? 2 * CASE_MAX_W : k2;
  // gate form of the additive attentions: the contexts only feed the mixture gate, so 3 gate-projected numbers
  // per key replace the value rows (needs the sparse tail, which merges gate partials instead of contexts)
  const bool gate = !(opt & CASE_OPT_NO_GATE) && sparse && dt == CASE_BF16 && a->Gv[0] != nullptr && a->Gv[1] != nullptr;
  // attns[i]: query = [dec_out ; norm2(answer_rep)]   (Model.py:108), then the fused additive attention
  auto stack_attention = [&](int i, const float* hsrc, float* qa, cudaStream_t s2, bool have_qa = false) -> int {
    if (have_qa) goto additive;          // the query was produced by a post linear of the preceding cluster launch
    {
    case_rowlin_args_t q;
    memset(&q, 0, sizeof(q));
    q.seg[0] = seg(hsrc, H, H, 1);
    q.seg[1] = seg(a->feat, H, H, W);
    q.nseg = 2; q.K = 2 * H; q.Wt = a->Wqa_t[i]; q.bias = a->bqa[i]; q.N = H; q.out = qa; q.ldo = H;
    q.R = R; q.dtype = dt;
    TRY(case_row_linear(&q, s2));
    }
  additive:
    if (gate) {
      const bool cmp = i == 1 && a->xidx != nullptr && a->xcount != nullptr;
      return case_additive_attn_gate(qa, a->U[i], a->Gv[i], a->va[i], a->mask[i], a->prior[i], a->tok, TL, t, B, W, a->S[i],
                                     a->nsplit_a[i], a->attn_un[i], a->stats[i], a->ctxp[i], a->fast_tanh,
                                     cmp ? a->xidx : nullptr, cmp ? a->xcount : nullptr, cmp ? a->xorder : nullptr,
                                     cmp ? a->xns : nullptr, s2);
    }
    if (i == 1 && dt == CASE_BF16 && a->xidx != nullptr && a->xcount != nullptr)   // valid keys only, balanced splits
      return case_additive_attn_compact(qa, a->U[i], a->Mv[i], a->va[i], a->mask[i], a->prior[i], a->tok, TL, t, B, W,
                                        a->S[i], H, a->nsplit_a[i], a->attn_un[i], a->stats[i], a->ctxp[i],
                                        a->fast_tanh, a->xidx, a->xcount, a->xorder, s2);
    return case_additive_attn(qa, a->U[i], a->Mv[i], a->va[i], a->mask[i], a->prior[i], a->tok, TL, t, B, W, a->S[i],
                              H, a->nsplit_a[i], a->attn_un[i], a->stats[i], a->ctxp[i], a->fast_tanh, dt, s2);
  };
  auto gen0 = [&]() -> int {   // gen.0 on [dec_input ; norm1(dec_out) ; feat]   (Model.py:115)
    case_rowlin_args_t g;
    memset(&g, 0, sizeof(g));
    g.seg[0] = seg(a->x_in, H, H, 1);
    g.seg[1] = seg(a->hN, H, H, 1);
    g.seg[2] = seg(a->feat, H, H, W);
    g.nseg = 3; g.K = 3 * H; g.Wt = a->Wg_t; g.bias = a->bg; g.N = H; g.out = a->gfeat; g.ldo = H;
    g.R = R; g.dtype = dt;
    return case_row_linear(&g, st);
  };
  auto finalize = [&]() -> int {
    return case_finalize_rows(a->h, a->lnN_g, a->lnN_b, a->stats[0], a->ctxp[0], a->nsplit_a[0], a->stats[1],
                              a->ctxp[1], a->nsplit_a[1], a->Wm, a->bm, a->hN, a->ctx[0], a->ctx[1], a->gates, a->fac, R,
                              st);
  };
#define CUTRY(x)                                                         \
  do {                                                                   \
    cudaError_t _ce = (x);                                               \
    if (_ce != cudaSuccess) {                                            \
      set_error(cudaGetErrorString(_ce));                                \
      return (int)_ce;                                                   \
    }                                                                    \
  } while (0)
  // cross-attention over memory i for layer L: compacted + balanced partition where the prefill provided it
  const bool xpart = dt == CASE_BF16 && a->xcount != nullptr && a->xprefix != nullptr && a->xslots > 0;
  auto big_xattn = [&](int L) -> int {
    const int i = L / 4;
    if (i == 1 && xpart)
      return case_cross_attn_part(a->q2, a->Kx[L], a->xcount, a->xprefix, B, W, a->S[1], a->xslots, a->part_ml, a->part_acc,
                                  st);
    return case_cross_attn_partial_tc(a->q2, a->Kx[L], a->mask[i], B, W, a->S[i], a->nsplit_x[i], a->part_ml,
                                      a->part_acc, st);
  };
  auto nparts_of = [&](int L) -> int { return (L / 4 == 1 && xpart) ? a->xslots : a->nsplit_x[L / 4]; };
  const bool chain = dt == CASE_BF16 && !(opt & CASE_OPT_NO_CHAIN) && a->layers[0].Wc != nullptr && a->Tmax <= case_layer_chain_max_tmax();
  if (chain) {
    // Cluster kernels: [embed + front 0] x [back 0 + front 1] x ... x [back 7], one launch between
    // cross-attentions.  The two additive attentions only feed the mixture gates and the copy scatter,
    // so they run on a side stream: attns[0] beside the whole second stack, attns[1] beside norm1 ->
    // gen.0 -> vocabulary GEMM (fork/join by events, captured into the graph like any other edge).
    const bool fork = !(opt & CASE_OPT_NO_FORK) && a->fork != nullptr && a->h0 != nullptr && a->qa1 != nullptr;
    cudaStream_t aux = fork ? a->fork->aux : st;
    cudaEvent_t* ev_fork = fork ? a->fork->ev_fork : nullptr;
    cudaEvent_t* ev_join = fork ? a->fork->ev_join : nullptr;
    // the whole first stack (4 layers over the S0 <= 64 keys of the query memory, cross-attention included)
    // plus the first half-layer of the second stack is ONE launch; otherwise one launch per half-layer pair
    const bool stack0 = !(opt & CASE_OPT_NO_STACK) && a->S[0] <= case_layer_chain_max_s0();
    // attention queries, norm1 and gen.0 ride on the cluster launches as post linears (no row_linear launches)
    const bool post = !(opt & CASE_OPT_NO_POST) && a->Wqa_c[0] != nullptr && a->Wqa_c[1] != nullptr && a->Wg_c != nullptr;
    auto qa_post = [&](int i, float* out) {
      case_chain_post_t p;
      memset(&p, 0, sizeof(p));
      p.npost = 1; p.W = W; p.feat = a->feat;
      p.lin[0].Wc = a->Wqa_c[i]; p.lin[0].bias = a->bqa[i]; p.lin[0].out = out; p.lin[0].nchunk = 2;
      p.lin[0].seg[0] = CASE_SEG_H; p.lin[0].seg[1] = CASE_SEG_FEAT;
      return p;
    };
    int Lstart = 0;
    if (stack0) {
      float* hdst0 = fork ? a->h0 : a->h;
      void* kcs[5]; void* vcs[5]; const void* kxs[4];
      for (int l = 0; l < 5; ++l) { kcs[l] = a->kcache[l]; vcs[l] = a->vcache[l]; }
      for (int l = 0; l < 4; ++l) kxs[l] = a->Kx[l];
      case_chain_post_t p0 = qa_post(0, a->qa);
      TRY(case_layer_stack(a->layers, 4, kcs, vcs, kxs, a->mask[0], W, a->S[0], nullptr, a->E, a->pe, 16.0f, a->x_in, hdst0,
                           anc, TL, a->tok, TL, a->prow, t, a->Tmax, a->bbuf, a->q2, R, 1, post ? &p0 : nullptr, st));
      if (fork) {
        CUTRY(cudaEventRecord(ev_fork[0], st));
        CUTRY(cudaStreamWaitEvent(aux, ev_fork[0], 0));
        TRY(stack_attention(0, hdst0, a->qa, aux, post));
        CUTRY(cudaEventRecord(ev_join[0], aux));
      } else {
        TRY(stack_attention(0, hdst0, a->qa, st, post));
      }
      TRY(big_xattn(4));
      Lstart = 5;
    }
    for (int L = Lstart; L <= 8; ++L) {
      const case_layer_weights_t* wb = L > 0 ? &a->layers[L - 1] : nullptr;
      const case_layer_weights_t* wf = L < 8 ? &a->layers[L] : nullptr;
      float* hdst = (L == 4 && fork) ? a->h0 : a->h;
      case_chain_post_t pl;
      memset(&pl, 0, sizeof(pl));
      if (post && L == 4) pl = qa_post(0, a->qa);
      if (post && L == 8) {
        pl = qa_post(1, fork ? a->qa1 : a->qa);
        pl.npost = 2; pl.x_in = a->x_in; pl.ln_g = a->lnN_g; pl.ln_b = a->lnN_b; pl.ln_out = a->hN;
        pl.lin[1].Wc = a->Wg_c; pl.lin[1].bias = a->bg; pl.lin[1].out = a->gfeat; pl.lin[1].nchunk = 3;
        pl.lin[1].seg[0] = CASE_SEG_XIN; pl.lin[1].seg[1] = CASE_SEG_HLN; pl.lin[1].seg[2] = CASE_SEG_FEAT;
      }
      TRY(case_layer_chain(wb, wf, nullptr, a->E, a->pe, 16.0f /* sqrt(256) */, a->x_in, a->bbuf, a->part_ml,
                           a->part_acc, L > 0 ? nparts_of(L - 1) : 1, hdst, wf ? a->kcache[L] : nullptr,
                           wf ? a->vcache[L] : nullptr, anc, TL, a->tok, TL, a->prow, t, a->Tmax, a->bbuf, a->q2, R,
                           L == 0, pl.npost ? &pl : nullptr, st));
      if (L == 4 || L == 8) {
        const int i = L / 4 - 1;
        if (fork) {
          CUTRY(cudaEventRecord(ev_fork[i], st));
          CUTRY(cudaStreamWaitEvent(aux, ev_fork[i], 0));
          TRY(stack_attention(i, hdst, i == 0 ? a->qa : a->qa1, aux, post));
          CUTRY(cudaEventRecord(ev_join[i], aux));
        } else {
          TRY(stack_attention(i, hdst, a->qa, st, post));
        }
      }
      if (L == 8) break;
      TRY(big_xattn(L));
    }
    if (!post) {
      TRY(case_layernorm_rows(a->h, a->lnN_g, a->lnN_b, a->hN, R, st));
      TRY(gen0());
    }
    TRY(case_vocab_gemm(a->gfeat, a->Wv, nullptr, a->logits, R, a->V, a->ldv, dt, a->vocab_impl, a->vocab_ws, st));
    if (sparse) TRY(case_vocab_base(a->logits, a->ldv, R, a->V, 0, k2b, a->base_ms, a->base_e, a->base_i, st));
    if (fork) {
      CUTRY(cudaStreamWaitEvent(st, ev_join[0], 0));
      CUTRY(cudaStreamWaitEvent(st, ev_join[1], 0));
    }
  } else {
  TRY(case_embed_rows(a->E, a->pe, a->tok, TL, t, 16.0f /* sqrt(256) */, a->x_in, R, st));
  const float* hin = a->x_in;
  for (int i = 0; i < 2; ++i) {
    for (int l = 0; l < 4; ++l) {
      const int L = i * 4 + l;
      TRY(case_layer_front(hin, &a->layers[L], a->kcache[L], a->vcache[L], anc, TL, a->tok, TL, t, a->Tmax,
                           a->bbuf, a->q2, R, dt, st));
      int nparts = nparts_of(L);
      if (dt == CASE_BF16) {   // tensor-core tiles (Kx holds the interleaved K|V tiles)
        TRY(big_xattn(L));
      } else {
        TRY(case_cross_attn_partial(a->q2, a->Kx[L], a->Vx[L], a->mask[i], B, W, a->S[i], a->nsplit_x[i],
                                    a->part_ml, a->part_acc, dt, st));
      }
      TRY(case_layer_back(a->bbuf, a->part_ml, a->part_acc, nparts, &a->layers[L], a->h, R, dt, st));
      hin = a->h;
    }
    TRY(stack_attention(i, a->h, a->qa, st));
  }
  TRY(case_layernorm_rows(a->h, a->lnN_g, a->lnN_b, a->hN, R, st));
  TRY(gen0());
  TRY(case_vocab_gemm(a->gfeat, a->Wv, nullptr, a->logits, R, a->V, a->ldv, dt, a->vocab_impl, a->vocab_ws, st));
  if (sparse) TRY(case_vocab_base(a->logits, a->ldv, R, a->V, 0, k2b, a->base_ms, a->base_e, a->base_i, st));
  }
  if (sparse || (use_tail && n_oov == 0 && a->V <= case_row_tail_max_vocab())) {
    // one launch: attention merge + gates, softmax x gate, both copy scatters, top-k; the [R, V]
    // distribution is written only for the `generate` face
    case_tail_args_t ta;
    memset(&ta, 0, sizeof(ta));
    ta.R = R; ta.V = a->V; ta.W = W; ta.K = W; ta.ldl = a->ldv; ta.ldd = a->ldv; ta.mask_col0 = 0; ta.nmem = 2;
    ta.do_finalize = 1; ta.fac_ld = 2 * CASE_MAX_SPLIT; ta.map_ld = a->map_ld;
    ta.logits = a->logits; ta.hN = a->hN; ta.Wm = a->Wm; ta.bm = a->bm; ta.gates = a->gates; ta.fac = a->fac;
    ta.map = a->map;
    for (int i = 0; i < 2; ++i) {
      ta.ns[i] = a->nsplit_a[i]; ta.fac_off[i] = i * CASE_MAX_SPLIT; ta.map_off[i] = a->map_off[i]; ta.S[i] = a->S[i];
      ta.stats[i] = a->stats[i]; ta.ctxp[i] = a->ctxp[i]; ta.ctx[i] = a->ctx[i]; ta.prior[i] = a->prior[i];
      ta.attn_un[i] = a->attn_un[i];
    }
    if (a->materialize_only) { ta.dist = a->dist; } else { ta.top_vals = a->top_vals; ta.top_idx = a->top_idx; }
    ta.gate_ctx = gate ? 1 : 0;
    ta.Vext = n_oov ? Vx : 0;
    if (sparse && !(opt & CASE_OPT_NO_COPY_PLAN) && a->cp_n != nullptr) {
      ta.cp_n = a->cp_n; ta.cp_uid = a->cp_uid; ta.cp_first = a->cp_first; ta.cp_start = a->cp_start; ta.cp_perm = a->cp_perm;
      ta.cp_ld = a->cp_ld;
    }
    if (attr) ta.attr = a->attr_cand;
    if (sparse) {
      const bool fuse_sel = a->qcount != nullptr && !(opt & CASE_OPT_NO_FUSED_SELECT);
      case_select_args_t sel = select_args(a->mode, B, W, t, a->max_len, a->Tmax, a->BOS, a->EOS, a->UNK, a->PAD,
                                           a->top_vals, a->top_idx, a->live, a->cum, a->length, a->tok, a->anc, a->parent,
                                           a->ended, a->best_key, a->best_len, a->out_tokens, a->n_live, a->nbest);
      if (n_oov) { sel.V_in = a->V; sel.tok_ext = a->tok_ext; }
      set_select_attr(sel, a->attr_cand, a->attr_hist, a->out_attr);
      set_tail_constr(ta, n_oov ? a->tok_ext : a->tok, anc, TL, t, a->EOS, a->no_repeat_ngram, a->min_len, a->ban_mask,
                      a->ban_tok, a->ban_len, a->ban_n);
      TRY(case_sparse_tail(&ta, a->base_ms, a->base_e, a->base_i, k2b, fuse_sel ? &sel : nullptr, a->qcount, st));
      if (fuse_sel) return 0;
    } else {
      TRY(case_row_tail(&ta, st));
    }
    if (a->materialize_only) return 0;
  } else {
    TRY(finalize());
    TRY(case_softmax_mix(a->logits, a->ldv, a->gates, a->dist, a->ldv, R, a->V, 0, st));
    if (n_oov)      // the dynamic columns start from zero: they only ever receive copy mass
      CUTRY(cudaMemset2DAsync(a->dist + a->V, (size_t)a->ldv * sizeof(float), 0, (size_t)n_oov * sizeof(float), R, st));
    for (int i = 0; i < 2; ++i) {
      TRY(case_copy_scatter(a->map, a->map_ld, a->map_off[i], a->prior[i], a->attn_un[i],
                            a->fac + (size_t)i * CASE_MAX_SPLIT, 2 * CASE_MAX_SPLIT, a->dist, a->ldv, B, W, a->S[i],
                            Vx, st));
    }
    if (a->materialize_only) return 0;
    TRY(case_topk_rows(a->dist, a->ldv, R, Vx, W, a->top_vals, a->top_idx, st));
  }
  {
    case_select_args_t sel = select_args(a->mode, B, W, t, a->max_len, a->Tmax, a->BOS, a->EOS, a->UNK, a->PAD, a->top_vals,
                                         a->top_idx, a->live, a->cum, a->length, a->tok, a->anc, a->parent, a->ended,
                                         a->best_key, a->best_len, a->out_tokens, a->n_live, a->nbest);
    if (n_oov) { sel.V_in = a->V; sel.tok_ext = a->tok_ext; }
    set_select_attr(sel, a->attr_cand, a->attr_hist, a->out_attr);
    return case_beam_select(&sel, st);
  }
}

// gh = Whh . h_prev + bhh (GRU hidden-side gates, GTTP/Model.py:124-126): depends on the previous state only
static int gttp_hidden_gates(const gttp_step_args_t* a, const float* s_in, int R, int dt, cudaStream_t st) {
  case_rowlin_args_t hh;
  memset(&hh, 0, sizeof(hh));
  hh.seg[0] = seg(s_in, H, H, 1, 1);
  hh.nseg = 1; hh.K = H; hh.Wt = a->Whh_t; hh.bias = a->bhh; hh.N = 3 * H; hh.out = a->gh; hh.ldo = 3 * H;
  hh.gather_idx = a->parent; hh.R = R; hh.dtype = dt;
  return case_row_linear(&hh, st);
}

extern "C" int gttp_decode_step(const gttp_step_args_t* a, int t, case_stream_t stream) {
  CB_REQUIRE(a, "gttp_decode_step: null args");
  CB_REQUIRE(a->R == a->B * a->W && a->W >= 1 && a->W <= CASE_MAX_W, "gttp_decode_step: R != B*W or W out of range");
  CB_REQUIRE(t >= 0 && t < a->Tmax && a->Tmax <= CASE_MAX_T, "gttp_decode_step: t out of range");
  TRY(check_nbest(a->nbest, a->W, a->mode));
  cudaStream_t st = (cudaStream_t)stream;
  const int R = a->R, B = a->B, W = a->W, TL = a->Tmax + 1, dt = a->dtype;
  const float* s_in = a->state[t & 1];
  float* s_out = a->state[(t + 1) & 1];
  const int opt = a->opt;
  OptScope scope(opt);
  const int use_tail = (opt & CASE_OPT_UNFUSED_TAIL) ? 0 : 1;
  // search path: the sparse tail of the CaSE step (base statistics of the logits + the copy mass hashed by vocabulary id,
  // accumulated in fixed point: the top-k never needs the [R, V] mixture and is reproducible run to run)
  const int k2 = 2 * W <= 2 * CASE_MAX_W ? 2 * W : 2 * CASE_MAX_W;
  const bool sparse = use_tail && !(opt & CASE_OPT_DENSE_TAIL) && !a->materialize_only && a->base_ms && a->base_e && a->base_i &&
                      a->V >= k2 && a->Lb <= case_sparse_tail_max_sources();
  TRY(check_step_attr(a->attr_cand, a->attr_hist, a->out_attr, sparse, "gttp_decode_step"));
  TRY(check_step_constr(a->no_repeat_ngram, a->min_len, a->mode, a->max_len, a->V, W, a->Tmax, sparse, "gttp_decode_step"));
  TRY(check_step_bans(a->ban_mask, a->ban_tok, a->ban_len, a->ban_n, a->mode, a->V, W, a->Tmax, sparse, "gttp_decode_step"));
  const int k2b = (a->no_repeat_ngram || a->min_len || a->ban_mask) ? 2 * CASE_MAX_W : k2;   // as in case_decode_step

  TRY(case_embed_rows(a->E, nullptr, a->tok, TL, t, 1.0f, a->emb, R, st));
  // two additive attentions with the previous GRU state as query (GTTP/Model.py:117-122)
  const void* Wq[2] = {a->Wqs_t, a->Wqb_t};
  const float* bq[2] = {a->bqs, a->bqb};
  const float* vv[2] = {a->vs, a->vb};
  const void* U[2] = {a->Us, a->Ub};
  const void* M[2] = {a->Ms, a->Mb};
  const uint8_t* mk[2] = {a->mask_c, a->mask_b};
  const int L[2] = {a->Lc, a->Lb};
  const int ns[2] = {a->nsplit_c, a->nsplit_b};
  // the two attentions are independent: with a fork handle the (short) context memory runs on the side stream beside the
  // background memory; the join is an event edge before the GRU cell (captured into the graph like any other edge)
  const bool fork = !(opt & CASE_OPT_NO_FORK) && a->fork != nullptr && a->qa1 != nullptr;
  if (fork) {
    int dev = -1;
    CUTRY(cudaGetDevice(&dev));
    CB_REQUIRE(dev == a->fork->device, "gttp_decode_step: the fork handle was created on another device");
    CUTRY(cudaEventRecord(a->fork->ev_fork[0], st));
    CUTRY(cudaStreamWaitEvent(a->fork->aux, a->fork->ev_fork[0], 0));
  }
  for (int i = 0; i < 2; ++i) {
    cudaStream_t si = (fork && i == 0) ? a->fork->aux : st;
    float* qbuf = (fork && i == 0) ? a->qa1 : a->qa;
    case_rowlin_args_t q;
    memset(&q, 0, sizeof(q));
    q.seg[0] = seg(s_in, H, H, 1, 1);
    q.nseg = 1; q.K = H; q.Wt = Wq[i]; q.bias = bq[i]; q.N = H; q.out = qbuf; q.ldo = H;
    q.gather_idx = a->parent; q.R = R; q.dtype = dt;
    TRY(case_row_linear(&q, si));
    TRY(case_additive_attn(qbuf, U[i], M[i], vv[i], mk[i], nullptr, nullptr, 0, t, B, W, L[i], 2 * H, ns[i],
                           a->attn_un[i], a->stats[i], a->ctxp[i], a->fast_tanh, dt, si));
    TRY(case_attn_merge(a->stats[i], a->ctxp[i], ns[i], 2 * H, a->ctx[i], i == 1 ? a->fac : nullptr, CASE_MAX_SPLIT,
                        R, si));
  }
  if (fork) {
    TRY(gttp_hidden_gates(a, s_in, R, dt, a->fork->aux));          // the side stream has time to spare: the GRU's hidden-side gates
    CUTRY(cudaEventRecord(a->fork->ev_join[0], a->fork->aux));
    CUTRY(cudaStreamWaitEvent(st, a->fork->ev_join[0], 0));
  }
  {  // GRU cell on [emb ; src_ctx ; bg_ctx]   (Model.py:124-126)
    case_rowlin_args_t g;
    memset(&g, 0, sizeof(g));
    g.seg[0] = seg(a->emb, H, H, 1);
    g.seg[1] = seg(a->ctx[0], 2 * H, 2 * H, 1);
    g.seg[2] = seg(a->ctx[1], 2 * H, 2 * H, 1);
    g.nseg = 3; g.K = 5 * H; g.Wt = a->Wih_t; g.bias = a->bih; g.N = 3 * H; g.out = a->gi; g.ldo = 3 * H;
    g.R = R; g.dtype = dt;
    TRY(case_row_linear(&g, st));
    if (!fork) TRY(gttp_hidden_gates(a, s_in, R, dt, st));
    TRY(case_gru_cell(a->gi, a->gh, s_in, a->parent, s_out, R, st));
  }
  {  // readout on [emb ; h' ; src_ctx ; bg_ctx]   (Model.py:128-130)
    case_rowlin_args_t r;
    memset(&r, 0, sizeof(r));
    r.seg[0] = seg(a->emb, H, H, 1);
    r.seg[1] = seg(s_out, H, H, 1);
    r.seg[2] = seg(a->ctx[0], 2 * H, 2 * H, 1);
    r.seg[3] = seg(a->ctx[1], 2 * H, 2 * H, 1);
    r.nseg = 4; r.K = 6 * H; r.Wt = a->Wr_t; r.bias = a->br; r.N = H; r.out = a->feat; r.ldo = H;
    r.R = R; r.dtype = dt;
    TRY(case_row_linear(&r, st));
  }
  TRY(case_vocab_gemm(a->feat, a->Wv, a->bv, a->logits, R, a->V, a->ldv, dt, a->vocab_impl, a->vocab_ws, st));
  TRY(case_gttp_gates(a->feat, a->wc, a->bc, a->gates, a->fac, CASE_MAX_SPLIT, ns[1], R, st));
  if (sparse) {
    TRY(case_vocab_base(a->logits, a->ldv, R, a->V, 1, k2b, a->base_ms, a->base_e, a->base_i, st));
    case_tail_args_t ta;
    memset(&ta, 0, sizeof(ta));
    ta.R = R; ta.V = a->V; ta.W = W; ta.K = W; ta.ldl = a->ldv; ta.ldd = a->ldv; ta.mask_col0 = 1; ta.nmem = 1;
    ta.do_finalize = 0; ta.fac_ld = CASE_MAX_SPLIT; ta.map_ld = a->map_ld;
    ta.logits = a->logits; ta.gates = a->gates; ta.fac = a->fac; ta.map = a->map;
    ta.S[0] = a->Lb; ta.attn_un[0] = a->attn_un[1];
    ta.top_vals = a->top_vals; ta.top_idx = a->top_idx;
    ta.attr = a->attr_cand;
    set_tail_constr(ta, a->tok, a->anc[t & 1], TL, t, a->EOS, a->no_repeat_ngram, a->min_len, a->ban_mask, a->ban_tok,
                    a->ban_len, a->ban_n);
    TRY(case_sparse_tail(&ta, a->base_ms, a->base_e, a->base_i, k2b, nullptr, nullptr, st));
  } else if (use_tail && a->V <= case_row_tail_max_vocab()) {
    case_tail_args_t ta;
    memset(&ta, 0, sizeof(ta));
    ta.R = R; ta.V = a->V; ta.W = W; ta.K = W; ta.ldl = a->ldv; ta.ldd = a->ldv; ta.mask_col0 = 1; ta.nmem = 1;
    ta.do_finalize = 0; ta.fac_ld = CASE_MAX_SPLIT; ta.map_ld = a->map_ld;
    ta.logits = a->logits; ta.gates = a->gates; ta.fac = a->fac; ta.map = a->map;
    ta.S[0] = a->Lb; ta.attn_un[0] = a->attn_un[1];
    if (a->materialize_only) { ta.dist = a->dist; } else { ta.top_vals = a->top_vals; ta.top_idx = a->top_idx; }
    TRY(case_row_tail(&ta, st));
    if (a->materialize_only) return 0;
  } else {
    TRY(case_softmax_mix(a->logits, a->ldv, a->gates, a->dist, a->ldv, R, a->V, 1, st));
    TRY(case_copy_scatter(a->map, a->map_ld, 0, nullptr, a->attn_un[1], a->fac, CASE_MAX_SPLIT, a->dist, a->ldv, B, W,
                          a->Lb, a->V, st));
    if (a->materialize_only) return 0;
    TRY(case_topk_rows(a->dist, a->ldv, R, a->V, W, a->top_vals, a->top_idx, st));
  }
  case_select_args_t sel = select_args(a->mode, B, W, t, a->max_len, a->Tmax, a->BOS, a->EOS, a->UNK, a->PAD, a->top_vals,
                                       a->top_idx, a->live, a->cum, a->length, a->tok, a->anc, a->parent, a->ended,
                                       a->best_key, a->best_len, a->out_tokens, a->n_live, a->nbest);
  set_select_attr(sel, a->attr_cand, a->attr_hist, a->out_attr);
  return case_beam_select(&sel, st);
}

/* layout self-check for FFI bindings: sizeof of each argument struct, by index */
extern "C" size_t case_struct_size(int which) {
  switch (which) {
    case 0: return sizeof(case_seg_t);
    case 1: return sizeof(case_rowlin_args_t);
    case 2: return sizeof(case_layer_weights_t);
    case 3: return sizeof(case_select_args_t);
    case 4: return sizeof(case_step_args_t);
    case 5: return sizeof(gttp_step_args_t);
    case 6: return sizeof(case_tail_args_t);
    case 7: return sizeof(case_chain_post_t);
    default: return 0;
  }
}
