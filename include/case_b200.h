/*
 * case_b200.h - C ABI of libcase_b200.so: the B200 (sm_100a) kernels behind the CaSE_RG
 * answer-decode hot path.
 *
 * The reference (PengjieRen/CaSE_RG) is pure Python/PyTorch and has no FFI of its own; the
 * drop-in boundary is the Python module face (CaSE/Model.py:50,125; GTTP/EncDecModel.py:11-42).
 * This header is the layer *under* that face: what a maintainer binds (ctypes / cffi / a torch
 * custom op) to replace the ATen calls of the reference's per-step decoder.  Each entry point
 * names the reference code it replaces.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller; nothing here allocates or frees;
 *  - launch-only: functions enqueue work on `stream` and return immediately (no sync);
 *  - return value: 0 on success, otherwise a cudaError_t (or CASE_EINVAL for bad arguments);
 *    case_last_error() gives a static message for the calling thread;
 *  - no process-global state: launchers are re-entrant and work on the calling thread's CURRENT device; per-kernel
 *    device attributes are set up per device on first use;
 *  - `dtype` selects the storage type of caches and weight matrices: CASE_F32 or CASE_BF16.
 *    Activations, softmax statistics and distributions are always fp32;
 *  - hidden size is fixed at 256 with 8 heads of 32 (CaSE/Model.py:261-265, Run.py:71);
 *  - rows: R = B * W, row r = b * W + w (query b, beam slot w).
 */
#ifndef CASE_B200_H
#define CASE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CASE_H 256
#define CASE_NH 8
#define CASE_HD 32
#define CASE_MAX_W 8
#define CASE_MAX_T 128
#define CASE_MAX_SPLIT 16   /* additive-attention key splits */
#define CASE_MAX_XSPLIT 64  /* cross-attention partials per (row, head) */
#define CASE_MAX_BAN_SEQ 256 /* banned sequences of length >= 2 (case_tail_args_t.ban_tok rows) */
#define CASE_MAX_BAN_LEN 16  /* tokens per banned sequence (case_tail_args_t.ban_tok columns) */

#define CASE_F32 0
#define CASE_BF16 1
#define CASE_EINVAL 100001

typedef void* case_stream_t; /* cudaStream_t */

/* Attribution record of one answer token y chosen from the mixture of its parent prefix (CaSE/Model.py:38-48,
 * GTTP/Model.py:25-43): part[0] = g0 * softmax(logits)[y] (generation; 0 for dynamic ids >= V and GTTP's masked id 0),
 * part[1] / part[2] = copy mass of y from memory 0 / memory 1 (CaSE: query / passages; GTTP: part[1] = the background,
 * part[2] = 0).  The parts sum to the mixture probability p(y).  source = the source position s (index of the
 * concatenated copy map [memory 0 ; memory 1]) with the largest single contribution gate_i * p_i[s] among positions with
 * map[s] == y, exact ties to the lowest s; -1 when no position contributes.  The zero record has source -1. */
typedef struct {
  float part[3];
  int32_t source;
} case_attr_t;

/* select modes (case_beam_select) */
#define CASE_MODE_MODULE_GREEDY 0 /* CaSE/Model.py:119-122: argmax, no EOS handling          */
#define CASE_MODE_PROTO_GREEDY 1  /* Generations.py:96-107: EOS->UNK at t0, PAD after the end */
#define CASE_MODE_BEAM 2          /* Generations.py:136-185                                   */

int case_abi_version(void);
const char* case_last_error(void);
/* sizeof() of the argument structs below, for binding self-checks: 0 case_seg_t, 1 case_rowlin_args_t,
 * 2 case_layer_weights_t, 3 case_select_args_t, 4 case_step_args_t, 5 gttp_step_args_t, 6 case_tail_args_t,
 * 7 case_chain_post_t */
size_t case_struct_size(int which);

/* ---------------------------------------------------------------- options and per-engine handles
 * The library keeps NO process-global state: every launcher is re-entrant, two engines on two host threads (or two
 * devices) never see each other.  What used to be library switches are bits of an option word carried by the step
 * argument blocks (case_step_args_t.opt / gttp_step_args_t.opt); 0 = the default fast path, a set bit switches one
 * feature OFF (A/B measurements, fallbacks under test). */
#define CASE_OPT_NO_PDL 0x001          /* no programmatic dependent launch attribute on the kernels                 */
#define CASE_OPT_NO_CHAIN 0x002        /* bf16: row-block layer kernels (case_layer_front / _back) instead of the
                                          cluster kernels (case_layer_chain / case_layer_stack)                      */
#define CASE_OPT_NO_STACK 0x004        /* no fusion of the first stack into one case_layer_stack launch              */
#define CASE_OPT_NO_FORK 0x008         /* additive attentions on the main stream even when a fork handle is given    */
#define CASE_OPT_NO_POST 0x010         /* attention queries / norm1 / gen.0 as own launches, not as post linears     */
#define CASE_OPT_NO_GATE 0x020         /* context form of the additive attentions on the search path                 */
#define CASE_OPT_NO_EVICT_FIRST 0x040  /* no L2 evict-first policy on the once-per-step K|V / Uk.mem streams         */
#define CASE_OPT_DENSE_TAIL 0x080      /* case_row_tail instead of case_vocab_base + case_sparse_tail                */
#define CASE_OPT_UNFUSED_TAIL 0x100    /* finalize + softmax_mix + copy_scatter + topk_rows launches                 */
#define CASE_OPT_NO_FUSED_SELECT 0x200 /* case_beam_select as its own launch                                         */
#define CASE_OPT_NO_COPY_PLAN 0x400    /* ignore a copy plan in the step arguments (hash-table sparse tail)          */

/* Options of the CALLING THREAD for direct launcher calls (only CASE_OPT_NO_PDL and CASE_OPT_NO_EVICT_FIRST apply
 * to single launchers); returns the previous word, a negative argument only queries.  The step orchestrators ignore
 * this and use the option word of their argument block. */
int case_thread_options(int opt);

/* Side stream + events for the fork/join inside case_decode_step (the additive attentions run beside the layer
 * stack / the vocabulary GEMM).  Created on the CURRENT device, owned by the caller - one per engine - and passed in
 * case_step_args_t.fork (NULL = no fork).  The only host objects the library ever creates. */
typedef struct case_fork_s case_fork_t;
int case_fork_create(case_fork_t** out);
int case_fork_destroy(case_fork_t* f);

/* ---------------------------------------------------------------- row-wise building blocks */

/* x[r] = E[tok[r*tok_ld + t]] * sqrt(H) + pe[t]   (nn.Embedding + PositionalEmbedding,
 * CaSE/Model.py:96, common/PositionalEmbedding.py:44-48).  pe == NULL -> plain gather * scale. */
int case_embed_rows(const float* E, const float* pe, const int32_t* tok, int tok_ld, int t, float scale,
                    float* x, int R, case_stream_t stream);

/* y = LayerNorm(x) row-wise, eps 1e-5 (norm2(answer_rep), CaSE/Model.py:98). */
int case_layernorm_rows(const float* x, const float* g, const float* b, float* y, int R, case_stream_t stream);

/* Generic row linear: y[r,:] = act( cat_j seg_j[r / div_j] . Wt + bias ) + res[r,:]
 * (nn.Linear call sites: BilinearAttention.py:31, Model.py:34, GTTP/Model.py:124-131).
 * Wt is the nn.Linear weight [N][K] re-tiled to [N/256][K][256] ("n-tile major") in `dtype`, so the
 * 256 output columns one CTA produces read one contiguous run that is streamed as 16 KB tiles;
 * K = sum of segment widths, K%32==0, N%256==0.  act: 0 none, 1 gelu(erf).  */
typedef struct {
  const float* p;
  int32_t ld;
  int32_t width;
  int32_t div; /* row index = r / div (1 for per-row tensors, W for per-query tensors) */
  int32_t gather; /* 0: none; 1: row index taken from gather_idx[r] (GTTP state under reorder) */
} case_seg_t;

typedef struct {
  case_seg_t seg[4];
  int32_t nseg;
  int32_t K;
  const void* Wt;
  const float* bias;
  int32_t N;
  int32_t act;
  const float* res;
  int32_t ldres;
  float* out;
  int32_t ldo;
  const int32_t* gather_idx;
  int32_t R;
  int32_t dtype;
} case_rowlin_args_t;

int case_row_linear(const case_rowlin_args_t* a, case_stream_t stream);

/* ---------------------------------------------------------------- decoder layer (CaSE) */

/* Weights of one TransformerDecoderLayer (common/TransformerDecoder.py:43-59), matrices re-tiled
 * to [N/256][K][256] in `dtype` (see case_row_linear), vectors fp32.  Wq* and bq* are pre-multiplied
 * by 1/sqrt(hd). */
typedef struct {
  const void* Wqkv_t; const float* bqkv;   /* self_attn.in_proj  [H][3H] */
  const void* Wo_t;   const float* bo;     /* self_attn.out_proj [H][H]  */
  const void* Wq2_t;  const float* bq2;    /* multihead_attn.in_proj[:H] */
  const void* Wo2_t;  const float* bo2;    /* multihead_attn.out_proj    */
  const void* W1_t;   const float* b1;     /* linear1 */
  const void* W2_t;   const float* b2;     /* linear2 */
  const float* ln1_g; const float* ln1_b;
  const float* ln2_g; const float* ln2_b;
  const float* ln3_g; const float* ln3_b;
  const void* Wc;     /* bf16 only, may be NULL: the eight matrices "cluster-packed" for case_layer_chain */
} case_layer_weights_t;

/* First half of a layer for the newest position t of every row (TransformerDecoder.py:76-80):
 *   a = LN1(h); qkv = a.Wqkv; K/V -> self cache at (row r, position t);
 *   c = self-attention of q over positions 0..t of the row's ancestry (keys whose input token is
 *       PAD are masked, Model.py:106); h1 = a + c.Wo; b = LN2(h1); q2 = b.Wq2 (pre-scaled)
 * kcache/vcache: [R][Tmax][H] in dtype for this layer; anc: int32 [R][anc_ld] physical row that
 * holds position j of row r's history; tok: int32 [R][tok_ld] input token of (physical row, pos). */
int case_layer_front(const float* h, const case_layer_weights_t* w, void* kcache, void* vcache,
                     const int32_t* anc, int anc_ld, const int32_t* tok, int tok_ld, int t, int Tmax,
                     float* b_out, float* q2_out, int R, int dtype, case_stream_t stream);

/* Cross-attention of q2 over one memory, flash-decoding style (TransformerDecoder.py:81, K4):
 * Kmem/Vmem: [B][NH][S][HD] in dtype (projected once per query); mask: uint8 [B][S] 1 = valid key;
 * the W rows of query b share every K/V tile.  Writes per-(row, head, split) partials:
 * part_ml [R][NH][nsplit][2] (max, sum) and part_acc [R][NH][nsplit][HD]. */
int case_cross_attn_partial(const float* q2, const void* Kmem, const void* Vmem, const uint8_t* mask,
                            int B, int W, int S, int nsplit, float* part_ml, float* part_acc, int dtype,
                            case_stream_t stream);

/* Tensor-core form of the above for bf16 K/V (mma.sync m16n8k16 tiles, FlashAttention-2 style; the W
 * beam rows are the M rows of the tile).  Same outputs as case_cross_attn_partial: one partial per
 * (row, head, split).  KV holds K and V of a head interleaved tile by tile so that one 8 KB bulk copy
 * fetches a whole stage: bf16 [B][NH][ceil(S/64)][2 (K,V)][64 keys][32], keys >= S zero, and inside
 * every 64-byte key row the four 16-byte chunks are stored at position chunk ^ ((key >> 1) & 3). */
int case_cross_attn_partial_tc(const float* q2, const void* KV, const uint8_t* mask, int B, int W, int S,
                               int nsplit, float* part_ml, float* part_acc, case_stream_t stream);

/* Cross-attention over a COMPACTED memory (bf16): the prefill packs only the valid keys of every query,
 * contiguously, into the KV tile layout above (case_pack_kv_tiles_gather: padding keys contribute nothing
 * and key order does not matter), so queries own different numbers of tiles.  ncount: int32 [B] valid
 * keys per query; tile_prefix: int32 [B + 1] running sum of ceil(ncount / 64).  The (query, head, tile)
 * stream is cut into equal contiguous ranges, one per warp of a persistent grid (one CTA of 8 warps per
 * SM), so every SM streams the same number of tiles whatever the padding pattern.  Partials: part_ml
 * [R][NH][nslot][2], part_acc [R][NH][nslot][HD] with nslot >= case_cross_attn_part_slots(S); slots a
 * (query, head) does not use are written as (m = -inf, l = 0). */
int case_cross_attn_part(const float* q2, const void* KV, const int32_t* ncount, const int32_t* tile_prefix, int B,
                         int W, int S, int nslot, float* part_ml, float* part_acc, case_stream_t stream);
int case_cross_attn_part_slots(int S);
/* Prefill projections of one memory as ONE tcgen05 GEMM whose epilogue writes the consumers' layouts (replaces
 * projected-rows GEMM + case_pack_kv_tiles[_gather] + the Uk.mem GEMM; TransformerDecoder.py:81 and
 * BilinearAttention.py:34 recompute both at every step):
 *   out[l] (l < nl): the K|V tile stream of layer l, layout of case_cross_attn_partial_tc; with cidx / ncount (both
 *     or neither) tile (b, j) holds the keys cidx[b][64 j ..] and keys >= ncount[b] are zero, tiles past a query's
 *     last one are not written (as case_pack_kv_tiles_gather);
 *   U (may be NULL): bf16 [B][S][H] = mem . Uk^T at the ORIGINAL positions of all S keys.
 * mem: bf16 [B][S][H].  Wp: nl*4 (+2 with U) weight blocks of 128 output rows in the canonical layout of
 * case_vocab_gemm_tc (64 KB each): rows (layer, K|V, head, dim) = multihead_attn.in_proj_weight[H:] of the nl
 * layers, then the H rows of linear_key.weight.  bias: fp32 [nl*2*H] (in_proj_bias[H:]).  cidx must list ALL S
 * positions of a query (valid ones first).  CTA = 128 keys of one query x all column blocks; accumulators double
 * buffered in TMEM. */
int case_prefill_project_tc(const void* mem, const void* Wp, const float* bias, int B, int S, const int32_t* cidx,
                            const int32_t* ncount, int nl, void* const* out, void* U, case_stream_t stream);
/* kv as in case_pack_kv_tiles (bf16 rows); cidx: int32 [B][S], cidx[b][j] = original position of the j-th
 * valid key of query b (ascending); key slots >= ncount[b] are zero. */
int case_pack_kv_tiles_gather(const void* kv, int ldkv, int B, int S, const int32_t* cidx, const int32_t* ncount,
                              int nl, void* const* out, case_stream_t stream);

/* Prefill helper: the output rows of the memory K/V projection GEMM, kv [B*S][ldkv] (fp32 or bf16,
 * src_dtype) with columns (layer, K|V, head, dim), re-packed into the KV layout above for `nl` (<= 4)
 * layers; out[l] = that layer's buffer.  (The projection itself, TransformerDecoder.py:81, is a plain
 * GEMM done once per batch.) */
int case_pack_kv_tiles(const void* kv, int src_dtype, int ldkv, int B, int S, int nl, void* const* out,
                       case_stream_t stream);

/* Second half (TransformerDecoder.py:82-89): ctx = merge(partials); h2 = b + ctx.Wo2;
 * c = LN3(h2); h_out = c + W2.gelu(W1.c). */
int case_layer_back(const float* b_in, const float* part_ml, const float* part_acc, int nsplit,
                    const case_layer_weights_t* w, float* h_out, int R, int dtype, case_stream_t stream);

/* Post linears of a cluster launch: y = [segments] . W^T + bias evaluated on the rows that leave the LAST
 * back half of the launch, at the end of the launch (CaSE: the attention query [h ; norm2(answer_rep)],
 * Model.py:108, and gen.0 on [x_in ; norm1(h) ; norm2(answer_rep)], Model.py:115).  Wc: the nn.Linear
 * weight [256][256 * nchunk] cluster-packed per 256-column chunk: bf16 [4 ranks][nchunk][64 n][256 k], chunk
 * kc of row n at kc ^ (n & 7).  seg[j] names the input of chunk j. */
#define CASE_SEG_H 1     /* the rows themselves            */
#define CASE_SEG_HLN 2   /* LayerNorm(rows; ln_g, ln_b), also written to ln_out */
#define CASE_SEG_FEAT 3  /* feat[row / W]   ([B][H] fp32)  */
#define CASE_SEG_XIN 4   /* x_in[row]       ([R][H] fp32; only in launches without a front half) */
typedef struct {
  const void* Wc; const float* bias; float* out; int32_t nchunk; int32_t seg[3];
} case_post_linear_t;
typedef struct {
  int32_t npost, W;
  case_post_linear_t lin[2];
  const float* feat; const float* x_in; const float* ln_g; const float* ln_b; float* ln_out;
} case_chain_post_t;

/* Cluster form of the two calls above for bf16 storage: ONE launch runs the second half of layer Lb
 * (wb, may be NULL) followed by the first half of layer Lf (wf, may be NULL) for all rows, i.e. all row
 * work between two cross-attention launches (TransformerDecoder.py:82-89 of layer Lb, then :76-80 of
 * layer Lf).  A thread-block cluster of 4 CTAs owns 8 rows; CTA c owns columns [64c, 64c+64) of every
 * linear (= heads 2c, 2c+1) and ingests only its slice of the weights and of the KV history; results
 * are exchanged through distributed shared memory.  Needs w->Wc: bf16 [4 ranks][8 matrices Wq,Wk,Wv,
 * Wo,Wq2,Wo2,W1,W2][64 n][256 k] with the 16-byte chunk kc of row n stored at chunk position
 * kc ^ (n & 7) (Wq/Wq2 pre-scaled like Wqkv_t/Wq2_t).
 * Input rows: wb != NULL -> h_out of the back half (also written to global memory); else E != NULL ->
 * the embedding x = E[tok[r][t]] * emb_scale + pe[t] (case_embed_rows), also written to x_out; else h_in.
 * prow (int32 [R][Tmax], may be NULL): per-step table "physical row | masked bit" of every history
 * position; the launch with first = 1 (the first of a step: anc/tok were written by the launch right
 * before it) derives it from anc/tok and publishes it, later launches of the step read it early.
 * Tmax <= case_layer_chain_max_tmax() (the KV history of the 8 rows lives in shared memory).
 * post (may be NULL): post linears on the rows leaving the back half (see case_chain_post_t). */
int case_layer_chain(const case_layer_weights_t* wb, const case_layer_weights_t* wf, const float* h_in,
                     const float* E, const float* pe, float emb_scale, float* x_out, const float* b_in,
                     const float* part_ml, const float* part_acc, int nsplit, float* h_out, void* kcache,
                     void* vcache, const int32_t* anc, int anc_ld, const int32_t* tok, int tok_ld, int32_t* prow,
                     int t, int Tmax, float* b_out, float* q2_out, int R, int first, const case_chain_post_t* post,
                     case_stream_t stream);
int case_layer_chain_max_tmax(void);

/* A whole decoder stack over a SHORT memory in one cluster launch: for f = 0 .. nfused-1 the first half
 * of layers[f], the cross-attention over the S0 <= case_layer_chain_max_s0() keys of that memory (K|V
 * tiles kx[f] in the case_cross_attn_partial_tc layout, mask0 uint8 [B][S0], W rows per query) and the
 * second half of layers[f] - then the first half of layers[nfused], whose b_out / q2_out feed the next
 * (big) cross-attention launch.  Replaces 2 * nfused + 1 launches (CaSE: the whole query-memory stack,
 * TransformerDecoder.py:191-218 with num_layers = 4, plus the first half-layer of the passage stack).
 * Input rows as in case_layer_chain (h_in, or the embedding when E != NULL); h_fused_out (may be NULL)
 * receives the output rows of layer nfused-1, i.e. the stack output.  kcache / vcache: nfused + 1
 * pointers, kx: nfused pointers; all layers need Wc. */
int case_layer_stack(const case_layer_weights_t* layers, int nfused, void* const* kcache, void* const* vcache,
                     const void* const* kx, const uint8_t* mask0, int W, int S0, const float* h_in, const float* E,
                     const float* pe, float emb_scale, float* x_out, float* h_fused_out, const int32_t* anc,
                     int anc_ld, const int32_t* tok, int tok_ld, int32_t* prow, int t, int Tmax, float* b_out,
                     float* q2_out, int R, int first, const case_chain_post_t* post, case_stream_t stream);
int case_layer_chain_max_s0(void);

/* ---------------------------------------------------------------- additive ("bilinear") attention */

/* Fused score + softmax-partials + context partials (BilinearAttention.py:24-60, K6-K8):
 *   e[r,s] = v . tanh(qa[r] + U[b,s]),  -inf where !mask[b,s] or !rowvalid[r]
 * qa: [R][H] = Wq.query + b (from case_row_linear); U: [B][S][H] (= Uk.mem) and Mv: [B][S][DV]
 * (values) in dtype; prior: fp32 [B][S] or NULL (CaSE/Model.py:110).  rowvalid: row r is valid iff
 * tok[r*tok_ld + t] != 0 (tok == NULL -> all valid).
 * Outputs: attn_un [R][S] = the raw masked scores e; per key split stats [R][nsplit][4] =
 * (m = max e, sum exp(e-m), sum prior*exp(e-m), 0) and ctx_part [R][nsplit][DV] = sum exp(e-m)*Mv.
 * fast_tanh: 1 = tanh.approx.f32. */
int case_additive_attn(const float* qa, const void* U, const void* Mv, const float* v, const uint8_t* mask,
                       const float* prior, const int32_t* tok, int tok_ld, int t, int B, int W, int S, int DV,
                       int nsplit, float* attn_un, float* stats, float* ctx_part, int fast_tanh, int dtype,
                       case_stream_t stream);

/* case_additive_attn over the VALID keys only (bf16): cidx int32 [B][S] = positions of the valid keys of
 * every query (ascending), ncount int32 [B]; every key split of a query walks the same number of valid
 * keys, and qorder int32 [B] (may be NULL) launches the heaviest queries first.  attn_un of padding
 * positions is NOT written: the caller fills those entries with -inf once (they never change). */
int case_additive_attn_compact(const float* qa, const void* U, const void* Mv, const float* v, const uint8_t* mask,
                               const float* prior, const int32_t* tok, int tok_ld, int t, int B, int W, int S, int DV,
                               int nsplit, float* attn_un, float* stats, float* ctx_part, int fast_tanh,
                               const int32_t* cidx, const int32_t* ncount, const int32_t* qorder,
                               case_stream_t stream);

/* Gate form (bf16 keys) for CaSE's search path: the contexts m_i are read only by the 3-way mixture gate
 * softmax(W_m [h; m_0; m_1] + b_m) (CaSE/Model.py:39,117), which is linear in m_i, so the prefill projects
 * every key once to G fp32 [B][S][4] = (W_m[:, H(1+i):H(2+i)] . mem_i[b][s], 0) and the step accumulates
 * gate_part [R][nsplit][4] = sum exp(e-m) * G instead of ctx_part (no value rows are read).  attn_un and
 * stats as in case_additive_attn; cidx / ncount / qorder as in case_additive_attn_compact or all NULL.
 * nsq int32 [B] (may be NULL): query b uses only its first nsq[b] <= nsplit splits, so that every CTA of the
 * launch walks about the same number of keys; unused slots are written as empty partials (m = -inf). */
int case_additive_attn_gate(const float* qa, const void* U, const float* G, const float* v, const uint8_t* mask,
                            const float* prior, const int32_t* tok, int tok_ld, int t, int B, int W, int S,
                            int nsplit, float* attn_un, float* stats, float* gate_part, int fast_tanh,
                            const int32_t* cidx, const int32_t* ncount, const int32_t* qorder, const int32_t* nsq,
                            case_stream_t stream);

/* Prefill of the gate form: G fp32 [N][4] = (Wg[0..2] . mem[n], 0) for N key rows mem bf16 [N][H];
 * Wg fp32 [3][H] = W_m[:, H(1+i):H(2+i)] of memory i (CaSE/Model.py:36,39). */
int case_gate_project(const void* mem, const float* Wg, float* G, long long N, case_stream_t stream);
/* Split plan for case_additive_attn_gate: nsq[b] = clamp(ceil(count[b] / c), 1, max_split), c = max(ceil(sum(count)
 * / slots), ceil(max(count) / max_split)) rounded up to 32 keys: about `slots` equally long CTAs per launch. */
int case_split_plan(const int32_t* count, int B, int slots, int max_split, int32_t* nsq, case_stream_t stream);

/* CaSE row finaliser (Model.py:110-113, 39): hN = LN(h); merges both attentions' partials into
 * ctx0/ctx1, computes the mixture gates softmax(Wm.[hN;ctx0;ctx1]+bm) and, per memory i, the pair
 * (F_i, M_i) = fac[r][i][0..1] such that copy weight(r,i,s) = F_i * prior_i[b,s] * exp(e_i[r,s] - M_i)
 * equals gate_{i+1} * p_i[r,s] of the reference.  gates: [R][4], fac: [R][2][CASE_MAX_SPLIT]. */
int case_finalize_rows(const float* h, const float* lnN_g, const float* lnN_b, const float* stats0,
                       const float* ctxp0, int nsplit0, const float* stats1, const float* ctxp1, int nsplit1,
                       const float* Wm, const float* bm, float* hN, float* ctx0, float* ctx1, float* gates,
                       float* fac, int R, case_stream_t stream);

/* ---------------------------------------------------------------- vocabulary side */

/* logits[R][ldl] = f[R][H] . Wv[V][H]^T (+ bias)   (gen.2, Model.py:34 / gen.linear GTTP/Model.py:8).
 * impl 0: fp32-accumulate SIMT tile kernel, Wv = [V][H] row-major in dtype, workspace unused.
 * impl 1: tcgen05 tensor-core kernel (bf16 x bf16 -> fp32 in TMEM).  Wv = the weight re-packed into
 *   128-row tiles in the UMMA K-major no-swizzle canonical layout: element (v, k) at byte
 *   (v/128)*65536 + (k/8)*2048 + ((v%128)/8)*128 + (v%8)*16 + (k%8)*2, rows >= V zero
 *   (case_vocab_tc_packed_weight_bytes(V) bytes); workspace = case_vocab_tc_workspace_bytes(R) bytes
 *   (holds the bf16 re-pack of f), both 16-byte aligned. */
int case_vocab_gemm(const float* f, const void* Wv, const float* bias, float* logits, int R, int V, int ldl,
                    int dtype, int impl, void* workspace, case_stream_t stream);
int case_vocab_gemm_tc(const float* f, const void* Wp, const float* bias, float* logits, int R, int V, int ldl,
                       void* workspace, case_stream_t stream);
size_t case_vocab_tc_workspace_bytes(int R);
size_t case_vocab_tc_packed_weight_bytes(int V);

/* dist[r,v] = gates[r][0] * softmax(logits[r,:V])[v]; mask_col0 sets logit 0 to -inf first
 * (GTTP/Model.py:26).  (Softmax of Model.py:34 fused with the first term of Model.py:41.) */
int case_softmax_mix(const float* logits, int ldl, const float* gates, float* dist, int ldd, int R, int V,
                     int mask_col0, case_stream_t stream);

/* dist[r, map[b,s]] += F[r] * prior[b,s] * exp(e[r,s] - M[r])   with (F, M) = fac[r*fac_ld + 0..1]
 * (replaces the one-hot bmm of Model.py:43 / GTTP Model.py:37-40 and build_map Utils.py:344-355;
 * indices are used exactly as given, so targets are bit-exact).  prior may be NULL (=1); e = -inf
 * marks a masked source position. */
int case_copy_scatter(const int32_t* map, int map_ld, int map_off, const float* prior, const float* attn_un,
                      const float* fac, int fac_ld, float* dist, int ldd, int B, int W, int S, int V,
                      case_stream_t stream);

/* copy_topk's folding step (common/Utils.py:170-178) on an extended row gen [R][ldg] = [V vocabulary entries | D dynamic
 * entries]: vocab[v] += sum over d with vocab_map[q][d] == v of dyn[d]; dyn[d] *= overlap[q][d]  (q = r / rows_per_map:
 * the maps are per query, the rows per hypothesis).  vocab_map int32 [Q][D] is the index form of the reference's one-hot
 * [Q][D][V]; overlap fp32 [Q][D] (1 = the dynamic word is NOT in the vocabulary).  In place; follow with
 * case_topk_rows over V + D columns. */
int case_oov_fold(float* gen, int ldg, int R, int V, int D, const int32_t* vocab_map, const float* overlap,
                  int rows_per_map, case_stream_t stream);

/* Per-row top-k, values descending, ties -> lower index first (Utils.topk, Utils.py:156-168). */
int case_topk_rows(const float* dist, int ldd, int R, int V, int k, float* vals, int32_t* idx,
                   case_stream_t stream);

/* Fused tail of a step, one CTA per row with the row's distribution in shared memory:
 *   [do_finalize: case_finalize_rows without the LayerNorm (hN is an input)] -> case_softmax_mix ->
 *   case_copy_scatter for nmem memories -> case_topk_rows (k = K),
 * reading the logits once and never writing the [R, V] tile unless dist != NULL.  top_idx == NULL skips
 * the top-k (then dist must be given).  Without do_finalize, gates[r][0] and the (F, M) pairs
 * fac[r*fac_ld + fac_off[i] + 0..1] are inputs (GTTP: case_attn_merge + case_gttp_gates).
 * V <= case_row_tail_max_vocab(); logits rows 16-byte aligned, ldl >= V rounded up to 4. */
typedef struct {
  int32_t R, V, W, K, ldl, ldd, mask_col0, nmem, do_finalize, fac_ld, map_ld;
  int32_t ns[2], fac_off[2], map_off[2], S[2];
  const float* logits;
  const float* hN; const float* stats[2]; const float* ctxp[2]; const float* Wm; const float* bm;
  float* ctx[2]; float* gates; float* fac;
  const int32_t* map; const float* prior[2]; const float* attn_un[2];
  float* top_vals; int32_t* top_idx; float* dist;
  int32_t gate_ctx;   /* case_sparse_tail only: ctxp[i] hold gate_part [R][ns][4] of case_additive_attn_gate (ctx[i] unused) */
  /* case_sparse_tail only, optional copy plan of case_copy_plan (cp_n == NULL: hash table + atomics): per query
   * the unique vocabulary ids of its VALID source positions (ascending), cp_first = first position | (occurrences
   * - 1) << 16, cp_start = offset of the id's run in cp_perm, cp_perm = the valid positions sorted by (id, position);
   * positions index the concatenation [memory 0 ; memory 1]; rows of cp_ld ints */
  int32_t cp_ld;
  const int32_t* cp_n; const int32_t* cp_uid; const int32_t* cp_first; const int32_t* cp_start; const int32_t* cp_perm;
  /* case_sparse_tail only: extended vocabulary (pointer-generator OOV extension).  Vext > V: copy targets map[b][s] may
   * lie in [V, Vext) - per-query dynamic entries that have no logit, so their mixture value is the copy mass alone -
   * and the top-k indices range over [0, Vext).  0 = V (no extension). */
  int32_t Vext;
  /* case_sparse_tail only, may be NULL: attribution record (case_attr_t) of every top-k entry, [R][K] like top_vals.  The
   * copy parts are accumulated in the fixed point of the hash table, so in hash-table mode part[1] + part[2] is exactly the
   * copy mass the ranking used; with a copy plan they match it to rounding. */
  case_attr_t* attr;
  /* case_sparse_tail only: search constraints (no_repeat_ngram = min_len = 0: off, the fields below are ignored).
   * Row r is at step t (0 <= t < CASE_MAX_T) and its answer so far is y_1 .. y_t, position j held by
   * hist_tok[((j == t) ? r : hist_anc[r][j])][j] (rows of hist_ld >= t + 1 ints; the select's tok / tok_ext and anc_in).
   * no_repeat_ngram = n (1..CASE_MAX_T): an id y with (y_{t-n+2} .. y_t, y) already a contiguous n-gram of y_1 .. y_t
   * is banned; min_len = m (0..CASE_MAX_T-1): eos is banned while t < m.  Banned ids leave the candidate set and nothing
   * is renormalised: top_vals / top_idx are the exact top-K of the mixture restricted to the allowed ids.  Needs
   * V >= 2K + hist_ld, so K allowed ids always exist. */
  const int32_t* hist_tok;
  const int32_t* hist_anc;
  int32_t hist_ld, t, eos;
  int32_t no_repeat_ngram, min_len;
  /* case_sparse_tail only: banned words (all four or none; NULL = off).  Like the constraints above they need the answer
   * history (hist_tok, hist_anc, hist_ld, t) and remove ids from the candidate set without renormalising; the banned set
   * of a row is the union of every rule.
   *   ban_mask: uint32 [ceil(V / 32)], bit (id & 31) of word id >> 5 set = id (0 <= id < V) is never a candidate.
   *   ban_tok [CASE_MAX_BAN_SEQ][CASE_MAX_BAN_LEN], ban_len [CASE_MAX_BAN_SEQ], *ban_n = the number of sequences:
   *     sequence i = (w_1 .. w_L), L = ban_len[i], bans w_L at step t when t >= L - 1 and y_{t-L+2} .. y_t == w_1 .. w_{L-1}.
   * The content is read on the device at every launch (a captured graph serves every list): *ban_n is clamped to
   * [0, CASE_MAX_BAN_SEQ] and a sequence whose length lies outside [2, CASE_MAX_BAN_LEN] is skipped.  The caller keeps the
   * ids in [0, V) and at least 2K + hist_ld allowed ids per step: V - (ids of ban_mask) >= 2K + hist_ld + *ban_n. */
  const uint32_t* ban_mask;
  const int32_t* ban_tok;
  const int32_t* ban_len;
  const int32_t* ban_n;
} case_tail_args_t;
int case_row_tail(const case_tail_args_t* a, case_stream_t stream);
int case_row_tail_max_vocab(void);

/* Sparse form of the tail for the search path (never builds the [R, V] mixture): every id of the final
 * top-k is a copy target of the row or one of the top entries of the base softmax.
 * case_vocab_base: the row is cut into 4 quarters; per (row, quarter) base_ms[r][4][2] = (max logit, sum
 *   exp(l - max)) and the k2 (K <= k2 <= 16; use 2K) largest logits base_l[r][4][k2] with their ids
 *   base_i[r][4][k2] (value desc, index asc; -inf / out-of-range id = no entry).  Needs only the logits,
 *   so it can run beside the additive attention.
 * case_sparse_tail: same inputs/outputs as case_row_tail (top_vals / top_idx required, dist ignored)
 *   plus the base statistics; sum of S[i] <= case_sparse_tail_max_sources(). */
int case_vocab_base(const float* logits, int ldl, int R, int V, int mask_col0, int k2, float* base_ms,
                    float* base_l, int32_t* base_i, case_stream_t stream);
int case_sparse_tail_max_sources(void);

/* ---------------------------------------------------------------- search bookkeeping */

typedef struct {
  int32_t mode, B, W, t, max_len, Tmax;
  int32_t BOS, EOS, UNK, PAD;
  const float* top_vals;   /* [R][W] */
  const int32_t* top_idx;  /* [R][W] */
  int32_t* live;           /* [R]  1 = slot holds a live hypothesis                      */
  double* cum;             /* [R]  cumulative cost (Node.cum_cost, Generations.py:198)   */
  int32_t* length;         /* [R]  node count incl. BOS (Node.length :199)               */
  int32_t* tok;            /* [R][Tmax+1] input token of (physical row, position)        */
  const int32_t* anc_in;   /* [R][Tmax+1]                                                */
  int32_t* anc_out;        /* [R][Tmax+1]                                                */
  int32_t* parent;         /* [R] physical parent row of the hypothesis now in slot r    */
  int32_t* ended;          /* [B] proto-greedy: row has emitted EOS                      */
  double* best_key;        /* [B] beam: best finished cum/length so far (+inf initially) */
  int32_t* best_len;       /* [B] tokens in best_seq                                     */
  int32_t* out_tokens;     /* [B][Tmax] greedy: per-step token; beam: best sequence      */
  int32_t* n_live;         /* [B] live hypotheses per query after this step (early-exit hint) */
  /* extended vocabulary: a selected id >= V_in (> 0) is a per-query dynamic (OOV) entry; it is fed back to the decoder as
   * UNK (it has no embedding row) while tok_ext [R][Tmax+1] keeps the extended id for the returned sequences.
   * V_in = 0 / tok_ext = NULL: no extension (tok holds both). */
  int32_t V_in;
  int32_t* tok_ext;
  /* n-best list (beam mode, 1 <= nbest <= W): the nbest best finished hypotheses of every query instead of the best one,
   * i.e. sorted(results[q], key=cum_cost/length)[:nbest] of Generations.py:183-185 - keys ascending, equal keys in
   * finishing order (earlier step first, then the better rank within a step).  best_key [B][nbest] (+inf initially),
   * best_len [B][nbest] and out_tokens [B][nbest][Tmax] (PAD initially) hold the entries in rank order; entry 0 is the
   * answer of nbest = 1.  0 or 1: the single best, layouts as above. */
  int32_t nbest;
  /* attribution (all three or none; NULL = off): attr_cand [R][W] the records of the top-k entries (index as top_vals,
   * written by case_sparse_tail), attr_hist [R][Tmax+1] the record of the token at (physical row, position) next to tok,
   * out_attr the records of out_tokens, same layout ([B][Tmax], or [B][nbest][Tmax] for nbest > 1; zero records with
   * source -1 initially).  Greedy: an EOS rewritten to UNK at t = 0 keeps its record, PAD after the end gets the zero
   * record. */
  const case_attr_t* attr_cand;
  case_attr_t* attr_hist;
  case_attr_t* out_attr;
} case_select_args_t;

int case_beam_select(const case_select_args_t* a, case_stream_t stream);

/* case_sparse_tail (see the vocabulary section): sel != NULL fuses case_beam_select into the launch - the
 * last CTA of a query's W rows runs the bookkeeping of that query (k must equal W); qcount: int32 [B],
 * zero before the first launch (the kernel leaves it zero). */
int case_sparse_tail(const case_tail_args_t* a, const float* base_ms, const float* base_l, const int32_t* base_i,
                     int k2, const case_select_args_t* sel, int32_t* qcount, case_stream_t stream);

/* ---------------------------------------------------------------- GTTP step pieces */

/* nn.GRU cell, gate order r,z,n (GTTP/Model.py:125): gi = x.Wih+bih, gh = h.Whh+bhh given. */
int case_gru_cell(const float* gi, const float* gh, const float* h_prev, const int32_t* gather_idx,
                  float* h_out, int R, case_stream_t stream);

/* GTTP row finaliser: merges one attention's partials -> ctx [R][DV]; optionally (fac != NULL)
 * fac[r][0..1] = (1/Z, M) so that the normalised attention is fac[0] * exp(e - fac[1]) */
int case_attn_merge(const float* stats, const float* ctx_part, int nsplit, int DV, float* ctx, float* fac,
                    int fac_ld, int R, case_stream_t stream);

/* p_copy = sigmoid(wc.f + bc); gates[r] = (1-p_copy, p_copy, 0, 0); fac[r][0] *= p_copy
 * (GTTP/Model.py:31-41). */
int case_gttp_gates(const float* f, const float* wc, const float* bc, float* gates, float* fac, int fac_ld,
                    int nsplit, int R, case_stream_t stream);

/* ---------------------------------------------------------------- pre-decode producers (SURVEY.md 8f N1)
 * What CaSE.do_test runs before the decoder (CaSE/Model.py:313-331): the shared TransformerSeqEncoder
 * (common/TransformerSeqEncoderDecoder.py:14-45), Interaction (common/Interaction.py:15-76), the TransformerBlock stacks
 * of passage selection / supporting-token identification (common/TransformerBlock.py:22-33, CaSE/Model.py:127-215) and the
 * prior / answer representation of ResponseGeneration.action (CaSE/Model.py:230-245).  Rows = tokens, row-major; GEMM
 * operands bf16, accumulation / statistics / residual streams fp32. */

/* x[m] = E[tok[m]] * scale + pe[m % L]   (nn.Embedding + PositionalEmbedding over [N][L] token ids); x fp32 [M][256]. */
int case_enc_embed(const float* E, const float* pe, const int32_t* tok, long long M, int L, float scale, float* x,
                   case_stream_t stream);

/* LayerNorm (eps 1e-5) of (x + add) over rows of width C = 256 or 1280; x / add fp32 or bf16 (in_dtype), add may be
 * NULL; outputs: y16 bf16 and / or y32 fp32 (either may be NULL). */
int case_ln_rows_wide(const void* x, const void* add, int in_dtype, const float* g, const float* b, void* y16, float* y32,
                      long long M, int C, case_stream_t stream);

/* nn.MultiheadAttention self-attention with a key padding mask over nseq sequences of L tokens (TransformerEncoder.py:66,
 * TransformerBlock.py:27): qkv bf16 [nseq * L][3C] = in_proj output (Q | K | V column blocks), kmask uint8 [nseq * L]
 * (1 = valid key), out bf16 [nseq * L][C] (before out_proj).  C = 256 (heads of 32) or 1280 (heads of 160), 8 heads;
 * the 1/sqrt(head dim) scale is applied here.  FlashAttention-2 style on mma.sync, 64-query x 64-key tiles. */
int case_enc_attention(const void* qkv, const uint8_t* kmask, int nseq, int L, int C, int nhead, void* out,
                       case_stream_t stream);

/* Interaction.forward (common/Interaction.py:15-76) for B queries x NP passages without its [B*NP][Lp][Lq][3H] tensor:
 * Eq fp32 [B][Lq][256] (one query sequence per query), Ep fp32 [B*NP][Lp][256], masks uint8, w fp32 [768] =
 * dual_att_linear.weight.  Outputs: Gp bf16 [B*NP*Lp][1280] (G_q_p, PAD rows zero) and Gq bf16 [B*Lq][1280] (G_p_q after
 * the max over the passages).  Scratch: Gq_scratch fp32 [B*NP*Lq][1280].  Lq <= 64, any Lp: the five products run on
 * mma.sync over passage tiles of 64 rows and the score matrix is never stored (case_interaction_smem_bytes: six 64-row
 * bf16 operand buffers, 199 KB). */
int case_interaction(const float* Eq, const float* Ep, const uint8_t* qmask, const uint8_t* pmask, const float* w, int B,
                     int NP, int Lq, int Lp, float* Gq_scratch, void* Gq_out, void* Gp_out, case_stream_t stream);
size_t case_interaction_smem_bytes(int Lq, int Lp);

/* y[r] = w . x[r * row_stride] + b over fp32 rows of width 256 (the scorer Linear(H, 1): CaSE/Model.py:164, 203). */
int case_rows_dot(const float* x, const float* w, const float* b, long long nrows, long long row_stride, float* y,
                  case_stream_t stream);

/* prior[b][s] = sigmoid(pscore[b][s / Lp]) * sigmoid(tscore[b][s]) (0 at PAD: token scores are masked to -1e6 first),
 * normalised by 1e-8 + its sum; answer[b] = sum_s prior[b][s] * memp[b][s]   (CaSE/Model.py:205-206, 239-243). */
int case_prior_answer(const float* pscore, const float* tscore, const uint8_t* pmask, const float* memp, int B, int NP,
                      int Lp, float* prior, float* answer, case_stream_t stream);

/* Y[M][N] = mask_rows( act( X[M][K] . W[N][K]^T + bias ) + residual ) on tcgen05 / TMEM.  X bf16 row-major; Wp = the
 * nn.Linear weight packed per 64-wide K block into 256-row tiles of the UMMA K-major no-swizzle canonical layout (element
 * (n, k) of a tile at byte (k/8)*4096 + (n/8)*128 + (n%8)*16 + (k%8)*2; [K/64][N/256][32 KB],
 * case_gemm_rows_packed_weight_bytes); N % 256 == 0, K % 64 == 0; act: 0 none, 1 gelu (erf),
 * 2 relu; residual [M][N] fp32 / bf16 or NULL; row_mask uint8 [M] or NULL (masked rows are written as zeros); Y bf16 or
 * fp32 (y_dtype). */
int case_gemm_rows_tc(const void* X, const void* Wp, const float* bias, long long M, int N, int K, int act,
                      const void* residual, int residual_dtype, const uint8_t* row_mask, void* Y, int y_dtype,
                      case_stream_t stream);
size_t case_gemm_rows_packed_weight_bytes(int N, int K);

/* Feed-forward of a TransformerEncoderLayer / TransformerBlock in one launch (common/TransformerEncoder.py:73-76,
 * TransformerBlock.py:30-32):  Y[M][256] = mask_rows( act( X[M][K1] . W1^T + b1 ) . W2^T + b2 + residual ), hidden and output
 * width 256; X bf16 row-major, W1p / W2p packed as for case_gemm_rows_tc ([K1/64][1][32 KB] and [4][1][32 KB]); act: 1 gelu
 * (erf), 2 relu; residual [M][256] fp32 / bf16 or NULL; row_mask uint8 [M] or NULL; Y bf16 or fp32.  The hidden activations
 * stay in shared memory (they become the A operand of the second product in place). */
int case_ffn_rows_tc(const void* X, const void* W1p, const float* b1, int K1, int act, const void* W2p, const float* b2,
                     long long M, const void* residual, int residual_dtype, const uint8_t* row_mask, void* Y, int y_dtype,
                     case_stream_t stream);

/* ---------------------------------------------------------------- whole-step orchestrators */

typedef struct {
  int32_t B, W, R, V, ldv, Tmax, dtype, fast_tanh, vocab_impl, mode;
  int32_t S[2], nsplit_x[2], nsplit_a[2], map_off[2];
  int32_t max_len, BOS, EOS, UNK, PAD, materialize_only;
  /* weights */
  const float* E; const float* pe;
  case_layer_weights_t layers[8];       /* decs.{0,1}.layers.{0..3} */
  const float* lnN_g; const float* lnN_b;            /* norm1 */
  const void* Wqa_t[2]; const float* bqa[2]; const float* va[2];   /* attns.i.linear_query, v */
  const void* Wg_t; const float* bg;                 /* gen.0 */
  const void* Wv; const float* Wm; const float* bm;  /* gen.2 [V][H] row-major, mix */
  /* per-batch (prefill) tensors */
  const float* feat;                    /* [B][H] = norm2(answer_rep) */
  const void* Kx[8]; const void* Vx[8]; /* fp32: [B][NH][S_i][HD] per layer; bf16: Kx = interleaved K|V tiles
                                           (case_cross_attn_partial_tc), Vx unused */
  const void* U[2]; const void* Mv[2];  /* [B][S_i][H] */
  const uint8_t* mask[2]; const float* prior[2]; const int32_t* map; int32_t map_ld;
  /* state */
  void* kcache[8]; void* vcache[8];
  int32_t* anc[2]; int32_t* tok; int32_t* live; double* cum; int32_t* length; int32_t* parent;
  int32_t* ended; double* best_key; int32_t* best_len; int32_t* out_tokens; int32_t* n_live;
  /* scratch (fp32 unless noted) */
  float* x_in; float* h; float* bbuf; float* q2; float* part_ml; float* part_acc;
  float* qa; float* attn_un[2]; float* stats[2]; float* ctxp[2]; float* hN; float* ctx[2];
  float* gates; float* fac; float* gfeat; float* logits; float* dist; float* top_vals; int32_t* top_idx;
  void* vocab_ws;                       /* case_vocab_tc_workspace_bytes(R) bytes when vocab_impl == 1 */
  int32_t* prow;                        /* [R][Tmax] scratch of case_layer_chain (may be NULL) */
  float* h0; float* qa1;                /* [R][H] each (may be NULL): stack-0 output and second attention query,
                                           private copies that let the additive attentions run on a side stream */
  float* base_ms; float* base_e; int32_t* base_i;   /* [R][4][2], [R][4][16], [R][4][16] (may be NULL): case_vocab_base */
  /* compacted second memory (may be NULL -> masks + case_cross_attn_partial_tc): Kx[4..7] then hold the
   * gathered tiles, part_ml / part_acc have xslots slots per (row, head) */
  const int32_t* xcount; const int32_t* xprefix; int32_t xslots;
  const int32_t* xidx; const int32_t* xorder;   /* [B][S1] valid positions, [B] queries by valid count (desc) */
  int32_t* qcount;                      /* [B] zeros (may be NULL): lets the sparse tail run the search bookkeeping */
  const void* Wqa_c[2]; const void* Wg_c;   /* attention-query / gen.0 weights as post linears of the cluster launches (may be NULL) */
  const int32_t* xns;                   /* [B] splits of the second memory's additive attention per query (may be NULL) */
  /* copy plan of the batch for the sparse tail (may be NULL -> hash table): see case_tail_args_t */
  const int32_t* cp_n; const int32_t* cp_uid; const int32_t* cp_first; const int32_t* cp_start; const int32_t* cp_perm;
  int32_t cp_ld;
  const float* Gv[2];                   /* [B][S_i][4] fp32 gate-projected memories (may be NULL): the search path then runs
                                           case_additive_attn_gate and never reads Mv */
  int32_t opt;                          /* CASE_OPT_* bits (0 = default fast path) */
  case_fork_t* fork;                    /* side stream + events of this engine (may be NULL: everything on `stream`) */
  /* extended vocabulary (pointer-generator OOV extension, the "extended (vocab + OOV) distribution"): map entries in
   * [V, V + n_oov) are per-query dynamic words; dist / top-k range over V + n_oov ids (ldv >= V + n_oov), an OOV id is
   * fed back as UNK and kept in tok_ext [R][Tmax+1] for the output.  n_oov = 0: off. */
  int32_t n_oov;
  int32_t* tok_ext;
  int32_t nbest;                        /* n-best list of the beam search (case_select_args_t.nbest); 0 or 1: the best only */
  /* attribution records of the search (case_select_args_t.attr_*; all three or none, NULL = off): attr_cand [R][W],
   * attr_hist [R][Tmax+1], out_attr like out_tokens.  Only the sparse tail computes them: a request on a step that would
   * not take it (CASE_OPT_DENSE_TAIL / CASE_OPT_UNFUSED_TAIL, materialize_only, no base_* buffers, V < 2W, more than
   * case_sparse_tail_max_sources() source positions) is refused before the first launch. */
  case_attr_t* attr_cand; case_attr_t* attr_hist; case_attr_t* out_attr;
  /* search constraints (case_tail_args_t.no_repeat_ngram / min_len; 0 = off), modes CASE_MODE_BEAM and
   * CASE_MODE_PROTO_GREEDY: 0 <= no_repeat_ngram <= max_len, 0 <= min_len < max_len.  The ids compared are the returned
   * ones (tok_ext with n_oov > 0; greedy: the emitted token).  Only the sparse tail applies them: a request on a step that
   * would not take it (as for attribution), in CASE_MODE_MODULE_GREEDY, or with V < 2W + Tmax + 1 is refused before the
   * first launch; the n-best and attribution refusals come first. */
  int32_t no_repeat_ngram, min_len;
  /* banned words (case_tail_args_t.ban_*; all four or none, NULL = off), same modes and the same sparse-tail requirement
   * as the constraints: a request on a step that cannot serve it, with only some of the four pointers, or with
   * V < 2W + Tmax + 1 is refused before the first launch, after the n-best, attribution and constraint checks.  The list
   * lives in device memory and is read at every launch, so the caller enforces its content limits (ids in [0, V), at
   * most CASE_MAX_BAN_SEQ sequences of 2 .. CASE_MAX_BAN_LEN tokens, V - (masked ids) >= 2W + Tmax + 1 + *ban_n). */
  const uint32_t* ban_mask; const int32_t* ban_tok; const int32_t* ban_len; const int32_t* ban_n;
} case_step_args_t;

/* Enqueue one full decode step t (embedding .. select) for all R rows: the body of the eval loop
 * CaSE/Model.py:94-122 for the newest position only, plus the search bookkeeping of
 * Generations.py:136-185 when mode == CASE_MODE_BEAM.  materialize_only: stop after the
 * distribution is complete (the `generate` face of the protocol). */
int case_decode_step(const case_step_args_t* a, int t, case_stream_t stream);

typedef struct {
  int32_t B, W, R, V, ldv, dtype, fast_tanh, vocab_impl, mode;
  int32_t Lc, Lb, nsplit_c, nsplit_b, max_len, BOS, EOS, UNK, PAD, materialize_only, Tmax;
  const float* E;                                        /* dec.embedding [V][E=H] */
  const void* Wqs_t; const float* bqs; const float* vs;  /* dec.src_attn  */
  const void* Wqb_t; const float* bqb; const float* vb;  /* dec.bg_attn   */
  const void* Wih_t; const float* bih; const void* Whh_t; const float* bhh;   /* dec.gru */
  const void* Wr_t; const float* br;                     /* dec.readout */
  const void* Wv; const float* bv; const float* wc; const float* bc;          /* gen.linear / linear_copy */
  const void* Us; const void* Ms; const void* Ub; const void* Mb;  /* [B][L][H], [B][L][2H] */
  const uint8_t* mask_c; const uint8_t* mask_b; const int32_t* map; int32_t map_ld;
  float* state[2];                                       /* [R][H] double-buffered by step parity */
  int32_t* anc[2]; int32_t* tok; int32_t* live; double* cum; int32_t* length; int32_t* parent;
  int32_t* ended; double* best_key; int32_t* best_len; int32_t* out_tokens; int32_t* n_live;
  float* emb; float* qa; float* attn_un[2]; float* stats[2]; float* ctxp[2]; float* ctx[2];
  float* gi; float* gh; float* feat; float* gates; float* fac; float* logits; float* dist;
  float* top_vals; int32_t* top_idx;
  void* vocab_ws;
  int32_t opt;                                           /* CASE_OPT_NO_PDL / CASE_OPT_UNFUSED_TAIL / CASE_OPT_DENSE_TAIL */
  /* statistics of case_vocab_base for the sparse tail (search path): base_ms [R][4][2], base_e / base_i [R][4][16];
   * NULL: the dense case_row_tail is used */
  float* base_ms; float* base_e; int32_t* base_i;
  /* optional: with a fork handle and a second query buffer qa1 [R][H] the attention over the context memory runs on the
   * handle's side stream beside the attention over the background (CASE_OPT_NO_FORK switches it off) */
  case_fork_t* fork; float* qa1;
  int32_t nbest;                                         /* n-best list of the beam search (case_select_args_t.nbest) */
  /* attribution records (as in case_step_args_t; part[1] = copy from the background, part[2] = 0); refused before the
   * first launch unless the step takes the sparse tail */
  case_attr_t* attr_cand; case_attr_t* attr_hist; case_attr_t* out_attr;
  int32_t no_repeat_ngram, min_len;                      /* search constraints (as in case_step_args_t) */
  /* banned words (as in case_step_args_t) */
  const uint32_t* ban_mask; const int32_t* ban_tok; const int32_t* ban_len; const int32_t* ban_n;
} gttp_step_args_t;

/* One GTTP decode step (GTTP/Model.py:176-193 -> BBCDecoder.forward :113-131 ->
 * CopyGenerator.forward :14-43 -> topk) plus the same search bookkeeping. */
int gttp_decode_step(const gttp_step_args_t* a, int t, case_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CASE_B200_H */
