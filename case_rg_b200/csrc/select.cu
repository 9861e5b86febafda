// Search bookkeeping on the device: greedy token hand-off and the beam step of
// common/Generations.py:136-185, with no host round trips.
//
// State layout (all int32 unless noted), R = B*W rows, TL = Tmax + 1:
//   tok[r][j]   input token consumed at position j by whichever hypothesis occupied physical row r
//               at step j (each (r, j) cell is written exactly once, by the select of step j-1)
//   anc[r][j]   physical row that holds position j (self-attention K/V, token) of the hypothesis
//               currently in slot r, for j < current position; double-buffered across steps
//   live/cum(double)/length per slot; live slots of a query are always compacted to the front in
//   rank order, which is the order Generations.beam keeps its fringe in (sorted per batch item).
#include "common.cuh"
#include "select.cuh"

namespace cb {

template <bool ATTR>
__global__ __launch_bounds__(32) void beam_select_kernel(case_select_args_t a) {
  pdl_trigger();
  pdl_wait();
  beam_select_query<ATTR>(a, blockIdx.x, threadIdx.x);
}

}  // namespace cb

using namespace cb;

extern "C" int case_beam_select(const case_select_args_t* a, case_stream_t stream) {
  CB_REQUIRE(a && a->top_idx && a->tok && a->anc_out && a->parent && a->out_tokens && a->live && a->n_live,
             "case_beam_select: null pointer");
  CB_REQUIRE(a->B > 0 && a->W >= 1 && a->W <= CASE_MAX_W && a->t >= 0 && a->t < a->max_len && a->max_len <= a->Tmax,
             "case_beam_select: bad sizes");
  int rc = check_nbest(a->nbest, a->W, a->mode);
  if (rc) return rc;
  rc = check_attr_select(*a);
  if (rc) return rc;
  if (a->mode == CASE_MODE_BEAM) {
    CB_REQUIRE(a->top_vals && a->cum && a->length && a->anc_in && a->best_key && a->best_len,
               "case_beam_select: beam mode needs top_vals/cum/length/anc_in/best_*");
  } else {
    CB_REQUIRE(a->W == 1, "case_beam_select: greedy modes need W == 1");
    CB_REQUIRE(a->mode != CASE_MODE_PROTO_GREEDY || a->ended, "case_beam_select: proto-greedy needs ended[]");
  }
  if (a->out_attr != nullptr)
    launch_k(beam_select_kernel<true>, a->B, 32, 0, (cudaStream_t)stream, *a);
  else
    launch_k(beam_select_kernel<false>, a->B, 32, 0, (cudaStream_t)stream, *a);
  return check_launch("case_beam_select");
}
