// extern "C" surface of libr2d2_b200 (declared in include/r2d2_b200.h).
#include <atomic>

#include "act.cuh"
#include "common.cuh"
#include "elementwise.cuh"
#include "gemm.cuh"
#include "learner.cuh"
#include "lstm_scan.cuh"
#include "net.cuh"
#include "replay.cuh"

namespace r2d2 {
static thread_local std::string g_last_error;
static std::atomic<long long> g_launches{0};
void set_last_error(const std::string& msg) { g_last_error = msg; }
const char* last_error() { return g_last_error.c_str(); }
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }
}  // namespace r2d2

using namespace r2d2;

static inline cudaStream_t S(r2d2_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline NetShape shape_of(const r2d2_net_shape* s) {
  return NetShape{s->obs_size, s->n_actions, s->hidden, s->is_critic != 0};
}

extern "C" {

int r2d2_version(void) { return 100; }
const char* r2d2_arch(void) { return "sm_100a"; }
const char* r2d2_last_error(void) { return last_error(); }

int r2d2_device_sm_count(int* out) {
  R2D2_REQUIRE(out, "null");
  int dev = 0;
  R2D2_CUDA_TRY(cudaGetDevice(&dev));
  R2D2_CUDA_TRY(cudaDeviceGetAttribute(out, cudaDevAttrMultiProcessorCount, dev));
  return R2D2_OK;
}

int r2d2_gemm_f32(int layout, int M, int N, int K, const float* A, long long lda, const float* B, long long ldb,
                  const float* A2, long long lda2, const float* B2, long long ldb2, int K2, float* C,
                  long long ldc, const float* bias, const float* Z, long long ldz, int epilogue, int split_k,
                  r2d2_stream_t stream) {
  R2D2_REQUIRE(layout >= 0 && layout <= 2, "layout");
  GemmParams p;
  p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.A2 = A2; p.lda2 = lda2; p.B2 = B2; p.ldb2 = ldb2; p.K2 = K2;
  p.C = C; p.ldc = ldc; p.M = M; p.N = N; p.K = K; p.bias = bias; p.Z = Z; p.ldz = ldz; p.epilogue = epilogue;
  p.split_k = split_k < 1 ? 1 : split_k;
  return gemm_f32(p, (GemmLayout)layout, S(stream));
}

size_t r2d2_net_param_count(const r2d2_net_shape* shape) { return shape ? shape_of(shape).param_count() : 0; }

size_t r2d2_net_workspace_floats(const r2d2_net_shape* shape, int T, int B, int repeat) {
  return shape ? ChainWs::floats(shape_of(shape), T, B, repeat) : 0;
}

int r2d2_lstm_net_forward(const r2d2_net_shape* shape, const float* params, const float* obs, const float* act,
                          const float* h0, const float* c0, int T, int B, int repeat, int head_first_row,
                          float* out, float* workspace, r2d2_stream_t stream) {
  R2D2_REQUIRE(shape && params && obs && workspace, "null");
  R2D2_REQUIRE(T > 0 && B > 0 && repeat >= 1, "shape");
  const NetShape s = shape_of(shape);
  const NetParams P = NetParams::from_flat(const_cast<float*>(params), s);
  const ChainWs ws = ChainWs::carve(workspace, s, T, B, repeat);
  R2D2_TRY(net_forward(s, P, ws, obs, act, h0, c0, T, B, repeat, S(stream)));
  if (out) {
    float* ho = ws.head_out + (size_t)head_first_row * B * s.act;
    R2D2_TRY(net_head_forward(s, P, ws, head_first_row, T, B, repeat, ho, s.act, S(stream)));
    R2D2_CUDA_TRY(cudaMemcpyAsync(out, ho, sizeof(float) * (size_t)(T - head_first_row) * B * s.act,
                                  cudaMemcpyDeviceToDevice, S(stream)));
  }
  return R2D2_OK;
}

int r2d2_lstm_net_backward(const r2d2_net_shape* shape, const float* params, const float* obs, const float* act,
                           const float* d_out, int T, int B, int repeat, int head_first_row, float* grads,
                           float* d_act, float* workspace, r2d2_stream_t stream) {
  R2D2_REQUIRE(shape && params && obs && d_out && workspace, "null");
  const NetShape s = shape_of(shape);
  const NetParams P = NetParams::from_flat(const_cast<float*>(params), s);
  const ChainWs ws = ChainWs::carve(workspace, s, T, B, repeat);
  const long long n = (long long)(T - head_first_row) * B * s.act;
  const float* d_pre = d_out;
  if (!s.critic) {  // through the output tanh (models.py:39) using the head outputs kept by the forward call
    R2D2_TRY(mul_dtanh(d_out, ws.head_out + (size_t)head_first_row * B * s.act, ws.d_pre, n, S(stream)));
    d_pre = ws.d_pre;
  }
  NetParams G;
  if (grads) G = NetParams::from_flat(grads, s);
  return net_backward(s, P, grads ? &G : nullptr, ws, obs, act, d_pre, head_first_row, T, B, repeat, d_act, nullptr,
                      S(stream));
}

int r2d2_lstm_scan_forward(const float* gin, const float* whh, const float* h0, const float* c0, float* gates,
                           float* hs, float* cs, float* head_in, int T, int B, int H, int repeat, float* scratch,
                           r2d2_stream_t stream) {
  ScanFwdParams p;
  p.gin = gin; p.whh = whh; p.h0 = h0; p.c0 = c0; p.gates = gates; p.hs = hs; p.cs = cs; p.head_in = head_in;
  p.T = T; p.B = B; p.H = H; p.repeat = repeat; p.scratch = scratch;
  return lstm_scan_forward(p, S(stream));
}

int r2d2_lstm_scan_backward(const float* gates, const float* hs, const float* cs, const float* whh,
                            const float* dh_head, int head_first_step, float* dgates, float* dgin, int T, int B,
                            int H, int repeat, float* scratch, r2d2_stream_t stream) {
  ScanBwdParams p;
  p.gates = gates; p.hs = hs; p.cs = cs; p.whh = whh; p.dh_head = dh_head; p.head_first_step = head_first_step;
  p.dgates = dgates; p.dgin = dgin; p.T = T; p.B = B; p.H = H; p.repeat = repeat; p.scratch = scratch;
  return lstm_scan_backward(p, S(stream));
}

int r2d2_debug_scan_forward_trace(const float* gin, const float* whh, float* gates, float* hs, float* cs, int T, int B,
                                  int H, long long* trace, r2d2_stream_t stream) {
  ScanFwdParams p;
  p.gin = gin; p.whh = whh; p.gates = gates; p.hs = hs; p.cs = cs; p.T = T; p.B = B; p.H = H; p.repeat = 1; p.trace = trace;
  return lstm_scan_forward(p, S(stream));
}

int r2d2_debug_scan_backward_trace(const float* gates, const float* hs, const float* cs, const float* whh,
                                   const float* dh_head, float* dgates, int T, int B, int H, long long* trace,
                                   r2d2_stream_t stream) {
  ScanBwdParams p;
  p.gates = gates; p.hs = hs; p.cs = cs; p.whh = whh; p.dh_head = dh_head; p.dgates = dgates; p.dgin = dgates;
  p.T = T; p.B = B; p.H = H; p.repeat = 1; p.trace = trace;
  return lstm_scan_backward(p, S(stream));
}

int r2d2_debug_max_active_clusters(int H, int nb, int backward) { return lstm_scan_max_active_clusters(H, nb, backward); }

int r2d2_set_gemm_impl(int impl) {
  gemm_set_impl(impl != 0);
  gemm_set_impl_skinny_mma(impl != 2);  // 2 = force the tcgen05 path even for skinny problems (tests)
  return R2D2_OK;
}
int r2d2_get_gemm_impl(void) { return gemm_get_impl(); }
int r2d2_set_scan_impl(int impl) { lstm_scan_set_impl(impl); return R2D2_OK; }
int r2d2_get_scan_impl(void) { return lstm_scan_get_impl(); }
int r2d2_scan_status(int* status, r2d2_stream_t stream) { return lstm_scan_error_status(status, S(stream)); }

int r2d2_td_priority(const float* q, const float* q_next, const float* rew, const float* term, int L, int B,
                     int A, int burn_in, int n_step, float gamma, float eta, float* target, float* dq,
                     float* td_sq, float* priority, float* critic_loss, r2d2_stream_t stream) {
  TdPriorityParams p;
  p.q = q; p.q_next = q_next; p.rew = rew; p.term = term; p.target = target; p.dq = dq; p.td_sq = td_sq;
  p.priority = priority; p.loss_sum = critic_loss; p.L = L; p.B = B; p.A = A; p.burn_in = burn_in; p.n_step = n_step;
  p.gamma_n = (float)pow((double)gamma, (double)n_step);
  p.eta = eta;
  return td_priority(p, S(stream));
}

int r2d2_nstep_rewards(const float* raw, const int* n_rows, int T, int B, int n_step, float gamma, float* out,
                       r2d2_stream_t stream) {
  return nstep_rewards(raw, n_rows, T, B, n_step, gamma, out, S(stream));
}
int r2d2_actor_priorities(const float* q, const float* q_next, const float* rew, const float* term, const int* n_rows,
                          int B, int A, int burn_in, int learning, int n_step, float gamma, float eta, int p_max,
                          float* prio, r2d2_stream_t stream) {
  return actor_priorities(q, q_next, rew, term, n_rows, B, A, burn_in, learning, n_step, gamma, eta, p_max, prio, S(stream));
}

int r2d2_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, int step,
                   float lr, float beta1, float beta2, float eps, float grad_scale, r2d2_stream_t stream) {
  return adam_step(params, grads, exp_avg, exp_avg_sq, n, step, lr, beta1, beta2, eps, grad_scale, S(stream));
}

// ---- replay ----
int r2d2_replay_create(r2d2_replay_t** out, const r2d2_replay_config* cfg) {
  return replay_create(reinterpret_cast<Replay**>(out), cfg);
}
int r2d2_replay_destroy(r2d2_replay_t* r) { return replay_destroy(reinterpret_cast<Replay*>(r)); }
int r2d2_replay_add_episode(r2d2_replay_t* r, const float* obs, const float* act, const float* rew,
                            const float* term, const float* states, int n_rows, int n_state_rows,
                            const float* priority, int n_starts, r2d2_stream_t stream) {
  return replay_add_episode(reinterpret_cast<Replay*>(r), obs, act, rew, term, states, n_rows, n_state_rows, priority,
                            n_starts, S(stream));
}
int r2d2_replay_add_episodes(r2d2_replay_t* r, int n_episodes, const int* n_rows, const int* n_starts,
                             const float* obs, const float* act, const float* rew, const float* term,
                             const float* states, const float* leaf_prio, long long* row_start_out,
                             long long* n_evicted_out, long long* sequence_counter_out, r2d2_stream_t stream) {
  return replay_add_episodes(reinterpret_cast<Replay*>(r), n_episodes, n_rows, n_starts, obs, act, rew, term, states,
                             leaf_prio, row_start_out, n_evicted_out, sequence_counter_out, S(stream));
}
int r2d2_replay_sample(r2d2_replay_t* r, const float* u, int batch, long long* leaf_idx, float* obs, float* act,
                       float* rew, float* term, float* states, r2d2_stream_t stream) {
  return replay_sample(reinterpret_cast<Replay*>(r), u, batch, leaf_idx, obs, act, rew, term, states, S(stream));
}
int r2d2_replay_gather(r2d2_replay_t* r, const long long* leaf_idx, int batch, float* obs, float* act, float* rew,
                       float* term, float* states, r2d2_stream_t stream) {
  return replay_gather(reinterpret_cast<Replay*>(r), leaf_idx, batch, obs, act, rew, term, states, S(stream));
}
int r2d2_replay_update_priorities(r2d2_replay_t* r, const long long* leaf_idx, const float* prio, int batch,
                                  r2d2_stream_t stream) {
  return replay_update_priorities(reinterpret_cast<Replay*>(r), leaf_idx, prio, batch, S(stream));
}
int r2d2_replay_stats(r2d2_replay_t* r, r2d2_replay_stats_t* out, r2d2_stream_t stream) {
  return replay_stats(reinterpret_cast<Replay*>(r), out, S(stream));
}
int r2d2_replay_decode(r2d2_replay_t* r, const long long* leaf_idx_host, int n, long long* episode_index,
                       long long* sequence_index) {
  return replay_decode(reinterpret_cast<Replay*>(r), leaf_idx_host, n, episode_index, sequence_index);
}
int r2d2_replay_tree_level(r2d2_replay_t* r, int level, const float** dev_ptr, long long* n) {
  return replay_tree_level(reinterpret_cast<Replay*>(r), level, dev_ptr, n);
}

// ---- learner ----
int r2d2_learner_create(r2d2_learner_t** out, const r2d2_learner_config* cfg) {
  return learner_create(reinterpret_cast<Learner**>(out), cfg);
}
int r2d2_learner_destroy(r2d2_learner_t* l) { return learner_destroy(reinterpret_cast<Learner*>(l)); }
int r2d2_learner_buffers_get(r2d2_learner_t* lh, r2d2_learner_buffers* o) {
  R2D2_REQUIRE(lh && o, "null");
  Learner* l = reinterpret_cast<Learner*>(lh);
  o->obs = l->obs; o->act = l->act; o->rew = l->rew; o->term = l->term; o->states = l->states;
  o->leaf_idx = l->leaf_idx; o->uniforms = l->uniforms; o->q_value = l->q; o->target_q_value = l->target;
  o->td_sq = l->td_sq; o->priority = l->priority; o->losses = l->losses;
  return R2D2_OK;
}
int r2d2_learner_buffers_get_slot(r2d2_learner_t* lh, int slot, r2d2_learner_buffers* o) {
  R2D2_REQUIRE(lh && o && (slot == 0 || slot == 1), "batch slot");
  Learner* l = reinterpret_cast<Learner*>(lh);
  R2D2_TRY(r2d2_learner_buffers_get(lh, o));
  const Learner::BatchSlot& b = l->slots[slot];
  o->obs = b.obs; o->act = b.act; o->rew = b.rew; o->term = b.term; o->states = b.states;
  o->leaf_idx = b.leaf_idx; o->uniforms = b.uniforms;
  return R2D2_OK;
}
int r2d2_learner_select_batch(r2d2_learner_t* l, int slot) {
  R2D2_REQUIRE(l, "null");
  return learner_select_batch(reinterpret_cast<Learner*>(l), slot);
}
int r2d2_learner_target_phase(r2d2_learner_t* l, int slot, r2d2_stream_t stream) {
  R2D2_REQUIRE(l, "null");
  return learner_target_phase(reinterpret_cast<Learner*>(l), slot, S(stream));
}
int r2d2_learner_discard_prefetch(r2d2_learner_t* l, r2d2_stream_t stream) {
  R2D2_REQUIRE(l, "null");
  return learner_discard_prefetch(reinterpret_cast<Learner*>(l), S(stream));
}
int r2d2_learner_critic_phase(r2d2_learner_t* l, r2d2_stream_t stream) {
  R2D2_REQUIRE(l, "null");
  return learner_critic_phase(reinterpret_cast<Learner*>(l), S(stream));
}
int r2d2_learner_actor_forward(r2d2_learner_t* l, r2d2_stream_t stream) {
  R2D2_REQUIRE(l, "null");
  return learner_actor_forward(reinterpret_cast<Learner*>(l), S(stream));
}
int r2d2_learner_actor_phase(r2d2_learner_t* l, float grad_scale, r2d2_stream_t stream) {
  R2D2_REQUIRE(l, "null");
  return learner_actor_phase(reinterpret_cast<Learner*>(l), grad_scale, S(stream));
}
int r2d2_learner_finish_phase(r2d2_learner_t* l, float grad_scale, r2d2_stream_t stream) {
  R2D2_REQUIRE(l, "null");
  return learner_finish_phase(reinterpret_cast<Learner*>(l), grad_scale, S(stream));
}
int r2d2_learner_step_count(r2d2_learner_t* l) { return l ? reinterpret_cast<Learner*>(l)->step : -1; }
int r2d2_learner_set_overlap_actor_inputs(r2d2_learner_t* l, int on) {
  R2D2_REQUIRE(l, "null");
  reinterpret_cast<Learner*>(l)->overlap_actor_inputs = on != 0;
  return R2D2_OK;
}
int r2d2_peer_layout_for(long long n_critic, long long n_actor, int world, r2d2_peer_layout* out) {
  R2D2_REQUIRE(out && n_critic > 0 && n_actor > 0 && world >= 2 && world <= kPeerMaxWorld, "peer layout arguments");
  const PeerLayout pl = peer_layout(n_critic, n_actor, world);
  out->bytes = pl.bytes;
  out->off_critic_grads = pl.off_grads[kPeerCritic];
  out->off_actor_grads = pl.off_grads[kPeerActor];
  out->off_critic_sums = pl.off_sums[kPeerCritic];
  out->off_actor_sums = pl.off_sums[kPeerActor];
  return R2D2_OK;
}
int r2d2_learner_peer_layout(r2d2_learner_t* lh, int world, r2d2_peer_layout* out) {
  R2D2_REQUIRE(lh && out && world >= 2 && world <= kPeerMaxWorld, "peer layout arguments");
  Learner* l = reinterpret_cast<Learner*>(lh);
  const PeerLayout pl = peer_layout((long long)l->critic_sh.param_count(), (long long)l->actor_sh.param_count(), world);
  out->bytes = pl.bytes;
  out->off_critic_grads = pl.off_grads[kPeerCritic];
  out->off_actor_grads = pl.off_grads[kPeerActor];
  out->off_critic_sums = pl.off_sums[kPeerCritic];
  out->off_actor_sums = pl.off_sums[kPeerActor];
  return R2D2_OK;
}
int r2d2_learner_attach_peers(r2d2_learner_t* l, int rank, int world, void* const* peer_bases) {
  return learner_attach_peers(reinterpret_cast<Learner*>(l), rank, world, peer_bases);
}
int r2d2_learner_peer_status(r2d2_learner_t* lh, int* status, r2d2_stream_t stream) {
  R2D2_REQUIRE(lh && status, "null");
  Learner* l = reinterpret_cast<Learner*>(lh);
  R2D2_REQUIRE(l->peer, "no peers attached");
  return peer_status(*l->peer, status, static_cast<cudaStream_t>(stream));
}
int r2d2_learner_peer_counters(r2d2_learner_t* lh, unsigned long long* out6, int reset, r2d2_stream_t stream) {
  R2D2_REQUIRE(lh && out6, "null");
  Learner* l = reinterpret_cast<Learner*>(lh);
  R2D2_REQUIRE(l->peer, "no peers attached");
  return peer_counters(*l->peer, out6, reset, static_cast<cudaStream_t>(stream));
}
int r2d2_learner_set_step_count(r2d2_learner_t* l, int step) {
  R2D2_REQUIRE(l && step >= 0, "step");
  reinterpret_cast<Learner*>(l)->step = step;
  return R2D2_OK;
}
int r2d2_learner_launches_per_iteration(r2d2_learner_t* lh) {
  if (!lh) return -1;
  Learner* l = reinterpret_cast<Learner*>(lh);
  return l->launches_phase[0] + l->launches_phase[1] + l->launches_phase[2] +
         (l->target_phase_standalone ? l->launches_target : 0);
}

// ---- batched acting ----
int r2d2_act_create(r2d2_act_t** out, const r2d2_net_shape* shape, int max_batch) {
  R2D2_REQUIRE(out && shape, "null");
  return act_create(reinterpret_cast<Act**>(out), shape->obs_size, shape->n_actions, shape->hidden, max_batch);
}
int r2d2_act_destroy(r2d2_act_t* a) { return act_destroy(reinterpret_cast<Act*>(a)); }
int r2d2_act_load(r2d2_act_t* a, const float* actor, const float* target_actor, const float* critic,
                  const float* target_critic, r2d2_stream_t stream) {
  const float* const params[4] = {actor, target_actor, critic, target_critic};
  return act_load(reinterpret_cast<Act*>(a), params, S(stream));
}
int r2d2_act_step(r2d2_act_t* a, const float* obs, const float* state_in, float* state_out, float* mu, int B,
                  r2d2_stream_t stream) {
  return act_step(reinterpret_cast<Act*>(a), obs, state_in, state_out, mu, B, S(stream));
}
int r2d2_act_status(r2d2_act_t* a, int* status, r2d2_stream_t stream) {
  return act_status(reinterpret_cast<Act*>(a), status, S(stream));
}

}  // extern "C"
