/* libr2d2_b200 - C ABI of the B200-native learner hot path of pytorch-r2d2-DPG.
 *
 * The reference (pure Python) has no FFI; its boundary for this path is the module surface
 * learner.py / replay_memory.py / models.py / utils.py.  Each entry point below replaces the
 * reference function(s) cited next to it; the host-side mirror in pytorch-r2d2-dpg_b200/*.py binds
 * them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; r2d2_last_error() (thread-local) has the text;
 *   - tensors are caller-owned device memory (fp32, contiguous, time-major [T,B,*] as produced by
 *     replay_memory.py:123-136), passed as raw pointers + explicit sizes; no torch types here;
 *   - the library owns only opaque handles (replay shard + sum tree, learner workspaces);
 *   - every launch goes to the cudaStream_t given (passed as void*); nothing synchronises the host
 *     unless stated; one host thread per handle.
 *   - parameter blocks are FLAT fp32 buffers in the reference's state_dict order
 *     (l1.weight[H,I], l1.bias[H], l2.weight_ih[4H,H], l2.weight_hh[4H,H], l2.bias_ih[4H],
 *      l2.bias_hh[4H], l3.weight[A,H], l3.bias[A]; models.py:17-19,59-61), I = O (actor) or O+A (critic).
 */
#ifndef R2D2_B200_H_
#define R2D2_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define R2D2_OK 0
#define R2D2_ERR_CUDA (-1)
#define R2D2_ERR_ARG (-2)
#define R2D2_ERR_UNSUPPORTED (-3)
#define R2D2_ERR_STATE (-4)

typedef void* r2d2_stream_t; /* cudaStream_t */

int r2d2_version(void);                /* 100 * major + minor */
const char* r2d2_arch(void);           /* "sm_100a" */
const char* r2d2_last_error(void);
int r2d2_device_sm_count(int* out);

/* ------------------------------------------------------------------------------------------------
 * Dense building block (x*W^T, dgrad, wgrad of models.py:33,37-39,76,80-82): fp32 in/out, bf16x3
 * tensor-core MMAs.  layout: 0 = NT (A[M,K] * B[N,K]^T), 1 = NN (A[M,K] * B[K,N]), 2 = TN (A[K,M]^T * B[K,N]).
 * epilogue: 0 none, 1 tanh(acc+bias), 2 (acc+bias)*(1-Z^2), 3 acc+bias+Z.  split_k > 1 adds into C.
 * ---------------------------------------------------------------------------------------------- */
int r2d2_gemm_f32(int layout, int M, int N, int K, const float* A, long long lda, const float* B, long long ldb,
                  const float* A2, long long lda2, const float* B2, long long ldb2, int K2, float* C,
                  long long ldc, const float* bias, const float* Z, long long ldz, int epilogue, int split_k,
                  r2d2_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Recurrent net chains: replace the per-timestep python loops over ActorNet/CriticNet.__call__
 * (models.py:32-40,74-83) at learner.py:92-95,102-106,120-123.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int obs_size;   /* O */
  int n_actions;  /* A */
  int hidden;     /* H (128 in the reference, models.py:17-19) */
  int is_critic;  /* 0: ActorNet, 1: CriticNet (input = cat(obs, action), head without tanh, A outputs) */
} r2d2_net_shape;

size_t r2d2_net_param_count(const r2d2_net_shape* shape);
/* floats of workspace needed by one chain of T input rows, `repeat` cell steps per row, batch B */
size_t r2d2_net_workspace_floats(const r2d2_net_shape* shape, int T, int B, int repeat);

/* Forward over T rows (S = T*repeat cell steps).  obs [T,B,O]; act [T,B,A] (critic only, else NULL);
 * h0/c0 [B,H] or NULL for the zero state (models.py:34-36).  Head outputs are produced for input rows
 * [head_first_row, T) (after the last of the `repeat` steps of each row) into out [(T-head_first_row),B,A].
 * workspace keeps the activations for r2d2_lstm_net_backward. */
int r2d2_lstm_net_forward(const r2d2_net_shape* shape, const float* params, const float* obs, const float* act,
                          const float* h0, const float* c0, int T, int B, int repeat, int head_first_row,
                          float* out, float* workspace, r2d2_stream_t stream);

/* BPTT through the chain saved in `workspace`.  d_out [(T-head_first_row),B,A] = dLoss/d(head output).
 * grads: flat buffer like params, ACCUMULATED into (zero it first); NULL -> data gradient only.
 * d_act [T,B,A]: dLoss/d(action input) (critic only, optional).  The workspace is consumed. */
int r2d2_lstm_net_backward(const r2d2_net_shape* shape, const float* params, const float* obs, const float* act,
                           const float* d_out, int T, int B, int repeat, int head_first_row, float* grads,
                           float* d_act, float* workspace, r2d2_stream_t stream);

/* The serial scan alone (the persistent-RNN kernel; bench.py times it for the roofline line):
 * gin [T,B,4H] pre-activation input projection, whh [4H,H], h0/c0 [B,H] or NULL; outputs gates [T*repeat,B,4H]
 * (may alias gin when repeat == 1), hs/cs [T*repeat+1,B,H], head_in [T,B,H] or NULL.  scratch: NULL for
 * H in {32,64,128,256}, else [B,4H] floats. */
int r2d2_lstm_scan_forward(const float* gin, const float* whh, const float* h0, const float* c0, float* gates,
                           float* hs, float* cs, float* head_in, int T, int B, int H, int repeat, float* scratch,
                           r2d2_stream_t stream);
/* BPTT twin: dgates [S,B,4H] (may alias gates), dgin [T,B,4H] (only when repeat > 1), dh_head [*,B,H] or NULL
 * consumed from step head_first_step on.  scratch: NULL for the cluster sizes, else [2,B,H]. */
int r2d2_lstm_scan_backward(const float* gates, const float* hs, const float* cs, const float* whh,
                            const float* dh_head, int head_first_step, float* dgates, float* dgin, int T, int B,
                            int H, int repeat, float* scratch, r2d2_stream_t stream);

/* debug: forward scan that also records per-step globaltimer stamps [grid][S][8] (thread 0 of every CTA) */
int r2d2_debug_scan_forward_trace(const float* gin, const float* whh, float* gates, float* hs, float* cs, int T, int B,
                                  int H, long long* trace, r2d2_stream_t stream);
/* debug: BPTT scan (H = 512 kernel) that also records per-step globaltimer stamps [grid][S][8] */
int r2d2_debug_scan_backward_trace(const float* gates, const float* hs, const float* cs, const float* whh,
                                   const float* dh_head, float* dgates, int T, int B, int H, long long* trace,
                                   r2d2_stream_t stream);
/* debug: clusters of a tcgen05 scan kernel the device can keep resident at once (-1 if not instantiated):
 * H in {32,64,128,256,512}, nb = 16 or 32 rows per tile (the kernels the batch tiling chooses between, forward or
 * backward); H = 512, nb = 80, backward = 0 is the H = 512 forward kernel of up to 80 rows per cluster. */
int r2d2_debug_max_active_clusters(int H, int nb, int backward);
/* GEMM implementation switch for A/B checks: 1 = tcgen05/TMEM with skinny problems (K<64, N<32 or M<32) on the
 * single-launch mma.sync kernel (default), 2 = tcgen05 for every shape, 0 = mma.sync v1 kernel only */
int r2d2_set_gemm_impl(int impl);
int r2d2_get_gemm_impl(void);
/* scan implementation switch for A/B checks: 1 = tcgen05/TMEM (default), 0 = mma.sync v1 kernels */
int r2d2_set_scan_impl(int impl);
int r2d2_get_scan_impl(void);
/* *status != 0 if a bounded mbarrier wait inside a tcgen05 scan kernel ever timed out; synchronises the stream */
int r2d2_scan_status(int* status, r2d2_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Fused n-step target + value rescaling + TD loss gradient + sequence priority
 * (learner.py:107-111,135-138; utils.py:17-21).  q, q_next [L,B,A]; rew, term [T',B].
 * Any output pointer may be NULL.
 * ---------------------------------------------------------------------------------------------- */
int r2d2_td_priority(const float* q, const float* q_next, const float* rew, const float* term, int L, int B,
                     int A, int burn_in, int n_step, float gamma, float eta, float* target, float* dq,
                     float* td_sq, float* priority, float* critic_loss, r2d2_stream_t stream);

/* Actor-side rows of the path (SURVEY 8f N2), batched over finished episodes (one episode per batch column, time-major,
 * zero padded): n-step discounted reward pre-sum (actor.py:74-76; rows i < n_rows[b] - n_step, later rows copied) and
 * the initial sequence priorities (actor.py:78-107): priority k = eta*max + (1-eta)*mean over j = k+burn_in+1 ..
 * k+burn_in+learning of (mean_A(q[j] - h(R[j] + gamma^n (1-term[j+n-1]) q_next[j+n])))^2 - the reference's deque is one
 * step ahead of the learner's window and squares the MEAN difference; both are kept.  prio [B, p_max], zero where
 * k >= n_rows[b] - n_step - burn_in - learning.  q, q_next come from r2d2_lstm_net_forward on the zero state. */
int r2d2_nstep_rewards(const float* raw, const int* n_rows, int T, int B, int n_step, float gamma, float* out,
                       r2d2_stream_t stream);
int r2d2_actor_priorities(const float* q, const float* q_next, const float* rew, const float* term, const int* n_rows,
                          int B, int A, int burn_in, int learning, int n_step, float gamma, float eta, int p_max,
                          float* prio, r2d2_stream_t stream);

/* torch.optim.Adam defaults (learner.py:50-53,114,128) on a flat buffer; grad is multiplied by grad_scale first. */
int r2d2_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, int step,
                   float lr, float beta1, float beta2, float eps, float grad_scale, r2d2_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * GPU-resident prioritized sequence replay (replaces LearnerReplayMemory, replay_memory.py:67-175).
 * Rows of all episodes live in HBM (SoA); one sum-tree leaf per row (priority 0 for rows that are
 * not valid sequence starts); 32-ary tree of fp32 partial sums.  P(start) is proportional to its
 * priority, which is what the reference's two-level draw (replay_memory.py:95-114) samples.
 * ---------------------------------------------------------------------------------------------- */
typedef struct r2d2_replay r2d2_replay_t;

typedef struct {
  int obs_size, n_actions, hidden;
  int burn_in, learning, n_step;   /* window rows T' = burn_in + learning + n_step (replay_memory.py:116) */
  long long capacity_rows;         /* physical rows in HBM (ring) */
  long long max_sequences;         /* eviction threshold on the sequence counter (replay_memory.py:148) */
} r2d2_replay_config;

int r2d2_replay_create(r2d2_replay_t** out, const r2d2_replay_config* cfg);
int r2d2_replay_destroy(r2d2_replay_t* r);

/* Append one episode (replay_memory.py:141-152).  HOST pointers: obs [n_rows,O], act [n_rows,A], rew [n_rows],
 * term [n_rows] (n_rows includes the n_step pad rows, actor.py:173), states [n_state_rows,4,2,H]
 * (actor, target_actor, critic, target_critic) x (hx,cx), priority [n_starts].  Oldest episodes are
 * evicted FIFO when the ring or max_sequences overflows.  Synchronises the stream. */
int r2d2_replay_add_episode(r2d2_replay_t* r, const float* obs, const float* act, const float* rew,
                            const float* term, const float* states, int n_rows, int n_state_rows,
                            const float* priority, int n_starts, r2d2_stream_t stream);

/* One actor file at a time (LearnerReplayMemory.load, replay_memory.py:138-157): all episodes of the file are appended,
 * THEN the oldest episodes are dropped while the sequence counter exceeds max_sequences - the reference's order.
 * HOST pointers, packed over the file's episodes with R = sum(n_rows): obs [R,O], act [R,A], rew [R], term [R],
 * states [R,4,2,H] (zero rows for the pad rows), leaf_prio [R] (the priority of a row that starts a sequence, else 0).
 * Contiguous runs in the ring are one copy per tensor; the tree is refreshed once; one stream synchronisation.
 * Outputs (host, optional): first ring row of each episode, episodes evicted by this call, the sequence counter. */
int r2d2_replay_add_episodes(r2d2_replay_t* r, int n_episodes, const int* n_rows, const int* n_starts,
                             const float* obs, const float* act, const float* rew, const float* term,
                             const float* states, const float* leaf_prio, long long* row_start_out,
                             long long* n_evicted_out, long long* sequence_counter_out, r2d2_stream_t stream);

/* Draw `batch` starts from DEVICE uniforms u[batch] in [0,1) and gather the time-major batch:
 * leaf_idx [batch] (int64, start row = tree leaf), obs [T',batch,O], act [T',batch,A], rew [T',batch],
 * term [T',batch], states [4,2,batch,H].  Any gather output may be NULL. */
int r2d2_replay_sample(r2d2_replay_t* r, const float* u, int batch, long long* leaf_idx, float* obs, float* act,
                       float* rew, float* term, float* states, r2d2_stream_t stream);

/* The gather half alone, for start rows the caller chose (DEVICE int64 leaf_idx): same outputs as r2d2_replay_sample. */
int r2d2_replay_gather(r2d2_replay_t* r, const long long* leaf_idx, int batch, float* obs, float* act, float* rew,
                       float* term, float* states, r2d2_stream_t stream);

/* priority[leaf_idx[i]] = prio[i] (DEVICE arrays; on duplicates the highest i wins, like the python
 * loop at learner.py:136-139) and recompute the touched tree paths. */
int r2d2_replay_update_priorities(r2d2_replay_t* r, const long long* leaf_idx, const float* prio, int batch,
                                  r2d2_stream_t stream);

typedef struct {
  long long n_episodes, n_rows_used, sequence_counter, capacity_rows, tree_levels, tree_nodes;
  long long last_row_start;        /* first row of the most recently added episode */
  double total_priority;
} r2d2_replay_stats_t;
int r2d2_replay_stats(r2d2_replay_t* r, r2d2_replay_stats_t* out, r2d2_stream_t stream); /* synchronises */

/* host-side decode of a start row into the reference's (episode_index, sequence_index) pair
 * (position of the episode in FIFO order, offset inside it); -1/-1 if the row is not live. */
int r2d2_replay_decode(r2d2_replay_t* r, const long long* leaf_idx_host, int n, long long* episode_index,
                       long long* sequence_index);
/* raw device views for tests: tree level pointer/size, leaf priorities */
int r2d2_replay_tree_level(r2d2_replay_t* r, int level, const float** dev_ptr, long long* n);

/* ------------------------------------------------------------------------------------------------
 * Learner iteration engine (learner.py:84-139 minus file I/O).  Parameters, gradients and Adam
 * moments are caller-owned flat device buffers; the engine owns batch buffers and workspaces.
 * ---------------------------------------------------------------------------------------------- */
typedef struct r2d2_learner r2d2_learner_t;

typedef struct {
  int obs_size, n_actions, hidden;
  int batch, burn_in, learning, n_step;
  float gamma, actor_lr, critic_lr, eta;
  int target_update_interval;      /* learner.py:45,131 */
  float* actor_params;  float* critic_params;  float* target_actor_params;  float* target_critic_params;
  float* actor_grads;   float* critic_grads;
  float* actor_exp_avg; float* actor_exp_avg_sq; float* critic_exp_avg; float* critic_exp_avg_sq;
} r2d2_learner_config;

typedef struct {
  /* device pointers into the engine-owned batch (fill them via r2d2_replay_sample or memcpy) */
  float* obs;      /* [T',B,O] */
  float* act;      /* [T',B,A] */
  float* rew;      /* [T',B]   */
  float* term;     /* [T',B]   */
  float* states;   /* [4,2,B,H] actor, target_actor, critic, target_critic */
  long long* leaf_idx; /* [B] */
  float* uniforms; /* [B] */
  /* results of the last iteration */
  float* q_value;        /* [L,B,A] */
  float* target_q_value; /* [L,B,A] */
  float* td_sq;          /* [L,B]   */
  float* priority;       /* [B]     */
  float* losses;         /* [2] critic_loss, actor_loss */
} r2d2_learner_buffers;

int r2d2_learner_create(r2d2_learner_t** out, const r2d2_learner_config* cfg);
int r2d2_learner_destroy(r2d2_learner_t* l);
int r2d2_learner_buffers_get(r2d2_learner_t* l, r2d2_learner_buffers* out);
/* The batch has two slots.  r2d2_learner_buffers_get returns slot 0 (the only one a simple caller needs); a pipelined
 * caller fills slot 1-s with batch i+1 while the phases of iteration i still read slot s, runs that batch's target
 * chains early with r2d2_learner_target_phase (they read only the target nets: learner.py:87,94-95,106) and switches
 * with r2d2_learner_select_batch before the next r2d2_learner_critic_phase.  Not allowed between an iteration whose
 * finish phase copies the weights into the target nets and that finish phase (the targets would be stale). */
int r2d2_learner_buffers_get_slot(r2d2_learner_t* l, int slot, r2d2_learner_buffers* out);
int r2d2_learner_select_batch(r2d2_learner_t* l, int slot);
int r2d2_learner_target_phase(r2d2_learner_t* l, int slot, r2d2_stream_t stream);
/* forget a target phase that ran ahead: the caller is about to overwrite that slot's batch */
int r2d2_learner_discard_prefetch(r2d2_learner_t* l, r2d2_stream_t stream);
/* phase 1: target chains (unless r2d2_learner_target_phase already ran for the selected slot), online critic chain,
 * TD/priority kernel, critic BPTT -> critic_grads */
int r2d2_learner_critic_phase(r2d2_learner_t* l, r2d2_stream_t stream);
/* optional, between phase 1 and phase 2: the actor's forward chain of the DPG update (learner.py:117,120-123; zero
 * state, 2 cell steps per row).  It does not read the critic, so a data-parallel caller issues it while the
 * all-reduce of critic_grads is in flight; phase 2 then skips it.  Without this call phase 2 runs it itself. */
int r2d2_learner_actor_forward(r2d2_learner_t* l, r2d2_stream_t stream);
/* phase 2: critic Adam (grads * grad_scale), actor chain unless r2d2_learner_actor_forward already ran, critic on
 * actor actions, dgrad through critic, actor BPTT -> actor_grads */
int r2d2_learner_actor_phase(r2d2_learner_t* l, float grad_scale, r2d2_stream_t stream);
/* phase 3: actor Adam, step counter, hard target update every target_update_interval steps */
int r2d2_learner_finish_phase(r2d2_learner_t* l, float grad_scale, r2d2_stream_t stream);
int r2d2_learner_step_count(r2d2_learner_t* l);
/* The critic phase pre-issues the input projection of the actor's DPG chain on a side stream (it reads the actor's
 * weights).  A caller that runs phase 3 of iteration i AFTER phase 1 of iteration i+1 (deferred actor all-reduce)
 * switches that off: the weights are not final yet. */
int r2d2_learner_set_overlap_actor_inputs(r2d2_learner_t* l, int on);
/* Data-parallel learner, one process per GPU (SURVEY 8e): the two gradient all-reduces of learner.py:113-114,127-128
 * as kernels of this library over NVLink peer memory, issued inside the phases on the learner's own stream (peer.cuh).
 * Every rank allocates `bytes` of zeroed device memory that all ranks of the node can map (CUDA IPC / fabric handles;
 * the Python host side uses torch's symmetric memory), exchanges the addresses and attaches them; the learner's
 * gradient blocks then live at off_*_grads of its own buffer and the optimiser kernels read off_*_sums.  The caller
 * keeps calling the phases in the same order on every rank and passes grad_scale = 1 / world.  Call order with the
 * loosest coupling: critic_phase(i), finish_phase(i-1), actor_forward(i), actor_phase(i). */
typedef struct {
  size_t bytes, off_critic_grads, off_actor_grads, off_critic_sums, off_actor_sums;
} r2d2_peer_layout;
int r2d2_learner_peer_layout(r2d2_learner_t* l, int world, r2d2_peer_layout* out);
/* the same from the two parameter counts (host arithmetic only) */
int r2d2_peer_layout_for(long long n_critic, long long n_actor, int world, r2d2_peer_layout* out);
int r2d2_learner_attach_peers(r2d2_learner_t* l, int rank, int world, void* const* peer_bases);
/* 0 = fine, 1 = a bounded wait (4 s) for a peer expired: the replicas are no longer in step (synchronises the stream) */
int r2d2_learner_peer_status(r2d2_learner_t* l, int* status, r2d2_stream_t stream);
/* diagnostics: nanoseconds summed since the last reset - [0..1] the slice-sum kernel waited for the peers' "gradients
 * complete" (critic, actor block), [2..3] the slice-sum kernel ran in total, [4..5] the wait kernel waited */
int r2d2_learner_peer_counters(r2d2_learner_t* l, unsigned long long* out6, int reset, r2d2_stream_t stream);
/* resume: completed iterations so far (drives Adam's bias correction and the target-update period, learner.py:82,131) */
int r2d2_learner_set_step_count(r2d2_learner_t* l, int step);
/* number of kernels launched by the three phases of one iteration (bench.py's gpu_launches) */
int r2d2_learner_launches_per_iteration(r2d2_learner_t* l);

/* ------------------------------------------------------------------------------------------------
 * Batched acting (the per-step loop body of actor.py:136-148 over B environments): one step of actor, target actor,
 * critic and target critic.  The critics are fed the UN-noised actions of their actors; noise and clipping stay on
 * the host (actor.py:146-148).  Supported: H a multiple of 32 in [32, 512], O >= 1, 1 <= A <= 32,
 * 1 <= B <= max_batch; anything else is rejected before any CUDA call.
 * ---------------------------------------------------------------------------------------------- */
typedef struct r2d2_act r2d2_act_t;

/* shape: obs_size, n_actions, hidden (is_critic ignored) */
int r2d2_act_create(r2d2_act_t** out, const r2d2_net_shape* shape, int max_batch);
int r2d2_act_destroy(r2d2_act_t* a);
/* flat DEVICE parameter blocks (state_dict order, see above) of actor, target_actor, critic, target_critic -> the
 * handle's packed weight images.  Stream-ordered; the blocks may be freed once the stream has passed this call. */
int r2d2_act_load(r2d2_act_t* a, const float* actor, const float* target_actor, const float* critic,
                  const float* target_critic, r2d2_stream_t stream);
/* obs [B,O]; state_in / state_out [4,2,B,H] in replay order (actor, target_actor, critic, target_critic) x (h, c),
 * 16-byte aligned; state_out must not alias state_in; mu [B,A] = the actor's un-noised action.  4 launches. */
int r2d2_act_step(r2d2_act_t* a, const float* obs, const float* state_in, float* state_out, float* mu, int B,
                  r2d2_stream_t stream);
/* *status != 0 if a bounded mbarrier wait inside an act kernel ever timed out; synchronises the stream */
int r2d2_act_status(r2d2_act_t* a, int* status, r2d2_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* R2D2_B200_H_ */
