/*
 * tsc_learn.h — C ABI of the per-intersection A2C learner kernels in libtsc (sm_100a).
 *
 * Replaces, for R lock-stepped replicas and all A agents at once, the TF1 graphs of the reference:
 *   fc / lstm layers                         agents/utils.py:66-74, 88-116
 *   LstmACPolicy / FPLstmACPolicy forward    agents/policies.py:99-136, 191-211
 *   ACPolicy.prepare_loss + backward         agents/policies.py:41-61, 138-155
 *   OnPolicyBuffer._add_R_Adv                agents/utils.py:202-214
 *   clip_by_global_norm + RMSPropOptimizer   agents/policies.py:54-61  (TF1 semantics: ms starts
 *                                            at 1, epsilon inside the sqrt, no momentum)
 * Two networks per agent (pi and V, agents/policies.py:87-96) = 2A "units"; unit u = 2*agent + net.
 *
 * All pointers are caller-owned DEVICE pointers; `stream` is a cudaStream_t as void*.
 * Every function returns 0 or <0 (message via tsc_last_error()).  The three plain time-batched
 * GEMMs of the update (X.Wx, dZ.Wx^T, X^T.dZ) are NOT in this ABI: the host calls the vendor
 * library for them (DESIGN.md §5) until the tcgen05 kernels replace them.
 */
#ifndef TSC_LEARN_H_
#define TSC_LEARN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Static shape/offset description of the A agents (host struct; arrays are HOST pointers, copied
 * by tscl_create).  Observation row of agent i (envs/env.py:163-205):
 *   [wave (n_wave[i]) | wait (n_wait[i]) | fingerprints (n_fp[i])] at obs_off[i]. */
typedef struct tscl_dims {
  int32_t n_agents;   /* A                                                                 */
  int32_t n_obs;      /* row stride of the observation matrix                              */
  int32_t max_na;     /* padded action dimension (row stride of pi / fingerprints)         */
  int32_t fw, ff, ft; /* fc widths: num_fw, num_fp (0 = no fingerprint branch), num_ft     */
  int32_t h;          /* num_lstm (must be 64)                                             */
  int32_t dx;         /* fw + ff + ft                                                      */
  const int32_t* obs_off;  /* [A]                                                          */
  const int32_t* n_wave;   /* [A]                                                          */
  const int32_t* n_wait;   /* [A]                                                          */
  const int32_t* n_fp;     /* [A]                                                          */
  const int32_t* n_a;      /* [A]                                                          */
  /* offsets (in floats) into the flat parameter / gradient / RMS-slot vectors             */
  const int64_t* off_fcw_w; /* [2A] ragged [n_wave][fw]   */ const int64_t* off_fcw_b; /* [2A] */
  const int64_t* off_fcf_w; /* [2A] ragged [n_fp][ff]     */ const int64_t* off_fcf_b; /* [2A] */
  const int64_t* off_fct_w; /* [2A] ragged [n_wait][ft]   */ const int64_t* off_fct_b; /* [2A] */
  int64_t off_wx;  /* [2A][dx][4h] */
  int64_t off_wh;  /* [2A][h][4h]  */
  int64_t off_bl;  /* [2A][4h]     */
  int64_t off_wo;  /* [2A][h][max_na]  (V units use column 0) */
  int64_t off_bo;  /* [2A][max_na] */
  int64_t n_params;
} tscl_dims;

typedef struct tscl_handle tscl_handle;

int tscl_create(const tscl_dims* dims, int32_t device, tscl_handle** out);
int tscl_destroy(tscl_handle* h);

/* fc front end (agents/policies.py:191-201): X[u][m][0:dx] = relu(fc(...)) for m in [0, M).
 * Row m reads obs + (m / rows_per_t) * stride_t + (m % rows_per_t) * n_obs  (floats). */
int tscl_fc_embed(tscl_handle* h, const float* params, const float* obs, int64_t M, int64_t rows_per_t,
                  int64_t stride_t, float* X, void* stream);

/* FcACPolicy hidden layer (agents/policies.py:236: `h = fc(h, out_type + '_fc', n_fc)`), own register-tiled fp32 GEMM
 * kernels (PolicyLayout(recurrent=False): wx [2A][dx][h], bl [2A][h]):
 *   fwd  H[u][m][:] = relu(X[u][m][:] . wx[u] + bl[u])                                  X [2A][M][dx], H [2A][M][h]
 *   bwd  dH <- dH * (H > 0);  dX = dH . wx^T;  grads.wx += X^T dH;  grads.bl += 1^T dH   (tf.gradients through relu + matmul) */
int tscl_fc_hidden_fwd(tscl_handle* h, const float* params, const float* X, int64_t M, float* H, void* stream);
int tscl_fc_hidden_bwd(tscl_handle* h, const float* params, const float* X, const float* H, float* dH, int64_t M,
                       float* dX, float* grads, void* stream);

/* LSTM over T steps (agents/utils.py:88-116): recurrent GEMM h.Wh + fused cell.
 *   ZG   [2A][T*Rc][4h]  in: X.Wx + b (time-major rows m = t*Rc + r); out: gate activations i,f,o,u
 *   C,H  [2A][T*Rc][h]   out (may be NULL when T == 1 and only states are wanted)
 *   Hprev [2A][T*Rc][h]  out, may be NULL: the masked h_{t-1} each step consumed (operand of dWh)
 *   c0,h0 [2A][ld_state][h] initial state rows r0 .. r0+Rc;  c1,h1: final state (may alias c0,h0, may be NULL)
 *   done [T] float (pre-step done: state is zeroed BEFORE the cell, agents/utils.py:104-105) */
int tscl_lstm_seq_fwd(tscl_handle* h, const float* params, float* ZG, float* C, float* H, float* Hprev,
                      const float* c0, const float* h0, float* c1, float* h1, const float* done, int32_t T,
                      int64_t Rc, int64_t ld_state, int64_t r0, void* stream);

/* Heads for one control step (agents/policies.py:18-26, utils.py:155-157): softmax policy, value,
 * categorical sample with the counter-based RNG keyed (seed, step, replica0 + r, agent).
 *   Hs [2A][R][h] -> pi [R][A][max_na] (zero padded), val [R][A], act [R][A] (may be NULL) */
int tscl_heads(tscl_handle* h, const float* params, const float* Hs, int64_t R, float* pi, float* val,
               int32_t* act, uint64_t seed, int64_t step, int64_t replica0, void* stream);

/* n-step returns (agents/utils.py:202-214): R_t = r_t + gamma*R_{t+1}*(1-done_post_t), Adv = R - v.
 *   rew,val,Rs,Adv [T][R][A]; boot [R][A]; done_post [T] float */
int tscl_returns(tscl_handle* h, const float* rew, const float* val, const float* boot, const float* done_post,
                 float gamma, int32_t T, int64_t R, float* Rs, float* Adv, void* stream);

/* Loss gradients at the heads for all (t, r) of a chunk (agents/policies.py:41-52):
 *   H [2A][M][h], act/Rs/Adv rows m -> base + (m / Rc)*stride_t + (m % Rc)*A
 *   dlog [2A][M][max_na] (out; V units use column 0), dH [2A][M][h] (out)
 *   stats [4] += {policy_loss, value_loss, entropy_loss, count} of agent 0 (agents/policies.py:63-72)
 *   scale = 1 / (n_step * total replicas): mean over the batch and over replicas
 *   h_bf16 (optional): read H from one chunk of the bf16 activation store ([2A][M][h]) instead of `H`
 *   grads (optional): also accumulate the head gradients  dWo += H^T dlog, dbo += sum dlog  into the flat
 *                     gradient vector; `dlog` may then be NULL */
int tscl_heads_loss(tscl_handle* h, const float* params, const float* H, const int32_t* act, const float* Rs,
                    const float* Adv, int64_t M, int64_t Rc, int64_t stride_t, float v_coef, float beta,
                    float scale, float* dlog, float* dH, float* stats, const void* h_bf16, float* grads,
                    void* stream);

/* BPTT through the LSTM (reverse of tscl_lstm_seq_fwd).  ZG holds gate activations on entry and
 * dZ (pre-activation gate gradients) on exit; dH holds head gradients on entry. */
int tscl_lstm_seq_bwd(tscl_handle* h, const float* params, float* ZG, const float* C, const float* dH,
                      const float* c0, const float* done, int32_t T, int64_t Rc, int64_t ld_state, int64_t r0,
                      void* stream);

/* fc front-end backward: grads[...] += obs^T . (dX * (X > 0)) and bias sums, rows as tscl_fc_embed. */
int tscl_fc_bwd(tscl_handle* h, const float* obs, const float* X, const float* dX, int64_t M,
                int64_t rows_per_t, int64_t stride_t, float* grads, void* stream);

/* The same contraction on the tensor cores (tcgen05, MN-major bf16 operands, fp32 accumulation in TMEM over
 * 128-row tiles; replaces the SIMT kernel in the training loop).  Pass the activations either as fp32 `X` or as one
 * chunk of the bf16 activation store `x_bf16` ([2A][M][dx]); `variant` must be 0. */
int tscl_fc_bwd_tc(tscl_handle* h, const float* obs, const float* X, const void* x_bf16, const float* dX,
                   const void* dx_bf16, int64_t M, int64_t rows_per_t, int64_t stride_t, float* grads, int32_t variant,
                   void* stream);
/* dX likewise as fp32 `dX` or bf16 `dx_bf16` ([2A][M][dx]). */

/* LSTM weight gradients of one chunk on the tensor cores:  grads.wx += X^T dZ, grads.wh += Hp^T dZ, grads.bl += 1^T dZ
 * (rows m = t * rc + r, M = T * rc; bf16 operands, fp32 accumulation in TMEM).  X as fp32 `X` or bf16 `x_bf16`
 * ([2A][M][dx]); Hp as fp32 `Hp` ([2A][M][h]) or rebuilt from the bf16 store chunk `h_bf16` ([2A][T][rc][h]) as
 * (1 - done[t]) * (t > 0 ? H[t-1] : h0[u][r0 + r]).  `variant` must be 0. */
int tscl_wgrad_tc(tscl_handle* h, const float* dZ, const void* dz_bf16, const float* X, const void* x_bf16,
                  const float* Hp, const void* h_bf16, const float* h0, const float* done, int32_t T, int64_t rc,
                  int64_t ld_state, int64_t r0, float* grads, int32_t variant, void* stream);
/* dZ likewise as fp32 `dZ` or bf16 `dz_bf16` ([2A][M][256], written by tscl_lstm_seq_bwd_tc). */

/* BPTT on the tensor cores (tcgen05): same contract as tscl_lstm_seq_bwd, with the recurrent product dz.Wh^T as
 * a bf16 MMA (M=128, N=64, K=256) per step; wt_bf16 [2A][32][64][8] comes from tscl_pack_wht (refresh after
 * every optimizer step).  With gates_bf16 / c_bf16 / dz_bf16 and ZG == NULL (the shipping call) the per-step operand tile
 * of 128 replicas (gates, c, dH: 112 KB) is fetched one step ahead by cp.async.bulk.tensor copies through tensor maps
 * built over the caller's arrays (cuTensorMapEncodeTiled via the driver entry point; TSC_BPTT_TMA=0 selects the
 * cp.async variant); the arrays must be 16-byte aligned and hold 2A * T * Rc rows. */
int tscl_pack_wht(tscl_handle* h, const float* params, void* wt_bf16, void* stream);
int tscl_lstm_seq_bwd_tc(tscl_handle* h, const void* wt_bf16, float* ZG, const float* C, const float* dH, const float* c0,
                         const float* done, int32_t T, int64_t Rc, int64_t ld_state, int64_t r0,
                         const void* gates_bf16, const void* c_bf16, void* dz_bf16, void* stream);
/* The same kernel with dX = dZ . Wx^T fused into every step (second tcgen05 product of the same dz tile, M=128, N=dx,
 * K=256, accumulator in TMEM columns 64..64+dx): wxt_bf16 [2A][32][dx][8] from tscl_pack_wxt (refresh after every
 * optimizer step), dx_bf16 [2A][T*Rc][dx] receives dX as bf16 — one way of replacing the last library GEMM of the update
 * (the shipping one is tscl_dx_tc below)
 * (reference: the tf.gradients chain through agents/utils.py:106, `tf.matmul(x, wx)`).  Both NULL = plain BPTT. */
int tscl_pack_wxt(tscl_handle* h, const float* params, void* wxt_bf16, void* stream);
int tscl_lstm_seq_bwd_tc_dx(tscl_handle* h, const void* wt_bf16, float* ZG, const float* C, const float* dH, const float* c0,
                            const float* done, int32_t T, int64_t Rc, int64_t ld_state, int64_t r0,
                            const void* gates_bf16, const void* c_bf16, void* dz_bf16, const void* wxt_bf16, void* dx_bf16,
                            void* stream);
/* Host-buffer loop, one call per replica range and control step (replaces the reference's per-step numpy hand-over of
 * ob / reward into `model.add_transition`, agents/models.py:222-229, main.py / utils.py:272-286): observations
 * host -> obs_dev (the rollout slot), rewards host -> rew_hist_dev = clip(reward / reward_norm) (0 = off for either),
 * global rewards host -> rew_acc_dev += (episode sum, utils.py:296-305).  *_stage_dev are device scratch of the same
 * size as the host arrays.  Host arrays should be page-locked; everything is enqueued on `stream`. */
int tscl_host_transition(tscl_handle* h, const float* obs_host, float* obs_dev, int64_t obs_floats, const float* rew_host,
                         float* rew_stage_dev, float* rew_hist_dev, int64_t rew_floats, float reward_norm, float reward_clip,
                         const float* grew_host, float* grew_stage_dev, float* rew_acc_dev, int64_t n, void* stream);
/* Same hand-over with the rewards already on the device (the device-resident loop): rew_hist_dev = clip(rew_dev /
 * reward_norm), rew_acc_dev += grew_dev, one launch. */
int tscl_device_transition(tscl_handle* h, const float* rew_dev, float* rew_hist_dev, int64_t rew_floats, float reward_norm,
                           float reward_clip, const float* grew_dev, float* rew_acc_dev, int64_t n, void* stream);
/* cudaMemcpyAsync on a caller-supplied stream; kind 1 = host->device, 2 = device->host, 3 = device->device */
int tscl_memcpy_async(tscl_handle* h, void* dst, const void* src, int64_t bytes, int32_t kind, void* stream);
/* dX = dZ . Wx^T as a stand-alone streaming product (the shipping path; reference: tf.gradients through
 * `tf.matmul(x, wx)`, agents/utils.py:106): dz_bf16 [2A][M][256], wxt_bf16 from tscl_pack_wxt, dx_bf16 [2A][M][dx] out.
 * Warp-specialised tcgen05 kernel (cp.async loaders -> 128B-swizzled operand stages, TMEM double buffer, bulk-copy stores).
 * dx must be a multiple of 16, <= 224 for the shared-memory budget. */
int tscl_dx_tc(tscl_handle* h, const void* dz_bf16, const void* wxt_bf16, void* dx_bf16, int64_t M, void* stream);
/* gates_bf16 / c_bf16 (both or neither): read gate activations and c_t straight from one chunk of the bf16
 * activation store instead of ZG / C (ZG is then write-only: it receives dZ).
 * dz_bf16 (optional): also write dZ as bf16 [2A][T*Rc][256]; with all three bf16 pointers ZG may be NULL. */

/* One replica chunk of the bf16 activation store ([2A][T][rc][w] contiguous) -> fp32 work buffers X, ZG (gates),
 * C, H and Hp[t] = (1 - done[t]) * (t > 0 ? H[t-1] : h0[:, r0 + r]).  Every output may be NULL (skipped): the
 * tensor-core kernels read the store themselves. */
int tscl_unpack_store(tscl_handle* h, const void* st_x, const void* st_g, const void* st_c, const void* st_h, float* X,
                      float* ZG, float* C, float* H, float* Hp, const float* h0, const float* done, int32_t T,
                      int64_t rc, int64_t ld_state, int64_t r0, void* stream);

/* Tools only (scripts/profile_policy_phases.py): per-phase clock64 sums of tscl_policy_step_v2 are added to 8 uint64
 * device counters while the pointer is set (NULL = off; a separate instantiation of the kernel, the hot one is unchanged). */
int tscl_debug_policy_prof(void* counters_dev);
/* same for the staged BPTT kernel: 8 counters (operand wait | smem->regs + cell backward + dZ stores | barrier | MMA + wait |
 * TMEM read-back), summed over CTAs; NULL switches profiling off */
int tscl_debug_bptt_prof(void* counters_dev);

/* Per-agent clip_by_global_norm(max_norm) + RMSProp step (TF1 semantics).  agent_of [n_params] u8.
 * norms [A] receives the pre-clip global norms. */
int tscl_clip_rmsprop(tscl_handle* h, float* params, float* grads, float* ms, const uint8_t* agent_of,
                      float max_norm, float lr, float alpha, float eps, float* norms, void* stream);

/* ---- fused tensor-core policy forward (tcgen05 + TMEM), csrc/tsc_policy_tc.cu -------------------------
 * tscl_pack_weights: per unit, [Wx;Wh] -> bf16 UMMA operand image [(dx+h)/8][4h][8] followed by the
 *   block-diagonal fc image [8][dx][8]; wpack holds 2A such records (call after every optimizer step).
 * tscl_policy_step: one decision for R replicas and all agents in ONE kernel: fc front end, gate GEMM on
 *   the tensor cores (bf16 operands, fp32 accumulate in TMEM), LSTM cell, heads, softmax, sampling.
 *   Replaces LstmACPolicy.forward / FPLstmACPolicy.forward for a whole batch (agents/policies.py:125-136).
 *   c_in/h_in/c_out/h_out [2A][R][h] (out may alias in); pi [R][A][max_na]; val [R][A]; act [R][A] or NULL;
 *   zdbg [2A][R][4h] raw gate accumulators (debug) or NULL; swap_lbo_sbo: debug switch, pass 0. */
int tscl_pack_weights(tscl_handle* h, const float* params, void* wpack_bf16, void* stream);
int tscl_policy_step(tscl_handle* h, const float* params, const void* wpack_bf16, const float* obs, int64_t R,
                     const float* c_in, const float* h_in, float* c_out, float* h_out, float* pi, float* val,
                     int32_t* act, int32_t done, uint64_t seed, int64_t step, int64_t replica0, float* zdbg,
                     int32_t swap_lbo_sbo, void* stream);

/* v2 of the fused forward: the fc front end runs on the tensor cores as well (observation slice tile x
 * block-diagonal fc weights -> TMEM -> relu/bf16 -> A operand).  Same arguments as tscl_policy_step
 * (without the descriptor debug switch); needs dx % 32 == 0.  wpack must come from tscl_pack_weights. */
int tscl_policy_step_v2(tscl_handle* h, const float* params, const void* wpack_bf16, const float* obs, int64_t R,
                        const float* c_in, const float* h_in, float* c_out, float* h_out, float* pi, float* val,
                        int32_t* act, int32_t done, uint64_t seed, int64_t step, int64_t replica0, float* zdbg,
                        void* st_x, void* st_g, void* st_c, void* st_h, int32_t t, int32_t T, int64_t rc, void* stream);
/* Replica-range form: R rows starting at absolute replica row0 of a batch of ld_state replicas.  Every pointer is the
 * base of the range's slice (obs + row0 * n_obs, c_in + row0 * h, pi + row0 * A * max_na, ...; the st_* pointers stay
 * the bases of the whole store); the per-unit state arrays keep ld_state rows per unit.  ld_state = 0: plain call. */
int tscl_policy_step_v2r(tscl_handle* h, const float* params, const void* wpack_bf16, const float* obs, int64_t R,
                         const float* c_in, const float* h_in, float* c_out, float* h_out, float* pi, float* val,
                         int32_t* act, int32_t done, uint64_t seed, int64_t step, int64_t replica0, float* zdbg,
                         void* st_x, void* st_g, void* st_c, void* st_h, int32_t t, int32_t T, int64_t rc,
                         int64_t ld_state, int64_t row0, void* stream);
/* st_x/st_g/st_c/st_h (all or none, may be NULL): bf16 activation store [R/rc][2A][T][rc][dx | 4h | h | h]
 * (replica-chunk major; rc must divide R) written at time index t — the relu'd fc outputs, the gate activations i,f,o,u, c_t and h_t — so that the update can
 * back-propagate through the rollout's own forward pass instead of recomputing it.
 * bf16 elements per unit in the packed weight image: ((dx+h)/8)*4h*8 + 8*dx*8 */

/* ---- batched independent Q-learning (IQL-LR / IQL-DQN), csrc/tsc_iql.cu ----------------------------------------
 * Replaces, for R lock-stepped replicas and all A agents at once, the reference's LRQPolicy / DeepQPolicy graphs
 * (agents/policies.py:285-389), epsilon-greedy acting (agents/models.py:347-362) and ReplayBuffer sampling
 * (agents/utils.py:231-263).  One Q network per agent, shared by all replicas.
 *   model 0 (lr):  q = S.Wq + bq
 *   model 1 (dqn): q = relu(relu([S_wave.Wf + bf | S_wait.Wt + bt]).W0 + b0).Wq + bq   (wait half only when n_w > 0,
 *                  width num_fc / 4; the wait inputs are the last n_w of the agent's n_s inputs)
 * Parameters of agent a lie contiguously in [par_off[a], par_off[a+1]) of one flat fp32 vector, in the order and
 * row-major [in][out] shapes of models.IQL: q_fcw/w, q_fcw/b, (q_fct/w, q_fct/b when n_w > 0), q_fc_0/w, q_fc_0/b,
 * q/w, q/b (dqn) or q/w, q/b (lr).  Gradients and the Adam moments use the same layout.
 * Replay ring of C transitions per replica (lock-step: every replica holds the same transition numbers n):
 *   obs [C+1][R][n_obs]  transition n reads s from slot n % (C+1) and s' from slot (n+1) % (C+1)
 *   act [C][R][A] int32, rew [C][R][A], done [C] float   transition n sits in slot n % C
 * n_total transitions have been stored; the live ones are the last min(n_total, C).
 * Limits (checked by tscl_iql_create): n_s <= 64, max_na <= 8, num_fc <= 128 (a multiple of 4), num_h <= 64. */
typedef struct tscl_iql_dims {
  int32_t n_agents;        /* A                                           */
  int32_t n_obs;           /* row stride of the observation matrix        */
  int32_t max_na;          /* row stride of the q output                  */
  int32_t model;           /* 0 = lr, 1 = dqn                             */
  int32_t num_fc, num_h;   /* dqn widths (ignored for lr)                 */
  const int32_t* obs_off;  /* [A] first input of agent a in an obs row    */
  const int32_t* n_s;      /* [A] inputs, wait inputs included            */
  const int32_t* n_w;      /* [A] wait inputs (dqn only)                  */
  const int32_t* n_a;      /* [A]                                         */
  const int64_t* par_off;  /* [A + 1]                                     */
} tscl_iql_dims;

typedef struct tscl_iql_handle tscl_iql_handle;

int tscl_iql_create(const tscl_iql_dims* dims, int32_t device, tscl_iql_handle** out);
int tscl_iql_destroy(tscl_iql_handle* h);
/* obs [R][n_obs] -> act [R][A]: argmax_j q (ties to the lowest j) or, when a uniform draw is < eps, a uniform action in
 * [0, n_a); draws keyed (seed, step, replica0 + r, agent).  q [R][A][max_na] (zero padded) may be NULL. */
int tscl_iql_forward(tscl_iql_handle* h, const float* params, const float* obs, int64_t R, float eps, uint64_t seed,
                     int64_t step, int64_t replica0, int32_t* act, float* q, void* stream);
/* idx [A][R][B]: B distinct ring slots in [0, size) per (agent, replica), keyed (seed, update, iter, agent,
 * replica0 + r).  Needs B <= size. */
int tscl_iql_sample(tscl_iql_handle* h, int64_t R, int32_t B, int64_t size, uint64_t seed, int64_t update, int32_t iter,
                    int64_t replica0, int32_t* idx, void* stream);
/* TD loss of the rows selected by idx [A][R][B] (ring slots):  loss_a = scale * sum (q(s)[a] - tq)^2 with
 * tq = done ? r : r + gamma max q(s') (same weights: no target network).  grads (whole flat vector) = d loss / d params;
 * stats [A][2] (may be NULL) = {loss_a, scale * sum q(s)[a]}.  Per-CTA partials summed in a fixed order: the same
 * inputs give the same bits. */
int tscl_iql_td_grad(tscl_iql_handle* h, const float* params, const float* obs_ring, const int32_t* act_ring,
                     const float* rew_ring, const float* done_ring, int64_t C, int64_t n_total, int64_t R, int32_t B,
                     const int32_t* idx, float gamma, float scale, float* grads, float* stats, void* stream);
/* per-agent clip_by_global_norm(max_norm) (0 = off) + TF1 Adam (beta1 0.9, beta2 0.999, epsilon 1e-8 outside the
 * sqrt) with lr_t = lr sqrt(1 - beta2^t) / (1 - beta1^t) computed by the caller.  norms [A] (may be NULL) receives the
 * pre-clip norms. */
int tscl_iql_clip_adam(tscl_iql_handle* h, float* params, const float* grads, float* m, float* v, float max_norm,
                       float lr_t, float* norms, void* stream);
/* reward hand-over into a ring slot, the arithmetic of tscl_device_transition: rew_slot = clip(rew / reward_norm),
 * rew_acc[0, n) += grew (0 = off for norm / clip) */
int tscl_iql_transition(tscl_iql_handle* h, const float* rew, float* rew_slot, int64_t rew_floats, float reward_norm,
                        float reward_clip, const float* grew, float* rew_acc, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TSC_LEARN_H_ */
