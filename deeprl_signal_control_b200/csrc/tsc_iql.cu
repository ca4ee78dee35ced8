// tsc_iql.cu — hand-written sm_100a kernels of the batched independent Q-learner (IQL) + C ABI (include/tsc_learn.h).
// fp32 storage and arithmetic (the reference is fp32 TF1).
//
//   iql_forward_kernel   Q network forward + epsilon-greedy actions       agents/models.py:347-362, policies.py:285-389
//   iql_sample_kernel    batch_size distinct ring indices per (agent, replica)   agents/utils.py:255-263 (random.sample)
//   iql_td_kernel        gather s, a, r, done, s' from the replay ring; forward on s' (target, no target network) and
//                        on s, backward on s, per-CTA gradient partials   agents/policies.py:307-338
//   iql_reduce_kernel    fixed-order sum of the per-CTA partials (deterministic: no float atomics)
//   iql_norm_kernel / iql_adam_kernel   per-agent clip_by_global_norm + TF1 Adam   agents/policies.py:325-329
//
// Networks (one per agent, ragged shapes; models.IQL._q):
//   lr    q = S.Wq + bq
//   dqn   h1 = [relu(S_wave.Wf + bf) | relu(S_wait.Wt + bt)]  (the wait half only when n_w > 0, width num_fc / 4)
//         h2 = relu(h1.W0 + b0),  q = h2.Wq + bq
// Agent a's tensors lie contiguously from par_off[a] in the order of models.IQL: q_fcw/w [n_s-n_w][num_fc], q_fcw/b,
// q_fct/w [n_w][num_fc/4], q_fct/b (n_w > 0 only), q_fc_0/w [width][num_h], q_fc_0/b, q/w [num_h][n_a], q/b  (dqn), or
// q/w [n_s][n_a], q/b (lr); weights row-major [in][out].  Gradients and the Adam moments use the same layout.
//
// A CTA works on one agent: the agent's weights are staged into shared memory once (row pitch padded by one float
// against bank conflicts) and the rows are processed in tiles of IQ_TR rows held feature-major ([feature][row]).
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/tsc_learn.h"

int tsc_set_error(const std::string& m);  // defined in tsc_sim.cu
// reward hand-over shared with tscl_device_transition (tsc_learn.cu)
int tscl_launch_reward_transition(int device, const float* rew, float* rew_hist, int64_t n_rew, float reward_norm,
                                  float reward_clip, const float* grew, float* rew_acc, int64_t n, cudaStream_t st);

#define ICK(call)                                                                  \
  do {                                                                             \
    cudaError_t e__ = (call);                                                      \
    if (e__ != cudaSuccess) return tsc_set_error(std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)

#define IQ_TR 64            // rows per tile
#define IQ_LD (IQ_TR + 1)   // pitch of the feature-major tile buffers
#define IQ_NT 512           // threads per CTA (dqn)
#define IQ_CTAS 296         // target CTAs of a dqn launch (2 per SM of a B200); fixed so that results do not depend on the device
// lr: the network is tiny and a tile is a chain of dependent gathers, so the TD kernel runs small CTAs, many per SM
#define IQ_NT_LR 128
#define IQ_CTAS_LR 1184     // 8 per SM of a B200

// shared-memory plan of one agent (offsets in floats); identical on host (sizing) and device
struct IqlLay {
  int dqn, ns, nw, na, nwv, nf, nt4, nh1, nh;
  int wf, bf, wt, bt, w0, b0, wq, bq;          // padded weights in shared memory
  int gf, gbf, gt, gbt, g0, gb0, gq, gbq;      // the same tensors in the agent's flat block
  int P;                                       // floats of the flat block
  int x, h1, h2, q, rows, grad, total;         // tile buffers, gradient accumulator (TD kernel only), size
};

__host__ __device__ inline IqlLay iql_lay(int dqn, int ns, int nw, int na, int nf, int nh, int max_na, bool td) {
  IqlLay L{};
  L.dqn = dqn; L.ns = ns; L.nw = dqn ? nw : 0; L.na = na;
  L.nwv = ns - L.nw; L.nf = nf; L.nt4 = L.nw > 0 ? nf / 4 : 0; L.nh1 = nf + L.nt4; L.nh = nh;
  int s = 0, g = 0;
  if (dqn) {
    L.wf = s; s += L.nwv * (nf + 1); L.gf = g; g += L.nwv * nf;
    L.bf = s; s += nf;               L.gbf = g; g += nf;
    L.wt = s; s += L.nw * (L.nt4 + 1); L.gt = g; g += L.nw * L.nt4;
    L.bt = s; s += L.nt4;            L.gbt = g; g += L.nt4;
    L.w0 = s; s += L.nh1 * (nh + 1); L.g0 = g; g += L.nh1 * nh;
    L.b0 = s; s += nh;               L.gb0 = g; g += nh;
    L.wq = s; s += nh * (na + 1);    L.gq = g; g += nh * na;
  } else {
    L.wq = s; s += ns * (na + 1);    L.gq = g; g += ns * na;
  }
  L.bq = s; s += na; L.gbq = g; g += na;
  L.P = g;
  L.x = s; s += ns * IQ_LD;
  L.h1 = s; s += (dqn ? L.nh1 : 0) * IQ_LD;
  L.h2 = s; s += (dqn ? nh : 0) * IQ_LD;
  L.q = s; s += max_na * IQ_LD;
  L.rows = s; s += 5 * IQ_TR;                  // reward, done, action, target, dloss/dq0 per row
  L.grad = s; if (td) s += g;
  L.total = s;
  return L;
}

struct IqlDev {
  int A, n_obs, max_na, dqn, nf, nh;
  const int32_t *obs_off, *n_s, *n_w, *n_a;
  const int64_t* par_off;
};

struct tscl_iql_handle {
  int device = 0;
  IqlDev d{};
  int64_t p_max = 0;          // largest flat block of one agent
  size_t smem_fwd = 0, smem_td = 0;
  std::vector<void*> owned;
  float* partial = nullptr;   // per-CTA gradient partials of the TD kernel
  size_t partial_floats = 0;
};

__device__ __forceinline__ uint64_t iq_mix(uint64_t z) {      // splitmix64 finaliser
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
// counter-based key: the same (seed, a, b, c, d) gives the same bits whatever the launch geometry
__device__ __forceinline__ uint64_t iq_key(uint64_t seed, uint64_t a, uint64_t b, uint64_t c, uint64_t d) {
  return iq_mix(iq_mix(iq_mix(iq_mix(iq_mix(seed) ^ a) ^ b) ^ c) ^ d);
}
__device__ __forceinline__ uint32_t iq_below(uint64_t h, uint32_t n) {      // uniform in [0, n) from 32 random bits
  return (uint32_t)(((uint64_t)(uint32_t)h * n) >> 32);
}

// OUT(i, c) = sum_t A[i*ai + t*at] * B[t*bt + c*bc] for i < NI, c < NC; 4 x 4 outputs per work item, epi(i, c, value).
// The item -> thread map depends on (NI, NC) only, so an accumulating epilogue always runs on the same thread.
template <class Epi>
__device__ __forceinline__ void iq_gemm(int NI, int NC, int K, const float* A, int ai, int at, const float* B, int bt,
                                        int bc, Epi epi) {
  const int ncb = (NC + 3) >> 2, items = ((NI + 3) >> 2) * ncb;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int i0 = (it / ncb) * 4, c0 = (it % ncb) * 4;
    const float* Ap[4];
    const float* Bp[4];
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      Ap[x] = A + min(i0 + x, NI - 1) * ai;
      Bp[x] = B + min(c0 + x, NC - 1) * bc;
    }
    float acc[4][4];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) acc[x][y] = 0.f;
    for (int t = 0; t < K; ++t) {
      float a[4], b[4];
#pragma unroll
      for (int x = 0; x < 4; ++x) { a[x] = Ap[x][t * at]; b[x] = Bp[x][t * bt]; }
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(a[x], b[y], acc[x][y]);
    }
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y)
        if (i0 + x < NI && c0 + y < NC) epi(i0 + x, c0 + y, acc[x][y]);
  }
}

__device__ inline IqlLay iq_agent_lay(const IqlDev& d, int a, bool td) {
  return iql_lay(d.dqn, d.n_s[a], d.n_w[a], d.n_a[a], d.nf, d.nh, d.max_na, td);
}

// flat [K][N] -> shared [K][N + 1]
__device__ __forceinline__ void iq_stage(float* dst, const float* src, int K, int N) {
  for (int e = threadIdx.x; e < K * N; e += blockDim.x) dst[(e / N) * (N + 1) + e % N] = src[e];
}
__device__ void iq_stage_weights(const IqlLay& L, float* sm, const float* P) {
  if (L.dqn) {
    iq_stage(sm + L.wf, P + L.gf, L.nwv, L.nf);
    iq_stage(sm + L.bf, P + L.gbf, 1, L.nf);
    if (L.nw > 0) {
      iq_stage(sm + L.wt, P + L.gt, L.nw, L.nt4);
      iq_stage(sm + L.bt, P + L.gbt, 1, L.nt4);
    }
    iq_stage(sm + L.w0, P + L.g0, L.nh1, L.nh);
    iq_stage(sm + L.b0, P + L.gb0, 1, L.nh);
    iq_stage(sm + L.wq, P + L.gq, L.nh, L.na);
  } else {
    iq_stage(sm + L.wq, P + L.gq, L.ns, L.na);
  }
  iq_stage(sm + L.bq, P + L.gbq, 1, L.na);
}

// q[j][r] for the IQ_TR rows in x (feature-major); leaves h1 / h2 (dqn) for the backward.  Ends synchronised.
__device__ void iq_q_forward(const IqlLay& L, float* sm) {
  float *X = sm + L.x, *Q = sm + L.q;
  const float* bq = sm + L.bq;
  const float* Hin = X;
  int K = L.ns;
  if (L.dqn) {
    float *H1 = sm + L.h1, *H2 = sm + L.h2;
    const float *bf = sm + L.bf, *bt = sm + L.bt, *b0 = sm + L.b0;
    iq_gemm(L.nf, IQ_TR, L.nwv, sm + L.wf, 1, L.nf + 1, X, IQ_LD, 1,
            [&](int i, int c, float v) { H1[i * IQ_LD + c] = fmaxf(v + bf[i], 0.f); });
    if (L.nw > 0)
      iq_gemm(L.nt4, IQ_TR, L.nw, sm + L.wt, 1, L.nt4 + 1, X + L.nwv * IQ_LD, IQ_LD, 1,
              [&](int i, int c, float v) { H1[(L.nf + i) * IQ_LD + c] = fmaxf(v + bt[i], 0.f); });
    __syncthreads();
    iq_gemm(L.nh, IQ_TR, L.nh1, sm + L.w0, 1, L.nh + 1, H1, IQ_LD, 1,
            [&](int i, int c, float v) { H2[i * IQ_LD + c] = fmaxf(v + b0[i], 0.f); });
    __syncthreads();
    Hin = H2;
    K = L.nh;
  }
  iq_gemm(L.na, IQ_TR, K, sm + L.wq, 1, L.na + 1, Hin, IQ_LD, 1,
          [&](int i, int c, float v) { Q[i * IQ_LD + c] = v + bq[i]; });
  __syncthreads();
}

// rows [0, nr) of the tile from `row(r)` (pointer to the agent's n_s inputs), zeros beyond
template <class RowPtr>
__device__ __forceinline__ void iq_load_x(const IqlLay& L, float* sm, int nr, RowPtr row) {
  float* X = sm + L.x;
  for (int e = threadIdx.x; e < IQ_TR * L.ns; e += blockDim.x) {
    const int r = e / L.ns, k = e % L.ns;
    X[k * IQ_LD + r] = r < nr ? row(r)[k] : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------
// acting: grid (chunks, A).  obs [R][n_obs] -> act [R][A], q [R][A][max_na] (optional, zero padded)
__global__ void __launch_bounds__(IQ_NT, 1)
iql_forward_kernel(IqlDev d, const float* __restrict__ params, const float* __restrict__ obs, int64_t R, float eps,
                   uint64_t seed, int64_t step, int64_t replica0, int32_t* __restrict__ act, float* __restrict__ qout) {
  extern __shared__ float sm[];
  const int a = blockIdx.y;
  const IqlLay L = iq_agent_lay(d, a, false);
  iq_stage_weights(L, sm, params + d.par_off[a]);
  const float* Q = sm + L.q;
  const int64_t n_tiles = (R + IQ_TR - 1) / IQ_TR;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * IQ_TR;
    const int nr = (int)min((int64_t)IQ_TR, R - r0);
    __syncthreads();                                  // previous tile's consumers of x / q are done
    const float* base = obs + r0 * d.n_obs + d.obs_off[a];
    iq_load_x(L, sm, nr, [&](int r) { return base + (int64_t)r * d.n_obs; });
    __syncthreads();
    iq_q_forward(L, sm);
    const int r = threadIdx.x;
    if (r < nr) {
      const int64_t rg = r0 + r;
      int best = 0;
      float qb = Q[r];
      for (int j = 1; j < L.na; ++j)                  // ties -> lowest index (np.argmax)
        if (Q[j * IQ_LD + r] > qb) { qb = Q[j * IQ_LD + r]; best = j; }
      if (eps > 0.f) {
        const uint64_t h = iq_key(seed, 0x51ull, (uint64_t)step, (uint64_t)(replica0 + rg), (uint64_t)a);
        if ((float)(h >> 40) * (1.0f / 16777216.0f) < eps) best = (int)iq_below(h, (uint32_t)L.na);
      }
      act[rg * d.A + a] = best;
      if (qout) {
        float* qo = qout + (rg * d.A + a) * d.max_na;
        for (int j = 0; j < d.max_na; ++j) qo[j] = j < L.na ? Q[j * IQ_LD + r] : 0.f;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// replay sampling: one thread per (agent, replica) row, Floyd's algorithm -> B distinct indices in [0, size).
__global__ void iql_sample_kernel(int A, int64_t R, int B, int64_t size, uint64_t seed, int64_t update, int iter,
                                  int64_t replica0, int32_t* __restrict__ idx) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)A * R) return;
  const int a = (int)(t / R);
  const int64_t r = t % R;
  int32_t* out = idx + t * B;
  const uint64_t key = iq_key(seed, 0x5a3ull, (uint64_t)update, ((uint64_t)iter << 32) | (uint32_t)a,
                              (uint64_t)(replica0 + r));
  int cnt = 0;
  for (int64_t j = size - B; j < size; ++j) {
    const int32_t v = (int32_t)iq_below(iq_mix(key + (uint64_t)j), (uint32_t)(j + 1));
    bool seen = false;
    for (int k = 0; k < cnt; ++k) seen |= (out[k] == v);
    out[cnt++] = seen ? (int32_t)j : v;
  }
}

// ------------------------------------------------------------------------------------------------
// TD loss gradient: grid (chunks, A).  Row m of agent a = (replica m / B, sample m % B); ring slot k = idx[a][r][b].
struct IqlRing {
  const float* obs;       // [C + 1][R][n_obs]
  const int32_t* act;     // [C][R][A]
  const float* rew;       // [C][R][A]
  const float* done;      // [C]
  int64_t C, n_total, R;
};

template <int NT, int MIN_CTAS>
__global__ void __launch_bounds__(NT, MIN_CTAS)
iql_td_kernel(IqlDev d, const float* __restrict__ params, IqlRing ring, int B, const int32_t* __restrict__ idx,
              float gamma, float scale, float* __restrict__ partial, int64_t p_max, float* __restrict__ stat_partial) {
  extern __shared__ float sm[];
  const int a = blockIdx.y;
  const IqlLay L = iq_agent_lay(d, a, true);
  iq_stage_weights(L, sm, params + d.par_off[a]);
  float* G = sm + L.grad;
  for (int e = threadIdx.x; e < L.P; e += blockDim.x) G[e] = 0.f;
  float *X = sm + L.x, *Q = sm + L.q, *H1 = sm + L.h1, *H2 = sm + L.h2;
  float *rr = sm + L.rows, *dn = rr + IQ_TR, *tq = rr + 3 * IQ_TR, *gq = rr + 4 * IQ_TR;
  int* ac = reinterpret_cast<int*>(rr + 2 * IQ_TR);
  const int64_t rows = ring.R * B, n_tiles = (rows + IQ_TR - 1) / IQ_TR;
  const int64_t base = ring.n_total - ring.C;         // first live transition when the ring is full
  const int A = d.A;
  float loss_acc = 0.f, q_acc = 0.f;
  __shared__ int64_t s_obs[IQ_TR], s_nxt[IQ_TR];      // float offsets of the rows' s and s' in the observation ring
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m0 = tile * IQ_TR;
    const int nr = (int)min((int64_t)IQ_TR, rows - m0);
    __syncthreads();
    if (threadIdx.x < IQ_TR) {
      const int r = threadIdx.x;
      if (r < nr) {
        const int64_t m = m0 + r, rep = m / B;
        const int64_t k = idx[((int64_t)a * ring.R + rep) * B + (m % B)];
        // transition number held by ring slot k (slot = n % C); observations of n and n + 1 sit at n % (C + 1), ...
        const int64_t n = ring.n_total <= ring.C ? k : base + (((k - base) % ring.C) + ring.C) % ring.C;
        s_obs[r] = ((n % (ring.C + 1)) * ring.R + rep) * d.n_obs + d.obs_off[a];
        s_nxt[r] = (((n + 1) % (ring.C + 1)) * ring.R + rep) * d.n_obs + d.obs_off[a];
        rr[r] = ring.rew[(k * ring.R + rep) * A + a];
        ac[r] = ring.act[(k * ring.R + rep) * A + a];
        dn[r] = ring.done[k];
      }
    }
    __syncthreads();
    // target: no target network, the same weights (agents/policies.py:318-322)
    iq_load_x(L, sm, nr, [&](int r) { return ring.obs + s_nxt[r]; });
    __syncthreads();
    iq_q_forward(L, sm);
    if (threadIdx.x < IQ_TR) {
      const int r = threadIdx.x;
      float mx = Q[r];
      for (int j = 1; j < L.na; ++j) mx = fmaxf(mx, Q[j * IQ_LD + r]);
      tq[r] = dn[r] != 0.f ? rr[r] : rr[r] + gamma * mx;
    }
    iq_load_x(L, sm, nr, [&](int r) { return ring.obs + s_obs[r]; });
    __syncthreads();
    iq_q_forward(L, sm);
    // dloss/dq = 2 (q0 - tq) * scale at the taken action; Q becomes dQ
    if (threadIdx.x < IQ_TR) {
      const int r = threadIdx.x;
      float g = 0.f;
      int ar = -1;
      if (r < nr) {
        ar = ac[r];
        const float q0 = Q[ar * IQ_LD + r], dlt = q0 - tq[r];
        loss_acc = fmaf(dlt, dlt, loss_acc);
        q_acc += q0;
        g = 2.f * dlt * scale;
      }
      gq[r] = g;
      for (int j = 0; j < L.na; ++j) Q[j * IQ_LD + r] = j == ar ? g : 0.f;
    }
    __syncthreads();
    const float* Hq = L.dqn ? H2 : X;                 // input of the q layer
    iq_gemm(L.dqn ? L.nh : L.ns, L.na, nr, Hq, IQ_LD, 1, Q, 1, IQ_LD,
            [&](int i, int c, float v) { G[L.gq + i * L.na + c] += v; });
    for (int j = threadIdx.x; j < L.na; j += blockDim.x) {
      float s = 0.f;
      for (int r = 0; r < nr; ++r) s += Q[j * IQ_LD + r];
      G[L.gbq + j] += s;
    }
    if (!L.dqn) continue;
    __syncthreads();
    // dZ2 = (h2 > 0) * Wq[:, a] * g, in place of h2
    {
      const float* Wq = sm + L.wq;
      for (int e = threadIdx.x; e < L.nh * IQ_TR; e += blockDim.x) {
        const int k = e / IQ_TR, r = e % IQ_TR;
        float& h = H2[k * IQ_LD + r];
        h = (r < nr && h > 0.f) ? Wq[k * (L.na + 1) + ac[r]] * gq[r] : 0.f;
      }
    }
    __syncthreads();
    iq_gemm(L.nh1, L.nh, nr, H1, IQ_LD, 1, H2, 1, IQ_LD,
            [&](int i, int c, float v) { G[L.g0 + i * L.nh + c] += v; });
    for (int j = threadIdx.x; j < L.nh; j += blockDim.x) {
      float s = 0.f;
      for (int r = 0; r < nr; ++r) s += H2[j * IQ_LD + r];
      G[L.gb0 + j] += s;
    }
    __syncthreads();
    // dZ1 = (h1 > 0) * (dZ2 . W0^T), in place of h1
    iq_gemm(L.nh1, IQ_TR, L.nh, sm + L.w0, L.nh + 1, 1, H2, IQ_LD, 1, [&](int i, int c, float v) {
      float& h = H1[i * IQ_LD + c];
      h = h > 0.f ? v : 0.f;
    });
    __syncthreads();
    iq_gemm(L.nwv, L.nf, nr, X, IQ_LD, 1, H1, 1, IQ_LD,
            [&](int i, int c, float v) { G[L.gf + i * L.nf + c] += v; });
    if (L.nw > 0)
      iq_gemm(L.nw, L.nt4, nr, X + L.nwv * IQ_LD, IQ_LD, 1, H1 + L.nf * IQ_LD, 1, IQ_LD,
              [&](int i, int c, float v) { G[L.gt + i * L.nt4 + c] += v; });
    for (int j = threadIdx.x; j < L.nh1; j += blockDim.x) {
      float s = 0.f;
      for (int r = 0; r < nr; ++r) s += H1[j * IQ_LD + r];
      G[(j < L.nf ? L.gbf + j : L.gbt + j - L.nf)] += s;
    }
  }
  __syncthreads();
  const int64_t cta = (int64_t)a * gridDim.x + blockIdx.x;
  for (int e = threadIdx.x; e < L.P; e += blockDim.x) partial[cta * p_max + e] = G[e];
  // per-CTA loss / q sums, fixed order
  if (threadIdx.x < IQ_TR) { tq[threadIdx.x] = loss_acc; gq[threadIdx.x] = q_acc; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float l = 0.f, q = 0.f;
    for (int r = 0; r < IQ_TR; ++r) { l += tq[r]; q += gq[r]; }
    stat_partial[cta * 2] = l * scale;
    stat_partial[cta * 2 + 1] = q * scale;
  }
}

// grads[par_off[a] + e] = sum over the agent's CTAs c = 0 .. n_cta-1 (in that order) of partial[a][c][e]
__global__ void iql_reduce_kernel(IqlDev d, const float* __restrict__ partial, int64_t p_max, int n_cta,
                                  float* __restrict__ grads, const float* __restrict__ stat_partial,
                                  float* __restrict__ stats) {
  const int a = blockIdx.y;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t P = d.par_off[a + 1] - d.par_off[a];
  if (e < P) {
    float s = 0.f;
    for (int c = 0; c < n_cta; ++c) s += partial[((int64_t)a * n_cta + c) * p_max + e];
    grads[d.par_off[a] + e] = s;
  }
  if (stats && blockIdx.x == 0 && threadIdx.x < 2) {
    float s = 0.f;
    for (int c = 0; c < n_cta; ++c) s += stat_partial[((int64_t)a * n_cta + c) * 2 + threadIdx.x];
    stats[a * 2 + threadIdx.x] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// per-agent global norm (one CTA per agent, fixed-order tree) and TF1 Adam
__global__ void __launch_bounds__(256) iql_norm_kernel(IqlDev d, const float* __restrict__ g, float* __restrict__ norm2) {
  __shared__ float red[8];
  const int a = blockIdx.x;
  float s = 0.f;
  for (int64_t e = d.par_off[a] + threadIdx.x; e < d.par_off[a + 1]; e += blockDim.x) s = fmaf(g[e], g[e], s);
  for (int o = 16; o; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    norm2[a] = t;
  }
}

__global__ void iql_adam_kernel(IqlDev d, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                float* __restrict__ v, const float* __restrict__ norm2, float max_norm, float lr_t,
                                float* __restrict__ norms) {
  const int a = blockIdx.y;
  const int64_t i = d.par_off[a] + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const float nrm = sqrtf(norm2[a]);
  if (norms && blockIdx.x == 0 && threadIdx.x == 0) norms[a] = nrm;
  if (i >= d.par_off[a + 1]) return;
  float gi = g[i];
  if (max_norm > 0.f) gi *= max_norm / fmaxf(nrm, max_norm);       // tf.clip_by_global_norm
  const float mi = m[i] + (gi - m[i]) * 0.1f;                       // beta1 = 0.9
  const float vi = v[i] + (gi * gi - v[i]) * 0.001f;                // beta2 = 0.999
  m[i] = mi;
  v[i] = vi;
  p[i] -= lr_t * mi / (sqrtf(vi) + 1e-8f);                          // epsilon outside the sqrt
}

// ================================================================================================
static int iq_up(tscl_iql_handle* h, const void* src, size_t bytes, const void** dst) {
  void* p = nullptr;
  ICK(cudaMalloc(&p, bytes ? bytes : 16));
  if (bytes) ICK(cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice));
  h->owned.push_back(p);
  *dst = p;
  return 0;
}

extern "C" int tscl_iql_destroy(tscl_iql_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  for (void* p : h->owned) cudaFree(p);
  if (h->partial) cudaFree(h->partial);
  delete h;
  return 0;
}

extern "C" int tscl_iql_create(const tscl_iql_dims* x, int32_t device, tscl_iql_handle** out) {
  if (!x || !out || x->n_agents <= 0 || !x->obs_off || !x->n_s || !x->n_w || !x->n_a || !x->par_off)
    return tsc_set_error("tscl_iql_create: bad argument");
  if (x->model != 0 && x->model != 1) return tsc_set_error("tscl_iql_create: model must be 0 (lr) or 1 (dqn)");
  if (x->max_na < 1 || x->max_na > 8) return tsc_set_error("tscl_iql_create: max_na must be in [1, 8]");
  if (x->model == 1 && (x->num_fc < 4 || x->num_fc > 128 || x->num_fc % 4 || x->num_h < 1 || x->num_h > 64))
    return tsc_set_error("tscl_iql_create: dqn needs num_fc in [4, 128] (a multiple of 4) and num_h in [1, 64]");
  int dev_count = 0;
  ICK(cudaGetDeviceCount(&dev_count));
  if (device < 0 || device >= dev_count) return tsc_set_error("tscl_iql_create: no such CUDA device");
  ICK(cudaSetDevice(device));
  const int A = x->n_agents;
  size_t smem_fwd = 0, smem_td = 0;
  int64_t p_max = 0, off = 0;
  for (int a = 0; a < A; ++a) {
    const int ns = x->n_s[a], nw = x->model == 1 ? x->n_w[a] : 0, na = x->n_a[a];
    if (ns < 1 || ns > 64 || nw < 0 || nw >= ns || na < 1 || na > x->max_na || x->obs_off[a] < 0 ||
        x->obs_off[a] + ns > x->n_obs)
      return tsc_set_error("tscl_iql_create: agent shapes out of range (n_s in [1, 64], n_w < n_s, n_a <= max_na)");
    const IqlLay Lf = iql_lay(x->model, ns, nw, na, x->num_fc, x->num_h, x->max_na, false);
    const IqlLay Lt = iql_lay(x->model, ns, nw, na, x->num_fc, x->num_h, x->max_na, true);
    if (x->par_off[a] != off) return tsc_set_error("tscl_iql_create: par_off does not match the agents' shapes");
    off += Lf.P;
    if (Lf.P > p_max) p_max = Lf.P;
    if ((size_t)Lf.total * 4 > smem_fwd) smem_fwd = (size_t)Lf.total * 4;
    if ((size_t)Lt.total * 4 > smem_td) smem_td = (size_t)Lt.total * 4;
  }
  if (x->par_off[A] != off) return tsc_set_error("tscl_iql_create: par_off[A] != total parameter count");
  int smem_max = 0;
  ICK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  if (smem_td + 2 * IQ_TR * 8 > (size_t)smem_max)
    return tsc_set_error("tscl_iql_create: an agent's network does not fit into shared memory");
  tscl_iql_handle* h = new tscl_iql_handle();
  h->device = device;
  h->p_max = p_max;
  h->smem_fwd = smem_fwd;
  h->smem_td = smem_td;
  IqlDev& d = h->d;
  d.A = A; d.n_obs = x->n_obs; d.max_na = x->max_na; d.dqn = x->model; d.nf = x->num_fc; d.nh = x->num_h;
  int rc = 0;
  const void* p;
  rc |= iq_up(h, x->obs_off, A * 4, &p); d.obs_off = (const int32_t*)p;
  rc |= iq_up(h, x->n_s, A * 4, &p); d.n_s = (const int32_t*)p;
  std::vector<int32_t> nw(A);
  for (int a = 0; a < A; ++a) nw[a] = x->model == 1 ? x->n_w[a] : 0;
  rc |= iq_up(h, nw.data(), A * 4, &p); d.n_w = (const int32_t*)p;
  rc |= iq_up(h, x->n_a, A * 4, &p); d.n_a = (const int32_t*)p;
  rc |= iq_up(h, x->par_off, (A + 1) * 8, &p); d.par_off = (const int64_t*)p;
  if (rc) { tscl_iql_destroy(h); return -1; }
  cudaError_t e1 = cudaFuncSetAttribute(iql_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fwd);
  cudaError_t e2 = cudaFuncSetAttribute(x->model == 1 ? iql_td_kernel<IQ_NT, 1> : iql_td_kernel<IQ_NT_LR, 8>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_td);
  if (e1 != cudaSuccess || e2 != cudaSuccess) {
    tscl_iql_destroy(h);
    return tsc_set_error(std::string("tscl_iql_create: cudaFuncSetAttribute: ") +
                         cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
  }
  *out = h;
  return 0;
}

static int iq_chunks(int64_t n_tiles, int A, int target = IQ_CTAS) {
  int64_t c = target / A;
  if (c < 1) c = 1;
  if (c > n_tiles) c = n_tiles;
  return (int)c;
}

extern "C" int tscl_iql_forward(tscl_iql_handle* h, const float* params, const float* obs, int64_t R, float eps,
                                uint64_t seed, int64_t step, int64_t replica0, int32_t* act, float* q, void* stream) {
  if (!h || !params || !obs || !act || R <= 0 || !(eps >= 0.f && eps <= 1.f))
    return tsc_set_error("tscl_iql_forward: bad argument");
  ICK(cudaSetDevice(h->device));
  const int64_t n_tiles = (R + IQ_TR - 1) / IQ_TR;
  dim3 grid((unsigned)iq_chunks(n_tiles, h->d.A), (unsigned)h->d.A);
  iql_forward_kernel<<<grid, IQ_NT, h->smem_fwd, (cudaStream_t)stream>>>(h->d, params, obs, R, eps, seed, step,
                                                                         replica0, act, q);
  ICK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_iql_sample(tscl_iql_handle* h, int64_t R, int32_t B, int64_t size, uint64_t seed, int64_t update,
                               int32_t iter, int64_t replica0, int32_t* idx, void* stream) {
  if (!h || !idx || R <= 0 || B <= 0 || size < B || size > INT32_MAX || replica0 < 0)
    return tsc_set_error("tscl_iql_sample: bad argument (needs 0 < batch <= size)");
  ICK(cudaSetDevice(h->device));
  const int64_t n = (int64_t)h->d.A * R;
  iql_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->d.A, R, B, size, seed, update,
                                                                                    iter, replica0, idx);
  ICK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_iql_td_grad(tscl_iql_handle* h, const float* params, const float* obs_ring, const int32_t* act_ring,
                                const float* rew_ring, const float* done_ring, int64_t C, int64_t n_total, int64_t R,
                                int32_t B, const int32_t* idx, float gamma, float scale, float* grads, float* stats,
                                void* stream) {
  if (!h || !params || !obs_ring || !act_ring || !rew_ring || !done_ring || !idx || !grads || C <= 0 || R <= 0 ||
      B <= 0 || n_total < B)
    return tsc_set_error("tscl_iql_td_grad: bad argument");
  ICK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int A = h->d.A;
  const int64_t n_tiles = (R * B + IQ_TR - 1) / IQ_TR;
  const bool dqn = h->d.dqn == 1;
  const int n_cta = iq_chunks(n_tiles, A, dqn ? IQ_CTAS : IQ_CTAS_LR);
  const size_t need = (size_t)A * n_cta * (h->p_max + 2);
  if (need > h->partial_floats) {
    if (h->partial) {
      ICK(cudaStreamSynchronize(st));
      ICK(cudaFree(h->partial));
      h->partial = nullptr;
      h->partial_floats = 0;
    }
    ICK(cudaMalloc(&h->partial, need * 4));
    h->partial_floats = need;
  }
  float* stat_partial = h->partial + (size_t)A * n_cta * h->p_max;
  IqlRing ring{obs_ring, act_ring, rew_ring, done_ring, C, n_total, R};
  if (dqn)
    iql_td_kernel<IQ_NT, 1><<<dim3((unsigned)n_cta, (unsigned)A), IQ_NT, h->smem_td, st>>>(
        h->d, params, ring, B, idx, gamma, scale, h->partial, h->p_max, stat_partial);
  else
    iql_td_kernel<IQ_NT_LR, 8><<<dim3((unsigned)n_cta, (unsigned)A), IQ_NT_LR, h->smem_td, st>>>(
        h->d, params, ring, B, idx, gamma, scale, h->partial, h->p_max, stat_partial);
  ICK(cudaGetLastError());
  iql_reduce_kernel<<<dim3((unsigned)((h->p_max + 255) / 256), (unsigned)A), 256, 0, st>>>(
      h->d, h->partial, h->p_max, n_cta, grads, stat_partial, stats);
  ICK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_iql_clip_adam(tscl_iql_handle* h, float* params, const float* grads, float* m, float* v,
                                  float max_norm, float lr_t, float* norms, void* stream) {
  if (!h || !params || !grads || !m || !v) return tsc_set_error("tscl_iql_clip_adam: bad argument");
  ICK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int A = h->d.A;
  float* norm2 = nullptr;
  ICK(cudaMallocAsync(&norm2, sizeof(float) * A, st));
  iql_norm_kernel<<<A, 256, 0, st>>>(h->d, grads, norm2);
  iql_adam_kernel<<<dim3((unsigned)((h->p_max + 255) / 256), (unsigned)A), 256, 0, st>>>(h->d, params, grads, m, v,
                                                                                          norm2, max_norm, lr_t, norms);
  ICK(cudaGetLastError());
  ICK(cudaFreeAsync(norm2, st));
  return 0;
}

extern "C" int tscl_iql_transition(tscl_iql_handle* h, const float* rew, float* rew_slot, int64_t rew_floats,
                                   float reward_norm, float reward_clip, const float* grew, float* rew_acc, int64_t n,
                                   void* stream) {
  if (!h || !rew || !rew_slot || !grew || !rew_acc || rew_floats <= 0 || n <= 0 || n > rew_floats)
    return tsc_set_error("tscl_iql_transition: bad argument");
  return tscl_launch_reward_transition(h->device, rew, rew_slot, rew_floats, reward_norm, reward_clip, grew, rew_acc, n,
                                       (cudaStream_t)stream);
}
