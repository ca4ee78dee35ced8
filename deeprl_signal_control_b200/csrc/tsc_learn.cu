// tsc_learn.cu — hand-written sm_100a kernels of the per-intersection A2C learner + C ABI
// (include/tsc_learn.h).  fp32 storage and arithmetic (the reference is fp32 TF1).
//
//   fc_embed_kernel       relu(fc) front end of all 2A networks            agents/policies.py:191-201
//   lstm_seq_fwd_kernel   T-step LSTM: recurrent GEMM h.Wh from smem + fused cell   agents/utils.py:88-116
//   heads_kernel          softmax / value / categorical sampling           agents/policies.py:18-26, utils.py:155-157
//   returns_kernel        n-step returns + advantages                      agents/utils.py:202-214
//   heads_loss_kernel     A2C loss gradients at the heads                  agents/policies.py:41-52
//   lstm_seq_bwd_kernel   BPTT: cell backward + dz.Wh^T from smem, carries in registers
//   fc_bwd_kernel         front-end weight/bias gradients (ragged, tiny K)
//   norm2_kernel / rmsprop_kernel   per-agent global-norm clip + TF1 RMSProp   agents/policies.py:54-61
//
// Layout conventions: unit u = 2*agent + net (0 = pi, 1 = V); time-major rows m = t*Rc + r.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/tsc_learn.h"

extern "C" const char* tsc_last_error(void);
int tsc_set_error(const std::string& m);  // defined in tsc_sim.cu

#define LCK(call)                                                                  \
  do {                                                                             \
    cudaError_t e__ = (call);                                                      \
    if (e__ != cudaSuccess) return tsc_set_error(std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)

#define H64 64
#define G4 256  // 4 * H64

struct DDims {
  int A, n_obs, max_na, fw, ff, ft, h, dx;
  const int32_t *obs_off, *n_wave, *n_wait, *n_fp, *n_a;
  const int64_t *off_fcw_w, *off_fcw_b, *off_fcf_w, *off_fcf_b, *off_fct_w, *off_fct_b;
  int64_t off_wx, off_wh, off_bl, off_wo, off_bo, n_params;
  int kw, ones_slot;   // ones_slot: spare input slot that carries 1.0 in tscl_fc_bwd_tc (-1: none); kw: width of the wave block in the 64-column tensor-core input tile: 32 (wave|fp16|wait16) or 48 (wave|fp16)
};

struct tscl_handle {
  int device = 0;
  DDims d{};
  std::vector<void*> owned;
  int max_in = 0;      // max n_wave + n_wait + n_fp
  int max_fcw = 0;     // max fc weight floats of a unit (incl. biases)
};

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }
__device__ __forceinline__ uint32_t lmix32(uint32_t h) {
  h ^= h >> 16; h *= 0x7feb352dU; h ^= h >> 15; h *= 0x846ca68bU; h ^= h >> 16;
  return h;
}

// ------------------------------------------------------------------------------------------------
// fc front end.  grid (n_row_groups, 2A), 256 threads.  Thread = output column (dx <= 256): its weight
// column (<= 32 values) lives in registers, each staged row costs one broadcast LDS.128 per 4 FMAs.
#define FE_ROWS 64
#define FE_KW_MAX 48   // padded inputs of the wave layer: template parameter KW = 32 (grid <= 30) or 48 (Monaco <= 34)
#define FE_KF 16   // fingerprint layer
#define FE_KT 16   // wait layer
#define FE_KTOT (KW + FE_KF + FE_KT)
template <int KW>
__global__ void __launch_bounds__(256)
fc_embed_kernel(const DDims d, const float* __restrict__ P, const float* __restrict__ obs, int64_t M,
                int64_t rows_per_t, int64_t stride_t, float* __restrict__ X) {
  __shared__ __align__(16) float sIn[FE_ROWS * FE_KTOT];
  const int u = blockIdx.y, a = u >> 1, tid = threadIdx.x;
  const int nw = d.n_wave[a], nt = d.n_wait[a], nf = d.ff > 0 ? d.n_fp[a] : 0;
  const int dx = d.dx, col = tid;
  // this thread's weight column
  float w[KW];
  float bias = 0.f;
  int kbase = 0, nk = 0;
#pragma unroll
  for (int k = 0; k < KW; ++k) w[k] = 0.f;
  if (col < dx) {
    if (col < d.fw) {
      nk = nw; kbase = 0;
      for (int k = 0; k < KW; ++k) if (k < nw) w[k] = P[d.off_fcw_w[u] + (int64_t)k * d.fw + col];
      bias = P[d.off_fcw_b[u] + col];
    } else if (col < d.fw + d.ff) {
      nk = nf; kbase = KW;
      for (int k = 0; k < FE_KF; ++k) if (k < nf) w[k] = P[d.off_fcf_w[u] + (int64_t)k * d.ff + (col - d.fw)];
      bias = P[d.off_fcf_b[u] + (col - d.fw)];
    } else {
      nk = nt; kbase = KW + FE_KF;
      for (int k = 0; k < FE_KT; ++k) if (k < nt) w[k] = P[d.off_fct_w[u] + (int64_t)k * d.ft + (col - d.fw - d.ff)];
      bias = P[d.off_fct_b[u] + (col - d.fw - d.ff)];
    }
  }
  const int nk4 = (nk + 3) >> 2;
  const int ooff = d.obs_off[a];
  const int n_in = nw + nt + nf;
  for (int64_t m0 = (int64_t)blockIdx.x * FE_ROWS; m0 < M; m0 += (int64_t)gridDim.x * FE_ROWS) {
    __syncthreads();
    // stage rows: [wave | pad][fp | pad][wait | pad]
    for (int i = tid; i < FE_ROWS * FE_KTOT; i += 256) sIn[i] = 0.f;
    __syncthreads();
    for (int i = tid; i < FE_ROWS * n_in; i += 256) {
      const int row = i / n_in, k = i - row * n_in;
      const int64_t m = m0 + row;
      if (m < M) {
        const float v = obs[(m / rows_per_t) * stride_t + (m % rows_per_t) * d.n_obs + ooff + k];
        int dst;
        if (k < nw) dst = k;
        else if (k < nw + nt) dst = KW + FE_KF + (k - nw);
        else dst = KW + (k - nw - nt);
        sIn[row * FE_KTOT + dst] = v;
      }
    }
    __syncthreads();
    if (col < dx) {
      const int rows = (M - m0) < FE_ROWS ? (int)(M - m0) : FE_ROWS;
      float* Xu = X + ((int64_t)u * M + m0) * dx + col;
      for (int row = 0; row < rows; ++row) {
        const float4* in4 = reinterpret_cast<const float4*>(&sIn[row * FE_KTOT + kbase]);
        float acc = bias;
#pragma unroll
        for (int k4 = 0; k4 < KW / 4; ++k4) {
          if (k4 < nk4) {
            const float4 x = in4[k4];
            acc = fmaf(x.x, w[4 * k4], acc); acc = fmaf(x.y, w[4 * k4 + 1], acc);
            acc = fmaf(x.z, w[4 * k4 + 2], acc); acc = fmaf(x.w, w[4 * k4 + 3], acc);
          }
        }
        Xu[(int64_t)row * dx] = fmaxf(acc, 0.f);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// LSTM sequence forward.  grid (ceil(Rc/32), 2A), 256 threads: thread (ty, tx) owns replicas
// 4*ty .. 4*ty+3 and hidden units 2*tx, 2*tx+1 (all four gates), so the cell update is thread-local.
#define LS_ROWS 32
__global__ void __launch_bounds__(256)
lstm_seq_fwd_kernel(const DDims d, const float* __restrict__ P, float* __restrict__ ZG, float* __restrict__ C,
                    float* __restrict__ Hout, float* __restrict__ Hprev, const float* __restrict__ c0,
                    const float* __restrict__ h0,
                    float* __restrict__ c1, float* __restrict__ h1, const float* __restrict__ done, int T,
                    int64_t Rc, int64_t ld_state, int64_t r0) {
  extern __shared__ float sm[];
  float* sWh = sm;                 // [64][256]
  float* sh = sm + H64 * G4;       // [32][64]
  const int u = blockIdx.y, tid = threadIdx.x, tx = tid & 31, ty = tid >> 5, j0 = 2 * tx;
  const float* Wh = P + d.off_wh + (int64_t)u * H64 * G4;
  for (int i = tid; i < H64 * G4 / 4; i += 256)
    reinterpret_cast<float4*>(sWh)[i] = reinterpret_cast<const float4*>(Wh)[i];
  for (int64_t rbase = (int64_t)blockIdx.x * LS_ROWS; rbase < Rc; rbase += (int64_t)gridDim.x * LS_ROWS) {
  __syncthreads();   // previous tile done with sh
  float c[4][2];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int64_t r = rbase + ty * 4 + q;
    float2 cv = make_float2(0.f, 0.f), hv = make_float2(0.f, 0.f);
    if (r < Rc) {
      const int64_t s = ((int64_t)u * ld_state + r0 + r) * H64 + j0;
      cv = *reinterpret_cast<const float2*>(c0 + s);
      hv = *reinterpret_cast<const float2*>(h0 + s);
    }
    c[q][0] = cv.x; c[q][1] = cv.y;
    *reinterpret_cast<float2*>(&sh[(ty * 4 + q) * H64 + j0]) = hv;
  }
  __syncthreads();
  for (int t = 0; t < T; ++t) {
    const bool dn = done[t] != 0.f;
    float acc[4][4][2];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t r = rbase + ty * 4 + q;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float2 z = make_float2(0.f, 0.f);
        if (r < Rc) z = *reinterpret_cast<const float2*>(ZG + (((int64_t)u * T + t) * Rc + r) * G4 + g * H64 + j0);
        acc[q][g][0] = z.x; acc[q][g][1] = z.y;
      }
      if (dn) { c[q][0] = 0.f; c[q][1] = 0.f; }
      if (Hprev && r < Rc) {
        float2 hp = make_float2(0.f, 0.f);
        if (!dn) hp = *reinterpret_cast<const float2*>(&sh[(ty * 4 + q) * H64 + j0]);
        *reinterpret_cast<float2*>(Hprev + (((int64_t)u * T + t) * Rc + r) * H64 + j0) = hp;
      }
    }
    if (!dn) {
#pragma unroll 4
      for (int k = 0; k < H64; ++k) {
        float hv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) hv[q] = sh[(ty * 4 + q) * H64 + k];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float2 w = *reinterpret_cast<const float2*>(&sWh[k * G4 + g * H64 + j0]);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            acc[q][g][0] = fmaf(hv[q], w.x, acc[q][g][0]);
            acc[q][g][1] = fmaf(hv[q], w.y, acc[q][g][1]);
          }
        }
      }
    }
    __syncthreads();   // every read of sh for step t is done
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t r = rbase + ty * 4 + q;
      float gi[2], gf[2], go[2], gu[2], hn[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        gi[e] = sigmoidf_(acc[q][0][e]); gf[e] = sigmoidf_(acc[q][1][e]);
        go[e] = sigmoidf_(acc[q][2][e]); gu[e] = tanhf(acc[q][3][e]);
        c[q][e] = gf[e] * c[q][e] + gi[e] * gu[e];
        hn[e] = go[e] * tanhf(c[q][e]);
      }
      *reinterpret_cast<float2*>(&sh[(ty * 4 + q) * H64 + j0]) = make_float2(hn[0], hn[1]);
      if (r < Rc) {
        const int64_t m = ((int64_t)u * T + t) * Rc + r;
        float* z = ZG + m * G4 + j0;
        *reinterpret_cast<float2*>(z) = make_float2(gi[0], gi[1]);
        *reinterpret_cast<float2*>(z + H64) = make_float2(gf[0], gf[1]);
        *reinterpret_cast<float2*>(z + 2 * H64) = make_float2(go[0], go[1]);
        *reinterpret_cast<float2*>(z + 3 * H64) = make_float2(gu[0], gu[1]);
        if (C) *reinterpret_cast<float2*>(C + m * H64 + j0) = make_float2(c[q][0], c[q][1]);
        if (Hout) *reinterpret_cast<float2*>(Hout + m * H64 + j0) = make_float2(hn[0], hn[1]);
      }
    }
    __syncthreads();
  }
  if (c1) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t r = rbase + ty * 4 + q;
      if (r < Rc) {
        const int64_t s = ((int64_t)u * ld_state + r0 + r) * H64 + j0;
        *reinterpret_cast<float2*>(c1 + s) = make_float2(c[q][0], c[q][1]);
        *reinterpret_cast<float2*>(h1 + s) = *reinterpret_cast<float2*>(&sh[(ty * 4 + q) * H64 + j0]);
      }
    }
  }
  }
}

// ------------------------------------------------------------------------------------------------
// Heads of one control step.  grid (ceil(R/128), A), 128 threads, thread = replica.
__global__ void __launch_bounds__(128)
heads_kernel(const DDims d, const float* __restrict__ P, const float* __restrict__ Hs, int64_t R,
             float* __restrict__ pi, float* __restrict__ val, int32_t* __restrict__ act, uint32_t seed_lo,
             uint32_t seed_hi, uint32_t step, int64_t replica0) {
  extern __shared__ float sm[];
  const int a = blockIdx.y, tid = threadIdx.x, na = d.n_a[a], mna = d.max_na;
  float* sWp = sm;                    // [64][mna]
  float* sWv = sWp + H64 * mna;       // [64]
  float* sb = sWv + H64;              // [mna + 1]
  const float* Wp = P + d.off_wo + (int64_t)(2 * a) * H64 * mna;
  const float* Wv = P + d.off_wo + (int64_t)(2 * a + 1) * H64 * mna;
  for (int i = tid; i < H64 * mna; i += 128) sWp[i] = Wp[i];
  for (int i = tid; i < H64; i += 128) sWv[i] = Wv[i * mna];
  for (int i = tid; i < mna; i += 128) sb[i] = P[d.off_bo + (int64_t)(2 * a) * mna + i];
  if (tid == 0) sb[mna] = P[d.off_bo + (int64_t)(2 * a + 1) * mna];
  __syncthreads();
  const int64_t r = (int64_t)blockIdx.x * 128 + tid;
  if (r >= R) return;
  const float4* hp = reinterpret_cast<const float4*>(Hs + ((int64_t)(2 * a) * R + r) * H64);
  const float4* hv = reinterpret_cast<const float4*>(Hs + ((int64_t)(2 * a + 1) * R + r) * H64);
  float lg[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) lg[j] = j < mna ? sb[j] : 0.f;
  float v = sb[mna];
  for (int k4 = 0; k4 < H64 / 4; ++k4) {
    const float4 x = hp[k4], y = hv[k4];
    const float xs[4] = {x.x, x.y, x.z, x.w}, ys[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = k4 * 4 + e;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < mna) lg[j] = fmaf(xs[e], sWp[k * mna + j], lg[j]);
      v = fmaf(ys[e], sWv[k], v);
    }
  }
  float mx = -1e30f;
#pragma unroll
  for (int j = 0; j < 8; ++j) if (j < na) mx = fmaxf(mx, lg[j]);
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) { lg[j] = j < na ? __expf(lg[j] - mx) : 0.f; s += lg[j]; }
  const float inv = 1.0f / s;
  float* po = pi + ((int64_t)r * d.A + a) * mna;
#pragma unroll
  for (int j = 0; j < 8; ++j) if (j < mna) po[j] = lg[j] * inv;
  val[(int64_t)r * d.A + a] = v;
  if (act) {
    uint32_t hsh = lmix32(seed_lo ^ (step * 0x9E3779B1U));
    hsh = lmix32(hsh ^ seed_hi ^ ((uint32_t)(replica0 + r) * 0x85EBCA77U));
    hsh = lmix32(hsh ^ ((uint32_t)a * 0xC2B2AE3DU));
    const float uu = (float)(hsh >> 8) * (1.0f / 16777216.0f);
    float cum = 0.f;
    int pick = na - 1;
    bool found = false;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < na) {
        cum += lg[j] * inv;
        if (!found && uu < cum) { pick = j; found = true; }
      }
    }
    act[(int64_t)r * d.A + a] = pick;
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void returns_kernel(const float* __restrict__ rew, const float* __restrict__ val,
                               const float* __restrict__ boot, const float* __restrict__ done_post, float gamma,
                               int T, int64_t RA, float* __restrict__ Rs, float* __restrict__ Adv) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= RA) return;
  float Rv = boot[i];
  for (int t = T - 1; t >= 0; --t) {
    Rv = rew[(int64_t)t * RA + i] + gamma * Rv * (1.0f - done_post[t]);
    Rs[(int64_t)t * RA + i] = Rv;
    Adv[(int64_t)t * RA + i] = Rv - val[(int64_t)t * RA + i];
  }
}

// ------------------------------------------------------------------------------------------------
// Loss gradients at the heads.  grid (<= HL_GX row-tile walkers, A), 128 threads, thread = row m of a 128-row tile.
// With `G` the head weight / bias gradients  dWo += H^T dlog,  dbo += sum dlog  are accumulated here too
// (rows staged in smem, thread = (hidden unit k, 4 logits); one atomic per output per CTA), and `dlog` may be null.
// `Hb`: read H from one chunk of the bf16 activation store instead of the fp32 buffer.
#define HL_GX 96
#define HL_LD 68                       // row pitch in floats: 16-byte aligned rows, conflict-free 128-bit row-owner accesses
#define HL_DL 12                       // dlog (8) | dv | pad
// Shared-memory traffic bounds this kernel (ncu: short scoreboard 6.3, mio throttle 3.3 per issue): rows and the head
// weights are therefore moved with 128-bit accesses only (Wp padded to 8 logits per hidden unit = two broadcast loads).
__global__ void __launch_bounds__(128)
heads_loss_kernel(const DDims d, const float* __restrict__ P, const float* __restrict__ Hm,
                  const __nv_bfloat16* __restrict__ Hb, const int32_t* __restrict__ act, const float* __restrict__ Rs,
                  const float* __restrict__ Adv, int64_t M, int64_t Rc, int64_t stride_t, float v_coef, float beta,
                  float scale, float* __restrict__ dlog, float* __restrict__ dH, float* __restrict__ stats,
                  float* __restrict__ G) {
  extern __shared__ __align__(16) float sm[];
  const int a = blockIdx.y, tid = threadIdx.x, na = d.n_a[a], mna = d.max_na;
  float* sWp = sm;                     // [64][8]
  float* sWv = sWp + H64 * 8;          // [64]
  float* sb = sWv + H64;               // [16]
  float* sH = sb + 16;                 // [128][HL_LD] rows of H (value unit, then policy unit)
  float* sdl = sH + 128 * HL_LD;       // [128][HL_DL]
  const float* Wp = P + d.off_wo + (int64_t)(2 * a) * H64 * mna;
  const float* Wv = P + d.off_wo + (int64_t)(2 * a + 1) * H64 * mna;
  for (int i = tid; i < H64 * 8; i += 128) { const int k = i >> 3, j = i & 7; sWp[i] = j < mna ? Wp[k * mna + j] : 0.f; }
  for (int i = tid; i < H64; i += 128) sWv[i] = Wv[i * mna];
  for (int i = tid; i < mna; i += 128) sb[i] = P[d.off_bo + (int64_t)(2 * a) * mna + i];
  if (tid == 0) sb[mna] = P[d.off_bo + (int64_t)(2 * a + 1) * mna];
  __syncthreads();
  float pl = 0.f, vl = 0.f, el = 0.f;
  float accp[4] = {0.f, 0.f, 0.f, 0.f}, accv = 0.f, accb = 0.f;
  const int kk = tid & 63, hh = tid >> 6;
  const int64_t n_tiles = (M + 127) / 128;
  float4* myH4 = reinterpret_cast<float4*>(sH + tid * HL_LD);
  const float4* sWp4 = reinterpret_cast<const float4*>(sWp);
  const float4* sWv4 = reinterpret_cast<const float4*>(sWv);
  auto load_row = [&](int64_t off) {       // one row of H (64 values) -> this thread's smem row
    if (Hb) {
      const uint4* p4 = reinterpret_cast<const uint4*>(Hb + off);
      uint4 x[H64 / 8];
#pragma unroll
      for (int k8 = 0; k8 < H64 / 8; ++k8) x[k8] = __ldg(p4 + k8);
#pragma unroll
      for (int k8 = 0; k8 < H64 / 8; ++k8) {
        myH4[2 * k8] = make_float4(__uint_as_float(x[k8].x << 16), __uint_as_float(x[k8].x & 0xffff0000u),
                                   __uint_as_float(x[k8].y << 16), __uint_as_float(x[k8].y & 0xffff0000u));
        myH4[2 * k8 + 1] = make_float4(__uint_as_float(x[k8].z << 16), __uint_as_float(x[k8].z & 0xffff0000u),
                                       __uint_as_float(x[k8].w << 16), __uint_as_float(x[k8].w & 0xffff0000u));
      }
    } else {
      const float4* p4 = reinterpret_cast<const float4*>(Hm + off);
#pragma unroll
      for (int k4 = 0; k4 < H64 / 4; ++k4) myH4[k4] = __ldg(p4 + k4);
    }
  };
  auto st8 = [](float* p, const float* v) {      // 256-bit store: one full sector per thread and instruction
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(__float_as_uint(v[0])),
                 "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
                 "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])) : "memory");
  };
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m = tile * 128 + tid;
    const bool valid = m < M;
    const int64_t op = ((int64_t)(2 * a) * M + (valid ? m : 0)) * H64, ov = ((int64_t)(2 * a + 1) * M + (valid ? m : 0)) * H64;
    const int64_t io = valid ? (m / Rc) * stride_t + (m % Rc) * d.A + a : 0;
    // ---- value unit ----
    __syncthreads();                       // previous tile's readers of sH / sdl are done
    float dv = 0.f, v = 0.f, ret = 0.f;
    if (valid) {
      load_row(ov);
      v = sb[mna]; ret = Rs[io];
#pragma unroll
      for (int k4 = 0; k4 < H64 / 4; ++k4) {
        const float4 x = myH4[k4], w = sWv4[k4];
        v = fmaf(x.x, w.x, v); v = fmaf(x.y, w.y, v); v = fmaf(x.z, w.z, v); v = fmaf(x.w, w.w, v);
      }
      dv = scale * v_coef * (v - ret);
#pragma unroll
      for (int k8 = 0; k8 < H64 / 8; ++k8) {
        const float4 w0 = sWv4[2 * k8], w1 = sWv4[2 * k8 + 1];
        const float o[8] = {dv * w0.x, dv * w0.y, dv * w0.z, dv * w0.w, dv * w1.x, dv * w1.y, dv * w1.z, dv * w1.w};
        st8(dH + ov + 8 * k8, o);
      }
    } else {
#pragma unroll
      for (int k4 = 0; k4 < H64 / 4; ++k4) myH4[k4] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    sdl[tid * HL_DL + 8] = dv;
    if (G) {
      __syncthreads();
      if (hh == 0) for (int row = 0; row < 128; ++row) accv = fmaf(sH[row * HL_LD + kk], sdl[row * HL_DL + 8], accv);
      __syncthreads();
    }
    // ---- policy unit ----
    float dl[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) dl[j] = 0.f;
    if (valid) {
      load_row(op);
      float lg[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) lg[j] = j < mna ? sb[j] : 0.f;
#pragma unroll 4
      for (int k4 = 0; k4 < H64 / 4; ++k4) {
        const float4 x4 = myH4[k4];
        const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float4 w0 = sWp4[2 * (4 * k4 + e)], w1 = sWp4[2 * (4 * k4 + e) + 1];
          lg[0] = fmaf(xs[e], w0.x, lg[0]); lg[1] = fmaf(xs[e], w0.y, lg[1]); lg[2] = fmaf(xs[e], w0.z, lg[2]);
          lg[3] = fmaf(xs[e], w0.w, lg[3]); lg[4] = fmaf(xs[e], w1.x, lg[4]); lg[5] = fmaf(xs[e], w1.y, lg[5]);
          lg[6] = fmaf(xs[e], w1.z, lg[6]); lg[7] = fmaf(xs[e], w1.w, lg[7]);
        }
      }
      float mx = -1e30f;
#pragma unroll
      for (int j = 0; j < 8; ++j) if (j < na) mx = fmaxf(mx, lg[j]);
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) { lg[j] = j < na ? __expf(lg[j] - mx) : 0.f; s += lg[j]; }
      const float inv = 1.0f / s;
      const int at = act[io];
      const float adv = Adv[io];
      float lp[8], ent = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        lg[j] *= inv;                                             // pi_j
        lp[j] = j < na ? __logf(fminf(fmaxf(lg[j], 1e-10f), 1.0f)) : 0.f;   // agents/policies.py:47
        ent -= lg[j] * lp[j];
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float g = 0.f;
        if (j < na) g = scale * (-adv * ((j == at ? 1.f : 0.f) - lg[j]) + beta * lg[j] * (lp[j] + ent));
        dl[j] = g;
      }
      if (dlog) {
        float* dlp = dlog + ((int64_t)(2 * a) * M + m) * mna;
        float* dlv = dlog + ((int64_t)(2 * a + 1) * M + m) * mna;
#pragma unroll
        for (int j = 0; j < 8; ++j) if (j < mna) { dlp[j] = dl[j]; dlv[j] = j == 0 ? dv : 0.f; }
      }
#pragma unroll 2
      for (int k8 = 0; k8 < H64 / 8; ++k8) {
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float4 w0 = sWp4[2 * (8 * k8 + e)], w1 = sWp4[2 * (8 * k8 + e) + 1];
          float t = 0.f;
          t = fmaf(dl[0], w0.x, t); t = fmaf(dl[1], w0.y, t); t = fmaf(dl[2], w0.z, t); t = fmaf(dl[3], w0.w, t);
          t = fmaf(dl[4], w1.x, t); t = fmaf(dl[5], w1.y, t); t = fmaf(dl[6], w1.z, t); t = fmaf(dl[7], w1.w, t);
          o[e] = t;
        }
        st8(dH + op + 8 * k8, o);
      }
      if (a == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) if (j == at) pl += -lp[j] * adv;
        vl += 0.5f * v_coef * (ret - v) * (ret - v);
        el += -beta * ent;
      }
    } else {
#pragma unroll
      for (int k4 = 0; k4 < H64 / 4; ++k4) myH4[k4] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (G) {      // head weight gradients of this tile: thread = (hidden unit kk, 4 logits)
      *reinterpret_cast<float4*>(sdl + tid * HL_DL) = make_float4(dl[0], dl[1], dl[2], dl[3]);
      *reinterpret_cast<float4*>(sdl + tid * HL_DL + 4) = make_float4(dl[4], dl[5], dl[6], dl[7]);
      __syncthreads();
#pragma unroll 8
      for (int row = 0; row < 128; ++row) {
        const float x = sH[row * HL_LD + kk];
        const float4 q = *reinterpret_cast<const float4*>(sdl + row * HL_DL + hh * 4);
        accp[0] = fmaf(x, q.x, accp[0]); accp[1] = fmaf(x, q.y, accp[1]);
        accp[2] = fmaf(x, q.z, accp[2]); accp[3] = fmaf(x, q.w, accp[3]);
      }
      if (tid < 9) for (int row = 0; row < 128; ++row) accb += sdl[row * HL_DL + tid];
    }
  }
  if (G) {
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int j = hh * 4 + jj;
      if (j < mna) atomicAdd(&G[d.off_wo + ((int64_t)(2 * a) * H64 + kk) * mna + j], accp[jj]);
    }
    if (hh == 0) atomicAdd(&G[d.off_wo + ((int64_t)(2 * a + 1) * H64 + kk) * mna], accv);
    if (tid < mna) atomicAdd(&G[d.off_bo + (int64_t)(2 * a) * mna + tid], accb);
    if (tid == 8) atomicAdd(&G[d.off_bo + (int64_t)(2 * a + 1) * mna], accb);
  }
  if (a == 0 && stats) {
    for (int o = 16; o; o >>= 1) {
      pl += __shfl_down_sync(0xffffffffu, pl, o);
      vl += __shfl_down_sync(0xffffffffu, vl, o);
      el += __shfl_down_sync(0xffffffffu, el, o);
    }
    if ((tid & 31) == 0) {
      atomicAdd(&stats[0], pl * scale); atomicAdd(&stats[1], vl * scale); atomicAdd(&stats[2], el * scale);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// BPTT through the LSTM.  Same thread mapping as the forward kernel.  smem: WhT [256][64] + dz [32][256].
__global__ void __launch_bounds__(256)
lstm_seq_bwd_kernel(const DDims d, const float* __restrict__ P, float* __restrict__ ZG, const float* __restrict__ C,
                    const float* __restrict__ dH, const float* __restrict__ c0, const float* __restrict__ done, int T,
                    int64_t Rc, int64_t ld_state, int64_t r0) {
  extern __shared__ float sm[];
  float* sWT = sm;                 // [256][64] : WhT[col][k]
  float* sdz = sm + G4 * H64;      // [32][256]
  const int u = blockIdx.y, tid = threadIdx.x, tx = tid & 31, ty = tid >> 5, j0 = 2 * tx;
  const float* Wh = P + d.off_wh + (int64_t)u * H64 * G4;
  for (int i = tid; i < H64 * G4; i += 256) {
    const int k = i / G4, col = i - k * G4;
    sWT[col * H64 + k] = Wh[i];
  }
  const int64_t rbase = (int64_t)blockIdx.x * LS_ROWS;
  float dc[4][2], dhc[4][2];
#pragma unroll
  for (int q = 0; q < 4; ++q) { dc[q][0] = dc[q][1] = 0.f; dhc[q][0] = dhc[q][1] = 0.f; }
  __syncthreads();
  for (int t = T - 1; t >= 0; --t) {
    const float keep = 1.0f - done[t];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t r = rbase + ty * 4 + q;
      float dz[4][2] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
      float dcp[2] = {0.f, 0.f};
      if (r < Rc) {
        const int64_t m = ((int64_t)u * T + t) * Rc + r;
        float* z = ZG + m * G4 + j0;
        const float2 gi = *reinterpret_cast<const float2*>(z), gf = *reinterpret_cast<const float2*>(z + H64);
        const float2 go = *reinterpret_cast<const float2*>(z + 2 * H64), gu = *reinterpret_cast<const float2*>(z + 3 * H64);
        const float2 ct = *reinterpret_cast<const float2*>(C + m * H64 + j0);
        float2 cp;
        if (t > 0) cp = *reinterpret_cast<const float2*>(C + (m - Rc) * H64 + j0);
        else cp = *reinterpret_cast<const float2*>(c0 + ((int64_t)u * ld_state + r0 + r) * H64 + j0);
        const float2 dh_in = *reinterpret_cast<const float2*>(dH + m * H64 + j0);
        const float i_[2] = {gi.x, gi.y}, f_[2] = {gf.x, gf.y}, o_[2] = {go.x, go.y}, u_[2] = {gu.x, gu.y};
        const float c_[2] = {ct.x, ct.y}, p_[2] = {cp.x * keep, cp.y * keep}, h_[2] = {dh_in.x, dh_in.y};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float dh = h_[e] + dhc[q][e];
          const float tc = tanhf(c_[e]);
          const float dcc = dc[q][e] + dh * o_[e] * (1.0f - tc * tc);
          dz[0][e] = dcc * u_[e] * i_[e] * (1.0f - i_[e]);
          dz[1][e] = dcc * p_[e] * f_[e] * (1.0f - f_[e]);
          dz[2][e] = dh * tc * o_[e] * (1.0f - o_[e]);
          dz[3][e] = dcc * i_[e] * (1.0f - u_[e] * u_[e]);
          dcp[e] = dcc * f_[e];
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) *reinterpret_cast<float2*>(z + g * H64) = make_float2(dz[g][0], dz[g][1]);
      }
#pragma unroll
      for (int g = 0; g < 4; ++g)
        *reinterpret_cast<float2*>(&sdz[(ty * 4 + q) * G4 + g * H64 + j0]) = make_float2(dz[g][0], dz[g][1]);
      dc[q][0] = dcp[0] * keep; dc[q][1] = dcp[1] * keep;
    }
    __syncthreads();
    if (keep != 0.f && t > 0) {
      float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
      for (int col = 0; col < G4; col += 4) {
        float2 w[4];
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) w[cc] = *reinterpret_cast<const float2*>(&sWT[(col + cc) * H64 + j0]);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 z = *reinterpret_cast<const float4*>(&sdz[(ty * 4 + q) * G4 + col]);   // warp-wide broadcast
          a0[q] = fmaf(z.x, w[0].x, a0[q]); a1[q] = fmaf(z.x, w[0].y, a1[q]);
          a0[q] = fmaf(z.y, w[1].x, a0[q]); a1[q] = fmaf(z.y, w[1].y, a1[q]);
          a0[q] = fmaf(z.z, w[2].x, a0[q]); a1[q] = fmaf(z.z, w[2].y, a1[q]);
          a0[q] = fmaf(z.w, w[3].x, a0[q]); a1[q] = fmaf(z.w, w[3].y, a1[q]);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) { dhc[q][0] = a0[q] * keep; dhc[q][1] = a1[q] * keep; }
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) { dhc[q][0] = 0.f; dhc[q][1] = 0.f; }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// fc front-end backward.  grid (n_groups, 2A), 256 threads.  Thread = column c of dX: accumulates
// dW[k][c] for every input k of its layer (<= 32 registers) + the bias gradient; rows staged 32 at a time.
#define FB_ROWS 32
template <int KW>
__global__ void __launch_bounds__(256)
fc_bwd_kernel(const DDims d, const float* __restrict__ obs, const float* __restrict__ X, const float* __restrict__ dX,
              int64_t M, int64_t rows_per_t, int64_t stride_t, float* __restrict__ G) {
  __shared__ __align__(16) float sIn[FB_ROWS * FE_KTOT];
  const int u = blockIdx.y, a = u >> 1, tid = threadIdx.x;
  const int nw = d.n_wave[a], nt = d.n_wait[a], nf = d.ff > 0 ? d.n_fp[a] : 0;
  const int n_in = nw + nt + nf, dx = d.dx, col = tid;
  int kbase = 0, nk = 0;
  if (col < d.fw) { nk = nw; kbase = 0; }
  else if (col < d.fw + d.ff) { nk = nf; kbase = KW; }
  else if (col < dx) { nk = nt; kbase = KW + FE_KF; }
  const int nk4 = (nk + 3) >> 2;
  float acc[KW];
#pragma unroll
  for (int k = 0; k < KW; ++k) acc[k] = 0.f;
  float accb = 0.f;
  const int ooff = d.obs_off[a];
  for (int i = tid; i < FB_ROWS * FE_KTOT; i += 256) sIn[i] = 0.f;
  for (int64_t m0 = (int64_t)blockIdx.x * FB_ROWS; m0 < M; m0 += (int64_t)gridDim.x * FB_ROWS) {
    __syncthreads();
    for (int i = tid; i < FB_ROWS * n_in; i += 256) {
      const int row = i / n_in, k = i - row * n_in;
      const int64_t m = m0 + row;
      float v = 0.f;
      if (m < M) v = obs[(m / rows_per_t) * stride_t + (m % rows_per_t) * d.n_obs + ooff + k];
      int dst;
      if (k < nw) dst = k;
      else if (k < nw + nt) dst = KW + FE_KF + (k - nw);
      else dst = KW + (k - nw - nt);
      sIn[row * FE_KTOT + dst] = v;
    }
    __syncthreads();
    if (col < dx) {
      const int rows = (M - m0) < FB_ROWS ? (int)(M - m0) : FB_ROWS;
      const int64_t o0 = ((int64_t)u * M + m0) * dx + col;
      // rows in groups of 8: all 16 global loads of a group are issued before they are consumed
      // (16-row groups were measured 2x slower: register pressure)
      for (int r0 = 0; r0 < rows; r0 += 8) {
        float g[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int64_t o = o0 + (int64_t)(r0 + j) * dx;
          float xv = 0.f, dv = 0.f;
          if (r0 + j < rows) { xv = __ldg(X + o); dv = __ldg(dX + o); }
          g[j] = xv > 0.f ? dv : 0.f;                   // relu mask
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          accb += g[j];
          const float4* in4 = reinterpret_cast<const float4*>(&sIn[(r0 + j) * FE_KTOT + kbase]);
#pragma unroll
          for (int k4 = 0; k4 < KW / 4; ++k4) {
            if (k4 < nk4) {
              const float4 x = in4[k4];
              acc[4 * k4] = fmaf(x.x, g[j], acc[4 * k4]); acc[4 * k4 + 1] = fmaf(x.y, g[j], acc[4 * k4 + 1]);
              acc[4 * k4 + 2] = fmaf(x.z, g[j], acc[4 * k4 + 2]); acc[4 * k4 + 3] = fmaf(x.w, g[j], acc[4 * k4 + 3]);
            }
          }
        }
      }
    }
  }
  if (col < dx) {
    int64_t wo, bo; int ld, c;
    if (col < d.fw) { wo = d.off_fcw_w[u]; bo = d.off_fcw_b[u]; ld = d.fw; c = col; }
    else if (col < d.fw + d.ff) { wo = d.off_fcf_w[u]; bo = d.off_fcf_b[u]; ld = d.ff; c = col - d.fw; }
    else { wo = d.off_fct_w[u]; bo = d.off_fct_b[u]; ld = d.ft; c = col - d.fw - d.ff; }
#pragma unroll
    for (int k = 0; k < KW; ++k)
      if (k < nk) atomicAdd(&G[wo + (int64_t)k * ld + c], acc[k]);
    atomicAdd(&G[bo + c], accb);
  }
}

// ------------------------------------------------------------------------------------------------
// Activation-store chunk -> fp32 work buffers in one pass: X, gates, C, H (8 bf16 = 16 B per thread-iteration)
// and Hp[t] = keep[t] * (t > 0 ? H[t-1] : h0).  All arrays are [2A][T][rc][w] contiguous.
__global__ void unpack_store_kernel(const uint4* __restrict__ sx, const uint4* __restrict__ sg, const uint4* __restrict__ sc,
                                    const uint4* __restrict__ shh, float4* __restrict__ X, float4* __restrict__ ZG,
                                    float4* __restrict__ Cc, float4* __restrict__ H, float4* __restrict__ Hp,
                                    const float* __restrict__ h0, const float* __restrict__ done, int64_t nx8, int64_t ng8,
                                    int64_t nh8, int T, int64_t rc, int64_t ld_state, int64_t r0) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  auto cvt = [](const uint4 v, float4& a, float4& b) {
    a.x = __uint_as_float(v.x << 16); a.y = __uint_as_float(v.x & 0xffff0000u);
    a.z = __uint_as_float(v.y << 16); a.w = __uint_as_float(v.y & 0xffff0000u);
    b.x = __uint_as_float(v.z << 16); b.y = __uint_as_float(v.z & 0xffff0000u);
    b.z = __uint_as_float(v.w << 16); b.w = __uint_as_float(v.w & 0xffff0000u);
  };
  if (X)
    for (int64_t i = i0; i < nx8; i += stride) { float4 a, b; cvt(sx[i], a, b); X[2 * i] = a; X[2 * i + 1] = b; }
  if (ZG)
    for (int64_t i = i0; i < ng8; i += stride) { float4 a, b; cvt(sg[i], a, b); ZG[2 * i] = a; ZG[2 * i + 1] = b; }
  if (!Cc && !H && !Hp) return;
  for (int64_t i = i0; i < nh8; i += stride) {
    float4 a, b;
    if (Cc) { cvt(sc[i], a, b); Cc[2 * i] = a; Cc[2 * i + 1] = b; }
    if (H) { cvt(shh[i], a, b); H[2 * i] = a; H[2 * i + 1] = b; }
    if (!Hp) continue;
    // element index -> (u, t, r, j8): 8 hidden per item, 8 items per row
    const int64_t row = i >> 3; const int j8 = (int)(i & 7);
    const int64_t r = row % rc; const int64_t ut = row / rc; const int t = (int)(ut % T); const int64_t u = ut / T;
    const float keep = 1.0f - done[t];
    float4 pa = make_float4(0.f, 0.f, 0.f, 0.f), pb = pa;
    if (keep != 0.f) {
      if (t > 0) { cvt(shh[i - rc * 8], pa, pb); }
      else {
        const float4* hp = reinterpret_cast<const float4*>(h0 + ((u * ld_state + r0 + r) * H64 + j8 * 8));
        pa = hp[0]; pb = hp[1];
      }
    }
    Hp[2 * i] = pa; Hp[2 * i + 1] = pb;
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void norm2_kernel(const float* __restrict__ g, const uint8_t* __restrict__ agent_of, int64_t n,
                             float* __restrict__ norm2) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float v = 0.f;
  int a = -1;
  if (i < n) { v = g[i]; v *= v; a = agent_of[i]; }
  const int a0 = __shfl_sync(0xffffffffu, a, 0);
  if (__all_sync(0xffffffffu, a == a0)) {
    for (int o = 16; o; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && a0 >= 0) atomicAdd(&norm2[a0], v);
  } else if (a >= 0) {
    atomicAdd(&norm2[a], v);
  }
}
__global__ void rmsprop_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ ms,
                               const uint8_t* __restrict__ agent_of, int64_t n, const float* __restrict__ norm2,
                               float max_norm, float lr, float alpha, float eps, float* __restrict__ norms) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int a = agent_of[i];
  const float nrm = sqrtf(norm2[a]);
  float scale = 1.0f;
  if (max_norm > 0.f) scale = max_norm / fmaxf(nrm, max_norm);      // tf.clip_by_global_norm
  const float gi = g[i] * scale;
  const float m = alpha * ms[i] + (1.0f - alpha) * gi * gi;          // TF1 RMSProp: ms starts at 1
  ms[i] = m;
  p[i] -= lr * gi / sqrtf(m + eps);                                  // epsilon inside the sqrt
  if (norms && (i == 0 || agent_of[i - 1] != a)) norms[a] = nrm;
}

// accessors for tsc_policy_tc.cu (DDimsTC there mirrors DDims member for member)
// ------------------------------------------------------------------------------------------------
// FcACPolicy hidden layer (agents/policies.py:236, `fc(h, out_type + '_fc', n_fc)`): register-tiled fp32 GEMMs.
//   forward   H[u][m][0:64]  = relu(X[u][m][0:dx] . W[u] + b[u])                       W = wx [2A][dx][64], b = bl
//   backward  dHm = dH * (H > 0) (written back),  dX = dHm . W^T,  g.bl += 1^T dHm     (one kernel)
//             g.wx += X^T dHm                                                           (row-split kernel, atomics)
// Tile = 64 rows x 64 columns per CTA of 256 threads (4 x 4 outputs per thread), K staged 32 at a time.
#define FH_T 128           // rows per tile
#define FH_K 32            // K staged per step of the forward
// forward: W [dx][64] resident in shared memory for all the row tiles of a CTA; thread = 8 rows x 4 columns
__global__ void __launch_bounds__(256)
fc_hidden_fwd_kernel(const DDims d, const float* __restrict__ P, const float* __restrict__ X, int64_t M,
                     float* __restrict__ H) {
  extern __shared__ float fh_sm[];
  float* Ws = fh_sm;                               // [dx][64]
  float* Xs = fh_sm + (size_t)d.dx * H64;          // [FH_T][FH_K + 1]
  const int u = blockIdx.y, tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const float* W = P + d.off_wx + (int64_t)u * d.dx * H64;
  const float* Xu = X + (int64_t)u * M * d.dx;
  for (int i = tid; i < d.dx * H64; i += 256) Ws[i] = W[i];
  const float4 bias = *reinterpret_cast<const float4*>(P + d.off_bl + (int64_t)u * H64 + tx * 4);
  const int64_t n_tiles = (M + FH_T - 1) / FH_T;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m0 = tile * FH_T;
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
    for (int k0 = 0; k0 < d.dx; k0 += FH_K) {
      __syncthreads();
      for (int i = tid; i < FH_T * FH_K; i += 256) {
        const int r = i / FH_K, k = i % FH_K;
        Xs[r * (FH_K + 1) + k] = (m0 + r < M && k0 + k < d.dx) ? Xu[(m0 + r) * d.dx + k0 + k] : 0.f;
      }
      __syncthreads();
      const int kmax = min(FH_K, d.dx - k0);
      for (int k = 0; k < kmax; ++k) {
        const float4 b = *reinterpret_cast<const float4*>(Ws + (size_t)(k0 + k) * H64 + tx * 4);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float x = Xs[(ty * 8 + i) * (FH_K + 1) + k];
          acc[i][0] = fmaf(x, b.x, acc[i][0]); acc[i][1] = fmaf(x, b.y, acc[i][1]);
          acc[i][2] = fmaf(x, b.z, acc[i][2]); acc[i][3] = fmaf(x, b.w, acc[i][3]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t m = m0 + ty * 8 + i;
      if (m < M)
        *reinterpret_cast<float4*>(H + ((int64_t)u * M + m) * H64 + tx * 4) =
            make_float4(fmaxf(acc[i][0] + bias.x, 0.f), fmaxf(acc[i][1] + bias.y, 0.f), fmaxf(acc[i][2] + bias.z, 0.f),
                        fmaxf(acc[i][3] + bias.w, 0.f));
    }
  }
}

// dHm = dH * (H > 0) (written back), dX = dHm . W^T in column passes of 64, bias gradient += column sums of dHm;
// W^T [64][dx] resident in shared memory for all the row tiles of a CTA
__global__ void __launch_bounds__(256)
fc_hidden_bwd_dx_kernel(const DDims d, const float* __restrict__ P, const float* __restrict__ H, float* __restrict__ dH,
                        int64_t M, float* __restrict__ dX, float* __restrict__ G) {
  extern __shared__ float fh_sm[];
  float* Wt = fh_sm;                               // [64][dxp]   Wt[k][n] = W[n][k], dxp = dx rounded up to 64
  const int dxp = (d.dx + 63) & ~63;
  float* Ds = fh_sm + (size_t)H64 * dxp;           // [FH_T][65]
  const int u = blockIdx.y, tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const float* W = P + d.off_wx + (int64_t)u * d.dx * H64;
  for (int i = tid; i < H64 * dxp; i += 256) {
    const int k = i / dxp, n = i % dxp;
    Wt[i] = n < d.dx ? W[(int64_t)n * H64 + k] : 0.f;
  }
  float bsum = 0.f;                                // threads 0..63: bias-gradient column sums over this CTA's tiles
  const int64_t n_tiles = (M + FH_T - 1) / FH_T;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m0 = tile * FH_T;
    __syncthreads();
    for (int i = tid; i < FH_T * H64; i += 256) {
      const int r = i >> 6, k = i & 63;
      float v = 0.f;
      if (m0 + r < M) {
        const int64_t o = ((int64_t)u * M + m0 + r) * H64 + k;
        v = H[o] > 0.f ? dH[o] : 0.f;
        dH[o] = v;                                 // the weight-gradient kernel reads the masked gradient
      }
      Ds[r * 65 + k] = v;
    }
    __syncthreads();
    if (tid < H64) {
      float sum = 0.f;
      for (int r = 0; r < FH_T; ++r) sum += Ds[r * 65 + tid];
      bsum += sum;
    }
    for (int n0 = 0; n0 < d.dx; n0 += 64) {
      float acc[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
#pragma unroll 4
      for (int k = 0; k < H64; ++k) {
        const float4 b = *reinterpret_cast<const float4*>(Wt + (size_t)k * dxp + n0 + tx * 4);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float x = Ds[(ty * 8 + i) * 65 + k];
          acc[i][0] = fmaf(x, b.x, acc[i][0]); acc[i][1] = fmaf(x, b.y, acc[i][1]);
          acc[i][2] = fmaf(x, b.z, acc[i][2]); acc[i][3] = fmaf(x, b.w, acc[i][3]);
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int64_t m = m0 + ty * 8 + i;
        if (m < M) {
          float* o = dX + ((int64_t)u * M + m) * d.dx + n0 + tx * 4;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (n0 + tx * 4 + j < d.dx) o[j] = acc[i][j];
        }
      }
    }
  }
  if (tid < H64) atomicAdd(G + d.off_bl + (int64_t)u * H64 + tid, bsum);
}

// g.wx[u][k][c] += sum_m X[u][m][k] * dHm[u][m][c] over the CTA's row slice; thread = (k-group, 4 columns)
#define FH_WROWS 32
__global__ void __launch_bounds__(256)
fc_hidden_wgrad_kernel(const DDims d, const float* __restrict__ X, const float* __restrict__ dHm, int64_t M,
                       int64_t rows_per_cta, float* __restrict__ G) {
  extern __shared__ float fh_sm[];
  float* Xs = fh_sm;                           // [FH_WROWS][dx]
  float* Ds = fh_sm + FH_WROWS * d.dx;         // [FH_WROWS][64]
  const int u = blockIdx.y, tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;     // 16 column groups x 16 k-groups
  const int kper = (d.dx + 15) / 16;           // k rows per thread (<= 16 for dx <= 256)
  const int64_t m_lo = (int64_t)blockIdx.x * rows_per_cta, m_hi = min(M, m_lo + rows_per_cta);
  float acc[16][4];
#pragma unroll
  for (int i = 0; i < 16; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
  for (int64_t mb = m_lo; mb < m_hi; mb += FH_WROWS) {
    const int nr = (int)min((int64_t)FH_WROWS, m_hi - mb);
    for (int i = tid; i < FH_WROWS * d.dx; i += 256) {
      const int r = i / d.dx;
      Xs[i] = r < nr ? X[((int64_t)u * M + mb) * d.dx + i] : 0.f;
    }
    for (int i = tid; i < FH_WROWS * H64; i += 256) {
      const int r = i >> 6;
      Ds[i] = r < nr ? dHm[((int64_t)u * M + mb) * H64 + i] : 0.f;
    }
    __syncthreads();
    for (int r = 0; r < FH_WROWS; ++r) {
      const float4 dv = *reinterpret_cast<const float4*>(Ds + r * H64 + tx * 4);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (i < kper) {
          const int k = ty * kper + i;
          const float x = k < d.dx ? Xs[r * d.dx + k] : 0.f;
          acc[i][0] = fmaf(x, dv.x, acc[i][0]); acc[i][1] = fmaf(x, dv.y, acc[i][1]);
          acc[i][2] = fmaf(x, dv.z, acc[i][2]); acc[i][3] = fmaf(x, dv.w, acc[i][3]);
        }
      }
    }
    __syncthreads();
  }
  float* Gw = G + d.off_wx + (int64_t)u * d.dx * H64;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    if (i < kper) {
      const int k = ty * kper + i;
      if (k < d.dx)
#pragma unroll
        for (int j = 0; j < 4; ++j) atomicAdd(Gw + (int64_t)k * H64 + tx * 4 + j, acc[i][j]);
    }
  }
}

struct DDimsTC;
const DDimsTC* tscl_dims_of(tscl_handle* h) { return reinterpret_cast<const DDimsTC*>(&h->d); }
int tscl_device_of(tscl_handle* h) { return h->device; }

// ================================================================================================
template <class T>
static int up(tscl_handle* h, const T* src, size_t n, const T** dst) {
  void* p = nullptr;
  LCK(cudaMalloc(&p, n ? n * sizeof(T) : 16));
  if (n) LCK(cudaMemcpy(p, src, n * sizeof(T), cudaMemcpyHostToDevice));
  h->owned.push_back(p);
  *dst = static_cast<const T*>(p);
  return 0;
}

extern "C" int tscl_create(const tscl_dims* x, int32_t device, tscl_handle** out) {
  if (!x || !out) return tsc_set_error("tscl_create: bad argument");
  if (x->h != H64) return tsc_set_error("tscl_create: num_lstm must be 64");
  if (x->max_na > 8) return tsc_set_error("tscl_create: max_na > 8");
  if (x->dx != x->fw + x->ff + x->ft) return tsc_set_error("tscl_create: dx != fw + ff + ft");
  LCK(cudaSetDevice(device));
  tscl_handle* h = new tscl_handle();
  h->device = device;
  DDims& d = h->d;
  d.A = x->n_agents; d.n_obs = x->n_obs; d.max_na = x->max_na; d.fw = x->fw; d.ff = x->ff; d.ft = x->ft;
  d.h = x->h; d.dx = x->dx; d.off_wx = x->off_wx; d.off_wh = x->off_wh; d.off_bl = x->off_bl; d.off_wo = x->off_wo;
  d.off_bo = x->off_bo; d.n_params = x->n_params;
  const size_t A = x->n_agents, U = 2 * A;
  int rc = 0;
  rc |= up(h, x->obs_off, A, &d.obs_off); rc |= up(h, x->n_wave, A, &d.n_wave); rc |= up(h, x->n_wait, A, &d.n_wait);
  rc |= up(h, x->n_fp, A, &d.n_fp); rc |= up(h, x->n_a, A, &d.n_a);
  rc |= up(h, x->off_fcw_w, U, &d.off_fcw_w); rc |= up(h, x->off_fcw_b, U, &d.off_fcw_b);
  rc |= up(h, x->off_fcf_w, U, &d.off_fcf_w); rc |= up(h, x->off_fcf_b, U, &d.off_fcf_b);
  rc |= up(h, x->off_fct_w, U, &d.off_fct_w); rc |= up(h, x->off_fct_b, U, &d.off_fct_b);
  if (rc) { tscl_destroy(h); return -1; }
  for (size_t a = 0; a < A; ++a) {
    const int nf = x->ff > 0 ? x->n_fp[a] : 0;
    const int n_in = x->n_wave[a] + x->n_wait[a] + nf;
    const int w = x->n_wave[a] * x->fw + nf * x->ff + x->n_wait[a] * x->ft + x->dx;
    if (n_in > h->max_in) h->max_in = n_in;
    if (w > h->max_fcw) h->max_fcw = w;
  }
  for (size_t a = 0; a < A; ++a)
    if (x->n_wave[a] > FE_KW_MAX || (x->ff > 0 && x->n_fp[a] > FE_KF) || x->n_wait[a] > FE_KT || x->dx > 256) {
      tscl_destroy(h);
      return tsc_set_error("tscl_create: fc input widths exceed the kernel limits (wave 48, fp 16, wait 16, dx 256)");
    }
  {
    int mw = 0, mt = 0;
    for (size_t a = 0; a < A; ++a) { if (x->n_wave[a] > mw) mw = x->n_wave[a]; if (x->n_wait[a] > mt) mt = x->n_wait[a]; }
    d.kw = mw <= 32 ? 32 : 48;
    if (d.kw == 48 && mt > 0 && x->ft > 0) d.kw = 0;   // no 64-column packing exists: tensor-core forward unavailable
    d.ones_slot = (d.kw > 0 && mw < d.kw) ? d.kw - 1 : -1;
  }
  LCK(cudaFuncSetAttribute(lstm_seq_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (H64 * G4 + LS_ROWS * H64) * 4));
  LCK(cudaFuncSetAttribute(lstm_seq_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (G4 * H64 + LS_ROWS * G4) * 4));
  *out = h;
  return 0;
}

extern "C" int tscl_destroy(tscl_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  for (void* p : h->owned) cudaFree(p);
  delete h;
  return 0;
}

extern "C" int tscl_fc_embed(tscl_handle* h, const float* params, const float* obs, int64_t M, int64_t rows_per_t,
                             int64_t stride_t, float* X, void* stream) {
  if (!h || M <= 0) return tsc_set_error("tscl_fc_embed: bad argument");
  LCK(cudaSetDevice(h->device));
  int64_t ng = (M + FE_ROWS - 1) / FE_ROWS;
  if (ng > 24) ng = 24;                 // 24 x 2A CTAs (~8 per SM): the weight column load is amortised over many rows
  dim3 grid((unsigned)ng, 2 * h->d.A);
  (h->d.kw == 32 ? fc_embed_kernel<32> : fc_embed_kernel<48>)<<<grid, 256, 0, (cudaStream_t)stream>>>(
      h->d, params, obs, M, rows_per_t, stride_t, X);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_fc_hidden_fwd(tscl_handle* h, const float* params, const float* X, int64_t M, float* H, void* stream) {
  if (!h || !params || !X || !H || M <= 0) return tsc_set_error("tscl_fc_hidden_fwd: bad argument");
  if (h->d.dx > 256) return tsc_set_error("tscl_fc_hidden_fwd: dx > 256");
  LCK(cudaSetDevice(h->device));
  static int attr_dev = -1;
  if (attr_dev != h->device) {
    LCK(cudaFuncSetAttribute(fc_hidden_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    LCK(cudaFuncSetAttribute(fc_hidden_bwd_dx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    attr_dev = h->device;
  }
  const int64_t n_tiles = (M + FH_T - 1) / FH_T;
  dim3 grid((unsigned)(n_tiles < 16 ? n_tiles : 16), 2 * h->d.A);      // 16 x 2A persistent CTAs: W is loaded once per CTA
  const size_t smem = ((size_t)h->d.dx * H64 + (size_t)FH_T * (FH_K + 1)) * sizeof(float);
  fc_hidden_fwd_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(h->d, params, X, M, H);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_fc_hidden_bwd(tscl_handle* h, const float* params, const float* X, const float* H, float* dH, int64_t M,
                                  float* dX, float* grads, void* stream) {
  if (!h || !params || !X || !H || !dH || !dX || !grads || M <= 0) return tsc_set_error("tscl_fc_hidden_bwd: bad argument");
  if (h->d.dx > 256) return tsc_set_error("tscl_fc_hidden_bwd: dx > 256");
  LCK(cudaSetDevice(h->device));
  static int attr_dev = -1;
  if (attr_dev != h->device) {
    LCK(cudaFuncSetAttribute(fc_hidden_bwd_dx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    LCK(cudaFuncSetAttribute(fc_hidden_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * 1024));
    attr_dev = h->device;
  }
  const int64_t n_tiles = (M + FH_T - 1) / FH_T;
  dim3 g1((unsigned)(n_tiles < 16 ? n_tiles : 16), 2 * h->d.A);
  const int dxp = (h->d.dx + 63) & ~63;
  const size_t smem1 = ((size_t)H64 * dxp + (size_t)FH_T * 65) * sizeof(float);
  fc_hidden_bwd_dx_kernel<<<g1, 256, smem1, (cudaStream_t)stream>>>(h->d, params, H, dH, M, dX, grads);
  LCK(cudaGetLastError());
  int64_t splits = (M + 2047) / 2048;
  if (splits > 64) splits = 64;
  const int64_t rows_per = ((M + splits - 1) / splits + FH_WROWS - 1) / FH_WROWS * FH_WROWS;
  dim3 g2((unsigned)((M + rows_per - 1) / rows_per), 2 * h->d.A);
  const size_t smem = (size_t)FH_WROWS * (h->d.dx + H64) * sizeof(float);
  fc_hidden_wgrad_kernel<<<g2, 256, smem, (cudaStream_t)stream>>>(h->d, X, dH, M, rows_per, grads);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_lstm_seq_fwd(tscl_handle* h, const float* params, float* ZG, float* C, float* H, float* Hprev,
                                 const float* c0, const float* h0, float* c1, float* h1, const float* done, int32_t T,
                                 int64_t Rc, int64_t ld_state, int64_t r0, void* stream) {
  if (!h || T <= 0 || Rc <= 0) return tsc_set_error("tscl_lstm_seq_fwd: bad argument");
  LCK(cudaSetDevice(h->device));
  int64_t nt = (Rc + LS_ROWS - 1) / LS_ROWS;
  if (T == 1 && nt > 9) nt = 9;        // rollout step: 9 x 2A CTAs = 3 per SM, each walks many row tiles with Wh resident
  dim3 grid((unsigned)nt, 2 * h->d.A);
  lstm_seq_fwd_kernel<<<grid, 256, (H64 * G4 + LS_ROWS * H64) * 4, (cudaStream_t)stream>>>(
      h->d, params, ZG, C, H, Hprev, c0, h0, c1, h1, done, T, Rc, ld_state, r0);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_heads(tscl_handle* h, const float* params, const float* Hs, int64_t R, float* pi, float* val,
                          int32_t* act, uint64_t seed, int64_t step, int64_t replica0, void* stream) {
  if (!h || R <= 0) return tsc_set_error("tscl_heads: bad argument");
  LCK(cudaSetDevice(h->device));
  dim3 grid((unsigned)((R + 127) / 128), h->d.A);
  const int smem = (H64 * h->d.max_na + H64 + h->d.max_na + 1) * 4;
  heads_kernel<<<grid, 128, smem, (cudaStream_t)stream>>>(h->d, params, Hs, R, pi, val, act, (uint32_t)seed,
                                                          (uint32_t)(seed >> 32), (uint32_t)step, replica0);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_returns(tscl_handle* h, const float* rew, const float* val, const float* boot,
                            const float* done_post, float gamma, int32_t T, int64_t R, float* Rs, float* Adv,
                            void* stream) {
  if (!h) return tsc_set_error("tscl_returns: null handle");
  LCK(cudaSetDevice(h->device));
  const int64_t RA = R * h->d.A;
  returns_kernel<<<(unsigned)((RA + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rew, val, boot, done_post, gamma, T, RA,
                                                                                  Rs, Adv);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_heads_loss(tscl_handle* h, const float* params, const float* H, const int32_t* act,
                               const float* Rs, const float* Adv, int64_t M, int64_t Rc, int64_t stride_t,
                               float v_coef, float beta, float scale, float* dlog, float* dH, float* stats,
                               const void* h_bf16, float* grads, void* stream) {
  if (!h || M <= 0 || (!H && !h_bf16) || !dH) return tsc_set_error("tscl_heads_loss: bad argument");
  if (h->d.max_na > 8) return tsc_set_error("tscl_heads_loss: more than 8 actions");
  LCK(cudaSetDevice(h->device));
  const int64_t n_tiles = (M + 127) / 128;
  dim3 grid((unsigned)(grads ? (n_tiles < HL_GX ? n_tiles : HL_GX) : n_tiles), h->d.A);
  const int smem = (H64 * 8 + H64 + 16 + 128 * HL_LD + 128 * HL_DL) * 4;
  heads_loss_kernel<<<grid, 128, smem, (cudaStream_t)stream>>>(h->d, params, H, (const __nv_bfloat16*)h_bf16, act, Rs, Adv,
                                                               M, Rc, stride_t, v_coef, beta, scale, dlog, dH, stats, grads);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_lstm_seq_bwd(tscl_handle* h, const float* params, float* ZG, const float* C, const float* dH,
                                 const float* c0, const float* done, int32_t T, int64_t Rc, int64_t ld_state,
                                 int64_t r0, void* stream) {
  if (!h || T <= 0 || Rc <= 0) return tsc_set_error("tscl_lstm_seq_bwd: bad argument");
  LCK(cudaSetDevice(h->device));
  dim3 grid((unsigned)((Rc + LS_ROWS - 1) / LS_ROWS), 2 * h->d.A);
  lstm_seq_bwd_kernel<<<grid, 256, (G4 * H64 + LS_ROWS * G4) * 4, (cudaStream_t)stream>>>(h->d, params, ZG, C, dH, c0,
                                                                                           done, T, Rc, ld_state, r0);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_fc_bwd(tscl_handle* h, const float* obs, const float* X, const float* dX, int64_t M,
                           int64_t rows_per_t, int64_t stride_t, float* grads, void* stream) {
  if (!h || M <= 0) return tsc_set_error("tscl_fc_bwd: bad argument");
  LCK(cudaSetDevice(h->device));
  int64_t ng = (M + FB_ROWS - 1) / FB_ROWS;
  if (ng > 24) ng = 24;
  dim3 grid((unsigned)ng, 2 * h->d.A);
  (h->d.kw == 32 ? fc_bwd_kernel<32> : fc_bwd_kernel<48>)<<<grid, 256, 0, (cudaStream_t)stream>>>(h->d, obs, X, dX, M, rows_per_t, stride_t, grads);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_unpack_store(tscl_handle* h, const void* st_x, const void* st_g, const void* st_c, const void* st_h,
                                 float* X, float* ZG, float* Cc, float* H, float* Hp, const float* h0, const float* done,
                                 int32_t T, int64_t rc, int64_t ld_state, int64_t r0, void* stream) {
  if (!h || !st_x || T <= 0 || rc <= 0) return tsc_set_error("tscl_unpack_store: bad argument");
  LCK(cudaSetDevice(h->device));
  const int64_t rows = (int64_t)2 * h->d.A * T * rc;
  unpack_store_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(
      (const uint4*)st_x, (const uint4*)st_g, (const uint4*)st_c, (const uint4*)st_h, (float4*)X, (float4*)ZG, (float4*)Cc,
      (float4*)H, (float4*)Hp, h0, done, rows * h->d.dx / 8, rows * G4 / 8, rows * H64 / 8, T, rc, ld_state, r0);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_clip_rmsprop(tscl_handle* h, float* params, float* grads, float* ms, const uint8_t* agent_of,
                                 float max_norm, float lr, float alpha, float eps, float* norms, void* stream) {
  if (!h) return tsc_set_error("tscl_clip_rmsprop: null handle");
  LCK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  float* norm2 = nullptr;
  LCK(cudaMallocAsync(&norm2, sizeof(float) * h->d.A, st));
  LCK(cudaMemsetAsync(norm2, 0, sizeof(float) * h->d.A, st));
  const int64_t n = h->d.n_params;
  norm2_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(grads, agent_of, n, norm2);
  rmsprop_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(params, grads, ms, agent_of, n, norm2, max_norm, lr, alpha,
                                                              eps, norms);
  LCK(cudaGetLastError());
  LCK(cudaFreeAsync(norm2, st));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Host-buffer (e2e) loop helpers: one call per replica range and control step replaces a dozen framework-level
// copies / elementwise launches (the host loop was issue-bound: 0.22 ms of Python per range and step).
//   tscl_host_transition: observations host -> rollout slot, rewards host -> normalised / clipped rollout slot
//   (envs/env.py reward hand-over + agents/models.py:222-229 `add_transition`, utils.py reward_norm / reward_clip),
//   global rewards host -> running episode sum (utils.py:296-305).
__global__ void host_transition_kernel(const float* __restrict__ rew_in, float* __restrict__ rew_hist, int64_t n_rew,
                                       float inv_norm, float clip, const float* __restrict__ grew_in,
                                       float* __restrict__ rew_acc, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_rew) {
    float r = rew_in[i];
    if (inv_norm != 0.f) r = r * inv_norm;
    if (clip > 0.f) r = fminf(fmaxf(r, -clip), clip);
    rew_hist[i] = r;
  }
  if (i < n) rew_acc[i] += grew_in[i];
}

extern "C" int tscl_host_transition(tscl_handle* h, const float* obs_host, float* obs_dev, int64_t obs_floats,
                                    const float* rew_host, float* rew_stage_dev, float* rew_hist_dev, int64_t rew_floats,
                                    float reward_norm, float reward_clip, const float* grew_host, float* grew_stage_dev,
                                    float* rew_acc_dev, int64_t n, void* stream) {
  if (!h || !obs_host || !obs_dev || !rew_host || !rew_stage_dev || !rew_hist_dev || !grew_host || !grew_stage_dev ||
      !rew_acc_dev || obs_floats <= 0 || rew_floats <= 0 || n <= 0 || n > rew_floats)
    return tsc_set_error("tscl_host_transition: bad argument");
  LCK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  LCK(cudaMemcpyAsync(obs_dev, obs_host, (size_t)obs_floats * 4, cudaMemcpyHostToDevice, st));
  LCK(cudaMemcpyAsync(rew_stage_dev, rew_host, (size_t)rew_floats * 4, cudaMemcpyHostToDevice, st));
  LCK(cudaMemcpyAsync(grew_stage_dev, grew_host, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  host_transition_kernel<<<(unsigned)((rew_floats + 255) / 256), 256, 0, st>>>(
      rew_stage_dev, rew_hist_dev, rew_floats, reward_norm != 0.f ? 1.0f / reward_norm : 0.f, reward_clip, grew_stage_dev,
      rew_acc_dev, n);
  LCK(cudaGetLastError());
  return 0;
}

// the same hand-over for the device-resident loop (rewards already on the device): one launch instead of six; also the
// reward store of the IQL replay ring (tscl_iql_transition, tsc_iql.cu)
int tscl_launch_reward_transition(int device, const float* rew, float* rew_hist, int64_t n_rew, float reward_norm,
                                  float reward_clip, const float* grew, float* rew_acc, int64_t n, cudaStream_t st) {
  LCK(cudaSetDevice(device));
  host_transition_kernel<<<(unsigned)((n_rew + 255) / 256), 256, 0, st>>>(
      rew, rew_hist, n_rew, reward_norm != 0.f ? 1.0f / reward_norm : 0.f, reward_clip, grew, rew_acc, n);
  LCK(cudaGetLastError());
  return 0;
}

extern "C" int tscl_device_transition(tscl_handle* h, const float* rew_dev, float* rew_hist_dev, int64_t rew_floats,
                                      float reward_norm, float reward_clip, const float* grew_dev, float* rew_acc_dev,
                                      int64_t n, void* stream) {
  if (!h || !rew_dev || !rew_hist_dev || !grew_dev || !rew_acc_dev || rew_floats <= 0 || n <= 0 || n > rew_floats)
    return tsc_set_error("tscl_device_transition: bad argument");
  return tscl_launch_reward_transition(h->device, rew_dev, rew_hist_dev, rew_floats, reward_norm, reward_clip, grew_dev,
                                       rew_acc_dev, n, (cudaStream_t)stream);
}

// plain asynchronous copy on a caller-supplied stream (kind: 1 host->device, 2 device->host, 3 device->device)
extern "C" int tscl_memcpy_async(tscl_handle* h, void* dst, const void* src, int64_t bytes, int32_t kind, void* stream) {
  if (!h || !dst || !src || bytes <= 0 || kind < 1 || kind > 3) return tsc_set_error("tscl_memcpy_async: bad argument");
  LCK(cudaSetDevice(h->device));
  LCK(cudaMemcpyAsync(dst, src, (size_t)bytes, kind == 1 ? cudaMemcpyHostToDevice : kind == 2 ? cudaMemcpyDeviceToHost
                                                                                              : cudaMemcpyDeviceToDevice,
                      (cudaStream_t)stream));
  return 0;
}
