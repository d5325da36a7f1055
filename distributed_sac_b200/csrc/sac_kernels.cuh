// Fused non-GEMM stages of the SAC gradient step: minibatch ingest / replay sampling,
// policy head (reparameterise + tanh squash + log-prob), critic heads (TD target, MSE
// gradient), actor-pass heads (min-Q), small-N layer backward, Adam (+Polyak) and the
// temperature update.  Everything that the reference evaluates in fp32 in an
// ill-conditioned way (1 - tanh^2 + 1e-6, u - mu) is evaluated in the SAME order here,
// transcendental functions are computed in fp64 and rounded once (== torch CPU's result on
// >98 % of inputs) and the file is compiled with -fmad=false so that only explicit fmaf()
// fuses.  Math reference: oracle/sac_manual.py; reference sites cited per kernel.
#pragma once
#include "common.cuh"

namespace bsac {

constexpr int kMaxAct = 8;      // act_dim <= 8  (head width 2*act <= 16)
constexpr int kMaxHeadOut = 16;
constexpr int kSaveW = 8;       // floats saved per (row, action) by the policy head
constexpr int kLossSlots = 1024;

// Per-learner constant block (device copy lives in the handle).
struct StepConst {
  int B, obs, act, T, xw;         // obs = raw observation width (state + one-hot); xw = in_w + act
  int in_w;                       // width of the state part of the MLP inputs: obs, or ctx_out + mix_out with CARE
  int care;
  int ldxa, ldx;                  // row pitches of XA ([2B][in_w]) and of XQ/XT/XP/dx ([B][xw]): multiples of 4 floats
  int Ha, Hc;                     // last hidden widths (actor / critic)
  float gamma, reward_scale, action_scale;
  float c_loss;                   // 1/B or 1/B^2 (weighted_loss)
  float inv_B;
  float tau, one_minus_tau;
  float hbar;                     // -act
  double lr_actor, lr_critic, lr_alpha, beta1, beta2, adam_eps;
  unsigned long long seed;
};

// Mutable per-replica counters in device memory: v[0..2] Adam steps critic/actor/alpha, v[3] step index;
// b1p/b2p[i] = beta^v[i], kept as running products so no kernel needs a double-precision pow().
// v[4] = Adam step of the CARE(O) context encoder.
struct Counters { long long v[5]; double b1p[5]; double b2p[5]; };

// ------------------------------------------------------------------------------------------
// Ingest: scatter one minibatch into the four pre-concatenated layer-0 inputs
//   XA [2B][obs]   = [s2 ; s]          (actor runs once over both halves)
//   XQ [B][obs+act] = [s | a]           critic update pass
//   XT [B][obs+act] = [s2 | a_next]     target pass   (a_next filled by the policy head)
//   XP [B][obs+act] = [s | a_cur]       actor pass    (a_cur  filled by the policy head)
// plus r, d, task id (argmax of the one-hot, MT10_Distributed_MTSAC/src/model.py:105-106) and
// the noise buffer.  Also bumps the Adam step counters (torch increments before use).
// Replaces ReplayBuffer.sample()'s 5x vstack + .to(device) (LL/replay_buffer.py:63-73).
// ------------------------------------------------------------------------------------------
struct IngestOut {
  float *XA, *XQ, *XT, *XP, *r, *d, *eps;   // replica 0 bases
  float* XS;                                 // CARE: raw [s' ; s] rows
  int* tid;
  Counters* cnt;
  long long rsXA, rsXQ, rsR, rsEps, rsXS;    // per-replica strides
  // temperature of this step, alpha[t] = exp(log_alpha[t]) as update() snapshots it before anything moves
  // (LL/learner.py:250, MS/learner.py:337): evaluated ONCE here (fp64, rounded once) for the layer-chained kernels
  const float* log_alpha; long long rsP;     // parameter arena pointer
  float* alpha; long long rsAlpha;           // [max(T,1)] per replica
};

B200_D void ingest_row(const StepConst& K, const IngestOut& O, int rep, int i, const float* s, const float* a,
                       float r, const float* s2, float d, int lane, int nl) {
  const int obs = K.obs, act = K.act, xw = K.ldx, xa = K.ldxa, B = K.B;
  float* XQ = O.XQ + rep * O.rsXQ;
  if (K.care) {
    // CARE: the MLP inputs are encoded states produced later by care_mix_kernel; keep the raw rows [s' ; s]
    float* XS = O.XS + rep * O.rsXS;
    for (int j = lane; j < obs; j += nl) {
      XS[(long long)i * obs + j] = s2[j];
      XS[(long long)(B + i) * obs + j] = s[j];
    }
  } else {
    float* XA = O.XA + rep * O.rsXA;
    float* XT = O.XT + rep * O.rsXQ;
    float* XP = O.XP + rep * O.rsXQ;
    for (int j = lane; j < obs; j += nl) {
      float v = s[j], v2 = s2[j];
      XA[(long long)i * xa + j] = v2;
      XA[(long long)(B + i) * xa + j] = v;
      XQ[(long long)i * xw + j] = v;
      XP[(long long)i * xw + j] = v;
      XT[(long long)i * xw + j] = v2;
    }
  }
  for (int j = lane; j < act; j += nl) XQ[(long long)i * xw + K.in_w + j] = a[j];
  if (lane == 0) {
    (O.r + rep * O.rsR)[i] = r;
    (O.d + rep * O.rsR)[i] = d;
    int t = 0;
    if (K.T > 0) {                       // first maximum, like torch.argmax
      float best = s[obs - K.T];
      for (int q = 1; q < K.T; ++q) {
        float v = s[obs - K.T + q];
        if (v > best) { best = v; t = q; }
      }
    }
    (O.tid + rep * O.rsR)[i] = t;
  }
}

B200_D void snapshot_alpha(const StepConst& K, const IngestOut& O, int rep, int t) {
  if (O.alpha != nullptr && t < (K.T > 0 ? K.T : 1))
    (O.alpha + rep * O.rsAlpha)[t] = (float)exp((double)(O.log_alpha + rep * O.rsP)[t]);
}

B200_D void bump_counters(Counters* cnt, int rep, double beta1, double beta2) {
  Counters* c = cnt + rep;
  c->v[0] += 1; c->v[1] += 1; c->v[2] += 1; c->v[3] += 1; c->v[4] += 1;
#pragma unroll
  for (int i = 0; i < 5; ++i) { c->b1p[i] *= beta1; c->b2p[i] *= beta2; }
}

// minibatch given as five separate arrays [R][B][w]
__global__ void ingest_split_kernel(StepConst K, IngestOut O, const float* __restrict__ s,
                                    const float* __restrict__ a, const float* __restrict__ r,
                                    const float* __restrict__ s2, const float* __restrict__ d,
                                    const float* __restrict__ eps_next, const float* __restrict__ eps_cur) {
  KStamp ks_;
  const int rep = blockIdx.y;
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32, wpb = blockDim.x / 32;
  const int B = K.B;
  if (blockIdx.x == 0 && threadIdx.x == 0) bump_counters(O.cnt, rep, K.beta1, K.beta2);
  if (blockIdx.x == gridDim.x - 1) snapshot_alpha(K, O, rep, threadIdx.x);
  for (int i = blockIdx.x * wpb + warp; i < B; i += gridDim.x * wpb) {
    const long long ri = (long long)rep * B + i;
    ingest_row(K, O, rep, i, s + ri * K.obs, a + ri * K.act, r[ri], s2 + ri * K.obs, d[ri], lane, 32);
    if (eps_next != nullptr) {
      float* E = O.eps + rep * O.rsEps;
      for (int j = lane; j < K.act; j += 32) {
        E[(long long)i * K.act + j] = eps_next[ri * K.act + j];
        E[(long long)(B + i) * K.act + j] = eps_cur[ri * K.act + j];
      }
    }
  }
}

// minibatch given as packed rows [s | a | r | s2 | d] (+pad), either gathered through idx
// (device replay ring) or dense (pinned-host staging after the H2D copy).
__global__ void ingest_rows_kernel(StepConst K, IngestOut O, const float* __restrict__ rows, long long rs_rows,
                                   int row_stride, const int* __restrict__ idx, long long rs_idx) {
  KStamp ks_;
  const int rep = blockIdx.y;
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32, wpb = blockDim.x / 32;
  const int B = K.B;
  if (blockIdx.x == 0 && threadIdx.x == 0) bump_counters(O.cnt, rep, K.beta1, K.beta2);
  if (blockIdx.x == gridDim.x - 1) snapshot_alpha(K, O, rep, threadIdx.x);
  for (int i = blockIdx.x * wpb + warp; i < B; i += gridDim.x * wpb) {
    const long long src = idx ? (long long)idx[rep * rs_idx + i] : (long long)i;
    const float* row = rows + rep * rs_rows + src * row_stride;
    ingest_row(K, O, rep, i, row, row + K.obs, row[K.obs + K.act], row + K.obs + K.act + 1,
               row[2 * K.obs + K.act + 1], lane, 32);
  }
}

// ------------------------------------------------------------------------------------------
// Replay index sampling: uniform WITHOUT replacement (random.sample, LL/replay_buffer.py:65),
// per task B/T when T > 0 (MS/replay_buffers.py:73-74).  One CTA per replica.  Duplicates are
// resolved deterministically (lowest batch slot keeps a contested index, the others redraw
// with the next Philox sub-counter), so a given (seed, step) always yields the same minibatch.
// ------------------------------------------------------------------------------------------
constexpr int kHashSlots = 4096;   // >= 2 * max batch (batch <= 2048)

__global__ void sample_indices_kernel(StepConst K, const Counters* __restrict__ cnt, const long long* __restrict__ fill,
                                      long long cap_per_task, int* __restrict__ idx_out, long long rs_idx,
                                      unsigned long long seed) {
  KStamp ks_;
  __shared__ int keys[kHashSlots];
  __shared__ int owner[kHashSlots];
  __shared__ int unresolved;
  const int rep = blockIdx.x;
  const int B = K.B, Teff = K.T > 0 ? K.T : 1, per = B / Teff;
  const long long step = cnt[rep].v[3];   // value BEFORE this step's bump
  Philox ph(seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(rep + 1));
  int* out = idx_out + rep * rs_idx;
  for (int i = threadIdx.x; i < kHashSlots; i += blockDim.x) { keys[i] = -1; owner[i] = 0x7fffffff; }
  // per-slot state lives in registers of the thread that owns slots i = threadIdx.x + j*blockDim.x
  constexpr int kMaxPer = 8;     // batch <= 8 * blockDim.x
  int cur[kMaxPer], att[kMaxPer], pos[kMaxPer];
  bool done[kMaxPer];
#pragma unroll
  for (int j = 0; j < kMaxPer; ++j) { att[j] = 0; done[j] = false; cur[j] = -1; pos[j] = 0; }
  __syncthreads();
  for (int round = 0; round < 64; ++round) {
    if (threadIdx.x == 0) unresolved = 0;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kMaxPer; ++j) {
      const int i = threadIdx.x + j * blockDim.x;
      if (i >= B || done[j]) continue;
      const int task = i / per;
      const long long n = fill[rep * Teff + (task < Teff ? task : Teff - 1)];
      uint32_t rnd[4];
      ph((uint32_t)step, (uint32_t)(step >> 32), (uint32_t)i, (uint32_t)att[j], rnd);
      const unsigned long long r64 = ((unsigned long long)rnd[0] << 32) | rnd[1];
      const long long local = (long long)(r64 % (unsigned long long)n);
      const int key = (int)((long long)task * cap_per_task + local);
      cur[j] = key;
      unsigned h = ((unsigned)key * 2654435761u) >> 20;   // 12 bits
      int probes = 0;
      for (; probes < kHashSlots; ++probes) {
        int prev = atomicCAS(&keys[h], -1, key);
        if (prev == -1 || prev == key) break;
        h = (h + 1) & (kHashSlots - 1);
      }
      if (probes == kHashSlots) {     // table full (cannot happen for fill >= 4 * batch): accept the draw
        pos[j] = -1;
        continue;
      }
      pos[j] = (int)h;
      atomicMin(&owner[h], i);
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kMaxPer; ++j) {
      const int i = threadIdx.x + j * blockDim.x;
      if (i >= B || done[j]) continue;
      out[i] = cur[j];                 // always leave a valid index behind
      if (pos[j] < 0 || owner[pos[j]] == i) {
        done[j] = true;
      } else {
        att[j] += 1;
        atomicAdd(&unresolved, 1);
      }
    }
    __syncthreads();
    // read the round's verdict NOW: thread 0 resets the counter at the top of the next round, and the only barrier between
    // here and there is the one below -- reading it after that barrier raced with the reset (compute-sanitizer racecheck)
    const int pending = unresolved;
    // winners lock their table entry so that a lower slot redrawing later cannot steal it
#pragma unroll
    for (int j = 0; j < kMaxPer; ++j) {
      const int i = threadIdx.x + j * blockDim.x;
      if (i < B && done[j] && pos[j] >= 0 && owner[pos[j]] == i) owner[pos[j]] = -1;
    }
    __syncthreads();
    if (pending == 0) break;
  }
}

// ------------------------------------------------------------------------------------------
// Policy head: last actor layer (width 2*act) + rsample + tanh squash + log-prob, one warp per
// row over the 2B rows [s2 ; s].  LL/model.py:38-65 (Actor.forward, get_action_log_prob),
// MS/model.py:35-56.  Writes the action into the critic input buffers (XT for the s2 half, XP
// for the s half) so no concat is ever materialised.
// ------------------------------------------------------------------------------------------
struct PolicyHeadArgs {
  const float* h; long long rsH; int ldh;     // last hidden activations [2B][Ha]
  const float* W; const float* b; long long rsP;   // head weight [2A][Ha], bias; param-arena replica stride
  const float* eps; long long rsEps;          // [2B][A] (used when use_eps_buf != 0)
  int use_eps_buf;
  float* pout; long long rsPout;              // [2B][2A] raw head output
  float* psave; long long rsSave;             // [2B][A][kSaveW]
  float* XT; float* XP; long long rsX;
  float* act_out; long long rsAct;            // [2B][A]
  float* logp; long long rsLogp;              // [2B]
  float* logstd_sum;                          // [2B] sum_j log(std) (entropy statistic, MS/learner.py:310)
  const Counters* cnt;
  int rows;                                   // 0: all 2B rows (a training step); n: only rows [0, n) (b200sac_act)
};

struct PolicyPoint {   // everything the backward needs for one (row, action)
  float std, diff, t, act, jac, eps, mask, logp_j, logstd;
};

// fp64-evaluated, once-rounded transcendentals as out-of-line functions: their bodies (70-150 instructions each) exist once
// per kernel instead of once per call site.  The kernels that use them run each code path once per CTA, i.e. out of a cold
// instruction cache (32 KB L1.5 against 70 KB kernels): straight-line code costs several cycles per instruction there.
__device__ __noinline__ float exp_f64r(float x) { return (float)exp((double)x); }
__device__ __noinline__ float tanh_f64r(float x) { return (float)tanh((double)x); }
__device__ __noinline__ float log_f64r(float x) { return (float)log((double)x); }

B200_D PolicyPoint policy_point(float mu, float raw, float eps, float k) {
  PolicyPoint p;
  const float ls = fminf(fmaxf(raw, -20.f), 2.f);          // torch.clamp(x, -20, 2)
  p.mask = (raw >= -20.f && raw <= 2.f) ? 1.f : 0.f;
  p.std = exp_f64r(ls);
  p.eps = eps;
  const float u = mu + p.std * eps;                        // Normal.rsample: loc + eps * scale
  p.t = tanh_f64r(u);
  p.act = k * p.t;
  p.diff = u - mu;                                         // as rounded, NOT std*eps
  const float var = p.std * p.std;
  p.logstd = log_f64r(p.std);
  const float gauss = -(p.diff * p.diff) / (2.f * var) - p.logstd - 0.91893853320467274178f;
  const float q = p.act / k;
  p.jac = k * (1.f - q * q + 1e-6f);
  p.logp_j = gauss - log_f64r(p.jac);
  return p;
}

// noise of one (row, action): from the injected buffer, or Philox keyed by (seed, replica, step, row, action)
B200_D float policy_noise(const StepConst& K, const PolicyHeadArgs& P, int rep, int row, int lane) {
  float e = 0.f;
  if (lane < K.act) {
    if (P.use_eps_buf) {
      e = (P.eps + rep * P.rsEps)[(long long)row * K.act + lane];
    } else {
      Philox ph(K.seed ^ (0xA0761D6478BD642Full * (unsigned long long)(rep + 1)));
      const long long step = P.cnt[rep].v[3];
      uint32_t rnd[4];
      ph((uint32_t)step, (uint32_t)(step >> 32), (uint32_t)row, 0x51u + (uint32_t)lane, rnd);
      float z0, z1;
      box_muller(rnd[0], rnd[1], z0, z1);
      e = z0;
    }
  }
  return e;
}

// One CTA = 8 rows: every warp does the head GEMV of its row, then ONE warp evaluates the tanh-Gaussian of all 8 x A
// (row, action) pairs in parallel lanes.  The transcendentals are evaluated in fp64 (DESIGN.md 3) and a warp-wide fp64
// instruction costs the same with 4 or 32 active lanes: the warp-per-row version (4 active lanes per warp) queued on the
// FP64 pipe -- 11.5 us at 2 048 rows, 16.9 us at 2 560 (profiles/, round 2) -- this one issues an eighth of the instructions.
__global__ void __launch_bounds__(256) policy_head_kernel(StepConst K, PolicyHeadArgs P) {
  KStamp ks_;
  __shared__ float sd[8][kMaxHeadOut];
  __shared__ float lp_s[8][kMaxAct], ls_s[8][kMaxAct];
  const int rep = blockIdx.y;
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int row0 = blockIdx.x * 8, row = row0 + warp;
  const int B = K.B, A = K.act, NO = 2 * K.act, H = K.Ha;
  const int total = P.rows > 0 ? P.rows : 2 * B;
  if (row < total) {
    const float* hr = P.h + rep * P.rsH + (long long)row * P.ldh;
    const float* W = P.W + rep * P.rsP;
    const float* bias = P.b + rep * P.rsP;
    float bj[kMaxHeadOut];
#pragma unroll
    for (int j = 0; j < kMaxHeadOut; ++j) bj[j] = j < NO ? bias[j] : 0.f;
    float acc[kMaxHeadOut];
#pragma unroll
    for (int j = 0; j < kMaxHeadOut; ++j) acc[j] = 0.f;
    for (int k0 = 0; k0 < H; k0 += 128) {       // four lane-strides of h and of every head row in flight per round trip
      float hv[4], wv[4][kMaxHeadOut];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int k = k0 + lane + 32 * u;
        hv[u] = k < H ? hr[k] : 0.f;
#pragma unroll
        for (int j = 0; j < kMaxHeadOut; ++j) wv[u][j] = (j < NO && k < H) ? __ldg(W + (long long)j * H + k) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (k0 + lane + 32 * u < H) {
#pragma unroll
          for (int j = 0; j < kMaxHeadOut; ++j)
            if (j < NO) acc[j] = fmaf(hv[u], wv[u][j], acc[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < kMaxHeadOut; ++j)
      if (j < NO) {
        const float v = warp_sum(acc[j]) + bj[j];
        if (lane == j) sd[warp][j] = v;
      }
  }
  __syncthreads();
  if (warp != 0) return;
  const int nrows = total - row0 < 8 ? total - row0 : 8;
  for (int e0 = 0; e0 < nrows * A; e0 += 32) {
    const int e = e0 + lane;
    if (e < nrows * A) {
      const int m = e / A, j = e - m * A, r = row0 + m;
      const float mu = sd[m][j], raw = sd[m][A + j];
      const float eps = policy_noise(K, P, rep, r, j);
      const PolicyPoint pp = policy_point(mu, raw, eps, K.action_scale);
      lp_s[m][j] = pp.logp_j;
      ls_s[m][j] = pp.logstd;
      float* sv = P.psave + rep * P.rsSave + ((long long)r * A + j) * kSaveW;
      sv[0] = pp.std; sv[1] = pp.diff; sv[2] = pp.t; sv[3] = pp.act; sv[4] = pp.jac; sv[5] = pp.eps; sv[6] = pp.mask;
      sv[7] = pp.logp_j;
      (P.act_out + rep * P.rsAct)[(long long)r * A + j] = pp.act;
      float* pout = P.pout + rep * P.rsPout + (long long)r * NO;
      pout[j] = mu;
      pout[A + j] = raw;
      if (r < B) (P.XT + rep * P.rsX)[(long long)r * K.ldx + K.in_w + j] = pp.act;
      else (P.XP + rep * P.rsX)[(long long)(r - B) * K.ldx + K.in_w + j] = pp.act;
    }
  }
  __syncwarp();
  if (lane < nrows) {                            // sums over the actions in index order, like the per-row version
    float tot = 0.f, tls = 0.f;
    for (int j = 0; j < A; ++j) { tot += lp_s[lane][j]; tls += ls_s[lane][j]; }
    (P.logp + rep * P.rsLogp)[row0 + lane] = tot;
    (P.logstd_sum + rep * P.rsLogp)[row0 + lane] = tls;
  }
}

// ------------------------------------------------------------------------------------------
// Critic heads for the critic update: scalar heads of Qt1,Qt2 (target pass) and Q1,Q2 (s,a),
// TD target and MSE gradient in one pass, one warp per row.
//   y = rs*r + gamma*(1-d)*(min(Qt1,Qt2) - alpha*logp')          LL/learner.py:210
//   dL/dQk = 2c (Qk - y)                                        LL/model.py:139-140
// ------------------------------------------------------------------------------------------
struct CriticHeadArgs {
  const float* hT; const float* hQ; long long rsHnet, rsHrep; int ldh;   // [net][B][Hc] per replica
  const float* Wt[2]; const float* bt[2]; const float* Wq[2]; const float* bq[2]; long long rsP;
  const float* r; const float* d; const int* tid; long long rsR;
  const float* logp; long long rsLogp;   // logp[0..B) = next-state half
  const float* log_alpha;                // param arena pointer (per replica rsP)
  float* y; float* q; float* dq; float* lq; long long rsY;   // y[B], q[2][B], dq[2][B], lq[B]
};

// Lane-strided dot product; eight strides (256 columns) of both operands are in flight before the first FMA so a
// 256-wide head costs one memory round trip instead of eight.  Per-lane accumulation order is unchanged (k ascending).
B200_D float warp_dot_partial(const float* __restrict__ x, const float* __restrict__ w, int n, int lane) {
  float a = 0.f;
  for (int k0 = 0; k0 < n; k0 += 256) {
    float xv[8], wv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int k = k0 + lane + 32 * u;
      xv[u] = k < n ? x[k] : 0.f;
      wv[u] = k < n ? __ldg(w + k) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (k0 + lane + 32 * u < n) a = fmaf(xv[u], wv[u], a);
  }
  return a;
}
B200_D float warp_dot(const float* __restrict__ x, const float* __restrict__ w, int n, int lane) {
  return warp_sum(warp_dot_partial(x, w, n, lane));
}

__global__ void critic_heads_kernel(StepConst K, CriticHeadArgs P) {
  KStamp ks_;
  const int rep = blockIdx.y;
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int row = blockIdx.x * (blockDim.x / 32) + warp;
  const int B = K.B, H = K.Hc;
  if (row >= B) return;
  const float* hT = P.hT + rep * P.rsHrep + (long long)row * P.ldh;
  const float* hQ = P.hQ + rep * P.rsHrep + (long long)row * P.ldh;
  const long long po = rep * P.rsP;
  // per-row scalars and the four heads' operands are all requested before anything is consumed
  const int t = (P.tid + rep * P.rsR)[row];
  const float r = (P.r + rep * P.rsR)[row], d = (P.d + rep * P.rsR)[row];
  const float lp = (P.logp + rep * P.rsLogp)[row];
  const float b_t1 = (P.bt[0] + po)[0], b_t2 = (P.bt[1] + po)[0], b_q1 = (P.bq[0] + po)[0], b_q2 = (P.bq[1] + po)[0];
  const float p_t1 = warp_dot_partial(hT, P.Wt[0] + po, H, lane), p_t2 = warp_dot_partial(hT + P.rsHnet, P.Wt[1] + po, H, lane);
  const float p_q1 = warp_dot_partial(hQ, P.Wq[0] + po, H, lane), p_q2 = warp_dot_partial(hQ + P.rsHnet, P.Wq[1] + po, H, lane);
  const float la_t = (P.log_alpha + po)[t];
  const float qt1 = warp_sum(p_t1) + b_t1, qt2 = warp_sum(p_t2) + b_t2, q1 = warp_sum(p_q1) + b_q1, q2 = warp_sum(p_q2) + b_q2;
  if (lane == 0) {
    const float alpha = (float)exp((double)la_t);
    const float t1 = K.reward_scale * r;
    const float t2 = K.gamma * (1.f - d);
    const float t3 = fminf(qt1, qt2) - alpha * lp;
    const float y = t1 + t2 * t3;
    const float e1 = y - q1, e2 = y - q2;
    float* Y = P.y + rep * P.rsY;
    Y[row] = y;
    float* Q = P.q + rep * 2 * P.rsY;
    Q[row] = q1; Q[B + row] = q2;
    float* DQ = P.dq + rep * 2 * P.rsY;
    DQ[row] = 2.f * K.c_loss * (q1 - y);
    DQ[B + row] = 2.f * K.c_loss * (q2 - y);
    (P.lq + rep * P.rsY)[row] = e1 * e1 + e2 * e2;
  }
}

// ------------------------------------------------------------------------------------------
// Actor-pass heads: Q1,Q2 at (s, a~) with the already-updated critics, min and its gradient
// routing (LL/learner.py:222-223; torch.minimum backward: the smaller head gets the gradient,
// ties split it), plus the per-row policy-loss term (LL/model.py:84-88).
// ------------------------------------------------------------------------------------------
struct ActorQHeadArgs {
  const float* hP; long long rsHnet, rsHrep; int ldh;
  const float* Wq[2]; const float* bq[2]; long long rsP;
  const int* tid; long long rsR;
  const float* logp; long long rsLogp;    // +B offset applied by the host: current-state half
  const float* log_alpha;
  float* dqa; float* la; float* qmin; long long rsY;   // dqa[2][B], la[B], qmin[B]
};

__global__ void actor_q_heads_kernel(StepConst K, ActorQHeadArgs P) {
  KStamp ks_;
  const int rep = blockIdx.y;
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int row = blockIdx.x * (blockDim.x / 32) + warp;
  const int B = K.B, H = K.Hc;
  if (row >= B) return;
  const float* hP = P.hP + rep * P.rsHrep + (long long)row * P.ldh;
  const long long po = rep * P.rsP;
  const int t = (P.tid + rep * P.rsR)[row];
  const float lp = (P.logp + rep * P.rsLogp)[row];
  const float b_q1 = (P.bq[0] + po)[0], b_q2 = (P.bq[1] + po)[0];
  const float p_q1 = warp_dot_partial(hP, P.Wq[0] + po, H, lane), p_q2 = warp_dot_partial(hP + P.rsHnet, P.Wq[1] + po, H, lane);
  const float la_t = (P.log_alpha + po)[t];
  const float q1 = warp_sum(p_q1) + b_q1, q2 = warp_sum(p_q2) + b_q2;
  if (lane == 0) {
    const float alpha = (float)exp((double)la_t);
    const float qm = fminf(q1, q2);
    float g1, g2;
    if (q1 == q2) { g1 = g2 = -0.5f * K.c_loss; }
    else if (q1 < q2) { g1 = -K.c_loss; g2 = 0.f; }
    else { g1 = 0.f; g2 = -K.c_loss; }
    float* DQ = P.dqa + rep * 2 * P.rsY;
    DQ[row] = g1; DQ[B + row] = g2;
    (P.la + rep * P.rsY)[row] = -(qm - alpha * lp);
    (P.qmin + rep * P.rsY)[row] = qm;
  }
}

// ------------------------------------------------------------------------------------------
// Backward of a narrow output layer (N_out <= 16: the scalar Q heads and the 2*act policy
// head).  One CTA per 32-column slab of the hidden width, looping over all rows:
//   dh[m][k] = (sum_j dout[m][j] W[j][k]) * [h[m][k] > 0]
//   dW[j][k] = sum_m dout[m][j] h[m][k],  db[j] = sum_m dout[m][j]
// In policy mode dout is produced on the fly from d(action) and the values saved by the
// policy head (closed-form backward of LL/model.py:50-60, oracle/sac_manual.py).
// ------------------------------------------------------------------------------------------
struct HeadBwdArgs {
  int M, NO, Kdim, nets;
  const float* dout; long long rsDoutNet, rsDoutRep;         // [net][M][NO] (critic mode)
  const float* W[2]; long long rsP;                          // head weights [NO][Kdim]
  const float* h; long long rsHnet, rsHrep; int ldh;         // [net][M][Kdim]
  float* dh; long long rsDhNet, rsDhRep; int lddh;
  float* dW[2]; float* db[2]; long long rsG;                 // grad arena (null -> no wgrad)
  int row_slices;                                            // rows are cut into this many slices (grid.x = col blocks x slices);
  float* dWx[2]; float* dbx[2]; long long xs;                // slice s >= 1 writes gradient slice s (summed by Adam, like split-K)
  int policy_mode;
  const float* dx; long long rsDxNet, rsDxRep; int lddx;     // [2][B][xw] critic input grads
  const float* psave; long long rsSave;                      // rows B..2B-1 pre-offset by host
  const int* tid; long long rsR;
  const float* log_alpha;
  float* dout_dbg; long long rsDbg;                          // optional dump of dout / d_action
  float* dact_dbg;
};

// d(loss)/d(mu | log_std) of one (row, action) from the values the policy head saved: the closed-form backward of
// LL/model.py:50-60 in the reference's evaluation order (oracle/sac_manual.py).
B200_D void policy_dout_point(const StepConst& K, const float* __restrict__ sv, float da, float alpha, float& dmu, float& dls) {
  const float k = K.action_scale;
  const float std = sv[0], diff = sv[1], t = sv[2], act = sv[3], jac = sv[4], eps = sv[5], mask = sv[6];
  const float glp = K.c_loss * alpha;
  const float var = std * std;
  const float d_act = da + glp * (2.f * (act / k) / k) * k / jac;
  const float g_u_t = d_act * k * (1.f - t * t);
  const float g_u = g_u_t + glp * (-(diff) / var);
  dmu = g_u + glp * (diff / var);
  const float dstd = g_u * eps + glp * ((diff * diff) / (var * std) - 1.f / std);
  dls = dstd * std * mask;
}

struct PolicyDoutArgs {
  const float* dx; long long rsDxNet, rsDxRep; int lddx;
  const float* psave; long long rsSave;
  const int* tid; long long rsR;
  const float* log_alpha; long long rsP;
  float* dout; float* dact; long long rsDout;     // [M][2A], [M][A]
  int M;
};

// Large batches: compute the policy-head output gradient once (instead of in every head_bwd CTA).
__global__ void __launch_bounds__(256) policy_dout_kernel(StepConst K, PolicyDoutArgs P) {
  KStamp ks_;
  const int rep = blockIdx.y, A = K.act;
  const int e = blockIdx.x * 256 + threadIdx.x;
  if (e >= P.M * A) return;
  const int m = e / A, j = e % A;
  const float* __restrict__ sv = P.psave + rep * P.rsSave + ((long long)m * A + j) * kSaveW;
  const float* __restrict__ dx0 = P.dx + rep * P.rsDxRep + (long long)m * P.lddx + K.in_w + j;
  const float da = dx0[0] + dx0[P.rsDxNet];
  const float alpha = (float)exp((double)(P.log_alpha + rep * P.rsP)[(P.tid + rep * P.rsR)[m]]);
  float dmu, dls;
  policy_dout_point(K, sv, da, alpha, dmu, dls);
  float* o = P.dout + rep * P.rsDout + (long long)m * 2 * A;
  o[j] = dmu;
  o[A + j] = dls;
  (P.dact + rep * P.rsDout)[(long long)m * A + j] = da;
}

constexpr int kHbCols = 8;     // hidden columns per CTA
constexpr int kHbRows = 32;    // row groups per CTA (256 threads = 8 cols x 32 row groups)

__global__ void __launch_bounds__(256) head_bwd_kernel(StepConst K, HeadBwdArgs P) {
  KStamp ks_;
  extern __shared__ float sm[];
  const int net = blockIdx.y, rep = blockIdx.z;
  const int NO = P.NO, KD = P.Kdim;
  const int ncb = (KD + kHbCols - 1) / kHbCols;
  const int slice = blockIdx.x / ncb, cb = blockIdx.x - slice * ncb;
  const int rows_per = (P.M + P.row_slices - 1) / P.row_slices;
  const int r0 = slice * rows_per, r1 = (r0 + rows_per < P.M) ? r0 + rows_per : P.M;
  const int M = r1 - r0;                // rows of this slice (>= 1 by construction of the grid)
  if (M <= 0) return;
  float* sd = sm;                       // [M][NO]
  float* red = sm + (size_t)rows_per * NO;     // [32][8][NO] partial dW / scratch (>= 256 floats)
  const int tid = threadIdx.x, tx = tid % kHbCols, ty = tid / kHbCols;

  if (P.policy_mode) {
    const int A = K.act;
    __shared__ float s_alpha[64];                       // exp(log_alpha[t]) once per task, not per (row, action)
    const int Teff = K.T > 0 ? K.T : 1;
    if (tid < Teff) s_alpha[tid] = (float)exp((double)(P.log_alpha + rep * P.rsP)[tid]);
    __syncthreads();
    for (int e = tid; e < M * A; e += 256) {
      const int ml = e / A, j = e % A, m = r0 + ml;
      const float* __restrict__ sv = P.psave + rep * P.rsSave + ((long long)m * A + j) * kSaveW;
      const float* __restrict__ dx0 = P.dx + rep * P.rsDxRep + (long long)m * P.lddx + K.in_w + j;
      const float da = dx0[0] + dx0[P.rsDxNet];
      const int tk = (P.tid + rep * P.rsR)[m];
      float dmu, dls;
      policy_dout_point(K, sv, da, s_alpha[tk], dmu, dls);
      sd[ml * NO + j] = dmu;
      sd[ml * NO + A + j] = dls;
      if (P.dout_dbg && cb == 0) {
        (P.dout_dbg + rep * P.rsDbg)[(long long)m * NO + j] = dmu;
        (P.dout_dbg + rep * P.rsDbg)[(long long)m * NO + A + j] = dls;
        (P.dact_dbg + rep * P.rsDbg)[(long long)m * A + j] = da;
      }
    }
  } else {
    const float* __restrict__ src = P.dout + rep * P.rsDoutRep + net * P.rsDoutNet + (long long)r0 * NO;
    for (int e = tid; e < M * NO; e += 256) sd[e] = src[e];
  }

  const int kcol = cb * kHbCols + tx;
  const bool kin = kcol < KD;
  const float* __restrict__ W = P.W[net] + rep * P.rsP;
  float w[kMaxHeadOut], gw[kMaxHeadOut];
#pragma unroll
  for (int j = 0; j < kMaxHeadOut; ++j) {        // head weights requested before the staging barrier
    w[j] = (j < NO && kin) ? W[(long long)j * KD + kcol] : 0.f;
    gw[j] = 0.f;
  }
  __syncthreads();
  const float* __restrict__ h = P.h + rep * P.rsHrep + net * P.rsHnet + (long long)r0 * P.ldh;
  float* __restrict__ dh = P.dh + rep * P.rsDhRep + net * P.rsDhNet + (long long)r0 * P.lddh;
  constexpr int U = 8;                                   // rows in flight per thread
  for (int mb = ty; mb < M; mb += kHbRows * U) {
    float hv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int m = mb + u * kHbRows;
      hv[u] = (kin && m < M) ? h[(long long)m * P.ldh + kcol] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int m = mb + u * kHbRows;
      if (m < M) {
        float ds = 0.f;
#pragma unroll
        for (int j = 0; j < kMaxHeadOut; ++j) {
          if (j < NO) {
            const float dv = sd[m * NO + j];
            ds = fmaf(dv, w[j], ds);
            gw[j] = fmaf(dv, hv[u], gw[j]);
          }
        }
        if (kin) dh[(long long)m * P.lddh + kcol] = hv[u] > 0.f ? ds : 0.f;
      }
    }
  }
  if (P.dW[net] != nullptr) {
    float* __restrict__ dWp = (slice == 0 ? P.dW[net] : P.dWx[net] + (long long)(slice - 1) * P.xs) + rep * P.rsG;
    float* __restrict__ dbp = (slice == 0 ? P.db[net] : P.dbx[net] + (long long)(slice - 1) * P.xs) + rep * P.rsG;
#pragma unroll
    for (int j = 0; j < kMaxHeadOut; ++j)
      if (j < NO) red[(ty * kHbCols + tx) * NO + j] = gw[j];
    __syncthreads();
    if (ty < NO && kin) {                 // thread (ty = output j, tx = column): fixed-order sum over row groups
      float ssum = 0.f;
      for (int q = 0; q < kHbRows; ++q) ssum += red[(q * kHbCols + tx) * NO + ty];
      dWp[(long long)ty * KD + kcol] = ssum;
    }
    if (cb == 0) {                     // bias gradient: per-thread row sums -> warp shuffle tree -> 8 warp partials (fixed order)
      __syncthreads();
      float part[kMaxHeadOut];
#pragma unroll
      for (int j = 0; j < kMaxHeadOut; ++j) part[j] = 0.f;
      for (int m = tid; m < M; m += 256) {
#pragma unroll
        for (int j = 0; j < kMaxHeadOut; ++j)
          if (j < NO) part[j] += sd[m * NO + j];
      }
#pragma unroll
      for (int j = 0; j < kMaxHeadOut; ++j)
        if (j < NO) {
          const float v = warp_sum(part[j]);
          if ((tid & 31) == 0) red[(tid >> 5) * kMaxHeadOut + j] = v;
        }
      __syncthreads();
      if (tid < NO) {
        float ssum = 0.f;
#pragma unroll
        for (int wq = 0; wq < 8; ++wq) ssum += red[wq * kMaxHeadOut + tid];
        dbp[tid] = ssum;
      }
    }
  }
}

// The same backward with 128-bit column accesses: thread = 4 consecutive hidden columns x one of 16 row groups, CTA = 64
// columns x one row slice.  The 8-column mapping above reads and writes 32 bytes per row per warp quarter (four sectors per
// warp instruction) and needs 50 column blocks x 4 slices x 2 nets = 400 CTAs at the 400-wide shapes -- 10.4 us at B = 1 024,
// 13 us at 1 280 (profiles/r2_bench_VS.json, round 2); here a warp instruction moves two full 256-byte row segments.  Used
// when the hidden width is a multiple of 4 (row pitches then are too); same fixed-order reductions, different grouping.
constexpr int kHb4Cols = 64;   // hidden columns per CTA (16 threads x float4)
constexpr int kHb4Rows = 16;   // row groups per CTA

template <int NOMAX>
__global__ void __launch_bounds__(256) head_bwd4_kernel(StepConst K, HeadBwdArgs P) {
  KStamp ks_;
  extern __shared__ float sm[];
  const int net = blockIdx.y, rep = blockIdx.z;
  const int NO = P.NO, KD = P.Kdim;
  const int ncb = (KD + kHb4Cols - 1) / kHb4Cols;
  const int slice = blockIdx.x / ncb, cb = blockIdx.x - slice * ncb;
  const int rows_per = (P.M + P.row_slices - 1) / P.row_slices;
  const int r0 = slice * rows_per, r1 = (r0 + rows_per < P.M) ? r0 + rows_per : P.M;
  const int M = r1 - r0;
  if (M <= 0) return;
  float* sd = sm;                                   // [M][NO]
  // [16 row groups][16 col quads][NO][4], stored as float4: 16-B aligned behind sd whatever rows_per * NO is (an odd batch)
  float* red = sm + (((size_t)rows_per * NO + 3) & ~(size_t)3);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

  if (P.policy_mode) {
    const int A = K.act;
    __shared__ float s_alpha[64];
    const int Teff = K.T > 0 ? K.T : 1;
    if (tid < Teff) s_alpha[tid] = (float)exp((double)(P.log_alpha + rep * P.rsP)[tid]);
    __syncthreads();
    for (int e = tid; e < M * A; e += 256) {
      const int ml = e / A, j = e % A, m = r0 + ml;
      const float* __restrict__ sv = P.psave + rep * P.rsSave + ((long long)m * A + j) * kSaveW;
      const float* __restrict__ dx0 = P.dx + rep * P.rsDxRep + (long long)m * P.lddx + K.in_w + j;
      const float da = dx0[0] + dx0[P.rsDxNet];
      const int tk = (P.tid + rep * P.rsR)[m];
      float dmu, dls;
      policy_dout_point(K, sv, da, s_alpha[tk], dmu, dls);
      sd[ml * NO + j] = dmu;
      sd[ml * NO + A + j] = dls;
      if (P.dout_dbg && cb == 0) {
        (P.dout_dbg + rep * P.rsDbg)[(long long)m * NO + j] = dmu;
        (P.dout_dbg + rep * P.rsDbg)[(long long)m * NO + A + j] = dls;
        (P.dact_dbg + rep * P.rsDbg)[(long long)m * A + j] = da;
      }
    }
  } else {
    const float* __restrict__ src = P.dout + rep * P.rsDoutRep + net * P.rsDoutNet + (long long)r0 * NO;
    for (int e = tid; e < M * NO; e += 256) sd[e] = src[e];
  }

  const int kcol = cb * kHb4Cols + 4 * tx;          // first of this thread's four columns (KD % 4 == 0: all four valid or none)
  const bool kin = kcol < KD;
  const float* __restrict__ W = P.W[net] + rep * P.rsP;
  float4 w[NOMAX], gw[NOMAX];
#pragma unroll
  for (int j = 0; j < NOMAX; ++j) {                 // head weights requested before the staging barrier
    w[j] = (j < NO && kin) ? *reinterpret_cast<const float4*>(W + (long long)j * KD + kcol) : make_float4(0.f, 0.f, 0.f, 0.f);
    gw[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  const float* __restrict__ h = P.h + rep * P.rsHrep + net * P.rsHnet + (long long)r0 * P.ldh;
  float* __restrict__ dh = P.dh + rep * P.rsDhRep + net * P.rsDhNet + (long long)r0 * P.lddh;
  constexpr int U = 8;                              // rows in flight per thread
  for (int mb = ty; mb < M; mb += kHb4Rows * U) {
    float4 hv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int m = mb + u * kHb4Rows;
      hv[u] = (kin && m < M) ? *reinterpret_cast<const float4*>(h + (long long)m * P.ldh + kcol) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int m = mb + u * kHb4Rows;
      if (m < M) {
        float4 ds = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < NOMAX; ++j) {
          if (j < NO) {
            const float dv = sd[m * NO + j];
            ds.x = fmaf(dv, w[j].x, ds.x); ds.y = fmaf(dv, w[j].y, ds.y); ds.z = fmaf(dv, w[j].z, ds.z); ds.w = fmaf(dv, w[j].w, ds.w);
            gw[j].x = fmaf(dv, hv[u].x, gw[j].x); gw[j].y = fmaf(dv, hv[u].y, gw[j].y);
            gw[j].z = fmaf(dv, hv[u].z, gw[j].z); gw[j].w = fmaf(dv, hv[u].w, gw[j].w);
          }
        }
        if (kin)
          *reinterpret_cast<float4*>(dh + (long long)m * P.lddh + kcol) =
              make_float4(hv[u].x > 0.f ? ds.x : 0.f, hv[u].y > 0.f ? ds.y : 0.f, hv[u].z > 0.f ? ds.z : 0.f, hv[u].w > 0.f ? ds.w : 0.f);
      }
    }
  }
  if (P.dW[net] != nullptr) {
    float* __restrict__ dWp = (slice == 0 ? P.dW[net] : P.dWx[net] + (long long)(slice - 1) * P.xs) + rep * P.rsG;
    float* __restrict__ dbp = (slice == 0 ? P.db[net] : P.dbx[net] + (long long)(slice - 1) * P.xs) + rep * P.rsG;
#pragma unroll
    for (int j = 0; j < NOMAX; ++j)
      if (j < NO) *reinterpret_cast<float4*>(red + ((size_t)(ty * 16 + tx) * NO + j) * 4) = gw[j];
    __syncthreads();
    for (int o = tid; o < NO * kHb4Cols; o += 256) {   // (output j, column cc): fixed-order sum over the 16 row groups
      const int j = o / kHb4Cols, cc = o - j * kHb4Cols;
      const int col = cb * kHb4Cols + cc;
      if (col < KD) {
        float ssum = 0.f;
#pragma unroll
        for (int q = 0; q < kHb4Rows; ++q) ssum += red[((size_t)(q * 16 + (cc >> 2)) * NO + j) * 4 + (cc & 3)];
        dWp[(long long)j * KD + col] = ssum;
      }
    }
    if (cb == 0) {                     // bias gradient: per-thread row sums -> warp shuffle tree -> 8 warp partials (fixed order)
      __syncthreads();
      float part[NOMAX];
#pragma unroll
      for (int j = 0; j < NOMAX; ++j) part[j] = 0.f;
      for (int m = tid; m < M; m += 256) {
#pragma unroll
        for (int j = 0; j < NOMAX; ++j)
          if (j < NO) part[j] += sd[m * NO + j];
      }
#pragma unroll
      for (int j = 0; j < NOMAX; ++j)
        if (j < NO) {
          const float v = warp_sum(part[j]);
          if ((tid & 31) == 0) red[(tid >> 5) * kMaxHeadOut + j] = v;
        }
      __syncthreads();
      if (tid < NO) {
        float ssum = 0.f;
#pragma unroll
        for (int wq = 0; wq < 8; ++wq) ssum += red[wq * kMaxHeadOut + tid];
        dbp[tid] = ssum;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// Adam (torch.optim.adam._single_tensor_adam, defaults) over a contiguous slice of the
// trainable arena, optionally fused with the Polyak update of the matching target slice
// (LL/learner.py:126-137,236-237).  The target critics are only read at the start of a step
// and the local critics do not change after critic_optimizer.step(), so doing the Polyak
// write here is exactly equivalent to the reference's end-of-step soft_update.
// The extra last CTA runs a "tail job": scalar reductions that must be deterministic.
// ------------------------------------------------------------------------------------------
enum { TAIL_NONE = 0, TAIL_CRITIC_LOSS = 1, TAIL_ALPHA_AND_LOSSES = 2, TAIL_ALL = 3 };   // ALL = critic loss + actor loss / entropy / temperature

struct AdamArgs {
  float* p; float* m; float* v; const float* g;     // slice bases (replica 0)
  const float* gx; long long xs; int nx;             // nx extra gradient slices (split-K weight gradients), slice stride xs
  long long rsP, rsM;                                // replica strides: param arena / trainable arena
  long long n;
  long long target_delta;                            // p[i + target_delta] is the Polyak target (0 = none)
  long long tau2_begin;                              // elements i >= tau2_begin use (tau2, 1 - tau2): CARE state encoder
  float tau2, one_minus_tau2;
  int which;                                         // counter index (0 critic, 1 actor)
  double lr;
  const Counters* cnt;
  int tail;
  // tail inputs
  const float* lq; const float* la; const float* logp_cur; const float* logstd_sum; const int* tid;
  long long rsY, rsLogp, rsR;
  float* log_alpha; float* m_alpha; float* v_alpha; float* g_alpha;   // arena pointers
  float* losses;                                     // [kLossSlots][R][4] device ring
  float* losses_host;                                // same ring in mapped pinned host memory (zero-copy D2H)
  int R;
};

B200_D void adam_scalars(double lr, double b1_pow_t, double b2_pow_t, float& step_size, float& bc2_sqrt) {
  const double bc1 = 1.0 - b1_pow_t;        // bias_correction1 = 1 - beta1 ** step
  const double bc2 = 1.0 - b2_pow_t;
  step_size = (float)(lr / bc1);
  bc2_sqrt = (float)sqrt(bc2);
}

B200_D void adam_one(float& p, float& m, float& v, float g, float w1, float b2, float omb2, float step_size,
                     float bc2_sqrt, float eps) {
  m = m + w1 * (g - m);                       // exp_avg.lerp_(grad, 1 - beta1)
  v = v * b2 + omb2 * g * g;                  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1-beta2)
  const float denom = sqrtf(v) / bc2_sqrt + eps;
  p = p - step_size * (m / denom);            // param.addcdiv_(exp_avg, denom, value=-step_size)
}

__global__ void __launch_bounds__(256) adam_kernel(StepConst K, AdamArgs P) {
  KStamp ks_;
  const int rep = blockIdx.y;
  __shared__ float red[256];
  __shared__ float s_ss, s_bc;
  const bool is_tail = (P.tail != TAIL_NONE) && (blockIdx.x == gridDim.x - 1);
  if (!is_tail) {
    if (threadIdx.x == 0) {
      float a, b;
      adam_scalars(P.lr, P.cnt[rep].b1p[P.which], P.cnt[rep].b2p[P.which], a, b);
      s_ss = a; s_bc = b;
    }
    __syncthreads();
    const float step_size = s_ss, bc2_sqrt = s_bc;
    const float w1 = (float)(1.0 - K.beta1), b2 = (float)K.beta2, omb2 = (float)(1.0 - K.beta2);
    const float eps = (float)K.adam_eps;
    const int nb = (P.tail != TAIL_NONE) ? gridDim.x - 1 : gridDim.x;
    float* p = P.p + rep * P.rsP;
    float* m = P.m + rep * P.rsM;
    float* v = P.v + rep * P.rsM;
    const float* g = P.g + rep * P.rsM;
    // 128-bit accesses, all five streams of an element group in flight before the math (slices are
    // multiples of 4 floats and 16-B aligned by construction of the arena)
    const long long n4 = P.n >> 2;
    float4* __restrict__ p4 = reinterpret_cast<float4*>(p);
    float4* __restrict__ m4 = reinterpret_cast<float4*>(m);
    float4* __restrict__ v4 = reinterpret_cast<float4*>(v);
    const float4* __restrict__ g4 = reinterpret_cast<const float4*>(g);
    float4* __restrict__ t4 = P.target_delta != 0 ? reinterpret_cast<float4*>(p + P.target_delta) : nullptr;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)nb * 256) {
      float4 pv = p4[i], mv = m4[i], vv = v4[i];
      float4 gv = g4[i];
      // split-K slices, added in index order; the first three are requested together with everything else (a run-time loop
      // kept each slice's load behind the previous slice's add: three extra round trips per element group)
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4* __restrict__ gx4 = reinterpret_cast<const float4*>(P.gx + rep * P.rsM);
      const long long xs4 = P.xs >> 2;               // (slice stride: a multiple of 4 floats like every arena)
      const float4 ge0 = P.nx > 0 ? gx4[i] : z4, ge1 = P.nx > 1 ? gx4[xs4 + i] : z4, ge2 = P.nx > 2 ? gx4[2 * xs4 + i] : z4;
      float4 tv = z4;
      if (t4) tv = t4[i];
      if (P.nx > 0) { gv.x += ge0.x; gv.y += ge0.y; gv.z += ge0.z; gv.w += ge0.w; }
      if (P.nx > 1) { gv.x += ge1.x; gv.y += ge1.y; gv.z += ge1.z; gv.w += ge1.w; }
      if (P.nx > 2) { gv.x += ge2.x; gv.y += ge2.y; gv.z += ge2.z; gv.w += ge2.w; }
      for (int sx = 3; sx < P.nx; ++sx) {
        const float4 ge = gx4[(long long)sx * xs4 + i];
        gv.x += ge.x; gv.y += ge.y; gv.z += ge.z; gv.w += ge.w;
      }
      adam_one(pv.x, mv.x, vv.x, gv.x, w1, b2, omb2, step_size, bc2_sqrt, eps);
      adam_one(pv.y, mv.y, vv.y, gv.y, w1, b2, omb2, step_size, bc2_sqrt, eps);
      adam_one(pv.z, mv.z, vv.z, gv.z, w1, b2, omb2, step_size, bc2_sqrt, eps);
      adam_one(pv.w, mv.w, vv.w, gv.w, w1, b2, omb2, step_size, bc2_sqrt, eps);
      p4[i] = pv; m4[i] = mv; v4[i] = vv;
      if (t4) {
        const bool second = (i << 2) >= P.tau2_begin;         // tau2_begin is a multiple of 4 (tensor offsets are)
        const float ta = second ? P.tau2 : K.tau, tb = second ? P.one_minus_tau2 : K.one_minus_tau;
        tv.x = ta * pv.x + tb * tv.x; tv.y = ta * pv.y + tb * tv.y;
        tv.z = ta * pv.z + tb * tv.z; tv.w = ta * pv.w + tb * tv.w;
        t4[i] = tv;
      }
    }
    return;
  }
  // ---- tail jobs (one CTA per replica) ----
  const int tid = threadIdx.x, B = K.B, lane = tid & 31, warp = tid >> 5;
  // two block sums at once: warp shuffle trees, then the 8 warp partials in index order (fixed order -> reproducible)
  auto block_sum2 = [&](float x, float y, float& sx, float& sy) {
    x = warp_sum(x); y = warp_sum(y);
    if (lane == 0) { red[warp] = x; red[8 + warp] = y; }
    __syncthreads();
    sx = 0.f; sy = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) { sx += red[q]; sy += red[8 + q]; }
    __syncthreads();
  };
  const long long slot = (P.cnt[rep].v[3] - 1) % kLossSlots;
  float* L = P.losses + ((long long)slot * P.R + rep) * 4;
  float* LH = P.losses_host + ((long long)slot * P.R + rep) * 4;
  if (P.tail == TAIL_CRITIC_LOSS || P.tail == TAIL_ALL) {
    float s = 0.f, dummy;
    for (int i = tid; i < B; i += 256) s += (P.lq + rep * P.rsY)[i];
    block_sum2(s, 0.f, s, dummy);
    if (tid == 0) { L[0] = s * K.c_loss; LH[0] = L[0]; }
    if (P.tail == TAIL_CRITIC_LOSS) return;
  }
  // TAIL_ALPHA_AND_LOSSES: actor loss, entropy, temperature gradient + its Adam step
  {
    const int Teff = K.T > 0 ? K.T : 1;
    float* la = P.log_alpha + rep * P.rsP;
    __shared__ float s_gs[64];
    __shared__ float s_la[64], s_m[64], s_v[64];
    // everything the serial part needs is requested up front, next to the reduction inputs
    if (tid < Teff) { s_la[tid] = la[tid]; s_m[tid] = (P.m_alpha + rep * P.rsM)[tid]; s_v[tid] = (P.v_alpha + rep * P.rsM)[tid]; }
    const double b1p = P.cnt[rep].b1p[2], b2p = P.cnt[rep].b2p[2];
    float s = 0.f, e = 0.f;
    for (int i = tid; i < B; i += 256) {
      s += (P.la + rep * P.rsY)[i];
      e += (P.logstd_sum + rep * P.rsLogp)[i];
    }
    {   // per-task sums of (logp + Hbar): one warp per task, lanes stride the rows, shuffle tree -> fixed order
      const int* __restrict__ tv = P.tid + rep * P.rsR;
      const float* __restrict__ lp = P.logp_cur + rep * P.rsLogp;
      for (int t = warp; t < Teff; t += 8) {
        float gs = 0.f;
        for (int i = lane; i < B; i += 32)
          if (tv[i] == t) gs += lp[i] + K.hbar;
        gs = warp_sum(gs);
        if (lane == 0) s_gs[t] = gs;
      }
    }
    block_sum2(s, e, s, e);          // its barriers also publish s_gs / s_la / s_m / s_v
    if (tid == 0) {
      L[1] = s * K.c_loss;
      L[3] = 0.5f * K.act * (1.0f + 1.8378770664093453f) + e * K.inv_B;   // 0.5 A (1+log 2pi) + mean(sum log_std)
      LH[1] = L[1]; LH[3] = L[3];
      float ss, bc;
      adam_scalars(K.lr_alpha, b1p, b2p, ss, bc);
      float aloss = 0.f;
      for (int t = 0; t < Teff; ++t) {
        const float grad = -s_gs[t] * K.inv_B;         // d/dlog_alpha[t] of -mean(log_alpha_i (logp_i + Hbar))
        aloss += s_la[t] * grad;                       // loss value = sum_t log_alpha[t] * grad[t]
        (P.g_alpha + rep * P.rsM)[t] = grad;
        float pi = s_la[t], mi = s_m[t], vi = s_v[t];
        adam_one(pi, mi, vi, grad, (float)(1.0 - K.beta1), (float)K.beta2, (float)(1.0 - K.beta2), ss, bc,
                 (float)K.adam_eps);
        la[t] = pi; (P.m_alpha + rep * P.rsM)[t] = mi; (P.v_alpha + rep * P.rsM)[t] = vi;
      }
      L[2] = aloss; LH[2] = aloss;     // mapped pinned memory: visible to the host once the stream has drained
    }
  }
}

// Stand-alone Polyak (Learner.soft_update outside a step; tau = 1 -> hard copy).
__global__ void polyak_kernel(float* p, long long rsP, long long n, long long target_delta, float tau,
                              float one_minus_tau, long long n_tau1 = -1, float tau2 = 0.f, float one_minus_tau2 = 0.f) {
  float* q = p + blockIdx.y * rsP;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const bool second = n_tau1 >= 0 && i >= n_tau1;
    q[i + target_delta] = second ? tau2 * q[i] + one_minus_tau2 * q[i + target_delta] : tau * q[i] + one_minus_tau * q[i + target_delta];
  }
}

// randn init of the mixture-of-encoders weights (state_encoder.py:146-153)
__global__ void randn_kernel(float* w, long long rsP, long long n, unsigned long long seed, int tag) {
  const int rep = blockIdx.y;
  Philox ph(seed + (unsigned long long)rep);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    uint32_t rnd[4];
    ph((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)tag, 0x9A11u, rnd);
    float z0, z1;
    box_muller(rnd[0], rnd[1], z0, z1);
    (w + rep * rsP)[i] = z0;
  }
}

// Synthetic replay fill (bench helper): rows [s | a | r | s2 | d | pad], SURVEY 8(d) distributions.
__global__ void fill_synthetic_kernel(float* rows, long long rs_rows, int row_stride, long long n_per_task,
                                      long long cap_per_task, int state_dim, int act, int T,
                                      unsigned long long seed) {
  const int rep = blockIdx.y;
  const int Teff = T > 0 ? T : 1;
  const int obs = state_dim + T;
  Philox ph(seed + 77ull * (unsigned long long)(rep + 1));
  const long long total = n_per_task * Teff;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    const int task = (int)(e / n_per_task);
    const long long local = e % n_per_task;
    float* row = rows + rep * rs_rows + (task * cap_per_task + local) * row_stride;
    const int nrand = 2 * state_dim + act + 2;
    for (int c = 0; c < nrand; c += 4) {
      uint32_t rnd[4];
      ph((uint32_t)e, (uint32_t)(e >> 32), (uint32_t)c, 0xF111u, rnd);
      float z[4];
      box_muller(rnd[0], rnd[1], z[0], z[1]);
      box_muller(rnd[2], rnd[3], z[2], z[3]);
      for (int q = 0; q < 4 && c + q < nrand; ++q) {
        const int j = c + q;
        if (j < state_dim) row[j] = z[q];                                                 // s
        else if (j < state_dim + act) row[obs + (j - state_dim)] = 2.f * u01(rnd[q]) - 1.f;   // a
        else if (j == state_dim + act) row[obs + act] = z[q];                                 // r
        else if (j < 2 * state_dim + act + 1) row[obs + act + 1 + (j - state_dim - act - 1)] = z[q];   // s2
        else row[2 * obs + act + 1] = (u01(rnd[q]) < 0.01f) ? 1.f : 0.f;                      // d
      }
    }
    for (int q = 0; q < T; ++q) {
      const float oh = (q == task) ? 1.f : 0.f;
      row[state_dim + q] = oh;
      row[obs + act + 1 + state_dim + q] = oh;
    }
  }
}

// Xavier-uniform init of one [out][in] matrix (nn.init.xavier_uniform_, gain 1), bias zero.
__global__ void xavier_kernel(float* w, long long rsP, int rows, int cols, int ld, unsigned long long seed, int tag) {
  const int rep = blockIdx.y;
  Philox ph(seed + (unsigned long long)rep);
  const float bound = sqrtf(6.f / (float)(rows + cols));
  const long long n = (long long)rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    uint32_t rnd[4];
    ph((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)tag, 0x1417u, rnd);
    (w + rep * rsP)[(i / cols) * ld + (i % cols)] = (2.f * u01(rnd[0]) - 1.f) * bound;
  }
}

}  // namespace bsac
