// Persistent Broyden root solver for small-d MLP branches (toy d=2, tabular d=6/43/63, hidden 128):
// ONE cooperative launch performs the whole solve of
//        g(z) = x_embed - f(z) - z = 0          (implicit_block.py:68-80, broyden.py:123-193)
// including every branch evaluation f(z) (fused fp32 MLP with the activation in registers), the
// batch-global residual norm (one grid.sync per iteration), the reference's break rules and
// best-iterate tracking, and the per-sample rank-1 updates (one warp per sample, history U^T/V^T in
// global memory that stays L2-resident: B*T*d*8 bytes = 15 MB at B=1000, d=63, T=30).
// The host reads back the 600-byte state once, after the solve — the reference synchronises the host
// on every iteration (broyden.py:145,157).
//
// Work split: a CTA owns tiles of kTile samples.  The MLP is evaluated per tile with activations in
// shared memory and weights (stored transposed, [in][out], so a warp reads consecutive neurons)
// streamed through L1/L2; each thread accumulates 4 samples x 1 neuron.  The decision logic is
// replicated in every CTA from the same partial sums in the same order, so all CTAs take identical
// branches without a second grid barrier.
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace impflow {

constexpr int kMlpThreads = 256;
constexpr int kMlpWarps = kMlpThreads / 32;
constexpr int kTile = 16;        // samples per tile
constexpr int kMaxLayers = 8;
constexpr int kMaxWidth = 256;   // widest layer (incl. d)

struct MlpDesc {
  int L;                       // number of linear layers
  int dims[kMaxLayers + 1];    // dims[0] = d, ..., dims[L] = d
  const float* Wt[kMaxLayers]; // [in][out], row stride ld
  int ld[kMaxLayers];
  const float* bias[kMaxLayers];
  const float* dmul[kMaxLayers];   // vjp mode: per-sample multiplier (B, dims[l+1]) on the output of layer l, or null
  int act_kind;
  const float* beta[kMaxLayers];   // softplus(beta) of the LipSwish behind layer l (every Swish module owns its beta)
  int mode;                    // 0: g(z) = x_embed - f(z) - z (forward / inverse solve)
                               // 1: g(v) = v^T J + v - rhs   (implicit backward; f is the transposed linear chain)
};

// out[s][n] = act?( bias[n] + sum_k in[s][k] * Wt[k][n] ) for the kTile samples of one tile.
__device__ void mlp_layer(const float* __restrict__ Wt, int ld, const float* __restrict__ bias, const float* in,
                          float* out, int K, int N, int act_kind, float beta, bool apply_act,
                          const float* __restrict__ dmul, int s0, int B) {
  // thread -> (neuron n, group of 4 samples)
  for (int idx = threadIdx.x; idx < N * (kTile / 4); idx += kMlpThreads) {
    const int n = idx % N;
    const int sg = idx / N;
    float acc[4];
    const float b = bias != nullptr ? __ldg(bias + n) : 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j] = b;
    const float* i0 = in + (sg * 4 + 0) * kMaxWidth;
    int k = 0;
    for (; k + 3 < K; k += 4) {
      const float w0 = __ldg(Wt + (long long)(k + 0) * ld + n);
      const float w1 = __ldg(Wt + (long long)(k + 1) * ld + n);
      const float w2 = __ldg(Wt + (long long)(k + 2) * ld + n);
      const float w3 = __ldg(Wt + (long long)(k + 3) * ld + n);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 h = *reinterpret_cast<const float4*>(i0 + j * kMaxWidth + k);
        acc[j] = fmaf(h.x, w0, acc[j]);
        acc[j] = fmaf(h.y, w1, acc[j]);
        acc[j] = fmaf(h.z, w2, acc[j]);
        acc[j] = fmaf(h.w, w3, acc[j]);
      }
    }
    for (; k < K; ++k) {
      const float w0 = __ldg(Wt + (long long)k * ld + n);
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = fmaf(i0[j * kMaxWidth + k], w0, acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v = apply_act ? act_dispatch(act_kind, acc[j], 0, beta) : acc[j];
      if (dmul != nullptr) {
        const int b = s0 + sg * 4 + j;
        v = b < B ? v * __ldg(dmul + (long long)b * N + n) : 0.f;
      }
      out[(sg * 4 + j) * kMaxWidth + n] = v;
    }
  }
}

// f(zin) for the tile's samples; result left in the returned smem buffer ([kTile][kMaxWidth], first d cols).
__device__ float* mlp_eval(const MlpDesc& net, const float* __restrict__ zin, int s0, int B, float* bufA, float* bufB) {
  const int d = net.dims[0];
  for (int i = threadIdx.x; i < kTile * d; i += kMlpThreads) {
    const int s = i / d, c = i % d;
    bufA[s * kMaxWidth + c] = (s0 + s < B) ? zin[(long long)(s0 + s) * d + c] : 0.f;
  }
  __syncthreads();
  float* cur = bufA;
  float* nxt = bufB;
  for (int l = 0; l < net.L; ++l) {
    const float beta = net.beta[l] != nullptr ? __ldg(net.beta[l]) : 0.f;
    mlp_layer(net.Wt[l], net.ld[l], net.bias[l], cur, nxt, net.dims[l], net.dims[l + 1], net.act_kind, beta,
              net.mode == 0 && l + 1 < net.L, net.dmul[l], s0, B);
    __syncthreads();
    float* t = cur;
    cur = nxt;
    nxt = t;
  }
  return cur;
}

struct LocalState {   // replica of impflow_broyden_state kept in shared memory by every CTA
  int nstep, lowest_step, active, prot_break, converged, stagnated, do_update, new_lowest, threshold;
  double eps, init_objective, lowest, objective;
  double trace[64];
};

__device__ void local_decide(LocalState* st, double total, bool init) {
  const double obj = (double)(float)sqrt(total);
  st->objective = obj;
  if (init) {
    st->nstep = 0; st->lowest_step = 0; st->init_objective = obj; st->lowest = obj; st->trace[0] = obj;
    st->prot_break = st->converged = st->stagnated = st->do_update = st->new_lowest = 0;
    st->active = (obj >= st->eps && 0 < st->threshold) ? 1 : 0;
    return;
  }
  const int T = st->threshold;
  const int nstep = ++st->nstep;
  st->trace[nstep] = obj;
  int new_low = 0;
  if (obj < st->lowest) { st->lowest = obj; st->lowest_step = nstep; new_low = 1; }
  st->new_lowest = new_low;
  const int conv = obj < st->eps ? 1 : 0;
  int stag = 0;
  if (!conv && obj < 3.0 * st->eps && nstep == T) {
    double mx = st->trace[nstep - T + 1], mn = mx;
    for (int i = nstep - T + 1; i <= nstep; ++i) { mx = fmax(mx, st->trace[i]); mn = fmin(mn, st->trace[i]); }
    stag = (mx / mn < 1.3) ? 1 : 0;
  }
  const int prot = (!conv && !stag && obj > st->init_objective * 1e6) ? 1 : 0;
  st->converged = conv; st->stagnated = stag; st->prot_break = prot;
  const int upd = (conv || stag || prot) ? 0 : 1;
  st->do_update = upd;
  st->active = (upd && obj >= st->eps && nstep < T) ? 1 : 0;
}

// rank-1 update of one sample by one warp (d <= 128), same algebra as k_update_small (broyden.cu).
__device__ void warp_update(float* x_old, const float* g_old, const float* xn, const float* gn, float* Ut, float* Vt,
                            int d, int T, int k, int lane) {
  float dx[4], dg[4], gg[4], xv[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int i = lane + 32 * e;
    if (i < d) {
      xv[e] = xn[i]; gg[e] = gn[i]; dx[e] = xv[e] - x_old[i]; dg[e] = gg[e] - g_old[i];
    } else {
      xv[e] = gg[e] = dx[e] = dg[e] = 0.f;
    }
  }
  float vT[4], w[4], S[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) { vT[e] = -dx[e]; w[e] = -dg[e]; S[e] = 0.f; }
  for (int j = 0; j < k; ++j) {
    float u1[4], v1[4], a = 0.f, bb = 0.f, c = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int i = lane + 32 * e;
      u1[e] = i < d ? Ut[(long long)j * d + i] : 0.f;
      v1[e] = i < d ? Vt[(long long)j * d + i] : 0.f;
      a += dx[e] * u1[e]; bb += v1[e] * dg[e]; c += v1[e] * gg[e];
    }
    a = warp_sum(a); bb = warp_sum(bb); c = warp_sum(c);
#pragma unroll
    for (int e = 0; e < 4; ++e) { vT[e] += a * v1[e]; w[e] += bb * u1[e]; S[e] += c * u1[e]; }
  }
  float den = 0.f, ck = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    den += vT[e] * dg[e];
    vT[e] = (vT[e] != vT[e]) ? 0.f : vT[e];
    ck += vT[e] * gg[e];
  }
  den = warp_sum(den);
  ck = warp_sum(ck);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int i = lane + 32 * e;
    if (i < d) {
      float u = (dx[e] - w[e]) / den;
      u = (u != u) ? 0.f : u;
      Ut[(long long)k * d + i] = u;
      Vt[(long long)k * d + i] = vT[e];
      x_old[i] = xv[e] + (-((-gg[e]) + (S[e] + u * ck)));
    }
  }
}

__global__ void __launch_bounds__(kMlpThreads)
k_mlp_broyden(MlpDesc net, const float* __restrict__ x_embed, float* za, float* ga, float* zb, float* gb,
              float* __restrict__ low_z, float* __restrict__ low_g, float* __restrict__ Ut, float* __restrict__ Vt,
              float* __restrict__ sample_sq, float* __restrict__ low_sq, double* __restrict__ partial,
              impflow_broyden_state* state, int B, int T, double eps) {
  cg::grid_group grid = cg::this_grid();
  __shared__ __align__(16) float bufA[kTile * kMaxWidth];
  __shared__ __align__(16) float bufB[kTile * kMaxWidth];
  __shared__ LocalState st;
  __shared__ double red[kMlpWarps];
  __shared__ float tile_sq[kTile];
  const int d = net.dims[0];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = (B + kTile - 1) / kTile;
  float *z_old = za, *g_old = ga, *zn = zb, *gn = gb;

  if (tid == 0) { st.threshold = T; st.eps = eps; }

  // evaluates g(zin) -> gout for this CTA's tiles, per-sample ||g||^2 -> sample_sq, returns the CTA partial
  auto eval_residual = [&](const float* zin, float* gout) -> double {
    double cta_sum = 0.0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int s0 = tile * kTile;
      float* f = mlp_eval(net, zin, s0, B, bufA, bufB);
      if (tid < kTile) tile_sq[tid] = 0.f;
      __syncthreads();
      // g = x_embed - f(z) - z (mode 0) or f(v) + v - rhs (mode 1), one warp handles samples warp, warp+8
      for (int s = warp; s < kTile; s += kMlpWarps) {
        const int b = s0 + s;
        if (b >= B) continue;
        float sq = 0.f;
        for (int c = lane; c < d; c += 32) {
          const long long i = (long long)b * d + c;
          const float fv = f[s * kMaxWidth + c];
          const float gv = net.mode == 0 ? x_embed[i] - fv - zin[i] : fv + zin[i] - x_embed[i];
          gout[i] = gv;
          sq += gv * gv;
        }
        sq = warp_sum(sq);
        if (lane == 0) { tile_sq[s] = sq; sample_sq[b] = sq; }
      }
      __syncthreads();
      if (tid == 0)
        for (int s = 0; s < kTile; ++s) cta_sum += (double)tile_sq[s];
      __syncthreads();
    }
    return cta_sum;
  };
  // all CTAs: identical fixed-order sum of the per-CTA partials of parity `p`
  auto total_of = [&](int p) -> double {
    double acc = 0.0;
    for (int i = tid; i < (int)gridDim.x; i += kMlpThreads) acc += partial[p * gridDim.x + i];
    acc = warp_sum_d(acc);
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < kMlpWarps; ++w) t += red[w];
    __syncthreads();
    return t;
  };

  // ---- g0 = g(z0), init bookkeeping, zn = z0 - g0 (broyden.py:136-151) ----
  {
    const double s = eval_residual(z_old, g_old);
    if (tid == 0) partial[blockIdx.x] = s;
  }
  grid.sync();
  {
    const double tot = total_of(0);
    if (tid == 0) local_decide(&st, tot, true);
    __syncthreads();
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
      for (int i = tid; i < kTile * d; i += kMlpThreads) {
        const int b = tile * kTile + i / d;
        if (b < B) {
          const long long idx = (long long)b * d + i % d;
          const float x = z_old[idx], g = g_old[idx];
          low_z[idx] = x; low_g[idx] = g; zn[idx] = x + (-g);
          if (i % d == 0) low_sq[b] = sample_sq[b];
        }
      }
    __syncthreads();
  }
  int parity = 1;
  while (st.active) {
    const double s = eval_residual(zn, gn);
    if (tid == 0) partial[parity * gridDim.x + blockIdx.x] = s;
    grid.sync();
    const double tot = total_of(parity);
    if (tid == 0) local_decide(&st, tot, false);
    __syncthreads();
    const int k = st.nstep - 1;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int s = warp; s < kTile; s += kMlpWarps) {
        const int b = tile * kTile + s;
        if (b >= B) continue;
        const long long base = (long long)b * d;
        if (st.new_lowest) {
          for (int c = lane; c < d; c += 32) { low_z[base + c] = zn[base + c]; low_g[base + c] = gn[base + c]; }
          if (lane == 0) low_sq[b] = sample_sq[b];
        }
        if (st.do_update)
          warp_update(z_old + base, g_old + base, zn + base, gn + base, Ut + (long long)b * T * d,
                      Vt + (long long)b * T * d, d, T, k, lane);
      }
    }
    __syncthreads();
    // the next iterate was written into z_old's buffer: swap roles (uniform over the grid)
    float* t = z_old; z_old = zn; zn = t;
    t = g_old; g_old = gn; gn = t;
    parity ^= 1;
  }
  if (blockIdx.x == 0 && tid == 0) {
    state->nstep = st.nstep; state->lowest_step = st.lowest_step; state->active = 0;
    state->prot_break = st.prot_break; state->converged = st.converged; state->stagnated = st.stagnated;
    state->do_update = st.do_update; state->new_lowest = st.new_lowest; state->threshold = T; state->counter = 0;
    state->eps = st.eps; state->init_objective = st.init_objective; state->lowest = st.lowest;
    state->objective = st.objective;
    for (int i = 0; i <= st.nstep; ++i) state->trace[i] = st.trace[i];
  }
}


// ------------------------------------------------------------------------------------------------------------
// Banach fixed-point iteration of the same branches in ONE cooperative launch (iresblock.py:69-79,
// implicit_block.py:17-28; the contract is in the header at impflow_conv3_fixed_point):
//     x_k = rhs - f(x_{k-1}),  x_0 = start,  stop when k - 1 > T or every (x_k - x_{k-1})^2 / (atol + |start| rtol) < 1.
// A CTA owns its tiles for the whole solve (it reads only the iterates it wrote), so the one grid.sync per evaluation
// is for the failing-element counts alone.  They are integers, summed by every CTA in the same way, so every CTA takes
// the same decision.  The counts are double-buffered by the parity of k: a CTA that is already in evaluation k + 1
// writes the other half while a slower one still reads the counts of evaluation k.
// ------------------------------------------------------------------------------------------------------------
// (3 CTAs per SM: without the hint ptxas keeps 40 registers and spills around the mlp_eval calls)
__global__ void __launch_bounds__(kMlpThreads, 3)
k_mlp_fixed_point(MlpDesc net, const float* __restrict__ rhs, const float* __restrict__ start, float* __restrict__ out,
                  float* xa, float* xb, int* __restrict__ counts, impflow_fixed_point_state* state, int B, float atol,
                  float rtol, int T) {
  cg::grid_group grid = cg::this_grid();
  __shared__ __align__(16) float bufA[kTile * kMaxWidth];
  __shared__ __align__(16) float bufB[kTile * kMaxWidth];
  __shared__ int red[kMlpWarps];
  const int d = net.dims[0];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = (B + kTile - 1) / kTile;
  int k = 1;
  for (;; ++k) {
    float* cur = (k & 1) ? xb : xa;                                 // evaluation k writes xa (k even) / xb (k odd)
    const float* prev = k == 1 ? start : ((k & 1) ? xa : xb);       // and reads what evaluation k - 1 wrote
    int fails = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int s0 = tile * kTile;
      const float* f = mlp_eval(net, prev, s0, B, bufA, bufB);
      for (int i = tid; i < kTile * d; i += kMlpThreads) {
        const int s = i / d, c = i % d;
        if (s0 + s >= B) continue;
        const long long idx = (long long)(s0 + s) * d + c;
        // one rounding per operation, as the torch expression of the reference loop
        const float x = __fsub_rn(rhs[idx], f[s * kMaxWidth + c]);
        const float tol = __fadd_rn(atol, __fmul_rn(fabsf(start[idx]), rtol));
        const float dx = __fsub_rn(x, prev[idx]);
        fails += (__fdiv_rn(__fmul_rn(dx, dx), tol) < 1.f) ? 0 : 1;
        cur[idx] = x;
      }
      __syncthreads();      // bufA / bufB are reused by the next tile
    }
    fails = __reduce_add_sync(0xffffffffu, fails);
    if (lane == 0) red[warp] = fails;
    __syncthreads();
    if (tid == 0) {
      int t = 0;
      for (int w = 0; w < kMlpWarps; ++w) t += red[w];
      counts[(k & 1) * gridDim.x + blockIdx.x] = t;
    }
    grid.sync();
    int total = 0;
    for (int i = tid; i < (int)gridDim.x; i += kMlpThreads) total += __ldcg(&counts[(k & 1) * gridDim.x + i]);
    total = __reduce_add_sync(0xffffffffu, total);
    __syncthreads();      // every warp has read red[] above before it is overwritten
    if (lane == 0) red[warp] = total;
    __syncthreads();
    total = 0;
    for (int w = 0; w < kMlpWarps; ++w) total += red[w];
    __syncthreads();      // red[] is reused by the next evaluation
    if (k - 1 > T || total == 0) break;
  }
  // the final iterate of this CTA's tiles into the caller's buffer
  const float* fin = (k & 1) ? xb : xa;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
    for (int i = tid; i < kTile * d; i += kMlpThreads) {
      const long long idx = (long long)tile * kTile * d + i;
      if (idx < (long long)B * d) out[idx] = fin[idx];
    }
  if (blockIdx.x == 0 && tid == 0) {
    state->iterations = k - 1;
    state->active = 0;
    state->fails = 0;
    state->ticket = 0;
  }
}

// ------------------------------------------------------------------------------------------------------------
// Power series of a small-d MLP branch in ONE launch (north-star kernel (c) for the MLP flows): the training path of
// the basic estimator (implicit_block.py:418-426 with create_graph=True) needs, at one saved point and for one probe v,
//     left vectors   l_k = (J^T)^k v, k = 1..n      (vjp chain)          S = sum_k c_k <l_k, v>
//     right vectors  r_m = J^m v,     m = 1..n-1    (tangent chain)
//     combinations   w_m = sum_{a=0}^{n-1-m} c_{a+m} l_a, m = 0..n-1     (left factors of the n bilinear-form gradients)
// Host-driven this is ~60 launches per call (5 GEMMs + 4 multiplier passes per chain step, n row dots, n(n+1)/2 linear
// combinations, 2 concatenations).  Here a CTA takes 16 samples through both chains with the activations in shared
// memory (mlp_eval in its linear-chain mode: no bias, no activation, the saved act' multipliers on the layer outputs).
// ------------------------------------------------------------------------------------------------------------
constexpr int kSeriesMaxTerms = 32;
struct SeriesCoeffs {
  float c[kSeriesMaxTerms];
};

__global__ void __launch_bounds__(kMlpThreads)
k_mlp_series(MlpDesc vjp, MlpDesc tan, SeriesCoeffs co, const float* __restrict__ v, float* Ls, float* Rs,
             float* __restrict__ Wm, float* __restrict__ S, int B, int n) {
  __shared__ __align__(16) float bufA[kTile * kMaxWidth];
  __shared__ __align__(16) float bufB[kTile * kMaxWidth];
  __shared__ float vt[kTile * 128];
  __shared__ float sacc[kTile];
  const int d = vjp.dims[0];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long plane = (long long)B * d;
  // the two chains of a tile are independent: even CTAs take the vjp chain (+ combinations, estimate), odd CTAs the
  // tangent chain, so a batch of 1000 samples (63 tiles) covers 126 SMs instead of 63
  const int chain = blockIdx.x & 1;
  for (int s0 = (blockIdx.x >> 1) * kTile; s0 < B; s0 += (gridDim.x >> 1) * kTile) {
    for (int i = tid; i < kTile * d; i += kMlpThreads) {
      const int s = i / d, c = i % d;
      const float x = (s0 + s < B) ? v[(long long)(s0 + s) * d + c] : 0.f;
      vt[s * 128 + c] = x;
      if (s0 + s < B) {
        if (chain == 0) Ls[(long long)(s0 + s) * d + c] = x;      // l_0 = r_0 = v
        else Rs[(long long)(s0 + s) * d + c] = x;
      }
    }
    if (tid < kTile) sacc[tid] = 0.f;
    __syncthreads();
    if (chain == 1) {
      // ---- tangent chain: r_m = J r_{m-1} ----
      for (int m = 1; m < n; ++m) {
        const float* cur = mlp_eval(tan, Rs + (m - 1) * plane, s0, B, bufA, bufB);
        for (int i = tid; i < kTile * d; i += kMlpThreads) {
          const int s = i / d, c = i % d;
          if (s0 + s < B) Rs[m * plane + (long long)(s0 + s) * d + c] = cur[s * kMaxWidth + c];
        }
        __syncthreads();
      }
      continue;
    }
    // ---- vjp chain: l_k = J^T l_{k-1}, S += c_k <l_k, v> ----
    for (int k = 1; k <= n; ++k) {
      const float* cur = mlp_eval(vjp, Ls + (k - 1) * plane, s0, B, bufA, bufB);
      for (int i = tid; i < kTile * d; i += kMlpThreads) {
        const int s = i / d, c = i % d;
        if (s0 + s < B) Ls[k * plane + (long long)(s0 + s) * d + c] = cur[s * kMaxWidth + c];
      }
      for (int s = warp; s < kTile; s += kMlpWarps) {
        float acc = 0.f;
        for (int c = lane; c < d; c += 32) acc += cur[s * kMaxWidth + c] * vt[s * 128 + c];
        acc = warp_sum(acc);
        if (lane == 0) sacc[s] = fmaf(co.c[k - 1], acc, sacc[s]);
      }
      __syncthreads();      // l_k is in global memory (visible to this block) before the next step reads it
    }
    // ---- w_m = sum_a c_{a+m} l_a (a ascending, as the host loop of linear combinations did) ----
    for (int i = tid; i < n * kTile * d; i += kMlpThreads) {
      const int m = i / (kTile * d), rest = i % (kTile * d);
      const int s = rest / d, c = rest % d;
      if (s0 + s >= B) continue;
      const long long off = (long long)(s0 + s) * d + c;
      float w = co.c[m] * Ls[off];
      for (int a = 1; a < n - m; ++a) w = fmaf(co.c[a + m], Ls[a * plane + off], w);
      Wm[m * plane + off] = w;
    }
    if (tid < kTile && s0 + tid < B) S[s0 + tid] = sacc[tid];
    __syncthreads();
  }
}

}  // namespace impflow

namespace impflow {
int mlp_cooperative_grid(const void* kernel, int B, int* grid);
int launch_mlp_solver(MlpDesc net, const float* x_embed, float* za, float* ga, float* zb, float* gb, float* low_z,
                      float* low_g, float* Ut, float* Vt, float* sample_sq, float* low_sq, double* partial,
                      impflow_broyden_state* state, int B, int threshold, double eps_scaled, void* stream);
}
using namespace impflow;

extern "C" int impflow_mlp_solver_limits(int* max_layers, int* max_width, int* max_d) {
  if (max_layers) *max_layers = kMaxLayers;
  if (max_width) *max_width = kMaxWidth;
  if (max_d) *max_d = 128;
  return 0;
}

extern "C" size_t impflow_mlp_solver_partial_doubles(void) { return 2 * 148 * 8; }

// params: L transposed weight matrices Wt_l [dims[l]][dims[l+1]] and L bias vectors (pointers on the HOST,
// pointing to device memory); biases may be NULL.
extern "C" int impflow_mlp_broyden_solve(const float* x_embed, const float* const* Wt, const float* const* bias,
                                         const int* dims, int L, int act_kind, const float* const* beta_sp, float* za,
                                         float* ga, float* zb, float* gb, float* low_z, float* low_g, float* Ut,
                                         float* Vt, float* sample_sq, float* low_sq, double* partial,
                                         impflow_broyden_state* state, int B, int threshold, double eps_scaled,
                                         void* stream) {
  IMPFLOW_REQUIRE(L >= 1 && L <= kMaxLayers, "mlp_broyden_solve: %d layers not in [1,%d]", L, kMaxLayers);
  IMPFLOW_REQUIRE(threshold >= 1 && threshold <= 63, "mlp_broyden_solve: threshold %d not in [1,63]", threshold);
  IMPFLOW_REQUIRE(dims[0] == dims[L] && dims[0] <= 128, "mlp_broyden_solve: needs d_in == d_out <= 128");
  IMPFLOW_REQUIRE(act_kind != IMPFLOW_ACT_LIPSWISH || beta_sp != nullptr, "mlp_broyden_solve: LipSwish needs beta");
  if (act_kind == IMPFLOW_ACT_LIPSWISH)
    for (int l = 0; l + 1 < L; ++l)
      IMPFLOW_REQUIRE(beta_sp[l] != nullptr, "mlp_broyden_solve: LipSwish behind layer %d has no beta", l);
  MlpDesc net;
  memset(&net, 0, sizeof(net));
  net.L = L;
  for (int l = 0; l <= L; ++l) {
    IMPFLOW_REQUIRE(dims[l] >= 1 && dims[l] <= kMaxWidth, "mlp_broyden_solve: width %d not in [1,%d]", dims[l],
                    kMaxWidth);
    net.dims[l] = dims[l];
  }
  for (int l = 0; l < L; ++l) {
    net.Wt[l] = Wt[l];
    net.bias[l] = bias ? bias[l] : nullptr;
  }
  for (int l = 0; l < L; ++l) net.ld[l] = dims[l + 1];
  net.act_kind = act_kind;
  for (int l = 0; l + 1 < L; ++l) net.beta[l] = beta_sp != nullptr ? beta_sp[l] : nullptr;
  net.mode = 0;
  return launch_mlp_solver(net, x_embed, za, ga, zb, gb, low_z, low_g, Ut, Vt, sample_sq, low_sq, partial, state, B,
                           threshold, eps_scaled, stream);
}

/* Implicit-backward solve of v^T (I + J) = rhs for the same MLP (implicit_block.py:199-207) in the same persistent
 * kernel: f becomes the transposed linear chain v -> (((v W_{L-1}) * D_{L-1}) W_{L-2} * D_{L-2}) ... W_0 with the
 * saved act' multipliers D_l = act'(pre-activation in front of layer l), (B, dims[l]) each.
 *   W[l]   : DEVICE pointer to the effective weight of layer l, [dims[l+1]][ldw[l]] (HOST array of L)
 *   dmul[l]: DEVICE pointer to D_l or NULL (HOST array of L; dmul[0] must be NULL) */
extern "C" int impflow_mlp_broyden_solve_vjp(const float* rhs, const float* const* W, const int* ldw,
                                             const float* const* dmul, const int* dims, int L, float* za, float* ga,
                                             float* zb, float* gb, float* low_z, float* low_g, float* Ut, float* Vt,
                                             float* sample_sq, float* low_sq, double* partial,
                                             impflow_broyden_state* state, int B, int threshold, double eps_scaled,
                                             void* stream) {
  IMPFLOW_REQUIRE(L >= 1 && L <= kMaxLayers, "mlp_broyden_solve_vjp: %d layers not in [1,%d]", L, kMaxLayers);
  IMPFLOW_REQUIRE(threshold >= 1 && threshold <= 63, "mlp_broyden_solve_vjp: threshold %d not in [1,63]", threshold);
  IMPFLOW_REQUIRE(dims[0] == dims[L] && dims[0] <= 128, "mlp_broyden_solve_vjp: needs d_in == d_out <= 128");
  IMPFLOW_REQUIRE(dmul[0] == nullptr, "mlp_broyden_solve_vjp: no activation in front of the first layer");
  MlpDesc net;
  memset(&net, 0, sizeof(net));
  net.L = L;
  for (int l = 0; l <= L; ++l) {
    IMPFLOW_REQUIRE(dims[l] >= 1 && dims[l] <= kMaxWidth, "mlp_broyden_solve_vjp: width %d not in [1,%d]", dims[l],
                    kMaxWidth);
    net.dims[l] = dims[L - l];          // the chain runs from the output side
  }
  for (int j = 0; j < L; ++j) {
    const int l = L - 1 - j;            // forward layer applied transposed at step j: [out][in] is [K][N] here
    IMPFLOW_REQUIRE(ldw[l] >= dims[l], "mlp_broyden_solve_vjp: row stride %d < %d", ldw[l], dims[l]);
    net.Wt[j] = W[l];
    net.ld[j] = ldw[l];
    net.dmul[j] = dmul[l];
  }
  net.act_kind = IMPFLOW_ACT_NONE;
  net.mode = 1;
  return launch_mlp_solver(net, rhs, za, ga, zb, gb, low_z, low_g, Ut, Vt, sample_sq, low_sq, partial, state, B,
                           threshold, eps_scaled, stream);
}

namespace impflow {
int launch_mlp_solver(MlpDesc net, const float* x_embed, float* za, float* ga, float* zb, float* gb, float* low_z,
                      float* low_g, float* Ut, float* Vt, float* sample_sq, float* low_sq, double* partial,
                      impflow_broyden_state* state, int B, int threshold, double eps_scaled, void* stream) {
  int grid = 0;
  if (mlp_cooperative_grid((const void*)k_mlp_broyden, B, &grid)) return -1;
  int T = threshold;
  double eps = eps_scaled;
  void* args[] = {&net, &x_embed, &za, &ga, &zb, &gb, &low_z, &low_g, &Ut, &Vt, &sample_sq, &low_sq,
                  &partial, &state, &B, &T, &eps};
  cudaError_t e = cudaLaunchCooperativeKernel((void*)k_mlp_broyden, dim3(grid), dim3(kMlpThreads), args, 0,
                                              (cudaStream_t)stream);
  if (e != cudaSuccess) {
    set_error("mlp_broyden_solve: cooperative launch failed: %s", cudaGetErrorString(e));
    return -1;
  }
  return check_launch("k_mlp_broyden");
}

// Grid of a persistent cooperative kernel: every CTA resident (up to 8 per SM), no more CTAs than tiles, at most
// 148 * 8 (the size of the per-CTA partial buffers).
int mlp_cooperative_grid(const void* kernel, int B, int* grid) {
  int dev = 0, sms = 0, per_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kMlpThreads, 0) != cudaSuccess || per_sm < 1) {
    set_error("mlp solver: occupancy query failed");
    return -1;
  }
  const int n_tiles = (B + kTile - 1) / kTile;
  int g = sms * (per_sm > 8 ? 8 : per_sm);
  if (g > n_tiles) g = n_tiles;
  if (g > 148 * 8) g = 148 * 8;
  *grid = g;
  return 0;
}
}  // namespace impflow

extern "C" int impflow_mlp_fixed_point(const float* rhs, const float* start, float* out, const float* const* Wt,
                                       const float* const* bias, const int* dims, int L, int act_kind,
                                       const float* const* beta_sp, float* xa, float* xb, int* counts,
                                       impflow_fixed_point_state* state_dev, impflow_fixed_point_state* state_host,
                                       int B, float atol, float rtol, int threshold, void* stream) {
  IMPFLOW_REQUIRE(L >= 1 && L <= kMaxLayers, "mlp_fixed_point: %d layers not in [1,%d]", L, kMaxLayers);
  IMPFLOW_REQUIRE(threshold >= 0 && threshold <= 1000, "mlp_fixed_point: threshold %d not in [0,1000]", threshold);
  IMPFLOW_REQUIRE(dims[0] == dims[L] && dims[0] <= 128, "mlp_fixed_point: needs d_in == d_out <= 128");
  IMPFLOW_REQUIRE(B >= 1, "mlp_fixed_point: empty batch");
  IMPFLOW_REQUIRE(act_kind != IMPFLOW_ACT_LIPSWISH || beta_sp != nullptr, "mlp_fixed_point: LipSwish needs beta");
  if (act_kind == IMPFLOW_ACT_LIPSWISH)
    for (int l = 0; l + 1 < L; ++l)
      IMPFLOW_REQUIRE(beta_sp[l] != nullptr, "mlp_fixed_point: LipSwish behind layer %d has no beta", l);
  MlpDesc net;
  memset(&net, 0, sizeof(net));
  net.L = L;
  for (int l = 0; l <= L; ++l) {
    IMPFLOW_REQUIRE(dims[l] >= 1 && dims[l] <= kMaxWidth, "mlp_fixed_point: width %d not in [1,%d]", dims[l],
                    kMaxWidth);
    net.dims[l] = dims[l];
  }
  for (int l = 0; l < L; ++l) {
    net.Wt[l] = Wt[l];
    net.ld[l] = dims[l + 1];
    net.bias[l] = bias ? bias[l] : nullptr;
  }
  net.act_kind = act_kind;
  for (int l = 0; l + 1 < L; ++l) net.beta[l] = beta_sp != nullptr ? beta_sp[l] : nullptr;
  net.mode = 0;
  int grid = 0;
  if (mlp_cooperative_grid((const void*)k_mlp_fixed_point, B, &grid)) return -1;
  int T = threshold;
  void* args[] = {&net, &rhs, &start, &out, &xa, &xb, &counts, &state_dev, &B, &atol, &rtol, &T};
  cudaStream_t s = (cudaStream_t)stream;
  const cudaError_t e = cudaLaunchCooperativeKernel((void*)k_mlp_fixed_point, dim3(grid), dim3(kMlpThreads), args, 0, s);
  if (e != cudaSuccess) {
    set_error("mlp_fixed_point: cooperative launch failed: %s", cudaGetErrorString(e));
    return -1;
  }
  if (check_launch("k_mlp_fixed_point")) return -1;
  if (cudaMemcpyAsync(state_host, state_dev, sizeof(impflow_fixed_point_state), cudaMemcpyDeviceToHost, s) !=
          cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess) {
    set_error("mlp_fixed_point: state read-back failed: %s", cudaGetErrorString(cudaGetLastError()));
    return -1;
  }
  return 0;
}

/* One-launch power series of a small-d MLP branch at a saved point (see k_mlp_series):
 *   W[l], ldw[l] : effective weight of layer l, [dims[l+1]][ldw[l]] row-major (vjp chain, as in ..._solve_vjp)
 *   Wt[l]        : its transpose [dims[l]][dims[l+1]] contiguous (tangent chain, as in impflow_mlp_broyden_solve)
 *   dmul[l]      : act'(pre-activation in front of layer l), (B, dims[l]); dmul[0] must be NULL
 *   v            : probe (B, d); coeffs: n HOST doubles c_1..c_n
 *   Ls (n+1, B, d): l_0 = v, l_k = (J^T)^k v;  Rs (n, B, d): r_0 = v, r_m = J^m v;  Wm (n, B, d): w_m;  S (B) */
extern "C" int impflow_mlp_series(const float* v, const float* const* W, const int* ldw, const float* const* Wt,
                                  const float* const* dmul, const int* dims, int L, int B, int n, const double* coeffs,
                                  float* Ls, float* Rs, float* Wm, float* S, void* stream) {
  IMPFLOW_REQUIRE(L >= 1 && L <= kMaxLayers, "mlp_series: %d layers not in [1,%d]", L, kMaxLayers);
  IMPFLOW_REQUIRE(n >= 1 && n <= kSeriesMaxTerms, "mlp_series: %d terms not in [1,%d]", n, kSeriesMaxTerms);
  IMPFLOW_REQUIRE(dims[0] == dims[L] && dims[0] <= 128, "mlp_series: needs d_in == d_out <= 128");
  IMPFLOW_REQUIRE(dmul[0] == nullptr, "mlp_series: no activation in front of the first layer");
  IMPFLOW_REQUIRE(B >= 1, "mlp_series: empty batch");
  MlpDesc vjp, tan;
  memset(&vjp, 0, sizeof(vjp));
  memset(&tan, 0, sizeof(tan));
  vjp.L = tan.L = L;
  for (int l = 0; l <= L; ++l) {
    IMPFLOW_REQUIRE(dims[l] >= 1 && dims[l] <= kMaxWidth, "mlp_series: width %d not in [1,%d]", dims[l], kMaxWidth);
    vjp.dims[l] = dims[L - l];          // the vjp chain runs from the output side
    tan.dims[l] = dims[l];
  }
  for (int j = 0; j < L; ++j) {
    const int l = L - 1 - j;
    IMPFLOW_REQUIRE(ldw[l] >= dims[l], "mlp_series: row stride %d < %d", ldw[l], dims[l]);
    vjp.Wt[j] = W[l];
    vjp.ld[j] = ldw[l];
    vjp.dmul[j] = dmul[l];
    tan.Wt[j] = Wt[j];
    tan.ld[j] = dims[j + 1];
    tan.dmul[j] = (j + 1 < L) ? dmul[j + 1] : nullptr;
  }
  vjp.act_kind = tan.act_kind = IMPFLOW_ACT_NONE;
  vjp.mode = tan.mode = 1;
  SeriesCoeffs co;
  memset(&co, 0, sizeof(co));
  for (int k = 0; k < n; ++k) co.c[k] = (float)coeffs[k];
  const int n_tiles = (B + kTile - 1) / kTile;
  const int grid = 2 * (n_tiles < 148 * 2 ? n_tiles : 148 * 2);      // (vjp CTA, tangent CTA) per tile
  k_mlp_series<<<grid, kMlpThreads, 0, (cudaStream_t)stream>>>(vjp, tan, co, v, Ls, Rs, Wm, S, B, n);
  return check_launch("k_mlp_series");
}
