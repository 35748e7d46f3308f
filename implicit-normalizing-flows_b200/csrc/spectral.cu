// Induced 2-norm power iteration for a dense (out,in) matrix, entirely on the device:
// replaces the host loop of mixed_lipschitz.py:85-123 (InducedNormLinear.compute_weight) and
// :276-319 (InducedNormConv2d._compute_weight_1x1) with its per-iteration tolerance test
// (:114-120, including the signed max(u) quirk).  One CTA; u, v live in shared memory.
#include "common.cuh"

namespace impflow {

constexpr int kSnThreads = 1024;
constexpr int kSnWarps = kSnThreads / 32;

__device__ float block_sum(float v, float* scratch) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  for (int w = 0; w < kSnWarps; ++w) t += scratch[w];
  return t;
}
__device__ float block_max(float v, float* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = scratch[0];
  for (int w = 1; w < kSnWarps; ++w) t = fmaxf(t, scratch[w]);
  return t;
}

// y[r] = sum_c W[r,c] x[c]   (warp per row, coalesced)
__device__ void mat_vec(const float* __restrict__ W, const float* x, float* y, int out_f, int in_f) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < out_f; r += kSnWarps) {
    float acc = 0.f;
    for (int c = lane; c < in_f; c += 32) acc += W[(long long)r * in_f + c] * x[c];
    acc = warp_sum(acc);
    if (lane == 0) y[r] = acc;
  }
  __syncthreads();
}
// y[c] = sum_r W[r,c] x[r].  Rows are dealt round-robin to the warps (one coalesced row segment per load, 32
// independent rows in flight per CTA instead of one dependent chain per column); the per-warp partial sums are
// combined in warp order through `part` ([kSnWarps][in_f] floats of shared memory): deterministic.
__device__ void mat_t_vec(const float* __restrict__ W, const float* x, float* y, int out_f, int in_f, float* part) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (part == nullptr) {            // no room for the partials: one thread per column
    for (int c = threadIdx.x; c < in_f; c += kSnThreads) {
      float acc = 0.f;
      for (int r = 0; r < out_f; ++r) acc += W[(long long)r * in_f + c] * x[r];
      y[c] = acc;
    }
    __syncthreads();
    return;
  }
  for (int c0 = 0; c0 < in_f; c0 += 32 * 8) {          // 8 columns per lane and pass
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int r = warp; r < out_f; r += kSnWarps) {
      const float xr = x[r];
      const float* row = W + (long long)r * in_f + c0 + lane;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (c0 + lane + 32 * j < in_f) acc[j] = fmaf(row[32 * j], xr, acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (c0 + lane + 32 * j < in_f) part[warp * in_f + c0 + lane + 32 * j] = acc[j];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < in_f; c += kSnThreads) {
    float t = 0.f;
#pragma unroll 8
    for (int w = 0; w < kSnWarps; ++w) t += part[w * in_f + c];
    y[c] = t;
  }
  __syncthreads();
}
// F.normalize(p=2, dim=0, eps=1e-12)
__device__ void l2_normalize(float* y, int n, float* scratch) {
  float ss = 0.f;
  for (int i = threadIdx.x; i < n; i += kSnThreads) ss += y[i] * y[i];
  const float nrm = fmaxf(sqrtf(block_sum(ss, scratch)), 1e-12f);
  for (int i = threadIdx.x; i < n; i += kSnThreads) y[i] = y[i] / nrm;
  __syncthreads();
}

// one CTA: the whole power iteration of one dense layer (body shared by the single-layer and the batched kernel)
__device__ void sn_power_iter_body(const float* __restrict__ W, float* __restrict__ u_g, float* __restrict__ v_g,
                                   float* __restrict__ sigma, int* __restrict__ iters, int out_f, int in_f,
                                   int n_iterations, float atol, float rtol, int with_partials, float* sm) {
  float* u = sm;
  float* v = u + out_f;
  float* ou = v + in_f;
  float* ov = ou + out_f;
  float* part = with_partials ? ov + in_f : nullptr;     // [kSnWarps][in_f]
  __shared__ float scratch[kSnWarps];
  for (int i = threadIdx.x; i < out_f; i += kSnThreads) u[i] = u_g[i];
  for (int i = threadIdx.x; i < in_f; i += kSnThreads) v[i] = v_g[i];
  __syncthreads();
  const bool tol_mode = n_iterations < 0;
  const int max_it = tol_mode ? 200 : n_iterations;
  int used = 0;
  for (int it = 0; it < max_it; ++it) {
    for (int i = threadIdx.x; i < out_f; i += kSnThreads) ou[i] = u[i];
    for (int i = threadIdx.x; i < in_f; i += kSnThreads) ov[i] = v[i];
    __syncthreads();
    mat_vec(W, v, u, out_f, in_f);
    l2_normalize(u, out_f, scratch);
    mat_t_vec(W, u, v, out_f, in_f, part);
    l2_normalize(v, in_f, scratch);
    ++used;
    if (tol_mode) {
      float du = 0.f, dv = 0.f, mu = -INFINITY, mv = -INFINITY;
      for (int i = threadIdx.x; i < out_f; i += kSnThreads) {
        const float t = u[i] - ou[i];
        du += t * t;
        mu = fmaxf(mu, u[i]);
      }
      for (int i = threadIdx.x; i < in_f; i += kSnThreads) {
        const float t = v[i] - ov[i];
        dv += t * t;
        mv = fmaxf(mv, v[i]);
      }
      const float err_u = sqrtf(block_sum(du, scratch)) / sqrtf((float)out_f);
      const float err_v = sqrtf(block_sum(dv, scratch)) / sqrtf((float)in_f);
      const float tol_u = atol + rtol * block_max(mu, scratch);
      const float tol_v = atol + rtol * block_max(mv, scratch);
      if (err_u < tol_u && err_v < tol_v) break;  // uniform: all threads hold the same totals
    }
  }
  // sigma = u^T W v (mixed_lipschitz.py:125)
  mat_vec(W, v, ou, out_f, in_f);
  float s = 0.f;
  for (int i = threadIdx.x; i < out_f; i += kSnThreads) s += u[i] * ou[i];
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) {
    sigma[0] = s;
    if (iters) iters[0] = used;
  }
  if (used > 0) {
    for (int i = threadIdx.x; i < out_f; i += kSnThreads) u_g[i] = u[i];
    for (int i = threadIdx.x; i < in_f; i += kSnThreads) v_g[i] = v[i];
  }
}

__global__ void __launch_bounds__(kSnThreads)
k_sn_power_iter(const float* __restrict__ W, float* __restrict__ u_g, float* __restrict__ v_g,
                float* __restrict__ sigma, int* __restrict__ iters, int out_f, int in_f, int n_iterations,
                float atol, float rtol, int with_partials) {
  extern __shared__ float sm[];
  sn_power_iter_body(W, u_g, v_g, sigma, iters, out_f, in_f, n_iterations, atol, rtol, with_partials, sm);
}

// All dense layers of a model in ONE launch, one CTA per layer (the refresh after every optimiser step touches every
// layer; the layers are independent): update_lipschitz issued one launch per layer (100+ for a tabular flow).
__global__ void __launch_bounds__(kSnThreads)
k_sn_power_iter_batch(const impflow_sn_desc* __restrict__ descs, int n_iterations, float atol, float rtol,
                      int smem_floats) {
  extern __shared__ float sm[];
  const impflow_sn_desc d = descs[blockIdx.x];
  // the single-layer launch's rule (200 KB with the per-warp partials, else without); the host sized the shared
  // memory as min(200 KB, need of the widest layer), so a layer that passes this test fits
  const long long need = 2LL * (d.out_f + d.in_f) + (long long)kSnWarps * d.in_f;
  sn_power_iter_body(d.W, d.u, d.v, d.sigma, d.iters, d.out_f, d.in_f, n_iterations, atol, rtol,
                     (need * 4 <= 200 * 1024 && need <= smem_floats) ? 1 : 0, sm);
}

// W / max(1, sigma/coeff) with sigma read from the device (mixed_lipschitz.py:128-131), and its
// gradient chain  dL/dW = s*G + <G,W> * ds/dsigma * D,  D = dsigma/dW (sigma = <W, D> is linear in W).
__global__ void __launch_bounds__(256)
k_sn_scale(const float* __restrict__ W, const float* __restrict__ sigma, float coeff, float* __restrict__ out,
           float* __restrict__ scale_out, long long n) {
  const float sg = __ldg(sigma);
  const float factor = fmaxf(1.f, sg / coeff);
  if (blockIdx.x == 0 && threadIdx.x == 0 && scale_out != nullptr) scale_out[0] = sg;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    out[i] = W[i] / factor;
}
__global__ void __launch_bounds__(256)
k_sn_scale_grad(const float* __restrict__ G, const float* __restrict__ D, const float* __restrict__ sigma,
                const float* __restrict__ gw_dot, float coeff, float* __restrict__ out, long long n) {
  const float sg = __ldg(sigma);
  const float ratio = sg / coeff;
  const float s = ratio > 1.f ? 1.f / ratio : 1.f;
  const float ds = ratio > 1.f ? -coeff / (sg * sg) : 0.f;
  const float c2 = ds * __ldg(gw_dot);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    out[i] = s * G[i] + c2 * D[i];
}

// ---- gradient of the effective weight, straight from the GEMM-layout weight gradient --------------------------
// The weight-gradient GEMMs produce dL/dW_eff in the layout the forward GEMM consumes (k_prep_weights, fwd side);
// the chain through the soft rescale needs t = <G, W> first.  Two launches (partial dots, then the combination)
// read the GEMM layout through the index map below instead of materialising flip / permute / contiguous copies.
__device__ __forceinline__ long long wbar_index(int kind, int cout, int cin, long long ldw, long long i) {
  if (kind == 0) return (i / cin) * ldw + (i % cin);
  const int co = (int)(i / (cin * 9)), r = (int)(i % (cin * 9)), ci = r / 9, t = r % 9;
  if (kind == 1) return (long long)co * ldw + t * cin + ci;          // fwd[co][(ky,kx,ci)]
  return ((long long)(8 - t) * cout + co) * ldw + ci;                // fwd[(2-ky,2-kx,co)][ci]
}
__global__ void __launch_bounds__(256)
k_sn_grad_dot(const float* __restrict__ Wbar, long long ldw, const float* __restrict__ W, int kind, int cout, int cin,
              long long n, float* __restrict__ partial) {
  float acc = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    acc = fmaf(Wbar[wbar_index(kind, cout, cin, ldw, i)], W[i], acc);
  __shared__ float red[256];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = red[0];
}
__global__ void __launch_bounds__(256)
k_sn_scale_grad_layout(const float* __restrict__ Wbar, long long ldw, const float* __restrict__ D,
                       const float* __restrict__ sigma, const float* __restrict__ partial, int n_partial, float coeff,
                       int kind, int cout, int cin, long long n, float* __restrict__ out) {
  __shared__ float red[256];
  float acc = 0.f;
  for (int j = threadIdx.x; j < n_partial; j += 256) acc += partial[j];     // same order in every block
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  const float sg = __ldg(sigma);
  const float ratio = sg / coeff;
  const float sc = ratio > 1.f ? 1.f / ratio : 1.f;
  const float c2 = (ratio > 1.f ? -coeff / (sg * sg) : 0.f) * red[0];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = sc * Wbar[wbar_index(kind, cout, cin, ldw, i)] + c2 * D[i];
}

// Effective weight of one layer in every layout the branch kernels consume, in ONE launch: the soft spectral
// rescale W / max(1, sigma/coeff) (mixed_lipschitz.py:128-131), the GEMM re-layouts of both directions
// (K zero-padded) and their tf32 hi/lo planes.  Replaces ~12 permute / pad / split launches per layer and step.
//   kind 0 (linear, 1x1):            fwd[co][ci]                   bwd[ci][co]
//   kind 1 (3x3, cin <= cout):       fwd[co][(ky,kx,ci)]           bwd[(ky,kx,ci)][co]
//   kind 2 (3x3, cin >  cout):       fwd[(ky',kx',co)][ci]         bwd[ci][(ky',kx',co)]     taps flipped: ky' = 2-ky
// The divisor comes from `fac` by group mode (kGroup): kPrepSigma, the induced-norm layers' W / max(1, sigma/coeff);
// or a closed-form operator norm (LopLinear / LopConv2d, lipschitz.py:72-79) with ratio n * (1/coeff) as torch forms
// it: one norm for the whole layer (kPrepLopOne), per output row (kPrepLopRow) or per input channel (kPrepLopCol).
struct PrepOut {
  float* f32;
  float* hi;   // may be null (CUDA-core path: no planes)
  float* lo;
  int N, Kp;   // rows, padded row length
};
constexpr int kPrepSigma = -1, kPrepLopOne = 0, kPrepLopRow = 1, kPrepLopCol = 2;
template <int kGroup>
__global__ void __launch_bounds__(256)
k_prep_weights(const float* __restrict__ W, const float* __restrict__ fac, float coeff, int kind, int cout,
               int cin, PrepOut fwd, PrepOut bwd) {
  const float rcoeff = 1.f / coeff;
  float factor = 1.f;
  if (kGroup == kPrepSigma) factor = fmaxf(1.f, __ldg(fac) / coeff);
  if (kGroup == kPrepLopOne) factor = fmaxf(1.f, __ldg(fac) * rcoeff);
  const int nf = fwd.N * fwd.Kp, nb = bwd.N * bwd.Kp;
  const int taps = kind == 0 ? 1 : 9;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nf + nb; i += gridDim.x * blockDim.x) {
    const bool is_fwd = i < nf;
    const PrepOut& o = is_fwd ? fwd : bwd;
    const int j = is_fwd ? i : i - nf;
    const int r = j / o.Kp, k = j - r * o.Kp;
    int co = -1, ci = 0, tap = 0;       // source element W[co][ci][tap]; co = -1: zero padding
    if (kind == 0) {
      if (is_fwd) { if (k < cin) co = r, ci = k; } else { if (k < cout) co = k, ci = r; }
    } else if (kind == 1) {
      if (is_fwd) { if (k < 9 * cin) co = r, tap = k / cin, ci = k - tap * cin; }
      else { if (k < cout) co = k, tap = r / cin, ci = r - tap * cin; }
    } else {
      if (is_fwd) { if (k < cin) { const int t = r / cout; co = r - t * cout, ci = k, tap = 8 - t; } }
      else { if (k < 9 * cout) { const int t = k / cout; co = k - t * cout, ci = r, tap = 8 - t; } }
    }
    float f = factor;
    if (kGroup == kPrepLopRow && co >= 0) f = fmaxf(1.f, __ldg(fac + co) * rcoeff);
    if (kGroup == kPrepLopCol && co >= 0) f = fmaxf(1.f, __ldg(fac + ci) * rcoeff);
    const float v = co >= 0 ? W[((long long)co * cin + ci) * taps + tap] / f : 0.f;
    o.f32[j] = v;
    if (o.hi != nullptr) {
      uint32_t hb;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(v));
      o.hi[j] = __uint_as_float(hb);
      o.lo[j] = v - __uint_as_float(hb);
    }
  }
}


// ---- closed-form operator norms (LopLinear / LopConv2d) -------------------------------------------------------------
// Group k of a [cout][cin][taps] weight is output row k (axis 0) or input channel k (axis 1).  Norm type 1: sum |w|,
// 2: sqrt(sum w^2), 3: the SIGNED maximum (the reference's _max_except_dim, lipschitz.py:51).  One warp per group, a
// fixed lane order and a butterfly: deterministic, no atomics.
constexpr int kLopGroupsPerCta = 8;
__device__ __forceinline__ long long lop_elem(int axis, int cin, int taps, int k, int j) {
  if (axis == 0) return (long long)k * cin * taps + j;
  const int co = j / taps, t = j - co * taps;
  return ((long long)co * cin + k) * taps + t;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__global__ void __launch_bounds__(32 * kLopGroupsPerCta)
k_lop_norms(const float* __restrict__ W, int cout, int cin, int taps, int axis, int norm_type,
            float* __restrict__ norms) {
  const int k = blockIdx.x * kLopGroupsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int groups = axis == 0 ? cout : cin, len = (axis == 0 ? cin : cout) * taps;
  if (k >= groups) return;
  float acc = norm_type == 3 ? -INFINITY : 0.f;
  for (int j = lane; j < len; j += 32) {
    const float w = __ldg(W + lop_elem(axis, cin, taps, k, j));
    acc = norm_type == 3 ? fmaxf(acc, w) : (norm_type == 1 ? acc + fabsf(w) : fmaf(w, w, acc));
  }
  acc = norm_type == 3 ? warp_max(acc) : warp_sum(acc);
  if (lane == 0) norms[k] = norm_type == 2 ? sqrtf(acc) : acc;
}
// norms[groups] = the largest group norm (the global constraint's norm and the `scale` buffer, lipschitz.py:74-77)
__global__ void __launch_bounds__(1024)
k_lop_norm_max(float* __restrict__ norms, int groups, float* __restrict__ scale_out) {
  __shared__ float scratch[32];
  float m = -INFINITY;
  for (int k = threadIdx.x; k < groups; k += 1024) m = fmaxf(m, norms[k]);
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = scratch[0];
    for (int w = 1; w < 32; ++w) t = fmaxf(t, scratch[w]);
    norms[groups] = t;
    if (scale_out != nullptr) scale_out[0] = t;
  }
}

// Gradient chain of W / f_k, f_k = max(1, n_k/coeff), from the GEMM-layout gradient (read through wbar_index):
//   dL/dW = Gbar/f_k - c_k t_k / (coeff f_k^2) dn_k/dW,   t_k = sum_{group k} Gbar W,
// c_k = 1 above the bound, 1/2 exactly at it (torch.max's even split), 0 below.  Phase 1: t_k and, for the signed
// maximum, the number of entries equal to n_k (amax's backward splits evenly among them), one warp per group.
__global__ void __launch_bounds__(32 * kLopGroupsPerCta)
k_lop_grad_dot(const float* __restrict__ Wbar, long long ldw, const float* __restrict__ W,
               const float* __restrict__ norms, int kind, int cout, int cin, int axis, float* __restrict__ ws) {
  const int taps = kind == 0 ? 1 : 9;
  const int k = blockIdx.x * kLopGroupsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int groups = axis == 0 ? cout : cin, len = (axis == 0 ? cin : cout) * taps;
  if (k >= groups) return;
  const float nk = norms[k];
  float t = 0.f, ties = 0.f;
  for (int j = lane; j < len; j += 32) {
    const long long i = lop_elem(axis, cin, taps, k, j);
    const float w = __ldg(W + i);
    t = fmaf(Wbar[wbar_index(kind, cout, cin, ldw, i)], w, t);
    ties += w == nk ? 1.f : 0.f;
  }
  t = warp_sum(t);
  ties = warp_sum(ties);
  if (lane == 0) {
    ws[k] = t;
    ws[groups + k] = ties;
  }
}
// Phase 2, elementwise.  local = 0: one factor from the largest norm N = norms[groups]; t = sum_k t_k and the
// derivative of N is split evenly among the groups whose norm equals N (every block sums the same values in the
// same order).
__global__ void __launch_bounds__(256)
k_lop_scale_grad_layout(const float* __restrict__ Wbar, long long ldw, const float* __restrict__ W,
                        const float* __restrict__ norms, const float* __restrict__ ws, float coeff, int kind,
                        int cout, int cin, int axis, int norm_type, int local, float* __restrict__ out) {
  const int taps = kind == 0 ? 1 : 9;
  const int groups = axis == 0 ? cout : cin;
  const float rcoeff = 1.f / coeff;
  __shared__ float red[2][256];
  float t_all = 0.f, n_tied = 0.f;
  if (!local) {
    const float N = norms[groups];
    float a = 0.f, b = 0.f;
    for (int k = threadIdx.x; k < groups; k += 256) {
      a += ws[k];
      b += norms[k] == N ? 1.f : 0.f;
    }
    red[0][threadIdx.x] = a;
    red[1][threadIdx.x] = b;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
      if (threadIdx.x < s) {
        red[0][threadIdx.x] += red[0][threadIdx.x + s];
        red[1][threadIdx.x] += red[1][threadIdx.x + s];
      }
      __syncthreads();
    }
    t_all = red[0][0];
    n_tied = red[1][0];
  }
  const long long n = (long long)cout * cin * taps;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i / ((long long)cin * taps)), ci = (int)((i / taps) % cin);
    const int k = axis == 0 ? co : ci;
    const float nk = norms[k], N = local ? nk : norms[groups];
    const float ratio = N * rcoeff;
    const float f = fmaxf(1.f, ratio);
    const float g = Wbar[wbar_index(kind, cout, cin, ldw, i)];
    float r = g / f;
    const float c = ratio > 1.f ? 1.f : (ratio == 1.f ? 0.5f : 0.f);
    if (c != 0.f && nk == N) {
      const float w = W[i];
      float dn = norm_type == 1 ? (w > 0.f ? 1.f : (w < 0.f ? -1.f : 0.f))
                                : (norm_type == 2 ? w / nk : (w == nk ? 1.f / ws[groups + k] : 0.f));
      if (!local) dn /= n_tied;
      const float t = local ? ws[k] : t_all;
      r -= c * t / (coeff * f * f) * dn;
    }
    out[i] = r;
  }
}
}  // namespace impflow

using namespace impflow;

extern "C" int impflow_prep_weights(const float* W, const float* sigma, float coeff, int kind, int cout, int cin,
                                    float* fwd, float* fwd_hi, float* fwd_lo, int fwd_rows, int fwd_k, float* bwd,
                                    float* bwd_hi, float* bwd_lo, int bwd_rows, int bwd_k, void* stream) {
  IMPFLOW_REQUIRE(kind >= 0 && kind <= 2 && cout >= 1 && cin >= 1, "prep_weights: bad layer (kind=%d)", kind);
  IMPFLOW_REQUIRE(fwd != nullptr && bwd != nullptr, "prep_weights: outputs missing");
  IMPFLOW_REQUIRE((fwd_hi == nullptr) == (fwd_lo == nullptr) && (bwd_hi == nullptr) == (bwd_lo == nullptr),
                  "prep_weights: planes come in pairs");
  const long long total = (long long)fwd_rows * fwd_k + (long long)bwd_rows * bwd_k;
  IMPFLOW_REQUIRE(total < (1LL << 31), "prep_weights: layer too large");
  PrepOut f{fwd, fwd_hi, fwd_lo, fwd_rows, fwd_k}, b{bwd, bwd_hi, bwd_lo, bwd_rows, bwd_k};
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  k_prep_weights<kPrepSigma><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(W, sigma, coeff, kind, cout, cin, f, b);
  return check_launch("k_prep_weights");
}

extern "C" int impflow_prep_weights_lop(const float* W, const float* norms, int group, float coeff, int kind,
                                        int cout, int cin, float* fwd, float* fwd_hi, float* fwd_lo, int fwd_rows,
                                        int fwd_k, float* bwd, float* bwd_hi, float* bwd_lo, int bwd_rows, int bwd_k,
                                        void* stream) {
  IMPFLOW_REQUIRE(kind >= 0 && kind <= 2 && cout >= 1 && cin >= 1, "prep_weights_lop: bad layer (kind=%d)", kind);
  IMPFLOW_REQUIRE(group >= 0 && group <= 2, "prep_weights_lop: bad group mode %d", group);
  IMPFLOW_REQUIRE(norms != nullptr && fwd != nullptr && bwd != nullptr, "prep_weights_lop: operands missing");
  IMPFLOW_REQUIRE((fwd_hi == nullptr) == (fwd_lo == nullptr) && (bwd_hi == nullptr) == (bwd_lo == nullptr),
                  "prep_weights_lop: planes come in pairs");
  const long long total = (long long)fwd_rows * fwd_k + (long long)bwd_rows * bwd_k;
  IMPFLOW_REQUIRE(total < (1LL << 31), "prep_weights_lop: layer too large");
  PrepOut f{fwd, fwd_hi, fwd_lo, fwd_rows, fwd_k}, b{bwd, bwd_hi, bwd_lo, bwd_rows, bwd_k};
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  cudaStream_t s = (cudaStream_t)stream;
  if (group == kPrepLopOne)
    k_prep_weights<kPrepLopOne><<<(int)blocks, 256, 0, s>>>(W, norms, coeff, kind, cout, cin, f, b);
  else if (group == kPrepLopRow)
    k_prep_weights<kPrepLopRow><<<(int)blocks, 256, 0, s>>>(W, norms, coeff, kind, cout, cin, f, b);
  else
    k_prep_weights<kPrepLopCol><<<(int)blocks, 256, 0, s>>>(W, norms, coeff, kind, cout, cin, f, b);
  return check_launch("k_prep_weights");
}

extern "C" int impflow_lop_norms(const float* W, int cout, int cin, int taps, int axis, int norm_type, float* norms,
                                 float* scale_out, void* stream) {
  IMPFLOW_REQUIRE(W != nullptr && norms != nullptr && cout >= 1 && cin >= 1 && taps >= 1, "lop_norms: bad layer");
  IMPFLOW_REQUIRE((axis == 0 || axis == 1) && norm_type >= 1 && norm_type <= 3,
                  "lop_norms: axis %d / norm type %d", axis, norm_type);
  const int groups = axis == 0 ? cout : cin;
  k_lop_norms<<<(groups + kLopGroupsPerCta - 1) / kLopGroupsPerCta, 32 * kLopGroupsPerCta, 0, (cudaStream_t)stream>>>(
      W, cout, cin, taps, axis, norm_type, norms);
  if (check_launch("k_lop_norms")) return -1;
  k_lop_norm_max<<<1, 1024, 0, (cudaStream_t)stream>>>(norms, groups, scale_out);
  return check_launch("k_lop_norm_max");
}

extern "C" int impflow_lop_scale_grad_layout(const float* Wbar, long long ldw, const float* W, const float* norms,
                                             float coeff, int kind, int cout, int cin, int axis, int norm_type,
                                             int local, float* out, float* ws, void* stream) {
  IMPFLOW_REQUIRE(kind >= 0 && kind <= 2 && cout >= 1 && cin >= 1, "lop_scale_grad_layout: bad layer description");
  IMPFLOW_REQUIRE((axis == 0 || axis == 1) && norm_type >= 1 && norm_type <= 3,
                  "lop_scale_grad_layout: axis %d / norm type %d", axis, norm_type);
  IMPFLOW_REQUIRE(ws != nullptr && norms != nullptr, "lop_scale_grad_layout: workspace or norms missing");
  const int groups = axis == 0 ? cout : cin;
  cudaStream_t s = (cudaStream_t)stream;
  k_lop_grad_dot<<<(groups + kLopGroupsPerCta - 1) / kLopGroupsPerCta, 32 * kLopGroupsPerCta, 0, s>>>(
      Wbar, ldw, W, norms, kind, cout, cin, axis, ws);
  if (check_launch("k_lop_grad_dot")) return -1;
  const long long n = (long long)cout * cin * (kind == 0 ? 1 : 9);
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  k_lop_scale_grad_layout<<<(int)blocks, 256, 0, s>>>(Wbar, ldw, W, norms, ws, coeff, kind, cout, cin, axis, norm_type,
                                                     local, out);
  return check_launch("k_lop_scale_grad_layout");
}

extern "C" int impflow_sn_scale(const float* W, const float* sigma, float coeff, float* out, float* scale_out,
                                long long n, void* stream) {
  if (n <= 0) return 0;
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  k_sn_scale<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(W, sigma, coeff, out, scale_out, n);
  return check_launch("k_sn_scale");
}

extern "C" int impflow_sn_scale_grad(const float* G, const float* D, const float* sigma, const float* gw_dot,
                                     float coeff, float* out, long long n, void* stream) {
  if (n <= 0) return 0;
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  k_sn_scale_grad<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(G, D, sigma, gw_dot, coeff, out, n);
  return check_launch("k_sn_scale_grad");
}

extern "C" int impflow_sn_scale_grad_layout(const float* Wbar, long long ldw, const float* W, const float* D,
                                            const float* sigma, float coeff, int kind, int cout, int cin, float* out,
                                            float* ws, void* stream) {
  IMPFLOW_REQUIRE(kind >= 0 && kind <= 2 && cout >= 1 && cin >= 1, "sn_scale_grad_layout: bad layer description");
  IMPFLOW_REQUIRE(ws != nullptr, "sn_scale_grad_layout: workspace of 1024 floats missing");
  const long long n = (long long)cout * cin * (kind == 0 ? 1 : 9);
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  k_sn_grad_dot<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(Wbar, ldw, W, kind, cout, cin, n, ws);
  if (check_launch("k_sn_grad_dot")) return -1;
  k_sn_scale_grad_layout<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(Wbar, ldw, D, sigma, ws, (int)blocks, coeff, kind,
                                                                        cout, cin, n, out);
  return check_launch("k_sn_scale_grad_layout");
}

extern "C" int impflow_sn_power_iter(const float* W, float* u, float* v, float* sigma, int* iters, int out_f,
                                     int in_f, int n_iterations, float atol, float rtol, void* stream) {
  IMPFLOW_REQUIRE(out_f >= 1 && in_f >= 1, "sn_power_iter: empty matrix");
  size_t smem = sizeof(float) * 2 * ((size_t)out_f + in_f);
  IMPFLOW_REQUIRE(smem <= 200 * 1024, "sn_power_iter: out+in=%d too large for one CTA", out_f + in_f);
  const size_t with_part = smem + sizeof(float) * (size_t)kSnWarps * in_f;
  const int with_partials = with_part <= 200 * 1024 ? 1 : 0;
  if (with_partials) smem = with_part;
  if (smem > 48 * 1024) {
    if (cudaFuncSetAttribute(k_sn_power_iter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
        cudaSuccess) {
      set_error("sn_power_iter: cannot set dynamic shared memory");
      return -1;
    }
  }
  k_sn_power_iter<<<1, kSnThreads, smem, (cudaStream_t)stream>>>(W, u, v, sigma, iters, out_f, in_f,
                                                                  n_iterations, atol, rtol, with_partials);
  return check_launch("k_sn_power_iter");
}

extern "C" int impflow_sn_power_iter_batch(const impflow_sn_desc* descs_dev, int n, int max_out, int max_in,
                                           int n_iterations, float atol, float rtol, void* stream) {
  IMPFLOW_REQUIRE(n >= 1 && descs_dev != nullptr, "sn_power_iter_batch: no layers");
  IMPFLOW_REQUIRE(max_out >= 1 && max_in >= 1, "sn_power_iter_batch: empty matrix");
  size_t smem = sizeof(float) * 2 * ((size_t)max_out + max_in);
  IMPFLOW_REQUIRE(smem <= 200 * 1024, "sn_power_iter_batch: out+in=%d too large for one CTA", max_out + max_in);
  const size_t with_part = smem + sizeof(float) * (size_t)kSnWarps * max_in;
  smem = with_part <= 200 * 1024 ? with_part : 200 * 1024;      // narrow layers of a mixed batch keep their partials
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(k_sn_power_iter_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
          cudaSuccess) {
    set_error("sn_power_iter_batch: cannot set dynamic shared memory");
    return -1;
  }
  k_sn_power_iter_batch<<<n, kSnThreads, smem, (cudaStream_t)stream>>>(descs_dev, n_iterations, atol, rtol,
                                                                       (int)(smem / sizeof(float)));
  return check_launch("k_sn_power_iter_batch");
}
