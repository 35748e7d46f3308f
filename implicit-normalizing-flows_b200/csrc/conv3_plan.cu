// Native host runtime for the 3x3 / 1x1 / 3x3 conv residual branch of the image flows
// (implicit_flow.py:359-398): one C call per branch evaluation, per power-series chain and per Broyden
// solve, instead of a Python-driven sequence of kernel launches.
//
//   impflow_conv3_forward        nnet(x)                           (implicit_block.py:68-80)
//   impflow_conv3_prepare_vjp    D_l = act'(pre_l), once per saved forward
//   impflow_conv3_vjp            v^T J                             (:199-203, :432-435)
//   impflow_conv3_power_series   w = v + sum_k coeff_k v^T J^k     (Neumann chain, :431-435)
//   impflow_conv3_broyden        whole forward / implicit-backward root solve: branch evaluations, the
//                                residual, the solver algebra and the per-iteration state read-back
//                                (broyden.py:123-193 + implicit_block.py:68-80, 199-207)
//   impflow_conv3_fixed_point    whole Banach iteration x <- rhs - nnet(x) with its stopping test
//                                (iresblock.py:69-79, implicit_block.py:17-28)
//
// Everything works on NHWC "rows" (M = B*H*W rows of c floats): a sample is a contiguous block of
// d = H*W*c floats, which is all the solver's per-sample dot products need.  Shapes with 9c <= 32 and
// C % 256 == 0 take the one-launch tile kernel (branch_fused.cu); the others run im2col-planes +
// three tcgen05 GEMMs + col2im.  The caller owns every buffer (plan->ws included).
#include "common.cuh"

namespace impflow {

static inline size_t pad64(size_t n) { return (n + 63) / 64 * 64; }

struct Conv3Ws {
  float *xin, *x0, *h1, *h2, *Y, *Y2, *t_rows, *chain_a, *chain_b;
  size_t total;
};

static Conv3Ws carve(float* base, long long M, int c, int C, int k0) {
  Conv3Ws w;
  size_t off = 0;
  auto take = [&](size_t n) {
    float* p = base ? base + off : nullptr;
    off += pad64(n);
    return p;
  };
  w.xin = take((size_t)M * c);
  w.x0 = take(2 * (size_t)M * k0);
  w.h1 = take(2 * (size_t)M * C);
  w.h2 = take(2 * (size_t)M * C);
  w.Y = take((size_t)M * 9 * c * (size_t)(C % 128 == 0 ? C / 128 : 1));   // room for the chain23 partials
  // second tap accumulator of the power-series chain on the tile kernel (its two channel halves are summed into a
  // ZEROED accumulator: term k's epilogue zeroes the one term k + 1 accumulates into)
  w.Y2 = take((k0 == 32 && 9 * c <= 32) ? (size_t)M * 9 * c : 0);
  w.t_rows = take((size_t)M * c);
  w.chain_a = take((size_t)M * c);
  w.chain_b = take((size_t)M * c);
  w.total = off;
  return w;
}

static inline bool use_tile_kernel(const impflow_conv3_plan* p) {
  return p->allow_fused && p->k0 == 32 && (p->C % 256) == 0 && 9 * p->c <= 32;
}

// layers 2 + 3 in one launch (chain23_fused.cu) whenever the tile kernel does not apply and C splits into quarters
static int g_chain23 = 1;
static inline bool use_chain23(const impflow_conv3_plan* p) {
  return g_chain23 && p->allow_fused && !use_tile_kernel(p) && (p->C % 128) == 0;
}
static inline int y_parts(const impflow_conv3_plan* p) { return use_chain23(p) ? p->C / 128 : 1; }
// layer 1 hands layer 2 ONE fp32 plane (k_chain23 splits it on chip) instead of tf32 hi/lo planes.  Measured SLOWER
// (k_chain23 79 -> 101 us at M = 16384, step 69.3 -> 71.2 ms): the kernel is bound by the SM's shared-memory port
// (SS-form N = 128 MMAs read 128 B/clk, the TMA writes come on top), and the on-chip split adds 48 KB per chunk to it.
static int g_chain23_a32 = 0;

static int plan_check(const impflow_conv3_plan* p, const char* who) {
  if (p == nullptr || p->ws == nullptr) {
    set_error("%s: plan or workspace missing", who);
    return -3;
  }
  if (p->B < 1 || p->H < 1 || p->W < 1 || p->c < 1 || p->C < 8 || p->k0 < 9 * p->c || (p->k0 % 32) != 0) {
    set_error("%s: bad plan (B=%d H=%d W=%d c=%d C=%d k0=%d)", who, p->B, p->H, p->W, p->c, p->C, p->k0);
    return -3;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// Glue kernels either side of the tile kernel / GEMM chain, one launch each (they replace act_mul + im2col
// (+ memset) in front and col2im + lincomb3 behind):
//
//   k_conv3_in :  X0[p, (ky,kx,ci)] = act0(x)[p + (ky-1,kx-1), ci]   fp32 rows (tile kernel) or tf32 hi/lo planes
//                 (GEMM chain), tail columns zero; also zero-fills the tap accumulator Y when the tile kernel
//                 sums two channel halves into it.
//   k_conv3_out:  val = col2im(Y) (+ bias3)            forward
//                     = col2im(Y) * act0'(pre0)        transposed sweep with a leading activation
//                 and, in the same pass,
//                   plain    : out = val
//                   fwd resid: out = (rhs - val) - x           g(z) = x_embed - f(z) - z   (implicit_block.py:72)
//                   bwd resid: out = (val + x) - rhs           g(v) = v^T J + v - grad     (:199-203)
//                   chain    : out = val, acc = fma(val, coeff, acc)   w += c_k v^T J^k    (:431-435)
//                   fixed pt : out = rhs - val, and the element test of the Banach loop against the previous
//                              iterate x; the last block decides        (iresblock.py:69-79, see fixed_point_decide)
//                 (the same roundings, in the same order, as the separate lincomb3 launches they replace)
// Both honour the device gate of the sync-free solver loop (common.cuh).
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void split_tf32_1(float v, float& hi, float& lo) {
  uint32_t h;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
  hi = __uint_as_float(h);
  lo = v - hi;
}

__global__ void __launch_bounds__(256)
k_conv3_in(const float* __restrict__ x, float* __restrict__ col, float* __restrict__ col_lo, float* __restrict__ zero,
           long long zero_n4, int B, int H, int W, int C, int ld, int act0_kind, const float* __restrict__ beta0,
           const int* gate) {
  pdl_trigger();
  pdl_wait();
  if (gate_closed(gate)) return;
  const float beta = (beta0 != nullptr) ? __ldg(beta0) : 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (zero != nullptr) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long long i = tid; i < zero_n4; i += stride) reinterpret_cast<float4*>(zero)[i] = z;
  }
  const int groups = ld / 4;
  const long long total = (long long)B * H * W * groups;
  const int K = 9 * C;
  for (long long i = tid; i < total; i += stride) {
    const long long p = i / groups;
    const int k0 = (int)(i - p * groups) * 4;
    const int xx = (int)(p % W);
    const int yy = (int)((p / W) % H);
    const long long img = p - (long long)yy * W - xx;
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int k = k0 + u;
      v[u] = 0.f;
      if (k < K) {
        const int tap = k / C, c = k - tap * C;
        const int sy = yy + tap / 3 - 1, sx = xx + tap % 3 - 1;
        if (sy >= 0 && sy < H && sx >= 0 && sx < W) {
          const float xv = __ldg(x + (img + (long long)sy * W + sx) * C + c);
          v[u] = act0_kind == IMPFLOW_ACT_NONE ? xv : act_dispatch(act0_kind, xv, 0, beta);
        }
      }
    }
    float* dst = col + p * ld + k0;
    if (col_lo != nullptr) {
      float h[4], l[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) split_tf32_1(v[u], h[u], l[u]);
      *reinterpret_cast<float4*>(dst) = make_float4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<float4*>(col_lo + p * ld + k0) = make_float4(l[0], l[1], l[2], l[3]);
    } else {
      *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

enum { OUT_PLAIN = 0, OUT_FWD_RESIDUAL = 1, OUT_BWD_RESIDUAL = 2, OUT_CHAIN = 3, OUT_FIXED_POINT = 4 };

struct Conv3Out {
  int nparts;           // partial accumulators to sum (chain23: one per 128-channel quarter), fixed order
  long long part_stride;
  const float* col;     // [M, 9c] tap-major accumulator
  const float* bias;    // [c] or null
  const float* pre0;    // [M, c] or null: multiply by act0'(pre0)
  const float* beta0;
  int act0_kind;
  int mode;
  const float* x;       // residual modes: the iterate
  const float* rhs;     // residual modes: x_embed / incoming gradient
  float* out;           // [M, c]
  float* acc;           // chain mode: w
  float coeff;
  const int* gate;
  // power-series chain: the result is also the input of the NEXT evaluation, so its im2col rows are written here
  // (what a k_conv3_in launch would produce from `out`): fp32 rows, or tf32 hi / lo planes when next_lo is set
  float* next_col;
  float* next_lo;
  int next_ld;
  float* zero;          // tap accumulator of the next evaluation to clear (tile kernel), zero_n4 float4 groups
  long long zero_n4;
  // fixed-point mode: evaluation `iter` of the Banach loop (x = the previous iterate, rhs = the right-hand side)
  const float* start;   // |start| scales the tolerance (the reference's quirk in the Banach fallback: not |rhs|)
  impflow_fixed_point_state* fp;
  BroydenProgress* fp_progress;   // mapped pinned records, index iter - 1
  float atol, rtol;
  int iter, threshold;
};

// Sum of the blocks' failing-element counts (integers: the order of the atomic adds does not matter); the last block
// to arrive applies the stopping rule of evaluation a.iter, publishes it and re-arms the counters for the next one.
__device__ __forceinline__ void fixed_point_decide(const Conv3Out& a, int fails) {
  __shared__ int warp_fails[8];     // 256 threads (launch_out)
  fails = __reduce_add_sync(0xffffffffu, fails);
  if ((threadIdx.x & 31) == 0) warp_fails[threadIdx.x >> 5] = fails;
  __syncthreads();
  if (threadIdx.x != 0) return;
  int block = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) block += warp_fails[w];
  if (block != 0) atomicAdd(&a.fp->fails, block);
  __threadfence();
  if (atomicAdd(&a.fp->ticket, 1) != (int)gridDim.x - 1) return;
  __threadfence();
  const int total = atomicAdd(&a.fp->fails, 0);
  const int active = (a.iter - 1 > a.threshold || total == 0) ? 0 : 1;
  a.fp->iterations = a.iter - 1;
  a.fp->active = active;
  a.fp->fails = 0;
  a.fp->ticket = 0;
  __threadfence();
  if (a.fp_progress != nullptr) {
    volatile BroydenProgress* pr = a.fp_progress + (a.iter - 1);
    pr->active = active;
    __threadfence_system();
    pr->seq = a.iter - 1;
    __threadfence_system();
  }
}

__global__ void __launch_bounds__(256) k_conv3_out(int B, int H, int W, int C, Conv3Out a) {
  pdl_trigger();
  pdl_wait();
  if (gate_closed(a.gate)) return;
  const float beta = (a.beta0 != nullptr) ? __ldg(a.beta0) : 0.f;
  const long long total = (long long)B * H * W * C;
  int fails = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long long p = i / C;
    const int xx = (int)(p % W);
    const int yy = (int)((p / W) % H);
    const long long b = p / ((long long)W * H);
    float sum = 0.f;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int sy = yy - (tap / 3 - 1), sx = xx - (tap % 3 - 1);
      if (sy >= 0 && sy < H && sx >= 0 && sx < W) {
        const float* src = a.col + (((b * H + sy) * W + sx) * 9 + tap) * C + c;
        float v = src[0];
        for (int part = 1; part < a.nparts; ++part) v += src[part * a.part_stride];
        sum += v;
      }
    }
    float val;
    if (a.pre0 != nullptr) {
      val = sum * act_dispatch(a.act0_kind, a.pre0[i], 1, beta);
    } else {
      val = sum + (a.bias != nullptr ? a.bias[c] : 0.f);
    }
    float r = val;
    if (a.mode == OUT_FIXED_POINT) {
      // x = rhs - f (one rounding, as lincomb3(rhs, 1, f, -1)); test (x - x_prev)^2 / (atol + |start| rtol) < 1 with
      // the roundings of the torch expression: no contraction into FMAs, a NaN fails
      r = __fsub_rn(a.rhs[i], val);
      const float tol = __fadd_rn(a.atol, __fmul_rn(fabsf(a.start[i]), a.rtol));
      const float dx = __fsub_rn(r, a.x[i]);
      fails += (__fdiv_rn(__fmul_rn(dx, dx), tol) < 1.f) ? 0 : 1;
    } else if (a.mode == OUT_FWD_RESIDUAL) {
      r = a.rhs[i] - val;
      r = r - a.x[i];
    } else if (a.mode == OUT_BWD_RESIDUAL) {
      r = val + a.x[i];
      r = r - a.rhs[i];
    } else if (a.mode == OUT_CHAIN) {
      a.acc[i] = fmaf(val, a.coeff, a.acc[i]);
    }
    a.out[i] = r;
    if (a.next_col != nullptr) {
      // im2col of the next evaluation, scattered: X0[p - delta][tap][c] = r for every tap whose source pixel is p;
      // the slots of THIS row whose source pixel lies outside the image are zero
      float hi = r, lo = 0.f;
      if (a.next_lo != nullptr) split_tf32_1(r, hi, lo);
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int dy = tap / 3 - 1, dx = tap % 3 - 1;
        const int ty = yy - dy, tx = xx - dx;              // row that reads pixel p through `tap`
        if (ty >= 0 && ty < H && tx >= 0 && tx < W) {
          const long long slot = ((b * H + ty) * W + tx) * a.next_ld + tap * C + c;
          a.next_col[slot] = hi;
          if (a.next_lo != nullptr) a.next_lo[slot] = lo;
        }
        const int sy = yy + dy, sx = xx + dx;              // source pixel of this row's `tap`
        if (sy < 0 || sy >= H || sx < 0 || sx >= W) {
          const long long slot = p * a.next_ld + tap * C + c;
          a.next_col[slot] = 0.f;
          if (a.next_lo != nullptr) a.next_lo[slot] = 0.f;
        }
      }
    }
  }
  if (a.zero != nullptr) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.zero_n4;
         i += (long long)gridDim.x * blockDim.x)
      reinterpret_cast<float4*>(a.zero)[i] = z;
  }
  if (a.mode == OUT_FIXED_POINT) fixed_point_decide(a, fails);
}

static inline int grid_cap(long long n, int per) {
  long long g = (n + per - 1) / per;
  const long long cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

static int launch_in(const impflow_conv3_plan* p, const float* x_rows, int act0_kind, const float* beta0, float* col,
                     float* col_lo, int ld, float* zero, long long zero_n, cudaStream_t s) {
  const long long M = (long long)p->B * p->H * p->W;
  if ((zero_n & 3) != 0) {       // odd tap-accumulator size: fall back to a memset (never the case for M % 128 == 0)
    if (zero != nullptr && cudaMemsetAsync(zero, 0, sizeof(float) * (size_t)zero_n, s) != cudaSuccess) {
      set_error("conv3: memset failed");
      return -1;
    }
    zero = nullptr;
  }
  const cudaError_t e = launch_pdl(k_conv3_in, grid_cap(M * (ld / 4), 256), 256, s, x_rows, col, col_lo, zero,
                                   zero_n >> 2, p->B, p->H, p->W, p->c, ld, act0_kind, beta0, g_gate);
  if (e != cudaSuccess) {
    set_error("k_conv3_in: launch failed: %s", cudaGetErrorString(e));
    return -1;
  }
  return check_launch("k_conv3_in");
}

static int launch_out(const impflow_conv3_plan* p, Conv3Out a, cudaStream_t s) {
  const long long total = (long long)p->B * p->H * p->W * p->c;
  a.gate = g_gate;
  const cudaError_t e = launch_pdl(k_conv3_out, grid_cap(total, 256), 256, s, p->B, p->H, p->W, p->c, a);
  if (e != cudaSuccess) {
    set_error("k_conv3_out: launch failed: %s", cudaGetErrorString(e));
    return -1;
  }
  return check_launch("k_conv3_out");
}

// Y (tap accumulator, [M, 9c]) = the three-layer chain applied to x_rows, forward (act0 applied to the input on the fly).
static int conv3_chain_forward(const impflow_conv3_plan* p, const Conv3Ws& w, const float* x_rows, float* pre1,
                               float* pre2, void* stream) {
  const long long M = (long long)p->B * p->H * p->W;
  const int N3 = 9 * p->c;
  cudaStream_t s = (cudaStream_t)stream;
  if (use_tile_kernel(p)) {
    if (launch_in(p, x_rows, p->act0_kind, p->beta0, w.x0, nullptr, 32, p->C > 256 ? w.Y : nullptr, M * N3, s)) return -1;
    return impflow_branch3_tc(w.x0, 32, p->W1f_hi, p->W1f_lo, p->W2f_hi, p->W2f_lo, p->W3f_hi, p->W3f_lo, p->b1, p->b2,
                              nullptr, nullptr, pre1, pre2, w.Y, N3, M, p->C, N3, p->act_kind, p->beta1, p->beta2,
                              stream);
  }
  float* x0_hi = w.x0;
  float* x0_lo = w.x0 + (size_t)M * p->k0;
  float* h1_hi = w.h1;
  float* h1_lo = w.h1 + (size_t)M * p->C;
  float* h2_hi = w.h2;
  float* h2_lo = w.h2 + (size_t)M * p->C;
  if (launch_in(p, x_rows, p->act0_kind, p->beta0, x0_hi, x0_lo, p->k0, nullptr, 0, s)) return -1;
  const bool a32 = use_chain23(p) && g_chain23_a32;
  if (impflow_gemm_nt_tc(x0_hi, x0_lo, p->k0, p->W1f_hi, p->W1f_lo, p->k0, p->b1, pre1, a32 ? h1_hi : nullptr, nullptr,
                         a32 ? nullptr : h1_hi, a32 ? nullptr : h1_lo, p->C, M, p->C, p->k0, p->act_kind, p->beta1,
                         nullptr, stream))
    return -1;
  if (use_chain23(p))
    return impflow_chain23_tc(h1_hi, a32 ? nullptr : h1_lo, p->C, p->W2f_hi, p->W2f_lo, p->W3f_hi, p->W3f_lo, p->b2, nullptr, pre2, w.Y,
                              N3, M * N3, M, p->C, N3, p->act_kind, p->beta2, stream);
  if (impflow_gemm_nt_tc(h1_hi, h1_lo, p->C, p->W2f_hi, p->W2f_lo, p->C, p->b2, pre2, nullptr, nullptr, h2_hi, h2_lo,
                         p->C, M, p->C, p->C, p->act_kind, p->beta2, nullptr, stream))
    return -1;
  return impflow_gemm_nt_tc(h2_hi, h2_lo, p->C, p->W3f_hi, p->W3f_lo, p->C, nullptr, w.Y, nullptr, nullptr, nullptr,
                            nullptr, N3, M, N3, p->C, IMPFLOW_ACT_NONE, nullptr, nullptr, stream);
}

// Y = the transposed chain applied to v_rows (d1, d2 = act'(pre) of the two hidden layers).
// skip_in: the im2col rows of v_rows (and, for the tile kernel, the cleared accumulator) were already produced by the
// epilogue of the previous evaluation (power-series chain); Yt: tap accumulator to use (default w.Y)
static int conv3_chain_vjp(const impflow_conv3_plan* p, const Conv3Ws& w, const float* d1, const float* d2,
                           const float* v_rows, void* stream, bool skip_in = false, float* Yt = nullptr) {
  const long long M = (long long)p->B * p->H * p->W;
  const int N3 = 9 * p->c;
  cudaStream_t s = (cudaStream_t)stream;
  float* const Y = Yt != nullptr ? Yt : w.Y;
  if (use_tile_kernel(p)) {
    if (!skip_in &&
        launch_in(p, v_rows, IMPFLOW_ACT_NONE, nullptr, w.x0, nullptr, 32, p->C > 256 ? Y : nullptr, M * N3, s))
      return -1;
    return impflow_branch3_tc(w.x0, 32, p->W3b_hi, p->W3b_lo, p->W2b_hi, p->W2b_lo, p->W1b_hi, p->W1b_lo, nullptr,
                              nullptr, d2, d1, nullptr, nullptr, Y, N3, M, p->C, N3, IMPFLOW_ACT_NONE, nullptr, nullptr,
                              stream);
  }
  float* x0_hi = w.x0;
  float* x0_lo = w.x0 + (size_t)M * p->k0;
  float* t3_hi = w.h1;
  float* t3_lo = w.h1 + (size_t)M * p->C;
  float* t2_hi = w.h2;
  float* t2_lo = w.h2 + (size_t)M * p->C;
  if (!skip_in && launch_in(p, v_rows, IMPFLOW_ACT_NONE, nullptr, x0_hi, x0_lo, p->k0, nullptr, 0, s)) return -1;
  const bool a32 = use_chain23(p) && g_chain23_a32;     // dmul mode: pre_out receives acc * act'(d2)
  if (impflow_gemm_nt_tc(x0_hi, x0_lo, p->k0, p->W3b_hi, p->W3b_lo, p->k0, nullptr, a32 ? t3_hi : nullptr, nullptr, d2,
                         a32 ? nullptr : t3_hi, a32 ? nullptr : t3_lo, p->C, M, p->C, p->k0, IMPFLOW_ACT_MULTIPLIER,
                         nullptr, nullptr, stream))
    return -1;
  if (use_chain23(p))
    return impflow_chain23_tc(t3_hi, a32 ? nullptr : t3_lo, p->C, p->W2b_hi, p->W2b_lo, p->W1b_hi, p->W1b_lo, nullptr, d1, nullptr, w.Y,
                              N3, M * N3, M, p->C, N3, IMPFLOW_ACT_NONE, nullptr, stream);
  if (impflow_gemm_nt_tc(t3_hi, t3_lo, p->C, p->W2b_hi, p->W2b_lo, p->C, nullptr, nullptr, nullptr, d1, t2_hi, t2_lo,
                         p->C, M, p->C, p->C, IMPFLOW_ACT_MULTIPLIER, nullptr, nullptr, stream))
    return -1;
  return impflow_gemm_nt_tc(t2_hi, t2_lo, p->C, p->W1b_hi, p->W1b_lo, p->C, nullptr, w.Y, nullptr, nullptr, nullptr,
                            nullptr, N3, M, N3, p->C, IMPFLOW_ACT_NONE, nullptr, nullptr, stream);
}

static Conv3Out out_forward(const impflow_conv3_plan* p, const Conv3Ws& w, float* out) {
  Conv3Out a;
  memset(&a, 0, sizeof(a));
  a.nparts = y_parts(p);
  a.part_stride = (long long)p->B * p->H * p->W * 9 * p->c;
  a.col = w.Y;
  a.bias = p->b3;
  a.act0_kind = IMPFLOW_ACT_NONE;
  a.mode = OUT_PLAIN;
  a.out = out;
  return a;
}

static Conv3Out out_vjp(const impflow_conv3_plan* p, const Conv3Ws& w, const float* pre0, float* out) {
  Conv3Out a;
  memset(&a, 0, sizeof(a));
  a.nparts = y_parts(p);
  a.part_stride = (long long)p->B * p->H * p->W * 9 * p->c;
  a.col = w.Y;
  a.act0_kind = p->act0_kind;
  a.beta0 = p->beta0;
  a.pre0 = p->act0_kind != IMPFLOW_ACT_NONE ? pre0 : nullptr;
  a.mode = OUT_PLAIN;
  a.out = out;
  return a;
}

// power-series chain: the col2im epilogue of term k also writes the im2col rows of term k + 1 (one k_conv3_in launch
// less per term); impflow_conv3_set_chain_fuse for A/B
static int g_chain_fuse = 1;
static int g_runahead = 2;     // iterations the host may enqueue beyond the last decision it has seen (0 = sync per iteration)

}  // namespace impflow

using namespace impflow;

extern "C" size_t impflow_conv3_workspace_floats(int B, int H, int W, int c, int C, int k0) {
  return carve(nullptr, (long long)B * H * W, c, C, k0).total;
}

extern "C" int impflow_conv3_forward(const impflow_conv3_plan* plan, const float* x_rows, float* y_rows, float* pre1,
                                     float* pre2, void* stream) {
  if (plan_check(plan, "conv3_forward")) return -3;
  const long long M = (long long)plan->B * plan->H * plan->W;
  const Conv3Ws w = carve(plan->ws, M, plan->c, plan->C, plan->k0);
  GateScope ungated(nullptr);
  if (conv3_chain_forward(plan, w, x_rows, pre1, pre2, stream)) return -1;
  return launch_out(plan, out_forward(plan, w, y_rows), (cudaStream_t)stream);
}

extern "C" int impflow_conv3_prepare_vjp(const impflow_conv3_plan* plan, const float* pre1, const float* pre2,
                                         float* d1, float* d2, void* stream) {
  if (plan_check(plan, "conv3_prepare_vjp")) return -3;
  const long long n = (long long)plan->B * plan->H * plan->W * plan->C;
  if (impflow_act_mul(pre1, nullptr, d1, n, plan->act_kind, 1, plan->beta1, stream)) return -1;
  return impflow_act_mul(pre2, nullptr, d2, n, plan->act_kind, 1, plan->beta2, stream);
}

extern "C" int impflow_conv3_vjp(const impflow_conv3_plan* plan, const float* pre0, const float* d1, const float* d2,
                                 const float* v_rows, float* out_rows, void* stream) {
  if (plan_check(plan, "conv3_vjp")) return -3;
  IMPFLOW_REQUIRE(plan->act0_kind == IMPFLOW_ACT_NONE || pre0 != nullptr, "conv3_vjp: pre0 missing");
  const long long M = (long long)plan->B * plan->H * plan->W;
  const Conv3Ws w = carve(plan->ws, M, plan->c, plan->C, plan->k0);
  GateScope ungated(nullptr);
  if (conv3_chain_vjp(plan, w, d1, d2, v_rows, stream)) return -1;
  return launch_out(plan, out_vjp(plan, w, pre0, out_rows), (cudaStream_t)stream);
}

extern "C" int impflow_conv3_power_series(const impflow_conv3_plan* plan, const float* pre0, const float* d1,
                                          const float* d2, const float* v_rows, const double* coeffs, int n,
                                          float* w_rows, const double* dot_coeffs, float* dot_out, void* stream) {
  if (plan_check(plan, "conv3_power_series")) return -3;
  IMPFLOW_REQUIRE(plan->act0_kind == IMPFLOW_ACT_NONE || pre0 != nullptr, "conv3_power_series: pre0 missing");
  IMPFLOW_REQUIRE((w_rows != nullptr && coeffs != nullptr) || (dot_out != nullptr && dot_coeffs != nullptr),
                  "conv3_power_series: neither the Neumann sum nor the Hutchinson dots were requested");
  IMPFLOW_REQUIRE((dot_out == nullptr) == (dot_coeffs == nullptr), "conv3_power_series: dot_out and dot_coeffs go together");
  const long long M = (long long)plan->B * plan->H * plan->W;
  const long long nel = M * plan->c;
  const long long d = nel / plan->B;
  const Conv3Ws w = carve(plan->ws, M, plan->c, plan->C, plan->k0);
  cudaStream_t s = (cudaStream_t)stream;
  GateScope ungated(nullptr);
  if (w_rows != nullptr && impflow_lincomb3(v_rows, 1.f, nullptr, 0.f, nullptr, 0.f, w_rows, nel, stream)) return -1;
  const float* cur = v_rows;
  float* bufs[2] = {w.chain_a, w.chain_b};
  const bool tile = use_tile_kernel(plan);
  const int N3 = 9 * plan->c;
  const bool fuse = g_chain_fuse && ((M * N3) % 4 == 0) && (!tile || w.Y2 != nullptr);
  for (int k = 0; k < n; ++k) {
    float* nxt = bufs[k & 1];
    float* Yk = (tile && fuse && (k & 1)) ? w.Y2 : w.Y;
    if (conv3_chain_vjp(plan, w, d1, d2, cur, stream, fuse && k > 0, Yk)) return -1;
    Conv3Out a = out_vjp(plan, w, pre0, nxt);
    a.col = Yk;
    if (fuse && k + 1 < n) {        // this epilogue prepares the next evaluation's input
      a.next_col = w.x0;
      a.next_lo = tile ? nullptr : w.x0 + (size_t)M * plan->k0;
      a.next_ld = tile ? 32 : plan->k0;
      if (tile && plan->C > 256) {
        a.zero = (k & 1) ? w.Y : w.Y2;
        a.zero_n4 = (M * N3) >> 2;
      }
    }
    if (w_rows != nullptr) {        // w += c_k v^T J^k in the col2im epilogue (implicit_block.py:435)
      a.mode = OUT_CHAIN;
      a.acc = w_rows;
      a.coeff = (float)coeffs[k];
    }
    if (launch_out(plan, a, s)) return -1;
    if (dot_out != nullptr &&       // Hutchinson term alpha_k <v^T J^k, v> per sample (:423)
        impflow_rowdot(nxt, v_rows, dot_out, plan->B, d, (float)dot_coeffs[k], k == 0 ? 0.f : 1.f, stream))
      return -1;
    cur = nxt;
  }
  return 0;
}

extern "C" int impflow_conv3_set_chain23(int on) {
  const int prev = g_chain23;
  g_chain23 = on ? 1 : 0;
  return prev;
}

extern "C" int impflow_conv3_set_chain23_a32(int on) {
  const int prev = g_chain23_a32;
  g_chain23_a32 = on ? 1 : 0;
  return prev;
}

extern "C" int impflow_conv3_set_chain_fuse(int on) {
  const int prev = g_chain_fuse;
  g_chain_fuse = on ? 1 : 0;
  return prev;
}

extern "C" int impflow_conv3_set_runahead(int iterations) {
  const int prev = g_runahead;
  g_runahead = iterations < 0 ? 0 : (iterations > 8 ? 8 : iterations);
  return prev;
}

extern "C" size_t impflow_conv3_broyden_host_bytes(int threshold) {
  return sizeof(impflow_broyden_state) + sizeof(BroydenProgress) * (size_t)(threshold + 2);
}

extern "C" int impflow_conv3_broyden(const impflow_conv3_plan* plan, int mode, const float* rhs_rows,
                                     const float* pre0, const float* d1, const float* d2, float* xa, float* xb,
                                     float* ga, float* gb, float* low_x, float* low_g, float* Ut, float* Vt,
                                     float* sample_sq, float* low_sq, float* partial,
                                     impflow_broyden_state* state_dev, impflow_broyden_state* state_host,
                                     int threshold, double eps_scaled, void* stream) {
  if (plan_check(plan, "conv3_broyden")) return -3;
  IMPFLOW_REQUIRE(mode == 0 || mode == 1, "conv3_broyden: mode must be 0 (forward) or 1 (implicit backward)");
  IMPFLOW_REQUIRE(mode == 0 || plan->act0_kind == IMPFLOW_ACT_NONE || pre0 != nullptr, "conv3_broyden: pre0 missing");
  IMPFLOW_REQUIRE(threshold >= 1 && threshold <= 63, "conv3_broyden: threshold %d not in [1,63]", threshold);
  const long long M = (long long)plan->B * plan->H * plan->W;
  const long long d = (long long)plan->H * plan->W * plan->c;
  const Conv3Ws w = carve(plan->ws, M, plan->c, plan->C, plan->k0);
  cudaStream_t s = (cudaStream_t)stream;
  // residual, written by the col2im epilogue:  forward  g(z) = x_embed - f(z) - z   (implicit_block.py:72)
  //                                            backward g(v) = v^T J + v - grad      (:199-203)
  auto eval_g = [&](const float* x, float* g) -> int {
    Conv3Out a;
    if (mode == 0) {
      if (conv3_chain_forward(plan, w, x, nullptr, nullptr, stream)) return -1;
      a = out_forward(plan, w, g);
      a.mode = OUT_FWD_RESIDUAL;
    } else {
      if (conv3_chain_vjp(plan, w, d1, d2, x, stream)) return -1;
      a = out_vjp(plan, w, pre0, g);
      a.mode = OUT_BWD_RESIDUAL;
    }
    a.x = x;
    a.rhs = rhs_rows;
    return launch_out(plan, a, s);
  };
  auto read_state = [&]() -> int {
    if (cudaMemcpyAsync(state_host, state_dev, sizeof(impflow_broyden_state), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess) {
      set_error("conv3_broyden: state read-back failed: %s", cudaGetErrorString(cudaGetLastError()));
      return -1;
    }
    return 0;
  };
  float* xs[2] = {xa, xb};      // iteration it evaluates g at xs[it & 1] (the update kernel writes the next iterate
  float* gs[2] = {ga, gb};      // into the other buffer): the roles alternate unconditionally, so they are known ahead

  // progress records in mapped pinned memory behind the state record (impflow_conv3_broyden_host_bytes)
  BroydenProgress* prog_host = reinterpret_cast<BroydenProgress*>(state_host + 1);
  BroydenProgress* prog_dev = nullptr;
  int runahead = g_runahead;
  if (runahead > 0 &&
      cudaHostGetDevicePointer(reinterpret_cast<void**>(&prog_dev), prog_host, 0) != cudaSuccess) {
    cudaGetLastError();
    runahead = 0;               // not mapped memory: fall back to one synchronisation per iteration
    prog_dev = nullptr;
  }

  if (runahead == 0) {
    GateScope ungated(nullptr);
    if (eval_g(xs[0], gs[0])) return -1;
    if (impflow_broyden_begin(xs[0], gs[0], xs[1], low_x, low_g, sample_sq, low_sq, partial, state_dev, plan->B, d,
                              threshold, eps_scaled, stream))
      return -1;
    if (read_state()) return -1;
    for (int it = 1; state_host->active; ++it) {
      if (eval_g(xs[it & 1], gs[it & 1])) return -1;
      if (impflow_broyden_step(xs[(it - 1) & 1], gs[(it - 1) & 1], xs[it & 1], gs[it & 1], Ut, Vt, low_x, low_g,
                               sample_sq, low_sq, partial, state_dev, plan->B, d, threshold, stream))
        return -1;
      if (read_state()) return -1;
    }
    return 0;
  }

  // ---- sync-free loop: the host enqueues up to `runahead` iterations beyond the last decision it has seen; the
  // device decides (k_norm_decide), speculative kernels behind the end of the loop are no-ops (gate), and the host
  // learns the decisions from the progress records instead of draining the stream (broyden.py:153-181 unchanged)
  volatile BroydenProgress* vp = prog_host;
  for (int i = 0; i <= threshold + 1; ++i) vp[i].seq = -1;
  auto wait_for = [&](int it) -> int {
    long long spins = 0;
    while (vp[it].seq != it) {
      if ((++spins & 0x3ff) == 0) {
        const cudaError_t q = cudaStreamQuery(s);
        if (q != cudaSuccess && q != cudaErrorNotReady) {
          set_error("conv3_broyden: stream failed while waiting for iteration %d: %s", it, cudaGetErrorString(q));
          return -1;
        }
        if (q == cudaSuccess && vp[it].seq != it) {
          set_error("conv3_broyden: iteration %d never reported (stream idle)", it);
          return -1;
        }
      }
    }
    return 0;
  };
  {
    GateScope ungated(nullptr);
    if (eval_g(xs[0], gs[0])) return -1;
    if (broyden_begin_ex(xs[0], gs[0], xs[1], low_x, low_g, sample_sq, low_sq, partial, state_dev, plan->B, d, threshold,
                         eps_scaled, prog_dev, stream))
      return -1;
  }
  int seen = -1, enq = 0;      // enq = iterations enqueued so far; record 0 belongs to the start point
  {
    GateScope gated(&state_dev->active);
    for (;;) {
      while (enq < seen + 1 + runahead && enq < threshold) {
        const int it = ++enq;
        if (eval_g(xs[it & 1], gs[it & 1])) return -1;
        if (broyden_step_ex(xs[(it - 1) & 1], gs[(it - 1) & 1], xs[it & 1], gs[it & 1], Ut, Vt, low_x, low_g, sample_sq,
                            low_sq, partial, state_dev, plan->B, d, threshold, 1, it, prog_dev, stream))
          return -1;
      }
      if (wait_for(seen + 1)) return -1;
      ++seen;
      if (!vp[seen].active) break;
    }
  }
  return read_state();        // full state record (trace, flags) + one stream drain per solve
}

extern "C" size_t impflow_conv3_fixed_point_host_bytes(int threshold) {
  return sizeof(impflow_fixed_point_state) + sizeof(BroydenProgress) * (size_t)(threshold + 2);
}

extern "C" int impflow_conv3_fixed_point(const impflow_conv3_plan* plan, const float* rhs_rows, const float* start_rows,
                                         float* out_rows, float* xa, float* xb, impflow_fixed_point_state* state_dev,
                                         impflow_fixed_point_state* state_host, float atol, float rtol, int threshold,
                                         void* stream) {
  if (plan_check(plan, "conv3_fixed_point")) return -3;
  IMPFLOW_REQUIRE(threshold >= 0 && threshold <= 1000, "conv3_fixed_point: threshold %d not in [0,1000]", threshold);
  const long long M = (long long)plan->B * plan->H * plan->W;
  const Conv3Ws w = carve(plan->ws, M, plan->c, plan->C, plan->k0);
  cudaStream_t s = (cudaStream_t)stream;
  // progress records in mapped pinned memory behind the state record (impflow_conv3_fixed_point_host_bytes), one per
  // evaluation: record k - 1 is written by the decision of evaluation k
  BroydenProgress* prog_host = reinterpret_cast<BroydenProgress*>(state_host + 1);
  BroydenProgress* prog_dev = nullptr;
  if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&prog_dev), prog_host, 0) != cudaSuccess) {
    cudaGetLastError();
    set_error("conv3_fixed_point: state_host is not mapped pinned host memory");
    return -3;
  }
  const int runahead = g_runahead;
  const int last = threshold + 2;            // evaluations at most
  float* xs[2] = {xa, xb};                   // evaluation k writes xs[k & 1]: the roles are known ahead
  auto eval = [&](int k) -> int {
    const float* prev = k == 1 ? start_rows : xs[(k - 1) & 1];
    if (conv3_chain_forward(plan, w, prev, nullptr, nullptr, stream)) return -1;
    Conv3Out a = out_forward(plan, w, xs[k & 1]);
    a.mode = OUT_FIXED_POINT;
    a.x = prev;
    a.rhs = rhs_rows;
    a.start = start_rows;
    a.fp = state_dev;
    a.fp_progress = prog_dev;
    a.atol = atol;
    a.rtol = rtol;
    a.iter = k;
    a.threshold = threshold;
    return launch_out(plan, a, s);
  };
  volatile BroydenProgress* vp = prog_host;
  for (int i = 0; i < last; ++i) vp[i].seq = -1;
  auto wait_for = [&](int rec) -> int {
    long long spins = 0;
    while (vp[rec].seq != rec) {
      if ((++spins & 0x3ff) == 0) {
        const cudaError_t q = cudaStreamQuery(s);
        if (q != cudaSuccess && q != cudaErrorNotReady) {
          set_error("conv3_fixed_point: stream failed while waiting for evaluation %d: %s", rec + 1,
                    cudaGetErrorString(q));
          return -1;
        }
        if (q == cudaSuccess && vp[rec].seq != rec) {
          set_error("conv3_fixed_point: evaluation %d never reported (stream idle)", rec + 1);
          return -1;
        }
      }
    }
    return 0;
  };
  // zero counters and ticket; evaluation 1 always runs (ungated), its decision opens or closes the gate
  if (cudaMemsetAsync(state_dev, 0, sizeof(impflow_fixed_point_state), s) != cudaSuccess) {
    set_error("conv3_fixed_point: state reset failed");
    return -1;
  }
  {
    GateScope ungated(nullptr);
    if (eval(1)) return -1;
  }
  int seen = 0, enq = 1;       // decisions seen / evaluations enqueued
  {
    GateScope gated(&state_dev->active);
    for (;;) {
      while (enq < seen + 1 + runahead && enq < last) {
        if (eval(++enq)) return -1;
      }
      if (wait_for(seen)) return -1;
      ++seen;
      if (!vp[seen - 1].active) break;
    }
  }
  // evaluation `seen` ended the loop; the gated evaluations behind it wrote nothing
  const size_t bytes = sizeof(float) * (size_t)M * plan->c;
  if (cudaMemcpyAsync(out_rows, xs[seen & 1], bytes, cudaMemcpyDeviceToDevice, s) != cudaSuccess ||
      cudaMemcpyAsync(state_host, state_dev, sizeof(impflow_fixed_point_state), cudaMemcpyDeviceToHost, s) !=
          cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess) {
    set_error("conv3_fixed_point: result copy failed: %s", cudaGetErrorString(cudaGetLastError()));
    return -1;
  }
  return 0;
}
