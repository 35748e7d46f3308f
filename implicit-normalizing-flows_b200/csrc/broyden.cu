// Broyden solver algebra on the device — replaces lib/layers/broyden.py:101-193.
//
// Data layout in HBM (all fp32, dense):
//   x, g, xn, gn, low_x, low_g : (B, d)
//   Ut, Vt (history)           : (B, T, d)   rank index j contiguous over d
//   sample_sq, low_sq          : (B)
// One solver iteration = one `norm_decide` launch (per-sample ||gn||^2, batch-global norm,
// bookkeeping and break rules in the elected last block) + one `update` launch (rank-1
// update and next iterate).  The update kernel gives each sample to a thread-block CLUSTER:
// every CTA owns a contiguous slice of d, slices exchange their partial dot products through
// distributed shared memory, so no global atomics and a fixed summation order.
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace impflow {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxT = 63;

// ------------------------------------------------------------------------------------------
// per-sample ||g||^2 partials + last-block bookkeeping
// ------------------------------------------------------------------------------------------
__device__ void decide(impflow_broyden_state* st, double total, bool init) {
  const double obj = (double)(float)sqrt(total);  // torch.norm(...).item(): fp32 value as a python float
  st->objective = obj;
  if (init) {  // broyden.py:136-151
    st->nstep = 0;
    st->lowest_step = 0;
    st->init_objective = obj;
    st->lowest = obj;
    st->trace[0] = obj;
    st->prot_break = 0;
    st->converged = 0;
    st->stagnated = 0;
    st->do_update = 0;
    st->new_lowest = 0;
    st->active = (obj >= st->eps && 0 < st->threshold) ? 1 : 0;
    return;
  }
  const int T = st->threshold;
  const int nstep = st->nstep + 1;  // :155
  st->nstep = nstep;
  st->trace[nstep] = obj;           // :158
  int new_low = 0;
  if (obj < st->lowest) {           // :159-162
    st->lowest = obj;
    st->lowest_step = nstep;
    new_low = 1;
  }
  st->new_lowest = new_low;
  const int conv = obj < st->eps ? 1 : 0;  // :163
  int stag = 0;
  if (!conv && obj < 3.0 * st->eps && nstep == T) {  // :165-168, trace[-T:]
    double mx = st->trace[nstep - T + 1], mn = mx;
    for (int i = nstep - T + 1; i <= nstep; ++i) {
      mx = fmax(mx, st->trace[i]);
      mn = fmin(mn, st->trace[i]);
    }
    stag = (mx / mn < 1.3) ? 1 : 0;
  }
  int prot = 0;
  if (!conv && !stag && obj > st->init_objective * 1e6) prot = 1;  // :169-172
  st->converged = conv;
  st->stagnated = stag;
  st->prot_break = prot;
  const int upd = (conv || stag || prot) ? 0 : 1;
  st->do_update = upd;
  st->active = (upd && obj >= st->eps && nstep < T) ? 1 : 0;  // while-condition :153
}

// grid (S, B): CTA (s,b) reduces slice s of sample b.
__global__ void __launch_bounds__(kThreads)
k_norm_decide(const float* __restrict__ g, float* __restrict__ partial, float* __restrict__ sample_sq,
              float* __restrict__ low_sq, impflow_broyden_state* st, int B, long long d, int S, int init, int gated,
              BroydenProgress* progress) {
  // speculative iteration of the sync-free loop: the while-condition already failed on the device (uniform)
  if (gated && ((volatile impflow_broyden_state*)st)->active == 0) return;
  const int b = blockIdx.y, s = blockIdx.x;
  const long long chunk = (d + S - 1) / S;
  const long long lo = (long long)s * chunk;
  const long long hi = lo + chunk < d ? lo + chunk : d;
  const float* gp = g + (long long)b * d;
  float acc = 0.f;
  if (((d & 3) == 0) && ((chunk & 3) == 0)) {
    const float4* g4 = reinterpret_cast<const float4*>(gp);
    for (long long i = (lo >> 2) + threadIdx.x; i < (hi >> 2); i += kThreads) {
      const float4 v = g4[i];
      acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += kThreads) acc += gp[i] * gp[i];
  }
  __shared__ float wsum[kWarps];
  __shared__ double dsum[kWarps];
  __shared__ int is_last;
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kWarps; ++w) t += wsum[w];
    partial[(long long)b * S + s] = t;
    __threadfence();
    const int done = atomicAdd(&st->counter, 1);
    is_last = (done == S * B - 1) ? 1 : 0;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // elected block: fixed-order finalisation (deterministic)
  double tot = 0.0;
  for (int i = threadIdx.x; i < B; i += kThreads) {
    float t = 0.f;
    for (int k = 0; k < S; ++k) t += __ldcg(&partial[(long long)i * S + k]);
    sample_sq[i] = t;
    tot += (double)t;
  }
  tot = warp_sum_d(tot);
  if ((threadIdx.x & 31) == 0) dsum[threadIdx.x >> 5] = tot;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kWarps; ++w) t += dsum[w];
    st->counter = 0;
    decide(st, t, init != 0);
    __threadfence();
    if (progress != nullptr) {      // mapped pinned host memory: the host polls this record instead of syncing
      volatile BroydenProgress* pr = progress + st->nstep;
      pr->active = st->active;
      __threadfence_system();
      pr->seq = st->nstep;
      __threadfence_system();
    }
  }
  __syncthreads();
  if (init || ((volatile impflow_broyden_state*)st)->new_lowest) {
    for (int i = threadIdx.x; i < B; i += kThreads) low_sq[i] = sample_sq[i];
  }
}

// ------------------------------------------------------------------------------------------
// begin: low_x = x0, low_g = g0, xn = x0 - g0
// ------------------------------------------------------------------------------------------
__global__ void k_begin(const float* __restrict__ x0, const float* __restrict__ g0, float* __restrict__ xn,
                        float* __restrict__ low_x, float* __restrict__ low_g, long long n,
                        impflow_broyden_state* st, int threshold, double eps) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    st->threshold = threshold;
    st->eps = eps;
    st->counter = 0;
  }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const float x = x0[i], g = g0[i];
    low_x[i] = x;
    low_g[i] = g;
    xn[i] = x + (-g);
  }
}

// ------------------------------------------------------------------------------------------
// rank-1 update, cluster per sample.  VEC = 4 (float4 path, d % 4 == 0) or 1.  Two CTAs of 8 warps per SM.
// dynamic smem: sdx[SL] sdg[SL] sgn[SL] | wsum[3*T][kWarps] | part0[3*T] part1[2] | tot[3*T+2]
// ------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(kThreads, 2)
k_update(float* __restrict__ x_old, const float* __restrict__ g_old, const float* __restrict__ xn,
         const float* __restrict__ gn, float* __restrict__ Ut, float* __restrict__ Vt,
         float* __restrict__ low_x, float* __restrict__ low_g, const impflow_broyden_state* st, long long d,
         int T, int SL, int expect_nstep) {
  // local copies of the block shape: without them nvcc assigns two accumulators other registers than in the build
  // whose speed profiles/ records (same instructions, same register count)
  constexpr int kThreads = impflow::kThreads;
  constexpr int kWarps = impflow::kWarps;
  const int do_update = st->do_update;
  const int new_low = st->new_lowest;
  if (!do_update && !new_low) return;  // uniform over the whole grid
  if (expect_nstep >= 0 && st->nstep != expect_nstep) return;   // this iteration's decision kernel was gated off

  cg::cluster_group cluster = cg::this_cluster();
  const int C = cluster.num_blocks();
  const int r = cluster.block_rank();
  const int b = blockIdx.x / C;
  const int k = st->nstep - 1;  // history entries already stored = slot to write (:174)

  extern __shared__ __align__(16) float smem[];
  float* sdx = smem;
  float* sdg = sdx + SL;
  float* sgn = sdg + SL;
  float* wsum = sgn + SL;                 // [3*T][kWarps]
  float* part0 = wsum + 3 * T * kWarps;   // [3*T]
  float* part1 = part0 + 3 * T;           // [2]
  float* tot = part1 + 2;                 // [3*T + 2]

  const long long base = (long long)b * d + (long long)r * SL;
  long long rem = d - (long long)r * SL;
  const int len = rem <= 0 ? 0 : (rem < SL ? (int)rem : SL);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // ---- phase 0: deltas into smem, best-iterate copy (:159-162, :94-99) ----
  if (VEC == 4) {
    constexpr int UN = 4;       // 16 independent loads per thread in flight
    for (int i0 = tid * 4; i0 < len; i0 += kThreads * 4 * UN) {
      float4 xo[UN], xv[UN], go[UN], gv[UN];
#pragma unroll
      for (int q = 0; q < UN; ++q) {
        const int i = i0 + q * kThreads * 4;
        if (i < len) {
          xo[q] = *reinterpret_cast<const float4*>(x_old + base + i);
          xv[q] = *reinterpret_cast<const float4*>(xn + base + i);
          go[q] = *reinterpret_cast<const float4*>(g_old + base + i);
          gv[q] = *reinterpret_cast<const float4*>(gn + base + i);
        }
      }
#pragma unroll
      for (int q = 0; q < UN; ++q) {
        const int i = i0 + q * kThreads * 4;
        if (i < len) {
          *reinterpret_cast<float4*>(sdx + i) =
              make_float4(xv[q].x - xo[q].x, xv[q].y - xo[q].y, xv[q].z - xo[q].z, xv[q].w - xo[q].w);
          *reinterpret_cast<float4*>(sdg + i) =
              make_float4(gv[q].x - go[q].x, gv[q].y - go[q].y, gv[q].z - go[q].z, gv[q].w - go[q].w);
          *reinterpret_cast<float4*>(sgn + i) = gv[q];
          if (new_low) {
            *reinterpret_cast<float4*>(low_x + base + i) = xv[q];
            *reinterpret_cast<float4*>(low_g + base + i) = gv[q];
          }
        }
      }
    }
  }
  for (int i = tid * VEC; VEC != 4 && i < len; i += kThreads * VEC) {
    if (VEC == 4) {
    } else {
      const float xv = xn[base + i], gv = gn[base + i];
      sdx[i] = xv - x_old[base + i];
      sdg[i] = gv - g_old[base + i];
      sgn[i] = gv;
      if (new_low) {
        low_x[base + i] = xv;
        low_g[base + i] = gv;
      }
    }
  }
  if (!do_update) return;  // uniform
  __syncthreads();

  const float* Ub = Ut + (long long)b * T * d + (long long)r * SL;
  const float* Vb = Vt + (long long)b * T * d + (long long)r * SL;

  // ---- phase 1: a_j = dx.U_j, b_j = V_j.dg, c_j = V_j.gn for j < k (:108,:119) ----
  // Rows in DESCENDING order: phase 2 must accumulate in ascending order and then starts with the rows this pass
  // read last, which are still in L2 when the history in flight exceeds it (same-order passes over a working set
  // larger than the cache hit nothing).  The dots of different rows are independent: results unchanged.
  for (int j = k - 1; j >= 0; --j) {
    const float* uj = Ub + (long long)j * d;
    const float* vj = Vb + (long long)j * d;
    float a = 0.f, bb = 0.f, c = 0.f;
    if (VEC == 4) {
      // the kernel is bound by load latency, not by DRAM bytes: 16 independent 16-byte loads per thread in flight
      // (same per-thread summation order as a plain loop)
      constexpr int UN = 8;
      for (int i0 = tid * 4; i0 < len; i0 += kThreads * 4 * UN) {
        float4 u4[UN], v4[UN];
#pragma unroll
        for (int q = 0; q < UN; ++q) {
          const int i = i0 + q * kThreads * 4;
          if (i < len) {
            u4[q] = __ldg(reinterpret_cast<const float4*>(uj + i));
            v4[q] = __ldg(reinterpret_cast<const float4*>(vj + i));
          }
        }
#pragma unroll
        for (int q = 0; q < UN; ++q) {
          const int i = i0 + q * kThreads * 4;
          if (i < len) {
            const float4 dx = *reinterpret_cast<const float4*>(sdx + i);
            const float4 dg = *reinterpret_cast<const float4*>(sdg + i);
            const float4 gg = *reinterpret_cast<const float4*>(sgn + i);
            a += dx.x * u4[q].x + dx.y * u4[q].y + dx.z * u4[q].z + dx.w * u4[q].w;
            bb += v4[q].x * dg.x + v4[q].y * dg.y + v4[q].z * dg.z + v4[q].w * dg.w;
            c += v4[q].x * gg.x + v4[q].y * gg.y + v4[q].z * gg.z + v4[q].w * gg.w;
          }
        }
      }
    } else {
      for (int i = tid; i < len; i += kThreads) {
        const float u1 = uj[i], v1 = vj[i];
        a += sdx[i] * u1;
        bb += v1 * sdg[i];
        c += v1 * sgn[i];
      }
    }
    a = warp_sum(a);
    bb = warp_sum(bb);
    c = warp_sum(c);
    if (lane == 0) {
      wsum[(3 * j + 0) * kWarps + warp] = a;
      wsum[(3 * j + 1) * kWarps + warp] = bb;
      wsum[(3 * j + 2) * kWarps + warp] = c;
    }
  }
  __syncthreads();
  for (int t = tid; t < 3 * k; t += kThreads) {
    float s = 0.f;
    for (int w = 0; w < kWarps; ++w) s += wsum[t * kWarps + w];
    part0[t] = s;
  }
  cluster.sync();
  for (int t = tid; t < 3 * k; t += kThreads) {
    float s = 0.f;
    for (int q = 0; q < C; ++q) s += cluster.map_shared_rank(part0, q)[t];
    tot[t] = s;
  }
  __syncthreads();

  // ---- phase 2: vT, w = matvec(dg), S = sum_j c_j U_j; den = vT.dg, c_k = vT_scrubbed.gn ----
  float den = 0.f, ck = 0.f;
  float* vk = Vt + (long long)b * T * d + (long long)k * d + (long long)r * SL;
  for (int i = tid * VEC; i < len; i += kThreads * VEC) {
    float dx[VEC], dg[VEC], gg[VEC], vT[VEC], w[VEC], S[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      dx[e] = sdx[i + e];
      dg[e] = sdg[i + e];
      gg[e] = sgn[i + e];
      vT[e] = -dx[e];
      w[e] = -dg[e];
      S[e] = 0.f;
    }
    int j = 0;
    if (VEC == 4) {
      constexpr int UJ = 8;       // 16 independent loads in flight per thread; accumulation order over j unchanged
      for (; j + UJ <= k; j += UJ) {
        float4 u4[UJ], v4[UJ];
#pragma unroll
        for (int q = 0; q < UJ; ++q) {
          u4[q] = __ldg(reinterpret_cast<const float4*>(Ub + (long long)(j + q) * d + i));
          v4[q] = __ldg(reinterpret_cast<const float4*>(Vb + (long long)(j + q) * d + i));
        }
#pragma unroll
        for (int q = 0; q < UJ; ++q) {
          const float aj = tot[3 * (j + q) + 0], bj = tot[3 * (j + q) + 1], cj = tot[3 * (j + q) + 2];
          const float u1[4] = {u4[q].x, u4[q].y, u4[q].z, u4[q].w};
          const float v1[4] = {v4[q].x, v4[q].y, v4[q].z, v4[q].w};
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            vT[e] += aj * v1[e % 4];
            w[e] += bj * u1[e % 4];
            S[e] += cj * u1[e % 4];
          }
        }
      }
    }
    for (; j < k; ++j) {
      float u1[VEC], v1[VEC];
      if (VEC == 4) {
        const float4 u4 = __ldg(reinterpret_cast<const float4*>(Ub + (long long)j * d + i));
        const float4 v4 = __ldg(reinterpret_cast<const float4*>(Vb + (long long)j * d + i));
        u1[0] = u4.x; u1[1 % VEC] = u4.y; u1[2 % VEC] = u4.z; u1[3 % VEC] = u4.w;
        v1[0] = v4.x; v1[1 % VEC] = v4.y; v1[2 % VEC] = v4.z; v1[3 % VEC] = v4.w;
      } else {
        u1[0] = __ldg(Ub + (long long)j * d + i);
        v1[0] = __ldg(Vb + (long long)j * d + i);
      }
      const float aj = tot[3 * j + 0], bj = tot[3 * j + 1], cj = tot[3 * j + 2];
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        vT[e] += aj * v1[e];
        w[e] += bj * u1[e];
        S[e] += cj * u1[e];
      }
    }
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      den += vT[e] * dg[e];                          // unscrubbed vT in the denominator (:176)
      vT[e] = (vT[e] != vT[e]) ? 0.f : vT[e];        // :177
      ck += vT[e] * gg[e];
      sdx[i + e] = dx[e] - w[e];                     // numerator of u
      sdg[i + e] = S[e];
    }
    if (VEC == 4) {
      *reinterpret_cast<float4*>(vk + i) = make_float4(vT[0], vT[1 % VEC], vT[2 % VEC], vT[3 % VEC]);  // :179
    } else {
      vk[i] = vT[0];
    }
  }
  den = warp_sum(den);
  ck = warp_sum(ck);
  if (lane == 0) {
    wsum[warp] = den;
    wsum[kWarps + warp] = ck;
  }
  __syncthreads();
  if (tid < 2) {
    float s = 0.f;
    for (int w = 0; w < kWarps; ++w) s += wsum[tid * kWarps + w];
    part1[tid] = s;
  }
  cluster.sync();
  if (tid < 2) {
    float s = 0.f;
    for (int q = 0; q < C; ++q) s += cluster.map_shared_rank(part1, q)[tid];
    tot[3 * T + tid] = s;
  }
  __syncthreads();
  const float den_t = tot[3 * T + 0], ck_t = tot[3 * T + 1];

  // ---- phase 3: u (scrub), next direction and next iterate (:176-181, :90) ----
  float* uk = Ut + (long long)b * T * d + (long long)k * d + (long long)r * SL;
  constexpr int U3 = 8;       // VEC == 4: the iterate is fetched 8 groups ahead (one round of load latency per slice)
  float4 xpre[U3];
  for (int i = tid * VEC, it = 0; i < len; i += kThreads * VEC, ++it) {
    float u[VEC], xnext[VEC], xv[VEC];
    if (VEC == 4) {
      if ((it % U3) == 0) {
#pragma unroll
        for (int q = 0; q < U3; ++q) {
          const int iq = i + q * kThreads * 4;
          if (iq < len) xpre[q] = *reinterpret_cast<const float4*>(xn + base + iq);
        }
      }
      float4 x4 = xpre[0];
#pragma unroll
      for (int q = 1; q < U3; ++q) x4 = ((it % U3) == q) ? xpre[q] : x4;
      xv[0] = x4.x; xv[1 % VEC] = x4.y; xv[2 % VEC] = x4.z; xv[3 % VEC] = x4.w;
    } else {
      xv[0] = xn[base + i];
    }
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      float q = sdx[i + e] / den_t;
      q = (q != q) ? 0.f : q;                        // :178
      u[e] = q;
      const float upd = -((-sgn[i + e]) + (sdg[i + e] + q * ck_t));  // -matvec(U[:nstep], V[:nstep], gx) :181
      xnext[e] = xv[e] + upd;
    }
    if (VEC == 4) {
      *reinterpret_cast<float4*>(uk + i) = make_float4(u[0], u[1 % VEC], u[2 % VEC], u[3 % VEC]);   // :180
      *reinterpret_cast<float4*>(x_old + base + i) =
          make_float4(xnext[0], xnext[1 % VEC], xnext[2 % VEC], xnext[3 % VEC]);
    } else {
      uk[i] = u[0];
      x_old[base + i] = xnext[0];
    }
  }
  cluster.sync();  // peers may still be reading part1 through DSMEM
}

// small-d variant: one warp per sample, d <= 128 (toy / tabular shapes).
__global__ void __launch_bounds__(kThreads)
k_update_small(float* __restrict__ x_old, const float* __restrict__ g_old, const float* __restrict__ xn,
               const float* __restrict__ gn, float* __restrict__ Ut, float* __restrict__ Vt,
               float* __restrict__ low_x, float* __restrict__ low_g, const impflow_broyden_state* st, int B,
               int d, int T, int expect_nstep) {
  const int do_update = st->do_update;
  const int new_low = st->new_lowest;
  if (!do_update && !new_low) return;
  if (expect_nstep >= 0 && st->nstep != expect_nstep) return;
  const int b = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (b >= B) return;
  const int lane = threadIdx.x & 31;
  const int k = st->nstep - 1;
  const long long base = (long long)b * d;
  float dx[4], dg[4], gg[4], xv[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int i = lane + 32 * e;
    if (i < d) {
      xv[e] = xn[base + i];
      gg[e] = gn[base + i];
      dx[e] = xv[e] - x_old[base + i];
      dg[e] = gg[e] - g_old[base + i];
      if (new_low) {
        low_x[base + i] = xv[e];
        low_g[base + i] = gg[e];
      }
    } else {
      xv[e] = gg[e] = dx[e] = dg[e] = 0.f;
    }
  }
  if (!do_update) return;
  const float* Ub = Ut + (long long)b * T * d;
  const float* Vb = Vt + (long long)b * T * d;
  float vT[4], w[4], S[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    vT[e] = -dx[e];
    w[e] = -dg[e];
    S[e] = 0.f;
  }
  for (int j = 0; j < k; ++j) {
    float u1[4], v1[4], a = 0.f, bb = 0.f, c = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int i = lane + 32 * e;
      u1[e] = i < d ? Ub[(long long)j * d + i] : 0.f;
      v1[e] = i < d ? Vb[(long long)j * d + i] : 0.f;
      a += dx[e] * u1[e];
      bb += v1[e] * dg[e];
      c += v1[e] * gg[e];
    }
    a = warp_sum(a);
    bb = warp_sum(bb);
    c = warp_sum(c);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      vT[e] += a * v1[e];
      w[e] += bb * u1[e];
      S[e] += c * u1[e];
    }
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
      Ut[(long long)b * T * d + (long long)k * d + i] = u;
      Vt[(long long)b * T * d + (long long)k * d + i] = vT[e];
      const float upd = -((-gg[e]) + (S[e] + u * ck));
      x_old[base + i] = xv[e] + upd;
    }
  }
}

static int pick_splits(int B, long long d) {
  int S = 1;
  while ((long long)B * S < 592 && d / (S * 2) >= 2048 && S < 64) S *= 2;
  return S;
}

static void pick_cluster(int B, long long d, int* C_out, int* SL_out) {
  const int kMaxSlice = 8192;
  int C = 1;
  while (C < 8 && (d + C - 1) / C > kMaxSlice) C *= 2;
  while (C < 8 && (long long)B * C < 296 && (d / (C * 2)) >= 512) C *= 2;
  long long sl = (d + C - 1) / C;
  sl = (sl + 3) / 4 * 4;
  *C_out = C;
  *SL_out = (int)sl;
}

}  // namespace impflow

using namespace impflow;

extern "C" size_t impflow_broyden_state_bytes(void) { return sizeof(impflow_broyden_state); }

extern "C" size_t impflow_broyden_workspace_floats(int B, long long d, int threshold) {
  (void)threshold;
  return (size_t)B * 64;
}

static int launch_norm(const float* g, float* partial, float* sample_sq, float* low_sq,
                       impflow_broyden_state* state, int B, long long d, int init, int gated,
                       BroydenProgress* progress, cudaStream_t s);

extern "C" int impflow_broyden_begin(const float* x0, const float* g0, float* xn, float* low_x, float* low_g,
                                     float* sample_sq, float* low_sq, float* partial,
                                     impflow_broyden_state* state, int B, long long d, int threshold,
                                     double eps_scaled, void* stream) {
  return broyden_begin_ex(x0, g0, xn, low_x, low_g, sample_sq, low_sq, partial, state, B, d, threshold, eps_scaled,
                          nullptr, stream);
}

int impflow::broyden_begin_ex(const float* x0, const float* g0, float* xn, float* low_x, float* low_g,
                              float* sample_sq, float* low_sq, float* partial, impflow_broyden_state* state, int B,
                              long long d, int threshold, double eps_scaled, BroydenProgress* progress,
                              void* stream) {
  IMPFLOW_REQUIRE(threshold >= 1 && threshold <= kMaxT, "broyden: threshold %d not in [1,%d]", threshold, kMaxT);
  IMPFLOW_REQUIRE(B >= 1 && d >= 1, "broyden: empty problem B=%d d=%lld", B, d);
  cudaStream_t s = (cudaStream_t)stream;
  const long long n = (long long)B * d;
  int blocks = (int)((n + 1023) / 1024);
  if (blocks > 148 * 8) blocks = 148 * 8;
  k_begin<<<blocks, 256, 0, s>>>(x0, g0, xn, low_x, low_g, n, state, threshold, eps_scaled);
  if (check_launch("k_begin")) return -1;
  return launch_norm(g0, partial, sample_sq, low_sq, state, B, d, 1, 0, progress, s);
}

static int launch_norm(const float* g, float* partial, float* sample_sq, float* low_sq,
                       impflow_broyden_state* state, int B, long long d, int init, int gated,
                       BroydenProgress* progress, cudaStream_t s) {
  const int S = pick_splits(B, d);
  dim3 grid(S, B);
  k_norm_decide<<<grid, kThreads, 0, s>>>(g, partial, sample_sq, low_sq, state, B, d, S, init, gated, progress);
  return check_launch("k_norm_decide");
}

extern "C" int impflow_broyden_step(float* x_old, const float* g_old, const float* xn, const float* gn,
                                    float* Ut, float* Vt, float* low_x, float* low_g, float* sample_sq,
                                    float* low_sq, float* partial, impflow_broyden_state* state, int B,
                                    long long d, int threshold, void* stream) {
  return broyden_step_ex(x_old, g_old, xn, gn, Ut, Vt, low_x, low_g, sample_sq, low_sq, partial, state, B, d,
                         threshold, 0, -1, nullptr, stream);
}

int impflow::broyden_step_ex(float* x_old, const float* g_old, const float* xn, const float* gn, float* Ut,
                             float* Vt, float* low_x, float* low_g, float* sample_sq, float* low_sq, float* partial,
                             impflow_broyden_state* state, int B, long long d, int threshold, int gated,
                             int expect_nstep, BroydenProgress* progress, void* stream) {
  IMPFLOW_REQUIRE(threshold >= 1 && threshold <= kMaxT, "broyden: threshold %d not in [1,%d]", threshold, kMaxT);
  cudaStream_t s = (cudaStream_t)stream;
  if (launch_norm(gn, partial, sample_sq, low_sq, state, B, d, 0, gated, progress, s)) return -1;
  if (d <= 128) {
    const int blocks = (B + kWarps - 1) / kWarps;
    k_update_small<<<blocks, kThreads, 0, s>>>(x_old, g_old, xn, gn, Ut, Vt, low_x, low_g, state, B, (int)d,
                                               threshold, expect_nstep);
    return check_launch("k_update_small");
  }
  IMPFLOW_REQUIRE(d <= 8LL * 8192, "broyden: d=%lld exceeds the cluster kernel limit 65536", d);
  int C, SL;
  pick_cluster(B, d, &C, &SL);
  // wsum is sized for 16 warps although k_update runs 8: the bytes bound how many CTAs share an SM, so shrinking
  // them is a performance change of its own
  const size_t smem = sizeof(float) * ((size_t)3 * SL + (size_t)3 * threshold * 16 + 3 * threshold + 2 +
                                       3 * threshold + 2 + 8);
  // The two-pass kernel is kept on purpose: read-once variants (history streamed through a bulk-copy ring, or walked
  // in L2-sized row chunks) were measured slower, 512-thread / L1-bypassing ones within a few per cent and not adopted
  // (profiles/r02_update_bench.txt; their source is in commits de6f192 and 74f3be3).
  void (*kern)(float*, const float*, const float*, const float*, float*, float*, float*, float*,
               const impflow_broyden_state*, long long, int, int, int) = d % 4 == 0 ? k_update<4> : k_update<1>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    set_error("broyden_step: cannot set %zu bytes of dynamic shared memory", smem);
    return -1;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(B * C));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, x_old, g_old, xn, gn, Ut, Vt, low_x, low_g,
                                     (const impflow_broyden_state*)state, d, threshold, SL, expect_nstep);
  if (e != cudaSuccess) {
    set_error("broyden_step: cluster launch failed: %s", cudaGetErrorString(e));
    return -1;
  }
  return check_launch("k_update");
}
