// Fused layers 2 + 3 of the 3x3 / 1x1 / 3x3 conv residual branch at the WIDER scales of the image flows
// (implicit_flow.py:359-398 with c = 12 / 48 narrow channels: 9c = 108 / 432 tap columns) — forward or transposed
// (vjp) — in ONE launch:
//
//     H  = A1 W2^T                  [M,C] x [C,C]^T        A1 = tf32 hi/lo planes written by the layer-1 GEMM
//     A2 = psi2(H)                  bias + activation (forward)  |  H * D (D = act'(pre), vjp)
//     Y_q = A2[:, q] W3[:, q]^T     [M,128] x [N3,128]^T   partial sums over the 128-channel quarter q of layer 2
//
// The narrow side is too wide for the all-in-tensor-memory scheme of branch_fused.cu (the im2col row alone would
// need 2 * 9c columns), so layer 1 stays a GEMM of its own and this kernel removes the other two launches together
// with the C-wide intermediate between them (67 MB of hi/lo planes per evaluation at c = 12, B = 64) and the
// N = 108 / 432 GEMMs that ran at 45-55 TFLOP/s.
//
// Work item = (128-row tile, 128-channel quarter q of layer 2's output); persistent, one CTA per SM.
// Tensor memory (512 columns):  [0,128) ACC2 | [128,256) A2 hi | [256,384) A2 lo | [384,512) ACC3
//   phase A  (tensor pipe): ACC2 = A1[tile] W2[q]^T, both operands streamed by TMA through a 3-stage 64 KB ring
//   transform (16 warps)  : ACC2 -> psi2 -> tf32 hi/lo -> A2 (stays in tensor memory; pre2_out optional)
//   phase B  (tensor pipe): for every pass of <= 128 tap columns: ACC3 = A2 W3[pass, q]^T (A from tensor memory,
//                           W3 chunks through the same ring), read back by the 16 warps into the partial Y_q
// Operand traffic: a single CTA pulls 64 KB (A1 chunk + W2 chunk) through L2 per 768 tensor-pipe cycles, twice
// what the L2 delivers to every SM at once.  Sharing the A1 chunk among the four quarter-CTAs of a row tile by TMA
// multicast was measured slower (91 vs 123 TFLOP/s, DESIGN.md §4) and removed.
// The Q = C/128 partials are summed in fixed order by the col2im kernel that follows (k_conv3_out), so the result
// does not depend on the order in which the quarters finish.  Everything is fp32-accurate 3xTF32.
#include "tile_common.cuh"

namespace impflow {

constexpr int C23_NS = 3;
constexpr int C23_PLANE = 128 * TC_BK * 4;            // 16 KB: 128 rows x 32 fp32
constexpr int C23_STAGE_BYTES = 4 * C23_PLANE;        // A hi | A lo | B hi | B lo
constexpr int C23_SMEM_BYTES = C23_NS * C23_STAGE_BYTES + 1024 + 256;
constexpr int C23_THREADS = 128 + 32 * BF_XF_WARPS;
constexpr uint32_t C23_COL_ACC2 = 0, C23_COL_A2HI = 128, C23_COL_A2LO = 256, C23_COL_ACC3 = 384;

// round to nearest, ties away (= cvt.rna.tf32.f32 for finite values) in two full-rate integer ops - the same
// expression as the GEMM epilogue's split, so both routes give the layer-2 MMAs bit-identical operands
__device__ __forceinline__ void split_tf32_c23(float v, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
  lo = v - hi;
}

struct Chain23Args {
  const float* bias2;    // [C] or null
  const float* mul2;     // [M, C] or null: psi2 = H * mul2
  float* pre2_out;       // [M, C] or null
  float* out;            // partials [Q][M][ldo]
  long long ldo;
  long long part_stride; // floats between two partials
  long long M;
  int C;
  int N3;
  int npass;             // ceil(N3 / 128)
  int PW;                // MMA N of a pass: 128, or N3 rounded up to 16 when npass == 1
  const float* beta2;
  const int* gate;
};

// A32: the layer-2 input arrives as ONE plain fp32 plane (what the layer-1 GEMM writes with half the bytes); warps 2
// and 3 split every landed chunk into tf32 hi / lo planes in shared memory (round-to-nearest hi in place, lo = a - hi
// beside it) before the MMAs read it.  A CTA then pulls 48 KB instead of 64 KB through L2 per K chunk - the stream that
// bounds this kernel - and the layer-1 GEMM's epilogue writes 4 instead of 8 bytes per element.
template <int ACT, bool A32>
__global__ void __launch_bounds__(C23_THREADS, 1)
k_chain23(const __grid_constant__ CUtensorMap mapAhi, const __grid_constant__ CUtensorMap mapAlo,
          const __grid_constant__ CUtensorMap mapW2hi, const __grid_constant__ CUtensorMap mapW2lo,
          const __grid_constant__ CUtensorMap mapW3hi, const __grid_constant__ CUtensorMap mapW3lo,
          const Chain23Args args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C23_NS * C23_STAGE_BYTES);
  uint64_t* full = bars;                    // [NS] TMA -> MMA
  uint64_t* empty = full + C23_NS;          // [NS] MMA -> TMA
  uint64_t* acc2_full = empty + C23_NS;     // MMA -> transform
  uint64_t* acc2_empty = acc2_full + 1;     // transform -> MMA (ACC2 read out)
  uint64_t* a2_full = acc2_empty + 1;       // transform -> MMA (A2 written)
  uint64_t* a2_empty = a2_full + 1;         // MMA -> transform (phase B retired: A2 may be overwritten)
  uint64_t* acc3_full = a2_empty + 1;       // MMA -> epilogue
  uint64_t* acc3_empty = acc3_full + 1;     // epilogue -> MMA
  uint64_t* ready = acc3_empty + 1;         // [NS] split warps -> MMA (A32: hi / lo planes of the stage are in place)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ready + C23_NS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int NC = args.C / TC_BK;            // K chunks of layer 2
  const int Q = args.C / 128;               // quarters (items per row tile)
  const int NC3 = 128 / TC_BK;              // K chunks of layer 3 per item
  const long long m_tiles = (args.M + TC_BM - 1) / TC_BM;
  long long num_items = m_tiles * Q;

  pdl_trigger();
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapAhi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapAlo)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapW2hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapW2lo)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapW3hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapW3lo)) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C23_NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
      mbar_init(&ready[s], 2);               // warps 2 and 3
    }
    mbar_init(acc2_full, 1);
    mbar_init(acc2_empty, BF_XF_WARPS);
    mbar_init(a2_full, BF_XF_WARPS);
    mbar_init(a2_empty, 1);
    mbar_init(acc3_full, 1);
    mbar_init(acc3_empty, BF_XF_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();        // the set-up above overlapped the predecessor (the layer-1 GEMM); no global memory touched yet
  if (gate_closed(args.gate)) num_items = 0;   // speculative solver iteration after the loop ended (uniform)

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      uint32_t gw = 0;
      for (long long item = blockIdx.x; item < num_items; item += gridDim.x) {
        const int q = (int)(item % Q);
        const int m0 = (int)(item / Q) * TC_BM;
        for (int kc = 0; kc < NC; ++kc, ++gw) {
          const int st = gw % C23_NS;
          mbar_wait(&empty[st], ((gw / C23_NS) & 1) ^ 1);
          uint8_t* sp = smem + st * C23_STAGE_BYTES;
          mbar_expect_tx(&full[st], A32 ? 3 * C23_PLANE : C23_STAGE_BYTES);
          if (A32) {     // one fp32 plane; the lo plane of the stage is produced on chip
            tma_load_2d(&mapAhi, &full[st], sp, kc * TC_BK, m0);
          } else {
            tma_load_2d(&mapAhi, &full[st], sp, kc * TC_BK, m0);
            tma_load_2d(&mapAlo, &full[st], sp + C23_PLANE, kc * TC_BK, m0);
          }
          tma_load_2d(&mapW2hi, &full[st], sp + 2 * C23_PLANE, kc * TC_BK, q * 128);
          tma_load_2d(&mapW2lo, &full[st], sp + 3 * C23_PLANE, kc * TC_BK, q * 128);
        }
        for (int j = 0; j < args.npass; ++j) {
          for (int c2 = 0; c2 < NC3; ++c2, ++gw) {
            const int st = gw % C23_NS;
            mbar_wait(&empty[st], ((gw / C23_NS) & 1) ^ 1);
            uint8_t* sp = smem + st * C23_STAGE_BYTES;
            mbar_expect_tx(&full[st], 2 * C23_PLANE);
            tma_load_2d(&mapW3hi, &full[st], sp + 2 * C23_PLANE, q * 128 + c2 * TC_BK, j * 128);
            tma_load_2d(&mapW3lo, &full[st], sp + 3 * C23_PLANE, q * 128 + c2 * TC_BK, j * 128);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    const uint32_t idesc_base = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TC_BM >> 4) << 24);
    const uint32_t idesc2 = idesc_base | ((uint32_t)(128 >> 3) << 17);
    const uint32_t idesc3 = idesc_base | ((uint32_t)(args.PW >> 3) << 17);
    const uint32_t t_acc2 = tmem_base + C23_COL_ACC2;
    const uint32_t t_a2hi = tmem_base + C23_COL_A2HI;
    const uint32_t t_a2lo = tmem_base + C23_COL_A2LO;
    const uint32_t t_acc3 = tmem_base + C23_COL_ACC3;
    uint32_t gw = 0, gp = 0, it = 0;
    for (long long item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      // ---- phase A: layer 2 into ACC2 (free once the previous item's transform has read it)
      if (it > 0) mbar_wait(acc2_empty, (it - 1) & 1);
      tc_fence_after();
      for (int kc = 0; kc < NC; ++kc, ++gw) {
        const uint32_t st = gw % C23_NS;
        mbar_wait(A32 ? &ready[st] : &full[st], (gw / C23_NS) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_hi = smem_u32(smem + st * C23_STAGE_BYTES);
          const uint32_t a_lo = a_hi + C23_PLANE;
          const uint32_t b_hi = a_hi + 2 * C23_PLANE;
          const uint32_t b_lo = a_hi + 3 * C23_PLANE;
#pragma unroll
          for (int k = 0; k < TC_BK / 8; ++k) {
            const uint64_t dah = make_kmajor_sw128_desc(a_hi + k * 32);
            const uint64_t dal = make_kmajor_sw128_desc(a_lo + k * 32);
            const uint64_t dbh = make_kmajor_sw128_desc(b_hi + k * 32);
            const uint64_t dbl = make_kmajor_sw128_desc(b_lo + k * 32);
            umma_tf32(t_acc2, dal, dbh, idesc2, (kc != 0 || k != 0) ? 1u : 0u);   // lo * hi
            umma_tf32(t_acc2, dah, dbl, idesc2, 1u);                               // hi * lo
            umma_tf32(t_acc2, dah, dbh, idesc2, 1u);                               // hi * hi
          }
          umma_commit(&empty[st]);
          if (kc == NC - 1) umma_commit(acc2_full);
        }
        __syncwarp();
      }
      // ---- phase B: layer 3, A operand = the transformed accumulator kept in tensor memory
      mbar_wait(a2_full, it & 1);
      tc_fence_after();
      for (int j = 0; j < args.npass; ++j, ++gp) {
        if (gp > 0) mbar_wait(acc3_empty, (gp - 1) & 1);
        tc_fence_after();
        for (int c2 = 0; c2 < NC3; ++c2, ++gw) {
          const uint32_t st = gw % C23_NS;
          mbar_wait(A32 ? &ready[st] : &full[st], (gw / C23_NS) & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t b_hi = smem_u32(smem + st * C23_STAGE_BYTES + 2 * C23_PLANE);
            const uint32_t b_lo = b_hi + C23_PLANE;
#pragma unroll
            for (int k = 0; k < TC_BK / 8; ++k) {
              const uint64_t dbh = make_kmajor_sw128_desc(b_hi + k * 32);
              const uint64_t dbl = make_kmajor_sw128_desc(b_lo + k * 32);
              const uint32_t col = c2 * TC_BK + k * 8;
              umma_tf32_ts(t_acc3, t_a2lo + col, dbh, idesc3, (c2 != 0 || k != 0) ? 1u : 0u);
              umma_tf32_ts(t_acc3, t_a2hi + col, dbl, idesc3, 1u);
              umma_tf32_ts(t_acc3, t_a2hi + col, dbh, idesc3, 1u);
            }
            umma_commit(&empty[st]);
            if (c2 == NC3 - 1) {
              umma_commit(acc3_full);
              if (j == args.npass - 1) umma_commit(a2_empty);
            }
          }
          __syncwarp();
        }
      }
    }
  } else if (A32 && (warp == 2 || warp == 3)) {
    // ================= split warps: fp32 A chunk -> tf32 hi / lo planes, in shared memory =================
    uint32_t gw = 0;
    for (long long item = blockIdx.x; item < num_items; item += gridDim.x) {
      for (int kc = 0; kc < NC; ++kc, ++gw) {
        const uint32_t st = gw % C23_NS;
        mbar_wait(&full[st], (gw / C23_NS) & 1);
        float4* ph = reinterpret_cast<float4*>(smem + st * C23_STAGE_BYTES);
        float4* pl = ph + C23_PLANE / 16;
#pragma unroll 4
        for (int i = (warp - 2) * 32 + lane; i < C23_PLANE / 16; i += 64) {
          const float4 v = ph[i];
          float4 h, l;
          split_tf32_c23(v.x, h.x, l.x);
          split_tf32_c23(v.y, h.y, l.y);
          split_tf32_c23(v.z, h.z, l.z);
          split_tf32_c23(v.w, h.w, l.w);
          ph[i] = h;
          pl[i] = l;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> the MMA's async proxy
        __syncwarp();
        if (lane == 0) mbar_arrive(&ready[st]);
      }
      for (int u = 0; u < args.npass * NC3; ++u, ++gw) {     // layer-3 stages carry weights only: pass them on
        const uint32_t st = gw % C23_NS;
        mbar_wait(&full[st], (gw / C23_NS) & 1);
        if (lane == 0) mbar_arrive(&ready[st]);
      }
    }
  } else if (warp >= 4) {
    // ================= transform / epilogue warps =================
    const int ql = warp & 3;                    // TMEM lane quarter
    const int grp = (warp - 4) >> 2;            // 0..3
    const int cw0 = grp * BF_CW;                // this warp's columns inside a 32-column chunk (transform)
    const uint32_t lane_base = (uint32_t)(ql * 32) << 16;
    const float beta2 = args.beta2 != nullptr ? __ldg(args.beta2) : 0.f;
    const float nbl2 = -1.4426950408889634f * beta2;
    const bool has_mul2 = args.mul2 != nullptr;
    const int C = args.C;
    uint32_t gp = 0, it = 0;
    for (long long item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int q = (int)(item % Q);
      const long long m = (item / Q) * TC_BM + ql * 32 + lane;
      const bool valid = m < args.M;
      uint32_t hi[BF_CW], lo[BF_CW];
      float a[BF_CW], mul[BF_CW];
      // the multiplier rows of the first chunk are fetched while layer 2 still runs
      if (has_mul2) {
        if (valid) ld8(args.mul2 + m * C + q * 128 + cw0, mul);
        else {
#pragma unroll
          for (int j = 0; j < BF_CW; ++j) mul[j] = 0.f;
        }
      }
      mbar_wait(acc2_full, it & 1);
      if (it > 0) mbar_wait(a2_empty, (it - 1) & 1);
      tc_fence_after();
      for (int c2 = 0; c2 < NC3; ++c2) {
        const int n0 = q * 128 + c2 * TC_BK + cw0;
        uint32_t r[BF_CW];
        tmem_ld8(tmem_base + lane_base + C23_COL_ACC2 + c2 * TC_BK + cw0, r);
        psi8<ACT>(r, a, args.bias2 != nullptr ? args.bias2 + n0 : nullptr, mul, has_mul2,
                  args.pre2_out != nullptr ? args.pre2_out + m * C + n0 : nullptr, args.pre2_out != nullptr && valid,
                  beta2, nbl2);
        if (has_mul2 && c2 + 1 < NC3) {
          if (valid) ld8(args.mul2 + m * C + n0 + TC_BK, mul);
        }
        split8(a, hi, lo);
        tmem_st8(tmem_base + lane_base + C23_COL_A2HI + c2 * TC_BK + cw0, hi);
        tmem_st8(tmem_base + lane_base + C23_COL_A2LO + c2 * TC_BK + cw0, lo);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(acc2_empty);
        mbar_arrive(a2_full);
      }
      // ---- layer-3 accumulator of every pass -> partial Y_q: warp group `grp` owns columns [32 grp, 32 grp + 32)
      float* out_q = args.out + (long long)q * args.part_stride;
      for (int j = 0; j < args.npass; ++j, ++gp) {
        mbar_wait(acc3_full, gp & 1);
        tc_fence_after();
        const int col0 = j * 128 + grp * 32;
        const bool any = grp * 32 < args.PW && col0 < args.N3;     // columns the MMA really wrote and the problem has
        uint32_t r[32];
        if (any) tmem_ld32(tmem_base + lane_base + C23_COL_ACC3 + grp * 32, r);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc3_empty);
        if (any && valid) {
          float* dst = out_q + m * args.ldo + col0;
          const int nvalid = args.N3 - col0 < 32 ? args.N3 - col0 : 32;
          if (nvalid == 32 && ((reinterpret_cast<uintptr_t>(dst) & 31) == 0)) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float v[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(r[8 * g + e]);
              st_global_v8(dst + 8 * g, v);
            }
          } else {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (e < nvalid) dst[e] = __uint_as_float(r[e]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

template <int ACT, bool A32>
static int launch_chain23(const CUtensorMap* maps, const Chain23Args& a, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(k_chain23<ACT, A32>, cudaFuncAttributeMaxDynamicSharedMemorySize, C23_SMEM_BYTES) !=
        cudaSuccess) {
      set_error("chain23_tc: cannot set %d bytes of dynamic shared memory", C23_SMEM_BYTES);
      return -1;
    }
    attr_set = true;
  }
  const long long items = ((a.M + TC_BM - 1) / TC_BM) * (a.C / 128);
  const int grid = (int)(items < 148 ? items : 148);     // persistent: at most one CTA per SM
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(C23_THREADS);
  cfg.dynamicSmemBytes = C23_SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  cfg.attrs = attr;
  cfg.numAttrs = pdl_attr(&attr[0]);
  const cudaError_t err = cudaLaunchKernelEx(&cfg, k_chain23<ACT, A32>, maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], a);
  if (err != cudaSuccess) {
    set_error("k_chain23: launch failed: %s", cudaGetErrorString(err));
    return -1;
  }
  return check_launch("k_chain23");
}

}  // namespace impflow

using namespace impflow;

extern "C" int impflow_chain23_parts(int C) { return C / 128; }

extern "C" int impflow_chain23_tc(const float* A_hi, const float* A_lo, long long lda, const float* W2_hi,
                                  const float* W2_lo, const float* W3_hi, const float* W3_lo, const float* bias2,
                                  const float* mul2, float* pre2_out, float* out, long long ldo, long long part_stride,
                                  long long M, int C, int N3, int act_kind, const float* beta2, void* stream) {
  IMPFLOW_REQUIRE(M >= 1 && C >= 128 && N3 >= 1, "chain23_tc: empty problem M=%lld C=%d N3=%d", M, C, N3);
  if (C % 128 != 0 || lda < C || (lda % 4) != 0 || ldo < N3 || part_stride < M * ldo) {
    set_error("chain23_tc: needs C %% 128 == 0, 16-byte aligned rows and room for C/128 partials (C=%d lda=%lld "
              "ldo=%lld part_stride=%lld)", C, lda, ldo, part_stride);
    return -2;
  }
  IMPFLOW_REQUIRE(A_hi != nullptr, "chain23_tc: A missing");
  const uintptr_t al = reinterpret_cast<uintptr_t>(A_hi) | reinterpret_cast<uintptr_t>(A_lo) |
                       reinterpret_cast<uintptr_t>(W2_hi) | reinterpret_cast<uintptr_t>(W2_lo) |
                       reinterpret_cast<uintptr_t>(W3_hi) | reinterpret_cast<uintptr_t>(W3_lo) |
                       reinterpret_cast<uintptr_t>(mul2) | reinterpret_cast<uintptr_t>(pre2_out) |
                       reinterpret_cast<uintptr_t>(bias2);
  if (al & 15) {
    set_error("chain23_tc: operand base pointers must be 16-byte aligned");
    return -2;
  }
  const bool a32 = A_lo == nullptr;              // one fp32 plane, split on chip
  CUtensorMap maps[6];
  if (make_map(&maps[0], A_hi, M, C, lda, 128) || make_map(&maps[1], a32 ? A_hi : A_lo, M, C, lda, 128) ||
      make_map(&maps[2], W2_hi, C, C, C, 128) || make_map(&maps[3], W2_lo, C, C, C, 128) ||
      make_map(&maps[4], W3_hi, N3, C, C, 128) || make_map(&maps[5], W3_lo, N3, C, C, 128))
    return -1;
  Chain23Args a;
  memset(&a, 0, sizeof(a));
  a.bias2 = bias2, a.mul2 = mul2, a.pre2_out = pre2_out, a.out = out, a.ldo = ldo, a.part_stride = part_stride;
  a.M = M, a.C = C, a.N3 = N3;
  a.npass = (N3 + 127) / 128;
  a.PW = a.npass == 1 ? (N3 + 15) / 16 * 16 : 128;
  a.beta2 = beta2;
  a.gate = g_gate;
  cudaStream_t s = (cudaStream_t)stream;
  if (a32) {
    switch (act_kind) {
      case IMPFLOW_ACT_LIPSWISH: return launch_chain23<IMPFLOW_ACT_LIPSWISH, true>(maps, a, s);
      case IMPFLOW_ACT_RELU: return launch_chain23<IMPFLOW_ACT_RELU, true>(maps, a, s);
      case IMPFLOW_ACT_SIN: return launch_chain23<IMPFLOW_ACT_SIN, true>(maps, a, s);
      default: return launch_chain23<IMPFLOW_ACT_NONE, true>(maps, a, s);
    }
  }
  switch (act_kind) {
    case IMPFLOW_ACT_LIPSWISH: return launch_chain23<IMPFLOW_ACT_LIPSWISH, false>(maps, a, s);
    case IMPFLOW_ACT_RELU: return launch_chain23<IMPFLOW_ACT_RELU, false>(maps, a, s);
    case IMPFLOW_ACT_SIN: return launch_chain23<IMPFLOW_ACT_SIN, false>(maps, a, s);
    default: return launch_chain23<IMPFLOW_ACT_NONE, false>(maps, a, s);
  }
}
