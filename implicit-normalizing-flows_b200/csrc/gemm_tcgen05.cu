// tcgen05 / TMA / TMEM GEMM for the residual-branch contractions (sm_100a only):
//
//     C[M,N] = A[M,K] * B[N,K]^T       fp32 in, fp32 out, "3xTF32" error-compensated:
//     A = A_hi + A_lo, B = B_hi + B_lo  (tf32-representable planes, see k_split_tf32)
//     C ~= A_lo*B_hi + A_hi*B_lo + A_hi*B_hi   accumulated in fp32 in TMEM.
//
// Why 3xTF32: the Broyden solves converge to eps*sqrt(B*d) with eps down to 1e-10 — i.e. fp32
// round-off — so the branch must be evaluated to fp32 accuracy (SURVEY.md §7 hard part 1).
//
// Structure (one persistent CTA per SM, 256 threads, warp-specialised):
//   warp 0   : TMA producer  — cp.async.bulk.tensor.2d, 128B-swizzled K-major tiles, 4 tiles/stage
//   warp 1   : MMA issuer    — one elected thread issues tcgen05.mma.kind::tf32 (M=128, N=BN, K=8)
//   warp 2   : TMEM allocator (2 accumulator stages of BN columns)
//   warps 4-7: epilogue      — tcgen05.ld 32x32b, fused bias / activation / act' product /
//                              hi-lo split for the next GEMM, direct coalesced-per-row stores
// smem ring: STAGES x {A_hi, A_lo, B_hi, B_lo}, full/empty mbarriers; TMEM full/empty mbarriers
// let the epilogue of tile i overlap the MMAs of tile i+1.
#include "tc_common.cuh"

namespace impflow {

constexpr int TC_EPI_WARPS = 8;   // two warps per TMEM lane quarter, interleaved over the 32-column chunks
constexpr int TC_THREADS = 128 + 32 * TC_EPI_WARPS;

struct TcEpilogue {
  Epilogue e;
  float* split_hi;  // optional tf32 hi plane of the "next layer input" value
  float* split_lo;
};

// PAIR: two CTAs of a cluster (one TPC) work on one 256 x BN tile with tcgen05.mma.cta_group::2 — each CTA
// stages its own 128 rows of A and HALF of the B tile, so the operand bytes a CTA pulls through L2 per MMA
// drop from 96 KB to 64 KB per K chunk (BN = 256): the single-CTA kernel is bound by exactly that stream.
template <int BN, bool PAIR = false>
struct TcCfg {
  static constexpr int kStages = PAIR ? 3 : (BN >= 256) ? 2 : (BN >= 128) ? 3 : 4;
  static constexpr int kABytes = TC_BM * TC_BK * 4;  // 16 KB per plane
  static constexpr int kBRows = PAIR ? BN / 2 : BN;  // B rows this CTA stages
  static constexpr int kBBytes = kBRows * TC_BK * 4;
  static constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;
  static constexpr int kTxBytes = PAIR ? 2 * kStageBytes : kStageBytes;   // bytes landing per stage, both CTAs
  static constexpr int kTileM = PAIR ? 2 * TC_BM : TC_BM;
  static constexpr int kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128
                                   : (2 * BN <= 256) ? 256 : 512;
  static constexpr int kStagingBytes = TC_EPI_WARPS * 4096;   // one 32x32 fp32 tile per epilogue warp (TMA stores)
  static constexpr int kSmemBytes = kStages * kStageBytes + kStagingBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // shared::cluster address of the same offset in the pair's CTA 0

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load issued by either CTA of a pair; the bytes are counted on CTA 0's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_pair(uint32_t tmem_c, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_c),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at the same offset in BOTH CTAs of the pair once the MMAs issued so far retire
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta0(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask)
               : "memory");
}

template <int BN, bool PAIR>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_gemm_tc3(const __grid_constant__ CUtensorMap mapAhi, const __grid_constant__ CUtensorMap mapAlo,
           const __grid_constant__ CUtensorMap mapBhi, const __grid_constant__ CUtensorMap mapBlo,
           const __grid_constant__ CUtensorMap mapPre, const __grid_constant__ CUtensorMap mapAct,
           const __grid_constant__ CUtensorMap mapShi, const __grid_constant__ CUtensorMap mapSlo, int tma_store,
           long long M, int N, int K, TcEpilogue ep, int splits, float* __restrict__ splitk_ws, const int* gate) {
  using Cfg = TcCfg<BN, PAIR>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* staging = smem + Cfg::kStages * Cfg::kStageBytes;        // 1024-byte aligned 4 KB tiles, one per epilogue warp
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + Cfg::kStagingBytes);
  uint64_t* full = bars;                       // [kStages]
  uint64_t* empty = bars + Cfg::kStages;       // [kStages]
  uint64_t* tfull = bars + 2 * Cfg::kStages;   // [2]
  uint64_t* tempty = tfull + 2;                // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  pdl_trigger();     // a dependent tile kernel may be scheduled as this one's CTAs retire
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = K / TC_BK;
  const long long m_tiles = (M + Cfg::kTileM - 1) / Cfg::kTileM;
  const int n_tiles = (N + BN - 1) / BN;
  // a work stream is one CTA, or one CTA pair (both CTAs walk the same tile sequence)
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
  const long long stream0 = PAIR ? (blockIdx.x >> 1) : blockIdx.x;
  const long long n_streams = PAIR ? (gridDim.x >> 1) : gridDim.x;
  // split-K (weight-gradient shapes: small M x N, K = all pixels): work item = (tile, k-slice);
  // raw partial accumulators go to splitk_ws[slice][M][N] and k_splitk_reduce finishes the job.
  long long num_tiles = m_tiles * n_tiles * splits;
  const int kb_per = (num_kb + splits - 1) / splits;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapAhi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapAlo)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapBhi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapBlo)) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], PAIR ? 2 * TC_EPI_WARPS : TC_EPI_WARPS);  // one arrive per epilogue warp (of both CTAs)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if (PAIR) {   // the same warp of both CTAs allocates the pair's columns
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"((uint32_t)Cfg::kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"((uint32_t)Cfg::kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();        // everything above overlapped the predecessor; no global memory was touched yet
  if (gate_closed(gate)) num_tiles = 0;   // speculative solver iteration after the loop ended: no tiles (uniform)

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (long long tile = stream0; tile < num_tiles; tile += n_streams) {
        const long long mn = tile / splits;
        const int ks = (int)(tile % splits);
        const int m_idx = (int)(mn / n_tiles) * Cfg::kTileM + (int)cta_rank * TC_BM;
        const int n_idx = (int)(mn % n_tiles) * BN + (int)cta_rank * (PAIR ? Cfg::kBRows : 0);
        const int kb_end = min(num_kb, (ks + 1) * kb_per);
        for (int kb = ks * kb_per; kb < kb_end; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* st = smem + stage * Cfg::kStageBytes;
          if (PAIR) {
            // CTA 0's barrier counts the bytes of both CTAs (the peer's may land before the expect: the
            // phase cannot complete without CTA 0's own arrival)
            if (cta_rank == 0) mbar_expect_tx(&full[stage], Cfg::kTxBytes);
            tma_load_2d_pair(&mapAhi, &full[stage], st, kb * TC_BK, m_idx);
            tma_load_2d_pair(&mapAlo, &full[stage], st + Cfg::kABytes, kb * TC_BK, m_idx);
            tma_load_2d_pair(&mapBhi, &full[stage], st + 2 * Cfg::kABytes, kb * TC_BK, n_idx);
            tma_load_2d_pair(&mapBlo, &full[stage], st + 2 * Cfg::kABytes + Cfg::kBBytes, kb * TC_BK, n_idx);
          } else {
            mbar_expect_tx(&full[stage], Cfg::kStageBytes);
            tma_load_2d(&mapAhi, &full[stage], st, kb * TC_BK, m_idx);
            tma_load_2d(&mapAlo, &full[stage], st + Cfg::kABytes, kb * TC_BK, m_idx);
            tma_load_2d(&mapBhi, &full[stage], st + 2 * Cfg::kABytes, kb * TC_BK, n_idx);
            tma_load_2d(&mapBlo, &full[stage], st + 2 * Cfg::kABytes + Cfg::kBBytes, kb * TC_BK, n_idx);
          }
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      if (PAIR) {
        // tail: every stage released (CTA 0's commits also arrive on the peer's barriers — nobody may exit
        // while such an arrive is in flight)
        for (int i = 0; i < Cfg::kStages; ++i) {
          mbar_wait(&empty[stage], phase ^ 1);
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 && cta_rank == 0) {
    // ================= MMA issuer (CTA 0 of a pair issues for both) =================
    // instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 [4,6)=1, a=TF32 [7,10)=2,
    // b=TF32 [10,13)=2, K-major both, N>>3 at [17,23), M>>4 at [24,29)
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) |
                           ((uint32_t)(Cfg::kTileM >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (long long tile = stream0; tile < num_tiles; tile += n_streams) {
      mbar_wait(&tempty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t tmem_c = tmem_base + (uint32_t)(acc * BN);
      const int ks = (int)(tile % splits);
      const int kb_begin = ks * kb_per;
      const int kb_end = min(num_kb, kb_begin + kb_per);
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_hi = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t a_lo = a_hi + Cfg::kABytes;
          const uint32_t b_hi = a_hi + 2 * Cfg::kABytes;
          const uint32_t b_lo = b_hi + Cfg::kBBytes;
#pragma unroll
          for (int k = 0; k < TC_BK / 8; ++k) {
            const uint32_t koff = k * 32;  // 8 tf32 = 32 bytes inside the 128B swizzle row
            const uint64_t dah = make_kmajor_sw128_desc(a_hi + koff);
            const uint64_t dal = make_kmajor_sw128_desc(a_lo + koff);
            const uint64_t dbh = make_kmajor_sw128_desc(b_hi + koff);
            const uint64_t dbl = make_kmajor_sw128_desc(b_lo + koff);
            if (PAIR) {
              umma_tf32_pair(tmem_c, dal, dbh, idesc, (kb != kb_begin || k != 0) ? 1u : 0u);
              umma_tf32_pair(tmem_c, dah, dbl, idesc, 1u);
              umma_tf32_pair(tmem_c, dah, dbh, idesc, 1u);
            } else {
              umma_tf32(tmem_c, dal, dbh, idesc, (kb != kb_begin || k != 0) ? 1u : 0u);
              umma_tf32(tmem_c, dah, dbl, idesc, 1u);
              umma_tf32(tmem_c, dah, dbh, idesc, 1u);
            }
          }
        }
        __syncwarp();
        if (elect_one()) {   // frees the smem stage (of both CTAs) when the MMAs retire
          if (PAIR) umma_commit_pair(&empty[stage]);
          else umma_commit(&empty[stage]);
        }
        __syncwarp();
        if (++stage == Cfg::kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one()) {   // accumulator ready for the epilogue
        if (PAIR) umma_commit_pair(&tfull[acc]);
        else umma_commit(&tfull[acc]);
      }
      __syncwarp();
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue =================
    const int q = warp & 3;           // TMEM lane quarter this warp may touch (warp % 4)
    const int chunk0 = (warp - 4) >> 2;  // first 32-column chunk of this warp; stride TC_EPI_WARPS / 4
    int acc = 0;
    uint32_t acc_phase = 0;
    const Epilogue e = resolve_beta(ep.e);
    // Output path.  tma_store: every 32x32 chunk is staged in this warp's shared-memory tile (128-byte rows,
    // SWIZZLE_128B, conflict-free row-per-thread writes) and leaves through ONE bulk tensor store, which also
    // clips ragged M / N; the per-thread 32-byte global stores of the fallback touch 32 different lines per
    // instruction and are limited by the L1 request rate.
    const bool use_tma = tma_store != 0 && splits == 1;
    uint8_t* const my_stage = staging + (warp - 4) * 4096;
    auto emit = [&](const CUtensorMap* map, float* out, const float* vals, long long row, int n0, long long m0w,
                    bool full_vec) {
      if (use_tma) {
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // previous store has read the tile
        __syncwarp();
        const uint32_t sbase = smem_u32(my_stage) + lane * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(sbase + (uint32_t)((j ^ (lane & 7)) << 4)),
                       "f"(vals[4 * j]), "f"(vals[4 * j + 1]), "f"(vals[4 * j + 2]), "f"(vals[4 * j + 3])
                       : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                           reinterpret_cast<uint64_t>(map)),
                       "r"(smem_u32(my_stage)), "r"(n0), "r"((int)m0w)
                       : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        return;
      }
      if (full_vec) {
#pragma unroll
        for (int j = 0; j < 32; j += 8) st_global_v8(out + row + n0 + j, vals + j);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (n0 + j < N) out[row + n0 + j] = vals[j];
      }
    };
    for (long long tile = stream0; tile < num_tiles; tile += n_streams) {
      const long long mn = tile / splits;
      const int ks = (int)(tile % splits);
      const long long m_cta = (mn / n_tiles) * Cfg::kTileM + (long long)cta_rank * TC_BM;   // first row of this CTA
      const long long m = m_cta + q * 32 + lane;
      const int n_base = (int)(mn % n_tiles) * BN;
      // The act' / multiplier operand of a chunk is requested one chunk ahead (the first one before the
      // accumulator is even complete), so its global-memory latency hides behind the MMAs / the previous chunk.
      float dm[32], dm_next[32];
      const bool dm_rows = e.dmul_pre != nullptr && splits == 1 && m < M && ((e.ldc & 7) == 0);
      auto dm_fetch = [&](int c) {
        const int n0f = n_base + c * 32;
        if (dm_rows && c < BN / 32 && n0f + 32 <= N) {
#pragma unroll
          for (int j = 0; j < 32; j += 8) ld_global_v8(e.dmul_pre + m * e.ldc + n0f + j, dm_next + j);
        }
      };
      dm_fetch(chunk0);
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int c = chunk0; c < BN / 32; c += TC_EPI_WARPS / 4) {
        uint32_t r[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + c * 32);
        const int n0 = n_base + c * 32;
#pragma unroll
        for (int j = 0; j < 32; ++j) dm[j] = dm_next[j];
        dm_fetch(c + TC_EPI_WARPS / 4);
        tmem_ld32(taddr, r);
        if (splits > 1) {
          if (m < M && n0 < N) {
            float* dst = splitk_ws + ((long long)ks * M + m) * N + n0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n0 + j < N) dst[j] = __uint_as_float(r[j]);
          }
          continue;
        }
        const long long m0w = m_cta + q * 32;          // first row of this warp's chunk
        if (use_tma ? (m0w < M && n0 < N) : (m < M && n0 < N)) {
          const long long row = m * e.ldc;
          const bool full_vec = (n0 + 32 <= N) && ((e.ldc & 7) == 0);   // 32-byte aligned row chunks
          float v[32];
          if (e.dmul_pre != nullptr) {
            if (e.act_out != nullptr) {      // dmul mode: act_out receives the raw accumulator
              float raw[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) raw[j] = __uint_as_float(r[j]);
              emit(&mapAct, e.act_out, raw, row, n0, m0w, full_vec);
            }
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              float p[8];
              if (full_vec && m < M) {
#pragma unroll
                for (int u = 0; u < 8; ++u) p[u] = dm[j + u];
              } else {
#pragma unroll
                for (int u = 0; u < 8; ++u) p[u] = (m < M && n0 + j + u < N) ? e.dmul_pre[row + n0 + j + u] : 0.f;
              }
#pragma unroll
              for (int u = 0; u < 8; ++u)
                v[j + u] = __uint_as_float(r[j + u]) * act_dispatch(e.act_kind, p[u], 1, e.beta);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float b = (e.bias != nullptr && n0 + j < N) ? __ldg(e.bias + n0 + j) : 0.f;
              v[j] = __uint_as_float(r[j]) + b;
            }
            if (e.pre_out != nullptr) emit(&mapPre, e.pre_out, v, row, n0, m0w, full_vec);
            if (e.act_kind == IMPFLOW_ACT_LIPSWISH) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = lipswish_fast(v[j], e.beta);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = act_dispatch(e.act_kind, v[j], 0, e.beta);
            }
          }
          if (e.dmul_pre != nullptr) {
            if (e.pre_out != nullptr) emit(&mapPre, e.pre_out, v, row, n0, m0w, full_vec);
          } else if (e.act_out != nullptr) {
            emit(&mapAct, e.act_out, v, row, n0, m0w, full_vec);
          }
          if (ep.split_hi != nullptr) {
            float h[32], l[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              // round to nearest, ties away (= cvt.rna.tf32.f32 for finite values) in two integer ops
              const uint32_t hb = (__float_as_uint(v[j]) + 0x1000u) & 0xffffe000u;
              h[j] = __uint_as_float(hb);
              l[j] = v[j] - h[j];
            }
            emit(&mapShi, ep.split_hi, h, row, n0, m0w, full_vec);
            emit(&mapSlo, ep.split_lo, l, row, n0, m0w, full_vec);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cta0(&tempty[acc]);
        else mbar_arrive(&tempty[acc]);
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (use_tma && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores complete before exit
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                   "r"((uint32_t)Cfg::kTmemCols)
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                   "r"((uint32_t)Cfg::kTmemCols)
                   : "memory");
  }
}

__global__ void __launch_bounds__(256)
k_splitk_reduce(const float* __restrict__ ws, const float* __restrict__ bias, float* __restrict__ out,
                long long M, int N, long long ldc, int splits) {
  const long long total = M * N;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int s = 0; s < splits; ++s) acc += ws[(long long)s * total + i];   // fixed order: deterministic
    const long long m = i / N;
    const int n = (int)(i % N);
    out[m * ldc + n] = acc + (bias != nullptr ? bias[n] : 0.f);
  }
}

static int g_tma_store = 1;   // A/B switch (impflow_gemm_tc_set_tma_store)

static int pick_splits(long long M, int N, int K, int BN) {
  const long long tiles = ((M + TC_BM - 1) / TC_BM) * ((N + BN - 1) / BN);
  const int num_kb = K / TC_BK;
  if (tiles >= 96 || num_kb < 64) return 1;
  long long s = (296 + tiles - 1) / tiles;
  if (s > num_kb / 16) s = num_kb / 16;
  if (s > 64) s = 64;
  return s < 2 ? 1 : (int)s;
}

template <int BN, bool PAIR = false>
static int launch_tc(const float* Ahi, const float* Alo, long long lda, const float* Bhi, const float* Blo,
                     long long ldb, long long M, int N, int K, const TcEpilogue& ep, int splits, float* ws,
                     cudaStream_t s) {
  CUtensorMap mAh, mAl, mBh, mBl;
  if (make_map(&mAh, Ahi, M, K, lda, TC_BM) || make_map(&mAl, Alo, M, K, lda, TC_BM) ||
      make_map(&mBh, Bhi, N, K, ldb, TcCfg<BN, PAIR>::kBRows) || make_map(&mBl, Blo, N, K, ldb, TcCfg<BN, PAIR>::kBRows))
    return -1;
  // outputs leave through bulk tensor stores when every output plane can be described by a tensor map
  // (16-byte aligned base and row stride); split-K partials keep the plain stores
  CUtensorMap mo[4];
  memset(mo, 0, sizeof(mo));
  float* outs[4] = {ep.e.pre_out, ep.e.act_out, ep.split_hi, ep.split_lo};
  int tma_store = (g_tma_store && splits == 1 && (ep.e.ldc % 4) == 0) ? 1 : 0;
  for (int i = 0; i < 4 && tma_store; ++i)
    if (outs[i] != nullptr && (reinterpret_cast<uintptr_t>(outs[i]) & 15) != 0) tma_store = 0;
  for (int i = 0; i < 4 && tma_store; ++i)
    if (outs[i] != nullptr && make_map(&mo[i], outs[i], M, N, ep.e.ldc, 32)) return -1;
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(k_gemm_tc3<BN, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             TcCfg<BN, PAIR>::kSmemBytes) != cudaSuccess) {
      set_error("gemm_tc: cannot set %d bytes of dynamic shared memory", TcCfg<BN, PAIR>::kSmemBytes);
      return -1;
    }
    attr_set = true;
  }
  constexpr int kTileM = TcCfg<BN, PAIR>::kTileM;
  const long long tiles = ((M + kTileM - 1) / kTileM) * ((N + BN - 1) / BN) * splits;
  if (PAIR) {
    // one cluster of two CTAs (a TPC's two SMs) per work stream
    const int pairs = (int)(tiles < 74 ? tiles : 74);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(TC_THREADS);
    cfg.dynamicSmemBytes = TcCfg<BN, PAIR>::kSmemBytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1 + pdl_attr(&attr[1]);
    const cudaError_t err = cudaLaunchKernelEx(&cfg, k_gemm_tc3<BN, PAIR>, mAh, mAl, mBh, mBl, mo[0], mo[1], mo[2], mo[3],
                                               tma_store, M, N, K, ep, splits, ws, g_gate);
    if (err != cudaSuccess) {
      set_error("k_gemm_tc3 (pair): launch failed: %s", cudaGetErrorString(err));
      return -1;
    }
    return check_launch("k_gemm_tc3<pair>");
  }
  const int grid = (int)(tiles < 148 ? tiles : 148);
  {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(TC_THREADS);
    cfg.dynamicSmemBytes = TcCfg<BN, PAIR>::kSmemBytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    cfg.attrs = attr;
    cfg.numAttrs = pdl_attr(&attr[0]);
    const cudaError_t err = cudaLaunchKernelEx(&cfg, k_gemm_tc3<BN, PAIR>, mAh, mAl, mBh, mBl, mo[0], mo[1], mo[2], mo[3],
                                               tma_store, M, N, K, ep, splits, ws, g_gate);
    if (err != cudaSuccess) {
      set_error("k_gemm_tc3: launch failed: %s", cudaGetErrorString(err));
      return -1;
    }
  }
  if (check_launch("k_gemm_tc3")) return -1;
  if (splits > 1) {
    long long blocks = (M * N + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    k_splitk_reduce<<<(int)blocks, 256, 0, s>>>(ws, ep.e.bias, ep.e.pre_out, M, N, ep.e.ldc, splits);
    return check_launch("k_splitk_reduce");
  }
  return 0;
}

int gemm_nt_simt(const float* A, long long lda, const float* Bm, long long ldb, long long M, int N, int K,
                 const Epilogue& ep, cudaStream_t s);
int gemm_strided_simt(const float* A, long long sAm, long long sAk, const float* Bm, long long sBn, long long sBk,
                      const float* bias, float* out, long long ldc, long long M, int N, int K, cudaStream_t s);

}  // namespace impflow

using namespace impflow;

extern "C" int impflow_gemm_nt(const float* A, long long lda, const float* Bm, long long ldb, const float* bias,
                               float* pre_out, float* act_out, const float* dmul_pre, long long ldc, long long M,
                               int N, int K, int act_kind, const float* beta_sp, void* stream) {
  IMPFLOW_REQUIRE(M >= 1 && N >= 1 && K >= 1, "gemm_nt: empty problem M=%lld N=%d K=%d", M, N, K);
  IMPFLOW_REQUIRE(pre_out != nullptr || act_out != nullptr, "gemm_nt: no output given");
  IMPFLOW_REQUIRE(dmul_pre == nullptr || pre_out != nullptr || act_out != nullptr,
                  "gemm_nt: dmul_pre needs pre_out or act_out");
  Epilogue ep{bias, pre_out, act_out, dmul_pre, ldc, act_kind, beta_sp, 0.f};
  return gemm_nt_simt(A, lda, Bm, ldb, M, N, K, ep, (cudaStream_t)stream);
}

extern "C" int impflow_gemm_strided(const float* A, long long sAm, long long sAk, const float* Bm, long long sBn,
                                    long long sBk, const float* bias, float* out, long long ldc, long long M, int N,
                                    int K, void* stream) {
  IMPFLOW_REQUIRE(M >= 1 && N >= 1 && K >= 1, "gemm_strided: empty problem M=%lld N=%d K=%d", M, N, K);
  IMPFLOW_REQUIRE(out != nullptr, "gemm_strided: no output given");
  return gemm_strided_simt(A, sAm, sAk, Bm, sBn, sBk, bias, out, ldc, M, N, K, (cudaStream_t)stream);
}

// Tile width: 256 halves the A-operand re-reads, but a problem with few row tiles fills more SMs (and
// finishes in fewer, cheaper rounds) with 128-wide tiles: compare rounds x relative tile cost.
static int tc_bn(int N, long long M = 1LL << 40) {
  if (N <= 32) return 32;
  if (N <= 64) return 64;
  if (N < 256) return 128;
  const long long m_tiles = (M + TC_BM - 1) / TC_BM;
  const long long r256 = (m_tiles * ((N + 255) / 256) + 147) / 148;
  const long long r128 = (m_tiles * ((N + 127) / 128) + 147) / 148;
  return (r128 * 55 < r256 * 100) ? 128 : 256;
}

static int g_pair = 1;   // A/B switch (impflow_gemm_tc_set_pair)
// CTA pairs (cta_group::2, 256 x 256 tiles) when they finish the problem in fewer cost-weighted rounds than
// single CTAs: a pair tile streams 64 KB per CTA and K chunk (MMA-paced), a single 128 x 256 tile 96 KB
// (about 1.5x the MMA time at the L2 -> SM rate), a 128 x 128 tile 64 KB for half the columns.
static bool tc_use_pair(long long M, int N) {
  if (!g_pair || N < 256) return false;
  const long long n256 = (N + 255) / 256;
  const long long r_pair = (((M + 255) / 256) * n256 + 73) / 74;
  const long long m_tiles = (M + TC_BM - 1) / TC_BM;
  const long long r256 = (m_tiles * n256 + 147) / 148;
  const long long r128 = (m_tiles * ((N + 127) / 128) + 147) / 148;
  return r_pair * 100 < r256 * 140 && r_pair * 100 < r128 * 95;
}

extern "C" int impflow_gemm_tc_set_pair(int on) {
  const int prev = g_pair;
  g_pair = on ? 1 : 0;
  return prev;
}

extern "C" int impflow_gemm_tc_set_tma_store(int on) {
  const int prev = g_tma_store;
  g_tma_store = on ? 1 : 0;
  return prev;
}

extern "C" int impflow_gemm_tc_splits(long long M, int N, int K) {
  if (K % TC_BK != 0) return 1;
  return pick_splits(M, N, K, tc_bn(N, M));
}

extern "C" int impflow_gemm_nt_tc(const float* A_hi, const float* A_lo, long long lda, const float* B_hi,
                                  const float* B_lo, long long ldb, const float* bias, float* pre_out,
                                  float* act_out, const float* dmul_pre, float* split_hi, float* split_lo,
                                  long long ldc, long long M, int N, int K, int act_kind,
                                  const float* beta_sp, float* splitk_ws, void* stream) {
  IMPFLOW_REQUIRE(M >= 1 && N >= 1 && K >= 1, "gemm_nt_tc: empty problem M=%lld N=%d K=%d", M, N, K);
  IMPFLOW_REQUIRE(pre_out != nullptr || act_out != nullptr || split_hi != nullptr, "gemm_nt_tc: no output given");
  IMPFLOW_REQUIRE(dmul_pre == nullptr || pre_out != nullptr || split_hi != nullptr || act_out != nullptr,
                  "gemm_nt_tc: dmul_pre needs pre_out, act_out or split planes");
  IMPFLOW_REQUIRE((split_hi == nullptr) == (split_lo == nullptr), "gemm_nt_tc: split planes come in pairs");
  if (K % TC_BK != 0 || (lda % 4) != 0 || (ldb % 4) != 0) {
    set_error("gemm_nt_tc: needs K %% 32 == 0 and 16-byte aligned rows (K=%d lda=%lld ldb=%lld)", K, lda, ldb);
    return -2;
  }
  const uintptr_t al = reinterpret_cast<uintptr_t>(A_hi) | reinterpret_cast<uintptr_t>(A_lo) |
                       reinterpret_cast<uintptr_t>(B_hi) | reinterpret_cast<uintptr_t>(B_lo);
  if (al & 15) {
    set_error("gemm_nt_tc: operand base pointers must be 16-byte aligned");
    return -2;
  }
  TcEpilogue ep{{bias, pre_out, act_out, dmul_pre, ldc, act_kind, beta_sp, 0.f}, split_hi, split_lo};
  cudaStream_t s = (cudaStream_t)stream;
  // split-K only for the plain epilogue (weight-gradient GEMMs) and only if the caller gave a workspace
  int splits = 1;
  if (splitk_ws != nullptr && act_out == nullptr && dmul_pre == nullptr && split_hi == nullptr && pre_out != nullptr)
    splits = pick_splits(M, N, K, tc_bn(N, M));
  const int bn = tc_bn(N, M);
  if (splits == 1 && tc_use_pair(M, N))
    return launch_tc<256, true>(A_hi, A_lo, lda, B_hi, B_lo, ldb, M, N, K, ep, 1, splitk_ws, s);
  if (bn == 32) return launch_tc<32>(A_hi, A_lo, lda, B_hi, B_lo, ldb, M, N, K, ep, splits, splitk_ws, s);
  if (bn == 64) return launch_tc<64>(A_hi, A_lo, lda, B_hi, B_lo, ldb, M, N, K, ep, splits, splitk_ws, s);
  if (bn == 256) return launch_tc<256>(A_hi, A_lo, lda, B_hi, B_lo, ldb, M, N, K, ep, splits, splitk_ws, s);
  return launch_tc<128>(A_hi, A_lo, lda, B_hi, B_lo, ldb, M, N, K, ep, splits, splitk_ws, s);
}
