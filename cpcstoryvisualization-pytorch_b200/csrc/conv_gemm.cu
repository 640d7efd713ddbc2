// tcgen05 implicit-GEMM kernel for every convolution-shaped contraction of the CP-CSV step.
//
// One persistent, warp-specialised kernel (sm_100a):
//   warp 0      TMA producer   : 5-D tiled tensor-map loads (128B swizzle) of the A pixel box
//                                (shifted per filter tap; TMA zero-fill = conv padding) and of
//                                the B tile, into a multi-stage shared-memory ring
//   warp 1      MMA issuer     : tcgen05.mma kind::f16 (bf16/fp16 in, fp32 accumulate in TMEM),
//                                1 or 3 MMAs per k-step (hi/lo split operands), tcgen05.commit
//                                releases smem stages / publishes the accumulator
//   warps 2..5  epilogue       : tcgen05.ld TMEM -> registers -> fp32 global (store or red.add)
// Two TMEM accumulator stages (2 x 256 columns) let the epilogue of tile i overlap the main
// loop of tile i+1.
//
// mode 0 (fprop / dgrad): D[pix, n] = sum_{tap, k} A[pix + tap, k] * B[tap][n, k]
//        A, B K-major; M tile = 128 output pixels (tile_n x tile_h x tile_w box)
// mode 1 (wgrad):         D[tap][ca, cb] = sum_pix A[pix + tapA, ca] * B[pix + tapB, cb]
//        A, B MN-major (channels contiguous); K step = 64 pixels
#include <cuda.h>
#include <cudaTypedefs.h>

#include <mutex>

#include "common.h"
#include "ptx.cuh"

namespace cpcsv {

constexpr int kThreads = 192;
constexpr int kBlockM = 128;
constexpr int kMaxStages = 8;
constexpr int kAPlaneBytes = kBlockM * 128;  // 128 rows x 64 16-bit (mode 0) / 2 x [64 pix x 64 ch] (mode 1)
constexpr int kSmemLimit = 227 * 1024;
// Shared memory a SINGLE-PLANE job takes: 144 KB = 3 pipeline stages of a pair job.  The single-plane jobs are the
// backward pass and the no-grad forward; with the whole 227 KB (6 stages) a resident GEMM CTA leaves no room for any
// other block that needs shared memory, and the optimiser's Adam + re-layout kernels (10-28 KB per block, issued
// during the backward pass) queue up behind the last GEMM.  Measured (bench.py, two boxes): 227 KB 20.21 /
// 20.59-20.61 ms per step; 160 KB 19.97 / 20.35; 144 KB 19.87-19.96; 128 KB 19.94-20.03 -- and no measurable change
// of the GEMMs' own serial time (15.4-15.9 ms either way).
constexpr int kSinglePlaneSmemLimit = 144 * 1024;
constexpr int kBarrierBytes = 256;
// Epilogue staging: each epilogue warp transposes its 32 rows x 32 columns through shared memory
// so that global stores / red.adds cover whole 128 B row segments (4 rows per instruction)
// instead of 32 different rows per instruction.  Row pitch 36 floats: conflict-free for the
// row-per-lane v4 writes and for the 8-lanes-per-row v4 reads.
constexpr int kEpiPitch = 36;
constexpr int kEpiWarpFloats = 32 * kEpiPitch;
constexpr int kEpiStageBytes = 4 * kEpiWarpFloats * 4;
// Column statistics (optional, GemmParams::stats): fp32 sums / sums of squares of the current tile's
// columns, one region per epilogue warp (its 32 rows; plain stores, no shared-memory atomics), combined
// and flushed to the fp64 totals between two named barriers of the four epilogue warps.
constexpr int kColAccFloats = 4 * 2 * 256;
constexpr int kEpiBytes = kEpiStageBytes + kColAccFloats * 4;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kAccStride = 256;  // columns between the two accumulator stages

struct GemmParams {
  int32_t mode, planes;
  int32_t N, H, W;
  int32_t tile_n, tile_h, tile_w;
  int32_t tiles_n, tiles_h, tiles_w;
  int32_t groups, taps_per_group, k_blocks;
  int32_t m_tiles, n_tiles, block_n;
  int32_t m_units;     // m_tiles, or pairs of m tiles in CTA-pair mode
  int32_t m_valid, n_valid;
  int32_t splits, iters_total;
  int32_t accumulate;
  int32_t stages, b_plane_bytes, stage_bytes;
  uint32_t idesc;
  uint32_t total_tiles;
  int64_t osn, osh, osw, ldc;
  const float* alpha;
  float* out;
  double* stats;      // optional [2][stats_ld]: per-column sum / sum of squares of the stored values
  int64_t stats_ld;
  cpcsv_tap_t taps[CPCSV_MAX_TAPS];
};

struct TileCoord {
  int32_t group, split, n_idx, m_idx;
  int32_t it0, it1;
};

// `t` counts work units: 128-row tiles, or (CTA-pair mode) pairs of them of which CTA `rank`
// takes the `rank`-th; an odd tail unit has m_idx == m_tiles (every row out of range)
__device__ __forceinline__ TileCoord decode_tile(const GemmParams& P, uint32_t t, uint32_t pair,
                                                 uint32_t rank) {
  TileCoord c;
  c.m_idx = static_cast<int32_t>((t % P.m_units) * (pair ? 2u : 1u) + rank);
  t /= P.m_units;
  c.n_idx = t % P.n_tiles;
  t /= P.n_tiles;
  c.split = t % P.splits;
  c.group = t / P.splits;
  c.it0 = static_cast<int32_t>((static_cast<int64_t>(P.iters_total) * c.split) / P.splits);
  c.it1 = static_cast<int32_t>((static_cast<int64_t>(P.iters_total) * (c.split + 1)) / P.splits);
  return c;
}

// pixel-tile index -> origin of the (n, h, w) box
__device__ __forceinline__ void pixel_tile_origin(const GemmParams& P, int32_t q, int32_t& n0,
                                                  int32_t& h0, int32_t& w0) {
  w0 = (q % P.tiles_w) * P.tile_w;
  q /= P.tiles_w;
  h0 = (q % P.tiles_h) * P.tile_h;
  n0 = (q / P.tiles_h) * P.tile_n;
}

// kPair: the two CTAs of a cluster work as one cta_group::2 unit: each loads its own 128 pixel
// rows of A and HALF of the B tile, the leader issues M = 256 MMAs that read B from both CTAs'
// shared memory, each CTA's TMEM receives its own 128 accumulator rows.  Per CTA and k-step that
// is 16 + block_n/16 KB instead of 16 + block_n/8 KB from L2 -- the L2 -> SM feed is what bounds
// the single-CTA kernel (ncu: 11.7 TB/s of 12.4 TB/s on single-plane jobs).
template <bool kPair>
__global__ void __launch_bounds__(kThreads, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                 const __grid_constant__ CUtensorMap tmB0, const __grid_constant__ CUtensorMap tmB1,
                 const __grid_constant__ GemmParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + P.stages * P.stage_bytes);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tmem_full = empty_bar + kMaxStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* epi_stage = reinterpret_cast<float*>(smem + P.stages * P.stage_bytes + kBarrierBytes);
  float* colacc = epi_stage + 4 * kEpiWarpFloats;   // [4 warps][sum | sumsq][256]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;
  const uint32_t tile0 = kPair ? (blockIdx.x >> 1) : blockIdx.x;
  const uint32_t tstep = kPair ? (gridDim.x >> 1) : gridDim.x;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    tma_prefetch_desc(&tmB0);
    if (P.planes == 2) {
      tma_prefetch_desc(&tmA1);
      tma_prefetch_desc(&tmB1);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < P.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], kPair ? 8 : 4);   // pair: the peer's epilogue warps arrive remotely
    }
    fence_barrier_init();
  }
  // Pair mode: the two CTAs of a cluster do not necessarily START at the same time.  Round 1 / 2 dead-lock
  // (profiles/r02_pair_hang_rootcause.md, cuda-gdb on two hung replays): the leader had allocated its
  // TMEM, given up its allocation permit with tcgen05.relinquish_alloc_permit.cta_group::2 -- which
  // speaks for the PAIR -- and was waiting at the cluster barrier below, while the late peer never got
  // through its own tcgen05.alloc.cta_group::2.  So: first make sure both CTAs are running, then both
  // allocate, and the permit is only given up once both allocations are known to be done.
  if (kPair) cluster_sync_all();
  if (warp == 2) {
    if (kPair) {
      tmem_alloc_pair(tmem_slot, kTmemCols);
    } else {
      tmem_alloc(tmem_slot, kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (kPair) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  if (kPair && warp == 2) tmem_relinquish_pair();
  const uint32_t tmem_base = *tmem_slot;

  const uint32_t stage_tx = static_cast<uint32_t>(P.planes) * (kAPlaneBytes + P.b_plane_bytes);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (uint32_t tile = tile0; tile < P.total_tiles; tile += tstep) {
        const TileCoord tc = decode_tile(P, tile, kPair, rank);
        int32_t n0 = 0, h0 = 0, w0 = 0;
        if (P.mode == 0) pixel_tile_origin(P, tc.m_idx, n0, h0, w0);
        for (int32_t it = tc.it0; it < tc.it1; ++it) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * P.stage_bytes;
          uint8_t* sb = sa + P.planes * kAPlaneBytes;
          if (kPair && P.mode == 1) {
            // weight gradient as a pair: each CTA loads its own 128 output-channel columns of A (dy) and HALF of
            // the B (x) channel block for the same 64 pixels
            if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * stage_tx);
            const uint32_t bar = mapa_u32(&full_bar[stage], 0);
            const cpcsv_tap_t& tap = P.taps[tc.group];
            pixel_tile_origin(P, it, n0, h0, w0);
            const int32_t half_n = P.block_n / 2;
            for (int pl = 0; pl < P.planes; ++pl) {
              for (int j = 0; j < 2; ++j)
                tma_load_5d_pair(pl ? &tmA1 : &tmA0, bar, sa + pl * kAPlaneBytes + j * 8192,
                                 tap.a[0] + tc.m_idx * kBlockM + j * 64, w0 + tap.a[1], tap.a[2],
                                 h0 + tap.a[3], n0);
              for (int j = 0; j < half_n / 64; ++j)
                tma_load_5d_pair(pl ? &tmB1 : &tmB0, bar, sb + pl * P.b_plane_bytes + j * 8192,
                                 tap.b[0] + tc.n_idx * P.block_n + static_cast<int32_t>(rank) * half_n + j * 64,
                                 w0 + tap.b[1], tap.b[2], h0 + tap.b[3], n0);
            }
          } else if (kPair) {
            // both CTAs' bytes are accounted on the leader's barrier
            if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * stage_tx);
            const uint32_t bar = mapa_u32(&full_bar[stage], 0);
            const int32_t t = it / P.k_blocks;
            const int32_t kb = it - t * P.k_blocks;
            const cpcsv_tap_t& tap = P.taps[tc.group * P.taps_per_group + t];
            for (int pl = 0; pl < P.planes; ++pl) {
              tma_load_5d_pair(pl ? &tmA1 : &tmA0, bar, sa + pl * kAPlaneBytes, tap.a[0] + kb * 64,
                               w0 + tap.a[1], tap.a[2], h0 + tap.a[3], n0);
              tma_load_5d_pair(pl ? &tmB1 : &tmB0, bar, sb + pl * P.b_plane_bytes, kb * 64,
                               tap.b[0] + tc.n_idx * P.block_n + static_cast<int32_t>(rank) * (P.block_n / 2),
                               0, 0, 0);
            }
          } else if (P.mode == 0) {
            mbar_expect_tx(&full_bar[stage], stage_tx);
            const int32_t t = it / P.k_blocks;
            const int32_t kb = it - t * P.k_blocks;
            const cpcsv_tap_t& tap = P.taps[tc.group * P.taps_per_group + t];
            for (int pl = 0; pl < P.planes; ++pl) {
              tma_load_5d(pl ? &tmA1 : &tmA0, &full_bar[stage], sa + pl * kAPlaneBytes,
                          tap.a[0] + kb * 64, w0 + tap.a[1], tap.a[2], h0 + tap.a[3], n0);
              tma_load_5d(pl ? &tmB1 : &tmB0, &full_bar[stage], sb + pl * P.b_plane_bytes, kb * 64,
                          tap.b[0] + tc.n_idx * P.block_n, 0, 0, 0);
            }
          } else {
            mbar_expect_tx(&full_bar[stage], stage_tx);
            const cpcsv_tap_t& tap = P.taps[tc.group];
            pixel_tile_origin(P, it, n0, h0, w0);
            for (int pl = 0; pl < P.planes; ++pl) {
              for (int j = 0; j < 2; ++j)
                tma_load_5d(pl ? &tmA1 : &tmA0, &full_bar[stage], sa + pl * kAPlaneBytes + j * 8192,
                            tap.a[0] + tc.m_idx * kBlockM + j * 64, w0 + tap.a[1], tap.a[2],
                            h0 + tap.a[3], n0);
              for (int j = 0; j < P.block_n / 64; ++j)
                tma_load_5d(pl ? &tmB1 : &tmB0, &full_bar[stage],
                            sb + pl * P.b_plane_bytes + j * 8192,
                            tap.b[0] + tc.n_idx * P.block_n + j * 64, w0 + tap.b[1], tap.b[2],
                            h0 + tap.b[3], n0);
            }
          }
          if (++stage == P.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      if (kPair) {
        // Producer tail (pair mode): the commits that release the last `stages` ring slots are
        // multicast arrives into BOTH CTAs' shared memory and nobody waits for them in the main
        // loop.  Drain them before this CTA may exit, so that none of them can land in the
        // barriers of whatever block is scheduled on this SM next.  (Slots that were never
        // filled pass immediately: a fresh barrier is complete for the preceding parity.)
        for (int i = 0; i < P.stages; ++i) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (++stage == P.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0 && rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t acc = 0, acc_phase = 0;
      for (uint32_t tile = tile0; tile < P.total_tiles; tile += tstep) {
        const TileCoord tc = decode_tile(P, tile, kPair, rank);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * kAccStride;
        for (int32_t it = tc.it0; it < tc.it1; ++it) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * P.stage_bytes);
          const uint32_t sb = sa + P.planes * kAPlaneBytes;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            // K-major: 16 elements (32 B) along the 128 B swizzled row per MMA;
            // MN-major: 16 k-rows (2048 B) per MMA, 64-channel atoms 8192 B apart.
            const uint32_t koff = (P.mode == 0) ? k * 32 : k * 2048;
            const uint32_t lbo = (P.mode == 0) ? 16 : 8192;
            const uint64_t a_hi = make_smem_desc(sa + koff, lbo, 1024);
            const uint64_t b_hi = make_smem_desc(sb + koff, lbo, 1024);
            const uint32_t first = (it > tc.it0 || k > 0) ? 1u : 0u;
            if (kPair) umma_f16_pair(tmem_d, a_hi, b_hi, P.idesc, first);
            else umma_f16(tmem_d, a_hi, b_hi, P.idesc, first);
            if (P.planes == 2) {
              const uint64_t a_lo = make_smem_desc(sa + kAPlaneBytes + koff, lbo, 1024);
              const uint64_t b_lo = make_smem_desc(sb + P.b_plane_bytes + koff, lbo, 1024);
              if (kPair) {
                umma_f16_pair(tmem_d, a_lo, b_hi, P.idesc, 1u);
                umma_f16_pair(tmem_d, a_hi, b_lo, P.idesc, 1u);
              } else {
                umma_f16(tmem_d, a_lo, b_hi, P.idesc, 1u);
                umma_f16(tmem_d, a_hi, b_lo, P.idesc, 1u);
              }
            }
          }
          if (kPair) umma_commit_pair(&empty_bar[stage]); else umma_commit(&empty_bar[stage]);
          if (++stage == P.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (kPair) umma_commit_pair(&tmem_full[acc]); else umma_commit(&tmem_full[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ epilogue (4 warps)
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    float* stg = epi_stage + q * kEpiWarpFloats;
    const int sub = lane >> 3;  // coalesced phase: this lane stores rows 4 * i + sub ...
    const int cq = lane & 7;    // ... columns [4 * cq, 4 * cq + 4) of the 32-column chunk
    uint32_t acc = 0, acc_phase = 0;
    const float alpha = P.alpha ? __ldg(P.alpha) : 1.0f;
    const bool atomic = (P.accumulate != 0) || (P.splits > 1);
    const bool want_stats = P.stats != nullptr;
    float* cacc = colacc + q * 512;
    for (uint32_t tile = tile0; tile < P.total_tiles; tile += tstep) {
      const TileCoord tc = decode_tile(P, tile, kPair, rank);
      float* row_ptr;
      bool row_valid;
      if (P.mode == 0) {
        int32_t n0, h0, w0;
        pixel_tile_origin(P, tc.m_idx, n0, h0, w0);
        const int32_t rw = row % P.tile_w;
        const int32_t rh = (row / P.tile_w) % P.tile_h;
        const int32_t rn = row / (P.tile_w * P.tile_h);
        const int32_t n = n0 + rn, h = h0 + rh, w = w0 + rw;
        row_valid = (n < P.N) && (h < P.H) && (w < P.W);
        row_ptr = P.out + P.taps[tc.group * P.taps_per_group].out_off + n * P.osn + h * P.osh +
                  w * P.osw;
      } else {
        const int32_t m = tc.m_idx * kBlockM + row;
        row_valid = m < P.m_valid;
        row_ptr = P.out + P.taps[tc.group].out_off + static_cast<int64_t>(m) * P.ldc;
      }
      // output rows this lane writes in the coalesced phase (owned by lane 4 * i + sub)
      float* rp[8];
      uint32_t rv = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int src = 4 * i + sub;
        rp[i] = reinterpret_cast<float*>(
            __shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(row_ptr), src));
        rv |= (__shfl_sync(0xffffffffu, row_valid ? 1u : 0u, src) & 1u) << i;
      }
      const int32_t col0 = tc.n_idx * P.block_n;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kAccStride;
      for (int32_t c0 = 0; c0 < P.block_n; c0 += 32) {
        if (P.block_n - c0 >= 32) {
          uint32_t r[32];
          tmem_ld_32x32(taddr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 v;
            v.x = __uint_as_float(r[j]) * alpha;
            v.y = __uint_as_float(r[j + 1]) * alpha;
            v.z = __uint_as_float(r[j + 2]) * alpha;
            v.w = __uint_as_float(r[j + 3]) * alpha;
            *reinterpret_cast<float4*>(stg + lane * kEpiPitch + j) = v;
          }
          __syncwarp();
          const int32_t col = col0 + c0 + 4 * cq;
          float cs[4] = {0.f, 0.f, 0.f, 0.f}, cq2[4] = {0.f, 0.f, 0.f, 0.f};
          if (col < P.n_valid) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              if ((rv >> i) & 1u) {
                const float4 v =
                    *reinterpret_cast<const float4*>(stg + (4 * i + sub) * kEpiPitch + 4 * cq);
                float* dst = rp[i] + col;
                if (atomic) {
                  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst),
                               "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                               : "memory");
                } else {
                  *reinterpret_cast<float4*>(dst) = v;
                }
                cs[0] += v.x; cs[1] += v.y; cs[2] += v.z; cs[3] += v.w;
                cq2[0] = fmaf(v.x, v.x, cq2[0]); cq2[1] = fmaf(v.y, v.y, cq2[1]);
                cq2[2] = fmaf(v.z, v.z, cq2[2]); cq2[3] = fmaf(v.w, v.w, cq2[3]);
              }
            }
          }
          if (want_stats) {
            // sum over the 4 row groups (lane bits 3, 4): lanes 0..7 end up with the 32-row sums of
            // their 4 columns, added to the CTA's per-tile column accumulators
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              cs[j] += __shfl_xor_sync(0xffffffffu, cs[j], 8);
              cs[j] += __shfl_xor_sync(0xffffffffu, cs[j], 16);
              cq2[j] += __shfl_xor_sync(0xffffffffu, cq2[j], 8);
              cq2[j] += __shfl_xor_sync(0xffffffffu, cq2[j], 16);
            }
            if (sub == 0) {
              *reinterpret_cast<float4*>(cacc + c0 + 4 * cq) = make_float4(cs[0], cs[1], cs[2], cs[3]);
              *reinterpret_cast<float4*>(cacc + 256 + c0 + 4 * cq) = make_float4(cq2[0], cq2[1], cq2[2], cq2[3]);
            }
          }
          __syncwarp();
        } else {
          // 16-column tail (narrow heads): one row per lane
          uint32_t r16[16];
          tmem_ld_32x16(taddr + c0, r16);
          tmem_ld_wait();
          if (row_valid) {
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
              const int32_t col = col0 + c0 + j;
              if (col < P.n_valid) {
                float4 v;
                v.x = __uint_as_float(r16[j]) * alpha;
                v.y = __uint_as_float(r16[j + 1]) * alpha;
                v.z = __uint_as_float(r16[j + 2]) * alpha;
                v.w = __uint_as_float(r16[j + 3]) * alpha;
                float* dst = row_ptr + col;
                if (atomic) {
                  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst),
                               "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                               : "memory");
                } else {
                  *reinterpret_cast<float4*>(dst) = v;
                }
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kPair && rank != 0) mbar_arrive_cluster(mapa_u32(&tmem_empty[acc], 0));
        else mbar_arrive(&tmem_empty[acc]);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
      if (want_stats) {
        // all four epilogue warps have written their 32-row column sums: combine, add to the fp64 totals
        asm volatile("bar.sync 1, 128;" ::: "memory");
        for (int c = row; c < P.block_n; c += 128) {
          if (col0 + c < P.n_valid) {
            const float s1 = colacc[c] + colacc[512 + c] + colacc[1024 + c] + colacc[1536 + c];
            const float s2 = colacc[256 + c] + colacc[768 + c] + colacc[1280 + c] + colacc[1792 + c];
            atomicAdd(P.stats + col0 + c, static_cast<double>(s1));
            atomicAdd(P.stats + P.stats_ld + col0 + c, static_cast<double>(s2));
          }
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");   // regions are overwritten by the next tile
      }
    }
  }

  tc_fence_before();
  if (kPair) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    if (kPair) tmem_dealloc_pair(tmem_base, kTmemCols);
    else tmem_dealloc(tmem_base, kTmemCols);
  }
  // Pair mode: neither CTA may exit (and hand its SM to a block of another kernel that allocates
  // TMEM there) before BOTH halves of the cta_group::2 deallocation have been issued.
  if (kPair) cluster_sync_all();
}

// ------------------------------------------------------------------------------ host side
static PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess) p = nullptr;
    return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }();
  return fn;
}

static int make_map(CUtensorMap* tm, const cpcsv_view5_t& v, const uint32_t box[5], int dtype,
                    const char* what) {
  auto fn = encode_fn();
  if (!fn) return fail(-2, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < 5; ++i) {
    gdim[i] = static_cast<cuuint64_t>(v.dims[i]);
    bx[i] = box[i];
    es[i] = 1;
    if (v.dims[i] <= 0) return fail(-1, "%s: dim %d is %lld", what, i, (long long)v.dims[i]);
    if (box[i] == 0 || box[i] > 256) return fail(-1, "%s: box %d is %u", what, i, box[i]);
  }
  for (int i = 1; i < 5; ++i) {
    if (v.strides[i] <= 0 || (v.strides[i] & 15))
      return fail(-1, "%s: stride %d = %lld not a positive multiple of 16 B", what, i,
                  (long long)v.strides[i]);
    gstr[i - 1] = static_cast<cuuint64_t>(v.strides[i]);
  }
  if (reinterpret_cast<uintptr_t>(v.ptr) & 15) return fail(-1, "%s: base not 16 B aligned", what);
  CUresult r = fn(tm, dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                  5, const_cast<void*>(v.ptr), gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(-3, "%s: cuTensorMapEncodeTiled failed (%d)", what, (int)r);
  return 0;
}

int num_sms() {
  static int n = [] {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  return n;
}

}  // namespace cpcsv

using namespace cpcsv;

extern "C" int cpcsv_conv_gemm(const cpcsv_gemm_t* job, cpcsv_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  CPCSV_REQUIRE(job != nullptr, "conv_gemm: null job");
  const cpcsv_gemm_t& J = *job;
  CPCSV_REQUIRE(J.mode == 0 || J.mode == 1, "conv_gemm: mode %d", J.mode);
  CPCSV_REQUIRE(J.dtype == 0 || J.dtype == 1, "conv_gemm: dtype %d", J.dtype);
  CPCSV_REQUIRE(J.planes == 1 || J.planes == 2, "conv_gemm: planes %d", J.planes);
  CPCSV_REQUIRE(J.N > 0 && J.H > 0 && J.W > 0, "conv_gemm: empty pixel grid");
  const int box_pix = J.tile_n * J.tile_h * J.tile_w;
  CPCSV_REQUIRE(J.tile_n > 0 && J.tile_h > 0 && J.tile_w > 0 && box_pix == (J.mode == 0 ? 128 : 64),
                "conv_gemm: pixel box %dx%dx%d", J.tile_n, J.tile_h, J.tile_w);
  CPCSV_REQUIRE(J.block_n >= 16 && J.block_n <= 256 && J.block_n % 16 == 0, "conv_gemm: block_n %d",
                J.block_n);
  CPCSV_REQUIRE(J.mode == 0 || J.block_n % 64 == 0, "conv_gemm: mode 1 needs block_n %% 64 == 0");
  CPCSV_REQUIRE(J.n_tiles > 0 && J.n_valid > 0 && J.n_valid <= J.n_tiles * J.block_n &&
                    J.n_valid % 4 == 0,
                "conv_gemm: n_valid %d", J.n_valid);
  CPCSV_REQUIRE(J.groups > 0 && J.splits > 0, "conv_gemm: groups/splits");
  CPCSV_REQUIRE(J.out != nullptr && (reinterpret_cast<uintptr_t>(J.out) & 15) == 0,
                "conv_gemm: out pointer");

  GemmParams P;
  memset(&P, 0, sizeof(P));
  P.mode = J.mode;
  P.planes = J.planes;
  P.N = J.N; P.H = J.H; P.W = J.W;
  P.tile_n = J.tile_n; P.tile_h = J.tile_h; P.tile_w = J.tile_w;
  P.tiles_n = static_cast<int32_t>(ceil_div(J.N, J.tile_n));
  P.tiles_h = static_cast<int32_t>(ceil_div(J.H, J.tile_h));
  P.tiles_w = static_cast<int32_t>(ceil_div(J.W, J.tile_w));
  const int64_t pixel_tiles = static_cast<int64_t>(P.tiles_n) * P.tiles_h * P.tiles_w;
  P.groups = J.groups;
  P.block_n = J.block_n;
  P.n_tiles = J.n_tiles;
  P.n_valid = J.n_valid;
  P.splits = J.splits;
  P.accumulate = J.accumulate;
  P.alpha = J.alpha;
  P.out = J.out;
  CPCSV_REQUIRE(J.stats == nullptr || (J.mode == 0 && J.splits == 1 && J.accumulate == 0 && J.block_n % 32 == 0 &&
                                       J.stats_ld >= J.n_valid),
                "conv_gemm: column statistics need mode 0 without split-K / accumulation and block_n %% 32 == 0");
  P.stats = J.stats;
  P.stats_ld = J.stats_ld;
  int ntaps;
  if (J.mode == 0) {
    CPCSV_REQUIRE(J.taps_per_group > 0 && J.k_blocks > 0, "conv_gemm: taps/k_blocks");
    ntaps = J.groups * J.taps_per_group;
    P.taps_per_group = J.taps_per_group;
    P.k_blocks = J.k_blocks;
    P.m_tiles = static_cast<int32_t>(pixel_tiles);
    P.iters_total = J.taps_per_group * J.k_blocks;
    P.osn = J.out_stride_n; P.osh = J.out_stride_h; P.osw = J.out_stride_w;
    CPCSV_REQUIRE((P.osn % 4) == 0 && (P.osh % 4) == 0 && (P.osw % 4) == 0,
                  "conv_gemm: output strides must be multiples of 4 elements");
  } else {
    ntaps = J.groups;
    P.taps_per_group = 1;
    CPCSV_REQUIRE(J.m_valid > 0, "conv_gemm: m_valid");
    P.m_valid = J.m_valid;
    P.m_tiles = static_cast<int32_t>(ceil_div(J.m_valid, kBlockM));
    CPCSV_REQUIRE(pixel_tiles < (1ll << 31), "conv_gemm: too many pixel tiles");
    P.iters_total = static_cast<int32_t>(pixel_tiles);
    P.ldc = J.ldc;
    CPCSV_REQUIRE(J.ldc % 4 == 0 && J.ldc >= J.n_valid, "conv_gemm: ldc %lld", (long long)J.ldc);
  }
  CPCSV_REQUIRE(ntaps <= CPCSV_MAX_TAPS, "conv_gemm: %d taps > %d", ntaps, CPCSV_MAX_TAPS);
  CPCSV_REQUIRE(J.splits <= P.iters_total, "conv_gemm: splits %d > iterations %d", J.splits,
                P.iters_total);
  for (int i = 0; i < ntaps; ++i) {
    P.taps[i] = J.taps[i];
    CPCSV_REQUIRE(J.taps[i].out_off % 4 == 0, "conv_gemm: tap %d out_off alignment", i);
  }
  // CTA-pair mode (cta_group::2): jobs with at least two 128-row tiles whose B tile can be halved
  // (fprop / dgrad: any block_n >= 32 in steps of 16; wgrad: whole 64-channel atoms per CTA).
  // Alone a pair job is 0.79-0.87x the time of the single-CTA job on hi/lo-plane jobs and never slower
  // (profiles/r01_sweep_pair.txt); in the step 21.4-21.6 ms vs 22.1-22.3 ms with single CTAs
  // (profiles/r02_pair_soak.log).  The intermittent dead-lock of round 1 (6 of 12 runs) and of round 2's first
  // soaks (2 of 7 processes) was the TMEM allocation handshake between the two CTAs of a cluster (kernel prologue
  // above; profiles/r02_pair_hang_rootcause.md); with the fix 32 of 32 processes x 150 whole-step graph replays ran
  // clean under the conditions that hung before (profiles/r02_pair_trace_after_fix.log).
  CPCSV_REQUIRE(J.cta_pair == 0 || (J.mode == 0 && J.block_n >= 32 && (J.block_n / 2) % 8 == 0) ||
                    (J.mode == 1 && (J.block_n / 2) % 64 == 0),
                "conv_gemm: cta_pair needs block_n a multiple of 16 >= 32 (mode 0) or of 128 (mode 1)");
  const bool pair = J.cta_pair != 0 && P.m_tiles >= 2;
  P.m_units = pair ? (P.m_tiles + 1) / 2 : P.m_tiles;
  const int64_t total = static_cast<int64_t>(P.groups) * P.splits * P.n_tiles * P.m_units;
  CPCSV_REQUIRE(total > 0 && total < (1ll << 31), "conv_gemm: tile count %lld", (long long)total);
  P.total_tiles = static_cast<uint32_t>(total);
  P.idesc = make_idesc(static_cast<uint32_t>(J.dtype), static_cast<uint32_t>(J.mode),
                       pair ? 2 * kBlockM : kBlockM, static_cast<uint32_t>(J.block_n));
  P.b_plane_bytes = (pair ? J.block_n / 2 : J.block_n) * 128;
  P.stage_bytes = J.planes * (kAPlaneBytes + P.b_plane_bytes);
  const int smem_limit = J.planes == 1 ? kSinglePlaneSmemLimit : kSmemLimit;
  int stages = (smem_limit - 1024 - kBarrierBytes - kEpiBytes) / P.stage_bytes;
  if (stages > kMaxStages) stages = kMaxStages;
  CPCSV_REQUIRE(stages >= 2, "conv_gemm: tile does not fit shared memory");
  P.stages = stages;
  const size_t smem_bytes =
      static_cast<size_t>(stages) * P.stage_bytes + 1024 + kBarrierBytes + kEpiBytes;

  CUtensorMap tmA[2], tmB[2];
  uint32_t boxA[5], boxB[5];
  boxA[0] = 64; boxA[1] = J.tile_w; boxA[2] = 1; boxA[3] = J.tile_h; boxA[4] = J.tile_n;
  if (J.mode == 0) {
    boxB[0] = 64; boxB[1] = pair ? J.block_n / 2 : J.block_n; boxB[2] = 1; boxB[3] = 1; boxB[4] = 1;
  } else {
    for (int i = 0; i < 5; ++i) boxB[i] = boxA[i];
  }
  for (int pl = 0; pl < 2; ++pl) {
    const int src = pl < J.planes ? pl : 0;
    int rc = make_map(&tmA[pl], J.a[src], boxA, J.dtype, "conv_gemm A");
    if (rc) return rc;
    rc = make_map(&tmB[pl], J.b[src], boxB, J.dtype, "conv_gemm B");
    if (rc) return rc;
  }

  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(conv_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    kSmemLimit);
    if (attr_err == cudaSuccess)
      attr_err = cudaFuncSetAttribute(conv_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      kSmemLimit);
  });
  if (attr_err != cudaSuccess)
    return fail(static_cast<int>(attr_err), "conv_gemm: cudaFuncSetAttribute: %s",
                cudaGetErrorString(attr_err));

  const uint32_t sms = static_cast<uint32_t>(num_sms());
  if (pair) {
    const uint32_t clusters = P.total_tiles < sms / 2 ? P.total_tiles : sms / 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * clusters);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, conv_gemm_kernel<true>, tmA[0], tmA[1], tmB[0], tmB[1], P);
    if (e != cudaSuccess)
      return fail(static_cast<int>(e), "conv_gemm (pair): %s", cudaGetErrorString(e));
    return launched("conv_gemm");
  }
  const uint32_t grid = P.total_tiles < sms ? P.total_tiles : sms;
  conv_gemm_kernel<false><<<grid, kThreads, smem_bytes, stream>>>(tmA[0], tmA[1], tmB[0], tmB[1], P);
  return launched("conv_gemm");
}
