// DecoderKernelDU: kernel D of the decoder (decoder_2/simple .. last_layer -> int16 PCM) on the 5th-generation tensor cores.
//
// This is the kernel that runs when the context's decoder mode is LYRA_B200_DECODER_TENSOR.  Every fp32 GEMM of the tile
// (913 k MAC per stream-frame) is issued as split-precision TF32 `tcgen05.mma` (x = hi + lo, three MMAs per product, fp32
// accumulators in tensor memory); the CUDA cores only run the depthwise passes, the epilogues and the state I/O.
// Same inputs, outputs and streaming state as DecoderKernelD (net_kernels.cuh), so the two can alternate on one stream.
//
//   rows        a GEMM row of the T = 20 layers is (time row t, stream s) of the tile: m = t * 8 + s, owned by thread m
//               (warps 0..4).  Rows 0..127 are UMMA row block 0 (TMEM lane = m), rows 128..159 row block 1 (TMEM lane = m - 128;
//               its other lanes hold stale data, which only reaches accumulator rows nobody reads - GEMM rows are independent).
//   residual    A operand in TENSOR MEMORY, written by the row's own thread with tcgen05.st (hi and lo column blocks): the
//   units       activations never take a round trip through shared memory between the depthwise conv, the two 1x1 convolutions
//               and last_layer.  B = weights from shared memory.  The A operand is staged one k-half (32 channels) at a time in
//               the same 64 columns: the row warps write channels 32..63 once the MMAs that read 0..31 have completed (a_free).
//               With D that is 128 columns per row block, 256 per tile: two blocks share the SM's tensor memory.
//   decoder_2/  computed TRANSPOSED: the 640 weight rows (tap j, phase r, cout) are the M dimension (five 128-row blocks, A operand
//   simple      from shared memory) and the tile's 32 (input row, stream) pairs the N dimension (B operand, 16 KB per half): a
//               16-cycle MMA instead of an 80-cycle one whose 128 rows would be three-quarters padding, and an epilogue in
//               which every TMEM lane carries live data.  The two taps land in different lanes; they meet in shared memory.
//   last_layer  ONE 64 x 64 GEMM P[row][tap * 16 + n] = sum_ci lrelu(u')[row][ci] * W[(tap, ci)][n] on the A operand the last
//               residual unit's epilogue leaves in tensor memory; the four taps are summed across time rows afterwards.
//   weights     pre-split on the host into hi / lo core-matrix chunks (net_params.h kDuChunkBytes), streamed by one producer
//               thread with TMA bulk copies through a 2-stage shared-memory ring; a stage is released by tcgen05.commit when
//               the MMAs that read it have completed.  Build switch LYRA_DU_RAW=1: decoder_2/simple's chunks (three quarters of
//               the stream) travel unsplit - half the bytes - and the row warps split them in place.  Measured slower (that
//               phase 26 k -> 34 k cycles): with two stages the TMA -> split -> MMA -> release chain is longer than the bytes saved.
//   state       the overlap tail, the last_layer tail and the ring blocks of units 0 and 1 move by TMA bulk copies in both directions
//               (written back whole, with the lanes of inactive streams left as loaded); kernel C's tile and unit 2's 36 KB ring
//               block are read from / written to global memory directly so that the block stays at 110 KB of shared memory.
//   roles       warps 0..7: rows / epilogues / state;  warp 8 lane 0: MMA issue;  warp 9 lane 0: TMA producer.
// Arithmetic: products carry fp32-level accuracy (error terms below 2^-21 relative) but not the oracle's fmaf-chain rounding or
// summation order: decoded PCM is compared with a tolerance (tests/parity_cases.py TENSOR_PCM_TOL_LSB), never bit for bit.
#pragma once

#include <type_traits>

#include "net_kernels.cuh"

namespace lyra_b200 {

struct DecDU {
  static constexpr int S = 8;
  static constexpr int kRowWarps = 8, kRowThreads = kRowWarps * 32;
  static constexpr int kMmaWarp = 8, kTmaWarp = 9;
  static constexpr int NT = 320;
  static constexpr int kStagesW = 2;
  static constexpr int LDU = 161;                             // u: f32 [64][LDU], element (c, row = t * 8 + s); odd stride: lanes that
                                                              // differ in c (decoder_2/simple epilogue) hit different banks
  // shared memory (bytes): 110 KB, sized so that a kernel-A block (105 KB, 96 registers x 320 threads) fits on the SM beside this
  // kernel's block: the FMA-bound encoder front end then fills the issue slots this latency-bound kernel leaves empty.
  //   u        the residual stream of the three units, f32 [64][LDU]
  //   region   decoder_2/simple's B operand X (hi | lo, 32 KB)  ->  once its MMAs are done: the carried overlap tail (10 KB), the ring
  //            blocks of units 0 and 1 (4 + 12 KB), PCM staging.  Unit 2's ring block (36 KB, dilation 9) stays in global memory (L2):
  //            its rows are read and replaced in place.  Kernel C's tile is read from global memory as well.
  static constexpr int kU = 0;
  static constexpr int kXc = kU + 64 * LDU * 4;               // decoder_2/simple B operand: hi | lo, each [128/4][4][8][4] f32
  static constexpr int kXPart = 32 * 4 * 32 * 4;              // 16,384
  static constexpr int kRegion = kXc, kRegionBytes = 2 * kXPart;
  static constexpr int kOv = kRegion;                         // decoder_2/simple overlap tail f32 [64][5][8]: loaded, consumed, rewritten, stored
  static constexpr int kRing0 = kOv + 64 * 5 * S * 4, kRing1 = kRing0 + 64 * 2 * S * 4;     // ring blocks [64][R][8] f32, R = 2, 6
  static constexpr int kStage = kRing1 + 64 * 6 * S * 4;      // at the end: PCM staging int16 [8][320]
  static constexpr int kSl = kRegion + kRegionBytes;          // last_layer carried tail f32 [48][8]
  static constexpr int kSlOut = kSl + 48 * S * 4;             // ... and its successor
  static constexpr int kDw4 = kSlOut + 48 * S * 4;            // depthwise parameters per channel: float4 {w0, w1, w2, bias} [3][64]
  static constexpr int kW = kDw4 + 3 * 256 * 4;               // weight ring
  static constexpr int kI = kW + kStagesW * kDuChunkBytes;    // slot[S], active[S], n18[S]
  // LYRA_DU_SMEM_PAD: request more than the layout needs, e.g. 6144 -> 116 KB = at most one block of this kernel per SM (the rest of
  // the SM is left to a kernel-A / B / C block)
#ifndef LYRA_DU_SMEM_PAD
#define LYRA_DU_SMEM_PAD 0
#endif
  static constexpr int kSmemBytes = kI + 3 * S * 4 + 16 + LYRA_DU_SMEM_PAD;     // + n18[S]
  static_assert(kStage + S * 320 * 2 <= kRegion + kRegionBytes, "overlap tail, two ring blocks and PCM staging must fit in the X region");
  static_assert(kXc % 128 == 0 && kOv % 128 == 0 && kRing0 % 128 == 0 && kRing1 % 128 == 0 && kW % 128 == 0 && kSl % 16 == 0 && kDw4 % 16 == 0,
                "bulk-copy / descriptor alignment");
  static_assert(kSmemBytes - LYRA_DU_SMEM_PAD <= 113 * 1024, "must leave room for a kernel-A block on the SM");
  // tensor memory columns: 256, half of the SM's, so that two blocks of this kernel run at once.  decoder_2/simple: block mb at
  // columns 32 mb.  Afterwards per row block rb: A hi | A lo of ONE k-half (channels 0..31, then 32..63 in the same columns) | D
  static constexpr int kTmemCols = 256;
  static constexpr int kColAhi = 0, kColAlo = 32, kColD = 64, kRbStride = 128;
  static_assert(5 * 32 <= kTmemCols && 2 * kRbStride <= kTmemCols, "decoder_2/simple's accumulators and both row blocks fit");
};

struct DecDUShared {
  LyraMbar w_full[DecDU::kStagesW], w_empty[DecDU::kStagesW];
  LyraMbar raw_full[DecDU::kStagesW];   // producer -> row warps: an unsplit decoder_2/simple chunk has landed in the stage's hi half
  LyraMbar s_full[DecDU::kStagesW];     // row warps -> MMA issuer: the chunk is split (hi | lo) in place
  LyraMbar in_full;        // producer -> row warps: the last_layer tail has landed
  LyraMbar ov_full;        // producer -> row warps: the overlap tail has landed (in the X region, after decoder_2/simple's MMAs)
  LyraMbar a_ready;        // row warps -> MMA issuer: the operand of the next GEMM (or k-half of it) is in place
  LyraMbar a_free;         // MMA issuer -> row warps: the MMAs that read the A operand's first k-half have completed
  LyraMbar d_ready;        // MMA issuer -> row warps: the accumulators of the GEMM are complete
  LyraMbar ring_full[2];   // producer -> row warps: ring block u (units 0, 1) has landed
  LyraMbar tmem_ready;     // MMA warp -> everybody: tensor memory is allocated, tmem_base is valid
  LyraMbar tmem_done;      // row warps -> MMA warp: the last tcgen05.ld of the tile has completed (LYRA_DU_EARLY_DEALLOC)
  uint32_t tmem_base;
};

__device__ __forceinline__ void DuSplit(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(__fsub_rn(x, __uint_as_float(hi)));
}

// All row threads: publish the TMEM / shared-memory operand of the next GEMM to the MMA issuer.
__device__ __forceinline__ void DuArriveA(DecDUShared* sh) {
  lyra_tmem_wait_st();
  lyra_tmem_wait_ld();
  lyra_fence_proxy_async();
  lyra_tc_fence_before_sync();
  __syncwarp();
  if ((threadIdx.x & 31) == 0) lyra_mbar_arrive(&sh->a_ready);
}

// The thread's 64 accumulator columns in four groups of 16, with the tcgen05.ld of group g + 1 in flight while f(g, v) runs
// (tcgen05.wait::ld covers every earlier load, so the next one is issued right after the wait).  Warp-collective.
#ifndef LYRA_DU_PIPE
#define LYRA_DU_PIPE 1
#endif
#ifndef LYRA_DU_EARLY_DEALLOC
#define LYRA_DU_EARLY_DEALLOC 1
#endif
template <typename F>
__device__ __forceinline__ void DuForEachAccGroup(uint32_t taddr, F f) {
  uint32_t v[2][16];
  lyra_tmem_ld<16>(taddr, v[0]);
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    lyra_tmem_wait_ld();
    if (LYRA_DU_PIPE && g < 3) lyra_tmem_ld<16>(taddr + (uint32_t)(16 * (g + 1)), v[(g + 1) & 1]);
    f(g * 16, v[g & 1]);
    if (!LYRA_DU_PIPE && g < 3) lyra_tmem_ld<16>(taddr + (uint32_t)(16 * (g + 1)), v[(g + 1) & 1]);
  }
}

// All row threads: between the two k-halves of an A operand, wait until the MMAs that read the first half have completed.
__device__ __forceinline__ void DuWaitAFree(DecDUShared* sh, unsigned& par) {
  lyra_mbar_wait(&sh->a_free, par);
  par ^= 1;
  lyra_tc_fence_after_sync();
}

// All row threads: the next GEMM's A operand, 16 channels at a time, make(c0, hi, lo) for c0 = 0, 16 | 32, 48, written to
// the row's A columns in two k-halves: channels 0..31 are published, then 32..63 overwrite them once the MMAs that read the
// first half have completed.
template <typename F>
__device__ __forceinline__ void DuWriteA(DecDUShared* sh, uint32_t trow, bool has_row, unsigned& f_par, F make) {
#pragma unroll 1
  for (int h = 0; h < 2; ++h) {
    if (h == 1) DuWaitAFree(sh, f_par);
    if (has_row) {
#pragma unroll 1
      for (int c0 = 32 * h; c0 < 32 * h + 32; c0 += 16) {
        uint32_t hi[16], lo[16];
        make(c0, hi, lo);
        lyra_tmem_st<16>(trow + DecDU::kColAhi + (uint32_t)(c0 - 32 * h), hi);
        lyra_tmem_st<16>(trow + DecDU::kColAlo + (uint32_t)(c0 - 32 * h), lo);
      }
    }
    DuArriveA(sh);
  }
}

// All row threads: the GEMM's accumulators (64 columns at trow + kColD) -> the next GEMM's A operand in two k-halves,
// f(c0, v, hi, lo) converting 16 channels.  The next GEMM's first MMAs overwrite D, so columns 32..63 are loaded into
// registers before the first half is published and converted after a_free.  Warp-collective.
template <typename F>
__device__ __forceinline__ void DuAccToA(DecDUShared* sh, uint32_t trow, bool has_row, unsigned& f_par, F f) {
  uint32_t v[2][16];
  auto put = [&](int c0, const uint32_t (&x)[16]) {
    uint32_t hi[16], lo[16];
    f(c0, x, hi, lo);
    lyra_tmem_st<16>(trow + DecDU::kColAhi + (uint32_t)(c0 % 32), hi);
    lyra_tmem_st<16>(trow + DecDU::kColAlo + (uint32_t)(c0 % 32), lo);
  };
  if (has_row) {
    const uint32_t td = trow + DecDU::kColD;
    lyra_tmem_ld<16>(td, v[0]);
    lyra_tmem_wait_ld();
    lyra_tmem_ld<16>(td + 16u, v[1]);
    put(0, v[0]);
    lyra_tmem_wait_ld();
    lyra_tmem_ld<16>(td + 32u, v[0]);
    put(16, v[1]);
    lyra_tmem_ld<16>(td + 48u, v[1]);
  }
  DuArriveA(sh);                                             // (waits for the loads: D is read in full)
  DuWaitAFree(sh, f_par);
  if (has_row) {
    put(32, v[0]);
    put(48, v[1]);
  }
  DuArriveA(sh);
}

__global__ void __launch_bounds__(DecDU::NT, 2)
DecoderKernelDU(const uint8_t* __restrict__ blob, DecoderParams P, TileIo io, const float* __restrict__ mid,
                float* __restrict__ state, int* __restrict__ n18g, int16_t* __restrict__ pcm, int ntiles) {
  using L = DecDU;
  constexpr int S = L::S, LDU = L::LDU;
  unsigned char* smem = LYRA_DYN_SMEM();
  float* smf = reinterpret_cast<float*>(smem);                // every f32 buffer below is addressed as smf[float offset]
  float* u = smf + L::kU / 4;
  unsigned char* wring = smem + L::kW;
  float* ov = smf + L::kOv / 4;
  float* sl = smf + L::kSl / 4;
  float* slo = smf + L::kSlOut / 4;
  int* slot = reinterpret_cast<int*>(smem + L::kI);
  int* active = slot + S;
  int* n18 = active + S;                                      // n18[S]: tile summary (LoadTileMeta)
  LYRA_STATIC_SMEM(DecDUShared, sh, 1);
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // Launched as clusters of two CTAs (engine.cu): when both tiles of the pair have work, the CTAs share the weight stream - each
  // producer loads one half of every chunk and multicasts it into both CTAs' rings, halving the L2 traffic of the kernel's
  // dominant stream (883 KB of weights per tile).  A CTA whose partner is a padding block or an idle tile runs on its own.
  if ((int)blockIdx.x >= ntiles) return;                    // padding block of an odd grid (its partner sees that and runs solo)
  bool pair = false;
  if (lyra_cluster_nctarank() == 2) {
    auto live = [&](int block) {
      if (block >= ntiles) return false;
      const int tl = io.tile_list[block];
      bool any = false;
      for (int ss = 0; ss < S; ++ss) {
        const int sl = io.slot_of_stream[tl * S + ss];
        any |= sl >= 0 && !(io.skip != nullptr && io.skip[sl]);
      }
      return any;
    };
    pair = live((int)blockIdx.x) && live((int)blockIdx.x ^ 1);      // the same value in both CTAs of the pair
  }
  const unsigned rank = lyra_cluster_ctarank();

  if (tid == 0) {
    for (int i = 0; i < L::kStagesW; ++i) {
      lyra_mbar_init(&sh->w_full[i], 1);
      lyra_mbar_init(&sh->w_empty[i], pair ? 2u : 1u);
      lyra_mbar_init(&sh->raw_full[i], 1);
      lyra_mbar_init(&sh->s_full[i], L::kRowWarps);
    }
    lyra_mbar_init(&sh->in_full, 1);
    lyra_mbar_init(&sh->ov_full, 1);
    lyra_mbar_init(&sh->tmem_ready, 1);
    lyra_mbar_init(&sh->tmem_done, 5);
    lyra_mbar_init(&sh->a_ready, L::kRowWarps);
    lyra_mbar_init(&sh->a_free, 1);
    lyra_mbar_init(&sh->d_ready, 1);
    for (int i = 0; i < 2; ++i) lyra_mbar_init(&sh->ring_full[i], 1);
    lyra_mbar_fence_init();
  }
  int tile;
  LoadTileMeta<S>(io, n18g, slot, active, n18, tile);       // two block barriers inside: the barrier inits are visible after it
  if (pair) lyra_cluster_sync();                              // both CTAs' barriers exist before any remote copy or arrival
  float* st = state + (size_t)tile * DecStateD::kUnits * S;
  const uint8_t* chunks = blob + P.du_chunks;
  int ph = 0;
  const bool idle = n18[S] == kTileIdle;
  if (!idle) PrefetchTileState<LYRA_PREFETCH_STATE>(st, DecStateD::kUnits * S * 4);      // unit 2 reads its ring block from global memory
  // Tensor memory is taken AFTER the block barriers above, by the MMA warp alone.  A block takes 256 of the SM's 512 columns, so
  // the two blocks of this kernel that fit on an SM (shared memory, registers) run at once: one tile's latency-bound residual
  // units overlap the other's stream-bound decoder_2/simple phase.
  if (!idle && warp == L::kMmaWarp) {
    lyra_tmem_alloc(&sh->tmem_base, L::kTmemCols);
    lyra_tc_fence_before_sync();
    if (lane == 0) lyra_mbar_arrive(&sh->tmem_ready);
  }
  auto tmem_address = [&]() { lyra_mbar_wait(&sh->tmem_ready, 0); lyra_tc_fence_after_sync(); return sh->tmem_base; };                      // every stream of the tile sits this call out: nothing to do (pair is false then)

  // ================================================= TMA producer =================================================
  if (idle) {
  } else if (warp == L::kTmaWarp) {
    if (lane == 0) {
      lyra_bulk_g2s(sl, st + (size_t)DecStateD::kLast * S, 48u * S * 4, &sh->in_full);
      for (int c = 0; c < kDuNumChunks; ++c) {
        const int stg = c % L::kStagesW;
        if (c >= L::kStagesW) lyra_mbar_wait(&sh->w_empty[stg], (unsigned)((c / L::kStagesW - 1) & 1));
        // decoder_2/simple chunks arrive unsplit (half the bytes; the row warps split them in place), the others pre-split
        const bool raw = kDuRawUp2 && c < kDuUp2Chunks;
        const unsigned bytes = raw ? (unsigned)kDuRawChunkBytes : (unsigned)kDuChunkBytes;
        const uint8_t* src = c < kDuUp2Chunks ? chunks + (size_t)c * kDuRawChunkBytes
                                              : chunks + (size_t)kDuUp2Chunks * kDuRawChunkBytes + (size_t)(c - kDuUp2Chunks) * kDuChunkBytes;
        LyraMbar* full = raw ? &sh->raw_full[stg] : &sh->w_full[stg];
        if (pair) {
          // arm this CTA's barrier for the whole chunk; this producer fetches its half and multicasts it to both CTAs
          const unsigned half = bytes / 2;
          lyra_bulk_multi_begin(full, bytes);
          lyra_bulk_g2s_mc(wring + (size_t)stg * kDuChunkBytes + rank * half, src + rank * half, half, full, 3u);
        } else {
          lyra_bulk_g2s(wring + (size_t)stg * kDuChunkBytes, src, bytes, full);
        }
        if (c == kDuUp2Chunks + L::kStagesW - 1) {
          // the wait above covered the last decoder_2/simple chunk's MMAs, the last readers of X: the overlap tail and the ring
          // blocks of units 0 and 1 may land on it
          lyra_bulk_g2s(ov, st + (size_t)DecStateD::kUp2 * S, 64u * 5 * S * 4, &sh->ov_full);
          lyra_bulk_g2s(smem + L::kRing0, st + (size_t)DecStateD::kRing0 * S, 64u * 2 * S * 4, &sh->ring_full[0]);
          lyra_bulk_g2s(smem + L::kRing1, st + (size_t)DecStateD::kRing1 * S, 64u * 6 * S * 4, &sh->ring_full[1]);
        }
      }
    }
  }

  // ================================================= MMA issuer ===================================================
  else if (warp == L::kMmaWarp) {
    if (lane == 0) {
      const uint32_t tmem = tmem_address();
      unsigned a_par = 0;
      int c = 0;                                             // weight chunk counter
      auto wait_a = [&]() { lyra_mbar_wait(&sh->a_ready, a_par); a_par ^= 1; lyra_tc_fence_after_sync(); };
      static_assert(kDuUp2Chunks % L::kStagesW == 0, "the split and the pre-split chunks use separate barrier phase sequences");
      auto wait_chunk_at = [&](int ci) -> const unsigned char* {
        if (!kDuRawUp2) lyra_mbar_wait(&sh->w_full[ci % L::kStagesW], (unsigned)((ci / L::kStagesW) & 1));
        else if (ci < kDuUp2Chunks) lyra_mbar_wait(&sh->s_full[ci % L::kStagesW], (unsigned)((ci / L::kStagesW) & 1));
        else lyra_mbar_wait(&sh->w_full[ci % L::kStagesW], (unsigned)(((ci - kDuUp2Chunks) / L::kStagesW) & 1));
        lyra_tc_fence_after_sync();
        return wring + (size_t)(ci % L::kStagesW) * kDuChunkBytes;
      };
      auto wait_chunk = [&]() -> const unsigned char* { return wait_chunk_at(c); };
      auto release_chunk = [&]() {                           // the stage is free once the MMAs of BOTH CTAs of a pair have read it
        if (pair) lyra_umma_commit_mc(&sh->w_empty[c % L::kStagesW], 3u);
        else lyra_umma_commit(&sh->w_empty[c % L::kStagesW]);
        ++c;
      };
      // ---- decoder_2/simple, transposed: D_mb[128 x 32] = Wt_mb[128 x 128] * X[32 x 128]^T for the five row blocks of Wt.
      //      This phase is bound by the delivery of its 640 KB of weights (about 30 bytes per cycle and SM with every SM streaming,
      //      measured; neither a deeper ring nor multicast changes it), not by the 240 small MMAs.
      wait_a();
      {
        const uint32_t idesc = lyra_umma_idesc_tf32(128, 32);
        const uint32_t lboW = 16u * 128u, lboX = 4u * 128u;
        const unsigned char* xh = smem + L::kXc;
        const unsigned char* xl = xh + L::kXPart;
        for (int mb = 0; mb < 5; ++mb)
          for (int kc = 0; kc < 8; ++kc) {
            const unsigned char* wst = wait_chunk();
            for (int k2 = 0; k2 < 2; ++k2) {
              const int ks = kc * 2 + k2;
              const uint64_t ah = lyra_umma_desc(wst + (size_t)k2 * 2 * lboW, lboW, 128);
              const uint64_t al = lyra_umma_desc(wst + kDuChunkBytes / 2 + (size_t)k2 * 2 * lboW, lboW, 128);
              const uint64_t bh = lyra_umma_desc(xh + (size_t)ks * 2 * lboX, lboX, 128);
              const uint64_t bl = lyra_umma_desc(xl + (size_t)ks * 2 * lboX, lboX, 128);
              const uint32_t d = tmem + (uint32_t)(mb * 32);
              lyra_umma_tf32(d, al, bh, idesc, ks > 0);                             // small terms first
              lyra_umma_tf32(d, ah, bl, idesc, true);
              lyra_umma_tf32(d, ah, bh, idesc, true);
            }
            release_chunk();
          }
        lyra_umma_commit(&sh->d_ready);
      }
      // ---- 3 x (pw1, pw2) and last_layer: K = N = 64, A in tensor memory, two row blocks
      {
        const uint32_t idesc = lyra_umma_idesc_tf32(128, 64);
        const uint32_t lboW = 8u * 128u;
        for (int g = 0; g < 7; ++g) {
          for (int kc = 0; kc < 2; ++kc) {                   // k-half kc: channels 32 kc .. 32 kc + 31, in the same A columns for both
            wait_a();
            const unsigned char* wst = wait_chunk();
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
              const int ks = kc * 4 + k4;
              const uint64_t bh = lyra_umma_desc(wst + (size_t)k4 * 2 * lboW, lboW, 128);
              const uint64_t bl = lyra_umma_desc(wst + kDuChunkBytes / 2 + (size_t)k4 * 2 * lboW, lboW, 128);
#pragma unroll
              for (int term = 0; term < 3; ++term)
#pragma unroll
                for (int rb = 0; rb < 2; ++rb) {             // alternate the two row blocks' accumulators: MMAs into one TMEM tile run as
                                                             // a dependent chain (measured 56 cycles each here), interleaved ones overlap (24)
                  const uint32_t base = tmem + (uint32_t)(rb * L::kRbStride);
                  lyra_umma_tf32_ts(base + L::kColD, base + (term == 0 ? L::kColAlo : L::kColAhi) + (uint32_t)(8 * k4), term == 1 ? bl : bh, idesc,
                                    ks > 0 || term > 0);
                }
            }
            release_chunk();
            if (kc == 0) lyra_umma_commit(&sh->a_free);      // the row warps may overwrite the A columns with the second half
          }
          lyra_umma_commit(&sh->d_ready);
        }
      }
    }
#if LYRA_DU_EARLY_DEALLOC
    // Tensor memory goes back as soon as the row warps have read the last accumulators - not at block exit, after the PCM and
    // state stores - so that a block that asks for it meanwhile does not wait for those stores.
    __syncwarp();
    lyra_mbar_wait(&sh->tmem_done, 0);
    lyra_tc_fence_after_sync();
    lyra_tmem_dealloc(sh->tmem_base, L::kTmemCols);
#endif
  }

  // ================================================= row warps ====================================================
  else {
    const int row = tid;                                     // rows 0..159 (warps 0..4) are GEMM rows (t, s)
    const int t = row / S, s = row % S;
    const int rb = row / 128;
    const bool has_row = warp < 5;                           // whole warps: tcgen05.ld / st are warp-collective
    unsigned d_par = 0, f_par = 0;
    LYRA_PHASE(3, ph);
    auto wait_d = [&]() { lyra_mbar_wait(&sh->d_ready, d_par); d_par ^= 1; lyra_tc_fence_after_sync(); };
    auto row_sync = [&]() { lyra_named_bar_sync(1, L::kRowThreads); };

    // ---- X: kernel C's tile [128 ch][4 rows][8 streams] -> B operand (split, core-matrix layout, row = (x-row, stream), k = ch)
    if (tid < 3 * 64) {                                       // depthwise parameters per channel (read after several barriers)
      const int un = tid / 64, c = tid % 64;
      const float* w = BlobPtr<float>(blob, P.r2[un].dw.w);
      reinterpret_cast<float4*>(smf + L::kDw4 / 4)[tid] = make_float4(w[c], w[64 + c], w[128 + c], BlobPtr<float>(blob, P.r2[un].dw.bias)[c]);
    }
    {
      const float* in = mid + (size_t)tile * 128 * 4 * S;     // kernel C's tile, straight from global memory (L2): 16 floats per thread
      float* xh = smf + L::kXc / 4;
      float* xl = xh + L::kXPart / 4;
      for (int item = tid; item < 32 * 4 * 8; item += L::kRowThreads) {
        const int i = item % 8, g = (item / 8) % 4, kg = item / 32;
        uint32_t hh[4], ll[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) DuSplit(in[((4 * kg + j) * 4 + g) * S + i], hh[j], ll[j]);
        const int o = ((kg * 4 + g) * 8 + i) * 4;
        *reinterpret_cast<float4*>(xh + o) = make_float4(__uint_as_float(hh[0]), __uint_as_float(hh[1]), __uint_as_float(hh[2]), __uint_as_float(hh[3]));
        *reinterpret_cast<float4*>(xl + o) = make_float4(__uint_as_float(ll[0]), __uint_as_float(ll[1]), __uint_as_float(ll[2]), __uint_as_float(ll[3]));
      }
    }
    DuArriveA(sh);
    LYRA_PHASE(3, ph);

    // ---- decoder_2/simple weights: every chunk lands as plain fp32 in the hi half of its stage; split it in place (hi stays,
    //      lo goes to the other half) while the tensor core works on the previous one.  All eight row warps: they have nothing
    //      else to do until the layer's accumulators are complete.
    for (int c = 0; kDuRawUp2 && c < kDuUp2Chunks; ++c) {
      const int stg = c % L::kStagesW;
      lyra_mbar_wait(&sh->raw_full[stg], (unsigned)((c / L::kStagesW) & 1));
      float4* wh = reinterpret_cast<float4*>(wring + (size_t)stg * kDuChunkBytes);
      float4* wl = wh + kDuRawChunkBytes / 16;
#pragma unroll
      for (int i = tid; i < kDuRawChunkBytes / 16; i += L::kRowThreads) {
        const float4 v = wh[i];
        uint32_t h0, h1, h2, h3, l0, l1, l2, l3;
        DuSplit(v.x, h0, l0); DuSplit(v.y, h1, l1); DuSplit(v.z, h2, l2); DuSplit(v.w, h3, l3);
        wh[i] = make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(h2), __uint_as_float(h3));
        wl[i] = make_float4(__uint_as_float(l0), __uint_as_float(l1), __uint_as_float(l2), __uint_as_float(l3));
      }
      lyra_fence_proxy_async();                              // the tensor core reads the stage through the asynchronous proxy
      __syncwarp();
      if (lane == 0) lyra_mbar_arrive(&sh->s_full[stg]);
    }
    LYRA_PHASE(3, ph);

    // ---- decoder_2/simple epilogue.  TMEM lane = weight row m = (tap j, phase r, cout), column = (x-row, stream).
    //      out[q][r][co] = (P[j=1][x=q] + bias + carried overlap (q = 0)) + P[j=0][x=q-1]; q = 4 is the new overlap tail.
    //      Pass 0 stores the j = 1 terms (every element of u), pass 1 adds the j = 0 terms.  j is uniform per (warp, block).
    wait_d();
    const uint32_t tq = tmem_address() + ((uint32_t)(32 * (warp % 4)) << 16);      // this warp's TMEM lane window
    const uint32_t trow = tq + (uint32_t)(rb * L::kRbStride);                      // ... at the thread's row block (residual units)
    lyra_mbar_wait(&sh->ov_full, 0);                         // the carried overlap tail (it landed on X once the MMAs above were done)
    LYRA_PHASE(3, ph);
    {
      const float* b = BlobPtr<float>(blob, P.up2.bias);
      const int mb0 = warp < 4 ? 0 : 3, mb1 = warp < 4 ? 3 : 5;
      for (int pass = 0; pass < 2; ++pass) {
        for (int mb = mb0; mb < mb1; ++mb) {
          const int m = mb * 128 + 32 * (warp % 4) + lane;
          const int j = m / 320;
          if (j != 1 - pass) continue;                       // warp-uniform
          const int r = (m % 320) / 64, co = m % 64;
          const float bias = b[co];
          float* uc = u + co * LDU + r * S;
          float* oc = ov + (co * 5 + r) * S;
          uint32_t v2[2][16];                                // both halves of the row in flight before the first is consumed
          lyra_tmem_ld<16>(tq + (uint32_t)(mb * 32), v2[0]);
          lyra_tmem_ld<16>(tq + (uint32_t)(mb * 32 + 16), v2[1]);
          lyra_tmem_wait_ld();
#pragma unroll
          for (int half = 0; half < 2; ++half) {
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              const int x = half * 2 + k / 8, ss = k % 8;
              const float p = __uint_as_float(v2[half][k]);
              if (pass == 0) {
                const float y = __fadd_rn(p, bias);
                uc[(5 * x) * S + ss] = __fadd_rn(y, x == 0 ? oc[ss] : 0.0f);
              } else if (x < 3) {
                float* o = uc + (5 * (x + 1)) * S + ss;
                *o = __fadd_rn(*o, p);
              } else if (active[ss]) {
                oc[ss] = __fsub_rn(__fadd_rn(__fadd_rn(p, bias), 0.0f), bias);
              }
            }
          }
        }
        lyra_fence_proxy_async();                            // pass 1: the rewritten overlap block, before its bulk store
        row_sync();
      }
      if (tid == 0) { lyra_bulk_s2g(st + (size_t)DecStateD::kUp2 * S, ov, 64u * 5 * S * 4); lyra_bulk_commit(); }
    }
    LYRA_PHASE(3, ph);

    // ---- decoder_2: three residual units, d = dw(lrelu(u)); h = lrelu(pw1(d)); u' = pw2(h) + u
    auto unit_body = [&](auto unit_c) {
      constexpr int unit = decltype(unit_c)::value;
      constexpr int dil = unit == 0 ? 1 : (unit == 1 ? 3 : 9), R = 2 * dil;
      // units 0, 1: ring block in shared memory (bulk-loaded, bulk-stored); unit 2 (R = 18, 36 KB): rows are read from and written
      // to the global block directly - a thread touches 32-byte runs of 8 streams, and every read precedes the row barrier
      // that the writes follow, exactly as for the shared-memory blocks
      constexpr bool ring_in_smem = unit < 2;
      constexpr int ring_off = (unit == 0 ? L::kRing0 : L::kRing1) / 4;                             // [64][R][S] f32 (units 0, 1)
      const ResF32& p = P.r2[unit];
      float* gring = st + (size_t)(unit == 0 ? DecStateD::kRing0 : (unit == 1 ? DecStateD::kRing1 : DecStateD::kRing2)) * S;
      const float* ringp = ring_in_smem ? smf + ring_off : gring;
      const int base = (n18[s] * 20) % R;                    // ring slot of this frame's row 0 for this stream
      if (ring_in_smem) lyra_mbar_wait(&sh->ring_full[unit < 2 ? unit : 0], 0);
      LYRA_PHASE(3, ph);
      // depthwise conv (k = 3, dilation dil) over LeakyReLU(u) -> A operand (hi, lo) of pw1, in two k-halves.  Rows before this
      // frame come from the ring (already activated): source pointer, channel stride and negative slope are selected once, the
      // loop is branch-free
      {
        const float4* w4 = reinterpret_cast<const float4*>(smf + L::kDw4 / 4) + unit * 64;      // per channel {w0, w1, w2, bias}
        const bool r1 = t - dil < 0, r0 = t - 2 * dil < 0;
        const float* p2 = u + row;
        const float* p1 = r1 ? ringp + ((base + t - dil + 2 * R) % R) * S + s : u + row - dil * S;
        const float* p0 = r0 ? ringp + ((base + t - 2 * dil + 2 * R) % R) * S + s : u + row - 2 * dil * S;
        const int st1 = r1 ? R * S : LDU, st0 = r0 ? R * S : LDU;
        const float n1 = r1 ? 1.0f : 0.3f, n0 = r0 ? 1.0f : 0.3f;
        DuWriteA(sh, trow, has_row, f_par, [&](int c0, uint32_t (&hi)[16], uint32_t (&lo)[16]) {
          float x1v[16], x0v[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) { x1v[j] = p1[(c0 + j) * st1]; x0v[j] = p0[(c0 + j) * st0]; }      // the (possibly global) loads first
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int c = c0 + j;
            float x2 = p2[c * LDU], x1 = x1v[j], x0 = x0v[j];
            const float4 wc = w4[c];
            x2 = fmaxf(x2, __fmul_rn(x2, 0.3f));            // LeakyReLU; ring rows are stored activated: slope 1 leaves them as they are
            x1 = fmaxf(x1, __fmul_rn(x1, n1));
            x0 = fmaxf(x0, __fmul_rn(x0, n0));
            float acc = __fmaf_rn(x0, wc.x, 0.0f);
            acc = __fmaf_rn(x1, wc.y, acc);
            acc = __fmaf_rn(x2, wc.z, acc);
            DuSplit(__fadd_rn(acc, wc.w), hi[j], lo[j]);
          }
        });
      }
      LYRA_PHASE(3, ph);
      // The newest min(20, R) rows of lrelu(u) replace the ring's oldest entries (every slot: R <= 20).  The copy runs in two
      // halves, each behind one of the unit's two GEMMs, so the row threads are busy while the tensor core works.
      row_sync();                                            // all ring reads are done
      const bool upd = has_row && t >= 20 - R && active[s];
      auto ring_update = [&](int c_lo) {
        if (!upd) return;
        float* wp = (ring_in_smem ? smf + ring_off : gring) + ((base + t) % R) * S + s;
        const float* ip = u + row;
#pragma unroll 16
        for (int c = c_lo; c < c_lo + 32; ++c) wp[c * (R * S)] = LeakyRelu(ip[c * LDU]);
      };
      ring_update(0);
      LYRA_PHASE(3, ph);
      // pw1 epilogue: bias, LeakyReLU, split -> A operand of pw2 (same TMEM columns: pw1's MMAs have completed)
      wait_d();
      LYRA_PHASE(3, ph);
      {
        const float* b1 = BlobPtr<float>(blob, p.pw1.bias);
        DuAccToA(sh, trow, has_row, f_par, [&](int c0, const uint32_t (&v)[16], uint32_t (&hi)[16], uint32_t (&lo)[16]) {
#pragma unroll
          for (int j = 0; j < 16; ++j) DuSplit(LeakyRelu(__fadd_rn(__uint_as_float(v[j]), b1[c0 + j])), hi[j], lo[j]);
        });
      }
      ring_update(32);
      lyra_fence_proxy_async();
      row_sync();
      if (ring_in_smem && tid == 0) { lyra_bulk_s2g(gring, smf + ring_off, (unsigned)(64 * R * S * 4)); lyra_bulk_commit(); }
      LYRA_PHASE(3, ph);
      // pw2 epilogue: bias + residual.  Units 0, 1: u' back to shared memory (the next depthwise conv reads neighbouring rows);
      // unit 2: LeakyReLU(u') straight into tensor memory as the A operand of last_layer
      wait_d();
      LYRA_PHASE(3, ph);
      {
        const float* b2 = BlobPtr<float>(blob, p.pw2.bias);
        float* uc = u + row;
        if constexpr (unit == 2) {
          DuAccToA(sh, trow, has_row, f_par, [&](int c0, const uint32_t (&v)[16], uint32_t (&hi)[16], uint32_t (&lo)[16]) {
            float res[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) res[j] = uc[(c0 + j) * LDU];               // the residual: loads first, one exposed latency
#pragma unroll
            for (int j = 0; j < 16; ++j) DuSplit(LeakyRelu(__fadd_rn(__fadd_rn(__uint_as_float(v[j]), b2[c0 + j]), res[j])), hi[j], lo[j]);
          });
        } else {
          if (has_row) {
            DuForEachAccGroup(trow + L::kColD, [&](int c0, const uint32_t (&v)[16]) {
              float res[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) res[j] = uc[(c0 + j) * LDU];             // the residual: loads first, one exposed latency
#pragma unroll
              for (int j = 0; j < 16; ++j) uc[(c0 + j) * LDU] = __fadd_rn(__fadd_rn(__uint_as_float(v[j]), b2[c0 + j]), res[j]);
            });
          }
          row_sync();                                        // u' complete before anybody reads a neighbour's rows
        }
      }
      LYRA_PHASE(3, ph);
    };
    unit_body(std::integral_constant<int, 0>());
    unit_body(std::integral_constant<int, 1>());
    unit_body(std::integral_constant<int, 2>());

    // ---- last_layer.  P[row][tap * 16 + n] from the GEMM goes to shared memory (the u buffer, same [column][row] layout; a
    //      thread only touches its own row), then output row q (0..22) sums its four taps: out[q][n] = sum_tap P[q + tap - 3][tap][n]
    wait_d();
    LYRA_PHASE(3, ph);
    if (has_row) {
      float* uc = u + row;
      DuForEachAccGroup(trow + L::kColD, [&](int c0, const uint32_t (&v)[16]) {
#pragma unroll
        for (int j = 0; j < 16; ++j) uc[(c0 + j) * LDU] = __uint_as_float(v[j]);
      });
#if LYRA_DU_EARLY_DEALLOC
      lyra_tc_fence_before_sync();                           // that was the tile's last tensor-memory access: let the MMA warp free it
      __syncwarp();
      if (lane == 0) lyra_mbar_arrive(&sh->tmem_done);
#endif
    }
    lyra_mbar_wait(&sh->in_full, 0);                         // the carried last_layer tail (loaded at kernel start)
    row_sync();
    int16_t* stage = reinterpret_cast<int16_t*>(smem + L::kStage);      // [S][320]
    if (tid < 23 * S) {
      const int q = tid / S;
      const float bias = BlobPtr<float>(blob, P.last.bias)[0];
#pragma unroll
      for (int n = 0; n < 16; ++n) {
        float acc = 0.0f;
#pragma unroll
        for (int tap = 0; tap < 4; ++tap) {
          const int tr = q + tap - 3;
          if (tr >= 0 && tr < 20) acc = __fadd_rn(acc, u[(tap * 16 + n) * LDU + tr * S + s]);
        }
        const int tt = 16 * q + n;
        const float y = __fadd_rn(__fadd_rn(acc, bias), tt < 48 ? sl[tt * S + s] : 0.0f);
        if (tt < 320) {
          // UnitToInt16Scalar (dsp_utils.h:53-60,79-88): scale, clip in float, truncate
          float x = __fmul_rn(y, 32768.0f);
          x = x > -32768.0f ? x : -32768.0f;
          x = x < 32767.0f ? x : 32767.0f;
          stage[s * 320 + tt] = (int16_t)(int)x;
        } else {
          slo[(tt - 320) * S + s] = active[s] ? __fsub_rn(y, bias) : sl[(tt - 320) * S + s];
        }
      }
    }
    lyra_fence_proxy_async();
    row_sync();
    if (tid == 0) { lyra_bulk_s2g(st + (size_t)DecStateD::kLast * S, slo, 48u * S * 4); lyra_bulk_commit(); }
    for (int i = tid; i < S * 320 / 2; i += L::kRowThreads) {         // two samples per store
      const int ss = (2 * i) / 320;
      if (active[ss]) *reinterpret_cast<uint32_t*>(pcm + (size_t)slot[ss] * 320 + (2 * i) % 320) = reinterpret_cast<const uint32_t*>(stage)[i];
    }
    if (tid < S && active[tid]) n18g[tile * S + tid] = (n18[tid] + 1) % 18;
    if (tid == 0) lyra_bulk_wait_all();                      // every state block is in global memory before the block exits
    LYRA_PHASE(3, ph);
  }

  lyra_tc_fence_before_sync();
  __syncthreads();
  if (pair) lyra_cluster_sync();                              // no CTA leaves while its partner may still signal its barriers
#if !LYRA_DU_EARLY_DEALLOC
  if (!idle && warp == L::kMmaWarp) lyra_tmem_dealloc(sh->tmem_base, L::kTmemCols);
#endif
}

}  // namespace lyra_b200
