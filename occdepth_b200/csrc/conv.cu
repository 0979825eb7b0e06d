// Generalised N-d convolution as implicit GEMM.
//   TC path  : TMA (5-D tiled tensor maps, zero-filled halos, traversal strides) -> swizzled smem ->
//              tcgen05.mma (M=128 positions x N<=256 channels, fp32 accumulators in TMEM) ->
//              tcgen05.ld epilogue (bias + residuals + activation, channels-last / fp32 planar stores)
//   SIMT path: CUDA-core direct convolution with identical semantics (cross-check and odd shapes)
// Two operand types share every kernel (template parameter T, see Elem<T> / tc::Mma<T>):
//   float (TF32 values, tcgen05 kind::tf32, K chunk = 32 / 16 / 8 channels)  -- reference-precision mode
//   __nv_bfloat16 (tcgen05 kind::f16, K chunk = 64 / 32 / 16 channels)       -- throughput mode
// A K chunk is always one swizzled smem row of RB = 128 / 64 / 32 bytes; one tcgen05.mma consumes 32 bytes of it.
// See include/occdepth_b200.h for the reference call sequences this replaces.
#include "conv_common.cuh"
#include "conv_tc.cuh"
#include <new>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

namespace {

constexpr int kTcThreads = 576;  // warp 0: TMA producer, warp 1: MMA issuer (+TMEM alloc), warps 2-17: four epilogue groups
constexpr int kMaxStages = 24;   // smem ring stages of the per-tap kernel
constexpr int kHaloMaxStages = 4;

// mbarriers of a persistent tcgen05 conv CTA, placed after its operand buffers: full[max_stages], empty[max_stages],
// two TMEM accumulator pairs tfull[2] / tempty[2], the resident-weight barrier w (halo kernels), and the 4-byte slot
// tcgen05.alloc writes the TMEM base address to
struct CtaBarriers {
  uint32_t full, empty, tfull, tempty, w, slot;
};

__device__ __forceinline__ CtaBarriers cta_barriers(uint32_t base, int max_stages) {
  CtaBarriers b;
  b.full = base;
  b.empty = base + 8u * max_stages;
  b.tfull = base + 16u * max_stages;
  b.tempty = b.tfull + 16u;
  b.w = b.tempty + 16u;
  b.slot = b.w + 8u;
  return b;
}

// Prologue of the three persistent kernels: tensor-map prefetch and barrier init (thread 0), TMEM alloc (warp 1),
// then the wait for the previous grid (programmatic dependent launch, common.cuh; without it griddepcontrol.wait
// returns at once).  Everything before the wait overlaps the tail of the previous grid, whose results are only
// touched after it.  Returns the TMEM base address.
__device__ __forceinline__ uint32_t cta_prologue(const CtaBarriers& bar, int stages, bool w_bar, int tmem_cols,
                                                 const CUtensorMap* tmA, const CUtensorMap* tmW) {
  if (threadIdx.x == 0) {
    tc::prefetch_tmap(tmA);
    tc::prefetch_tmap(tmW);
    for (int s = 0; s < stages; ++s) {
      tc::mbar_init(bar.full + 8u * s, 1);
      tc::mbar_init(bar.empty + 8u * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      tc::mbar_init(bar.tfull + 8u * a, 1);
      tc::mbar_init(bar.tempty + 8u * a, 256);  // every epilogue thread of the two groups arrives
    }
    if (w_bar) tc::mbar_init(bar.w, 1);
    tc::fence_barrier_init();
  }
  if ((threadIdx.x >> 5) == 1) {
    __syncwarp();
    tc::tmem_alloc(bar.slot, (uint32_t)tmem_cols);
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(bar.slot));
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  return tmem_base;
}

__device__ __forceinline__ void cta_teardown(uint32_t tmem_base, int tmem_cols) {
  tc::fence_before_sync();
  __syncthreads();
  if ((threadIdx.x >> 5) == 1) {
    __syncwarp();
    tc::tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
  }
}

// Debug timeline (occd_conv_debug_trace, tools/conv_trace.py): clock64 stamp k of pipeline step j of CTA 0 into
// trace[64][8].  k = 0 / 1: TMA producer, 2 / 3: MMA issuer, 4 / 5 / 6: epilogue wait / go / done (thread 64 only)
__device__ __forceinline__ void trace_stamp(long long* trace, uint32_t j, int k) {
  if (trace && blockIdx.x == 0 && j < 64u && (k < 4 || threadIdx.x == 64)) trace[j * 8 + k] = clock64();
}

// Fast epilogue (conv_common.cuh) of this thread's accumulator row: TMEM columns [c_begin, c_end) from taddr, each
// chunk's bias / residual loads in flight together with its TMEM load
template <typename T>
__device__ __forceinline__ void epi_drain_fast(const EpiRow<T>& er, uint32_t taddr, int c_begin, int c_end) {
  uint32_t ra[16];
  EpiPre q;
  for (int c0 = c_begin; c0 < c_end; c0 += 16) {
    tc::tmem_ld16_issue(taddr + (uint32_t)c0, ra);
    epi_prefetch<T>(er, c0, q);
    tc::tmem_ld_wait16(ra);
    epi_finish<T>(er, c0, ra, q);
  }
}

struct TcParams {
  ConvEpi epi;
  int n_taps;
  int n_kchunks[OCCD_CONV_MAX_SRC];
  int tiles_w, tiles_h, tiles_d, num_m_tiles;
  int src_d0;
  int w_batch_rows;  // weight rows per image (0: shared weights)
  int TD, TH, TW;
  int TWv;           // output columns per tile row: TW, or 30 for the x-packed variant (one halo column each side)
  int stride[3];
  int Cout_pad, N_tile;
  int stages, group;
  int a_bytes, b_stride, b_bytes;
  int tmem_cols;
  long long* trace;  // optional [tile][8] clock64 stamps of CTA 0 (occd_conv_debug_trace, tools/conv_trace.py)
  signed char tap_src[OCCD_CONV_MAX_TAPS];
  short tap_dz[OCCD_CONV_MAX_TAPS], tap_dy[OCCD_CONV_MAX_TAPS], tap_dx[OCCD_CONV_MAX_TAPS];
  // tap groups: n_groups convolutions over the same sources and iteration space in one launch (the sub-pixel phases
  // of a stride-2 transposed conv).  Tiles are ordered group-major, so every CTA of the persistent grid takes the
  // same share of each group (the groups differ in tap count).  n_groups == 1: the whole tap list, epi.oadd.
  int n_groups;
  short grp_tap0[OCCD_CONV_MAX_GROUPS + 1];
  short grp_iters[OCCD_CONV_MAX_GROUPS];
  signed char grp_oadd[OCCD_CONV_MAX_GROUPS][3];
};

// XP: x-packed variant: the pipeline items are (source, dz, dy) groups whose B operand stacks the three W taps
// (N_tile = 3 * Cout_pad: with taps in lexicographic order that is 3 consecutive tap slices of the ordinary weight
// tensor), tiles are 32 wide with one halo column on each side so that one smem row == one TMEM lane == one lane of
// an epilogue warp, and the epilogue forms out[r] = Q_0[r-1] + Q_1[r] + Q_2[r+1] from the three column groups with
// two warp shuffles per channel.  One A fetch then feeds 3x the output columns (measured on B200, round 2: the
// Cout = 80 decoder convs 0.154 -> 0.102 ms).
template <typename T, int RB, bool XP>
__global__ void __launch_bounds__(kTcThreads)
conv_tc_kernel(const __grid_constant__ TcParams p, const __grid_constant__ CUtensorMap tmA0,
               const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
               const __grid_constant__ CUtensorMap tmW) {
  // Persistent, warp-specialised implicit GEMM.  Each CTA walks tiles blockIdx.x, +gridDim.x, ...:
  //   warp 0 (one lane): TMA producer -- runs ahead across tile boundaries, the smem ring never drains
  //   warp 1 (one lane): tcgen05.mma issuer, accumulating into one of TWO TMEM accumulators
  //   warps 2-17       : four epilogue groups of 4 warps: group g drains accumulator (g & 1) -- even / odd
  //                      tiles -- and column half (g >> 1) of it: TMEM -> regs -> global while the MMAs of the
  //                      following tiles run (the epilogue is latency bound: 16 warps keep the SM's LSU busy)
  constexpr int KCH = RB / (int)sizeof(T);  // channels per K chunk
  constexpr int NMMA = RB / 32;             // tcgen05.mma instructions per chunk (32 bytes of K each)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // dynamic smem is only guaranteed 16-byte aligned: round the base up to 1024 (swizzle atom alignment)
  const uint32_t smem_base = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base;
  const uint32_t smem_b = smem_a + (uint32_t)(p.stages * p.group) * p.a_bytes;
  // barriers: 8-byte aligned (the buffers before them are multiples of 1024 bytes)
  const CtaBarriers bar = cta_barriers(smem_b + (uint32_t)(p.stages * p.group) * p.b_stride, kMaxStages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tiles_n = XP ? 1 : p.Cout_pad / p.N_tile;
  const int tiles_per_group = p.num_m_tiles * n_tiles_n;
  const int num_tiles = tiles_per_group * p.n_groups;

  const uint32_t tmem_base = cta_prologue(bar, p.stages, false, p.tmem_cols, &tmA0, &tmW);
  const uint32_t acc_stride = (uint32_t)p.tmem_cols >> 1;  // column offset of the second accumulator

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer =====
      const CUtensorMap* maps[3] = {&tmA0, &tmA1, &tmA2};
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int grp = tile / tiles_per_group;
        const int tg = tile - grp * tiles_per_group;
        const int nt = tg % n_tiles_n;
        int t = tg / n_tiles_n;
        const int tw = t % p.tiles_w; t /= p.tiles_w;
        const int th = t % p.tiles_h; t /= p.tiles_h;
        const int td = t % p.tiles_d; t /= p.tiles_d;
        const int b = t;
        const int iw0 = XP ? tw * 30 - 1 : tw * p.TW * p.stride[2], ih0 = th * p.TH * p.stride[1],
                  id0 = td * p.TD * p.stride[0] + p.src_d0;
        const int n0 = nt * p.N_tile;
        // items (tap, k-chunk) are loaded in groups of p.group per pipeline stage: one barrier hand-off per group
        int g = 0;
        int remaining = p.grp_iters[grp];
        const int jt = (tile - blockIdx.x) / gridDim.x;
        trace_stamp(p.trace, jt, 0);
        for (int tp = p.grp_tap0[grp]; tp < p.grp_tap0[grp + 1]; ++tp) {
          const int src = p.tap_src[tp];
          const int cw = iw0 + p.tap_dx[tp], ch = ih0 + p.tap_dy[tp], cd = id0 + p.tap_dz[tp];
          const int wrow = b * p.w_batch_rows + (XP ? tp * p.N_tile : tp * p.Cout_pad + n0);
          const int nk = p.n_kchunks[src];
          for (int kc = 0; kc < nk; ++kc) {
            if (g == 0) {
              const int cnt = remaining < p.group ? remaining : p.group;
              tc::mbar_wait(bar.empty + 8u * s, ph ^ 1u);
              tc::mbar_expect_tx(bar.full + 8u * s, (uint32_t)(cnt * (p.a_bytes + p.b_bytes)));
            }
            const uint32_t sa = smem_a + (uint32_t)(s * p.group + g) * p.a_bytes;
            const uint32_t sb = smem_b + (uint32_t)(s * p.group + g) * p.b_stride;
            tc::tma_load_5d(sa, maps[src], bar.full + 8u * s, kc * KCH, cw, ch, cd, b);
            tc::tma_load_2d(sb, &tmW, bar.full + 8u * s, kc * KCH, wrow);
            --remaining;
            if (++g == p.group || remaining == 0) {
              g = 0;
              if (++s == p.stages) { s = 0; ph ^= 1u; }
            }
          }
        }
        trace_stamp(p.trace, jt, 1);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc = tc::Mma<T>::idesc(128, p.N_tile);
      const uint64_t da0 = tc::make_sdesc(smem_a, RB);
      const uint64_t db0 = tc::make_sdesc(smem_b, RB);
      int s = 0;
      uint32_t ph = 0;
      int j = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++j) {
        const uint32_t acc = (uint32_t)j & 1u;
        tc::mbar_wait(bar.tempty + 8u * acc, (((uint32_t)j >> 1) & 1u) ^ 1u);  // epilogue drained this buffer
        tc::fence_after_sync();
        trace_stamp(p.trace, j, 2);
        const uint32_t d_tmem = tmem_base + acc * acc_stride;
        const int iters_per_tile = p.grp_iters[tile / tiles_per_group];
        for (int it = 0; it < iters_per_tile;) {
          tc::mbar_wait(bar.full + 8u * s, ph);
          tc::fence_after_sync();
          const int cnt = (iters_per_tile - it) < p.group ? (iters_per_tile - it) : p.group;
          for (int g = 0; g < cnt; ++g, ++it) {
            const uint64_t da = da0 + (uint64_t)((s * p.group + g) * (p.a_bytes >> 4));
            const uint64_t db = db0 + (uint64_t)((s * p.group + g) * (p.b_stride >> 4));
            tc::mma_kchunk<T, NMMA>(d_tmem, da, db, idesc, it == 0);
          }
          tc::mma_commit(bar.empty + 8u * s);  // frees the smem stage when these MMAs retire
          if (++s == p.stages) { s = 0; ph ^= 1u; }
        }
        tc::mma_commit(bar.tfull + 8u * acc);  // accumulator complete
        trace_stamp(p.trace, j, 3);
      }
    }
  } else {
    // ===== epilogue: TMEM -> registers -> (bias, residuals, activation) -> global =====
    // (a shared-memory-staged TMA-store epilogue was measured on B200, round 2: same 4-5 B/cycle/SM as these direct
    // stores -- the write path, not the store instruction mix, is the limit -- and the 64 KB of staging cost the
    // large-K convs a third of their smem ring: 4.0 -> 5.4 ms for the decoder 3x3 convs.  Removed.)
    const int q = warp & 3;                  // TMEM lane quarter this warp may access
    const int egrp = (warp - 2) >> 2;        // epilogue group 0..3 (128 threads == 128 tile rows)
    const int grp = egrp & 1;                // accumulator index (tile parity)
    const int half = egrp >> 1;              // this group takes the first / second half of the 16-column chunks
    const int ncols = XP ? p.Cout_pad : p.N_tile;        // output channels of one tile
    const int n_chunks = ncols >> 4;
    const int c_begin = half == 0 ? 0 : ((n_chunks + 1) >> 1) * 16;   // contiguous per thread: whole lines fill up
    const int c_end = half == 0 ? ((n_chunks + 1) >> 1) * 16 : ncols;
    const int row = q * 32 + lane;
    const int rw = row % p.TW;
    const int rh = (row / p.TW) % p.TH;
    const int rd = row / (p.TW * p.TH);
    int j = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++j) {
      if ((j & 1) != grp) continue;
      const int tgrp = tile / tiles_per_group;       // tap group (sub-pixel phase) of this tile
      const int tg = tile - tgrp * tiles_per_group;
      const int nt = tg % n_tiles_n;
      int t = tg / n_tiles_n;
      const int tw = t % p.tiles_w; t /= p.tiles_w;
      const int th = t % p.tiles_h; t /= p.tiles_h;
      const int td = t % p.tiles_d; t /= p.tiles_d;
      const int b = t;
      const int od = td * p.TD + rd, oh = th * p.TH + rh, ow = XP ? tw * 30 + rw - 1 : tw * p.TW + rw;
      const bool valid = od < p.epi.OD && oh < p.epi.OH && ow < p.epi.OW && (!XP || (rw >= 1 && rw <= 30));
      const int n0 = nt * p.N_tile;
      const uint32_t acc = (uint32_t)grp;
      trace_stamp(p.trace, j, 4);
      tc::mbar_wait(bar.tfull + 8u * acc, ((uint32_t)j >> 1) & 1u);
      tc::fence_after_sync();
      trace_stamp(p.trace, j, 5);
      const uint32_t taddr = tmem_base + acc * acc_stride + ((uint32_t)(q * 32) << 16);
      if constexpr (XP) {
        // TW == 32: lane == tile column, so the W neighbours' partial sums sit in the neighbouring lanes
        for (int c0 = c_begin; c0 < c_end; c0 += 16) {
          float lo[16], v[16], hi[16];
          tc::tmem_ld16(taddr + (uint32_t)c0, lo);
          tc::tmem_ld16(taddr + (uint32_t)(p.Cout_pad + c0), v);
          tc::tmem_ld16(taddr + (uint32_t)(2 * p.Cout_pad + c0), hi);
#pragma unroll
          for (int i = 0; i < 16; ++i)
            v[i] += __shfl_up_sync(0xffffffffu, lo[i], 1) + __shfl_down_sync(0xffffffffu, hi[i], 1);
          if (valid) conv_epilogue_row<T, 16>(p.epi, b, od, oh, ow, c0, v);
        }
      } else if (epi_fast_ok(p.epi)) {
        // fast path: pointers formed once per tile
        const EpiRow<T> er = p.n_groups > 1 ? epi_row<T>(p.epi, valid, b, od, oh, ow, n0, p.grp_oadd[tgrp][0],
                                                         p.grp_oadd[tgrp][1], p.grp_oadd[tgrp][2])
                                            : epi_row<T>(p.epi, valid, b, od, oh, ow, n0);
        epi_drain_fast<T>(er, taddr, c_begin, c_end);
      } else {
        // software-pipelined: the tcgen05.ld of this group's next 16 columns is in flight while these are stored
        uint32_t ra[16], rb[16];
        int c0 = c_begin;
        if (c0 < c_end) tc::tmem_ld16_issue(taddr + (uint32_t)c0, ra);
        for (; c0 < c_end; c0 += 32) {
          tc::tmem_ld_wait16(ra);
          const bool has_b = c0 + 16 < c_end;
          if (has_b) tc::tmem_ld16_issue(taddr + (uint32_t)(c0 + 16), rb);
          if (valid) {
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(ra[i]);
            conv_epilogue_row<T, 16>(p.epi, b, od, oh, ow, n0 + c0, v);
          }
          if (has_b) {
            tc::tmem_ld_wait16(rb);
            if (c0 + 32 < c_end) tc::tmem_ld16_issue(taddr + (uint32_t)(c0 + 32), ra);
            if (valid) {
              float v[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(rb[i]);
              conv_epilogue_row<T, 16>(p.epi, b, od, oh, ow, n0 + c0 + 16, v);
            }
          }
        }
      }
      tc::fence_before_sync();
      tc::mbar_arrive(bar.tempty + 8u * acc);  // this thread's TMEM reads of the buffer are done
      trace_stamp(p.trace, j, 6);
    }
  }
  cta_teardown(tmem_base, p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// Halo-tile variant for stride-1 3x3x3 convolutions with few channels (the full-resolution head):
// the per-tap TMA boxes of conv_tc_kernel re-load every input row 27 times and the TMA unit (~1.5 cycles per
// box row) becomes the limiter.  Here each CTA tile loads ONE zero-filled halo box (PD x PH x PW positions,
// rows of one K chunk) and feeds all 27 taps from row-shifted views of that box: with smem rows
// linearised as r = (pd*PH + ph)*PW + pw, the A operand of tap (a,b,c) for output rows [R, R+128) is simply
// rows [R + (a*PH + b)*PW + c, ...) -- a different UMMA start address, same data.  Rows that fall in the
// halo produce garbage accumulator rows that the epilogue never stores.  Dilation d runs the same scheme on
// the d^3 sub-sampled grids (TMA traversal stride d), so the halo is always one position.  Weights for all
// taps stay resident in shared memory.  The swizzled row-shifted UMMA start addresses use base-offset 0 (measured on
// B200: the XOR swizzle follows absolute smem address bits for both TMA and UMMA).
struct HaloParams {
  ConvEpi epi;
  int d;                      // dilation (== padding)
  int D, H, W;                // full grid (== output grid)
  int BD, BH, BW, PD, PH, PW;  // valid box / halo box (sub-sampled coordinates)
  int src_d0;                 // plane offset of the interior inside a halo-margin source buffer
  int hd, hh, hw;             // 1 where the taps reach into that dimension (halo of one sub-sampled position)
  int tilesD, tilesH, tilesW;
  int nM, R0;                 // M tiles per CTA tile, first valid row
  int box_bytes;              // bytes one TMA box delivers
  int a_stage_bytes;          // allocated per stage (box + slack rows read by garbage outputs)
  int stages;
  int n_taps;
  int N_tile, tmem_cols, set_stride;
  int b_stride, w_bytes;
  int tap_off16[27];          // (R0 + (a*PH + b)*PW + c) * row_bytes / 16: A-descriptor advance per tap
  long long* trace;
};

template <typename T, int RB>
__global__ void __launch_bounds__(kTcThreads)
conv_halo_kernel(const __grid_constant__ HaloParams p, const __grid_constant__ CUtensorMap tmA,
                 const __grid_constant__ CUtensorMap tmW) {
  constexpr int NMMA = RB / 32;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_w = smem_base;                                   // [n_taps][b_stride] resident weights
  const uint32_t smem_a = smem_w + (uint32_t)p.w_bytes;                 // [stages][a_stage_bytes]
  const CtaBarriers bar = cta_barriers(smem_a + (uint32_t)p.stages * p.a_stage_bytes, kHaloMaxStages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int d = p.d;
  const int per_res = p.tilesD * p.tilesH * p.tilesW;
  const int num_tiles = p.epi.B * d * d * d * per_res;

  const uint32_t tmem_base = cta_prologue(bar, p.stages, true, p.tmem_cols, &tmA, &tmW);

  // tile -> (batch, residue class, sub-grid tile origin)
  auto decode = [&](int tile, int& b, int& ra, int& rb, int& rc, int& td, int& th, int& tw) {
    int t = tile;
    tw = t % p.tilesW; t /= p.tilesW;
    th = t % p.tilesH; t /= p.tilesH;
    td = t % p.tilesD; t /= p.tilesD;
    rc = t % d; t /= d;
    rb = t % d; t /= d;
    ra = t % d; t /= d;
    b = t;
  };

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer: resident weights once, then one halo box per tile =====
      tc::mbar_expect_tx(bar.w, (uint32_t)(p.n_taps * p.N_tile * RB));
      for (int tp = 0; tp < p.n_taps; ++tp)
        tc::tma_load_2d(smem_w + (uint32_t)tp * p.b_stride, &tmW, bar.w, 0, tp * p.N_tile);
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int b, ra, rb, rc, td, th, tw;
        decode(tile, b, ra, rb, rc, td, th, tw);
        tc::mbar_wait(bar.empty + 8u * s, ph ^ 1u);
        tc::mbar_expect_tx(bar.full + 8u * s, (uint32_t)p.box_bytes);
        tc::tma_load_5d(smem_a + (uint32_t)s * p.a_stage_bytes, &tmA, bar.full + 8u * s, 0,
                        (tw * p.BW - p.hw) * d + rc, (th * p.BH - p.hh) * d + rb,
                        (td * p.BD - p.hd) * d + ra + p.src_d0, b);
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc = tc::Mma<T>::idesc(128, p.N_tile);
      const uint64_t db_w = tc::make_sdesc(smem_w, RB);
      const int w_step16 = p.b_stride / 16;
      tc::mbar_wait(bar.w, 0);
      int s = 0;
      uint32_t ph = 0;
      int j = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++j) {
        const uint32_t set = (uint32_t)j & 1u;
        const uint32_t use = (uint32_t)j >> 1;
        tc::mbar_wait(bar.tempty + 8u * set, (use & 1u) ^ 1u);
        tc::mbar_wait(bar.full + 8u * s, ph);
        tc::fence_after_sync();
        trace_stamp(p.trace, j, 2);
        // descriptors advance by plain 64-bit adds on the 16-byte-unit address field (smem < 256 KB: no carry out
        // of the 14-bit field), so the issue loop is ~4 instructions per tcgen05.mma
        const uint64_t da_stage = tc::make_sdesc(smem_a + (uint32_t)s * p.a_stage_bytes, RB);
        for (int m = 0; m < p.nM; ++m) {
          const uint32_t d_tmem = tmem_base + set * (uint32_t)p.set_stride + (uint32_t)(m * p.N_tile);
          const uint64_t da_m = da_stage + (uint64_t)(m * (128 * RB / 16));
          tc::mma_kchunk<T, NMMA>(d_tmem, da_m + (uint64_t)p.tap_off16[0], db_w, idesc, true);
#pragma unroll 3
          for (int tp = 1; tp < p.n_taps; ++tp)
            tc::mma_kchunk<T, NMMA>(d_tmem, da_m + (uint64_t)p.tap_off16[tp], db_w + (uint64_t)(tp * w_step16), idesc,
                                    false);
        }
        tc::mma_commit(bar.empty + 8u * s);
        tc::mma_commit(bar.tfull + 8u * set);
        trace_stamp(p.trace, j, 3);
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ===== epilogue =====
    const int q = warp & 3;
    const int grp = ((warp - 2) >> 2) & 1;   // accumulator set (tile parity)
    const int half = (warp - 2) >> 3;        // even / odd M tiles of the set
    int j = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++j) {
      const uint32_t set = (uint32_t)j & 1u;   // accumulator set == epilogue group
      const uint32_t use = (uint32_t)j >> 1;
      if ((int)set != grp) continue;
      int b, ra, rb, rc, td, th, tw;
      decode(tile, b, ra, rb, rc, td, th, tw);
      trace_stamp(p.trace, j, 4);
      tc::mbar_wait(bar.tfull + 8u * set, use & 1u);
      tc::fence_after_sync();
      trace_stamp(p.trace, j, 5);
      for (int m = half; m < p.nM; m += 2) {   // one epilogue group per M tile parity
        const int R = p.R0 + m * 128 + q * 32 + lane;
        const int pw = R % p.PW;
        const int phh = (R / p.PW) % p.PH;
        const int pd = R / (p.PW * p.PH);
        const int od = (td * p.BD + pd - p.hd) * d + ra, oh = (th * p.BH + phh - p.hh) * d + rb,
                  ow = (tw * p.BW + pw - p.hw) * d + rc;
        const bool valid = pd >= p.hd && pd < p.hd + p.BD && phh >= p.hh && phh < p.hh + p.BH && pw >= p.hw &&
                           pw < p.hw + p.BW && od < p.D && oh < p.H && ow < p.W;
        const uint32_t taddr = tmem_base + set * (uint32_t)p.set_stride + (uint32_t)(m * p.N_tile) +
                               ((uint32_t)(q * 32) << 16);
        if (epi_fast_ok(p.epi)) {
          epi_drain_fast<T>(epi_row<T>(p.epi, valid, b, od, oh, ow, 0), taddr, 0, p.N_tile);
        } else {
          for (int c0 = 0; c0 < p.N_tile; c0 += 16) {
            float v[16];
            tc::tmem_ld16(taddr + (uint32_t)c0, v);
            if (valid) conv_epilogue_row<T, 16>(p.epi, b, od, oh, ow, c0, v);
          }
        }
      }
      tc::fence_before_sync();
      tc::mbar_arrive(bar.tempty + 8u * set);
      trace_stamp(p.trace, j, 6);
    }
  }
  cta_teardown(tmem_base, p.tmem_cols);
}


// ------------------------------------------------------------------------------------------------
// x-packed halo kernel for grids whose innermost extent W is one warp wide or narrower (W in {8, 16, 32}: every
// 3-D activation of this network -- Z = 32 / 16 / 8).  Measured on B200 (tools/micro/mma_issue_bench.cu,
// profiles/r02_mma_issue_bench.txt): one tcgen05.mma costs max(59, N/2) cycles for M = 128 whatever the operand
// type, so a 32-output-channel conv issued tap by tap runs the tensor pipe at N/2 / 59 = 27 % (bf16) and, with
// K = 8 per instruction, 14 % (TF32).  Here the three W taps (dx = -d, 0, +d) of each (dz, dy) pair share ONE
// instruction: its B operand stacks the three taps' weights along N (N = 3 * Cout_pad: three consecutive tap slices
// of the ordinary weight tensor), its A operand is the un-shifted rows, and the accumulator holds
//     Q_c[r] = sum_{a,b} W[a][b][c] . in[r + (a*PH + b)*PW]      c = 0, 1, 2
// from which the epilogue forms out[r] = Q_0[r - d] + Q_1[r] + Q_2[r + d].  Smem rows are linearised with W
// fastest and PW == W divides 32, so r +- d stays inside the warp: two shuffles per channel, masked where the
// neighbour would fall outside [0, W) -- which is exactly the convolution's zero padding, so the W axis needs no
// halo columns and no sub-sampling.  D and H keep the halo-tile scheme (one zero-filled halo position per side on
// the d-sub-sampled grids, TMA traversal stride d).  27 taps become 9 instructions per 32 bytes of K.
// out[r] = Q0[r - d] + Q1[r] + Q2[r + d] for 16 channels of this lane's row: the three accumulator column groups of
// the x-packed MMA (lane == W position; lanes shifted out of [0, W) contribute the conv's zero padding).  The three
// tcgen05.ld are issued back to back and share ONE wait.
__device__ __forceinline__ void halox_gather16(uint32_t taddr, int c0, int CP, int d, bool lo_ok, bool hi_ok, float* v) {
  uint32_t lo[16], mid[16], hi[16];
  tc::tmem_ld16_issue(taddr + (uint32_t)c0, lo);
  tc::tmem_ld16_issue(taddr + (uint32_t)(CP + c0), mid);
  tc::tmem_ld16_issue(taddr + (uint32_t)(2 * CP + c0), hi);
  tc::tmem_ld_wait16(lo);
  tc::tmem_ld_dep16(mid);
  tc::tmem_ld_dep16(hi);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float l = __shfl_up_sync(0xffffffffu, __uint_as_float(lo[i]), (unsigned)d);
    const float h = __shfl_down_sync(0xffffffffu, __uint_as_float(hi[i]), (unsigned)d);
    v[i] = __uint_as_float(mid[i]) + (lo_ok ? l : 0.f) + (hi_ok ? h : 0.f);
  }
}

struct HaloxParams {
  ConvEpi epi;
  int d;                      // dilation (== padding) of the taps
  int D, H;                   // output grid (W == PW)
  int BD, BH, PD, PH, PW;     // valid box / halo box in sub-sampled (D, H) coordinates; PW == W
  int hd, hh;                 // 1 where the taps reach into D / H
  int src_d0;
  int tilesD, tilesH;
  int nM;                     // M tiles (128 smem rows = 128 / PW h-rows of one plane) per CTA tile, <= 2
  int mt_row[2], mt_pd[2], mt_ph0[2];
  int box_bytes, a_stage_bytes, stages;
  int n_groups;               // (dz, dy) groups = n_taps / 3
  int CP, N_tile;             // padded output channels, N_tile = 3 * CP
  int tmem_cols, set_stride;
  int b_stride, w_bytes;
  int grp_off[9];             // (a*PH + b)*PW: smem row offset of a group's A operand relative to the M tile
  long long* trace;
  // plane-ring mode (ring == 1; chosen when the halo box leaves room for ONE stage only, i.e. the TF32 head whose
  // resident weights take 110 KB): the output planes of all columns (image, residue class, H tile) form one sequence
  // of n_cols * sD M tiles; every CTA takes a contiguous, equal share of it (at most one column change inside).  The
  // four stages are a ring of single input planes, output plane z reads ring planes z-1, z, z+1, so every M tile costs
  // ONE new 6-row plane (prefetched a plane ahead) instead of half a 4-plane box loaded while the tensor pipe waits
  int ring, sD, n_cols;
  signed char grp_dz[9];      // -1 / 0 / +1: which ring plane a group reads
  short grp_row[9];           // (hh + dy) * PW: its row offset inside the plane
};

template <typename T, int RB>
__global__ void __launch_bounds__(kTcThreads)
conv_halox_kernel(const __grid_constant__ HaloxParams p, const __grid_constant__ CUtensorMap tmA,
                  const __grid_constant__ CUtensorMap tmW) {
  constexpr int NMMA = RB / 32;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_w = smem_base;                                   // [n_groups][b_stride] resident weights
  const uint32_t smem_a = smem_w + (uint32_t)p.w_bytes;                 // [stages][a_stage_bytes]
  const uint32_t bar_base = smem_a + (uint32_t)p.stages * p.a_stage_bytes;
  const CtaBarriers bar = cta_barriers(bar_base, kHaloMaxStages);      // ring mode: descriptor table at bar_base + 128

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int d = p.d;
  const int num_tiles = p.epi.B * d * d * p.tilesD * p.tilesH;
  // ring mode: this CTA's share [ring_lo, ring_hi) of the n_cols * sD output planes
  const long long ring_total = (long long)p.n_cols * p.sD;
  const long long ring_lo = p.ring ? ring_total * blockIdx.x / gridDim.x : 0;
  const long long ring_hi = p.ring ? ring_total * (blockIdx.x + 1) / gridDim.x : 0;

  const uint32_t tmem_base = cta_prologue(bar, p.stages, true, p.tmem_cols, &tmA, &tmW);

  // tile -> (batch, (D, H) residue class, sub-grid tile origin)
  auto decode = [&](int tile, int& b, int& ra, int& rb, int& td, int& th) {
    int t = tile;
    th = t % p.tilesH; t /= p.tilesH;
    td = t % p.tilesD; t /= p.tilesD;
    rb = t % d; t /= d;
    ra = t % d; t /= d;
    b = t;
  };

  // ring mode: position in the plane sequence -> (batch, residue class, H tile) and the run of planes [z0, z1) this CTA
  // takes from that column
  auto decode_ring = [&](long long pos, int& b, int& ra, int& rb, int& th, int& z0, int& z1) {
    int t = (int)(pos / p.sD);
    z0 = (int)(pos - (long long)t * p.sD);
    const long long left = ring_hi - pos;
    z1 = (long long)(p.sD - z0) < left ? p.sD : z0 + (int)left;
    th = t % p.tilesH; t /= p.tilesH;
    rb = t % d; t /= d;
    ra = t % d; t /= d;
    b = t;
  };

  if (warp == 0) {
    if (lane == 0 && p.ring) {
      // ===== TMA producer, ring mode: weights once, then planes z0-1 .. z1 of every unit, one ring slot each =====
      tc::mbar_expect_tx(bar.w, (uint32_t)(p.n_groups * p.N_tile * RB));
      for (int g = 0; g < p.n_groups; ++g)
        tc::tma_load_2d(smem_w + (uint32_t)g * p.b_stride, &tmW, bar.w, 0, g * p.N_tile);
      uint32_t n = 0;
      for (long long pos = ring_lo; pos < ring_hi;) {
        int b, ra, rb, th, z0, z1;
        decode_ring(pos, b, ra, rb, th, z0, z1);
        pos += z1 - z0;
        for (int z = z0 - 1; z <= z1; ++z, ++n) {
          const uint32_t slot = n & 3u;
          trace_stamp(p.trace, n, 0);
          tc::mbar_wait(bar.empty + 8u * slot, ((n >> 2) & 1u) ^ 1u);
          trace_stamp(p.trace, n, 1);
          tc::mbar_expect_tx(bar.full + 8u * slot, (uint32_t)p.box_bytes);
          tc::tma_load_5d(smem_a + slot * (uint32_t)p.a_stage_bytes, &tmA, bar.full + 8u * slot, 0, 0,
                          (th * p.BH - p.hh) * d + rb, z * d + ra + p.src_d0, b);
        }
      }
    } else if (lane == 0) {
      // ===== TMA producer: resident weights once, then one halo box per tile =====
      tc::mbar_expect_tx(bar.w, (uint32_t)(p.n_groups * p.N_tile * RB));
      for (int g = 0; g < p.n_groups; ++g)
        tc::tma_load_2d(smem_w + (uint32_t)g * p.b_stride, &tmW, bar.w, 0, g * p.N_tile);
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int b, ra, rb, td, th;
        decode(tile, b, ra, rb, td, th);
        tc::mbar_wait(bar.empty + 8u * s, ph ^ 1u);
        tc::mbar_expect_tx(bar.full + 8u * s, (uint32_t)p.box_bytes);
        tc::tma_load_5d(smem_a + (uint32_t)s * p.a_stage_bytes, &tmA, bar.full + 8u * s, 0, 0,
                        (th * p.BH - p.hh) * d + rb, (td * p.BD - p.hd) * d + ra + p.src_d0, b);
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && p.ring) {
      // ===== MMA issuer, ring mode =====
      const uint32_t idesc = tc::Mma<T>::idesc(128, p.N_tile);
      const uint64_t db_w = tc::make_sdesc(smem_w, RB);
      const int w_step16 = p.b_stride / 16;
      // A descriptors of the nine groups for each of the four ring rotations, built once (the issuing thread must not
      // spend its ~60 cycles per MMA on address arithmetic)
      uint64_t* dtab = reinterpret_cast<uint64_t*>(smem_raw + (bar_base - tc::smem_u32(smem_raw)) + 128u);
      for (int r = 0; r < 4; ++r)
        for (int g = 0; g < 9; ++g) {
          const uint32_t slot = (uint32_t)(r + (g < p.n_groups ? p.grp_dz[g] : 0)) & 3u;
          dtab[r * 9 + g] = tc::make_sdesc(smem_a + slot * (uint32_t)p.a_stage_bytes, RB) +
                            (uint64_t)((g < p.n_groups ? p.grp_row[g] : 0) * (RB / 16));
        }
      tc::mbar_wait(bar.w, 0);
      uint32_t n0 = 0;     // ring index of this unit's first plane (z0 - 1)
      uint32_t j = 0;      // output planes so far == accumulator uses
      for (long long pos = ring_lo; pos < ring_hi;) {
        int b, ra, rb, th, z0, z1;
        decode_ring(pos, b, ra, rb, th, z0, z1);
        pos += z1 - z0;
        const int K = z1 - z0;
        for (int k = 0; k < K; ++k, ++j) {
          const uint32_t set = j & 1u;
          tc::mbar_wait(bar.tempty + 8u * set, ((j >> 1) & 1u) ^ 1u);
          for (uint32_t i = (k == 0 ? 0u : 2u); i < 3u; ++i) {     // planes z-1 and z were waited for by plane z-1
            const uint32_t n = n0 + (uint32_t)k + i;
            tc::mbar_wait(bar.full + 8u * (n & 3u), (n >> 2) & 1u);
          }
          tc::fence_after_sync();
          trace_stamp(p.trace, j, 2);
          const uint32_t d_tmem = tmem_base + set * (uint32_t)p.set_stride;
          const uint64_t* drow = dtab + ((n0 + (uint32_t)k + 1u) & 3u) * 9u;
          uint64_t dg[9];
#pragma unroll
          for (int g = 0; g < 9; ++g) dg[g] = drow[g];
#pragma unroll
          for (int g = 0; g < 9; ++g)
            if (g < p.n_groups) tc::mma_kchunk<T, NMMA>(d_tmem, dg[g], db_w + (uint64_t)(g * w_step16), idesc, g == 0);
          tc::mma_commit(bar.tfull + 8u * set);
          trace_stamp(p.trace, j, 3);
          tc::mma_commit(bar.empty + 8u * ((n0 + (uint32_t)k) & 3u));            // plane z-1 is done with
          if (k == K - 1) {                                                       // ... and the unit's last two
            tc::mma_commit(bar.empty + 8u * ((n0 + (uint32_t)k + 1u) & 3u));
            tc::mma_commit(bar.empty + 8u * ((n0 + (uint32_t)k + 2u) & 3u));
          }
        }
        n0 += (uint32_t)K + 2u;
      }
    } else if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc = tc::Mma<T>::idesc(128, p.N_tile);
      const uint64_t db_w = tc::make_sdesc(smem_w, RB);
      const int w_step16 = p.b_stride / 16;
      tc::mbar_wait(bar.w, 0);
      int s = 0;
      uint32_t ph = 0;
      int j = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++j) {
        const uint32_t set = (uint32_t)j & 1u;
        const uint32_t use = (uint32_t)j >> 1;
        tc::mbar_wait(bar.tempty + 8u * set, (use & 1u) ^ 1u);
        tc::mbar_wait(bar.full + 8u * s, ph);
        tc::fence_after_sync();
        trace_stamp(p.trace, j, 2);
        const uint64_t da_stage = tc::make_sdesc(smem_a + (uint32_t)s * p.a_stage_bytes, RB);
        for (int m = 0; m < p.nM; ++m) {
          const uint32_t d_tmem = tmem_base + set * (uint32_t)p.set_stride + (uint32_t)(m * p.N_tile);
          tc::mma_kchunk<T, NMMA>(d_tmem, da_stage + (uint64_t)((p.mt_row[m] + p.grp_off[0]) * (RB / 16)), db_w, idesc,
                                  true);
#pragma unroll 2
          for (int g = 1; g < p.n_groups; ++g)
            tc::mma_kchunk<T, NMMA>(d_tmem, da_stage + (uint64_t)((p.mt_row[m] + p.grp_off[g]) * (RB / 16)),
                                    db_w + (uint64_t)(g * w_step16), idesc, false);
        }
        tc::mma_commit(bar.empty + 8u * s);
        tc::mma_commit(bar.tfull + 8u * set);
        trace_stamp(p.trace, j, 3);
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ===== epilogue: 16 warps; group (egrp & 1) drains accumulator set (tile parity), (egrp >> 1) picks the work
    // items (M tile, 16-channel chunk) it takes =====
    const int q = warp & 3;
    const int egrp = (warp - 2) >> 2;
    const int grp = egrp & 1;
    const int half = egrp >> 1;
    const int rr = q * 32 + lane;            // row inside an M tile
    const int hr = rr / p.PW;                // h-row inside the M tile
    const int pw = rr - hr * p.PW;           // == output w
    const bool lo_ok = pw >= d, hi_ok = pw + d < p.PW;
    const int chunks = p.CP >> 4;
    const int n_items = p.nM * chunks;
    if (p.ring) {
      // ring mode: one M tile (one plane, 128 / PW h-rows) per accumulator use
      uint32_t jr = 0;
      for (long long pos = ring_lo; pos < ring_hi;) {
        int b, ra, rb, th, z0, z1;
        decode_ring(pos, b, ra, rb, th, z0, z1);
        pos += z1 - z0;
        for (int z = z0; z < z1; ++z, ++jr) {
          const uint32_t set = jr & 1u;
          if ((int)set != grp) continue;
          trace_stamp(p.trace, jr, 4);
          tc::mbar_wait(bar.tfull + 8u * set, (jr >> 1) & 1u);
          tc::fence_after_sync();
          trace_stamp(p.trace, jr, 5);
          const int od = z * d + ra;
          const int oh = (th * p.BH + hr) * d + rb;
          const bool valid = od < p.D && oh < p.H;
          const uint32_t taddr = tmem_base + set * (uint32_t)p.set_stride + ((uint32_t)(q * 32) << 16);
          for (int it = half; it < chunks; it += 2) {
            const int c0 = it * 16;
            float v[16];
            halox_gather16(taddr, c0, p.CP, d, lo_ok, hi_ok, v);
            if (valid) conv_epilogue_row<T, 16>(p.epi, b, od, oh, pw, c0, v);
          }
          tc::fence_before_sync();
          tc::mbar_arrive(bar.tempty + 8u * set);
          trace_stamp(p.trace, jr, 6);
        }
      }
    }
    int j = 0;
    for (int tile = blockIdx.x; !p.ring && tile < num_tiles; tile += gridDim.x, ++j) {
      const uint32_t set = (uint32_t)j & 1u;
      const uint32_t use = (uint32_t)j >> 1;
      if ((int)set != grp) continue;
      int b, ra, rb, td, th;
      decode(tile, b, ra, rb, td, th);
      trace_stamp(p.trace, j, 4);
      tc::mbar_wait(bar.tfull + 8u * set, use & 1u);
      tc::fence_after_sync();
      trace_stamp(p.trace, j, 5);
      for (int it = half; it < n_items; it += 2) {
        const int m = it / chunks, c0 = (it - m * chunks) * 16;
        const int od = (td * p.BD + p.mt_pd[m] - p.hd) * d + ra;
        const int oh = (th * p.BH + p.mt_ph0[m] + hr - p.hh) * d + rb;
        const bool valid = od < p.D && oh < p.H;
        const uint32_t taddr = tmem_base + set * (uint32_t)p.set_stride + (uint32_t)(m * p.N_tile) +
                               ((uint32_t)(q * 32) << 16);
        float v[16];
        halox_gather16(taddr, c0, p.CP, d, lo_ok, hi_ok, v);
        if (valid) conv_epilogue_row<T, 16>(p.epi, b, od, oh, pw, c0, v);
      }
      tc::fence_before_sync();
      tc::mbar_arrive(bar.tempty + 8u * set);
      trace_stamp(p.trace, j, 6);
    }
  }
  cta_teardown(tmem_base, p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// SIMT direct convolution: one thread = one output position x 8 output channels
struct SimtParams {
  ConvEpi epi;
  int n_src, n_taps;
  const void* src[OCCD_CONV_MAX_SRC];
  int src_C[OCCD_CONV_MAX_SRC], src_cstride[OCCD_CONV_MAX_SRC], src_coff[OCCD_CONV_MAX_SRC];
  int ID, IH, IW, src_d0;
  int stride[3];
  const void* weight;
  int Cout_pad, Kpad;
  int w_batch_rows;
  signed char tap_src[OCCD_CONV_MAX_TAPS];
  short tap_dz[OCCD_CONV_MAX_TAPS], tap_dy[OCCD_CONV_MAX_TAPS], tap_dx[OCCD_CONV_MAX_TAPS];
};

template <typename T>
__global__ void __launch_bounds__(128) conv_simt_kernel(const __grid_constant__ SimtParams p) {
  const int ngroups = p.epi.Cout_store / 8;
  const long long total = (long long)p.epi.B * p.epi.OD * p.epi.OH * p.epi.OW * ngroups;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int g = (int)(idx % ngroups);
  long long pos = idx / ngroups;
  const int ow = (int)(pos % p.epi.OW); pos /= p.epi.OW;
  const int oh = (int)(pos % p.epi.OH); pos /= p.epi.OH;
  const int od = (int)(pos % p.epi.OD); pos /= p.epi.OD;
  const int b = (int)pos;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int tp = 0; tp < p.n_taps; ++tp) {
    const int s = p.tap_src[tp];
    const int id = od * p.stride[0] + p.tap_dz[tp] + p.src_d0;
    const int ih = oh * p.stride[1] + p.tap_dy[tp];
    const int iw = ow * p.stride[2] + p.tap_dx[tp];
    if (id < 0 || id >= p.ID || ih < 0 || ih >= p.IH || iw < 0 || iw >= p.IW) continue;
    const T* in = reinterpret_cast<const T*>(p.src[s]) +
                  ((((long long)b * p.ID + id) * p.IH + ih) * p.IW + iw) * p.src_cstride[s] + p.src_coff[s];
    const T* w = reinterpret_cast<const T*>(p.weight) +
                 ((long long)b * p.w_batch_rows + (long long)tp * p.Cout_pad + g * 8) * p.Kpad;
    const int C = p.src_C[s];
    for (int c = 0; c < C; c += 8) {
      float x[8];
      Elem<T>::ld8(in + c, x);
      if (c + 8 > C) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (c + i >= C) x[i] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float wv[8];
        Elem<T>::ld8_nc(w + (long long)j * p.Kpad + c, wv);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[j] = fmaf(x[i], wv[i], acc[j]);
      }
    }
  }
  conv_epilogue_row<T, 8>(p.epi, b, od, oh, ow, g * 8, acc);
}

// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !ptr) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

int round_up(int a, int b) { return (a + b - 1) / b * b; }

// K chunk (channels) for a source of C channels: the smallest swizzled row (32 / 64 / 128 bytes) that holds it,
// else the 128-byte row
int chunk_channels(int C, int esize) {
  for (int rb = 32; rb <= 128; rb *= 2)
    if (C <= rb / esize) return rb / esize;
  return 128 / esize;
}

long long* g_trace_buf = nullptr;

}  // namespace

// debug hook (tools/conv_trace.py): plans created while a buffer is set record per-role clock64 stamps of CTA 0
// into it ([64 tiles][8] int64, device memory owned by the caller); NULL switches tracing off again
extern "C" int occd_conv_debug_trace(long long* device_buf) {
  g_trace_buf = device_buf;
  return OCCD_OK;
}

struct occd_conv_plan {
  int impl;
  int dtype;
  int esize;
  int kc;   // channels per K chunk
  int rb;   // bytes per K chunk row (kc * esize): 128 / 64 / 32 == the swizzle mode
  TcParams tc;
  HaloParams halo;
  HaloxParams halox;
  SimtParams simt;
  CUtensorMap tmA[OCCD_CONV_MAX_SRC];
  CUtensorMap tmW;
  dim3 grid;
  size_t smem;
};

static int fill_epi(const occd_conv_desc* d, ConvEpi* e) {
  e->B = d->B; e->OD = d->OD; e->OH = d->OH; e->OW = d->OW;
  for (int i = 0; i < 3; ++i) { e->omul[i] = d->omul[i]; e->oadd[i] = d->oadd[i]; }
  e->ODf = d->ODf; e->OHf = d->OHf; e->OWf = d->OWf;
  e->Cout = d->Cout;
  e->Cout_store = round_up(d->Cout, 8);
  e->bias = d->bias;
  e->out0 = d->out0;
  e->out0_cstride = d->out0_cstride; e->out0_coff = d->out0_coff;
  e->act = d->act;
  e->out0_exact = d->out0_exact;
  e->res1 = d->res1;
  e->res1_cstride = d->res1_cstride; e->res1_coff = d->res1_coff;
  e->res2 = d->res2;
  e->res2_cstride = d->res2_cstride; e->res2_coff = d->res2_coff; e->res2_post = d->res2_post;
  e->out1_mode = d->out1_mode; e->out1 = d->out1;
  e->out1_cstride = d->out1_cstride; e->out1_coff = d->out1_coff; e->out1_C = d->out1_C;
  return 0;
}

static int n_sms_current() {
  static int n_sms[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (n_sms[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) n_sms[dev] = v;
    else n_sms[dev] = 148;
  }
  return n_sms[dev];
}

// persistent kernels: one CTA per SM, fewer when there are fewer tiles
static int persistent_grid(occd_conv_plan* pl, long long num_tiles) {
  if (num_tiles >= 2147483647LL) {
    occd_set_last_error("occd_conv_plan_create: too many tiles");
    return OCCD_ERR_UNSUPPORTED;
  }
  const int n_sms = n_sms_current();
  pl->grid = dim3((unsigned)(num_tiles < n_sms ? num_tiles : n_sms));
  return OCCD_OK;
}

static CUtensorMapSwizzle swizzle_for(int rb) {
  return rb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (rb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

static CUtensorMapDataType tm_dtype(int dtype) {
  return dtype == OCCD_DTYPE_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
}

// Tensor maps of a tcgen05 plan.  Source s: 5-D (channels, W, H, D, B) over its channel window; a box is one K chunk of
// channels x box[] positions, visited with traversal strides estr[] (box and estr in W, H, D order).  Weights: 2-D
// (Kpad, rows); a box is one K chunk x w_box_rows rows.
static int encode_maps(const occd_conv_desc* d, occd_conv_plan* pl, const int box[3], const int estr[3],
                       int w_box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    occd_set_last_error("occd_conv_plan_create: cuTensorMapEncodeTiled unavailable (no CUDA driver / GPU?)");
    return OCCD_ERR_CUDA;
  }
  const int es = pl->esize;
  const CUtensorMapSwizzle sw = swizzle_for(pl->rb);
  char msg[160];
  for (int s = 0; s < d->n_src; ++s) {
    const cuuint64_t cs = (cuuint64_t)d->src_cstride[s] * es;
    cuuint64_t gdim[5] = {(cuuint64_t)d->src_C[s], (cuuint64_t)d->IW, (cuuint64_t)d->IH, (cuuint64_t)d->ID,
                          (cuuint64_t)d->B};
    cuuint64_t gstr[4] = {cs, cs * d->IW, cs * d->IW * d->IH, cs * d->IW * d->IH * d->ID};
    cuuint32_t bx[5] = {(cuuint32_t)pl->kc, (cuuint32_t)box[0], (cuuint32_t)box[1], (cuuint32_t)box[2], 1};
    cuuint32_t ex[5] = {1, (cuuint32_t)estr[0], (cuuint32_t)estr[1], (cuuint32_t)estr[2], 1};
    void* base = (void*)((const char*)d->src[s] + (size_t)d->src_coff[s] * es);
    CUresult r = enc(&pl->tmA[s], tm_dtype(pl->dtype), 5, base, gdim, gstr, bx, ex, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      snprintf(msg, sizeof(msg), "occd_conv_plan_create: cuTensorMapEncodeTiled(source %d) failed with %d", s, (int)r);
      occd_set_last_error(msg);
      return OCCD_ERR_CUDA;
    }
  }
  for (int s = d->n_src; s < OCCD_CONV_MAX_SRC; ++s) pl->tmA[s] = pl->tmA[0];
  cuuint64_t gdim[2] = {(cuuint64_t)d->Kpad, (cuuint64_t)d->n_taps * d->Cout_pad * (d->weight_per_image ? d->B : 1)};
  cuuint64_t gstr[1] = {(cuuint64_t)d->Kpad * es};
  cuuint32_t bx[2] = {(cuuint32_t)pl->kc, (cuuint32_t)w_box_rows};
  cuuint32_t ex[2] = {1, 1};
  CUresult r = enc(&pl->tmW, tm_dtype(pl->dtype), 2, (void*)d->weight, gdim, gstr, bx, ex,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(msg, sizeof(msg), "occd_conv_plan_create: cuTensorMapEncodeTiled(weights) failed with %d", (int)r);
    occd_set_last_error(msg);
    return OCCD_ERR_CUDA;
  }
  return OCCD_OK;
}

// refusal of an impl whose kernel cannot run the described conv ("occd_conv_plan_create(<tag>): <msg>")
static int refuse(const char* tag, const char* msg) {
  char buf[256];
  snprintf(buf, sizeof(buf), "occd_conv_plan_create(%s): %s", tag, msg);
  occd_set_last_error(buf);
  return OCCD_ERR_UNSUPPORTED;
}
#define PLAN_REQUIRE(cond, tag, msg) do { if (!(cond)) return refuse(tag, msg); } while (0)

// preconditions shared by the halo kernels: a stride-1 "same" convolution of one source whose channels are one K chunk
// (Kpad == the chunk); sets the plan's K chunk
static int same_grid_one_chunk(const occd_conv_desc* d, occd_conv_plan* pl, const char* tag) {
  PLAN_REQUIRE(d->n_src == 1, tag, "one source only");
  PLAN_REQUIRE(d->stride[0] == 1 && d->stride[1] == 1 && d->stride[2] == 1, tag, "stride must be 1");
  PLAN_REQUIRE(d->omul[0] == 1 && d->omul[1] == 1 && d->omul[2] == 1 && d->oadd[0] == 0 && d->oadd[1] == 0 &&
               d->oadd[2] == 0, tag, "identity output mapping only");
  PLAN_REQUIRE(d->OD + 2 * d->src_d0 == d->ID && d->OH == d->IH && d->OW == d->IW, tag,
               "output grid must equal the input grid (plus symmetric halo margins)");
  const int KC = chunk_channels(d->src_C[0], pl->esize);
  PLAN_REQUIRE(d->src_C[0] <= KC && d->Kpad == KC, tag, "one K chunk: Kpad must equal the k-chunk");
  pl->kc = KC;
  pl->rb = KC * pl->esize;
  return OCCD_OK;
}

// Halo-tile plan (conv_halo_kernel): stride-1 "same" convolution whose taps are {-d,0,d} offsets, one source, one
// k-chunk, one N tile.  Host arithmetic, then the tensor maps.
static int plan_halo(const occd_conv_desc* d, occd_conv_plan* pl) {
  const int rc = same_grid_one_chunk(d, pl, "halo");
  if (rc != OCCD_OK) return rc;
  PLAN_REQUIRE(d->n_taps <= 27, "halo", "at most 27 taps");
  PLAN_REQUIRE(d->Cout_pad <= 128, "halo", "Cout_pad too large for the resident-weight scheme");
  int dil = 0;
  for (int i = 0; i < d->n_taps; ++i) {
    const int o[3] = {abs(d->taps[i].dz), abs(d->taps[i].dy), abs(d->taps[i].dx)};
    for (int k = 0; k < 3; ++k)
      if (o[k]) { if (!dil) dil = o[k]; PLAN_REQUIRE(o[k] == dil, "halo", "taps must be {-d,0,d} offsets"); }
  }
  PLAN_REQUIRE(dil >= 1 && dil <= 8, "halo", "dilation must be 1..8");
  int hal[3] = {0, 0, 0};
  for (int i = 0; i < d->n_taps; ++i) {
    if (d->taps[i].dz) hal[0] = 1;
    if (d->taps[i].dy) hal[1] = 1;
    if (d->taps[i].dx) hal[2] = 1;
  }
  HaloParams& h = pl->halo;
  fill_epi(d, &h.epi);
  const int row_bytes = pl->rb;
  h.d = dil; h.D = d->OD; h.H = d->IH; h.W = d->IW;
  h.src_d0 = d->src_d0;
  h.hd = hal[0]; h.hh = hal[1]; h.hw = hal[2];
  h.n_taps = d->n_taps;
  h.N_tile = d->Cout_pad;
  h.b_stride = round_up(h.N_tile * row_bytes, 1024);
  h.w_bytes = h.n_taps * h.b_stride;
  PLAN_REQUIRE(h.w_bytes <= 112 * 1024, "halo", "weights do not fit in shared memory");
  const int sD = (d->OD + dil - 1) / dil, sH = (d->IH + dil - 1) / dil, sW = (d->IW + dil - 1) / dil;
  const int smem_total = 224 * 1024 - h.w_bytes - 2048;
  // W extent of the box: the whole sub-sampled line when it fits, else equal splits of at most 62
  const int nW = (sW + 61) / 62;
  const int BW = (sW + nW - 1) / nW;
  long long best_cost = -1;
  for (int BD = 1; BD <= (hal[0] ? 4 : 1); ++BD)
    for (int BH = 1; BH <= sH && BH <= 96; ++BH) {
      const int PD = BD + 2 * hal[0], PH = BH + 2 * hal[1], PW = BW + 2 * hal[2];
      if ((PW - 1) * dil + 1 > 256 || (PH - 1) * dil + 1 > 256 || (PD - 1) * dil + 1 > 256) continue;
      const int R0 = (hal[0] * PH + hal[1]) * PW + hal[2];
      const int Rend = ((BD - 1 + hal[0]) * PH + (BH - 1 + hal[1])) * PW + BW - 1 + hal[2];
      const int nM = (Rend - R0 + 1 + 127) / 128;
      if (nM * h.N_tile > 256) continue;
      int rows_alloc = PD * PH * PW;
      if (R0 + nM * 128 + R0 > rows_alloc) rows_alloc = R0 + nM * 128 + R0;
      const int stage = round_up(rows_alloc * row_bytes, 1024);
      if (2 * stage > smem_total) continue;
      if (2 * BD * BH * BW < nM * 128) continue;  // < 50 % useful MMA rows: the per-tap kernel is the better choice
      const long long tiles = (long long)((sD + BD - 1) / BD) * ((sH + BH - 1) / BH) * nW;
      const long long cost = tiles * nM * 1000 + tiles;  // MMA work first, then tile count
      if (best_cost < 0 || cost < best_cost) {
        best_cost = cost;
        h.BD = BD; h.BH = BH; h.BW = BW; h.PD = PD; h.PH = PH; h.PW = PW;
        h.R0 = R0; h.nM = nM; h.a_stage_bytes = stage;
      }
    }
  PLAN_REQUIRE(best_cost >= 0, "halo", "no tile shape fits");
  h.tilesD = (sD + h.BD - 1) / h.BD; h.tilesH = (sH + h.BH - 1) / h.BH; h.tilesW = nW;
  h.box_bytes = h.PD * h.PH * h.PW * row_bytes;
  h.stages = smem_total / h.a_stage_bytes;
  if (h.stages > 4) h.stages = 4;
  h.set_stride = 32;
  while (h.set_stride < h.nM * h.N_tile) h.set_stride *= 2;
  h.tmem_cols = 2 * h.set_stride;
  for (int i = 0; i < d->n_taps; ++i)
    h.tap_off16[i] = (h.R0 + ((d->taps[i].dz / dil) * h.PH + d->taps[i].dy / dil) * h.PW + d->taps[i].dx / dil) *
                     row_bytes / 16;
  h.trace = g_trace_buf;
  pl->smem = (size_t)h.w_bytes + (size_t)h.stages * h.a_stage_bytes + 128 + 1024;
  const int rg = persistent_grid(pl, (long long)d->B * dil * dil * dil * h.tilesD * h.tilesH * h.tilesW);
  if (rg != OCCD_OK) return rg;
  const int box[3] = {(h.PW - 1) * dil + 1, (h.PH - 1) * dil + 1, (h.PD - 1) * dil + 1};
  const int estr[3] = {dil, dil, dil};
  return encode_maps(d, pl, box, estr, h.N_tile);
}


// x-packed halo plan (conv_halox_kernel): host arithmetic, then the tensor maps
static int plan_halox(const occd_conv_desc* d, occd_conv_plan* pl) {
  const int rc = same_grid_one_chunk(d, pl, "halox");
  if (rc != OCCD_OK) return rc;
  PLAN_REQUIRE(d->IW == 8 || d->IW == 16 || d->IW == 32, "halox",
               "innermost extent W must be 8, 16 or 32 (one warp row)");
  PLAN_REQUIRE(d->n_taps % 3 == 0 && d->n_taps <= 27, "halox", "taps must come as W triples");
  PLAN_REQUIRE(3 * d->Cout_pad <= 256, "halox", "3 * Cout_pad <= 256");
  const int dil = d->taps[2].dx;
  PLAN_REQUIRE(dil >= 1 && dil <= 8 && dil < d->IW, "halox", "W dilation");
  int hal[2] = {0, 0};
  for (int i = 0; i < d->n_taps; i += 3) {
    const occd_conv_tap &a = d->taps[i], &b = d->taps[i + 1], &c = d->taps[i + 2];
    PLAN_REQUIRE(a.dx == -dil && b.dx == 0 && c.dx == dil && a.dz == b.dz && a.dz == c.dz && a.dy == b.dy &&
                 a.dy == c.dy, "halox", "taps must be ordered (dz, dy) groups of dx = -d, 0, +d");
    PLAN_REQUIRE((a.dz == 0 || abs(a.dz) == dil) && (a.dy == 0 || abs(a.dy) == dil), "halox",
                 "D / H taps must be {-d, 0, d}");
    if (a.dz) hal[0] = 1;
    if (a.dy) hal[1] = 1;
  }
  HaloxParams& h = pl->halox;
  fill_epi(d, &h.epi);
  const int RB = pl->rb, NMMA = RB / 32;
  h.d = dil; h.D = d->OD; h.H = d->IH;
  h.src_d0 = d->src_d0;
  h.hd = hal[0]; h.hh = hal[1];
  h.n_groups = d->n_taps / 3;
  h.CP = d->Cout_pad;
  h.N_tile = 3 * d->Cout_pad;
  h.PW = d->IW;
  h.b_stride = round_up(h.N_tile * RB, 1024);
  h.w_bytes = h.n_groups * h.b_stride;
  const int smem_total = 227 * 1024 - h.w_bytes - 4096;   // barriers, TMEM slot, 1024-byte alignment slack
  PLAN_REQUIRE(smem_total > 0, "halox", "weights do not fit in shared memory");
  const int HR = 128 / h.PW;                               // h-rows of one plane per M tile
  const int sD = (d->OD + dil - 1) / dil, sH = (d->IH + dil - 1) / dil;
  // CTA tile = BD planes x nB blocks of HR h-rows (<= 2 M tiles: two accumulator sets of nM x N_tile columns)
  double best = -1.0;
  const int cand[3][2] = {{1, 1}, {1, 2}, {2, 1}};
  for (int ci = 0; ci < 3; ++ci) {
    const int BD = cand[ci][0], nB = cand[ci][1];
    const int BH = nB * HR, PD = BD + 2 * hal[0], PH = BH + 2 * hal[1];
    if ((PH - 1) * dil + 1 > 256 || (PD - 1) * dil + 1 > 256) continue;
    const int rows = PD * PH * h.PW;
    const int stage = round_up(rows * RB, 1024);
    if (stage > smem_total) continue;
    const int stages = smem_total / stage;
    const int nM = BD * nB;
    int set_stride = 32;
    while (set_stride < nM * h.N_tile) set_stride *= 2;
    if (2 * set_stride > 512) continue;
    // cycles per useful output: MMA issue floor (59 cycles per instruction at N <= 118) plus, single-buffered,
    // the un-overlapped L2 -> smem fill at the chip's ~42 B/cycle/SM
    const double eff_d = (double)(sD < BD ? sD : BD) / BD, eff_h = (double)(sH < BH ? sH : BH) / BH;
    const double mma = (double)nM * h.n_groups * NMMA * (h.N_tile > 118 ? h.N_tile / 2.0 : 59.0);
    const double fill = stages >= 2 ? 0.0 : (double)rows * RB / 42.0;
    // (tie-break: the tile that reloads the fewest halo rows per output)
    const double cost = (mma + fill + 1e-3 * rows * RB) / (BD * BH * h.PW * eff_d * eff_h);
    if (best < 0 || cost < best) {
      best = cost;
      h.BD = BD; h.BH = BH; h.PD = PD; h.PH = PH; h.nM = nM;
      h.a_stage_bytes = stage; h.stages = stages > 4 ? 4 : stages;
      h.set_stride = set_stride;
    }
  }
  PLAN_REQUIRE(best >= 0, "halox", "no tile shape fits");
  h.ring = 0;
  {
    // plane ring instead of a single-stage box (see HaloxParams): needs D taps and four single-plane stages
    const int PHr = HR + 2 * hal[1];
    const int plane = round_up(PHr * h.PW * RB, 1024);
    if (h.stages < 2 && hal[0] == 1 && 4 * plane <= smem_total && (PHr - 1) * dil + 1 <= 256) {
      h.ring = 1;
      h.BD = 1; h.BH = HR; h.PD = 3; h.PH = PHr; h.nM = 1;
      h.a_stage_bytes = plane; h.stages = 4;
      h.set_stride = 32;
      while (h.set_stride < h.N_tile) h.set_stride *= 2;
    }
  }
  {
    const int nB = h.BH / HR;
    int m = 0;
    for (int pd = 0; pd < h.BD; ++pd)
      for (int blk = 0; blk < nB; ++blk, ++m) {
        h.mt_pd[m] = pd + h.hd;
        h.mt_ph0[m] = h.hh + blk * HR;
        h.mt_row[m] = (h.mt_pd[m] * h.PH + h.mt_ph0[m]) * h.PW;
      }
  }
  h.tmem_cols = 2 * h.set_stride;
  h.tilesD = (sD + h.BD - 1) / h.BD; h.tilesH = (sH + h.BH - 1) / h.BH;
  h.box_bytes = (h.ring ? 1 : h.PD) * h.PH * h.PW * RB;
  for (int g = 0; g < h.n_groups; ++g) {
    h.grp_off[g] = ((d->taps[3 * g].dz / dil) * h.PH + d->taps[3 * g].dy / dil) * h.PW;
    h.grp_dz[g] = (signed char)(d->taps[3 * g].dz / dil);
    h.grp_row[g] = (short)((h.hh + d->taps[3 * g].dy / dil) * h.PW);
  }
  h.sD = sD;
  h.n_cols = d->B * dil * dil * h.tilesH;
  h.trace = g_trace_buf;
  pl->smem = (size_t)h.w_bytes + (size_t)h.stages * h.a_stage_bytes + 128 + 512 + 1024;   // barriers, ring-mode descriptor table, alignment slack
  const long long num_tiles = h.ring ? (long long)h.n_cols * sD      // ring mode: M tiles; each CTA takes a contiguous share
                                     : (long long)d->B * dil * dil * h.tilesD * h.tilesH;
  const int rg = persistent_grid(pl, num_tiles);
  if (rg != OCCD_OK) return rg;
  const int box[3] = {h.PW, (h.PH - 1) * dil + 1, h.ring ? 1 : (h.PD - 1) * dil + 1};   // ring mode: one plane per load
  const int estr[3] = {1, dil, dil};
  return encode_maps(d, pl, box, estr, h.N_tile);
}

// Per-tap (TC) plan: host arithmetic, then the tensor maps.  xp: x-packed variant (TCX)
static int plan_tc(const occd_conv_desc* d, occd_conv_plan* pl, bool xp) {
  int maxC = 0;
  for (int s = 0; s < d->n_src; ++s) maxC = d->src_C[s] > maxC ? d->src_C[s] : maxC;
  TcParams& t = pl->tc;
  fill_epi(d, &t.epi);
  const int KC = chunk_channels(maxC, pl->esize);
  pl->kc = KC;
  pl->rb = KC * pl->esize;
  const int RB = pl->rb;
  if (d->Kpad % KC != 0) {
    occd_set_last_error("occd_conv_plan_create: Kpad must be a multiple of the K chunk");
    return OCCD_ERR_ARG;
  }
  t.n_taps = xp ? d->n_taps / 3 : d->n_taps;  // x-packed: one pipeline item per (source, dz, dy) group
  const int n_groups = d->n_groups > 1 ? d->n_groups : 1;
  if (n_groups > 1) {
    bool ok = !xp && n_groups <= OCCD_CONV_MAX_GROUPS && d->group_tap0[0] == 0 && d->group_tap0[n_groups] == d->n_taps &&
              d->out1_mode == OCCD_OUT1_NONE && d->out0 != nullptr &&
              (d->res2 == nullptr || (d->res2_post && d->res1 == nullptr));
    for (int g = 0; ok && g < n_groups; ++g) {
      ok = d->group_tap0[g + 1] > d->group_tap0[g];
      for (int i = 0; i < 3; ++i) ok = ok && d->group_oadd[g][i] >= 0 && d->group_oadd[g][i] < d->omul[i];
    }
    if (!ok) {
      occd_set_last_error("occd_conv_plan_create: tap groups need the per-tap TC kernel, ascending non-empty tap "
                          "ranges covering all taps, 0 <= group_oadd < omul, no second output and at most one residual");
      return OCCD_ERR_UNSUPPORTED;
    }
  }
  t.n_groups = n_groups;
  t.src_d0 = d->src_d0;
  t.w_batch_rows = d->weight_per_image ? d->n_taps * d->Cout_pad : 0;
  for (int s = 0; s < OCCD_CONV_MAX_SRC; ++s) t.n_kchunks[s] = s < d->n_src ? (d->src_C[s] + KC - 1) / KC : 0;
  for (int i = 0; i < 3; ++i) t.stride[i] = d->stride[i];
  for (int g = 0; g < n_groups; ++g) {
    t.grp_tap0[g] = (short)(n_groups > 1 ? d->group_tap0[g] : 0);
    t.grp_tap0[g + 1] = (short)(n_groups > 1 ? d->group_tap0[g + 1] : t.n_taps);
    for (int i = 0; i < 3; ++i) t.grp_oadd[g][i] = (signed char)(n_groups > 1 ? d->group_oadd[g][i] : 0);
  }
  if (xp) {
    // groups of three W taps -1, 0, +1 share one MMA with N = 3 * Cout_pad; the tile is 32 positions wide (30
    // outputs + one halo column each side) so that lane == column in the epilogue
    if (d->n_taps % 3 || d->stride[2] != 1 || 3 * d->Cout_pad > 256) {
      occd_set_last_error("occd_conv_plan_create(tcx): needs W-tap triples, W stride 1 and 3 * Cout_pad <= 256");
      return OCCD_ERR_UNSUPPORTED;
    }
    for (int i = 0; i < d->n_taps; i += 3) {
      const occd_conv_tap &a = d->taps[i], &b = d->taps[i + 1], &c = d->taps[i + 2];
      if (!(a.dx == -1 && b.dx == 0 && c.dx == 1 && a.src == b.src && a.src == c.src && a.dz == b.dz &&
            a.dz == c.dz && a.dy == b.dy && a.dy == c.dy)) {
        occd_set_last_error("occd_conv_plan_create(tcx): taps must be ordered (src, dz, dy) groups of dx = -1, 0, +1");
        return OCCD_ERR_UNSUPPORTED;
      }
      t.tap_src[i / 3] = (signed char)b.src;
      t.tap_dz[i / 3] = (short)b.dz; t.tap_dy[i / 3] = (short)b.dy; t.tap_dx[i / 3] = 0;
    }
    t.TW = 32;
    long long best = -1;
    for (int th = 4; th >= 1; th >>= 1) {
      const int tdd = 4 / th;
      const long long vol = (long long)round_up(d->OH, th) * round_up(d->OD, tdd);
      if (best < 0 || vol < best) { best = vol; t.TH = th; t.TD = tdd; }
    }
  } else {
    for (int i = 0; i < d->n_taps; ++i) {
      t.tap_src[i] = (signed char)d->taps[i].src;
      t.tap_dz[i] = (short)d->taps[i].dz; t.tap_dy[i] = (short)d->taps[i].dy; t.tap_dx[i] = (short)d->taps[i].dx;
    }
    // tile box (TD,TH,TW), product 128: minimal padded volume, but a wide innermost extent (long contiguous TMA
    // runs, coalesced stores) wins whenever it costs < 4% extra positions
    long long best = -1;
    for (int pass = 0; pass < 2; ++pass)
      for (int tw = 128; tw >= 1; tw >>= 1)
        for (int th = 128 / tw; th >= 1; th >>= 1) {
          const int tdd = 128 / (tw * th);
          if (tw * d->stride[2] > 256 || th * d->stride[1] > 256 || tdd * d->stride[0] > 256) continue;
          const long long vol = (long long)round_up(d->OW, tw) * round_up(d->OH, th) * round_up(d->OD, tdd);
          if (pass == 0) {
            if (best < 0 || vol < best) best = vol;
          } else if (vol * 100 <= best * 104) {
            t.TW = tw; t.TH = th; t.TD = tdd;
            pass = 2; tw = 0; break;  // first hit in (widest TW, tallest TH) order
          }
        }
  }
  t.TWv = xp ? 30 : t.TW;
  t.tiles_w = (d->OW + t.TWv - 1) / t.TWv; t.tiles_h = (d->OH + t.TH - 1) / t.TH; t.tiles_d = (d->OD + t.TD - 1) / t.TD;
  // N tile: the divisor of Cout_pad (multiple of 16, <= 256) with the smallest estimated makespan.  Three measured
  // B200 constants drive the model (profiles/r02_mma_issue_bench.txt, r02_conv_role_traces.txt, r02_membw.txt):
  //   one tcgen05.mma costs max(59, N/2) cycles for M = 128, any operand type
  //   an SM pulls ~44 bytes/cycle from L2 when the whole chip does (6300 B/cycle chip-wide)
  //   the epilogue drains ~7-12 bytes/cycle/SM (fast path; 12 measured best for the whole forward, r02c)
  // A tile's main loop (TMA + MMA) overlaps the previous tile's epilogue, so a CTA's time is
  // waves * max(mainloop, epilogue) + min(mainloop, epilogue).  Small-M layers (late encoder stages: 9 M tiles) get
  // narrow N tiles that spread the write-bound epilogue over every SM; large-M layers get the widest tile (fewest
  // re-reads of the A operand).
  t.Cout_pad = d->Cout_pad;
  {
    int iters = 0;
    for (int i = 0; i < t.n_taps; ++i) iters += t.n_kchunks[t.tap_src[i]];
    iters = (iters + n_groups - 1) / n_groups;   // tap groups: the mean group; every CTA gets its share of each
    const long long m_tiles0 = (long long)d->B * t.tiles_d * t.tiles_h * t.tiles_w * n_groups;
    const int n_sms = n_sms_current();
    const double out_bytes_per_col = 128.0 * ((d->out0 ? pl->esize : 0) + (d->out1_mode == OCCD_OUT1_CL ? pl->esize : 0) +
                                              (d->out1_mode == OCCD_OUT1_F32_PLANAR ? 4 : 0));
    const double epi_rate = 12.0;
    double best = -1.0;
    t.N_tile = 16;
    for (int n = 16; n <= 256 && n <= d->Cout_pad; n += 16) {
      if (d->Cout_pad % n) continue;
      const double mma = (RB / 32) * (n > 118 ? n / 2.0 : 59.0);
      const double load = (128.0 + n) * RB / 44.0;
      const double mainloop = iters * (mma > load ? mma : load);
      const double epi = out_bytes_per_col * n / epi_rate;
      const long long tiles = m_tiles0 * (d->Cout_pad / n);
      const double waves = (double)((tiles + n_sms - 1) / n_sms);
      const double span = waves * (mainloop > epi ? mainloop : epi) + (mainloop > epi ? epi : mainloop);
      if (best < 0 || span <= best * 1.02) {   // within 2 %: the wider tile (fewer tiles, fewer A re-reads) wins
        if (best < 0 || span < best) best = span;
        t.N_tile = n;
      }
    }
  }
  if (xp) t.N_tile = 3 * d->Cout_pad;  // one N tile: the three taps' weights stacked
  t.tmem_cols = 32;
  while (t.tmem_cols < t.N_tile) t.tmem_cols *= 2;
  t.trace = g_trace_buf;
  t.tmem_cols *= 2;  // two accumulators: the epilogue of tile j overlaps the MMAs of tile j+1
  t.a_bytes = 128 * RB;
  t.b_bytes = t.N_tile * RB;
  t.b_stride = round_up(t.b_bytes, 1024);
  const int stage_bytes = t.a_bytes + t.b_stride;
  int total_iters = 0;   // (tap, k-chunk) items of one tile; with tap groups: of the largest group
  for (int g = 0; g < n_groups; ++g) {
    int it = 0;
    for (int i = t.grp_tap0[g]; i < t.grp_tap0[g + 1]; ++i) it += t.n_kchunks[t.tap_src[i]];
    t.grp_iters[g] = (short)it;
    if (it > total_iters) total_iters = it;
  }
  const int budget = 200 * 1024;  // persistent kernel: one CTA per SM owns the shared memory
  // (tap, k-chunk) items per pipeline stage: the single-thread producer/MMA hand-off costs ~0.25 us, so a stage
  // must carry >= ~512 tensor-pipe cycles of work (or up to 9 items) while leaving >= 3 stages in flight
  const int mma_cycles_per_item = (RB / 32) * (128 * t.N_tile / 256);
  int group = (512 + mma_cycles_per_item - 1) / mma_cycles_per_item;
  if (group > 9) group = 9;
  if (group > total_iters) group = total_iters;
  while (group > 1 && 3 * group * stage_bytes > budget) --group;
  t.group = group;
  int stages = budget / (group * stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  const int groups_per_tile = (total_iters + group - 1) / group;
  {
    // ring depth: two tiles' worth of stage groups, but never fewer than 8 stages when they fit (a conv with one
    // item per tile otherwise keeps only two TMA loads in flight)
    int cap = 2 * groups_per_tile;
    if (cap < 8) cap = 8;
    if (stages > cap) stages = cap;
  }
  if (stages < 1) stages = 1;
  t.stages = stages;
  pl->smem = (size_t)stages * group * stage_bytes + 16 * kMaxStages + 64 + 1024;  // + barriers + alignment slack
  const long long m_tiles = (long long)d->B * t.tiles_d * t.tiles_h * t.tiles_w;
  const int rg = persistent_grid(pl, m_tiles * (xp ? 1 : d->Cout_pad / t.N_tile) * n_groups);
  if (rg != OCCD_OK) return rg;
  t.num_m_tiles = (int)m_tiles;
  const int box[3] = {t.TW * d->stride[2], t.TH * d->stride[1], t.TD * d->stride[0]};
  const int estr[3] = {d->stride[2], d->stride[1], d->stride[0]};
  return encode_maps(d, pl, box, estr, t.N_tile);
}

// Hands the kernel instantiation of a tcgen05 plan (dtype x impl x K-chunk row bytes) and its arguments to
// f(kernel, args...)
template <typename T, int RB, typename F>
static cudaError_t with_tc_kernel_rb(const occd_conv_plan* pl, F&& f) {
  switch (pl->impl) {
    case OCCD_CONV_IMPL_TC: return f(conv_tc_kernel<T, RB, false>, pl->tc, pl->tmA[0], pl->tmA[1], pl->tmA[2], pl->tmW);
    case OCCD_CONV_IMPL_TCX: return f(conv_tc_kernel<T, RB, true>, pl->tc, pl->tmA[0], pl->tmA[1], pl->tmA[2], pl->tmW);
    case OCCD_CONV_IMPL_HALO: return f(conv_halo_kernel<T, RB>, pl->halo, pl->tmA[0], pl->tmW);
    default: return f(conv_halox_kernel<T, RB>, pl->halox, pl->tmA[0], pl->tmW);
  }
}

template <typename T, typename F>
static cudaError_t with_tc_kernel_t(const occd_conv_plan* pl, F&& f) {
  switch (pl->rb) {
    case 128: return with_tc_kernel_rb<T, 128>(pl, f);
    case 64: return with_tc_kernel_rb<T, 64>(pl, f);
    default: return with_tc_kernel_rb<T, 32>(pl, f);
  }
}

template <typename F>
static cudaError_t with_tc_kernel(const occd_conv_plan* pl, F&& f) {
  if (pl->dtype == OCCD_DTYPE_F32) return with_tc_kernel_t<float>(pl, f);
  return with_tc_kernel_t<__nv_bfloat16>(pl, f);
}

extern "C" int occd_conv_plan_create(const occd_conv_desc* d, occd_conv_plan** out) {
  OCCD_CHECK_ARG(d && out, "occd_conv_plan_create: null argument");
  OCCD_CHECK_ARG(d->dtype == OCCD_DTYPE_F32 || d->dtype == OCCD_DTYPE_BF16, "occd_conv_plan_create: dtype");
  OCCD_CHECK_ARG(d->n_src >= 1 && d->n_src <= OCCD_CONV_MAX_SRC, "occd_conv_plan_create: n_src");
  OCCD_CHECK_ARG(d->n_taps >= 1 && d->n_taps <= OCCD_CONV_MAX_TAPS, "occd_conv_plan_create: n_taps");
  OCCD_CHECK_ARG(d->src_d0 >= 0 && d->src_d0 < d->ID, "occd_conv_plan_create: src_d0");
  OCCD_CHECK_ARG(d->B > 0 && d->ID > 0 && d->IH > 0 && d->IW > 0 && d->OD > 0 && d->OH > 0 && d->OW > 0,
                 "occd_conv_plan_create: dims");
  OCCD_CHECK_ARG(d->Cout > 0 && d->Cout_pad >= d->Cout && d->Cout_pad % 16 == 0, "occd_conv_plan_create: Cout_pad");
  OCCD_CHECK_ARG(d->Kpad > 0 && d->Kpad % 8 == 0, "occd_conv_plan_create: Kpad must be a multiple of 8");
  OCCD_CHECK_ARG(d->weight && d->bias, "occd_conv_plan_create: weight/bias");
  OCCD_CHECK_ARG(d->out0 || d->out1_mode != OCCD_OUT1_NONE, "occd_conv_plan_create: no output");
  const int es = d->dtype == OCCD_DTYPE_F32 ? 4 : 2;
  auto aligned = [es](const void* p) { return (reinterpret_cast<uintptr_t>(p) % (8 * es)) == 0; };
  const int cst = round_up(d->Cout, 8);
  if (d->out0) OCCD_CHECK_ARG(d->out0_coff % 8 == 0 && d->out0_cstride % 8 == 0 && d->out0_coff + cst <= d->out0_cstride &&
                              aligned(d->out0), "occd_conv_plan_create: out0 channel window");
  if (d->res1) OCCD_CHECK_ARG(d->res1_coff % 8 == 0 && d->res1_cstride % 8 == 0 && d->res1_coff + cst <= d->res1_cstride &&
                              aligned(d->res1), "occd_conv_plan_create: res1 channel window");
  if (d->res2) OCCD_CHECK_ARG(d->res2_coff % 8 == 0 && d->res2_cstride % 8 == 0 && d->res2_coff + cst <= d->res2_cstride &&
                              aligned(d->res2), "occd_conv_plan_create: res2 channel window");
  if (d->out1_mode == OCCD_OUT1_CL)
    OCCD_CHECK_ARG(d->out1 && d->out1_coff % 8 == 0 && d->out1_cstride % 8 == 0 && d->out1_coff + cst <= d->out1_cstride &&
                   aligned(d->out1), "occd_conv_plan_create: out1 channel window");
  if (d->out1_mode == OCCD_OUT1_F32_PLANAR)
    OCCD_CHECK_ARG(d->out1 && d->out1_coff + d->Cout <= d->out1_C, "occd_conv_plan_create: out1 planar window");
  for (int i = 0; i < 3; ++i) {
    OCCD_CHECK_ARG(d->stride[i] >= 1 && d->stride[i] <= 8 && d->omul[i] >= 1, "occd_conv_plan_create: stride/omul");
  }
  OCCD_CHECK_ARG((long long)(d->OD - 1) * d->omul[0] + d->oadd[0] < d->ODf &&
                 (long long)(d->OH - 1) * d->omul[1] + d->oadd[1] < d->OHf &&
                 (long long)(d->OW - 1) * d->omul[2] + d->oadd[2] < d->OWf, "occd_conv_plan_create: output mapping");
  for (int s = 0; s < d->n_src; ++s) {
    OCCD_CHECK_ARG(d->src[s] && d->src_C[s] > 0 && d->src_cstride[s] % 8 == 0 && d->src_coff[s] % 8 == 0 &&
                   d->src_coff[s] + d->src_C[s] <= d->src_cstride[s] && aligned(d->src[s]),
                   "occd_conv_plan_create: source channel window");
    OCCD_CHECK_ARG(d->src_C[s] <= d->Kpad, "occd_conv_plan_create: Kpad smaller than a source");
  }
  for (int i = 0; i < d->n_taps; ++i) {
    OCCD_CHECK_ARG(d->taps[i].src >= 0 && d->taps[i].src < d->n_src, "occd_conv_plan_create: tap source");
    OCCD_CHECK_ARG(abs(d->taps[i].dz) < 30000 && abs(d->taps[i].dy) < 30000 && abs(d->taps[i].dx) < 30000,
                   "occd_conv_plan_create: tap offset");
  }
  OCCD_CHECK_ARG(d->impl == OCCD_CONV_IMPL_TC || d->impl == OCCD_CONV_IMPL_SIMT || d->impl == OCCD_CONV_IMPL_HALO ||
                 d->impl == OCCD_CONV_IMPL_TCX || d->impl == OCCD_CONV_IMPL_HALOX, "occd_conv_plan_create: impl");
  OCCD_CHECK_ARG(d->n_groups <= 1 || d->impl == OCCD_CONV_IMPL_TC, "occd_conv_plan_create: tap groups: TC impl only");
  OCCD_CHECK_ARG(!d->weight_per_image || (d->impl != OCCD_CONV_IMPL_HALO && d->impl != OCCD_CONV_IMPL_HALOX),
                 "occd_conv_plan_create: per-image weights: TC or SIMT impl");

  occd_conv_plan* pl = new (std::nothrow) occd_conv_plan;
  OCCD_CHECK_ARG(pl != nullptr, "occd_conv_plan_create: out of memory");
  memset(pl, 0, sizeof(*pl));
  pl->impl = d->impl;
  pl->dtype = d->dtype;
  pl->esize = es;

  if (d->impl == OCCD_CONV_IMPL_SIMT) {
    SimtParams& s = pl->simt;
    fill_epi(d, &s.epi);
    s.n_src = d->n_src; s.n_taps = d->n_taps;
    for (int i = 0; i < d->n_src; ++i) {
      s.src[i] = d->src[i];
      s.src_C[i] = d->src_C[i]; s.src_cstride[i] = d->src_cstride[i]; s.src_coff[i] = d->src_coff[i];
    }
    s.ID = d->ID; s.IH = d->IH; s.IW = d->IW; s.src_d0 = d->src_d0;
    for (int i = 0; i < 3; ++i) s.stride[i] = d->stride[i];
    s.weight = d->weight;
    s.Cout_pad = d->Cout_pad; s.Kpad = d->Kpad;
    s.w_batch_rows = d->weight_per_image ? d->n_taps * d->Cout_pad : 0;
    for (int i = 0; i < d->n_taps; ++i) {
      s.tap_src[i] = (signed char)d->taps[i].src;
      s.tap_dz[i] = (short)d->taps[i].dz; s.tap_dy[i] = (short)d->taps[i].dy; s.tap_dx[i] = (short)d->taps[i].dx;
    }
    const long long total = (long long)d->B * d->OD * d->OH * d->OW * (s.epi.Cout_store / 8);
    pl->grid = dim3((unsigned)((total + 127) / 128));
    *out = pl;
    return OCCD_OK;
  }

  int rc = d->impl == OCCD_CONV_IMPL_HALO    ? plan_halo(d, pl)
           : d->impl == OCCD_CONV_IMPL_HALOX ? plan_halox(d, pl)
                                             : plan_tc(d, pl, d->impl == OCCD_CONV_IMPL_TCX);
  if (rc == OCCD_OK) {
    // the plan's pointers belong to the device current at creation: its kernel may use up to 227 KB of smem there
    const cudaError_t e = with_tc_kernel(pl, [](auto kernel, const auto&...) {
      return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    });
    if (e != cudaSuccess) {
      occd_set_last_error(cudaGetErrorString(e));
      rc = OCCD_ERR_CUDA;
    }
  }
  if (rc != OCCD_OK) { delete pl; return rc; }
  *out = pl;
  return OCCD_OK;
}

extern "C" int occd_conv_plan_destroy(occd_conv_plan* plan) {
  delete plan;
  return OCCD_OK;
}

extern "C" int occd_conv_plan_info(const occd_conv_plan* pl, int* info) {
  OCCD_CHECK_ARG(pl && info, "occd_conv_plan_info: null");
  if (pl->impl == OCCD_CONV_IMPL_SIMT) {
    for (int i = 0; i < 8; ++i) info[i] = 0;
    info[6] = (int)pl->grid.x;
    return OCCD_OK;
  }
  if (pl->impl == OCCD_CONV_IMPL_HALO) {
    const HaloParams& h = pl->halo;
    info[0] = h.BD; info[1] = h.BH; info[2] = h.BW; info[3] = h.N_tile; info[4] = pl->kc;
    info[5] = h.stages * 100 + h.nM; info[6] = (int)pl->grid.x;
    info[7] = h.epi.B * h.d * h.d * h.d * h.tilesD * h.tilesH * h.tilesW;
    return OCCD_OK;
  }
  if (pl->impl == OCCD_CONV_IMPL_HALOX) {
    const HaloxParams& h = pl->halox;
    info[0] = h.BD; info[1] = h.BH; info[2] = h.PW; info[3] = h.N_tile; info[4] = pl->kc;
    info[5] = h.stages * 100 + h.nM; info[6] = (int)pl->grid.x;
    info[7] = h.epi.B * h.d * h.d * h.tilesD * h.tilesH;
    return OCCD_OK;
  }
  info[0] = pl->tc.TD; info[1] = pl->tc.TH; info[2] = pl->tc.TW; info[3] = pl->tc.N_tile;
  info[4] = pl->kc; info[5] = pl->tc.stages * 100 + pl->tc.group; info[6] = (int)pl->grid.x;
  info[7] = pl->tc.num_m_tiles * (pl->impl == OCCD_CONV_IMPL_TCX ? 1 : pl->tc.Cout_pad / pl->tc.N_tile);
  return OCCD_OK;
}

extern "C" int occd_conv_run(const occd_conv_plan* pl, void* stream) {
  OCCD_CHECK_ARG(pl != nullptr, "occd_conv_run: null plan");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (pl->impl == OCCD_CONV_IMPL_SIMT) {
    if (pl->dtype == OCCD_DTYPE_F32) conv_simt_kernel<float><<<pl->grid, 128, 0, st>>>(pl->simt);
    else conv_simt_kernel<__nv_bfloat16><<<pl->grid, 128, 0, st>>>(pl->simt);
    OCCD_CHECK_LAUNCH();
    return OCCD_OK;
  }
  // programmatic dependent launch (common.cuh): the prologue of the persistent kernels overlaps the tail of the
  // previous grid.  Measured on B200 (round 2, profiles/r02_ab_experiments.txt): 1.0 % of the config-2 forward,
  // results bit-identical.
  const cudaError_t e = with_tc_kernel(pl, [&](auto kernel, const auto&... args) {
    return occd_launch(kernel, pl->grid, dim3(kTcThreads), pl->smem, st, args...);
  });
  if (e != cudaSuccess) {
    occd_set_last_error(cudaGetErrorString(e));
    return OCCD_ERR_CUDA;
  }
  return OCCD_OK;
}
