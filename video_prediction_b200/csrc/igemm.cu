// Tensor-core implicit-GEMM convolution engine for B200 (sm_100a).
//
//   D[pixels, Cout] = sum_taps  A_tap[pixels, Cin] * W_tap[Cin, Cout]          (fwd / dgrad)
//   dW_tap[Cout, Cin] = sum_pixels dY[pixels, Cout]^T * X_tap[pixels, Cin]     (wgrad)
//
// Operands are fp32 in HBM/shared memory and are consumed by tcgen05.mma kind::tf32 with fp32
// accumulation in TMEM.  Activation tiles are fetched with 5-D TMA boxes straight from the NDHWC
// tensor: a box of bw x bh x bd x bn output positions is one 128-row (64-row for wgrad) operand
// tile whose rows are 32 channels = 128 bytes, written by TMA with the 128-byte swizzle the UMMA
// descriptor expects.  A filter tap is a coordinate shift of the box; TMA zero-fills out-of-bounds
// rows/channels, which *is* the convolution's zero padding.  Strided convolutions read one of
// s_d*s_h*s_w "parity" sub-lattices of the input (one tensor map each); transposed convolutions
// (upsample_conv2d forward, dgrad of strided convs) are split into output phases.
//
// Two forward / dgrad kernels compute the same convolution (the host layer times both per geometry): BOX mode above, and HALO
// mode (igemm_halo_kernel): M = 256 per CTA as two 128-row sub-tiles, one halo tile per (tap group, 32-channel chunk) on which
// every tap is a shifted K-major descriptor, weight tiles shared by both sub-tiles (two taps per ring stage), one MMA-issuing
// thread per sub-tile.  Weight gradients: row mode (one x halo tile per kernel row) and tap-group mode (merged-tap wide-N MMAs).
//
// Warp roles (224 threads; wgrad 192; halo 256): warp 0 (+ warp 6 in the forward kernel: weights) = TMA producer, warp 1 = TMEM allocator + single-thread MMA
// issuer, warps 2..5 = epilogue (TMEM -> registers -> bias/activation -> global).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <tuple>
#include <vector>

#include "common.h"
#include "ptx.cuh"
#include "tensormap.h"

namespace vp {

constexpr int kMaxTaps = 128;
constexpr int kMaxMaps = 8;
constexpr int kStagesFwd = 4;
constexpr int kKsubMinIters = 48;  // k-iterations per CTA from which two k-chunks per stage pay off
constexpr int kMaxStagesFwd = 6;
constexpr int kWgPix = 64;  // pixels (GEMM-K) per wgrad pipeline stage

struct Tap {
  int8_t map, cd, ch, cw;
  int32_t wslot;
};

struct alignas(64) IgemmArgs {
  CUtensorMap amap[kMaxMaps];  // shifted operand, one map per stride parity
  CUtensorMap bmap;            // fwd: packed weights (2-D);  wgrad: the un-shifted operand (5-D)
  int32_t tiles_w, tiles_h, tiles_d, tiles_n;
  int32_t bw, bh, bd, bn;
  int32_t kc, n_pad, bn_tile, tmem_cols;
  int32_t num_phases, splits;
  int32_t phase_begin[9];
  int8_t phase_ooff[8][4];
  int32_t os_d, os_h, os_w;
  float* out;
  long long so_n, so_d, so_h, so_w;
  int32_t out_n, out_d, out_h, out_w, out_c;
  const float* bias;
  int32_t act;
  float alpha;
  int32_t accumulate;
  const float* aux_y;    // optional: activation OUTPUT with the layout of `out`; result is multiplied by act'(aux_y)
  const float* aux_add;  // optional addend (same layout), added before the multiplication
  int32_t aux_act;
  // wgrad only
  int32_t rows_from_shifted, m_tiles, n_tiles, kpad;
  int32_t tap_group, num_taps, rows_valid, wg_stages, stages;
  int32_t ksub;          // 32-channel k-chunks per pipeline stage (1 or 2): two chunks halve the per-MMA cost of the issue loops
  int32_t halo_w, halo_sub, row_kw, row_pw;   // wgrad row mode: halo box width (pixels), padded bytes of one halo sub-tile, kw, pw
  int32_t k_tail;        // MMAs (K = 8 channels each) that hold real channels in the LAST k-chunk of a tap (1..4)
  int32_t dbg_trace, dbg_poll;
  int32_t dbg_skip;      // timing experiments only (VP_FWD_SKIP): 1 = no activation loads, 2 = no weight loads
  uint32_t wg_stage_bytes;
  Tap taps[kMaxTaps];
};

// Optional per-CTA timeline (VP_FWD_TRACE=1; read back with vp_debug_read_trace): 8 globaltimer stamps per CTA.
__device__ unsigned long long g_trace[16 * 2048];
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define VP_TRACE(slot)                                                                                       \
  do {                                                                                                       \
    if (DBG && a.dbg_trace) {                                                                                \
      const int cta_ = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);                        \
      if (cta_ < 2048) g_trace[cta_ * 16 + (slot)] = gtimer();                                                \
    }                                                                                                        \
  } while (0)

__device__ __forceinline__ float apply_act(float v, int act, float alpha) {
  switch (act) {
    case VP_ACT_RELU: return fmaxf(v, 0.f);
    case VP_ACT_LRELU: return fmaxf(alpha * v, v);
    case VP_ACT_SIGMOID: return 1.f / (1.f + __expf(-v));
    case VP_ACT_TANH: return tanhf(v);
    default: return v;
  }
}

// ------------------------------------------------------------------------------------------------
// forward / dgrad kernel.  A CTA owns one (BN-column tile, phase, k-split) and walks the 128-pixel tiles
// m = blockIdx.x, blockIdx.x + gridDim.x, ... (persistent): the TMA ring keeps streaming across tiles and the two TMEM
// accumulators alternate, so the epilogue of tile i overlaps the MMAs of tile i+1 and barriers / TMEM are set up once.
// ------------------------------------------------------------------------------------------------
template <int KSUB, bool DBG>
__global__ void __launch_bounds__(224, KSUB == 1 ? 2 : 1) igemm_fwd_kernel(const __grid_constant__ IgemmArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[kMaxStagesFwd], empty_bar[kMaxStagesFwd], tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t sub_bytes = 16384u + static_cast<uint32_t>(a.bn_tile) * 128u;
  const uint32_t stage_bytes = sub_bytes * static_cast<uint32_t>(KSUB);
  const int num_mtiles = a.tiles_w * a.tiles_h * a.tiles_d * a.tiles_n;
  const int n0 = blockIdx.y * a.bn_tile;
  const int phase = blockIdx.z / a.splits, split = blockIdx.z % a.splits;
  const int tb = a.phase_begin[phase], te = a.phase_begin[phase + 1];
  const int total = (te - tb) * a.kc;
  const int it0 = static_cast<int>(static_cast<long long>(total) * split / a.splits);
  const int it1 = static_cast<int>(static_cast<long long>(total) * (split + 1) / a.splits);
  if (it1 <= it0) return;
  if (threadIdx.x == 0) {
    VP_TRACE(0);
    if (DBG && a.dbg_trace) { unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); g_trace[(blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z)) % 2048 * 16 + 7] = smid; }
  }

  if (threadIdx.x == 0) {
    for (int i = 0; i < a.stages; ++i) { mbar_init(&full_bar[i], 2); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full_bar[i], 1); mbar_init(&tmem_empty_bar[i], 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, a.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  // ---- Issue loops.  Each runs in ONE elected thread and is a serial latency chain (~5 cycles per instruction), while
  // a stage of four N<=128 MMAs covers only 256 tensor-pipe cycles: the loops are kept to a few dozen instructions
  // (no divisions, byte offsets carried instead of indices, slow paths out of line, debug code compiled out), the
  // activation and weight streams have their own issuers, and narrow tiles carry KSUB = 2 k-chunks per stage.
  const uint32_t full0 = opaque_u32(smem_u32(&full_bar[0])), empty0 = opaque_u32(smem_u32(&empty_bar[0]));
  const uint32_t ring_end = static_cast<uint32_t>(a.stages) * 8u;
  if (warp == 0) {
    // activation boxes: one 5-D TMA per k-chunk; the tap is a coordinate shift, padding is the OOB zero fill
    if (elect_one_sync() && !(DBG && (a.dbg_skip & 8))) {
      const bool load = !(DBG && (a.dbg_skip & 1));
      const uint32_t smem0 = opaque_u32(smem_u32(smem));
      uint32_t s_off = 0, b_off = 0, ph = 0;
      const int tap0 = it0 / a.kc, c00 = (it0 - tap0 * a.kc) * 32, c0_end = a.kc * 32;
#pragma unroll 1
      for (int mtile = blockIdx.x; mtile < num_mtiles; mtile += gridDim.x) {
        int mt = mtile;
        const int tw = mt % a.tiles_w; mt /= a.tiles_w;
        const int th = mt % a.tiles_h; mt /= a.tiles_h;
        const int td = mt % a.tiles_d;
        const int tn = mt / a.tiles_d;
        const int x0 = tw * a.bw, y0 = th * a.bh, d0 = td * a.bd, s0 = tn * a.bn;
        int tap = tb + tap0, c0 = c00;
        Tap tp = a.taps[tap];
        int c1 = x0 + tp.cw, c2 = y0 + tp.ch, c3 = d0 + tp.cd;
        const CUtensorMap* map = &a.amap[tp.map];
#pragma unroll 1
        for (int it = it0; it < it1; it += KSUB) {
          if (a.dbg_poll) mbar_poll_addr(empty0 + b_off, ph ^ 1); else mbar_wait_addr(empty0 + b_off, ph ^ 1);
          const uint32_t fb = full0 + b_off;
          const bool two = KSUB == 2 && it + 1 < it1;
          if (load) mbar_expect_tx_addr(fb, two ? 32768u : 16384u);
          else mbar_arrive_addr(fb);
#pragma unroll
          for (int j = 0; j < KSUB; ++j) {
            if (j == 0 || two) {
              if (load) tma_load_5d_addr(smem0 + s_off + j * sub_bytes, map, fb, c0, c1, c2, c3, s0);
              c0 += 32;
              if (c0 == c0_end) {
                c0 = 0; ++tap;
                tp = a.taps[tap < te ? tap : tb];
                c1 = x0 + tp.cw; c2 = y0 + tp.ch; c3 = d0 + tp.cd;
                map = &a.amap[tp.map];
              }
            }
          }
          s_off += stage_bytes; b_off += 8;
          if (b_off == ring_end) { s_off = 0; b_off = 0; ph ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 6) {
    // weight tiles: one 2-D TMA per k-chunk (rows = tap slot * n_pad + n0)
    if (elect_one_sync() && !(DBG && (a.dbg_skip & 8))) {
      const bool load = !(DBG && (a.dbg_skip & 2));
      const uint32_t smem0 = opaque_u32(smem_u32(smem) + 16384u);
      const uint32_t b_bytes = sub_bytes - 16384u;
      uint32_t s_off = 0, b_off = 0, ph = 0;
      const int tap0 = it0 / a.kc, c00 = (it0 - tap0 * a.kc) * 32, c0_end = a.kc * 32;
#pragma unroll 1
      for (int mtile = blockIdx.x; mtile < num_mtiles; mtile += gridDim.x) {
        int tap = tb + tap0, c0 = c00;
        int c1 = a.taps[tap].wslot * a.n_pad + n0;
#pragma unroll 1
        for (int it = it0; it < it1; it += KSUB) {
          if (a.dbg_poll) mbar_poll_addr(empty0 + b_off, ph ^ 1); else mbar_wait_addr(empty0 + b_off, ph ^ 1);
          const uint32_t fb = full0 + b_off;
          const bool two = KSUB == 2 && it + 1 < it1;
          if (load) mbar_expect_tx_addr(fb, two ? 2 * b_bytes : b_bytes);
          else mbar_arrive_addr(fb);
#pragma unroll
          for (int j = 0; j < KSUB; ++j) {
            if (j == 0 || two) {
              if (load) tma_load_2d_addr(smem0 + s_off + j * sub_bytes, &a.bmap, fb, c0, c1);
              c0 += 32;
              if (c0 == c0_end) { c0 = 0; ++tap; c1 = a.taps[tap < te ? tap : tb].wslot * a.n_pad + n0; }
            }
          }
          s_off += stage_bytes; b_off += 8;
          if (b_off == ring_end) { s_off = 0; b_off = 0; ph ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one_sync()) {
      const uint32_t idesc = make_idesc_tf32(128, a.bn_tile, 0, 0);
      const uint64_t ad_base = make_smem_desc(smem_u32(smem), 16, 1024, 0);
      const uint32_t stage_adv = stage_bytes >> 4, sub_adv = sub_bytes >> 4;
      const bool ring = !(DBG && (a.dbg_skip & 8));
      const int kq_last = a.kc - 1;
      uint32_t b_off = 0, ph = 0;
      int ti = 0;
      uint64_t ad = ad_base;
      long long trace_c0 = 0;
#pragma unroll 1
      for (int mtile = blockIdx.x; mtile < num_mtiles; mtile += gridDim.x, ++ti) {
        const int acc = ti & 1, use = ti >> 1;
        if (!(DBG && (a.dbg_skip & 4))) mbar_wait(&tmem_empty_bar[acc], (use & 1) ^ 1);   // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * a.bn_tile;
        uint32_t accum = 0;
        int kq = it0 % a.kc;
#pragma unroll 1
        for (int it = it0; it < it1; it += KSUB) {
          if (ring) { if (a.dbg_poll) mbar_poll_addr(full0 + b_off, ph); else mbar_wait_addr(full0 + b_off, ph); }
          tc_fence_after();
          if (DBG && it == it0 && ti == 0) { VP_TRACE(2); trace_c0 = clock64(); }
          // the last k-chunk of a tap may hold fewer than 32 real channels (e.g. 72 = 32 + 32 + 8): the zero-filled
          // K = 8 slices are not multiplied at all
          const uint64_t bd = ad + (16384u >> 4);
          const int nk = kq == kq_last ? a.k_tail : 4;
          umma_tf32(d_tmem, ad, bd, idesc, accum);
          if (nk > 1) umma_tf32(d_tmem, ad + 2, bd + 2, idesc, 1u);
          if (nk > 2) umma_tf32(d_tmem, ad + 4, bd + 4, idesc, 1u);
          if (nk > 3) umma_tf32(d_tmem, ad + 6, bd + 6, idesc, 1u);
          kq = kq == kq_last ? 0 : kq + 1;
          if (KSUB == 2 && it + 1 < it1) {
            const uint64_t ad2 = ad + sub_adv, bd2 = bd + sub_adv;
            const int nk2 = kq == kq_last ? a.k_tail : 4;
            umma_tf32(d_tmem, ad2, bd2, idesc, 1u);
            if (nk2 > 1) umma_tf32(d_tmem, ad2 + 2, bd2 + 2, idesc, 1u);
            if (nk2 > 2) umma_tf32(d_tmem, ad2 + 4, bd2 + 4, idesc, 1u);
            if (nk2 > 3) umma_tf32(d_tmem, ad2 + 6, bd2 + 6, idesc, 1u);
            kq = kq == kq_last ? 0 : kq + 1;
          }
          if (ring) umma_commit_addr(empty0 + b_off);
          accum = 1u;
          ad += stage_adv; b_off += 8;
          if (b_off == ring_end) { b_off = 0; ph ^= 1; ad = ad_base; }
        }
        umma_commit(&tmem_full_bar[acc]);
        if (DBG) {
          VP_TRACE(3);
          if (a.dbg_trace) g_trace[(blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z)) % 2048 * 16 + 1] = clock64() - trace_c0;
        }
      }
    }
    __syncwarp();
  } else if (warp < 6) {
    // ---- epilogue: warp w owns TMEM lanes 32*(w%4)..+31, thread <-> one output pixel
    const int q = warp & 3;
    const int row = q * 32 + lane;
    int r = row;
    const int lw = r % a.bw; r /= a.bw;
    const int lh = r % a.bh; r /= a.bh;
    const int ld = r % a.bd;
    const int ln = r / a.bd;
    const bool add_bias = (a.bias != nullptr) && (split == 0);
    int ti = 0;
    for (int mtile = blockIdx.x; mtile < num_mtiles && !(DBG && (a.dbg_skip & 4)); mtile += gridDim.x, ++ti) {
      int mt = mtile;
      const int tw = mt % a.tiles_w; mt /= a.tiles_w;
      const int th = mt % a.tiles_h; mt /= a.tiles_h;
      const int td = mt % a.tiles_d;
      const int tn = mt / a.tiles_d;
      const int ow = (tw * a.bw + lw) * a.os_w + a.phase_ooff[phase][2];
      const int oh = (th * a.bh + lh) * a.os_h + a.phase_ooff[phase][1];
      const int od = (td * a.bd + ld) * a.os_d + a.phase_ooff[phase][0];
      const int on = tn * a.bn + ln;
      const bool rvalid = (ow < a.out_w) && (oh < a.out_h) && (od < a.out_d) && (on < a.out_n);
      const long long ooff = on * a.so_n + od * a.so_d + oh * a.so_h + ow * a.so_w;
      float* orow = a.out + ooff;
      const int acc = ti & 1, use = ti >> 1;
      mbar_wait(&tmem_full_bar[acc], use & 1);
      tc_fence_after();
      if (threadIdx.x == 64) VP_TRACE(4);
      const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * a.bn_tile;
      for (int c0 = 0; c0 < a.bn_tile; c0 += 16) {
        float v[16];
        __syncwarp();
        tmem_ld16(t_acc + c0, v);
        const int col0 = n0 + c0;
        if (rvalid && col0 < a.out_c) {
          if (a.accumulate == 2) {      // last pass of a multi-pass accumulation: the partial sum is added BEFORE bias / activation
#pragma unroll
            for (int j = 0; j < 16; ++j) if (col0 + j < a.out_c) v[j] += orow[col0 + j];
          }
          if (add_bias) {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (col0 + j < a.out_c) v[j] += __ldg(a.bias + col0 + j);
          }
          if (a.splits > 1) {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (col0 + j < a.out_c) atomicAdd(orow + col0 + j, v[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = apply_act(v[j], a.act, a.alpha);
            if (a.aux_y != nullptr) {   // fused backward of the previous layer's activation: (v + add) * act'(y)
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                if (col0 + j < a.out_c) {
                  const float yv = __ldg(a.aux_y + ooff + col0 + j);
                  float t = v[j];
                  if (a.aux_add != nullptr) t += __ldg(a.aux_add + ooff + col0 + j);
                  if (a.aux_act == VP_ACT_LRELU) t = yv > 0.f ? t : a.alpha * t;
                  else if (a.aux_act == VP_ACT_RELU) t = yv > 0.f ? t : 0.f;
                  else if (a.aux_act == VP_ACT_SIGMOID) t *= yv * (1.f - yv);
                  else if (a.aux_act == VP_ACT_TANH) t *= (1.f - yv * yv);
                  v[j] = t;
                }
              }
            }
            if (col0 + 16 <= a.out_c) {
              float4* o4 = reinterpret_cast<float4*>(orow + col0);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                if (a.accumulate == 1) { const float4 e = o4[j]; o.x += e.x; o.y += e.y; o.z += e.z; o.w += e.w; }
                o4[j] = o;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (col0 + j < a.out_c) orow[col0 + j] = a.accumulate == 1 ? orow[col0 + j] + v[j] : v[j];
            }
          }
        }
      }
      // this warp is done reading the accumulator: hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
      if (threadIdx.x == 64) VP_TRACE(5);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, a.tmem_cols);
  if (threadIdx.x == 0) VP_TRACE(6);
}

// ------------------------------------------------------------------------------------------------
// HALO MODE forward / dgrad kernel.
//
// The box-mode kernel above fetches a 16 KB activation tile for every (tap, 32-channel chunk) and a weight tile for every
// 128-pixel tile: 629 MB of L2 -> SM traffic for the 27 MB lstm_h0 gate convolution, which pins it at the L2 fabric limit
// (tensor pipe 37 %).  Here a CTA owns a tile of 256 output positions = two 128-row sub-tiles (8 positions x 16 lines each)
// and the taps are grouped by (stride parity, depth shift[, line shift]): for each (group, 32-channel chunk) ONE halo tile
// (tile + filter reach, <= 512 rows of 128 B, TMA zero-fills the padding) is loaded, and every tap of the group is the same
// shared-memory tile read through a UMMA descriptor whose start address is shifted by (dy * pitch + dx) rows and whose
// 8-row-group stride (SBO) is the halo line pitch: the 128-byte swizzle is a function of the absolute shared-memory address,
// so a row-shifted start addresses the shifted window.  Only the weight tile streams per tap, and it feeds both sub-tiles
// (M = 256 per CTA).  lstm_h0: 0.46 MB of operand loads per 200 MMAs instead of 3.2 MB.
//
// Warp roles (256 threads): w0 halo producer, w6 weight producer, w1 (TMEM allocator) and w7 MMA issuers (one per sub-tile),
// w2..5 epilogue.
// ------------------------------------------------------------------------------------------------
constexpr int kHaloMaxGroups = 72;
constexpr int kHaloMaxBStages = 14;
constexpr int kHaloMaxAStages = 3;

struct HaloGroup {
  int8_t map, cd0, ch0, cw0;    // tensor map (stride parity) and the smallest shifts of the group = halo origin
  int16_t tap_begin, tap_end;
};

struct alignas(64) HaloArgs {
  CUtensorMap amap[kMaxMaps];
  CUtensorMap bmap;
  int32_t tiles_w, tiles_h, tiles_d, tiles_n;
  int32_t tile_w, bh, bd, bn;      // a tile is tile_w (8|16) positions x (bh*bd*bn = 16|32) lines
  int32_t sub_off;                 // descriptor units (16 B) between the start addresses of the two sub-tiles
  int32_t sub_lines, sub_x;        // epilogue: line / x offset of sub-tile 1
  int32_t hw;                      // halo line pitch (rows)
  uint32_t halo_bytes, halo_stride;
  int32_t a_stages, b_stages, tps;  // tps: filter taps (weight tiles) per weight-ring stage
  int32_t kc, n_pad, bn_tile, tmem_cols, dbuf, k_tail;
  int32_t num_phases, splits, stagger, dbg_skip;
  int32_t group_begin[9];
  int8_t phase_ooff[8][4];
  int32_t os_d, os_h, os_w;
  float* out;
  long long so_n, so_d, so_h, so_w;
  int32_t out_n, out_d, out_h, out_w, out_c;
  const float* bias;
  int32_t act;
  float alpha;
  int32_t accumulate;
  const float* aux_y;
  const float* aux_add;
  int32_t aux_act;
  HaloGroup groups[kHaloMaxGroups];
  uint16_t tap_aoff[kMaxTaps];     // row offset of the tap's window inside its group's halo tile
  int32_t tap_wslot[kMaxTaps];
};

template <bool DBG>
__global__ void __launch_bounds__(256, 1) igemm_halo_kernel(const __grid_constant__ HaloArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t a_full[kHaloMaxAStages], a_empty[kHaloMaxAStages], b_full[kHaloMaxBStages], b_empty[kHaloMaxBStages];
  __shared__ uint64_t tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_mtiles = a.tiles_w * a.tiles_h * a.tiles_d * a.tiles_n;
  const int n0 = blockIdx.y * a.bn_tile;
  const int phase = blockIdx.z / a.splits, split = blockIdx.z % a.splits;
  const int g_begin = a.group_begin[phase];
  const int n_items = (a.group_begin[phase + 1] - g_begin) * a.kc;       // item = (group, 32-channel chunk)
  const int it0 = static_cast<int>(static_cast<long long>(n_items) * split / a.splits);
  const int it1 = static_cast<int>(static_cast<long long>(n_items) * (split + 1) / a.splits);
  if (it1 <= it0) return;
  const uint32_t b_bytes = static_cast<uint32_t>(a.bn_tile) * 128u;
  const int trace_cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
  if (DBG && threadIdx.x == 0 && trace_cta < 2048) g_trace[trace_cta * 16 + 0] = gtimer();

  if (threadIdx.x == 0) {
    // two MMA-issuing threads (one per sub-tile, warps 1 and 7) release the operand stages and publish the accumulators
    for (int i = 0; i < a.a_stages; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 2); }
    for (int i = 0; i < a.b_stages; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 2); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full_bar[i], 2); mbar_init(&tmem_empty_bar[i], 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, a.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  if (DBG && threadIdx.x == 0 && trace_cta < 2048) g_trace[trace_cta * 16 + 1] = gtimer();
  const uint32_t smem0 = smem_u32(smem);
  const uint32_t bring0 = smem0 + static_cast<uint32_t>(a.a_stages) * a.halo_stride;
  const int g_first = g_begin + it0 / a.kc, c_first = it0 % a.kc;
  const uint32_t rot = a.stagger ? (blockIdx.x * 7u + blockIdx.y * 3u) : 0u;      // tap-order rotation of this CTA

  if (warp == 0) {
    // ---- halo tiles: one 5-D TMA box per (group, chunk)
    if (elect_one_sync()) {
      const uint32_t af0 = opaque_u32(smem_u32(&a_full[0])), ae0 = opaque_u32(smem_u32(&a_empty[0]));
      uint32_t st = 0, ph = 0;
#pragma unroll 1
      for (int mtile = blockIdx.x; mtile < num_mtiles; mtile += gridDim.x) {
        int mt = mtile;
        const int tw = mt % a.tiles_w; mt /= a.tiles_w;
        const int th = mt % a.tiles_h; mt /= a.tiles_h;
        const int td = mt % a.tiles_d;
        const int tn = mt / a.tiles_d;
        const int x0 = tw * a.tile_w, y0 = th * a.bh, d0 = td * a.bd, s0 = tn * a.bn;
        int g = g_first, c = c_first;
#pragma unroll 1
        for (int it = it0; it < it1; ++it) {
          const HaloGroup G = a.groups[g];
          mbar_wait_addr(ae0 + st * 8, ph ^ 1);
          if (DBG && (a.dbg_skip & 1)) {
            mbar_arrive_addr(af0 + st * 8);       // timing experiment: no halo loads (wrong results)
          } else {
            mbar_expect_tx_addr(af0 + st * 8, a.halo_bytes);
            tma_load_5d_addr(smem0 + st * a.halo_stride, &a.amap[G.map], af0 + st * 8, c * 32, x0 + G.cw0, y0 + G.ch0, d0 + G.cd0, s0);
          }
          if (++st == static_cast<uint32_t>(a.a_stages)) { st = 0; ph ^= 1; }
          if (++c == a.kc) { c = 0; ++g; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 6) {
    // ---- weight tiles: one 2-D TMA per (tap, chunk)
    if (elect_one_sync()) {
      const uint32_t bf0 = opaque_u32(smem_u32(&b_full[0])), be0 = opaque_u32(smem_u32(&b_empty[0]));
      uint32_t st = 0, ph = 0;
#pragma unroll 1
      for (int mtile = blockIdx.x; mtile < num_mtiles; mtile += gridDim.x) {
        int g = g_first, c = c_first;
#pragma unroll 1
        for (int it = it0; it < it1; ++it) {
          // every CTA walks the taps of a group in a rotated order: at any moment the CTAs of a wave ask the L2 for
          // DIFFERENT weight tiles instead of all for the same 16 KB
          const int t0 = a.groups[g].tap_begin, t1 = a.groups[g].tap_end;
          int t = t0 + static_cast<int>(rot % static_cast<uint32_t>(t1 - t0));
#pragma unroll 1
          for (int i = t0; i < t1; i += a.tps) {
            // a stage holds the weight tiles of `tps` consecutive taps: one barrier round trip per stage, not per tap
            const int nt = min(a.tps, t1 - i);
            mbar_wait_addr(be0 + st * 8, ph ^ 1);
            if (DBG && (a.dbg_skip & 2)) {
              mbar_arrive_addr(bf0 + st * 8);     // timing experiment: no weight loads (wrong results)
              for (int j = 0; j < nt; ++j) if (++t == t1) t = t0;
            } else {
              mbar_expect_tx_addr(bf0 + st * 8, static_cast<uint32_t>(nt) * b_bytes);
              for (int j = 0; j < nt; ++j) {
                tma_load_2d_addr(bring0 + (st * static_cast<uint32_t>(a.tps) + j) * b_bytes, &a.bmap, bf0 + st * 8, c * 32,
                                 a.tap_wslot[t] * a.n_pad + n0);
                if (++t == t1) t = t0;
              }
            }
            if (++st == static_cast<uint32_t>(a.b_stages)) { st = 0; ph ^= 1; }
          }
          if (++c == a.kc) { c = 0; ++g; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1 || warp == 7) {
    // ---- MMA issue.  One elected thread per SUB-TILE: a thread retires ~1 instruction per 4-5 cycles and a tap costs ~60
    // instructions of barrier / descriptor work, which is about the tensor-pipe time of the tap's 8 MMAs; with two issuing
    // threads (independent TMEM accumulators, so their relative order does not matter) each has twice the budget.
    if (elect_one_sync()) {
      const uint32_t sub = warp == 1 ? 0u : 1u;
      const uint32_t idesc = make_idesc_tf32(128, a.bn_tile, 0, 0);
      // A: K-major, 128B swizzle, 8-row groups at the halo line pitch; B: the usual 1024-byte groups
      const uint64_t ad_base = make_smem_desc(smem0, 16, static_cast<uint32_t>(a.hw) * 128u, 0);
      const uint64_t bd_base = make_smem_desc(bring0, 16, 1024, 0);
      const uint32_t af0 = opaque_u32(smem_u32(&a_full[0])), ae0 = opaque_u32(smem_u32(&a_empty[0]));
      const uint32_t bf0 = opaque_u32(smem_u32(&b_full[0])), be0 = opaque_u32(smem_u32(&b_empty[0]));
      const uint32_t a_adv = a.halo_stride >> 4, b_adv = b_bytes >> 4, b_stage_adv = b_adv * static_cast<uint32_t>(a.tps);
      const uint32_t sub_off = sub * static_cast<uint32_t>(a.sub_off);
      uint32_t ast = 0, aph = 0, bst = 0, bph = 0;
      int ti = 0;
      long long w_a = 0, w_b = 0, w_t = 0, t_begin = 0;     // DBG: cycles this thread waited for halo tiles / weight tiles / TMEM
      if (DBG) t_begin = clock64();
#pragma unroll 1
      for (int mtile = blockIdx.x; mtile < num_mtiles; mtile += gridDim.x, ++ti) {
        const int acc = a.dbuf ? (ti & 1) : 0, use = a.dbuf ? (ti >> 1) : ti;
        long long c0 = 0;
        if (DBG) c0 = clock64();
        mbar_wait(&tmem_empty_bar[acc], (use & 1) ^ 1);
        if (DBG) w_t += clock64() - c0;
        tc_fence_after();
        const uint32_t d0 = tmem_base + (static_cast<uint32_t>(acc * 2) + sub) * static_cast<uint32_t>(a.bn_tile);
        uint32_t accum = 0;
        int g = g_first, c = c_first;
#pragma unroll 1
        for (int it = it0; it < it1; ++it) {
          if (DBG) c0 = clock64();
          mbar_wait_addr(af0 + ast * 8, aph);
          if (DBG) w_a += clock64() - c0;
          tc_fence_after();
          const uint64_t ad_s = ad_base + ast * a_adv + sub_off;
          const int nk = (c == a.kc - 1) ? a.k_tail : 4;
          const int t0 = a.groups[g].tap_begin, t1 = a.groups[g].tap_end;
          int t = t0 + static_cast<int>(rot % static_cast<uint32_t>(t1 - t0));
#pragma unroll 1
          for (int i = t0; i < t1; i += a.tps) {
            const int nt = min(a.tps, t1 - i);
            if (DBG) c0 = clock64();
            mbar_wait_addr(bf0 + bst * 8, bph);
            if (DBG) w_b += clock64() - c0;
            tc_fence_after();
            uint64_t bd = bd_base + bst * b_stage_adv;
#pragma unroll 1
            for (int j = 0; j < nt; ++j, bd += b_adv) {
              const uint64_t ad = ad_s + static_cast<uint32_t>(a.tap_aoff[t]) * 8u;    // rows * 128 B >> 4
              umma_tf32(d0, ad, bd, idesc, accum);
              if (nk > 1) umma_tf32(d0, ad + 2, bd + 2, idesc, 1u);
              if (nk > 2) umma_tf32(d0, ad + 4, bd + 4, idesc, 1u);
              if (nk > 3) umma_tf32(d0, ad + 6, bd + 6, idesc, 1u);
              accum = 1u;
              if (++t == t1) t = t0;
            }
            umma_commit_addr(be0 + bst * 8);
            if (++bst == static_cast<uint32_t>(a.b_stages)) { bst = 0; bph ^= 1; }
          }
          umma_commit_addr(ae0 + ast * 8);
          if (++ast == static_cast<uint32_t>(a.a_stages)) { ast = 0; aph ^= 1; }
          if (++c == a.kc) { c = 0; ++g; }
        }
        umma_commit(&tmem_full_bar[acc]);
      }
      if (DBG && sub == 0) {
        const int cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        if (cta < 2048) {
          g_trace[cta * 16 + 8] = static_cast<unsigned long long>(clock64() - t_begin);
          g_trace[cta * 16 + 9] = static_cast<unsigned long long>(w_a);
          g_trace[cta * 16 + 10] = static_cast<unsigned long long>(w_b);
          g_trace[cta * 16 + 11] = static_cast<unsigned long long>(w_t);
        }
      }
    }
    __syncwarp();
  } else {
    // ---- epilogue: warp w owns TMEM lanes 32*(w%4)..+31; thread <-> one output position of each sub-tile
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int px = row & 7, line0 = row >> 3;
    const bool add_bias = (a.bias != nullptr) && (split == 0);
    int ti = 0;
    for (int mtile = blockIdx.x; mtile < num_mtiles; mtile += gridDim.x, ++ti) {
      int mt = mtile;
      const int tw = mt % a.tiles_w; mt /= a.tiles_w;
      const int th = mt % a.tiles_h; mt /= a.tiles_h;
      const int td = mt % a.tiles_d;
      const int tn = mt / a.tiles_d;
      const int acc = a.dbuf ? (ti & 1) : 0, use = a.dbuf ? (ti >> 1) : ti;
      mbar_wait(&tmem_full_bar[acc], use & 1);
      tc_fence_after();
#pragma unroll 1
      for (int sub = 0; sub < 2; ++sub) {
        int line = line0 + sub * a.sub_lines;
        const int ly = line % a.bh; line /= a.bh;
        const int ld = line % a.bd;
        const int ln = line / a.bd;
        const int ow = (tw * a.tile_w + sub * a.sub_x + px) * a.os_w + a.phase_ooff[phase][2];
        const int oh = (th * a.bh + ly) * a.os_h + a.phase_ooff[phase][1];
        const int od = (td * a.bd + ld) * a.os_d + a.phase_ooff[phase][0];
        const int on = tn * a.bn + ln;
        const bool rvalid = (ow < a.out_w) && (oh < a.out_h) && (od < a.out_d) && (on < a.out_n);
        const long long ooff = on * a.so_n + od * a.so_d + oh * a.so_h + ow * a.so_w;
        float* orow = a.out + ooff;
        const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>((acc * 2 + sub) * a.bn_tile);
        for (int c0 = 0; c0 < a.bn_tile; c0 += 16) {
          float v[16];
          __syncwarp();
          tmem_ld16(t_acc + c0, v);
          const int col0 = n0 + c0;
          if (rvalid && col0 < a.out_c) {
            if (a.accumulate == 2) {
#pragma unroll
              for (int j = 0; j < 16; ++j) if (col0 + j < a.out_c) v[j] += orow[col0 + j];
            }
            if (add_bias) {
#pragma unroll
              for (int j = 0; j < 16; ++j) if (col0 + j < a.out_c) v[j] += __ldg(a.bias + col0 + j);
            }
            if (a.splits > 1) {
              if (col0 + 16 <= a.out_c) {
#pragma unroll
                for (int j = 0; j < 16; j += 4) red_add_v4(orow + col0 + j, v[j], v[j + 1], v[j + 2], v[j + 3]);
              } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) if (col0 + j < a.out_c) atomicAdd(orow + col0 + j, v[j]);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = apply_act(v[j], a.act, a.alpha);
              if (a.aux_y != nullptr) {   // fused backward of the previous layer's activation: (v + add) * act'(y)
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                  if (col0 + j < a.out_c) {
                    const float yv = __ldg(a.aux_y + ooff + col0 + j);
                    float t = v[j];
                    if (a.aux_add != nullptr) t += __ldg(a.aux_add + ooff + col0 + j);
                    if (a.aux_act == VP_ACT_LRELU) t = yv > 0.f ? t : a.alpha * t;
                    else if (a.aux_act == VP_ACT_RELU) t = yv > 0.f ? t : 0.f;
                    else if (a.aux_act == VP_ACT_SIGMOID) t *= yv * (1.f - yv);
                    else if (a.aux_act == VP_ACT_TANH) t *= (1.f - yv * yv);
                    v[j] = t;
                  }
                }
              }
              if (col0 + 16 <= a.out_c) {
                float4* o4 = reinterpret_cast<float4*>(orow + col0);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                  if (a.accumulate == 1) { const float4 e = o4[j]; o.x += e.x; o.y += e.y; o.z += e.z; o.w += e.w; }
                  o4[j] = o;
                }
              } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  if (col0 + j < a.out_c) orow[col0 + j] = a.accumulate == 1 ? orow[col0 + j] + v[j] : v[j];
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, a.tmem_cols);
  if (DBG && threadIdx.x == 0 && trace_cta < 2048) {
    g_trace[trace_cta * 16 + 2] = gtimer();
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    g_trace[trace_cta * 16 + 7] = smid;
  }
}

// ------------------------------------------------------------------------------------------------
// wgrad kernel: one CTA = (128 dy-channels x up-to-128 x-channels) x a GROUP of filter taps x a range of
// pixel boxes.  Both operands are MN-major (channel-contiguous) 64-pixel boxes; GEMM-K = pixels.
// The un-shifted operand (dy for a conv, x for a transposed conv) is fetched ONCE per pixel box and reused
// by every tap of the group (one TMEM accumulator per tap); only sub-tiles that hold real channels are
// fetched.  This cuts the L2->smem traffic of the many-pixel / few-channel layers by 4-9x.
// ------------------------------------------------------------------------------------------------
constexpr int kWgMaxStages = 4;
__global__ void __launch_bounds__(192, 1) igemm_wgrad_kernel(const __grid_constant__ IgemmArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[kWgMaxStages], empty_bar[kWgMaxStages], tmem_full_bar;
  __shared__ uint32_t tmem_base_smem;
  constexpr uint32_t kSub = kWgPix * 128;  // bytes of one 32-channel sub-tile

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mtile = blockIdx.x % a.m_tiles, ntile = blockIdx.x / a.m_tiles;
  const int m0 = mtile * 128;                                   // dy channel (row) origin
  const int c0 = ntile * 128;                                   // x channel (col) origin
  const int nb = min(4, a.kc - ntile * 4);                      // 32-channel boxes of x in this tile
  const int na = min(4, (a.rows_valid - m0 + 31) / 32);         // 32-channel boxes of dy that hold real channels
  const int t0 = blockIdx.y * a.tap_group;
  const int nt = min(a.tap_group, a.num_taps - t0);
  const int ncols = 32 * nb;
  const int stages = a.wg_stages;
  const uint32_t stage_bytes = a.wg_stage_bytes;
  const bool a_shifted = a.rows_from_shifted != 0;
  const int n_shared = a_shifted ? nb : na, n_per = a_shifted ? na : nb;
  const int total = a.tiles_w * a.tiles_h * a.tiles_d * a.tiles_n;
  const int it0 = static_cast<int>(static_cast<long long>(total) * blockIdx.z / a.splits);
  const int it1 = static_cast<int>(static_cast<long long>(total) * (blockIdx.z + 1) / a.splits);
  if (it1 <= it0 || na <= 0) return;

  if (threadIdx.x == 0) {
    for (int i = 0; i < stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, a.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  // Issue loops: one elected thread each, no divisions, byte offsets carried instead of indices (see igemm_fwd_kernel).
  const uint32_t full0 = opaque_u32(smem_u32(&full_bar[0])), empty0 = opaque_u32(smem_u32(&empty_bar[0]));
  const uint32_t ring_end = static_cast<uint32_t>(stages) * 8u;
  const uint32_t smem0 = opaque_u32(smem_u32(smem));
  if (warp == 0) {
    if (elect_one_sync()) {
      const uint32_t tx = static_cast<uint32_t>(n_shared + nt * n_per) * kSub;
      const int sh_c0 = a_shifted ? c0 : m0, pt_c0 = a_shifted ? m0 : c0;
      int mt = it0;
      int tw = mt % a.tiles_w; mt /= a.tiles_w;
      int th = mt % a.tiles_h; mt /= a.tiles_h;
      int td = mt % a.tiles_d;
      int tn = mt / a.tiles_d;
      uint32_t s_off = 0, b_off = 0, ph = 0;
#pragma unroll 1
      for (int it = it0; it < it1; ++it) {
        const int x0 = tw * a.bw, y0 = th * a.bh, d0 = td * a.bd, s0 = tn * a.bn;
        mbar_wait_addr(empty0 + b_off, ph ^ 1);
        const uint32_t fb = full0 + b_off;
        uint32_t dst = smem0 + s_off;
        mbar_expect_tx_addr(fb, tx);
        // shared (un-shifted) operand first, then one block per tap of the shifted operand
        for (int i = 0; i < n_shared; ++i, dst += kSub) tma_load_5d_addr(dst, &a.bmap, fb, sh_c0 + 32 * i, x0, y0, d0, s0);
#pragma unroll 1
        for (int t = 0; t < nt; ++t) {
          const Tap tp = a.taps[t0 + t];
          const CUtensorMap* map = &a.amap[tp.map];
          const int cx = x0 + tp.cw, cy = y0 + tp.ch, cz = d0 + tp.cd;
          for (int i = 0; i < n_per; ++i, dst += kSub) tma_load_5d_addr(dst, map, fb, pt_c0 + 32 * i, cx, cy, cz, s0);
        }
        if (++tw == a.tiles_w) { tw = 0; if (++th == a.tiles_h) { th = 0; if (++td == a.tiles_d) { td = 0; ++tn; } } }
        s_off += stage_bytes; b_off += 8;
        if (b_off == ring_end) { s_off = 0; b_off = 0; ph ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one_sync()) {
      const uint32_t idesc = make_idesc_tf32(128, ncols, 1, 1);
      // MN-major tf32: 32-channel x 4-pixel atoms (512 B) with the 32-byte-granular 128B swizzle;
      // LBO = stride between 32-channel groups, SBO = stride between 4-pixel groups.  M = 128 always reads
      // four 32-channel groups; groups beyond `na` alias neighbouring data and only feed rows never stored.
      const uint64_t sh_base = make_smem_desc(smem0, kSub, 512, 0, 1);
      const uint32_t per_adv = static_cast<uint32_t>(n_per) * kSub >> 4, sh_adv = static_cast<uint32_t>(n_shared) * kSub >> 4;
      const uint32_t stage_adv = stage_bytes >> 4;
      const int merge = (a.dbg_poll & 2) ? 1 : max(1, 256 / ncols);      // taps per merged MMA (dbg_poll bit 1: VP_WGRAD_MERGE=0)
      const uint32_t idesc_m = make_idesc_tf32(128, min(merge, nt) * ncols, 1, 1);
      uint32_t b_off = 0, ph = 0, adv = 0, first = 1;
#pragma unroll 1
      for (int it = it0; it < it1; ++it) {
        mbar_wait_addr(full0 + b_off, ph);
        tc_fence_after();
        const uint64_t shd = sh_base + adv;
        uint64_t ptd = shd + sh_adv;
        const uint32_t accum0 = first ? 0u : 1u;
        if (!a_shifted && merge > 1) {
          // the shifted x tiles of consecutive taps are consecutive 32-channel groups in shared memory (LBO = kSub), and the
          // taps' accumulators are consecutive TMEM columns: `merge` taps run as ONE MMA with N = merge * ncols (<= 256)
          // instead of `merge` narrow ones (an N = 32 MMA costs 40 cycles, an N = 256 one 128)
#pragma unroll 1
          for (int t = 0; t < nt; t += merge, ptd += merge * per_adv) {
            const uint32_t idesc_g = (nt - t >= merge) ? idesc_m : make_idesc_tf32(128, (nt - t) * ncols, 1, 1);
            const uint32_t d_tmem = tmem_base + t * ncols;
#pragma unroll
            for (int k = 0; k < kWgPix / 8; ++k) umma_tf32(d_tmem, shd + k * 64, ptd + k * 64, idesc_g, k == 0 ? accum0 : 1u);
          }
        } else {
#pragma unroll 1
          for (int t = 0; t < nt; ++t, ptd += per_adv) {
            const uint64_t ad0 = a_shifted ? ptd : shd, bd0 = a_shifted ? shd : ptd;
            const uint32_t d_tmem = tmem_base + t * ncols;
#pragma unroll
            for (int k = 0; k < kWgPix / 8; ++k) umma_tf32(d_tmem, ad0 + k * 64, bd0 + k * 64, idesc, k == 0 ? accum0 : 1u);
          }
        }
        umma_commit_addr(empty0 + b_off);
        first = 0;
        adv += stage_adv; b_off += 8;
        if (b_off == ring_end) { b_off = 0; ph ^= 1; adv = 0; }
      }
      umma_commit(&tmem_full_bar);
    }
    __syncwarp();
  } else {
    const int q = warp & 3;
    const int row = m0 + q * 32 + lane;
    const bool rvalid = row < a.n_pad && row < a.rows_valid;
    mbar_wait(&tmem_full_bar, 0);
    tc_fence_after();
    for (int t = 0; t < nt; ++t) {
      const Tap tp = a.taps[t0 + t];
      float* orow = a.out + (static_cast<long long>(tp.wslot) * a.n_pad + row) * a.kpad + c0;
      for (int cc = 0; cc < ncols; cc += 16) {
        float v[16];
        __syncwarp();
        tmem_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + t * ncols + cc, v);
        if (rvalid) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) red_add_v4(orow + cc + j, v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, a.tmem_cols);
}


// ------------------------------------------------------------------------------------------------
// wgrad, ROW MODE (stride-1 convolutions: the ConvLSTM gates).  One CTA = (128 dy-channels x up-to-96/128
// x-channels) x ONE KERNEL ROW (all kw taps) x a range of pixel boxes.  Per 64-pixel box the CTA loads dy once and ONE
// halo tile of x (bw + kw - 1 pixels per line, left/right padding by TMA OOB fill); the kw taps of the row read the
// same halo tile through descriptor start addresses shifted by s pixels (s * 128 B inside the 128B-swizzled MN-major
// tile).  L2 -> SM traffic per MMA drops ~3.3x against the tap-group kernel and the stage needs 7 TMA loads for 40 MMAs.
// ------------------------------------------------------------------------------------------------
template <int LINES>   // lines of bw = 64 / LINES pixels per 64-pixel box
__global__ void __launch_bounds__(192, 1) igemm_wgrad_row_kernel(const __grid_constant__ IgemmArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[kWgMaxStages], empty_bar[kWgMaxStages], tmem_full_bar;
  __shared__ uint32_t tmem_base_smem;
  constexpr uint32_t kSub = kWgPix * 128;  // bytes of one 32-channel dy sub-tile

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mtile = blockIdx.x % a.m_tiles, ntile = blockIdx.x / a.m_tiles;
  const int m0 = mtile * 128;
  const int nb_tile = a.tap_group;                               // 32-channel x groups per N tile (<= 512 / (32 kw))
  const int c0 = ntile * nb_tile * 32;
  const int nb = min(nb_tile, a.kc - ntile * nb_tile);
  const int na = min(4, (a.rows_valid - m0 + 31) / 32);
  const int row = blockIdx.y;                                    // kernel row (rd * kh + rh)
  const int ncols = min(32 * nb, (a.out_c - c0 + 15) / 16 * 16);  // exact N (multiple of 16): no MMA columns for channel padding
  const int stages = a.wg_stages;
  const uint32_t stage_bytes = a.wg_stage_bytes;
  const int total = a.tiles_w * a.tiles_h * a.tiles_d * a.tiles_n;
  const int it0 = static_cast<int>(static_cast<long long>(total) * blockIdx.z / a.splits);
  const int it1 = static_cast<int>(static_cast<long long>(total) * (blockIdx.z + 1) / a.splits);
  if (it1 <= it0 || na <= 0) return;

  if (threadIdx.x == 0) {
    for (int i = 0; i < stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, a.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  const uint32_t full0 = opaque_u32(smem_u32(&full_bar[0])), empty0 = opaque_u32(smem_u32(&empty_bar[0]));
  const uint32_t ring_end = static_cast<uint32_t>(stages) * 8u;
  const uint32_t smem0 = opaque_u32(smem_u32(smem));
  const uint32_t halo_off = static_cast<uint32_t>(na) * kSub;   // x halo sub-tiles follow the dy sub-tiles

  if (warp == 0) {
    if (elect_one_sync()) {
      const Tap tp = a.taps[row * a.row_kw];                    // first tap of the row: its (cd, ch) are the row's shift
      const uint32_t tx = static_cast<uint32_t>(na) * kSub + static_cast<uint32_t>(nb) * (static_cast<uint32_t>(a.halo_w) * (kWgPix / a.bw) * 128u);
      int mt = it0;
      int tw = mt % a.tiles_w; mt /= a.tiles_w;
      int th = mt % a.tiles_h; mt /= a.tiles_h;
      int td = mt % a.tiles_d;
      int tn = mt / a.tiles_d;
      uint32_t s_off = 0, b_off = 0, ph = 0;
#pragma unroll 1
      for (int it = it0; it < it1; ++it) {
        const int x0 = tw * a.bw, y0 = th * a.bh, d0 = td * a.bd, s0 = tn * a.bn;
        mbar_wait_addr(empty0 + b_off, ph ^ 1);
        const uint32_t fb = full0 + b_off, st = smem0 + s_off;
        mbar_expect_tx_addr(fb, tx);
        for (int i = 0; i < na; ++i) tma_load_5d_addr(st + i * kSub, &a.bmap, fb, m0 + 32 * i, x0, y0, d0, s0);
        for (int i = 0; i < nb; ++i)
          tma_load_5d_addr(st + halo_off + i * a.halo_sub, &a.amap[1], fb, c0 + 32 * i, x0 - a.row_pw, y0 + tp.ch, d0 + tp.cd, s0);
        if (++tw == a.tiles_w) { tw = 0; if (++th == a.tiles_h) { th = 0; if (++td == a.tiles_d) { td = 0; ++tn; } } }
        s_off += stage_bytes; b_off += 8;
        if (b_off == ring_end) { s_off = 0; b_off = 0; ph ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one_sync()) {
      const uint32_t idesc = make_idesc_tf32(128, ncols, 1, 1);
      // MN-major tf32 (32-channel x 4-pixel atoms, 32-byte-granular 128B swizzle): LBO = stride between 32-channel
      // groups, SBO = 512 (4 pixels).  The swizzle is keyed on the absolute shared-memory address, so a start address
      // shifted by whole pixels (128 B) addresses the shifted window of the same tile.
      const uint64_t ad_base = make_smem_desc(smem0, kSub, 512, 0, 1);
      const uint64_t bd_base = make_smem_desc(smem0 + halo_off, static_cast<uint32_t>(a.halo_sub), 512, 0, 1);
      const uint32_t stage_adv = stage_bytes >> 4;
      constexpr int J = 8 / LINES;                               // K = 8 MMAs per line
      const uint32_t b_line = static_cast<uint32_t>(a.halo_w) * 128u >> 4;
      uint32_t b_off = 0, ph = 0, adv = 0, first = 1;
      // N <= 128 MMAs last <= 64 cycles and the issuing thread retires one instruction every ~5 cycles: the 8 MMAs of a
      // tap are fully unrolled, the dy descriptors (i * 1024 B) are shared by the kw taps of the stage.
#pragma unroll 1
      for (int it = it0; it < it1; ++it) {
        mbar_wait_addr(full0 + b_off, ph);
        tc_fence_after();
        const uint64_t ad_s = ad_base + adv;
        uint64_t bd_s = bd_base + adv;
        const uint32_t accum0 = first ? 0u : 1u;
#pragma unroll 1
        for (int s = 0; s < a.row_kw; ++s, bd_s += 8) {          // next tap: + 1 pixel = 128 B = 8 descriptor units
          const uint32_t d_tmem = tmem_base + s * ncols;
#pragma unroll
          for (int l = 0; l < LINES; ++l) {
            const uint64_t bd_l = bd_s + l * b_line;
#pragma unroll
            for (int j = 0; j < J; ++j)
              umma_tf32(d_tmem, ad_s + (l * J + j) * 64, bd_l + j * 64, idesc, (l == 0 && j == 0) ? accum0 : 1u);
          }
        }
        umma_commit_addr(empty0 + b_off);
        first = 0;
        adv += stage_adv; b_off += 8;
        if (b_off == ring_end) { b_off = 0; ph ^= 1; adv = 0; }
      }
      umma_commit(&tmem_full_bar);
    }
    __syncwarp();
  } else {
    const int q = warp & 3;
    const int rowi = m0 + q * 32 + lane;
    const bool rvalid = rowi < a.n_pad && rowi < a.rows_valid;
    mbar_wait(&tmem_full_bar, 0);
    tc_fence_after();
    for (int s = 0; s < a.row_kw; ++s) {
      const Tap tp = a.taps[row * a.row_kw + s];
      float* orow = a.out + (static_cast<long long>(tp.wslot) * a.n_pad + rowi) * a.kpad + c0;
      for (int cc = 0; cc < ncols; cc += 16) {
        float v[16];
        __syncwarp();
        tmem_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + s * ncols + cc, v);
        if (rvalid) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) red_add_v4(orow + cc + j, v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, a.tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int floor_pow2(int v) { int p = 1; while (p * 2 <= v) p *= 2; return p; }
static int ceil_div(int a, int b) { return (a + b - 1) / b; }
static int pos_mod(int a, int b) { int r = a % b; return r < 0 ? r + b : r; }
static int floor_div(int a, int b) { return (a - pos_mod(a, b)) / b; }

// 5-D map over the (sd,sh,sw)-strided sub-lattice with parity (qd,qh,qw) of an NDHWC view.
static int make_act_map(CUtensorMap* m, const vp_tensor* t, int qd, int qh, int qw, int sd, int sh, int sw,
                        const int box[4] /*w,h,d,n*/, bool mn_major = false) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return set_error("cuTensorMapEncodeTiled entry point not found");
  const long long cs = t->cstride;
  float* base = t->ptr + ((static_cast<long long>(qd) * t->h + qh) * t->w + qw) * cs;
  cuuint64_t dims[5] = {static_cast<cuuint64_t>(t->c), static_cast<cuuint64_t>(std::max(1, ceil_div(t->w - qw, sw))),
                        static_cast<cuuint64_t>(std::max(1, ceil_div(t->h - qh, sh))),
                        static_cast<cuuint64_t>(std::max(1, ceil_div(t->d - qd, sd))), static_cast<cuuint64_t>(t->n)};
  cuuint64_t strides[4] = {static_cast<cuuint64_t>(cs * sw * 4), static_cast<cuuint64_t>(cs * t->w * sh * 4),
                           static_cast<cuuint64_t>(cs * t->w * t->h * sd * 4),
                           static_cast<cuuint64_t>(cs * t->w * t->h * t->d * 4)};
  cuuint32_t boxd[5] = {32, static_cast<cuuint32_t>(box[0]), static_cast<cuuint32_t>(box[1]),
                        static_cast<cuuint32_t>(box[2]), static_cast<cuuint32_t>(box[3])};
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, base, dims, strides, boxd, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error("cuTensorMapEncodeTiled(activation) failed with %d", static_cast<int>(r));
  return 0;
}

static int check_tensor(const vp_tensor* t, const char* what) {
  if (!t || !t->ptr) return set_error("%s: null tensor", what);
  if ((reinterpret_cast<uintptr_t>(t->ptr) & 15) || (t->cstride & 3))
    return set_error("%s: pointer must be 16B aligned and cstride a multiple of 4", what);
  if (t->n < 1 || t->d < 1 || t->h < 1 || t->w < 1 || t->c < 1 || t->c > t->cstride)
    return set_error("%s: bad dims", what);
  return 0;
}

// Fills taps / phases / output strides of the geometry; `lat` (w,h,d,n) is divided by the stride for transposed convs.
static int build_taps(IgemmArgs& A, const vp_conv_geom* g, int lat[4]) {
  int ntaps = 0;
  const int K = g->kd * g->kh * g->kw;
  if (K > kMaxTaps) return set_error("too many filter taps (%d)", K);
  if (!g->transposed) {
    if (g->sd * g->sh * g->sw > kMaxMaps) return set_error("stride product too large");
    A.num_phases = 1;
    A.phase_begin[0] = 0;
    A.os_d = A.os_h = A.os_w = 1;
    std::memset(A.phase_ooff, 0, sizeof(A.phase_ooff));
    for (int rd = 0; rd < g->kd; ++rd)
      for (int rh = 0; rh < g->kh; ++rh)
        for (int rw = 0; rw < g->kw; ++rw) {
          Tap& t = A.taps[ntaps++];
          const int qd = pos_mod(rd - g->pd, g->sd), qh = pos_mod(rh - g->ph, g->sh), qw = pos_mod(rw - g->pw, g->sw);
          t.map = static_cast<int8_t>((qd * g->sh + qh) * g->sw + qw);
          t.cd = static_cast<int8_t>(floor_div(rd - g->pd, g->sd));
          t.ch = static_cast<int8_t>(floor_div(rh - g->ph, g->sh));
          t.cw = static_cast<int8_t>(floor_div(rw - g->pw, g->sw));
          t.wslot = (rd * g->kh + rh) * g->kw + rw;
        }
    A.phase_begin[1] = ntaps;
  } else {
    const int P = g->sd * g->sh * g->sw;
    if (P > 8) return set_error("stride product too large");
    A.num_phases = P;
    A.os_d = g->sd; A.os_h = g->sh; A.os_w = g->sw;
    int p = 0;
    for (int fd = 0; fd < g->sd; ++fd)
      for (int fh = 0; fh < g->sh; ++fh)
        for (int fw = 0; fw < g->sw; ++fw, ++p) {
          A.phase_begin[p] = ntaps;
          A.phase_ooff[p][0] = static_cast<int8_t>(fd);
          A.phase_ooff[p][1] = static_cast<int8_t>(fh);
          A.phase_ooff[p][2] = static_cast<int8_t>(fw);
          A.phase_ooff[p][3] = 0;
          const int r0d = pos_mod(fd + g->pd, g->sd), r0h = pos_mod(fh + g->ph, g->sh), r0w = pos_mod(fw + g->pw, g->sw);
          for (int rd = r0d; rd < g->kd; rd += g->sd)
            for (int rh = r0h; rh < g->kh; rh += g->sh)
              for (int rw = r0w; rw < g->kw; rw += g->sw) {
                if (ntaps >= kMaxTaps) return set_error("too many taps");
                Tap& t = A.taps[ntaps++];
                t.map = 0;
                t.cd = static_cast<int8_t>((fd + g->pd - rd) / g->sd);   // exact: (f+p-r) is a multiple of s
                t.ch = static_cast<int8_t>((fh + g->ph - rh) / g->sh);
                t.cw = static_cast<int8_t>((fw + g->pw - rw) / g->sw);
                t.wslot = (rd * g->kh + rh) * g->kw + rw;
              }
        }
    A.phase_begin[P] = ntaps;
    lat[0] = ceil_div(lat[0], g->sw); lat[1] = ceil_div(lat[1], g->sh); lat[2] = ceil_div(lat[2], g->sd);
  }
  return 0;
}

// Fills taps / phases / maps for the tap-shifted tensor `sh_t`; the iteration lattice has dims `lat`.
static int build_geometry(IgemmArgs& A, const vp_conv_geom* g, const vp_tensor* sh_t, int rows_per_tile,
                          const int lat_in[4] /*w,h,d,n*/, bool mn_major = false) {
  int lat[4] = {lat_in[0], lat_in[1], lat_in[2], lat_in[3]};
  if (build_taps(A, g, lat)) return -1;
  // box shape: product == rows_per_tile, powers of two, w fastest
  int rem = rows_per_tile;
  A.bw = std::min(floor_pow2(lat[0]), rem); rem /= A.bw;
  A.bh = std::min(floor_pow2(lat[1]), rem); rem /= A.bh;
  A.bd = std::min(floor_pow2(lat[2]), rem); rem /= A.bd;
  A.bn = rem;
  A.tiles_w = ceil_div(lat[0], A.bw); A.tiles_h = ceil_div(lat[1], A.bh);
  A.tiles_d = ceil_div(lat[2], A.bd); A.tiles_n = ceil_div(lat[3], A.bn);
  const int box[4] = {A.bw, A.bh, A.bd, A.bn};
  if (!g->transposed) {
    for (int qd = 0; qd < g->sd; ++qd)
      for (int qh = 0; qh < g->sh; ++qh)
        for (int qw = 0; qw < g->sw; ++qw) {
          int rc = make_act_map(&A.amap[(qd * g->sh + qh) * g->sw + qw], sh_t, qd, qh, qw, g->sd, g->sh, g->sw, box, mn_major);
          if (rc) return rc;
        }
  } else {
    int rc = make_act_map(&A.amap[0], sh_t, 0, 0, 0, 1, 1, 1, box, mn_major);
    if (rc) return rc;
  }
  return 0;
}

static int next_pow2_cols(int n) { int c = 32; while (c < n) c *= 2; return c; }

}  // namespace vp

using namespace vp;

static thread_local int g_engine_override = -1;
extern "C" int vp_conv_set_engine(int engine) {
  if (engine < -1 || engine > 1) return set_error("vp_conv_set_engine: engine must be -1 (default), 0 (box) or 1 (halo)");
  g_engine_override = engine;
  return 0;
}

// {kernel, splits} of the calling thread's last engine launch (vp_conv_last_launch)
static thread_local int g_last_launch[2] = {-1, 0};
static void note_launch(int kernel, int splits) { g_last_launch[0] = kernel; g_last_launch[1] = splits; }
extern "C" int vp_conv_last_launch(int* info) {
  if (!info) return set_error("vp_conv_last_launch: null argument");
  info[0] = g_last_launch[0];
  info[1] = g_last_launch[1];
  return 0;
}

// Host side of halo mode.  Returns 0 = launched, 1 = not eligible (the caller uses box mode), -1 = error.
static int conv_halo_try(const vp_tensor* in, const vp_conv_geom* g, const float* wpacked, int n_pad, int kc,
                         const vp_tensor* out, const float* bias, int act, float alpha, int split_k, int accumulate,
                         const float* aux_y, const float* aux_add, int aux_act, int mode, vp_stream_t stream) {
  static thread_local IgemmArgs T;     // scratch: taps / phases of the geometry
  static thread_local HaloArgs A;
  std::memset(&A, 0, sizeof(A));
  int lat[4] = {out->w, out->h, out->d, out->n};
  if (build_taps(T, g, lat)) return -1;
  const int ntaps_all = T.phase_begin[T.num_phases];
  if (lat[0] % 8 != 0 || ntaps_all < 2) return 1;
  // tile shape: 8 positions per line; two sub-tiles side by side (16 x 16 lines) or stacked (8 x 32 lines)
  const bool side = lat[0] % 16 == 0;
  const int tile_w = side ? 16 : 8, lines = side ? 16 : 32;
  const int bh = std::min(floor_pow2(lat[1]), lines);
  const int bd = std::min(floor_pow2(lat[2]), lines / bh);
  const int bn = lines / (bh * bd);
  // halo line pitch: the exact width by default (measured: a pitch padded to 8 rows, i.e. SBO a multiple of 1024 B, is
  // never faster and 2.4x slower on the 8x8 planes); VP_HALO_PAD8=1 pads
  const bool pad8 = getenv("VP_HALO_PAD8") && atoi(getenv("VP_HALO_PAD8")) == 1;
  // groups: taps that share a halo tile.  With a y-halo the lines of a tile must all come from one (d, n) plane.
  bool yhalo = (bd * bn == 1);
  int hw = 0, hh = 0, ngroups = 0;
  std::vector<int> order(ntaps_all);
  for (int attempt = 0; attempt < 2; ++attempt) {
    ngroups = 0; hw = 0; hh = 0;
    bool ok = true;
    int ti = 0;
    for (int p = 0; p < T.num_phases && ok; ++p) {
      A.group_begin[p] = ngroups;
      const int tb = T.phase_begin[p], te = T.phase_begin[p + 1];
      std::vector<int> idx;
      for (int t = tb; t < te; ++t) idx.push_back(t);
      auto key = [&](int t) { const Tap& x = T.taps[t]; return std::make_tuple(int(x.map), int(x.cd), yhalo ? 0 : int(x.ch)); };
      std::stable_sort(idx.begin(), idx.end(), [&](int x, int y) { return key(x) < key(y); });
      size_t i = 0;
      while (i < idx.size()) {
        size_t j = i;
        int cw0 = 127, cw1 = -128, ch0 = 127, ch1 = -128;
        while (j < idx.size() && key(idx[j]) == key(idx[i])) {
          const Tap& x = T.taps[idx[j]];
          cw0 = std::min(cw0, int(x.cw)); cw1 = std::max(cw1, int(x.cw));
          ch0 = std::min(ch0, int(x.ch)); ch1 = std::max(ch1, int(x.ch));
          ++j;
        }
        if (ngroups >= kHaloMaxGroups) { ok = false; break; }
        HaloGroup& G = A.groups[ngroups++];
        const Tap& f = T.taps[idx[i]];
        G.map = f.map; G.cd0 = f.cd; G.ch0 = static_cast<int8_t>(ch0); G.cw0 = static_cast<int8_t>(cw0);
        G.tap_begin = static_cast<int16_t>(ti);
        for (size_t k = i; k < j; ++k) order[ti++] = idx[k];
        G.tap_end = static_cast<int16_t>(ti);
        hw = std::max(hw, tile_w + cw1 - cw0);
        hh = std::max(hh, bh + ch1 - ch0);
        i = j;
      }
    }
    A.group_begin[T.num_phases] = ngroups;
    if (pad8) hw = (hw + 7) / 8 * 8;
    if (ok && hw <= 256 && hh <= 256 && hw * hh * bd * bn <= 512) break;
    if (!yhalo || attempt == 1) return 1;
    yhalo = false;                  // the 2-D halo does not fit: one group per filter row
  }
  for (int gi = 0; gi < ngroups; ++gi) {
    const HaloGroup& G = A.groups[gi];
    for (int t = G.tap_begin; t < G.tap_end; ++t) {
      const Tap& x = T.taps[order[t]];
      A.tap_aoff[t] = static_cast<uint16_t>((x.ch - G.ch0) * hw + (x.cw - G.cw0));
      A.tap_wslot[t] = x.wslot;
    }
  }
  A.tile_w = tile_w; A.bh = bh; A.bd = bd; A.bn = bn; A.hw = hw;
  A.sub_off = side ? 8 * 8 : 16 * hw * 8;
  A.sub_lines = side ? 0 : 16; A.sub_x = side ? 8 : 0;
  A.halo_bytes = static_cast<uint32_t>(hw) * hh * bd * bn * 128u;
  A.halo_stride = (A.halo_bytes + 1023u) / 1024u * 1024u;
  A.tiles_w = ceil_div(lat[0], tile_w); A.tiles_h = ceil_div(lat[1], bh);
  A.tiles_d = ceil_div(lat[2], bd); A.tiles_n = ceil_div(lat[3], bn);
  A.num_phases = T.num_phases;
  std::memcpy(A.phase_ooff, T.phase_ooff, sizeof(A.phase_ooff));
  A.os_d = T.os_d; A.os_h = T.os_h; A.os_w = T.os_w;
  // tensor maps of the halo boxes (one per stride parity)
  const int box[4] = {hw, hh, bd, bn};
  if (!g->transposed) {
    for (int qd = 0; qd < g->sd; ++qd)
      for (int qh = 0; qh < g->sh; ++qh)
        for (int qw = 0; qw < g->sw; ++qw)
          if (make_act_map(&A.amap[(qd * g->sh + qh) * g->sw + qw], in, qd, qh, qw, g->sd, g->sh, g->sw, box)) return 1;
  } else {
    if (make_act_map(&A.amap[0], in, 0, 0, 0, 1, 1, 1, box)) return 1;
  }
  A.kc = kc; A.n_pad = n_pad;
  A.k_tail = std::min(4, std::max(1, ceil_div(in->c - (kc - 1) * 32, 8)));
  if (n_pad <= 128) A.bn_tile = n_pad;
  else if (n_pad % 128 == 0) A.bn_tile = 128;
  else if (n_pad <= 256) A.bn_tile = n_pad;
  else {
    const int tiles = ceil_div(n_pad, 256);
    if (n_pad % tiles == 0 && (n_pad / tiles) % 16 == 0) A.bn_tile = n_pad / tiles;
  }
  if (const char* e = getenv("VP_HALO_BN")) { const int v = atoi(e); if (v >= 16 && v <= 256 && v % 16 == 0 && n_pad % v == 0) A.bn_tile = v; }
  if (A.bn_tile == 0) return 1;
  A.dbuf = (4 * A.bn_tile <= 512) ? 1 : 0;
  A.tmem_cols = next_pow2_cols((A.dbuf ? 4 : 2) * A.bn_tile);
  const size_t b_bytes = static_cast<size_t>(A.bn_tile) * 128;
  const size_t smem_max = 227 * 1024 - 2048;
  A.a_stages = 2;
  long long b_budget = static_cast<long long>(smem_max) - 1024 - 2LL * A.halo_stride;
  A.b_stages = static_cast<int>(std::min<long long>(kHaloMaxBStages, b_budget / static_cast<long long>(b_bytes)));
  if (const char* e = getenv("VP_HALO_BSTAGES")) { const int v = atoi(e); if (v >= 2 && v <= A.b_stages) A.b_stages = v; }
  if (const char* e = getenv("VP_HALO_SKIP")) A.dbg_skip = atoi(e);
  if (A.b_stages < 3 && !getenv("VP_HALO_BSTAGES")) return 1;
  if (b_budget - A.b_stages * static_cast<long long>(b_bytes) >= static_cast<long long>(A.halo_stride) && A.b_stages >= 6) A.a_stages = 3;
  // two taps per weight stage when at least three such stages fit: halves the barrier round trips of the issuing threads
  A.tps = A.b_stages >= 6 ? 2 : 1;
  if (const char* e = getenv("VP_HALO_TPS")) { const int v = atoi(e); if (v == 1 || (v == 2 && A.b_stages >= 4)) A.tps = v; }
  A.b_stages /= A.tps;
  // split the (group, chunk) items over CTAs when the grid would leave SMs idle
  const int m_tiles = A.tiles_w * A.tiles_h * A.tiles_d * A.tiles_n;
  const int n_tiles = n_pad / A.bn_tile;
  int min_items = 1 << 30;
  for (int p = 0; p < A.num_phases; ++p) min_items = std::min(min_items, (A.group_begin[p + 1] - A.group_begin[p]) * kc);
  if (min_items < 1) return 1;
  const long long base_ctas = 1LL * m_tiles * n_tiles * A.num_phases;
  if (split_k <= 0) {
    split_k = 1;
    const bool dense = out->c == out->cstride;
    if (dense && act == VP_ACT_NONE && !accumulate && !aux_y && base_ctas * 2 <= 148) {
      split_k = static_cast<int>(std::min<long long>(std::min(min_items, 8), 148 / base_ctas));
    }
  }
  A.splits = std::max(1, std::min(split_k, min_items));
  // rotating the tap order per CTA (to spread simultaneous requests for the same weight tile over the L2) measured no gain
  // (the kernel is issue-bound, not load-bound) and makes a sample's summation order depend on its tile: off by default
  A.stagger = getenv("VP_HALO_STAGGER") && atoi(getenv("VP_HALO_STAGGER")) == 1;
  if (A.splits > 1) {
    if (act != VP_ACT_NONE || aux_y) return 1;
    if (!accumulate) {
      if (out->c != out->cstride) return 1;
      const size_t bytes = static_cast<size_t>(out->n) * out->d * out->h * out->w * out->cstride * sizeof(float);
      if (cudaMemsetAsync(out->ptr, 0, bytes, static_cast<cudaStream_t>(stream)) != cudaSuccess)
        return set_error("vp_conv_igemm(halo): cudaMemsetAsync failed");
    }
  }
  A.aux_y = aux_y; A.aux_add = aux_add; A.aux_act = aux_act;
  A.out = out->ptr;
  A.so_w = out->cstride; A.so_h = A.so_w * out->w; A.so_d = A.so_h * out->h; A.so_n = A.so_d * out->d;
  A.out_n = out->n; A.out_d = out->d; A.out_h = out->h; A.out_w = out->w; A.out_c = out->c;
  A.bias = bias; A.act = act; A.alpha = alpha; A.accumulate = (A.splits > 1) ? 0 : accumulate;   // as in box mode
  {
    EncodeTiledFn enc = get_encode();
    if (!enc) return set_error("cuTensorMapEncodeTiled entry point not found");
    const int slots = g->kd * g->kh * g->kw;
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(std::min(kc * 32, (in->c + 3) / 4 * 4)), static_cast<cuuint64_t>(slots) * n_pad};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(kc) * 128};
    cuuint32_t wbox[2] = {32, static_cast<cuuint32_t>(A.bn_tile)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&A.bmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(wpacked), dims, strides, wbox, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error("cuTensorMapEncodeTiled(weights) failed with %d", static_cast<int>(r));
  }
  const size_t smem = static_cast<size_t>(A.a_stages) * A.halo_stride + static_cast<size_t>(A.b_stages) * A.tps * b_bytes + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(igemm_halo_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_max)) != cudaSuccess ||
        cudaFuncSetAttribute(igemm_halo_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_max)) != cudaSuccess)
      return set_error("cudaFuncSetAttribute(igemm_halo_kernel) failed: %s", cudaGetErrorString(cudaGetLastError()));
    attr_set = true;
  }
  const bool trace = getenv("VP_FWD_TRACE") != nullptr || A.dbg_skip != 0;
  const int other = n_tiles * A.num_phases * A.splits;
  const int gx = std::min(m_tiles, std::max(1, 148 / other));
  dim3 grid(gx, n_tiles, A.num_phases * A.splits);
  if (trace) {
    fprintf(stderr, "[halo] grid (%d,%d,%d) tile_w %d bh %d bd %d bn %d hw %d halo %u B x%d, B tile %zu B x%d, N tile %d, groups %d, kc %d k_tail %d splits %d\n",
            gx, n_tiles, A.num_phases * A.splits, A.tile_w, A.bh, A.bd, A.bn, A.hw, A.halo_bytes, A.a_stages, b_bytes, A.b_stages,
            A.bn_tile, ngroups, kc, A.k_tail, A.splits);
    igemm_halo_kernel<true><<<grid, 256, std::max(smem, static_cast<size_t>(120 * 1024)), static_cast<cudaStream_t>(stream)>>>(A);
  } else {
    igemm_halo_kernel<false><<<grid, 256, std::max(smem, static_cast<size_t>(120 * 1024)), static_cast<cudaStream_t>(stream)>>>(A);
  }
  (void)mode;
  note_launch(1, A.splits);
  return check_launch("igemm_halo_kernel");
}

static int conv_igemm_impl(const vp_tensor* in, const vp_conv_geom* g, const float* wpacked, int n_pad, int kc,
                           const vp_tensor* out, const float* bias, int act, float alpha, int split_k, int accumulate,
                           const float* aux_y, const float* aux_add, int aux_act, vp_stream_t stream) {
  if (check_tensor(in, "vp_conv_igemm(in)") || check_tensor(out, "vp_conv_igemm(out)")) return -1;
  if (!g || !wpacked) return set_error("vp_conv_igemm: null argument");
  if (n_pad % 16 || n_pad < 16) return set_error("vp_conv_igemm: n_pad must be a positive multiple of 16");
  if (kc < 1 || kc * 32 < in->c) return set_error("vp_conv_igemm: kc*32 must cover in->c");
  if (out->c > n_pad) return set_error("vp_conv_igemm: out->c exceeds n_pad");
  if (in->n != out->n) return set_error("vp_conv_igemm: batch mismatch");
  if (split_k > 1 && act != VP_ACT_NONE) return set_error("vp_conv_igemm: split_k needs act NONE");
  if (aux_y && split_k > 1) return set_error("vp_conv_igemm: the fused activation gradient needs split_k <= 1");
  {
    // halo mode (one activation tile per tap GROUP, M = 256 per CTA) whenever the geometry allows it; VP_HALO=0 disables,
    // vp_conv_set_engine() overrides per thread (the host layer times both engines once per geometry and keeps the faster)
    const char* e = getenv("VP_HALO");
    const int halo_mode = g_engine_override >= 0 ? g_engine_override : (e ? atoi(e) : 1);
    if (halo_mode > 0) {
      const int rc = conv_halo_try(in, g, wpacked, n_pad, kc, out, bias, act, alpha, split_k, accumulate, aux_y, aux_add, aux_act,
                                   halo_mode, stream);
      if (rc <= 0) return rc;
    }
  }
  static thread_local IgemmArgs A;  // large POD; per-thread host-side scratch (ctypes releases the GIL during calls)
  std::memset(&A, 0, sizeof(A));
  const int lat[4] = {out->w, out->h, out->d, out->n};
  if (build_geometry(A, g, in, 128, lat)) return -1;
  A.kc = kc; A.n_pad = n_pad;
  A.k_tail = std::min(4, std::max(1, ceil_div(in->c - (kc - 1) * 32, 8)));
  if (getenv("VP_FWD_NOTAIL")) A.k_tail = 4;
  // N tiling: the whole N when it fits one UMMA (<= 256); 128-wide tiles for multiples of 128 (more CTAs for the
  // small-M ConvLSTM GEMMs); otherwise the fewest equal tiles that are multiples of 16 (n_pad = tiles * bn_tile).
  if (n_pad <= 256) A.bn_tile = n_pad;
  if (n_pad >= 256 && n_pad % 128 == 0) A.bn_tile = 128;
  if (A.bn_tile == 0) {
    const int tiles = ceil_div(n_pad, 256);
    if (n_pad % tiles == 0 && (n_pad / tiles) % 16 == 0) A.bn_tile = n_pad / tiles;
  }
  if (const char* e = getenv("VP_FWD_BN")) { const int v = atoi(e); if (v >= 16 && v <= 256 && v % 16 == 0 && n_pad % v == 0) A.bn_tile = v; }
  if (A.bn_tile == 0) return set_error("vp_conv_igemm: unsupported n_pad %d", n_pad);
  A.tmem_cols = next_pow2_cols(2 * A.bn_tile);   // two accumulators (double-buffered epilogue)
  int min_iters = 1 << 30;
  for (int p = 0; p < A.num_phases; ++p) min_iters = std::min(min_iters, (A.phase_begin[p + 1] - A.phase_begin[p]) * kc);
  if (min_iters < 1) return set_error("vp_conv_igemm: a phase has no taps");
  const long long base_ctas = 1LL * A.tiles_w * A.tiles_h * A.tiles_d * A.tiles_n * (n_pad / A.bn_tile) * A.num_phases;
  if (split_k <= 0) {
    // auto: an under-filled grid with a long K loop is split over K; the partial sums are reduced with atomics into a
    // zero-filled output (only when the output view is dense so that it can be cleared here, and the epilogue is linear)
    split_k = 1;
    const bool dense = out->c == out->cstride;
    if (dense && act == VP_ACT_NONE && !accumulate && !aux_y && base_ctas <= 148 && min_iters >= 24) {
      // cost model: the persistent grid holds floor(148 / (N tiles * phases * splits)) CTAs per column of work, each CTA
      // walks ceil(m_tiles / gx) pixel tiles of 1/splits of the K loop; every extra split costs atomics + a memset
      const int m_tiles_all = A.tiles_w * A.tiles_h * A.tiles_d * A.tiles_n;
      const int cols = (n_pad / A.bn_tile) * A.num_phases;
      double best = 1e30;
      for (int sp = 1; sp <= 4 && min_iters / sp >= 12; ++sp) {
        const int gx = std::min(m_tiles_all, std::max(1, 148 / (cols * sp)));
        const double cost = static_cast<double>(ceil_div(m_tiles_all, gx)) / sp + 0.06 * (sp - 1);
        if (cost < best - 1e-9) { best = cost; split_k = sp; }
      }
      if (split_k > 1) {
        const size_t bytes = static_cast<size_t>(out->n) * out->d * out->h * out->w * out->cstride * sizeof(float);
        if (cudaMemsetAsync(out->ptr, 0, bytes, static_cast<cudaStream_t>(stream)) != cudaSuccess)
          return set_error("vp_conv_igemm: cudaMemsetAsync failed");
      }
    }
  }
  A.splits = std::max(1, std::min(split_k, min_iters));
  A.aux_y = aux_y; A.aux_add = aux_add; A.aux_act = aux_act;
  A.out = out->ptr;
  A.so_w = out->cstride; A.so_h = A.so_w * out->w; A.so_d = A.so_h * out->h; A.so_n = A.so_d * out->d;
  A.out_n = out->n; A.out_d = out->d; A.out_h = out->h; A.out_w = out->w; A.out_c = out->c;
  // split over K, the partial sums are added atomically to the output as it stands: that already accumulates (accumulate
  // 1 and 2 are the same with act NONE), and reading the prior back in every split would add it `splits` times
  A.bias = bias; A.act = act; A.alpha = alpha; A.accumulate = A.splits > 1 ? 0 : accumulate;
  if (accumulate == 1 && act != VP_ACT_NONE) return set_error("vp_conv_igemm: accumulate = 1 needs act NONE");
  // weights: 2-D [slots*n_pad rows][kc*32]
  {
    EncodeTiledFn enc = get_encode();
    if (!enc) return set_error("cuTensorMapEncodeTiled entry point not found");
    const int slots = g->kd * g->kh * g->kw;
    // logical width = the real channel count: the zero padding of the last k-chunk is OOB-filled, not fetched
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(std::min(kc * 32, (in->c + 3) / 4 * 4)), static_cast<cuuint64_t>(slots) * n_pad};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(kc) * 128};
    cuuint32_t box[2] = {32, static_cast<cuuint32_t>(A.bn_tile)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&A.bmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(wpacked), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error("cuTensorMapEncodeTiled(weights) failed with %d", static_cast<int>(r));
  }
  const long long n_ctas = static_cast<long long>(A.tiles_w) * A.tiles_h * A.tiles_d * A.tiles_n * (n_pad / A.bn_tile) * A.num_phases * A.splits;
  // Pipeline shape.  The producer / MMA issue loops are single-thread latency chains (~5 cycles per instruction), and a
  // stage of four N<=128 MMAs covers only <= 256 tensor-pipe cycles, so narrow tiles carry TWO k-chunks per stage
  // (8 MMAs, 64 KB, 3 stages); wide tiles (N > 128) keep one chunk per stage and 4 stages.
  // ... but short K loops (3x3 heads, pooled / upsampled encoder-decoder convs) are epilogue-bound: they keep one chunk per
  // stage and 3 stages (<= 97 KB) so that TWO CTAs share an SM and eight epilogue warps drain the accumulators
  const int iters_cta = min_iters / std::max(1, split_k);
  A.ksub = (A.bn_tile <= 128 && iters_cta >= kKsubMinIters) ? 2 : 1;
  A.stages = A.ksub == 2 ? 3 : ((A.bn_tile <= 128 && n_ctas > 148) ? 3 : kStagesFwd);
  if (const char* e = getenv("VP_FWD_KSUB")) { const int v = atoi(e); if (v == 1 || v == 2) { A.ksub = v; A.stages = v == 2 ? 3 : ((A.bn_tile <= 128 && n_ctas > 148) ? 3 : kStagesFwd); } }
  if (const char* e = getenv("VP_FWD_SKIP")) A.dbg_skip = atoi(e);
  if (getenv("VP_FWD_TRACE")) A.dbg_trace = 1;
  if (const char* e = getenv("VP_FWD_POLL")) A.dbg_poll = atoi(e);
  const size_t sub_bytes = 16384 + static_cast<size_t>(A.bn_tile) * 128;
  if (const char* e = getenv("VP_FWD_STAGES")) { const int v = atoi(e); if (v >= 2 && v <= kMaxStagesFwd && static_cast<size_t>(v) * A.ksub * sub_bytes + 1024 <= 226 * 1024) A.stages = v; }
  const size_t smem = static_cast<size_t>(A.stages) * A.ksub * sub_bytes + 1024;
  typedef void (*FwdKernel)(const IgemmArgs);
  static const FwdKernel kernels[4] = {igemm_fwd_kernel<1, false>, igemm_fwd_kernel<2, false>, igemm_fwd_kernel<1, true>,
                                       igemm_fwd_kernel<2, true>};
  static bool attr_set = false;
  if (!attr_set) {
    for (FwdKernel k : kernels)
      if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024) != cudaSuccess)
        return set_error("cudaFuncSetAttribute(igemm_fwd_kernel) failed: %s", cudaGetErrorString(cudaGetLastError()));
    attr_set = true;
  }
  const FwdKernel kernel = kernels[(A.ksub == 2 ? 1 : 0) + ((A.dbg_skip || A.dbg_trace) ? 2 : 0)];
  // persistent over the pixel tiles: at most ~2 CTAs per SM in total; each CTA strides through the M tiles
  const int m_tiles = A.tiles_w * A.tiles_h * A.tiles_d * A.tiles_n;
  const int other = (n_pad / A.bn_tile) * A.num_phases * A.splits;
  const int resident = (smem <= 113 * 1024 ? 2 : 1) * 148;
  int gx = std::min(m_tiles, std::max(1, resident / other));
  if (const char* e = getenv("VP_FWD_NONPERSISTENT")) { if (atoi(e)) gx = m_tiles; }
  dim3 grid(gx, n_pad / A.bn_tile, A.num_phases * A.splits);
  kernel<<<grid, 224, smem, static_cast<cudaStream_t>(stream)>>>(A);
  count_launch(1);
  note_launch(0, A.splits);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error("igemm_fwd_kernel launch failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int vp_conv_igemm(const vp_tensor* in, const vp_conv_geom* g, const float* wpacked, int n_pad, int kc,
                             const vp_tensor* out, const float* bias, int act, float alpha, int split_k,
                             int accumulate, vp_stream_t stream) {
  return conv_igemm_impl(in, g, wpacked, n_pad, kc, out, bias, act, alpha, split_k, accumulate, nullptr, nullptr, 0, stream);
}

extern "C" int vp_conv_igemm_actgrad(const vp_tensor* in, const vp_conv_geom* g, const float* wpacked, int n_pad, int kc,
                                     const vp_tensor* out, const float* act_output, const float* addend, int act,
                                     float alpha, int accumulate, vp_stream_t stream) {
  if (!act_output) return set_error("vp_conv_igemm_actgrad: act_output is required");
  if (out->c != out->cstride) return set_error("vp_conv_igemm_actgrad: dense output required");
  if (accumulate != 0 && accumulate != 2) return set_error("vp_conv_igemm_actgrad: accumulate must be 0 or 2");
  return conv_igemm_impl(in, g, wpacked, n_pad, kc, out, nullptr, VP_ACT_NONE, alpha, 1, accumulate, act_output, addend, act, stream);
}

extern "C" int vp_conv_wgrad(const vp_tensor* x, const vp_tensor* dy, const vp_conv_geom* g, float* dwpacked,
                             int n_pad, int kc, int split_k, vp_stream_t stream) {
  if (check_tensor(x, "vp_conv_wgrad(x)") || check_tensor(dy, "vp_conv_wgrad(dy)")) return -1;
  if (!g || !dwpacked) return set_error("vp_conv_wgrad: null argument");
  if (n_pad % 16 || dy->c > n_pad || kc * 32 < x->c) return set_error("vp_conv_wgrad: bad n_pad / kc");
  static thread_local IgemmArgs A;
  std::memset(&A, 0, sizeof(A));
  // conv:  dW[r] += sum_o dy[o]^T x[s*o+r-p]   (x shifted, lattice = dy)
  // tconv: dW[r] += sum_o dy[s*o+r-p]^T x[o]   (dy shifted, lattice = x); as a gather this is a
  //        plain (non-transposed) strided access pattern, so build the geometry with transposed=0.
  vp_conv_geom gg = *g;
  gg.transposed = 0;
  const vp_tensor* shifted = g->transposed ? dy : x;
  const vp_tensor* plain = g->transposed ? x : dy;
  const int lat[4] = {plain->w, plain->h, plain->d, plain->n};
  if (build_geometry(A, &gg, shifted, kWgPix, lat, true)) return -1;
  const int box[4] = {A.bw, A.bh, A.bd, A.bn};
  if (make_act_map(&A.bmap, plain, 0, 0, 0, 1, 1, 1, box, true)) return -1;
  A.rows_from_shifted = g->transposed ? 1 : 0;
  A.kc = kc; A.n_pad = n_pad; A.kpad = kc * 32;
  A.rows_valid = dy->c;
  A.m_tiles = ceil_div(std::min(n_pad, ceil_div(dy->c, 32) * 32), 128);
  A.n_tiles = ceil_div(kc, 4);
  A.num_taps = A.phase_begin[1];
  // Row mode: stride-1, non-transposed convolutions with a box line that is a whole number of K = 8 MMAs.
  {
    const bool unit = g->sd == 1 && g->sh == 1 && g->sw == 1 && !g->transposed;
    const char* env = getenv("VP_WGRAD_ROW");
    const bool enabled = !(env && atoi(env) == 0);
    // (kc == 4 with kw = 5 would need two 64-column N tiles that re-read dy; the tap-group kernel is faster there)
    const bool narrow_tiles = kc > 512 / (32 * g->kw) && kc % ceil_div(kc, 512 / (32 * g->kw)) == 0 && kc / ceil_div(kc, 512 / (32 * g->kw)) < 3;
    static const int min_kw = getenv("VP_WGRAD_ROW_MINKW") ? atoi(getenv("VP_WGRAD_ROW_MINKW")) : 4;
    if (enabled && unit && g->kw >= min_kw && g->kw <= 8 && A.bw % 8 == 0 && g->kw * 32 <= 512 && !narrow_tiles) {
      const int halo_w = A.bw + g->kw - 1;
      const int lines = kWgPix / A.bw;
      const int hbox[4] = {halo_w, A.bh, A.bd, A.bn};
      if (halo_w <= 256 && make_act_map(&A.amap[1], x, 0, 0, 0, 1, 1, 1, hbox, true) == 0) {
        A.halo_w = halo_w; A.row_kw = g->kw; A.row_pw = g->pw;
        A.halo_sub = (halo_w * lines * 128 + 1023) / 1024 * 1024;
        const int nb_max = std::min(std::min(4, kc), 512 / (32 * g->kw));
        A.n_tiles = ceil_div(kc, nb_max);
        const int nb_tile = ceil_div(kc, A.n_tiles);  // balanced N tiles (kc = 4 -> 2 + 2, kc = 5 -> 3 + 2)
        A.tap_group = nb_tile;                       // reused: 32-channel x groups per N tile
        A.out_c = x->c;
        A.tmem_cols = next_pow2_cols(g->kw * 32 * nb_tile);
        const int na_max = std::min(4, ceil_div(dy->c, 32));
        A.wg_stage_bytes = static_cast<uint32_t>(na_max) * kWgPix * 128 + static_cast<uint32_t>(nb_tile) * A.halo_sub;
        A.wg_stages = std::max(2, std::min(kWgMaxStages, static_cast<int>((198u * 1024u) / A.wg_stage_bytes)));
        const int groups = g->kd * g->kh;
        const int total = A.tiles_w * A.tiles_h * A.tiles_d * A.tiles_n;
        const int ctas = A.m_tiles * A.n_tiles * groups;
        int sk = split_k;
        if (sk <= 0) sk = std::max(1, (2 * 148) / ctas);   // at most two full waves of one-CTA-per-SM (never a third partial wave)
        A.splits = std::max(1, std::min(sk, std::max(1, total / 4)));
        A.out = dwpacked;
        static bool row_attr_set = false;
        const size_t smem_max = 227 * 1024 - 2048;
        typedef void (*RowKernel)(const IgemmArgs);
        static const RowKernel row_kernels[4] = {igemm_wgrad_row_kernel<1>, igemm_wgrad_row_kernel<2>, igemm_wgrad_row_kernel<4>,
                                                 igemm_wgrad_row_kernel<8>};
        if (!row_attr_set) {
          for (RowKernel k : row_kernels)
            if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_max)) != cudaSuccess)
              return set_error("cudaFuncSetAttribute(igemm_wgrad_row_kernel) failed: %s", cudaGetErrorString(cudaGetLastError()));
          row_attr_set = true;
        }
        const RowKernel row_kernel = row_kernels[lines == 1 ? 0 : lines == 2 ? 1 : lines == 4 ? 2 : 3];
        // + 24 KB: M = 128 always reads four dy groups; groups beyond `na` alias the following bytes (rows never stored)
        const size_t smem = static_cast<size_t>(A.wg_stages) * A.wg_stage_bytes + 3 * kWgPix * 128 + 2048;
        if (smem <= smem_max) {
          dim3 grid(A.m_tiles * A.n_tiles, groups, A.splits);
          row_kernel<<<grid, 192, smem, static_cast<cudaStream_t>(stream)>>>(A);
          count_launch(1);
          note_launch(3, A.splits);
          cudaError_t e = cudaGetLastError();
          if (e != cudaSuccess) return set_error("igemm_wgrad_row_kernel launch failed: %s", cudaGetErrorString(e));
          return 0;
        }
      }
    }
  }
  // tap group: bounded by TMEM columns (one accumulator per tap) and by the per-stage shared-memory budget
  const int nb_max = std::min(4, kc), na_max = std::min(4, ceil_div(dy->c, 32));
  const int n_shared = A.rows_from_shifted ? nb_max : na_max, n_per = A.rows_from_shifted ? na_max : nb_max;
  int tg = std::min(512 / (32 * nb_max), (12 - n_shared) / n_per);
  tg = std::max(1, std::min(tg, A.num_taps));
  const int groups = ceil_div(A.num_taps, tg);
  tg = ceil_div(A.num_taps, groups);     // balance the groups
  A.tap_group = tg;
  if (const char* e = getenv("VP_WGRAD_MERGE")) { if (atoi(e) == 0) A.dbg_poll |= 2; }
  A.tmem_cols = next_pow2_cols(tg * 32 * nb_max);
  A.wg_stage_bytes = static_cast<uint32_t>(n_shared + tg * n_per) * kWgPix * 128;
  A.wg_stages = std::max(2, std::min(kWgMaxStages, static_cast<int>((200u * 1024u) / A.wg_stage_bytes)));
  const int total = A.tiles_w * A.tiles_h * A.tiles_d * A.tiles_n;
  const int ctas = A.m_tiles * A.n_tiles * groups;
  if (split_k <= 0) split_k = std::max(1, (2 * 148) / ctas);  // auto: at most two full waves (never a third partial wave)
  A.splits = std::max(1, std::min(split_k, std::max(1, total / 4)));
  A.out = dwpacked;
  static bool attr_set = false;
  const size_t smem_max = 227 * 1024 - 2048;
  if (!attr_set) {
    if (cudaFuncSetAttribute(igemm_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_max)) != cudaSuccess)
      return set_error("cudaFuncSetAttribute(igemm_wgrad_kernel) failed: %s", cudaGetErrorString(cudaGetLastError()));
    attr_set = true;
  }
  const size_t smem = static_cast<size_t>(A.wg_stages) * A.wg_stage_bytes + 3 * kWgPix * 128 + 1024;
  if (smem > smem_max) return set_error("vp_conv_wgrad: shared memory budget exceeded (%zu)", smem);
  dim3 grid(A.m_tiles * A.n_tiles, groups, A.splits);
  igemm_wgrad_kernel<<<grid, 192, smem, static_cast<cudaStream_t>(stream)>>>(A);
  count_launch(1);
  note_launch(2, A.splits);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error("igemm_wgrad_kernel launch failed: %s", cudaGetErrorString(e));
  return 0;
}

// Debug: copy the per-CTA timeline of the last traced forward launch (VP_FWD_TRACE=1) to host memory (n entries of 8).
extern "C" int vp_debug_read_trace(unsigned long long* host, int n_ctas) {
  if (n_ctas > 2048) n_ctas = 2048;
  if (cudaMemcpyFromSymbol(host, vp::g_trace, static_cast<size_t>(n_ctas) * 16 * sizeof(unsigned long long)) != cudaSuccess)
    return set_error("vp_debug_read_trace failed: %s", cudaGetErrorString(cudaGetLastError()));
  return 0;
}
