// Weight-gradient GEMM for sm_100a:   dW[cout, tap, cin] = sum_pixels dY[pixel, cout] * X_tap[pixel (+tap offset), cin]
//
// The reduction runs over pixels, so both operands are "MN-major" for the tensor core: a TMA box of 64 pixels x 64 channels
// (64 rows of 128 B, 128B swizzle) is exactly one canonical MN-major SWIZZLE_128B atom column (K = pixel rows). The same
// NHWC activation tensors and the same tap/phase tensor maps as the forward kernel are used - no transposes, no im2col.
// The pixel range is split across CTAs (split-K); each CTA writes its fp32 partial tile to a workspace which
// wgrad_reduce_rows_kernel sums deterministically (no atomics) into the OIHW gradient.
//
// 64-channel inputs with several taps (ResNet layer1 3x3, the space-to-depth stem) run in MERGED-TAP mode: the 64-column
// atoms of one B tile belong to DIFFERENT taps (same pixels, shifted TMA coordinates), so one dY tile feeds an N = 192 / 256
// MMA instead of one N = 64 MMA per tap (tcgen05.mma costs ~100 cycles however small N is).
//
// Replaces the cuDNN backward-filter / cuBLAS calls autograd issues for nn.Conv2d / nn.Linear in the reference
// (loss.backward(): classification/resnet/utils.py:43).
#pragma once
#include "common.cuh"
#include "conv_gemm.cuh"
#include "conv1x1_stream.cuh"   // lds128

namespace b200 {

struct alignas(64) WgradParams {
  CUtensorMap dy_map;     // 4-D (Cout, d1, d2, d3), box (64, b1, b2, b3), b1*b2*b3 = 64 pixels
  CUtensorMap x_maps[4];  // 4-D (Cin, ...), same box
  int num_taps;     // taps that are separate work items (1 in merged-tap mode)
  int merge_atoms;  // merged-tap mode: 64-channel atoms per tap (Cin / 64); 0 = one tap per work item
  int n_cols;       // valid columns of one partial row segment: Cin, or taps * Cin in merged-tap mode
  int Cout, Cin;
  int mg_tiles, ng_tiles;
  int tiles1, tiles2, tiles3;
  int box1, box2, box3;
  int splits, kb_per_split, kb_total;
  long long ld_partial;  // taps * Cin (row pitch of the partial matrix, in floats)
  int8_t tap_map[kMaxTaps];
  int8_t tap_o1[kMaxTaps];
  int8_t tap_o2[kMaxTaps];
  float* partial;  // [splits][Cout][taps*Cin]
  uint32_t desc_lbo, desc_sbo, desc_kstep;  // MN-major smem descriptor strides (bytes): 8192 / 1024 / 2048
  // kBias kernels: per-split column sums of dY (= the bias gradient of the layer), [splits][2][Cout] (plane 0 = sums,
  // plane 1 = 0: the layout b200_bn_bwd_finalize folds).  The dY tiles are already in shared memory for the tensor core:
  // four extra warps add up their rows, so the bias gradient costs no pass over dY (it used to be a separate HBM pass).
  float* bias_partial;
};

template <int BLOCK_NG>
struct WgradCfg {
  static constexpr int BLOCK_K = 64;                       // pixels per stage
  static constexpr int A_BYTES = 2 * 64 * 128;             // two 64-channel atoms of dY
  static constexpr int B_BYTES = (BLOCK_NG / 64) * 64 * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BLOCK_NG == 256) ? 4 : (BLOCK_NG == 192 ? 5 : (BLOCK_NG == 128 ? 6 : 8));
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BAR_BYTES + 1024;
  static constexpr int TMEM_COLS = (2 * BLOCK_NG <= 128) ? 128 : (2 * BLOCK_NG <= 256 ? 256 : 512);
};

template <int BLOCK_NG, bool kBias = false>
__global__ void __launch_bounds__(kBias ? 320 : 192, 1) wgrad_gemm_kernel(const __grid_constant__ WgradParams p) {
  pdl_launch_dependents();
  using Cfg = WgradCfg<BLOCK_NG>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // work item = (split, mg, ng, tap); tap fastest so CTAs sharing the same pixels run together (L2 reuse)
  const int items_per_split = p.mg_tiles * p.ng_tiles * p.num_taps;
  const int num_items = items_per_split * p.splits;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&p.dy_map);
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.x_maps[i]);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], kBias ? 5 : 1);   // the MMA commit (+ the four column-sum warps, on every stage)
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 4);
    }
    fence_mbar_init();
  }
  if (warp_idx == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();   // everything above touched only this CTA's shared memory / TMEM and the kernel parameters

  if (warp_idx == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        const int split = item / items_per_split;
        int r = item - split * items_per_split;
        const int tap = r % p.num_taps;
        r /= p.num_taps;
        const int ng = r % p.ng_tiles;
        const int mg = r / p.ng_tiles;
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        // per 64-column atom of the B tile: tensor map, channel offset and tap shift
        const CUtensorMap* xm[BLOCK_NG / 64];
        int ch0[BLOCK_NG / 64], o1[BLOCK_NG / 64], o2[BLOCK_NG / 64];
#pragma unroll
        for (int j = 0; j < BLOCK_NG / 64; ++j) {
          int tp = tap, ca = ng * (BLOCK_NG / 64) + j;
          if (p.merge_atoms) {
            tp = ca / p.merge_atoms;
            ca -= tp * p.merge_atoms;
          }
          xm[j] = &p.x_maps[p.tap_map[tp]];
          ch0[j] = ca * 64;
          o1[j] = p.tap_o1[tp], o2[j] = p.tap_o2[tp];
        }
        for (int kb = kb0; kb < kb1; ++kb) {
          const int t1 = kb % p.tiles1;
          const int t2 = (kb / p.tiles1) % p.tiles2;
          const int t3 = kb / (p.tiles1 * p.tiles2);
          const int c1 = t1 * p.box1, c2 = t2 * p.box2, c3 = t3 * p.box3;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* a_dst = smem + stage * Cfg::STAGE_BYTES;
          uint8_t* b_dst = a_dst + Cfg::A_BYTES;
          mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
          tma_load_4d(a_dst, &p.dy_map, &full_bar[stage], mg * 128, c1, c2, c3);
          tma_load_4d(a_dst + 8192, &p.dy_map, &full_bar[stage], mg * 128 + 64, c1, c2, c3);
#pragma unroll
          for (int j = 0; j < BLOCK_NG / 64; ++j)
            tma_load_4d(b_dst + j * 8192, xm[j], &full_bar[stage], ch0[j], c1 + o1[j], c2 + o2[j], c3);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp_idx == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(128, BLOCK_NG, 1, 1);  // both operands MN-major
      // descriptors of all stages / K steps by 64-bit adds on two base descriptors (see conv_gemm.cuh)
      const uint64_t desc_a0 = make_smem_desc_sw128(smem_u32(smem), p.desc_lbo, p.desc_sbo);
      const uint64_t desc_b0 = make_smem_desc_sw128(smem_u32(smem) + Cfg::A_BYTES, p.desc_lbo, p.desc_sbo);
      const uint64_t kstep = p.desc_kstep >> 4;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        const int split = item / items_per_split;
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_NG;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          // 16 pixel rows per MMA = 2048 B; LBO = next 64-channel atom (8192 B); SBO = next 8 pixel rows (1024 B)
          const uint64_t soff = static_cast<uint64_t>(stage) * (Cfg::STAGE_BYTES >> 4);
          const uint64_t da = desc_a0 + soff, db = desc_b0 + soff;
          umma_f16(tmem_d, da, db, idesc, kb > kb0 ? 1u : 0u);
#pragma unroll
          for (int k = 1; k < 4; ++k) umma_f16(tmem_d, da + k * kstep, db + k * kstep, idesc, 1u);
          umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&tmem_full[acc]);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (kBias && warp_idx >= 6) {
    // ===================== column sums of the dY tiles (bias gradient) =====================
    // Only the (ng == 0, tap == 0) item of every (split, mg) pair is summed, but these warps wait for and release every stage
    // of every item, in order, like any other consumer of the ring: a CTA that runs several items (more items than SMs)
    // keeps its phase bookkeeping exact, and no tile is refilled before they are done with it.
    // The dY stage is 64 pixel rows x 2 atoms x 128 B: thread t of the 128 reads 8 rows of ONE 16-byte chunk (8 channels),
    // chunk cc = t % 16 (atom cc / 8, chunk cc % 8 inside the 128-byte row, XOR-swizzled by row & 7), rows (t / 16) * 8 .. + 8.
    __shared__ float bias_red[8][128];
    const int t = (warp_idx - 6) * 32 + lane;
    const int cc = t & 15, rg = t >> 4;
    const uint32_t atom_off = static_cast<uint32_t>(cc >> 3) * 8192u;
    int stage = 0;
    uint32_t phase = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      const int split = item / items_per_split;
      int r = item - split * items_per_split;
      const int tap = r % p.num_taps;
      r /= p.num_taps;
      const int ng = r % p.ng_tiles;
      const int mg = r / p.ng_tiles;
      const int kb0 = split * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      const bool summed = ng == 0 && tap == 0;
      float sum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        if (summed) {
          const uint32_t base = smem_u32(smem + stage * Cfg::STAGE_BYTES) + atom_off;
          uint4 v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int row = rg * 8 + i;
            v[i] = lds128(base + row * 128 + ((static_cast<uint32_t>(cc & 7) ^ static_cast<uint32_t>(row & 7)) << 4));
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float f[8];
            unpack8(v[i], f);
#pragma unroll
            for (int j = 0; j < 8; ++j) sum[j] += f[j];
          }
          // the sums depend on every word loaded from the tile: computing them here means the loads have returned before
          // the release below lets the producer overwrite the stage
          asm volatile("" ::"f"(sum[0]), "f"(sum[1]), "f"(sum[2]), "f"(sum[3]), "f"(sum[4]), "f"(sum[5]), "f"(sum[6]),
                       "f"(sum[7]) : "memory");
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);   // this warp is done with the tile
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (!summed) continue;
      // fold the 8 row groups (fixed order: deterministic) and write this split's partial sums
      named_bar_sync(2, 128);   // previous item's readers are done with bias_red
#pragma unroll
      for (int j = 0; j < 8; ++j) bias_red[rg][cc * 8 + j] = sum[j];
      named_bar_sync(2, 128);
      {
        float tot = 0.f;
#pragma unroll
        for (int g2 = 0; g2 < 8; ++g2) tot += bias_red[g2][t];
        const int cout = mg * 128 + t;
        if (cout < p.Cout) {
          p.bias_partial[(static_cast<long long>(split) * 2) * p.Cout + cout] = tot;
          p.bias_partial[(static_cast<long long>(split) * 2 + 1) * p.Cout + cout] = 0.f;
        }
      }
    }
  } else {
    const int q = warp_idx & 3;
    const int row = q * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      const int split = item / items_per_split;
      int r = item - split * items_per_split;
      const int tap = r % p.num_taps;
      r /= p.num_taps;
      const int ng = r % p.ng_tiles;
      const int mg = r / p.ng_tiles;
      const int cout = mg * 128 + row;
      float* out_row = p.partial + (static_cast<long long>(split) * p.Cout + cout) * p.ld_partial +
                       static_cast<long long>(tap) * p.Cin + ng * BLOCK_NG;
      // (the host guarantees every split owns at least one pixel block)
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t tmem_acc = tmem_base + acc * BLOCK_NG + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
      for (int ch = 0; ch < BLOCK_NG / 32; ++ch) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_acc + ch * 32, v);
        tmem_ld_wait();
        if (cout < p.Cout) {
          const int cin0 = ng * BLOCK_NG + ch * 32;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (cin0 + j * 4 < p.n_cols) {  // a multiple of 8
              uint4 w = make_uint4(v[j * 4], v[j * 4 + 1], v[j * 4 + 2], v[j * 4 + 3]);
              *reinterpret_cast<uint4*>(out_row + ch * 32 + j * 4) = w;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// grad[cout][cin][tap] (OIHW, fp32) (+)= sum_s partial[s][cout][tap*Cin + cin]
// Row-block reduction: one block owns `chunk` input channels of one output channel for ALL taps, i.e. a contiguous run of
// chunk * taps gradient elements. The split range is folded by `SL` thread slices with float4 loads (coalesced along cin in
// the partial layout, two independent loads in flight per thread), staged in shared memory as [slice][tap][cin] and written
// out tap-innermost, so that both the partial reads and the OIHW gradient writes are fully coalesced. Fixed summation order.
__global__ void __launch_bounds__(256) wgrad_reduce_rows_kernel(const float* __restrict__ partial, float* __restrict__ grad,
                                                                int splits, int Cout, int Cin, int taps, int chunk, int SL,
                                                                int accumulate, const float* __restrict__ rowscale,
                                                                const float* __restrict__ bias_partial,
                                                                float* __restrict__ bias_out) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float4 rows_sm4[];
  const int cout = blockIdx.x;
  // the layer's bias gradient: the per-split column sums of dY the kBias wgrad kernel left in bias_partial[splits][2][Cout],
  // folded in split order by the first block of each output channel (it used to be a launch of its own per layer)
  if (bias_out != nullptr && blockIdx.y == 0 && threadIdx.x == 0) {
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += bias_partial[static_cast<long long>(k) * 2 * Cout + cout];
    bias_out[cout] = s;
  }
  const int c0 = blockIdx.y * chunk;
  const int cw = min(chunk, Cin - c0);
  const int vpt = cw >> 2;          // float4 vectors per tap
  const int nvec = taps * vpt;
  const long long slice4 = static_cast<long long>(Cout) * taps * Cin / 4;
  const float4* row4 = reinterpret_cast<const float4*>(partial + static_cast<long long>(cout) * taps * Cin + c0);
  const int cin4 = Cin >> 2;
  for (int w = threadIdx.x; w < nvec * SL; w += blockDim.x) {
    const int sl = w / nvec;
    const int v = w - sl * nvec;
    const int tap = v / vpt;
    const int cv = v - tap * vpt;
    const float4* src = row4 + tap * cin4 + cv;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    int k = sl;
    for (; k + SL < splits; k += 2 * SL) {
      const float4 x = __ldcs(src + k * slice4);
      const float4 y = __ldcs(src + (k + SL) * slice4);
      a.x += x.x, a.y += x.y, a.z += x.z, a.w += x.w;
      b.x += y.x, b.y += y.y, b.z += y.z, b.w += y.w;
    }
    if (k < splits) {
      const float4 x = __ldcs(src + k * slice4);
      a.x += x.x, a.y += x.y, a.z += x.z, a.w += x.w;
    }
    rows_sm4[w] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
  __syncthreads();
  const float* sm = reinterpret_cast<const float*>(rows_sm4);
  const float rs = rowscale != nullptr ? __ldg(rowscale + cout) : 1.f;
  float* out = grad + (static_cast<long long>(cout) * Cin + c0) * taps;
  for (int e = threadIdx.x; e < cw * taps; e += blockDim.x) {
    const int cin = e / taps;
    const int tap = e - cin * taps;
    float s = 0.f;
    for (int sl = 0; sl < SL; ++sl) s += sm[(sl * nvec) * 4 + tap * cw + cin];
    s *= rs;
    out[e] = accumulate ? out[e] + s : s;
  }
}

// Same reduction, one thread per element walking the splits: fallback for shapes the row kernel does not take.
__global__ void wgrad_reduce_flat_kernel(const float* __restrict__ partial, float* __restrict__ grad, int splits, int Cout,
                                    int Cin, int taps, int accumulate, const float* __restrict__ rowscale,
                                    const float* __restrict__ bias_partial, float* __restrict__ bias_out) {
  pdl_launch_dependents();
  pdl_wait();
  const long long total = static_cast<long long>(Cout) * Cin * taps;
  const long long slice = total;
  if (bias_out != nullptr) {
    for (int cout = blockIdx.x * blockDim.x + threadIdx.x; cout < Cout; cout += gridDim.x * blockDim.x) {
      float s = 0.f;
      for (int k = 0; k < splits; ++k) s += bias_partial[static_cast<long long>(k) * 2 * Cout + cout];
      bias_out[cout] = s;
    }
  }
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    // i indexes the partial layout (coalesced reads): [cout][tap][cin]
    const int cin = static_cast<int>(i % Cin);
    const long long t = i / Cin;
    const int tap = static_cast<int>(t % taps);
    const int cout = static_cast<int>(t / taps);
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += partial[k * slice + i];
    if (rowscale != nullptr) s *= __ldg(rowscale + cout);
    const long long o = (static_cast<long long>(cout) * Cin + cin) * taps + tap;
    grad[o] = accumulate ? grad[o] + s : s;
  }
}


}  // namespace b200
