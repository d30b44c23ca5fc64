// Implicit-GEMM convolution on tcgen05 tensor cores (sm_100a).
//
//   D[pixel m (128 per tile), channel n (BN per tile)] = sum over taps t, channel chunks c of
//       A_t,c [128 px x 64 ch]  (TMA 4-D box of the NHWC input, shifted by the tap, zero OOB fill,
//                                SWIZZLE_128B, K-major)
//     * B_t,c [BN co x 64 ch]   (TMA 3-D box of the packed weights [tap][co][ci], K-major)
//
// Warp roles (192 threads, 1 CTA/SM, persistent over tiles):
//   warp 0      TMA producer (one elected lane issues), smem ring of `stages` {A,B} slots
//   warp 1      TMEM allocator + tcgen05.mma issuer (one elected lane), fp32 accumulators in TMEM,
//               two accumulator buffers so the epilogue of tile i overlaps the MMAs of tile i+1
//   warps 2..5  epilogue: tcgen05.ld -> alpha/bias/residual/accumulate/LeakyReLU/mask -> bf16 ->
//               128-bit stores into a channel slice of the NHWC output (zero-copy concat), optional
//               2x2 store replication (nearest upsample folded into the store).
//
// Replaces, for the reference: nn.Conv2d fwd/dgrad (block.py:238), torch.cat (RRDBNet_arch.py:152-159),
// LeakyReLU (block.py:91), x5*0.2+x (RRDBNet_arch.py:163,96), ShortcutBlock add (block.py:191),
// F.interpolate nearest (block.py:358).
#include "common.cuh"
#include "sm100_ptx.cuh"

namespace b200 {

namespace {

constexpr int kThreads = 192;
constexpr int kMaxStages = 8;
constexpr uint32_t kABytes = 128 * 128;  // 128 pixel rows x 64 bf16

struct IgemmParams {
  CUtensorMap in_map;
  CUtensorMap w_map;
  int tw, th, tn;
  int tiles_x, tiles_y, tiles_n, n_blocks, total_tiles;
  int cls_tiles;   // tiles per output-parity class (== total_tiles when the launch is a single conv)
  int Nimg, Ho, Wo;
  int aux_h, aux_w, aux_my, aux_oy, aux_mx, aux_ox;  // grid of the residual / mask tensors
  int in_stride, in_off_y, in_off_x;
  int cin_off, k_chunks, last_k16;
  int ntaps;
  int8_t tap_dy[B200_MAX_TAPS], tap_dx[B200_MAX_TAPS], tap_w[B200_MAX_TAPS];
  int BN, Cout;
  int acc_cols;  // TMEM column stride between accumulator buffers
  int acc_stages;  // 256-row kernel: 2 when 4 * acc_cols <= 512, else 1
  uint32_t a_bytes;  // bytes of one A slot (128 or 256 pixel rows x 128 B)
  int stages;
  uint32_t b_bytes;  // BN * 128 (TMA transaction bytes of one B slot)
  uint32_t stage_bytes;
  // staged epilogue of the 256-row kernel: finished 64-channel slabs go through a SW128 staging buffer and leave as
  // TMA tile stores (out_map[parity class or 2x2 replica]); 0 = per-thread 16-byte stores
  int tma_store;
  int st_bufs;                // staging buffers per 128-row half (1 or 2), 16 KB each
  uint32_t st_off;            // byte offset of the staging area behind the operand ring
  int st_dy, st_dn;           // output-tile rows / images between the two halves
  int dbg;                    // B200_IGEMM_DBG (experiments): 1 skip the epilogue's global traffic
  long long* dbg_ptr;         // B200_IGEMM_DBG_PTR (tools/igemm_timeline.py): CTA 0 stamps clock64() per k-iteration
  CUtensorMap out_map[4];
  // EPI = 3: per-(tile, half) column sums and sums of squares of the bf16-rounded outputs -- BatchNorm statistics
  // without a pass over the stored tensor.  Output-major: stat_part[(which * Cout + c) * stat_rows + 2 * pixel_tile + half]
  float* stat_part;
  int stat_rows;
  // output placement
  __nv_bfloat16* out;
  long long o_sn, o_sy, o_sx;
  int o_coff, o_my, o_oy, o_mx, o_ox, upsample;
  // epilogue
  const float* bias;
  float alpha;
  int act;
  float slope;
  const __nv_bfloat16* res1;
  const __nv_bfloat16* res2;
  int res1_c, res1_coff, res2_c, res2_coff, res_nch;
  float beta1, beta2;
  int accumulate;
  const __nv_bfloat16* mask;
  int mask_c, mask_coff, mask_lo, mask_hi;
  float mask_slope;
};

struct TileCoord {
  int nb, x0, y0, n0;
  int cls;   // output-parity class of a merged launch: taps [cls * ntaps, +ntaps), output offset + (cls >> 1, cls & 1)
};

__device__ __forceinline__ TileCoord decode_tile(const IgemmParams& p, int tile) {
  TileCoord t;
  t.cls = tile / p.cls_tiles;
  tile -= t.cls * p.cls_tiles;
  t.nb = tile % p.n_blocks;
  int r = tile / p.n_blocks;
  t.x0 = (r % p.tiles_x) * p.tw;
  r /= p.tiles_x;
  t.y0 = (r % p.tiles_y) * p.th;
  t.n0 = (r / p.tiles_y) * p.tn;
  return t;
}

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return u;
}

// Epilogue for NC (16 or 32) accumulator columns of one pixel row.
template <int NC>
__device__ __forceinline__ void epilogue_columns(const IgemmParams& p, const uint32_t* acc, int cbase,
                                                 bool valid, long long pix_lin,
                                                 __nv_bfloat16* out_px) {
  if (!valid) return;
#pragma unroll
  for (int g = 0; g < NC / 8; ++g) {
    const int c = cbase + g * 8;
    if (c >= p.Cout) break;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[g * 8 + j]);
    if (p.bias) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + c));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + c + 4));
      v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
      v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= p.alpha;
    if (c < p.res_nch) {
      if (p.res1) {
        float r[8];
        unpack8(*reinterpret_cast<const uint4*>(p.res1 + pix_lin * p.res1_c + p.res1_coff + c), r);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(p.beta1, r[j], v[j]);
      }
      if (p.res2) {
        float r[8];
        unpack8(*reinterpret_cast<const uint4*>(p.res2 + pix_lin * p.res2_c + p.res2_coff + c), r);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(p.beta2, r[j], v[j]);
      }
    }
    __nv_bfloat16* dst = out_px + p.o_coff + c;
    if (p.accumulate) {
      float r[8];
      unpack8(*reinterpret_cast<const uint4*>(dst), r);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += r[j];
    }
    if (p.act) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * p.slope;
    }
    if (p.mask && c >= p.mask_lo && c < p.mask_hi) {
      float r[8];
      unpack8(*reinterpret_cast<const uint4*>(p.mask + pix_lin * p.mask_c + p.mask_coff + c), r);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = r[j] > 0.f ? v[j] : v[j] * p.mask_slope;
    }
    const uint4 o = pack8(v);
    *reinterpret_cast<uint4*>(dst) = o;
    if (p.upsample) {
      *reinterpret_cast<uint4*>(dst + p.o_sx) = o;
      *reinterpret_cast<uint4*>(dst + p.o_sy) = o;
      *reinterpret_cast<uint4*>(dst + p.o_sy + p.o_sx) = o;
    }
  }
}

__global__ void __launch_bounds__(kThreads, 1)
conv_igemm_kernel(const __grid_constant__ IgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem =
      reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[kMaxStages], empty_bar[kMaxStages], tfull_bar[2], tempty_bar[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&tfull_bar[0], 1);
    mbar_init(&tfull_bar[1], 1);
    mbar_init(&tempty_bar[0], 4);
    mbar_init(&tempty_bar[1], 4);
    mbar_fence_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.in_map);
    tma_prefetch_desc(&p.w_map);
  }
  if (warp == 1) {
    tmem_alloc(&tmem_base_s, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  // Dependents may be scheduled from here on: this CTA already owns its TMEM columns, so a co-resident
  // CTA of the next kernel can never make it wait for an allocation (which would deadlock, because that
  // CTA in turn waits for this grid to complete).
  pdl_trigger();
  pdl_wait();   // everything above overlapped the previous kernel's tail
  const int k_iters = p.ntaps * p.k_chunks;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(p, tile);
      for (int t0 = 0; t0 < p.ntaps; ++t0) {
        const int t = tc.cls * p.ntaps + t0;
        const int cx = tc.x0 * p.in_stride + p.in_off_x + p.tap_dx[t];
        const int cy = tc.y0 * p.in_stride + p.in_off_y + p.tap_dy[t];
        const int wt = p.tap_w[t];
        for (int c = 0; c < p.k_chunks; ++c) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
            uint8_t* sa = smem + (size_t)stage * p.stage_bytes;
            mbar_expect_tx(&full_bar[stage], kABytes + p.b_bytes);
            tma_load_4d(sa, &p.in_map, &full_bar[stage], p.cin_off + c * 64, cx, cy, tc.n0);
            tma_load_3d(sa + kABytes, &p.w_map, &full_bar[stage], c * 64, tc.nb * p.BN, wt);
          }
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    const uint32_t idesc = make_idesc_bf16(128, p.BN, 0, 0);
    const uint64_t desc_hi = make_smem_desc(0, 16, 1024, LAYOUT_SW128, 0);
    const uint32_t smem_base = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem + acc * p.acc_cols;
      int c = 0;
      for (int it = 0; it < k_iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const int nk = (c == p.k_chunks - 1) ? p.last_k16 : 4;
        const uint32_t a_addr = smem_base + stage * p.stage_bytes;
        const uint32_t b_addr = a_addr + kABytes;
        if (elect_one()) {
          for (int k = 0; k < nk; ++k) {
            const uint64_t ad = desc_hi | (uint64_t)(((a_addr + k * 32) >> 4) & 0x3FFF);
            const uint64_t bd = desc_hi | (uint64_t)(((b_addr + k * 32) >> 4) & 0x3FFF);
            umma_f16(d_tmem, ad, bd, idesc, (it | k) != 0);
          }
          umma_commit(&empty_bar[stage]);
          if (it == k_iters - 1) umma_commit(&tfull_bar[acc]);
        }
        __syncwarp();
        if (++c == p.k_chunks) c = 0;
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else {
    // ------------------------------------------------------------ epilogue (warps 2..5)
    const int quad = warp & 3;  // TMEM lane quadrant accessible by this warp
    const int m = quad * 32 + lane;
    const int ix = m % p.tw;
    const int iy = (m / p.tw) % p.th;
    const int in_ = m / (p.tw * p.th);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(p, tile);
      const int x = tc.x0 + ix, y = tc.y0 + iy, n = tc.n0 + in_;
      const bool valid = (x < p.Wo) && (y < p.Ho) && (n < p.Nimg);
      // residual / mask tensors live on the output buffer's grid at the placed coordinates
      // (or on the logical grid when the store replicates 2x2)
      const int cy_ = tc.cls >> 1, cx_ = tc.cls & 1;   // parity offsets of a merged launch (0 otherwise)
      const long long pix_lin = ((long long)n * p.aux_h + (y * p.aux_my + p.aux_oy + cy_)) * p.aux_w +
                                (x * p.aux_mx + p.aux_ox + cx_);
      __nv_bfloat16* out_px = p.out + (long long)n * p.o_sn +
                              (long long)(y * p.o_my + p.o_oy + cy_) * p.o_sy +
                              (long long)(x * p.o_mx + p.o_ox + cx_) * p.o_sx;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem + ((uint32_t)(quad * 32) << 16) + acc * p.acc_cols;
      const int cb = tc.nb * p.BN;
      int c0 = 0;
      for (; c0 + 32 <= p.BN; c0 += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(t_row + c0, r);
        tmem_ld_wait();
        epilogue_columns<32>(p, r, cb + c0, valid, pix_lin, out_px);
      }
      if (c0 < p.BN) {
        uint32_t r[16];
        tmem_ld_32x32b_x16(t_row + c0, r);
        tmem_ld_wait();
        epilogue_columns<16>(p, r, cb + c0, valid, pix_lin, out_px);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------
// 256-row variant: the tile is 256 output pixels (two 128-row MMA tiles sharing every weight slot),
// two MMA-issuing warps (one thread sustains only ~1 tcgen05.mma / 49 cycles plus ~300 cycles of
// barrier round trip per k-iteration -- profiles/r01_flat_v0_timeline.txt), 8 epilogue warps that
// request all their global operands before waiting on the TMEM load.  Used whenever the layer has
// enough 256-pixel tiles to fill the SMs; the 128-row kernel above serves the small layers.
constexpr int kThreads256 = 352;

template <int NC>
struct EpiLoads256 {
  uint4 a[NC / 8];   // previous output (accumulate) or residual 1
  uint4 r2[NC / 8];
  uint4 msk[NC / 8];
};

template <int NC>
__device__ __forceinline__ void epi256_load(const IgemmParams& p, EpiLoads256<NC>& L, int cbase, long long pix_lin,
                                            const __nv_bfloat16* out_px) {
#pragma unroll
  for (int g = 0; g < NC / 8; ++g) {
    const int c = cbase + g * 8;
    if (c >= p.Cout) break;
    if (p.accumulate) L.a[g] = *reinterpret_cast<const uint4*>(out_px + p.o_coff + c);
    if (p.mask && c >= p.mask_lo && c < p.mask_hi)
      L.msk[g] = __ldg(reinterpret_cast<const uint4*>(p.mask + pix_lin * p.mask_c + p.mask_coff + c));
    if (c < p.res_nch) {
      if (p.res1) L.a[g] = __ldg(reinterpret_cast<const uint4*>(p.res1 + pix_lin * p.res1_c + p.res1_coff + c));
      if (p.res2) L.r2[g] = __ldg(reinterpret_cast<const uint4*>(p.res2 + pix_lin * p.res2_c + p.res2_coff + c));
    }
  }
}

template <int NC>
__device__ __forceinline__ void epi256_store(const IgemmParams& p, const uint32_t* acc, const EpiLoads256<NC>& L,
                                             int cbase, __nv_bfloat16* out_px) {
#pragma unroll
  for (int g = 0; g < NC / 8; ++g) {
    const int c = cbase + g * 8;
    if (c >= p.Cout) break;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[g * 8 + j]);
    if (p.bias) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + c));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + c + 4));
      v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
      v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= p.alpha;
    if (c < p.res_nch) {
      if (p.res1) {
        float r[8];
        unpack8(L.a[g], r);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(p.beta1, r[j], v[j]);
      }
      if (p.res2) {
        float r[8];
        unpack8(L.r2[g], r);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(p.beta2, r[j], v[j]);
      }
    }
    __nv_bfloat16* dst = out_px + p.o_coff + c;
    if (p.accumulate) {
      float r[8];
      unpack8(L.a[g], r);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += r[j];
    }
    if (p.act) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * p.slope;
    }
    if (p.mask && c >= p.mask_lo && c < p.mask_hi) {
      float r[8];
      unpack8(L.msk[g], r);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = r[j] > 0.f ? v[j] : v[j] * p.mask_slope;
    }
    const uint4 o = pack8(v);
    *reinterpret_cast<uint4*>(dst) = o;
    if (p.upsample) {
      *reinterpret_cast<uint4*>(dst + p.o_sx) = o;
      *reinterpret_cast<uint4*>(dst + p.o_sy) = o;
      *reinterpret_cast<uint4*>(dst + p.o_sy + p.o_sx) = o;
    }
  }
}

// EPI = 0: general epilogue (residuals, accumulate, partial channel blocks, direct or staged stores).
// EPI = 1 / 2: the straight-line epilogue of the common case -- staged TMA stores, BN a multiple of 64, only
// bias / alpha / LeakyReLU (1) plus the activation-derivative mask (2).  The general code evaluates every feature
// flag per 8-channel group; with two epilogue warps per scheduler nothing hides those dependent branches and loads,
// and the epilogue (not the tensor pipe) set the pace of every layer (profiles/r02_igemm_epilogue.txt).
template <int EPI>
__global__ void __launch_bounds__(kThreads256, 1)
conv_igemm256_kernel(const __grid_constant__ IgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem =
      reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[kMaxStages], empty_bar[kMaxStages], tfull_bar[2], tempty_bar[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float sbias[EPI ? 256 : 4];   // this tile's bias slice (EPI != 0)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 2);
    }
    mbar_init(&tfull_bar[0], 2);
    mbar_init(&tfull_bar[1], 2);
    mbar_init(&tempty_bar[0], 8);
    mbar_init(&tempty_bar[1], 8);
    mbar_fence_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.in_map);
    tma_prefetch_desc(&p.w_map);
  }
  if (warp == 1) {
    tmem_alloc(&tmem_base_s, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  // Dependents may be scheduled from here on: this CTA already owns its TMEM columns, so a co-resident
  // CTA of the next kernel can never make it wait for an allocation (which would deadlock, because that
  // CTA in turn waits for this grid to complete).
  pdl_trigger();
  pdl_wait();   // everything above overlapped the previous kernel's tail
  const int k_iters = p.ntaps * p.k_chunks;

  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    int dbg_it = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(p, tile);
      for (int t0 = 0; t0 < p.ntaps; ++t0) {
        const int t = tc.cls * p.ntaps + t0;
        const int cx = tc.x0 * p.in_stride + p.in_off_x + p.tap_dx[t];
        const int cy = tc.y0 * p.in_stride + p.in_off_y + p.tap_dy[t];
        const int wt = p.tap_w[t];
        for (int c = 0; c < p.k_chunks; ++c) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (p.dbg_ptr && blockIdx.x == 0 && lane == 0 && dbg_it < 64) p.dbg_ptr[128 + dbg_it++] = clock64();
          if (elect_one()) {
            uint8_t* sa = smem + (size_t)stage * p.stage_bytes;
            mbar_expect_tx(&full_bar[stage], p.a_bytes + p.b_bytes);
            tma_load_4d(sa, &p.in_map, &full_bar[stage], p.cin_off + c * 64, cx, cy, tc.n0);
            tma_load_3d(sa + p.a_bytes, &p.w_map, &full_bar[stage], c * 64, tc.nb * p.BN, wt);
          }
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    const int half = warp - 1;
    const uint32_t idesc = make_idesc_bf16(128, p.BN, 0, 0);
    const uint64_t desc_hi = make_smem_desc(0, 16, 1024, LAYOUT_SW128, 0);
    const uint32_t smem_base = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    int dbg_it = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem + acc * 2 * p.acc_cols + half * p.acc_cols;
      int c = 0;
      for (int it = 0; it < k_iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const bool stamp = p.dbg_ptr && blockIdx.x == 0 && half == 0 && lane == 0 && dbg_it < 64;
        if (stamp) p.dbg_ptr[2 * dbg_it] = clock64();
        const int nk = (c == p.k_chunks - 1) ? p.last_k16 : 4;
        const uint32_t a_addr = smem_base + stage * p.stage_bytes + half * kABytes;
        const uint32_t b_addr = smem_base + stage * p.stage_bytes + p.a_bytes;
        if (elect_one()) {
          for (int k = 0; k < nk; ++k) {
            const uint64_t ad = desc_hi | (uint64_t)(((a_addr + k * 32) >> 4) & 0x3FFF);
            const uint64_t bd = desc_hi | (uint64_t)(((b_addr + k * 32) >> 4) & 0x3FFF);
            umma_f16(d_tmem, ad, bd, idesc, (it | k) != 0);
          }
          umma_commit(&empty_bar[stage]);
          if (it == k_iters - 1) umma_commit(&tfull_bar[acc]);
        }
        __syncwarp();
        if (stamp) p.dbg_ptr[2 * dbg_it++ + 1] = clock64();
        if (++c == p.k_chunks) c = 0;
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (p.acc_stages == 2) {
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      } else {
        acc_phase ^= 1;
      }
    }
  } else {
    const int quad = warp & 3;
    const int half = (warp - 3) >> 2;
    const int m = half * 128 + quad * 32 + lane;
    const int ix = m % p.tw;
    const int iy = (m / p.tw) % p.th;
    const int in_ = m / (p.tw * p.th);
    int acc = 0;
    uint32_t acc_phase = 0;
    int st_count = 0, st_tiles = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(p, tile);
      const int x = tc.x0 + ix, y = tc.y0 + iy, n = tc.n0 + in_;
      const bool valid = (x < p.Wo) && (y < p.Ho) && (n < p.Nimg) && !(p.dbg & 1);
      const int cy_ = tc.cls >> 1, cx_ = tc.cls & 1;   // parity offsets of a merged launch (0 otherwise)
      const long long pix_lin = ((long long)n * p.aux_h + (y * p.aux_my + p.aux_oy + cy_)) * p.aux_w +
                                (x * p.aux_mx + p.aux_ox + cx_);
      __nv_bfloat16* out_px = p.out + (long long)n * p.o_sn +
                              (long long)(y * p.o_my + p.o_oy + cy_) * p.o_sy +
                              (long long)(x * p.o_mx + p.o_ox + cx_) * p.o_sx;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const bool estamp = p.dbg_ptr && blockIdx.x == 0 && warp == 3 && lane == 0 && st_tiles < 8;
      if (estamp) p.dbg_ptr[256 + 2 * st_tiles] = clock64();
      const uint32_t t_row = tmem + ((uint32_t)(quad * 32) << 16) + acc * 2 * p.acc_cols + half * p.acc_cols;
      const int cb = tc.nb * p.BN;
      int c0 = 0;
      if constexpr (EPI != 0) {
        const int m_local = quad * 32 + lane;
        const bool issuer = (quad == 0) && (lane == 0);
        const int ty = tc.y0 + half * p.st_dy, tn_ = tc.n0 + half * p.st_dn;
        // bias slice of this tile -> shared memory (one copy for both halves)
        named_bar_sync(3, 256);   // everyone is done with the previous tile's slice
        {
          const int e = half * 128 + m_local;
          if (e < p.BN) sbias[e] = (p.bias && cb + e < p.Cout) ? __ldg(p.bias + cb + e) : 0.f;
        }
        named_bar_sync(3, 256);
        const float alpha = p.alpha, slope = p.slope, mslope = p.mask_slope;
        const bool act = p.act != 0;
        const __nv_bfloat16* mrow = (EPI == 2 && valid) ? p.mask + pix_lin * p.mask_c + p.mask_coff : nullptr;
        uint32_t r[2][32];
        tmem_ld_32x32b_x32(t_row, r[0]);
        tmem_ld_32x32b_x32(t_row + 32, r[1]);
        for (; c0 < p.BN; c0 += 64) {
          const int buf = st_count % p.st_bufs;
          ++st_count;
          uint8_t* sbuf = smem + p.st_off + (size_t)(half * p.st_bufs + buf) * (128 * 128);
          uint4 mk[8];
          if (EPI == 2) {
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              const int c = cb + c0 + g * 8;
              mk[g] = (mrow && c >= p.mask_lo && c < p.mask_hi) ? __ldg(reinterpret_cast<const uint4*>(mrow + c))
                                                               : make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u);
            }
          }
          if (issuer) {   // the store that last read this staging buffer has drained it
            if (p.st_bufs == 2) bulk_wait_group_read<1>(); else bulk_wait_group_read<0>();
          }
          if (half == 0) named_bar_sync(1, 128); else named_bar_sync(2, 128);
          tmem_ld_wait();
          const uint32_t srow = smem_u32(sbuf) + (uint32_t)m_local * 128;
          const int sx = m_local & 7;
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            float v[8];
            const float4 b0 = *reinterpret_cast<const float4*>(&sbias[c0 + g * 8]);
            const float4 b1 = *reinterpret_cast<const float4*>(&sbias[c0 + g * 8 + 4]);
            const uint32_t* a = &r[g >> 2][(g & 3) * 8];
            v[0] = (__uint_as_float(a[0]) + b0.x) * alpha; v[1] = (__uint_as_float(a[1]) + b0.y) * alpha;
            v[2] = (__uint_as_float(a[2]) + b0.z) * alpha; v[3] = (__uint_as_float(a[3]) + b0.w) * alpha;
            v[4] = (__uint_as_float(a[4]) + b1.x) * alpha; v[5] = (__uint_as_float(a[5]) + b1.y) * alpha;
            v[6] = (__uint_as_float(a[6]) + b1.z) * alpha; v[7] = (__uint_as_float(a[7]) + b1.w) * alpha;
            if (act) {
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * slope;
            }
            if (EPI == 2) {
              float mf[8];
              unpack8(mk[g], mf);
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = mf[j] > 0.f ? v[j] : v[j] * mslope;
            }
            const uint4 o = pack8(v);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + (uint32_t)((g ^ sx) << 4)), "r"(o.x),
                         "r"(o.y), "r"(o.z), "r"(o.w)
                         : "memory");
          }
          if (c0 + 64 < p.BN) {   // next slab's accumulators: in flight while this slab is stored
            tmem_ld_32x32b_x32(t_row + c0 + 64, r[0]);
            tmem_ld_32x32b_x32(t_row + c0 + 96, r[1]);
          }
          fence_proxy_async_smem();
          if (half == 0) named_bar_sync(1, 128); else named_bar_sync(2, 128);
          if (issuer && !(p.dbg & 1)) {
            const int ch = p.o_coff + cb + c0;
            if (p.upsample) {
#pragma unroll
              for (int rep = 0; rep < 4; ++rep) tma_store_4d(&p.out_map[rep], sbuf, ch, tc.x0, ty, tn_);
            } else {
              tma_store_4d(&p.out_map[tc.cls], sbuf, ch, tc.x0, ty, tn_);
            }
            bulk_commit_group();
          }
          if constexpr (EPI == 3) {
            // column statistics of the staged slab (the values the next layer will read): thread = (column, statistic),
            // 128 rows in row order; pixels outside the image are excluded.  The buffer is not rewritten before every
            // thread of this half has passed the "buffer free" barrier of its next use.
            const int col = m_local & 63, which = m_local >> 6;
            const int rows_x = p.Wo - tc.x0, rows_y = p.Ho - ty, rows_n = p.Nimg - tn_;
            float acc_s = 0.f;
            const uint32_t cbase_s = smem_u32(sbuf) + (uint32_t)((col & 7) * 2);
            const int hth = p.st_dn ? p.th : p.th / 2, htn = p.st_dn ? p.st_dn : 1;   // the half's rows and images
            auto ld_col = [&](int r) {
              uint16_t hv;
              asm volatile("ld.shared.u16 %0, [%1];" : "=h"(hv) : "r"(cbase_s + (uint32_t)(r * 128 + (((col >> 3) ^ (r & 7)) << 4))));
              return __uint_as_float((uint32_t)hv << 16);
            };
            if (rows_x >= p.tw && rows_y >= hth && rows_n >= htn) {
#pragma unroll 8
              for (int r = 0; r < 128; ++r) {
                const float f = ld_col(r);
                acc_s += which ? f * f : f;
              }
            } else {
              for (int r = 0; r < 128; ++r) {
                const int rx = r % p.tw, ry = (r / p.tw) % hth, rn = r / (p.tw * hth);
                if (rx >= rows_x || ry >= rows_y || rn >= rows_n) continue;
                const float f = ld_col(r);
                acc_s += which ? f * f : f;
              }
            }
            const int cglob = cb + c0 + col;
            if (cglob < p.Cout) {
              const int prow = 2 * (tile / p.n_blocks) + half;
              p.stat_part[((size_t)which * p.Cout + cglob) * p.stat_rows + prow] = acc_s;
            }
          }
        }
      } else {
      for (; c0 + 32 <= p.BN; c0 += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(t_row + c0, r);
        EpiLoads256<32> L;        if (valid) epi256_load<32>(p, L, cb + c0, pix_lin, out_px);
        tmem_ld_wait();
        if (valid) epi256_store<32>(p, r, L, cb + c0, out_px);
      }
      if (c0 < p.BN) {
        uint32_t r[16];
        tmem_ld_32x32b_x16(t_row + c0, r);
        EpiLoads256<16> L;
        if (valid) epi256_load<16>(p, L, cb + c0, pix_lin, out_px);
        tmem_ld_wait();
        if (valid) epi256_store<16>(p, r, L, cb + c0, out_px);
      }
      }   // EPI == 0
      if (estamp) p.dbg_ptr[256 + 2 * st_tiles++ + 1] = clock64();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (p.acc_stages == 2) {
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      } else {
        acc_phase ^= 1;
      }
    }
  }
  if (p.tma_store && warp >= 3 && (warp & 3) == 0 && lane == 0) bulk_wait_group<0>();   // staging buffers drained
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

inline int pow2_ceil(int v) {
  int r = 1;
  while (r < v) r <<= 1;
  return r;
}

}  // namespace
}  // namespace b200

using namespace b200;

// stat_part != nullptr: also produce the BatchNorm partial statistics (EPI = 3); stat_query != nullptr: launch
// nothing, only report how many partial rows that would produce (0 = this conv cannot: fall back to
// b200_bn_stats_finalize).
static int conv_igemm_impl(const b200_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                           const void* res1, const void* res2, const void* mask, void* y, float* stat_part,
                           int* stat_query, b200_stream_t stream) {
  B200_REQUIRE(d && (stat_query || (x && w_packed && y)), "b200_conv_igemm: null argument");
  B200_REQUIRE(d->cin > 0 && d->cin % 16 == 0, "b200_conv_igemm: cin=%d must be a multiple of 16", d->cin);
  B200_REQUIRE(d->cout > 0 && d->cout % 8 == 0, "b200_conv_igemm: cout=%d must be a multiple of 8", d->cout);
  B200_REQUIRE(d->cx % 8 == 0 && d->cy % 8 == 0 && d->cin_off % 8 == 0 && d->cout_off % 8 == 0,
               "b200_conv_igemm: channel pitches/offsets must be multiples of 8");
  B200_REQUIRE(d->ntaps >= 1 && d->ntaps <= B200_MAX_TAPS, "b200_conv_igemm: bad ntaps %d", d->ntaps);
  B200_REQUIRE(d->in_stride >= 1 && d->in_stride <= 8, "b200_conv_igemm: bad in_stride");
  B200_REQUIRE(d->w_cin_pad % 64 == 0 && d->w_cin_pad >= d->cin, "b200_conv_igemm: bad w_cin_pad");
  B200_REQUIRE(d->w_cout_pad % 16 == 0 && d->w_cout_pad >= d->cout, "b200_conv_igemm: bad w_cout_pad");
  B200_REQUIRE(!(d->upsample2x && (d->out_mul_y != 1 || d->out_mul_x != 1)),
               "b200_conv_igemm: upsample2x excludes output placement");

  const int kSmemBytes = 200 * 1024;
  B200_ENSURE_SMEM(conv_igemm_kernel, kSmemBytes);
  const int kSmem256 = 225 * 1024;   // the 256-row kernel also stages its output tiles
  B200_ENSURE_SMEM(conv_igemm256_kernel<0>, kSmem256);
  B200_ENSURE_SMEM(conv_igemm256_kernel<1>, kSmem256);
  B200_ENSURE_SMEM(conv_igemm256_kernel<2>, kSmem256);
  B200_ENSURE_SMEM(conv_igemm256_kernel<3>, kSmem256);

  IgemmParams p;
  memset(&p, 0, sizeof(p));
  // ---- tile geometry: 256-pixel tiles (two MMA issuers) when the layer has enough of them
  const int sms = sm_count();
  auto geometry = [&](int rows) {
    p.tw = d->w_out > 8 ? 16 : (d->w_out > 4 ? 8 : 4);
    int th_max = rows / p.tw;
    p.th = pow2_ceil(d->h_out) < th_max ? pow2_ceil(d->h_out) : th_max;
    p.tn = rows / (p.tw * p.th);
    p.tiles_x = (d->w_out + p.tw - 1) / p.tw;
    p.tiles_y = (d->h_out + p.th - 1) / p.th;
    p.tiles_n = (d->n + p.tn - 1) / p.tn;
    return p.tiles_x * p.tiles_y * p.tiles_n;
  };
  auto nblocks = [&](int bn) { return (d->cout + bn - 1) / bn; };
  // Tile shape (128 or 256 pixel rows x BN output channels) by a small cost model instead of "fill the SMs": many of
  // these layers are L2 -> shared-memory bound, and narrow tiles re-fetch the activation tile once per output-channel
  // block.  cost = max(tensor time of the slowest SM, operand bytes / L2 bandwidth), both in SM cycles; the model
  // reproduces the measured times within ~15 % (512->512 @16x16, 256 x 64 tiles: 82 k cycles; @32x32, 256 x 256: 143 k).
  const int ncls = d->parity_classes == 4 ? 4 : 1;
  const int bn0 = d->cout <= 256 ? ((d->cout + 15) / 16) * 16 : 256;
  const long long k_iters_h = (long long)d->ntaps * ((d->cin + 63) / 64);
  double best_cost = 1e30;
  int best_rows = 128, BN = bn0;
  for (int rows = 256; rows >= 128; rows -= 128) {
    const int px_tiles = geometry(rows);
    for (int bn = bn0;; bn /= 2) {
      const long long tiles = (long long)px_tiles * nblocks(bn) * ncls;
      const long long waves = (tiles + sms - 1) / sms;
      const double mma_one = bn / 2.0 > (4096.0 + bn * 32.0) / 128.0 ? bn / 2.0 : (4096.0 + bn * 32.0) / 128.0;
      const double t_mma = (double)waves * k_iters_h * 4.0 * (rows / 128) * mma_one;
      const double t_l2 = (double)tiles * k_iters_h * (rows * 128.0 + bn * 128.0) / 4500.0;   // chip-wide L2 -> SM bytes/cycle
      const double t_sm = (double)waves * k_iters_h * (rows * 128.0 + bn * 128.0) / 40.0;      // one SM's L2 ingest bytes/cycle
      double cost = t_mma > t_l2 ? t_mma : t_l2;
      cost = (cost > t_sm ? cost : t_sm) + 3000.0 * waves;
      if (cost < best_cost) {
        best_cost = cost;
        best_rows = rows;
        BN = bn;
      }
      if (!(bn >= 64 && bn % 32 == 0 && d->cout % (bn / 2) == 0)) break;
    }
  }
  static const bool igemm_debug = getenv("B200_IGEMM_DEBUG") != nullptr;
  if (igemm_debug)
    fprintf(stderr, "conv_igemm: cin %d cout %d %dx%dx%d taps %d x%d stride %d -> %d-row tile x BN %d (model %.0f cycles)\n",
            d->cin, d->cout, d->n, d->h_out, d->w_out, d->ntaps, ncls, d->in_stride, best_rows, BN, best_cost);
  const bool use256 = best_rows == 256;
  int pixel_tiles = geometry(best_rows);
  p.BN = BN;
  p.acc_cols = (BN + 31) & ~31;
  p.acc_stages = (4 * p.acc_cols <= 512) ? 2 : 1;
  p.a_bytes = use256 ? 2 * kABytes : kABytes;
  p.n_blocks = nblocks(BN);
  p.cls_tiles = pixel_tiles * p.n_blocks;
  p.total_tiles = p.cls_tiles * ncls;
  p.Nimg = d->n;
  p.Ho = d->h_out;
  p.Wo = d->w_out;
  p.in_stride = d->in_stride;
  p.in_off_y = d->in_off_y;
  p.in_off_x = d->in_off_x;
  p.cin_off = d->cin_off;
  p.k_chunks = (d->cin + 63) / 64;
  p.last_k16 = (d->cin % 64 == 0) ? 4 : (d->cin % 64) / 16;
  p.ntaps = d->ntaps;
  B200_REQUIRE(d->parity_classes == 0 || d->parity_classes == 1 || d->parity_classes == 4,
               "b200_conv_igemm: parity_classes must be 0, 1 or 4");
  B200_REQUIRE(d->ntaps * ncls <= B200_MAX_TAPS, "b200_conv_igemm: %d taps x %d classes exceed the tap table", d->ntaps, ncls);
  B200_REQUIRE(ncls == 1 || (d->out_mul_y == 2 && d->out_mul_x == 2 && !d->upsample2x),
               "b200_conv_igemm: parity classes need out_mul = (2, 2)");
  for (int t = 0; t < d->ntaps * ncls; ++t) {
    p.tap_dy[t] = d->tap_dy[t];
    p.tap_dx[t] = d->tap_dx[t];
    p.tap_w[t] = d->tap_w[t];
    B200_REQUIRE(d->tap_w[t] >= 0 && d->tap_w[t] < d->w_taps, "b200_conv_igemm: tap_w out of range");
  }
  p.Cout = d->cout;
  p.b_bytes = (uint32_t)BN * 128;
  p.stage_bytes = p.a_bytes + ((p.b_bytes + 1023) & ~1023u);
  p.stages = (kSmemBytes - 2048) / (int)p.stage_bytes;
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  B200_REQUIRE(p.stages >= 2, "b200_conv_igemm: not enough shared memory for 2 stages");
  static const int igemm_dbg = getenv("B200_IGEMM_DBG") ? atoi(getenv("B200_IGEMM_DBG")) : 0;
  p.dbg = igemm_dbg;
  static long long* const igemm_dbg_ptr =
      getenv("B200_IGEMM_DBG_PTR") ? reinterpret_cast<long long*>(strtoull(getenv("B200_IGEMM_DBG_PTR"), nullptr, 0)) : nullptr;
  p.dbg_ptr = igemm_dbg_ptr;
  // straight-line epilogue with staged TMA tile stores (conv_igemm256_kernel<1 / 2>): whole 64-channel slabs, no
  // residual / accumulate operands
  p.tma_store = use256 && BN % 64 == 0 && !res1 && !res2 && !d->accumulate;
  if (p.tma_store) {
    const int kSlab = 128 * 128;   // one half's 64-channel slab
    p.st_bufs = 2;
    int st = (kSmem256 - 1024 - 2 * p.st_bufs * kSlab) / (int)p.stage_bytes;
    if (st < 3) {
      p.st_bufs = 1;
      st = (kSmem256 - 1024 - 2 * p.st_bufs * kSlab) / (int)p.stage_bytes;
    }
    if (st < 2) {
      p.tma_store = 0;
    } else {
      p.stages = st > kMaxStages ? kMaxStages : st;
      p.st_off = (uint32_t)p.stages * p.stage_bytes;
    }
  }

  const bool stats_ok = p.tma_store && ncls == 1 && !d->upsample2x && !mask && !d->act;
  if (stat_query) {
    *stat_query = stats_ok ? 2 * pixel_tiles : 0;
    return 0;
  }
  B200_REQUIRE(!stat_part || stats_ok, "b200_conv_igemm_stats: this conv has no statistics epilogue (ask b200_conv_igemm_stat_rows first)");
  p.stat_part = stat_part;
  p.stat_rows = 2 * pixel_tiles;
  // ---- tensor maps
  {
    uint64_t dims[4] = {(uint64_t)(d->cin_off + d->cin), (uint64_t)d->w_in, (uint64_t)d->h_in,
                        (uint64_t)d->n};
    uint64_t strides[3] = {(uint64_t)d->cx * 2, (uint64_t)d->w_in * d->cx * 2,
                           (uint64_t)d->h_in * d->w_in * d->cx * 2};
    uint32_t box[4] = {64, (uint32_t)(p.tw * d->in_stride), (uint32_t)(p.th * d->in_stride),
                       (uint32_t)p.tn};
    uint32_t es[4] = {1, (uint32_t)d->in_stride, (uint32_t)d->in_stride, 1};
    if (make_tensor_map(&p.in_map, x, 4, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  {
    uint64_t dims[3] = {(uint64_t)d->w_cin_pad, (uint64_t)d->w_cout_pad, (uint64_t)d->w_taps};
    uint64_t strides[2] = {(uint64_t)d->w_cin_pad * 2, (uint64_t)d->w_cout_pad * d->w_cin_pad * 2};
    uint32_t box[3] = {64, (uint32_t)BN, 1};
    if (make_tensor_map(&p.w_map, w_packed, 3, dims, strides, box, nullptr,
                        CU_TENSOR_MAP_SWIZZLE_128B))
      return 1;
  }
  // ---- output placement
  p.out = reinterpret_cast<__nv_bfloat16*>(y);
  if (p.tma_store) {
    // strided views of the output, one per parity class / 2x2 replica: [channels, Wo, Ho, N] at pitch (mul_x, mul_y)
    const int mul_y = d->upsample2x ? 2 : (d->out_mul_y ? d->out_mul_y : 1);
    const int mul_x = d->upsample2x ? 2 : (d->out_mul_x ? d->out_mul_x : 1);
    const int off_y = d->upsample2x ? 0 : d->out_off_y, off_x = d->upsample2x ? 0 : d->out_off_x;
    const int nmaps = (ncls == 4 || d->upsample2x) ? 4 : 1;
    const int half_th = p.tn >= 2 ? p.th : p.th / 2, half_tn = p.tn >= 2 ? p.tn / 2 : 1;
    p.st_dy = p.tn >= 2 ? 0 : p.th / 2;
    p.st_dn = p.tn >= 2 ? p.tn / 2 : 0;
    for (int k = 0; k < nmaps; ++k) {
      const long long base = ((long long)(off_y + (k >> 1)) * d->w_buf + (off_x + (k & 1))) * d->cy;
      uint64_t dims[4] = {(uint64_t)(d->cout_off + d->cout), (uint64_t)d->w_out, (uint64_t)d->h_out, (uint64_t)d->n};
      uint64_t strides[3] = {(uint64_t)mul_x * d->cy * 2, (uint64_t)mul_y * d->w_buf * d->cy * 2,
                             (uint64_t)d->h_buf * d->w_buf * d->cy * 2};
      uint32_t box[4] = {64, (uint32_t)p.tw, (uint32_t)half_th, (uint32_t)half_tn};
      if (make_tensor_map(&p.out_map[k], reinterpret_cast<const __nv_bfloat16*>(y) + base, 4, dims, strides, box,
                          nullptr, CU_TENSOR_MAP_SWIZZLE_128B))
        return 1;
    }
  }
  p.o_sx = d->cy;
  p.o_sy = (long long)d->w_buf * d->cy;
  p.o_sn = (long long)d->h_buf * d->w_buf * d->cy;
  p.o_coff = d->cout_off;
  p.upsample = d->upsample2x;
  if (d->upsample2x) {
    p.o_my = 2; p.o_oy = 0; p.o_mx = 2; p.o_ox = 0;
    B200_REQUIRE(d->h_buf == 2 * d->h_out && d->w_buf == 2 * d->w_out, "b200_conv_igemm: upsample buffer dims");
  } else {
    p.o_my = d->out_mul_y ? d->out_mul_y : 1;
    p.o_oy = d->out_off_y;
    p.o_mx = d->out_mul_x ? d->out_mul_x : 1;
    p.o_ox = d->out_off_x;
    B200_REQUIRE((d->h_out - 1) * p.o_my + p.o_oy < d->h_buf && (d->w_out - 1) * p.o_mx + p.o_ox < d->w_buf,
                 "b200_conv_igemm: output placement exceeds buffer");
  }
  if (d->upsample2x) {
    p.aux_h = d->h_out; p.aux_w = d->w_out; p.aux_my = 1; p.aux_oy = 0; p.aux_mx = 1; p.aux_ox = 0;
  } else {
    p.aux_h = d->h_buf; p.aux_w = d->w_buf;
    p.aux_my = p.o_my; p.aux_oy = p.o_oy; p.aux_mx = p.o_mx; p.aux_ox = p.o_ox;
  }
  p.bias = bias;
  p.alpha = d->alpha;
  p.act = d->act;
  p.slope = d->slope;
  p.res1 = reinterpret_cast<const __nv_bfloat16*>(res1);
  p.res2 = reinterpret_cast<const __nv_bfloat16*>(res2);
  p.res1_c = d->res1_c; p.res1_coff = d->res1_coff;
  p.res2_c = d->res2_c; p.res2_coff = d->res2_coff;
  p.res_nch = (res1 || res2) ? (d->res_nch > 0 ? d->res_nch : d->cout) : 0;
  p.beta1 = d->beta1; p.beta2 = d->beta2;
  p.accumulate = d->accumulate;
  p.mask = reinterpret_cast<const __nv_bfloat16*>(mask);
  p.mask_c = d->mask_c; p.mask_coff = d->mask_coff;
  p.mask_lo = d->mask_lo; p.mask_hi = d->mask_hi;
  p.mask_slope = d->mask_slope;

  const int grid = p.total_tiles < sms ? p.total_tiles : sms;
  const size_t smem = (size_t)p.stages * p.stage_bytes + 1024 + (p.tma_store ? 2 * (size_t)p.st_bufs * 128 * 128 : 0);
  const bool fast = p.tma_store != 0;
  if (use256 && fast && stat_part)
    ::b200::launch_kernel(conv_igemm256_kernel<3>, grid, kThreads256, smem, as_stream(stream), p);
  else if (use256 && fast && mask)
    ::b200::launch_kernel(conv_igemm256_kernel<2>, grid, kThreads256, smem, as_stream(stream), p);
  else if (use256 && fast)
    ::b200::launch_kernel(conv_igemm256_kernel<1>, grid, kThreads256, smem, as_stream(stream), p);
  else if (use256)
    ::b200::launch_kernel(conv_igemm256_kernel<0>, grid, kThreads256, smem, as_stream(stream), p);
  else
    ::b200::launch_kernel(conv_igemm_kernel, grid, kThreads, smem, as_stream(stream), p);
  B200_LAUNCH_CHECK();
  return 0;
}

extern "C" int b200_conv_igemm(const b200_conv_desc* d, const void* x, const void* w_packed,
                               const float* bias, const void* res1, const void* res2,
                               const void* mask, void* y, b200_stream_t stream) {
  return conv_igemm_impl(d, x, w_packed, bias, res1, res2, mask, y, nullptr, nullptr, stream);
}

extern "C" int b200_conv_igemm_stat_rows(const b200_conv_desc* d) {
  int rows = 0;
  if (conv_igemm_impl(d, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, &rows, nullptr)) return -1;
  return rows;
}

extern "C" int b200_conv_igemm_stats(const b200_conv_desc* d, const void* x, const void* w_packed,
                                     const float* bias, void* y, float* stat_part, b200_stream_t stream) {
  B200_REQUIRE(stat_part, "b200_conv_igemm_stats: null stat_part");
  return conv_igemm_impl(d, x, w_packed, bias, nullptr, nullptr, nullptr, y, stat_part, nullptr, stream);
}
