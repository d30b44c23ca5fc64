// 3x3 stride-1 convolution on zero-bordered ("flat") NHWC activations -- the RDB trunk fast path.
//
// With a 1-pixel zero border stored in HBM, [n, h+2, w+2, c] flattens to a matrix X[P, c] and a
// conv tap (dy, dx) is the row shift dy*(w+2)+dx.  One CTA tile = 256 consecutive rows:
//   A region  rows [m0 - (w+3), m0 + 256 + (w+3)) x 64 channels, ONE TMA-loaded smem tile per
//             channel chunk (SWIZZLE_128B, K-major) shared by all 9 taps -- a tap is just a different
//             start address of the UMMA smem descriptor (row shifts need no realignment because the
//             128B swizzle is a function of the absolute smem address; tools/umma_probe.cu).
//   B         weights [BN co x 64 ci] per (tap, chunk) from the packed tensor, own smem ring.
//   D         two 128-row accumulators [128 x BN] fp32 in TMEM (the two halves share every B tile).
// L2->SMEM traffic per MMA drops ~4.4x vs per-tap loading (conv_igemm.cu), which is what bounds
// the per-tap kernel on the Cout=32 / Cin=32 trunk layers.
//
// Warp roles: warp 0 TMA producer (A ring + B ring), warps 1-2 MMA issuers (one per 128-row half),
// warps 3..10 epilogue (only interior rows are stored; the border stays zero).
// Reference: ResidualDenseBlock_5C / RRDB forward and autograd dgrad (RRDBNet_arch.py:89-163).
#include <stdlib.h>

#include "common.cuh"
#include "sm100_ptx.cuh"

namespace b200 {
namespace {

constexpr int kThreads = 352;  // producer, 2 MMA issuers (one per 128-row half), 8 epilogue warps
constexpr int kMaxAStages = 4;
constexpr int kMaxBStages = 8;
constexpr int kTileM = 256;

struct FlatParams {
  CUtensorMap in_map;  // 2-D [P rows][C extent], box (64, box_rows)
  CUtensorMap in2_map; // optional second input (extends the reduction axis)
  CUtensorMap w_map;   // 3-D packed weights, box (64, BN, 1)
  int P, Hp, Wp, HpWp, h, w, n;
  int total_tiles;
  int cin_off, k_chunks, last_k16;      // k_chunks = kc1 + kc2
  int kc1, last1_k16, cin2_off;
  int tap_shift[9];
  int tap_w[9];
  int halo;            // Wp + 1
  int nbox, box_rows;  // A region = nbox boxes of box_rows rows
  uint32_t a_bytes, a_stage_bytes, b_bytes, b_tap_bytes, b_stage_bytes;
  int a_stages, b_stages;
  int tpb;             // taps per B stage (9, 3 or 1): one barrier round-trip per tpb taps
  uint32_t b_ring_off;
  int BN, acc_cols, acc_stages, Cout;
  // output
  __nv_bfloat16* out;
  int out_mode, cy, o_coff;
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
  long long* dbg;  // optional per-CTA timeline (clock64), 16 slots per CTA; nullptr in production
};

#define DBG_T(slot) do { if (p.dbg && lane == 0) p.dbg[blockIdx.x * 16 + (slot)] = clock64(); } while (0)

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

// Global operands of the epilogue for NC columns of one row, fetched BEFORE the TMEM load is waited
// on so that all of them are in flight together (the serial load->use chains were the bottleneck of
// the read-modify-write dgrad epilogue; profiles/r01_flat_v0_timeline.txt).
template <int NC>
struct EpiLoads {
  uint4 a[NC / 8];    // previous output value (accumulate) or residual 1 -- never both (checked on the host)
  uint4 r2[NC / 8];
  uint4 msk[NC / 8];
};

template <int NC>
__device__ __forceinline__ void flat_epilogue_load(const FlatParams& p, EpiLoads<NC>& L, int cbase, long long m,
                                                   const __nv_bfloat16* out_px) {
#pragma unroll
  for (int g = 0; g < NC / 8; ++g) {
    const int c = cbase + g * 8;
    if (c >= p.Cout) break;
    if (p.accumulate) L.a[g] = *reinterpret_cast<const uint4*>(out_px + p.o_coff + c);
    if (p.mask && c >= p.mask_lo && c < p.mask_hi)
      L.msk[g] = __ldg(reinterpret_cast<const uint4*>(p.mask + m * p.mask_c + p.mask_coff + c));
    if (c < p.res_nch) {
      if (p.res1) L.a[g] = __ldg(reinterpret_cast<const uint4*>(p.res1 + m * p.res1_c + p.res1_coff + c));
      if (p.res2) L.r2[g] = __ldg(reinterpret_cast<const uint4*>(p.res2 + m * p.res2_c + p.res2_coff + c));
    }
  }
}

template <int NC>
__device__ __forceinline__ void flat_epilogue(const FlatParams& p, const uint32_t* acc, const EpiLoads<NC>& L,
                                              int cbase, __nv_bfloat16* out_px, long long up_sx,
                                              long long up_sy) {
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
    if (p.out_mode == 2) {
      *reinterpret_cast<uint4*>(dst + up_sx) = o;
      *reinterpret_cast<uint4*>(dst + up_sy) = o;
      *reinterpret_cast<uint4*>(dst + up_sy + up_sx) = o;
    }
  }
}

// One 64-channel K chunk of one 128-row half: 9 taps in groups of TPB taps per weight stage.  A single
// elected lane issues a whole group inside ONE elect region: tcgen05.mma issue is nearly synchronous (the
// queue is a few instructions deep), so every elect/reconverge boundary between MMAs is a bubble on the
// tensor pipe whenever both issuers reach it together (tools/umma_probe.cu "pipe": a boundary every
// 4 MMAs costs 57 cycles/MMA, every 12 or 36 MMAs the hardware's 40.7 / 48.5).
template <int TPB>
__device__ __forceinline__ void flat_issue_chunk(const FlatParams& p, const uint32_t (&sh16)[9], uint32_t a16,
                                                 int nk, bool first_c, bool last_c,
                                                 uint32_t d_tmem, uint32_t idesc, uint64_t desc_hi,
                                                 uint32_t b_ring16, uint32_t b_stage16, uint32_t btap16,
                                                 int& bs, uint32_t& bph, uint64_t* b_full, uint64_t* b_empty,
                                                 uint64_t* a_empty_bar, uint64_t* tfull) {
#pragma unroll
  for (int g = 0; g < 9 / TPB; ++g) {
    mbar_wait(&b_full[bs], bph);
    tc_fence_after();
    const uint32_t b16 = b_ring16 + bs * b_stage16;
    if (elect_one()) {
#pragma unroll
      for (int j = 0; j < TPB; ++j) {
        const int t = g * TPB + j;
        const uint32_t at = a16 + sh16[t], bt = b16 + j * btap16;
        if (nk == 4) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16(d_tmem, desc_hi | (uint64_t)(at + 2 * k), desc_hi | (uint64_t)(bt + 2 * k), idesc,
                     !(first_c && t == 0 && k == 0));
        } else {
          for (int k = 0; k < nk; ++k)
            umma_f16(d_tmem, desc_hi | (uint64_t)(at + 2 * k), desc_hi | (uint64_t)(bt + 2 * k), idesc,
                     !(first_c && t == 0 && k == 0));
        }
      }
      umma_commit(&b_empty[bs]);
      if (g == 9 / TPB - 1) {
        umma_commit(a_empty_bar);
        if (last_c) umma_commit(tfull);
      }
    }
    __syncwarp();
    if (++bs == p.b_stages) {
      bs = 0;
      bph ^= 1;
    }
  }
}

// One CTA per SM (all of shared memory and TMEM); each CTA walks the tiles with stride gridDim.x.
__global__ void __launch_bounds__(kThreads, 1)
conv_flat_kernel(const __grid_constant__ FlatParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem =
      reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t a_full[kMaxAStages], a_empty[kMaxAStages], b_full[kMaxBStages],
      b_empty[kMaxBStages], tfull_bar[2], tempty_bar[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // provably warp-uniform
  const int lane = threadIdx.x & 31;
  if (warp == 0) DBG_T(0);
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.a_stages; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&a_empty[s], 2);   // both MMA issuers commit
    }
    for (int s = 0; s < p.b_stages; ++s) {
      mbar_init(&b_full[s], 1);
      mbar_init(&b_empty[s], 2);
    }
    mbar_init(&tfull_bar[0], 2);
    mbar_init(&tfull_bar[1], 2);
    mbar_init(&tempty_bar[0], 8);   // all epilogue warps
    mbar_init(&tempty_bar[1], 8);
    mbar_fence_init();
  }
  if (warp == 0 && lane == 0) {
    if (p.kc1) tma_prefetch_desc(&p.in_map);
    if (p.k_chunks > p.kc1) tma_prefetch_desc(&p.in2_map);
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
  if (warp == 0) DBG_T(1);

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int as = 0, bs = 0;
    uint32_t aph = 0, bph = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const int row0 = tile * kTileM - p.halo;
      for (int c = 0; c < p.k_chunks; ++c) {
        mbar_wait(&a_empty[as], aph ^ 1);
        if (elect_one()) {
          uint8_t* sa = smem + (size_t)as * p.a_stage_bytes;
          mbar_expect_tx(&a_full[as], p.a_bytes);
          const CUtensorMap* im = (c < p.kc1) ? &p.in_map : &p.in2_map;
          const int ch = (c < p.kc1) ? p.cin_off + c * 64 : p.cin2_off + (c - p.kc1) * 64;
          for (int j = 0; j < p.nbox; ++j)
            tma_load_2d(sa + (size_t)j * p.box_rows * 128, im, &a_full[as], ch, row0 + j * p.box_rows);
        }
        __syncwarp();
        if (++as == p.a_stages) {
          as = 0;
          aph ^= 1;
        }
        for (int t0 = 0; t0 < 9; t0 += p.tpb) {
          mbar_wait(&b_empty[bs], bph ^ 1);
          if (elect_one()) {
            uint8_t* sb = smem + p.b_ring_off + (size_t)bs * p.b_stage_bytes;
            mbar_expect_tx(&b_full[bs], p.b_bytes * p.tpb);
            for (int j = 0; j < p.tpb; ++j)
              tma_load_3d(sb + (size_t)j * p.b_tap_bytes, &p.w_map, &b_full[bs], c * 64, 0, p.tap_w[t0 + j]);
          }
          __syncwarp();
          if (++bs == p.b_stages) {
            bs = 0;
            bph ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ------------------------------------------------------------ MMA issuers: warp 1 -> rows
    // [0,128) of the tile, warp 2 -> rows [128,256); each owns one TMEM accumulator.  Two issuing
    // threads because a single thread sustains only ~1 tcgen05.mma per 49 cycles
    // (profiles/r01_umma_issue_rate_probe.log), below the 40-cycle smem-bound rate of N = 32.
    const int half = warp - 1;
    const uint32_t idesc = make_idesc_bf16(128, p.BN, 0, 0);
    const uint64_t desc_hi = make_smem_desc(0, 16, 1024, LAYOUT_SW128, 0);
    const uint32_t smem_base = smem_u32(smem);
    // Everything the issue loop touches is warp-uniform (the warp index comes from a shuffle so that the
    // compiler can prove it) and the nine tap offsets live in registers: the descriptor of an MMA is then
    // two uniform adds away from the previous one.  With per-tap constant-bank loads and R2UR moves in
    // the loop the issuers managed only one MMA per ~130 cycles each (tools/umma_probe.cu "pipe" reaches
    // the hardware's 40/48 cycles per MMA with the same barrier structure).
    uint32_t sh16[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) sh16[t] = (uint32_t)(p.tap_shift[t] * 8);   // rows of 128 B, in 16-B units
    const uint32_t btap16 = p.b_tap_bytes >> 4;
    const uint32_t b_ring16 = (smem_base + p.b_ring_off) >> 4, b_stage16 = p.b_stage_bytes >> 4;
    int as = 0, bs = 0;
    uint32_t aph = 0, bph = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem + acc * 2 * p.acc_cols + half * p.acc_cols;
      for (int c = 0; c < p.k_chunks; ++c) {
        mbar_wait(&a_full[as], aph);
        tc_fence_after();
        if (half == 0 && tile == (int)blockIdx.x && c == 0) DBG_T(2);
        const int nk = (c == p.k_chunks - 1) ? p.last_k16 : ((c == p.kc1 - 1) ? p.last1_k16 : 4);
        const uint32_t a16 = (smem_base + as * p.a_stage_bytes + (uint32_t)(p.halo + half * 128) * 128) >> 4;
        const bool first_c = (c == 0), last_c = (c == p.k_chunks - 1);
        if (p.tpb == 9)
          flat_issue_chunk<9>(p, sh16, a16, nk, first_c, last_c, d_tmem, idesc, desc_hi, b_ring16, b_stage16,
                              btap16, bs, bph, b_full, b_empty, &a_empty[as], &tfull_bar[acc]);
        else if (p.tpb == 3)
          flat_issue_chunk<3>(p, sh16, a16, nk, first_c, last_c, d_tmem, idesc, desc_hi, b_ring16, b_stage16,
                              btap16, bs, bph, b_full, b_empty, &a_empty[as], &tfull_bar[acc]);
        else
          flat_issue_chunk<1>(p, sh16, a16, nk, first_c, last_c, d_tmem, idesc, desc_hi, b_ring16, b_stage16,
                              btap16, bs, bph, b_full, b_empty, &a_empty[as], &tfull_bar[acc]);
        if (++as == p.a_stages) {
          as = 0;
          aph ^= 1;
        }
      }
      if (half == 0) DBG_T(tile == (int)blockIdx.x ? 3 : 4);
      if (p.acc_stages == 2) {
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      } else {
        acc_phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue (warps 3..10)
    // warps 3..6 -> rows [0,128), warps 7..10 -> rows [128,256)
    const int quad = warp & 3;            // TMEM lane quadrant accessible by this warp
    const int half = (warp - 3) >> 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if (warp == 3) DBG_T(tile == (int)blockIdx.x ? 5 : 7);
      const long long m = (long long)tile * kTileM + half * 128 + quad * 32 + lane;
      const int nimg = (int)(m / p.HpWp);
      const int rem = (int)(m - (long long)nimg * p.HpWp);
      const int yp = rem / p.Wp, xp = rem - yp * p.Wp;
      const bool valid = (m < p.P) && yp >= 1 && yp <= p.h && xp >= 1 && xp <= p.w;
      __nv_bfloat16* out_px;
      long long up_sx = 0, up_sy = 0;
      if (p.out_mode == 0) {
        out_px = p.out + m * p.cy;
      } else if (p.out_mode == 1) {
        out_px = p.out + (((long long)nimg * p.h + (yp - 1)) * p.w + (xp - 1)) * p.cy;
      } else {
        up_sx = p.cy;
        up_sy = (long long)2 * p.w * p.cy;
        out_px = p.out + (((long long)nimg * 2 * p.h + 2 * (yp - 1)) * 2 * p.w + 2 * (xp - 1)) * p.cy;
      }
      const uint32_t t_row = tmem + ((uint32_t)(quad * 32) << 16) + acc * 2 * p.acc_cols + half * p.acc_cols;
      int c0 = 0;
      for (; c0 + 32 <= p.BN; c0 += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(t_row + c0, r);
        EpiLoads<32> L;
        if (valid) flat_epilogue_load<32>(p, L, c0, m, out_px);
        tmem_ld_wait();
        if (valid) flat_epilogue<32>(p, r, L, c0, out_px, up_sx, up_sy);
      }
      if (c0 < p.BN) {
        uint32_t r[16];
        tmem_ld_32x32b_x16(t_row + c0, r);
        EpiLoads<16> L;
        if (valid) flat_epilogue_load<16>(p, L, c0, m, out_px);
        tmem_ld_wait();
        if (valid) flat_epilogue<16>(p, r, L, c0, out_px, up_sx, up_sy);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (warp == 3) DBG_T(tile == (int)blockIdx.x ? 6 : 8);
      if (p.acc_stages == 2) {
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      } else {
        acc_phase ^= 1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) DBG_T(9);
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------- layout helpers
__global__ void pad_copy_kernel(__nv_bfloat16* __restrict__ dst, int dst_c, int dst_coff,
                                const __nv_bfloat16* __restrict__ src, int src_c, int src_coff, int n,
                                int h, int w, int c) {
  pdl_trigger();
  pdl_wait();
  const int cv = c / 8;
  const long long total = (long long)n * h * w * cv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % cv) * 8;
    long long r = i / cv;
    const int x = (int)(r % w);
    r /= w;
    const int y = (int)(r % h);
    const int b = (int)(r / h);
    const long long sp = ((long long)b * h + y) * w + x;
    const long long dp = ((long long)b * (h + 2) + y + 1) * (w + 2) + x + 1;
    *reinterpret_cast<uint4*>(dst + dp * dst_c + dst_coff + v) =
        *reinterpret_cast<const uint4*>(src + sp * src_c + src_coff + v);
  }
}

__global__ void unpad_add_kernel(__nv_bfloat16* __restrict__ dst, int dst_c,
                                 const __nv_bfloat16* __restrict__ src, int src_c, int src_coff,
                                 const __nv_bfloat16* __restrict__ add, int add_c, int n, int h, int w,
                                 int c) {
  pdl_trigger();
  pdl_wait();
  const int cv = c / 8;
  const long long total = (long long)n * h * w * cv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % cv) * 8;
    long long r = i / cv;
    const int x = (int)(r % w);
    r /= w;
    const int y = (int)(r % h);
    const int b = (int)(r / h);
    const long long dp = ((long long)b * h + y) * w + x;
    const long long sp = ((long long)b * (h + 2) + y + 1) * (w + 2) + x + 1;
    uint4 u = *reinterpret_cast<const uint4*>(src + sp * src_c + src_coff + v);
    if (add) {
      float a[8], t[8];
      unpack8(u, a);
      unpack8(*reinterpret_cast<const uint4*>(add + dp * add_c + v), t);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += t[j];
      u = pack8(a);
    }
    *reinterpret_cast<uint4*>(dst + dp * dst_c + v) = u;
  }
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" int b200_conv3x3_flat(const b200_flat_desc* d, const void* x, const void* x2,
                                 const void* w_packed, const float* bias, const void* res1,
                                 const void* res2, const void* mask, void* y, b200_stream_t stream) {
  B200_REQUIRE(d && w_packed && y, "b200_conv3x3_flat: null argument");
  B200_REQUIRE((d->cin > 0 && x) || (d->cin2 > 0 && x2), "b200_conv3x3_flat: no input");
  B200_REQUIRE(d->cin % 16 == 0 && d->cin2 % 16 == 0, "b200_conv3x3_flat: cin %% 16");
  B200_REQUIRE(d->cin2 == 0 || (x2 && d->cx2 % 8 == 0 && d->cin2_off % 8 == 0), "b200_conv3x3_flat: bad second input");
  B200_REQUIRE(d->cout > 0 && d->cout % 16 == 0 && d->cout <= 192, "b200_conv3x3_flat: cout %% 16, <= 192");
  B200_REQUIRE(d->cx % 8 == 0 && d->cy % 8 == 0 && d->cin_off % 8 == 0 && d->cout_off % 8 == 0,
               "b200_conv3x3_flat: channel pitches/offsets must be multiples of 8");
  const int kSmemBytes = 200 * 1024;
  B200_ENSURE_SMEM(conv_flat_kernel, kSmemBytes);
  FlatParams p;
  memset(&p, 0, sizeof(p));
  p.n = d->n; p.h = d->h; p.w = d->w;
  p.Hp = d->h + 2; p.Wp = d->w + 2; p.HpWp = p.Hp * p.Wp;
  const long long P = (long long)d->n * p.HpWp;
  B200_REQUIRE(P < (1ll << 31), "b200_conv3x3_flat: too many positions");
  p.P = (int)P;
  p.total_tiles = (int)((P + kTileM - 1) / kTileM);
  p.halo = p.Wp + 1;
  const int region = kTileM + 2 * p.halo;
  p.nbox = (region + 255) / 256;
  // every box must start on a 1024-byte (8-row) boundary of the swizzle-128B pattern
  p.box_rows = (((region + p.nbox - 1) / p.nbox) + 7) & ~7;
  if (p.box_rows > 256) { p.nbox += 1; p.box_rows = (((region + p.nbox - 1) / p.nbox) + 7) & ~7; }
  p.a_bytes = (uint32_t)p.nbox * p.box_rows * 128;
  p.a_stage_bytes = (p.a_bytes + 1023) & ~1023u;
  p.cin_off = d->cin_off;
  p.kc1 = (d->cin + 63) / 64;
  p.last1_k16 = (d->cin % 64 == 0) ? 4 : (d->cin % 64) / 16;
  const int kc2 = (d->cin2 + 63) / 64;
  p.cin2_off = d->cin2_off;
  p.k_chunks = p.kc1 + kc2;
  p.last_k16 = kc2 ? ((d->cin2 % 64 == 0) ? 4 : (d->cin2 % 64) / 16) : p.last1_k16;
  for (int t = 0; t < 9; ++t) {
    p.tap_shift[t] = d->tap_dy[t] * p.Wp + d->tap_dx[t];
    p.tap_w[t] = d->tap_w[t];
    B200_REQUIRE(d->tap_w[t] >= 0 && d->tap_w[t] < d->w_taps, "b200_conv3x3_flat: tap_w out of range");
    B200_REQUIRE(d->tap_dy[t] >= -1 && d->tap_dy[t] <= 1 && d->tap_dx[t] >= -1 && d->tap_dx[t] <= 1,
                 "b200_conv3x3_flat: taps must be within the 3x3 window");
  }
  p.BN = d->cout;
  p.Cout = d->cout;
  p.acc_cols = (p.BN + 31) & ~31;
  p.acc_stages = (4 * p.acc_cols <= 512) ? 2 : 1;
  p.b_bytes = (uint32_t)p.BN * 128;
  p.b_tap_bytes = (p.b_bytes + 1023) & ~1023u;
  // taps per B stage: fewer barrier round trips for the MMA issuers when the weight tiles are small
  p.tpb = (9 * p.b_tap_bytes <= 40 * 1024) ? 9 : ((3 * p.b_tap_bytes <= 50 * 1024) ? 3 : 1);
  p.b_stage_bytes = p.b_tap_bytes * p.tpb;
  {
    // Shared-memory fit: prefer 2-3 activation stages and the largest weight stage (fewest barrier round
    // trips); wide images (large A region: (256 + 2(w+3)) rows x 128 B per stage) fall back to fewer taps
    // per weight stage and finally to a single activation stage.  Widest LR input that fits: w ~ 580.
    const int budget = kSmemBytes - 2048;
    bool fit = false;
    const int tpb0 = p.tpb;
    for (int a_st = 2; a_st >= 1 && !fit; --a_st) {
      for (int tpb : {9, 3, 1}) {
        if (tpb > tpb0) continue;
        const int st = (int)p.b_tap_bytes * tpb;
        const int bs = (budget - a_st * (int)p.a_stage_bytes) / st;
        if (bs >= 2) {
          p.a_stages = a_st;
          p.tpb = tpb;
          p.b_stage_bytes = (uint32_t)st;
          p.b_stages = bs > kMaxBStages ? kMaxBStages : bs;
          fit = true;
          break;
        }
      }
    }
    B200_REQUIRE(fit, "b200_conv3x3_flat: image too wide for the shared-memory A region (w=%d; limit ~580)", d->w);
    while (p.a_stages < 3 && p.b_stages >= 3 &&
           budget - (p.a_stages + 1) * (int)p.a_stage_bytes >= 3 * (int)p.b_stage_bytes) {
      ++p.a_stages;
      p.b_stages = (budget - p.a_stages * (int)p.a_stage_bytes) / (int)p.b_stage_bytes;
      if (p.b_stages > kMaxBStages) p.b_stages = kMaxBStages;
    }
  }
  p.b_ring_off = (uint32_t)p.a_stages * p.a_stage_bytes;
  if (d->cin > 0) {
    uint64_t dims[2] = {(uint64_t)(d->cin_off + d->cin), (uint64_t)P};
    uint64_t strides[1] = {(uint64_t)d->cx * 2};
    uint32_t box[2] = {64, (uint32_t)p.box_rows};
    if (make_tensor_map(&p.in_map, x, 2, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  if (d->cin2 > 0) {
    uint64_t dims[2] = {(uint64_t)(d->cin2_off + d->cin2), (uint64_t)P};
    uint64_t strides[1] = {(uint64_t)d->cx2 * 2};
    uint32_t box[2] = {64, (uint32_t)p.box_rows};
    if (make_tensor_map(&p.in2_map, x2, 2, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  {
    uint64_t dims[3] = {(uint64_t)d->w_cin_pad, (uint64_t)d->w_cout_pad, (uint64_t)d->w_taps};
    uint64_t strides[2] = {(uint64_t)d->w_cin_pad * 2, (uint64_t)d->w_cout_pad * d->w_cin_pad * 2};
    uint32_t box[3] = {64, (uint32_t)p.BN, 1};
    if (make_tensor_map(&p.w_map, w_packed, 3, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B))
      return 1;
  }
  p.out = reinterpret_cast<__nv_bfloat16*>(y);
  p.out_mode = d->out_mode;
  p.cy = d->cy;
  p.o_coff = d->cout_off;
  B200_REQUIRE(!(d->out_mode != 0 && (d->accumulate || mask)), "b200_conv3x3_flat: accumulate/mask need flat output");
  B200_REQUIRE(!(d->accumulate && res1), "b200_conv3x3_flat: accumulate and res1 are mutually exclusive");
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
  {
    const char* e = getenv("B200_FLAT_DBG_PTR");
    p.dbg = e ? reinterpret_cast<long long*>(strtoull(e, nullptr, 0)) : nullptr;
  }
  const int sms = sm_count();
  const size_t smem = (size_t)p.a_stages * p.a_stage_bytes + (size_t)p.b_stages * p.b_stage_bytes + 1024;
  const int grid = p.total_tiles < sms ? p.total_tiles : sms;
  ::b200::launch_kernel(conv_flat_kernel, grid, kThreads, smem, as_stream(stream), p);
  B200_LAUNCH_CHECK();
  return 0;
}

extern "C" int b200_pad_copy(void* dst_flat, int32_t dst_c, int32_t dst_coff, const void* src_dense,
                             int32_t src_c, int32_t src_coff, int32_t n, int32_t h, int32_t w,
                             int32_t c, b200_stream_t stream) {
  B200_REQUIRE(c % 8 == 0 && dst_c % 8 == 0 && src_c % 8 == 0 && dst_coff % 8 == 0 && src_coff % 8 == 0,
               "b200_pad_copy: channels must be multiples of 8");
  long long total = (long long)n * h * w * (c / 8);
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  ::b200::launch_kernel(pad_copy_kernel, blocks < 1 ? 1 : blocks, 256, 0, as_stream(stream), 
      (__nv_bfloat16*)dst_flat, dst_c, dst_coff, (const __nv_bfloat16*)src_dense, src_c, src_coff, n, h, w, c);
  B200_LAUNCH_CHECK();
  return 0;
}

extern "C" int b200_unpad_add(void* dst_dense, int32_t dst_c, const void* src_flat, int32_t src_c,
                              int32_t src_coff, const void* add_dense, int32_t add_c, int32_t n,
                              int32_t h, int32_t w, int32_t c, b200_stream_t stream) {
  B200_REQUIRE(c % 8 == 0 && dst_c % 8 == 0 && src_c % 8 == 0 && src_coff % 8 == 0 && add_c % 8 == 0,
               "b200_unpad_add: channels must be multiples of 8");
  long long total = (long long)n * h * w * (c / 8);
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  ::b200::launch_kernel(unpad_add_kernel, blocks < 1 ? 1 : blocks, 256, 0, as_stream(stream), 
      (__nv_bfloat16*)dst_dense, dst_c, (const __nv_bfloat16*)src_flat, src_c, src_coff,
      (const __nv_bfloat16*)add_dense, add_c, n, h, w, c);
  B200_LAUNCH_CHECK();
  return 0;
}
