// Batched weight gradient of ALL residual dense blocks in one launch (sm_100a, tcgen05).
//
// Per RDB r (flat, zero-bordered layout, P = n*(h+2)*(w+2) positions):
//   X  = B[r]            [P, 192]   inputs of conv1..conv5 (channel prefixes 64/96/128/160/192)
//   dY = G[r][:, 64:192] [P, 128]   pre-activation gradients of conv1..conv4 (32 channels each)
//   dO = G[r+1][:, 0:64] [P, 64]    gradient of the RDB output (conv5's dY up to the factor `a`)
//   dW_k[co][ci][tap] = sum_m X[m + shift(tap), ci] * dYcat[m, co]     (GEMM with K = positions)
// Both operands are consumed MN-major straight from the TMA-landed [rows][64 ch] SWIZZLE_128B tiles;
// the three taps of one kernel row (dx = -1,0,1) share the same smem tiles through row-shifted UMMA
// descriptors, and all five convs of the block share the X tile (the output-channel axis of the
// GEMM is the concatenation of the five dY's), so N is 64..128 instead of 32.
//
// Work item = (rdb, dy, type); three item types cover exactly the needed (ci, co) blocks:
//   T1: D[ci 0..127][3 taps x (dY1..dY4 = 128 co)]     A = X atoms 0,1 (shifted), B = dY atoms 0,1
//   T2: D[ci 0..127][3 taps x (dO = 64 co)]             A = X atoms 0,1 (shifted), B = dO atom
//   T3: D[co' = dY3,dY4,dO (128)][3 taps x ci 128..191] A = dY atom 1 + dO atom, B = X atom 2 (shifted)
// fp32 accumulation in TMEM over all positions (no split-K, no atomics: every (conv, co, ci, tap)
// element is owned by exactly one item), then `+=` into the fp32 OIHW gradient tensors.
//
// Reference: autograd wgrad of the 5 convs of ResidualDenseBlock_5C (RRDBNet_arch.py:130-148).
#include "common.cuh"
#include "colsum.cuh"
#include "sm100_ptx.cuh"

namespace b200 {
namespace {

constexpr int kThreads = 192;
constexpr int kStages = 2;
constexpr int kXRows = 136;                       // 128 + 2 shifted rows, rounded to 8
constexpr uint32_t kXAtom = kXRows * 128;         // 17408 B
constexpr uint32_t kYAtom = 128 * 128;            // 16384 B
constexpr uint32_t kStageBytes = 2 * kXAtom + 2 * kYAtom;  // 67584 B (T1 is the largest)

struct RdbItemParams {
  const CUtensorMap* maps;     // device table: per rdb [x_map (box 64 x 136), g_map (box 64 x 128), do_map (box 64 x 128)]
  const b200_wgrad_rdb_entry* rdbs;  // device table
  int n_rdb, P, Wp, k_steps, total_items;
  int nf, gc;
  int k_split, k_per;   // positions are split into k_split slices of k_per k-steps (see the host entry)
  float* ws;            // [k_split][n_rdb][kSlabFloats] partial sums (nullptr when k_split == 1)
};

__device__ __forceinline__ void item_decode(const RdbItemParams& p, int item, int& r, int& dy, int& type,
                                            int& ks0, int& ks1, int* slice_out = nullptr) {
  // heaviest type first so that the static round-robin schedule balances; the 9 * k_split items of one
  // RDB are adjacent so that the CTAs running at any moment share the same two or three RDBs' tensors
  type = item % 3;
  int q = item / 3;
  dy = q % 3 - 1;
  q /= 3;
  const int slice = q % p.k_split;
  r = q / p.k_split;
  ks0 = slice * p.k_per;
  ks1 = ks0 + p.k_per < p.k_steps ? ks0 + p.k_per : p.k_steps;
  if (slice_out) *slice_out = slice;
}

// tap-major slab of one RDB in the split workspace: conv k at slab_off(k), element ((tap * cout_k + co) * cin_k + ci)
constexpr int kSlabFloats = 9 * (32 * 64 + 32 * 96 + 32 * 128 + 32 * 160 + 64 * 192);   // 239616 (nf = 64, gc = 32)
__host__ __device__ __forceinline__ int slab_off(int k, int nf, int gc) {
  // 9 * gc * sum_{k' < k} (nf + k' gc)
  return 9 * gc * (k * nf + gc * (k * (k - 1) / 2));
}

__global__ void __launch_bounds__(kThreads, 1)
wgrad_rdb_kernel(const __grid_constant__ RdbItemParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem =
      reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[kStages], empty_bar[kStages], tfull_bar, tempty_bar;
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&tfull_bar, 1);
    mbar_init(&tempty_bar, 4);
    mbar_fence_init();
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

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    for (int item = blockIdx.x; item < p.total_items; item += gridDim.x) {
      int r, dy, type, ks0, ks1;
      item_decode(p, item, r, dy, type, ks0, ks1);
      const CUtensorMap* xm = p.maps + 3 * r;
      const CUtensorMap* gm = xm + 1;
      const CUtensorMap* om = xm + 2;
      for (int ks = ks0; ks < ks1; ++ks) {
        const int m0 = ks * 128;
        const int xr = m0 + dy * p.Wp - 1;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elect_one()) {
          uint8_t* s0 = smem + (size_t)stage * kStageBytes;
          if (type == 0) {          // X atoms 0,1 | dY atoms 0,1
            mbar_expect_tx(&full_bar[stage], 2 * kXAtom + 2 * kYAtom);
            tma_load_2d(s0, xm, &full_bar[stage], 0, xr);
            tma_load_2d(s0 + kXAtom, xm, &full_bar[stage], 64, xr);
            tma_load_2d(s0 + 2 * kXAtom, gm, &full_bar[stage], p.nf, m0);
            tma_load_2d(s0 + 2 * kXAtom + kYAtom, gm, &full_bar[stage], p.nf + 64, m0);
          } else if (type == 1) {   // X atoms 0,1 | dO
            mbar_expect_tx(&full_bar[stage], 2 * kXAtom + kYAtom);
            tma_load_2d(s0, xm, &full_bar[stage], 0, xr);
            tma_load_2d(s0 + kXAtom, xm, &full_bar[stage], 64, xr);
            tma_load_2d(s0 + 2 * kXAtom, om, &full_bar[stage], 0, m0);
          } else {                  // dY atom 1 (dY3,dY4), dO | X atom 2
            mbar_expect_tx(&full_bar[stage], 2 * kYAtom + kXAtom);
            tma_load_2d(s0, gm, &full_bar[stage], p.nf + 64, m0);
            tma_load_2d(s0 + kYAtom, om, &full_bar[stage], 0, m0);
            tma_load_2d(s0 + 2 * kYAtom, xm, &full_bar[stage], 128, xr);
          }
        }
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    const uint32_t smem_base = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0, acc_phase = 0;
    for (int item = blockIdx.x; item < p.total_items; item += gridDim.x) {
      int r, dy, type, ks0, ks1;
      item_decode(p, item, r, dy, type, ks0, ks1);
      const int N = (type == 0) ? 128 : 64;
      const uint32_t idesc = make_idesc_bf16(128, N, 1, 1);
      mbar_wait(&tempty_bar, acc_phase ^ 1);
      tc_fence_after();
      for (int ks = ks0; ks < ks1; ++ks) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t s0 = smem_base + stage * kStageBytes;
        if (elect_one()) {
          // A/B bases, atom strides (LBO) and which operand carries the tap shift
          uint32_t a_base, b_base, a_lbo, b_lbo;
          int a_shift, b_shift;
          if (type == 2) {
            a_base = s0; a_lbo = kYAtom; a_shift = 0;
            b_base = s0 + 2 * kYAtom; b_lbo = kXAtom; b_shift = 1;
          } else {
            a_base = s0; a_lbo = kXAtom; a_shift = 1;
            b_base = s0 + 2 * kXAtom; b_lbo = kYAtom; b_shift = 0;
          }
          const uint64_t a_hi = make_smem_desc(0, a_lbo, 1024, LAYOUT_SW128, 0);
          const uint64_t b_hi = make_smem_desc(0, b_lbo, 1024, LAYOUT_SW128, 0);
#pragma unroll
          for (int t = 0; t < 3; ++t) {       // dx = t - 1 ; shifted operand starts at row (1 + dx) = t
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const uint32_t a_addr = a_base + (uint32_t)((a_shift ? t : 0) + k * 16) * 128;
              const uint32_t b_addr = b_base + (uint32_t)((b_shift ? t : 0) + k * 16) * 128;
              const uint64_t ad = a_hi | (uint64_t)((a_addr >> 4) & 0x3FFF);
              const uint64_t bd = b_hi | (uint64_t)((b_addr >> 4) & 0x3FFF);
              umma_f16(tmem + t * N, ad, bd, idesc, ks != ks0 || k != 0);
            }
          }
          umma_commit(&empty_bar[stage]);
          if (ks == ks1 - 1) umma_commit(&tfull_bar);
        }
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      acc_phase ^= 1;
    }
  } else {
    // ------------------------------------------------------------ epilogue (warps 2..5)
    const int quad = warp & 3;
    const int row = quad * 32 + lane;   // accumulator row: ci (T1, T2) or concatenated co' (T3)
    uint32_t acc_phase = 0;
    const int nf = p.nf, gc = p.gc;
    for (int item = blockIdx.x; item < p.total_items; item += gridDim.x) {
      int r, dy, type, ks0, ks1, slice;
      item_decode(p, item, r, dy, type, ks0, ks1, &slice);
      const b200_wgrad_rdb_entry e = p.rdbs[r];
      const int N = (type == 0) ? 128 : 64;
      mbar_wait(&tfull_bar, acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem + ((uint32_t)(quad * 32) << 16);
      if (p.ws && nf == 64 && gc == 32) {
        // Split-workspace path, specialised for the (64, 32) RDB the slab layout assumes: no per-element index
        // arithmetic (the generic loop below spends ~90 k cycles per item on divisions and branches, and this
        // epilogue is NOT overlapped -- one accumulator set fills TMEM), x32 TMEM loads issued one block ahead.
        float* slab = p.ws + ((size_t)slice * p.n_rdb + r) * kSlabFloats;
        const int nblk = 3 * (N / 32);          // 32-column blocks over the three taps
        uint32_t v0[32], v1[32];
        auto issue = [&](uint32_t* dst, int b) {
          tmem_ld_32x32b_x32(t_row + (b / (N / 32)) * N + (b % (N / 32)) * 32, dst);
        };
        auto emit = [&](const uint32_t* vv, int b) {
          const int t = b / (N / 32), c0 = (b % (N / 32)) * 32;
          const int tap = (dy + 1) * 3 + t;
          if (type == 0) {            // row = ci < 128 ; block c0/32 = conv k (cout 32, cin 64 + 32 k)
            const int k = c0 >> 5, cin_k = 64 + 32 * k;
            if (row < cin_k) {
              float* d = slab + slab_off(k, 64, 32) + (size_t)(tap * 32) * cin_k + row;
#pragma unroll
              for (int j = 0; j < 32; ++j) d[(size_t)j * cin_k] = __uint_as_float(vv[j]);
            }
          } else if (type == 1) {     // conv5: ci = row < 128, co = c0 + j
            float* d = slab + slab_off(4, 64, 32) + (size_t)(tap * 64 + c0) * 192 + row;
#pragma unroll
            for (int j = 0; j < 32; ++j) d[(size_t)j * 192] = __uint_as_float(vv[j]);
          } else {                    // row = co' in [dY3 | dY4 | dO], columns = ci - 128
            if (row >= 64) {          // dO -> conv5, ci = 128 + c0 + j
              float4* d = reinterpret_cast<float4*>(slab + slab_off(4, 64, 32) + (size_t)(tap * 64 + row - 64) * 192 + 128 + c0);
#pragma unroll
              for (int j = 0; j < 8; ++j)
                d[j] = make_float4(__uint_as_float(vv[4 * j]), __uint_as_float(vv[4 * j + 1]),
                                   __uint_as_float(vv[4 * j + 2]), __uint_as_float(vv[4 * j + 3]));
            } else if (row >= 32 && c0 == 0) {   // dY4 -> conv4 (cin 160): ci = 128 .. 159
              float4* d = reinterpret_cast<float4*>(slab + slab_off(3, 64, 32) + (size_t)(tap * 32 + row - 32) * 160 + 128);
#pragma unroll
              for (int j = 0; j < 8; ++j)
                d[j] = make_float4(__uint_as_float(vv[4 * j]), __uint_as_float(vv[4 * j + 1]),
                                   __uint_as_float(vv[4 * j + 2]), __uint_as_float(vv[4 * j + 3]));
            }                         // dY3 -> conv3 has only 128 inputs: nothing here
          }
        };
        issue(v0, 0);
        for (int b = 0; b < nblk; b += 2) {   // nblk is even (6 or 12): static ping-pong, no local-memory arrays
          tmem_ld_wait();
          issue(v1, b + 1);
          emit(v0, b);
          tmem_ld_wait();
          if (b + 2 < nblk) issue(v0, b + 2);
          emit(v1, b + 1);
        }
      } else
      for (int t = 0; t < 3; ++t) {
        const int tap = (dy + 1) * 3 + t;
        for (int c0 = 0; c0 < N; c0 += 16) {
          uint32_t v16[16];
          tmem_ld_32x32b_x16(t_row + t * N + c0, v16);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int col = c0 + j;
            // element (conv k, co, ci) of this tap; no atomics: it is owned by exactly one item per position slice
            int k = -1, co = 0, ci = 0;
            if (type == 0) {            // row = ci < 128 ; col -> conv k = col/gc, co = col % gc
              k = col / gc;
              co = col - k * gc;
              ci = row;
              if (row >= nf + k * gc) k = -1;
            } else if (type == 1) {     // conv5: ci = row < 128, co = col
              k = 4; co = col; ci = row;
            } else {                    // row = co' in [dY3 | dY4 | dO], col -> ci = 128 + col
              ci = 2 * nf + col;        // nf = 64: X atom 2 starts at channel 128
              if (row >= 2 * gc) {      // dO -> conv5
                k = 4; co = row - 2 * gc;
              } else if (row >= gc && ci < nf + 3 * gc) {   // dY4 -> conv4 (cin 160)
                k = 3; co = row - gc;
              }                         // dY3 -> conv3 has only 128 inputs: nothing here
            }
            if (k >= 0) {
              const int cin_k = nf + k * gc, cout_k = (k == 4) ? nf : gc;
              const float v = __uint_as_float(v16[j]);
              if (p.ws) {   // tap-major slab of this slice: lanes = consecutive ci (types 0, 1) / 16 consecutive ci per thread (type 2)
                p.ws[((size_t)slice * p.n_rdb + r) * kSlabFloats + slab_off(k, nf, gc) + ((size_t)tap * cout_k + co) * cin_k + ci] = v;
              } else {
                e.dw[k][((size_t)co * cin_k + ci) * 9 + tap] += (k == 4 ? e.scale5 : 1.f) * v;
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar);
      acc_phase ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// Second pass: dW_k (OIHW) += scale_k * sum over the position slices, in slice order (deterministic).
__global__ void __launch_bounds__(256) wgrad_rdb_reduce_kernel(const float* __restrict__ ws,
                                                               const b200_wgrad_rdb_entry* __restrict__ rdbs,
                                                               int n_rdb, int k_split, int nf, int gc) {
  pdl_trigger();
  pdl_wait();
  const int r = blockIdx.y;
  const b200_wgrad_rdb_entry e = rdbs[r];
  const size_t slice_stride = (size_t)n_rdb * kSlabFloats;
  const float* base = ws + (size_t)r * kSlabFloats;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kSlabFloats; i += gridDim.x * blockDim.x) {
    int k = 4;
    while (i < slab_off(k, nf, gc)) --k;
    const int cin_k = nf + k * gc, cout_k = (k == 4) ? nf : gc;
    const int o = i - slab_off(k, nf, gc);
    const int ci = o % cin_k, q = o / cin_k;
    const int co = q % cout_k, tap = q / cout_k;
    float s = 0.f;
    for (int sl = 0; sl < k_split; ++sl) s += base[(size_t)sl * slice_stride + i];
    e.dw[k][((size_t)co * cin_k + ci) * 9 + tap] += (k == 4 ? e.scale5 : 1.f) * s;
  }
}

__global__ void __launch_bounds__(256) colsum_multi_kernel(const b200_colsum_entry* __restrict__ table,
                                                           float* __restrict__ part, unsigned* __restrict__ counters,
                                                           int c_max) {
  pdl_trigger();
  pdl_wait();
  __shared__ float red[256 * 8];
  const b200_colsum_entry e = table[blockIdx.y];
  const int stride = gridDim.x + det_groups(gridDim.x);
  colsum_vec(reinterpret_cast<const __nv_bfloat16*>(e.src), e.npix, e.pitch, e.coff, e.c, e.scale, e.dst, red,
             part + (size_t)blockIdx.y * stride * c_max, counters + blockIdx.y * (1 + det_groups(gridDim.x)));
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" int b200_colsum_multi(const b200_colsum_entry* table_dev, int32_t count, b200_stream_t stream) {
  if (count <= 0) return 0;
  B200_REQUIRE(table_dev, "b200_colsum_multi: null table");
  // entries must have c % 8 == 0, c <= c_max = 256, pitch % 8 == 0, coff % 8 == 0 (16-byte vector loads)
  const int c_max = 256;
  dim3 grid(32, count);
  DetScratch ds;
  if (det_scratch(&ds, (size_t)count * (32 + det_groups(32)) * c_max, count * (1 + det_groups(32)))) return 1;
  ::b200::launch_kernel(colsum_multi_kernel, grid, 256, 0, as_stream(stream), table_dev, ds.part, ds.counters, c_max);
  B200_LAUNCH_CHECK();
  return 0;
}

extern "C" int b200_wgrad_rdb_make_maps(void* maps_host, int32_t n_rdb, const void* const* x_ptrs,
                                        const void* const* g_ptrs, const void* const* do_ptrs,
                                        const int32_t* do_pitch, int32_t n, int32_t h, int32_t w,
                                        int32_t c) {
  B200_REQUIRE(maps_host && x_ptrs && g_ptrs && do_ptrs && do_pitch, "b200_wgrad_rdb_make_maps: null argument");
  CUtensorMap* m = reinterpret_cast<CUtensorMap*>(maps_host);
  const uint64_t P = (uint64_t)n * (h + 2) * (w + 2);
  for (int r = 0; r < n_rdb; ++r) {
    uint64_t dims[2] = {(uint64_t)c, P};
    uint64_t strides[1] = {(uint64_t)c * 2};
    uint32_t boxx[2] = {64, (uint32_t)kXRows};
    uint32_t boxy[2] = {64, 128};
    if (make_tensor_map(&m[3 * r], x_ptrs[r], 2, dims, strides, boxx, nullptr, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    if (make_tensor_map(&m[3 * r + 1], g_ptrs[r], 2, dims, strides, boxy, nullptr, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    uint64_t dimso[2] = {64, P};
    uint64_t strideso[1] = {(uint64_t)do_pitch[r] * 2};
    if (make_tensor_map(&m[3 * r + 2], do_ptrs[r], 2, dimso, strideso, boxy, nullptr, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  return 0;
}

namespace {
// Split-K for L2 locality, not for parallelism: with one item per (rdb, kernel row, type) the 148 CTAs
// would stream 16 different RDBs (53 MB of X/dY each) at once and every operand byte would come from
// HBM (18.6 GB per launch at config 2).  With S slices the CTAs in flight cover 16/S RDBs.  Each slice
// writes its own tap-major slab of the caller's workspace with plain coalesced stores and a second kernel adds
// the slabs in slice order: deterministic (round 1 used fp32 atomics: S=1 3.76 ms, S=4 3.41 ms, S=8 4.32 ms
// because of the exposed atomic epilogue; operand phase alone 2.55 ms for S >= 4).
constexpr int kSplit = 4;   // measured (deterministic slabs): S=1 3.76 ms, S=4 3.31 ms, S=8 4.09 ms
void rdb_split(int k_steps, int* k_split, int* k_per) {
  int s = kSplit < k_steps ? kSplit : 1;
  *k_per = (k_steps + s - 1) / s;
  *k_split = (k_steps + *k_per - 1) / *k_per;   // no empty slices
}
}  // namespace

extern "C" int64_t b200_wgrad_rdb_ws_bytes(int32_t n_rdb, int32_t n, int32_t h, int32_t w) {
  const long long P = (long long)n * (h + 2) * (w + 2);
  int k_split, k_per;
  rdb_split((int)((P + 127) / 128), &k_split, &k_per);
  return k_split > 1 ? (int64_t)k_split * n_rdb * kSlabFloats * (int64_t)sizeof(float) : 0;
}

extern "C" int b200_wgrad_rdb(const void* maps_dev, const b200_wgrad_rdb_entry* entries_dev, int32_t n_rdb,
                              int32_t n, int32_t h, int32_t w, int32_t nf, int32_t gc, void* workspace,
                              int64_t ws_bytes, b200_stream_t stream) {
  B200_REQUIRE(maps_dev && entries_dev && n_rdb > 0, "b200_wgrad_rdb: null argument");
  B200_REQUIRE(nf == 64 && gc == 32, "b200_wgrad_rdb: the fused RDB weight-gradient kernel is specialised for nf=64, gc=32");
  const int kSmemBytes = kStages * kStageBytes + 1024;
  B200_ENSURE_SMEM(wgrad_rdb_kernel, kSmemBytes);
  RdbItemParams p;
  p.maps = reinterpret_cast<const CUtensorMap*>(maps_dev);
  p.rdbs = entries_dev;
  p.n_rdb = n_rdb;
  const long long P = (long long)n * (h + 2) * (w + 2);
  p.P = (int)P;
  p.Wp = w + 2;
  p.k_steps = (int)((P + 127) / 128);
  rdb_split(p.k_steps, &p.k_split, &p.k_per);
  p.total_items = n_rdb * 9 * p.k_split;
  p.nf = nf;
  p.gc = gc;
  p.ws = nullptr;
  if (p.k_split > 1) {
    const int64_t need = b200_wgrad_rdb_ws_bytes(n_rdb, n, h, w);
    B200_REQUIRE(workspace && ws_bytes >= need, "b200_wgrad_rdb: workspace of %lld bytes needed (b200_wgrad_rdb_ws_bytes)",
                 (long long)need);
    p.ws = reinterpret_cast<float*>(workspace);
  }
  const int sms = sm_count();
  const int grid = p.total_items < sms ? p.total_items : sms;
  ::b200::launch_kernel(wgrad_rdb_kernel, grid, kThreads, kSmemBytes, as_stream(stream), p);
  B200_LAUNCH_CHECK();
  if (p.ws) {
    dim3 rg(16, n_rdb);
    ::b200::launch_kernel(wgrad_rdb_reduce_kernel, rg, 256, 0, as_stream(stream), (const float*)p.ws, entries_dev, n_rdb,
                          p.k_split, nf, gc);
    B200_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int b200_tensor_map_bytes(void) { return (int)sizeof(CUtensorMap); }
