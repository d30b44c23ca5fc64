// Whole-trunk residual-dense-block chain in ONE persistent launch (sm_100a: tcgen05 + TMEM + TMA + clusters/DSMEM).
//
// A dense block is 5 stacked 3x3 convs where conv_k consumes [x, x1 .. x_{k-1}].  Computed conv by conv, four of them
// have only 32 output channels and tcgen05.mma is shared-memory-operand bound at 40 % of the tensor pipe (N = 32;
// profiles/r01_umma_pipe_probe.log).  Here a block is computed INPUT SLICE by input slice:
//   stage j consumes the newest slice S_j (x for j = 0, then x1..x4) and adds its contribution to ALL convs that still
//   need it:  D[:, 32j:192] += S_j (*) W_stage_j      (N = 192 - 32 j, K = 64 or 32 per tap)
// and the fp32 partial sums of a CTA's 256-position super-tile (two 128-row halves x 192 columns) stay in TMEM for
// the whole block.  After stage j the 32 (last stage: 64) columns that just became complete are finished (bias /
// LeakyReLU or mask / residuals), written to HBM (saved activation / gradient) and -- as bf16, already in the
// 128B-swizzled K-major layout -- straight back into the CTA's own shared-memory operand region: they ARE the next
// stage's A operand.  The output of stage 4 is the x slice of the NEXT block, so the whole trunk (69 blocks x 5
// stages) runs in one launch with the activations never leaving the SM except as stores.
//
// One CTA per super-tile of the flat (zero-bordered) position space, all co-resident; warp roles: TMA weight producer,
// two MMA issuers (one per 128-row half, sharing every weight tile), eight epilogue warps.  The stage weights stream
// through a TMA ring.  A stage is issued in two parts -- first the columns it completes, then the columns of the later
// convs -- so that the turnaround of the finished slice (TMEM -> registers -> smem, halo exchange) overlaps the second
// part on the tensor pipe.  The operand regions rotate (stage s reads region s % 3, fills region (s+1) % 3) so that a
// neighbour's halo rows can never land in rows the tensor core still reads.
//
// Halo rows (the +-(w+3) positions a 3x3 tap reaches beyond the super-tile) belong to the neighbouring CTAs:
//   * inside a thread-block cluster they travel through DISTRIBUTED SHARED MEMORY: one cp.async.bulk
//     shared::cta -> shared::cluster copy per side, straight from this CTA's operand region into the peer's (same
//     swizzle phase: the row offset is 256), completing on the peer's mbarrier;
//   * across cluster edges through L2 in "LL" form: every 16-byte store carries 8 bytes of data and two copies of a
//     4-byte sequence flag (8-byte atomicity), the receiver polls the data itself -- no fence, no separate flag
//     (a separate flag costs store -> fence -> flag -> acquire -> TMA, ~6.5 k cycles per stage in
//     profiles/r01_rdb_persist_timeline.txt).
//
// The gather-form input gradient of a block has exactly the same shape with the slices taken in reverse
// (dO, dY4 .. dY1 -> d(x4) .. d(x)), so the backward trunk is the same kernel with flipped taps.
// Measured history and the in-kernel timeline: DESIGN.md section 4, tools/time_chain.py.
//
// Reference: ResidualDenseBlock_5C.forward + RRDB residuals (RRDBNet_arch.py:89-96,150-163), the ShortcutBlock
// trunk (block.py:184-192) and their autograd input gradients.
#include <stdlib.h>

#include <map>
#include <mutex>

#include "common.cuh"
#include "sm100_ptx.cuh"

namespace b200 {
namespace {

constexpr int kThreads = 352;          // weights producer, 2 MMA issuers, 2 x 4 epilogue warps
constexpr int kTileM = 256;            // positions per CTA: two adjacent 128-row MMA halves sharing one operand region
constexpr int kNTotal = 192;
constexpr int kBStages = 5;            // at most; p.b_stages slots are used (what fits beside the operand regions)
constexpr uint32_t kBStageBytes = 24 * 1024;   // one 64-channel tap tile (24 KB) or 2-3 32-channel tap tiles (<= 24 KB)
constexpr int kLLRowBytes = 256;       // 128 B of data (64 channels) in LL form
constexpr int kMaxHalo = 128;          // w <= 125

struct ChainParams {
  CUtensorMap x_map;       // input of the first block: flat [P rows][>= 64 ch], box (64, box_rows)
  CUtensorMap w_map[5][2]; // stage weights [n_blocks*9 taps][N_j rows][K_j] as 3-D maps; [j][0]: box = all rows (split = 0) or the
                           // rows of the conv stage j completes; [j][1]: the remaining rows (split = 1 only)
  const b200_chain_stage* table;   // [n_blocks][5]
  int n_blocks;
  int x_ch;                // channel offset of the first block's input slice
  int Wp, HpWp, h, w, halo, nbox, box_rows;
  uint32_t a_bytes, a_region_bytes;
  int pos0, range_len, n_tiles;   // first position, positions and 256-position super-tiles of the image group
  int b_stages;            // weight ring slots in use
  int n_regions;           // operand regions in rotation (2, or 3 with split stages)
  int split;               // issue every stage as (completing columns, later convs) -- see part_rows()
  int tap_sign;            // +1 forward taps, -1 input-gradient taps
  uint8_t* ll;             // LL exchange buffers [tile][side][parity][halo rows][256 B]
  uint32_t ll_tile_stride; // bytes per tile
  const uint32_t* epoch;   // launch sequence number (bumped by a 1-thread kernel before this one)
  int cluster_size;        // CTAs per thread-block cluster (1: every halo goes through L2)
  long long* dbg;
};

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

__device__ __forceinline__ void st_shared_v4(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_global_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_volatile_v4(const void* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Operands of a stage epilogue that do not depend on the accumulator, requested BEFORE the wait on the MMAs.
struct EpiPre {
  uint4 lm[4], l1[4], l2[4];
  float4 b[8];
};

__device__ __forceinline__ void prefetch32(const b200_chain_stage& e, EpiPre& q, int c0, long long m) {
  const __nv_bfloat16* mask = reinterpret_cast<const __nv_bfloat16*>(e.mask);
  const __nv_bfloat16* res1 = reinterpret_cast<const __nv_bfloat16*>(e.res1);
  const __nv_bfloat16* res2 = reinterpret_cast<const __nv_bfloat16*>(e.res2);
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const int c = c0 + g * 8;
    if (mask) q.lm[g] = *reinterpret_cast<const uint4*>(mask + m * e.mask_c + e.mask_coff + c);
    if (res1) q.l1[g] = *reinterpret_cast<const uint4*>(res1 + m * e.res1_c + e.res1_coff + c);
    if (res2) q.l2[g] = *reinterpret_cast<const uint4*>(res2 + m * e.res2_c + e.res2_coff + c);
    if (e.bias) {
      q.b[2 * g] = __ldg(reinterpret_cast<const float4*>(e.bias + c));
      q.b[2 * g + 1] = __ldg(reinterpret_cast<const float4*>(e.bias + c + 4));
    }
  }
}

// finish 32 accumulator columns of one row -> 4 packed 16-byte chunks
__device__ __forceinline__ void finish32(const b200_chain_stage& e, const uint32_t* acc, const EpiPre& q, uint4* o) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[g * 8 + j]);
    if (e.bias) {
      const float4 b0 = q.b[2 * g], b1 = q.b[2 * g + 1];
      v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
      v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= e.alpha;
    if (e.res1) {
      float r[8];
      unpack8(q.l1[g], r);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf(e.beta1, r[j], v[j]);
    }
    if (e.res2) {
      float r[8];
      unpack8(q.l2[g], r);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf(e.beta2, r[j], v[j]);
    }
    if (e.act) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * e.slope;
    }
    if (e.mask) {
      float r[8];
      unpack8(q.lm[g], r);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = r[j] > 0.f ? v[j] : v[j] * e.mask_slope;
    }
    o[g] = pack8(v);
  }
}

#define CDBG(slot) do { if (p.dbg && lane == 0) p.dbg[(long long)blockIdx.x * 64 + (slot)] = clock64(); } while (0)

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// bulk copy local shared memory -> a peer CTA's shared memory; completes `bytes` on the PEER's mbarrier
__device__ __forceinline__ void dsmem_push(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes, uint32_t mbar_cluster) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   dst_cluster),
               "r"(src_cta), "r"(bytes), "r"(mbar_cluster)
               : "memory");
}
// A stage may be issued in two parts: part 0 = the 32 (j = 4: 64) accumulator columns that stage j COMPLETES, part 1 =
// the columns of the later convs, so that the epilogue / halo exchange of the completed columns overlaps part 1 on the
// tensor pipe (the N = 32 MMAs of part 0 are shared-memory-operand bound: the price of starting the turnaround early).
// split == 0: one part with all N = 192 - 32 j columns.
__host__ __device__ __forceinline__ int part_rows(int j, int part, int split) {
  if (!split) return part == 0 ? kNTotal - 32 * j : 0;
  return part == 0 ? (j == 4 ? 64 : 32) : (j == 4 ? 0 : kNTotal - 32 * (j + 1));
}
__host__ __device__ __forceinline__ int part_tpb(int rows, int j) {   // taps per 24 KB weight slot
  const int t = (int)kBStageBytes / (rows * (j == 0 ? 128 : 64));
  return t > 9 ? 9 : t;
}

__global__ void __launch_bounds__(kThreads, 1)
rdb_chain_kernel(const __grid_constant__ ChainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem =
      reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // slice_ready[parity]: operand region `parity` complete = 8 epilogue warps (own rows, cluster-edge halos) + 1
  // expect_tx arrival covering the bytes the in-cluster neighbours push through distributed shared memory
  __shared__ uint64_t b_full[kBStages], b_empty[kBStages], init_full, slice_ready[3], acc_ready;
  __shared__ uint32_t tmem_base_s;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int cta = blockIdx.x;
  const int crank = p.cluster_size > 1 ? (int)cluster_ctarank() : 0;
  const bool active = cta < p.n_tiles;   // CTAs that only pad the grid to a multiple of the cluster size do nothing
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.b_stages; ++s) {
      mbar_init(&b_full[s], 1);
      mbar_init(&b_empty[s], 2);       // both MMA issuers
    }
    mbar_init(&init_full, 1);
    for (int i = 0; i < 3; ++i) mbar_init(&slice_ready[i], 9);
    mbar_init(&acc_ready, 2);
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_base_s, 512);
    tmem_relinquish();
  }
  // Operand regions rotate: stage s reads region s % nreg, its epilogue (and the neighbours) fill region (s+1) % nreg.
  // nreg = 2 suffices when a stage is issued in one piece; with split stages the later-conv MMAs of stage s-1 may still
  // read region (s-1) % nreg while a neighbour already pushes its stage-s halo rows, so three regions rotate.
  // halo rows of the never TMA-loaded regions start as zeros: at the ends of the position range nobody
  // ever writes them (the neighbouring positions are border rows of other images)
  const int nreg = p.n_regions;
  for (int i = threadIdx.x; i < (nreg - 1) * 2 * p.halo * 8; i += kThreads) {
    const int reg = 1 + i / (2 * p.halo * 8), k = i % (2 * p.halo * 8);
    const int row = k >> 3, ch = k & 7;
    const uint32_t R = row < p.halo ? (uint32_t)row : (uint32_t)(kTileM + row);
    *reinterpret_cast<uint4*>(smem + (size_t)reg * p.a_region_bytes + (size_t)R * 128 + ch * 16) = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (p.cluster_size > 1) cluster_sync_all();   // every CTA's barriers are initialised before any peer pushes into it
  const uint32_t tmem = tmem_base_s;
  const uint32_t b_ring_off = (uint32_t)nreg * p.a_region_bytes;
  const int n_stages_total = p.n_blocks * 5;
  if (warp == 0) CDBG(0);

  if (warp == 0) {
    // ------------------------------------------------------------ producer: initial operand region, then weights
    if (active) {
      if (elect_one()) {
        tma_prefetch_desc(&p.x_map);
        for (int j = 0; j < 5; ++j) {
          tma_prefetch_desc(&p.w_map[j][0]);
          if (p.split && j < 4) tma_prefetch_desc(&p.w_map[j][1]);
        }
        const int row0 = p.pos0 + cta * kTileM - p.halo;
        mbar_expect_tx(&init_full, p.a_bytes);
        for (int bx = 0; bx < p.nbox; ++bx)
          tma_load_2d(smem + (size_t)bx * p.box_rows * 128, &p.x_map, &init_full, p.x_ch, row0 + bx * p.box_rows);
      }
      __syncwarp();
      int bs = 0;
      uint32_t bph = 0;
      for (int blk = 0; blk < p.n_blocks; ++blk) {
        for (int j = 0; j < 5; ++j) {
          for (int part = 0; part < 2; ++part) {
            const int rows = part_rows(j, part, p.split);
            if (rows == 0) continue;
            const int tpb = part_tpb(rows, j);
            const uint32_t tap_bytes = (uint32_t)rows * (j == 0 ? 128 : 64);
            const int row0 = part == 0 ? 0 : part_rows(j, 0, p.split);
            for (int t0 = 0; t0 < 9; t0 += tpb) {
              const int nt = (9 - t0) < tpb ? (9 - t0) : tpb;
              mbar_wait(&b_empty[bs], bph ^ 1);
              if (elect_one()) {
                mbar_expect_tx(&b_full[bs], tap_bytes * nt);
                for (int q = 0; q < nt; ++q)
                  tma_load_3d(smem + b_ring_off + (size_t)bs * kBStageBytes + (size_t)q * tap_bytes, &p.w_map[j][part],
                              &b_full[bs], 0, row0, blk * 9 + t0 + q);
              }
              __syncwarp();
              if (++bs == p.b_stages) {
                bs = 0;
                bph ^= 1;
              }
            }
          }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ------------------------------------------------------------ MMA issuer of half (warp - 1): rows [128 half, +128)
    const int half = warp - 1;
    if (active) {
      const uint64_t desc_hi = make_smem_desc(0, 16, 1024, LAYOUT_SW128, 0);
      const uint64_t desc_b64 = make_smem_desc(0, 16, 512, LAYOUT_SW64, 0);   // 32-channel weight tiles: 64-byte rows
      const uint32_t smem_base = smem_u32(smem);
      const uint32_t d_half = tmem + half * kNTotal;
      uint32_t sh16[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) sh16[t] = (uint32_t)((p.tap_sign * ((t / 3 - 1) * p.Wp + (t % 3 - 1))) * 8);   // 128-B rows in 16-B units
      int bs = 0;
      uint32_t bph = 0;
      for (int s = 0; s < n_stages_total; ++s) {
        const int j = s % 5;
        if (s == 0) {
          mbar_wait(&init_full, 0);
        } else {
          mbar_wait(&slice_ready[s % nreg], (uint32_t)(((s - 1) / nreg) & 1));
        }
        tc_fence_after();
        if (s < 7 && half == 0) CDBG(2 + 8 * s);   // operand slice ready
        const uint32_t a16 = (smem_base + (uint32_t)(s % nreg) * p.a_region_bytes + (uint32_t)(p.halo + half * 128) * 128) >> 4;
        const int nk = (j == 0) ? 4 : 2;
        const uint64_t bdesc_hi = (j == 0) ? desc_hi : desc_b64;
        for (int part = 0; part < 2; ++part) {
          const int rows = part_rows(j, part, p.split);
          if (rows == 0) continue;
          const uint32_t idesc = make_idesc_bf16(128, rows, 0, 0);
          const uint32_t d_tmem = d_half + 32 * j + (part ? part_rows(j, 0, p.split) : 0);
          const int tpb = part_tpb(rows, j);
          const uint32_t tap16 = ((uint32_t)rows * (j == 0 ? 128 : 64)) >> 4;
          for (int t0 = 0; t0 < 9; t0 += tpb) {
            const int nt = (9 - t0) < tpb ? (9 - t0) : tpb;
            mbar_wait(&b_full[bs], bph);
            tc_fence_after();
            const uint32_t b16 = (smem_base + b_ring_off + bs * kBStageBytes) >> 4;
            if (elect_one()) {
              for (int q = 0; q < nt; ++q) {
                const uint32_t at = a16 + sh16[t0 + q], bt = b16 + q * tap16;
                // the first tap of a block's first stage zero-initialises the accumulator columns of its part
                if (nk == 4) {
#pragma unroll
                  for (int k = 0; k < 4; ++k)
                    umma_f16(d_tmem, desc_hi | (uint64_t)((at + 2 * k) & 0x3FFF), bdesc_hi | (uint64_t)((bt + 2 * k) & 0x3FFF), idesc,
                             ((t0 + q) | k) != 0);
                } else {
#pragma unroll
                  for (int k = 0; k < 2; ++k)
                    umma_f16(d_tmem, desc_hi | (uint64_t)((at + 2 * k) & 0x3FFF), bdesc_hi | (uint64_t)((bt + 2 * k) & 0x3FFF), idesc, 1u);
                }
              }
              umma_commit(&b_empty[bs]);
              if (part == 0 && t0 + tpb >= 9) umma_commit(&acc_ready);   // the completing columns of this half are done
            }
            __syncwarp();
            if (++bs == p.b_stages) {
              bs = 0;
              bph ^= 1;
            }
          }
        }
        if (s < 7 && half == 0) CDBG(3 + 8 * s);   // stage MMAs issued
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 3..10: one 256-row super-tile
    if (active) {
      const int ew = warp - 3;                              // 0..7
      const int quad = warp & 3;                            // TMEM lane quadrant this warp may read
      const int half = ew >> 2;                             // warps 3..6 -> rows [0,128), 7..10 -> rows [128,256)
      const int r = half * 128 + quad * 32 + lane;          // row of the super-tile
      const int et = ew * 32 + lane;                        // 0..255: index among the epilogue threads
      const int lpos = cta * kTileM + r;                    // position within the range
      const long long m = (long long)p.pos0 + lpos;
      const int rem = (int)(m % p.HpWp);
      const int yp = rem / p.Wp, xp = rem - yp * p.Wp;
      const bool valid = lpos < p.range_len && yp >= 1 && yp <= p.h && xp >= 1 && xp <= p.w;
      const bool has_up = cta > 0, has_dn = cta + 1 < p.n_tiles;
      // neighbours inside the cluster are reached through distributed shared memory, the others through L2 (LL)
      const bool ds_up = has_up && crank > 0, ds_dn = has_dn && crank + 1 < p.cluster_size;
      const bool ll_up = has_up && !ds_up, ll_dn = has_dn && !ds_dn;
      const uint32_t t_row = tmem + ((uint32_t)(quad * 32) << 16) + half * kNTotal;
      const uint32_t region0 = smem_u32(smem);
      const uint32_t own_row = (uint32_t)(p.halo + r);
      const uint32_t own_xor = own_row & 7;
      uint8_t* ll_me = p.ll + (size_t)cta * p.ll_tile_stride;
      uint8_t* ll_upb = ll_me - p.ll_tile_stride;   // receive buffers of the super-tiles above / below
      uint8_t* ll_dnb = ll_me + p.ll_tile_stride;
      const uint32_t side_bytes = (uint32_t)p.halo * kLLRowBytes;   // one (side, parity) buffer
      const uint32_t flag0 = (*p.epoch) << 12;
      const uint32_t push_bytes = (uint32_t)p.halo * 128;
      const uint32_t ds_in_bytes = ((ds_up ? 1u : 0u) + (ds_dn ? 1u : 0u)) * push_bytes;
      // rows [0, halo) (needed by the super-tile above) and [256 - halo, 256) (below) and the warps that own them
      const bool in_top = r < p.halo, in_bot = r >= kTileM - p.halo;
      const bool top_member = half == 0 && quad * 32 < p.halo;
      const bool bot_member = half == 1 && (quad + 1) * 32 > 128 - p.halo;
      const int top_count = (p.halo + 31) / 32 < 4 ? (p.halo + 31) / 32 : 4;
      const int bot_count = 4 - ((128 - p.halo) > 0 ? (128 - p.halo) / 32 : 0);
      uint32_t acc_ph = 0;
      for (int s = 0; s < n_stages_total; ++s) {
        const int j = s % 5;
        const b200_chain_stage e = p.table[s];
        const int nch = (j == 4) ? 8 : 4;              // 16-byte chunks of the finished slice (64 or 32 channels)
        const uint32_t flag = flag0 + (uint32_t)s + 1u;
        const int par = s & 1, pn = (s + 1) % nreg;    // LL buffer parity; the finished slice becomes operand region `pn`
        const bool more = s + 1 < n_stages_total;
        const uint32_t region = region0 + (uint32_t)pn * p.a_region_bytes;
        const uint32_t own_addr = region + own_row * 128;
        if (more && et == 0) {
          // this phase of slice_ready[pn] also waits for the bytes the in-cluster neighbours push
          if (ds_in_bytes) mbar_expect_tx(&slice_ready[pn], ds_in_bytes);
          else mbar_arrive(&slice_ready[pn]);
        }
        EpiPre q;
        if (valid) prefetch32(e, q, 0, m);
        mbar_wait(&acc_ready, acc_ph);
        acc_ph ^= 1;
        tc_fence_after();
        if (s < 7 && warp == 3) CDBG(4 + 8 * s);   // stage MMAs (completing columns) done
        __nv_bfloat16* outp = reinterpret_cast<__nv_bfloat16*>(e.out);
        for (int c0 = 0; c0 < nch * 8; c0 += 32) {
          uint32_t acc[32];
          tmem_ld_32x32b_x32(t_row + 32 * j + c0, acc);
          if (c0 > 0 && valid) prefetch32(e, q, c0, m);
          tmem_ld_wait();
          if (s < 7 && warp == 3 && c0 == 0) CDBG(7 + 8 * s);
          uint4 o[4];
          if (valid) {
            finish32(e, acc, q, o);
          } else {
#pragma unroll
            for (int g = 0; g < 4; ++g) o[g] = make_uint4(0, 0, 0, 0);   // border / out-of-range positions stay zero
          }
          if (s < 7 && warp == 3 && c0 == 0) CDBG(8 + 8 * s);
          const int cb = c0 >> 3;   // first chunk index
          // (1) own rows of the next operand slice, 128B-swizzled K-major (the in-cluster halo pushes read them)
          if (more) {
#pragma unroll
            for (int g = 0; g < 4; ++g) st_shared_v4(own_addr + ((uint32_t)((cb + g) ^ own_xor) << 4), o[g]);
          }
          // (2) halo rows for neighbours in OTHER clusters through L2 (LL: data + flag in every 8 bytes)
          if (more && ll_up && in_top) {
            uint8_t* dst = ll_upb + (1 * 2 + par) * side_bytes + (size_t)r * kLLRowBytes + cb * 32;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              st_global_v4(dst + g * 32, o[g].x, flag, o[g].y, flag);
              st_global_v4(dst + g * 32 + 16, o[g].z, flag, o[g].w, flag);
            }
          }
          if (more && ll_dn && in_bot) {
            uint8_t* dst = ll_dnb + (0 * 2 + par) * side_bytes + (size_t)(r - (kTileM - p.halo)) * kLLRowBytes + cb * 32;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              st_global_v4(dst + g * 32, o[g].x, flag, o[g].y, flag);
              st_global_v4(dst + g * 32 + 16, o[g].z, flag, o[g].w, flag);
            }
          }
          // (3) saved activation / gradient in HBM
          if (valid && outp) {
            uint4* dst = reinterpret_cast<uint4*>(outp + m * e.out_c + e.out_coff + c0);
#pragma unroll
            for (int g = 0; g < 4; ++g) dst[g] = o[g];
          }
          if (s < 7 && warp == 3 && c0 == 0) CDBG(9 + 8 * s);
        }
        tc_fence_before();
        if (s < 7 && warp == 3) CDBG(6 + 8 * s);   // epilogue math + stores issued
        if (more) {
          fence_proxy_async();   // own rows (generic proxy) -> visible to the bulk-copy engine and the tensor core
          // (4) push the halo rows to the in-cluster neighbours: ONE bulk copy per side, straight from this CTA's operand
          //     region into the peer's (same 128B-swizzle phase: the row offset between the two is 256), completing on
          //     the peer's slice_ready barrier.  Only the warps that own those rows synchronise.
          if (ds_up && top_member) {
            named_bar_sync(1, 32 * top_count);
            if (quad == 0 && lane == 0) {   // my rows [0, halo) -> bottom halo of the super-tile above
              const uint32_t dst = mapa_cluster(region + (uint32_t)(p.halo + kTileM) * 128, (uint32_t)(crank - 1));
              const uint32_t bar = mapa_cluster(smem_u32(&slice_ready[pn]), (uint32_t)(crank - 1));
              dsmem_push(dst, region + (uint32_t)p.halo * 128, push_bytes, bar);
            }
          }
          if (ds_dn && bot_member) {
            named_bar_sync(2, 32 * bot_count);
            if (quad == 3 && lane == 0) {   // my rows [256 - halo, 256) -> top halo of the super-tile below
              const uint32_t dst = mapa_cluster(region, (uint32_t)(crank + 1));
              const uint32_t bar = mapa_cluster(smem_u32(&slice_ready[pn]), (uint32_t)(crank + 1));
              dsmem_push(dst, region + (uint32_t)kTileM * 128, push_bytes, bar);
            }
          }
          // (5) halo rows from neighbours in other clusters: poll the LL buffers (all of a thread's polls in flight
          //     together; items whose flags have not landed are polled again after a short sleep)
          if (ll_up || ll_dn) {
            const int per_side = p.halo * nch;
            constexpr int kBatch = 3;
            for (int base = et; base < 2 * per_side; base += 256 * kBatch) {
              const uint8_t* src[kBatch];
              uint32_t dst[kBatch];
              unsigned pending = 0;
#pragma unroll
              for (int qi = 0; qi < kBatch; ++qi) {
                const int i = base + qi * 256;
                src[qi] = nullptr;
                dst[qi] = 0;
                if (i < 2 * per_side) {
                  const int side = i >= per_side ? 1 : 0;
                  if (side == 0 ? ll_up : ll_dn) {
                    const int k = i - side * per_side;
                    const int row = k / nch, ch = k - row * nch;
                    src[qi] = ll_me + (side * 2 + par) * side_bytes + (size_t)row * kLLRowBytes + ch * 32;
                    const uint32_t R = side == 0 ? (uint32_t)row : (uint32_t)(p.halo + kTileM + row);
                    dst[qi] = region + R * 128 + ((uint32_t)(ch ^ (R & 7)) << 4);
                    pending |= 1u << qi;
                  }
                }
              }
              while (pending) {
                uint4 a[kBatch], b[kBatch];
#pragma unroll
                for (int qi = 0; qi < kBatch; ++qi)
                  if (pending & (1u << qi)) {
                    a[qi] = ld_volatile_v4(src[qi]);
                    b[qi] = ld_volatile_v4(src[qi] + 16);
                  }
#pragma unroll
                for (int qi = 0; qi < kBatch; ++qi)
                  if ((pending & (1u << qi)) && a[qi].y == flag && a[qi].w == flag && b[qi].y == flag && b[qi].w == flag) {
                    st_shared_v4(dst[qi], make_uint4(a[qi].x, a[qi].z, b[qi].x, b[qi].z));
                    pending &= ~(1u << qi);
                  }
                if (pending) __nanosleep(64);
              }
            }
            fence_proxy_async();
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&slice_ready[pn]);
        }
        if (s < 7 && warp == 3) CDBG(5 + 8 * s);   // slice turned around (this warp's part)
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (p.cluster_size > 1) cluster_sync_all();   // no CTA of the cluster exits while a peer may still push into it
  if (warp == 0) CDBG(1);
  if (warp == 1) tmem_dealloc(tmem, 512);
}

__global__ void chain_epoch_bump_kernel(uint32_t* epoch) {
  pdl_trigger();
  pdl_wait();
  *epoch = (*epoch + 1u) & 0xFFFFFu;   // flag = (epoch << 12) + stage + 1 stays below 2^32
  if (*epoch == 0u) *epoch = 1u;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" int b200_rdb_chain_geometry(int32_t n, int32_t h, int32_t w, int32_t* n_cta, int64_t* ll_bytes) {
  const int Hp = h + 2, Wp = w + 2;
  const long long len = (long long)n * Hp * Wp;
  // the last (w + 3) positions of the range are border positions of the last image: a super-tile holding only those has
  // nothing to compute (8 images of 66 x 66: 136 tiles = 34 clusters of 4 instead of 137)
  const int tiles = (int)((len - (Wp + 1) + kTileM - 1) / kTileM);
  if (n_cta) *n_cta = tiles;
  const int halo = Wp + 1;
  if (ll_bytes) *ll_bytes = (int64_t)tiles * 4 * halo * kLLRowBytes;
  // the shared-memory budget: two operand regions + at least three 24 KB weight slots
  const int region = kTileM + 2 * halo;
  const int nbox = (region + 255) / 256;
  const int box_rows = (((region + nbox - 1) / nbox) + 7) & ~7;
  const int a_region = (nbox * box_rows * 128 + 1023) & ~1023;
  return (halo <= kMaxHalo && 2 * a_region + 3 * (int)kBStageBytes + 1024 <= 227 * 1024) ? 0 : 1;
}

// One launch = a chain of n_blocks dense blocks (forward, or gather-form input gradient when flip_taps) over
// the n images starting at image `img0` of the flat tensors.  table_dev: [n_blocks][5] stage descriptors
// (device memory); w_stage[j]: packed stage weights [n_blocks][9][192-32j][K_j] bf16 (K_0 = 64, else 32).
extern "C" int b200_rdb_chain(const b200_chain_desc* d, const void* x0, const void* const* w_stage,
                              const b200_chain_stage* table_dev, void* ll_buf, int64_t ll_bytes,
                              uint32_t* epoch_dev, b200_stream_t stream) {
  B200_REQUIRE(d && x0 && w_stage && table_dev && ll_buf && epoch_dev, "b200_rdb_chain: null argument");
  B200_REQUIRE(d->n >= 1 && d->n_blocks >= 1 && d->w + 3 <= kMaxHalo, "b200_rdb_chain: bad geometry (w <= 128)");
  ChainParams p;
  memset(&p, 0, sizeof(p));
  p.h = d->h; p.w = d->w;
  p.Wp = d->w + 2;
  const int Hp = d->h + 2;
  p.HpWp = Hp * p.Wp;
  p.halo = p.Wp + 1;
  const int region = kTileM + 2 * p.halo;
  p.nbox = (region + 255) / 256;
  p.box_rows = (((region + p.nbox - 1) / p.nbox) + 7) & ~7;
  p.a_bytes = (uint32_t)p.nbox * p.box_rows * 128;
  p.a_region_bytes = (p.a_bytes + 1023) & ~1023u;
  p.split = 1;
  p.n_regions = 3;
  int b_stages = (227 * 1024 - 1024 - p.n_regions * (int)p.a_region_bytes) / (int)kBStageBytes;
  if (b_stages < 3) {   // not enough room for three regions (w >= 70): one-piece stages with two
    p.split = 0;
    p.n_regions = 2;
    b_stages = (227 * 1024 - 1024 - 2 * (int)p.a_region_bytes) / (int)kBStageBytes;
  }
  if (b_stages > kBStages) b_stages = kBStages;
  B200_REQUIRE(b_stages >= 3, "b200_rdb_chain: image too wide for the shared-memory operand regions (w=%d)", d->w);
  p.b_stages = b_stages;
  const int kSmemBytes = (int)(p.n_regions * p.a_region_bytes + b_stages * kBStageBytes + 1024);
  B200_ENSURE_SMEM(rdb_chain_kernel, kSmemBytes);
  const long long P_total = (long long)d->n_total * p.HpWp;
  p.pos0 = d->img0 * p.HpWp;
  p.range_len = d->n * p.HpWp;
  p.n_tiles = (p.range_len - p.halo + kTileM - 1) / kTileM;   // see b200_rdb_chain_geometry
  const int n_cta = p.n_tiles;
  const int sms = sm_count();
  B200_REQUIRE(n_cta <= sms, "b200_rdb_chain: %d super-tiles exceed the %d SMs (split the batch)", n_cta, sms);
  int n_cta_chk;
  int64_t need;
  B200_REQUIRE(b200_rdb_chain_geometry(d->n, d->h, d->w, &n_cta_chk, &need) == 0, "b200_rdb_chain: unsupported geometry");
  B200_REQUIRE(ll_bytes >= need, "b200_rdb_chain: exchange buffer of %lld bytes needed", (long long)need);
  p.ll = reinterpret_cast<uint8_t*>(ll_buf);
  p.ll_tile_stride = (uint32_t)(4 * p.halo * kLLRowBytes);
  p.epoch = epoch_dev;
  p.table = table_dev;
  p.n_blocks = d->n_blocks;
  p.x_ch = d->x_coff;
  p.tap_sign = d->flip_taps ? -1 : 1;
  {
    const char* e = getenv("B200_CHAIN_DBG_PTR");
    p.dbg = e ? reinterpret_cast<long long*>(strtoull(e, nullptr, 0)) : nullptr;
  }
  {
    uint64_t dims[2] = {(uint64_t)(d->x_coff + 64), (uint64_t)P_total};
    uint64_t strides[1] = {(uint64_t)d->cx * 2};
    uint32_t box[2] = {64, (uint32_t)p.box_rows};
    if (make_tensor_map(&p.x_map, x0, 2, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  for (int j = 0; j < 5; ++j) {
    B200_REQUIRE(w_stage[j], "b200_rdb_chain: null stage weights");
    const int N = kNTotal - 32 * j;
    const uint64_t kc = (j == 0) ? 64 : 32;
    for (int part = 0; part < 2; ++part) {
      const int rows = part_rows(j, part, p.split);
      if (rows == 0) continue;
      uint64_t dims[3] = {kc, (uint64_t)N, (uint64_t)d->n_blocks * 9};
      uint64_t strides[2] = {kc * 2, (uint64_t)N * kc * 2};
      uint32_t box[3] = {(uint32_t)kc, (uint32_t)rows, 1};
      if (make_tensor_map(&p.w_map[j][part], w_stage[j], 3, dims, strides, box, nullptr,
                          kc == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B))
        return 1;
    }
  }
  // Thread-block clusters: neighbouring tiles inside a cluster exchange their halo rows through distributed
  // shared memory (bulk copy + remote mbarrier), only the cluster-edge halos go through L2.  The largest cluster
  // size (<= 8, the portable maximum) whose clusters are all co-resident is used.
  int cs = 1, grid = n_cta;
  // decided once per grid size (the occupancy query must not run inside a stream capture)
  static std::mutex cs_mu;
  static std::map<int, int> cs_cache;
  bool cached = false;
  {
    std::lock_guard<std::mutex> g(cs_mu);
    auto it = cs_cache.find(n_cta);
    if (it != cs_cache.end()) {
      cs = it->second;
      grid = (n_cta + cs - 1) / cs * cs;
      cached = true;
    }
  }
  for (int c = cached ? 0 : 8; c >= 2; --c) {   // any size, not only powers of two: 6 fits where 4 + 4 + .. does not
    const int g = (n_cta + c - 1) / c * c;
    cudaLaunchConfig_t q = {};
    q.gridDim = dim3(g);
    q.blockDim = dim3(kThreads);
    q.dynamicSmemBytes = kSmemBytes;
    cudaLaunchAttribute qa[1];
    qa[0].id = cudaLaunchAttributeClusterDimension;
    qa[0].val.clusterDim.x = c;
    qa[0].val.clusterDim.y = 1;
    qa[0].val.clusterDim.z = 1;
    q.attrs = qa;
    q.numAttrs = 1;
    int max_clusters = 0;
    const cudaError_t qe = cudaOccupancyMaxActiveClusters(&max_clusters, rdb_chain_kernel, &q);
    // measured on B200 with this kernel's 226 KB of shared memory: 74 clusters of 2, 33 clusters of 4 (config 2 needs
    // 34: one short, so the default run uses pairs and half of the tile sides go through L2)
    if (getenv("B200_CHAIN_DEBUG"))
      fprintf(stderr, "rdb_chain: cluster size %d -> max active clusters %d (%s), need %d\n", c, max_clusters,
              cudaGetErrorString(qe), g / c);
    if (qe == cudaSuccess && max_clusters * c >= g) {
      cs = c;
      grid = g;
      break;
    }
    (void)cudaGetLastError();
  }
  if (!cached) {
    std::lock_guard<std::mutex> g(cs_mu);
    cs_cache[n_cta] = cs;
  }
  p.cluster_size = cs;
  ::b200::launch_kernel(chain_epoch_bump_kernel, 1, 1, 0, as_stream(stream), epoch_dev);
  B200_LAUNCH_CHECK();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = as_stream(stream);
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (cs > 1) {
    // all clusters co-resident (checked above with cudaOccupancyMaxActiveClusters): the neighbour exchange
    // cannot deadlock once every cluster is scheduled
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cs;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  } else {
    attr[na].id = cudaLaunchAttributeCooperative;   // all CTAs co-resident
    attr[na].val.cooperative = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  B200_CHECK_CUDA(cudaLaunchKernelEx(&cfg, rdb_chain_kernel, p));
  g_launches.fetch_add(1);
  return 0;
}
