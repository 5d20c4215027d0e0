// Sparse convolution filter gradient on the tensor cores (BF16x3-class precision, no atomics).
//
//   dW[k][ci][co] = sum over output rows o of  features[nbr[k][o]][ci] * out_grad[o][co]      (spconv_ops.h:363-456,
//   the `torch::mm_out(filterGradSub, inputBuffer.t(), outputBuffer)` per kernel offset of indiceConvBackward)
//
// The reduction runs over ROWS, so both operands are "MN-major" for the tensor core: a row of the operand tile is one
// reduction index and holds the M (or N) elements contiguously -- which is exactly how the split images of
// spconv_v6.cu store a row (per 16 channels: 16 bf16 hi | 16 bf16 lo).  The kernel therefore
//   * gathers the 128-byte channel slabs of 64 feature rows (through nbr, missing rows as zeros) with cp.async into
//     SWIZZLE_128B tiles, exactly like the forward kernel, and loads the matching 64 out-grad rows with TMA tile
//     copies (they are contiguous);
//   * treats the hi and lo halves of a row as SEPARATE M (N) elements: one M = 128 x N = 2 Cout x K = 16 MMA with
//     MN-major descriptors produces hi.hi, hi.lo, lo.hi and lo.lo partial products of 64 input channels at once, in
//     separate accumulator rows / columns; the epilogue adds the four (two columns in registers, two TMEM lanes
//     through one shuffle);
//   * gives every CTA work items (kernel offset k, chunk of rows): the accumulator (2 Cin x 2 Cout fp32 = up to all
//     512 TMEM columns) lives in TMEM for the whole item and is written once as a partial dW; a second kernel adds the
//     partials of the chunks in a fixed order (bit-reproducible, like the SIMT path it replaces).
// Warp roles (10 warps, one CTA per SM): 0-7 feature-row gather + epilogue, 8 MMA issue + TMEM allocation,
// 9 out-grad loader (TMA).
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace bevb200 {

int spconv_v6_split_rows_padded(const float *features, int n, int c_in, int c_eff, void *split, cudaStream_t st);

constexpr int kWgtThreads = 10 * 32;
constexpr int kWgtMaxStages = 8;
constexpr int kWgtMaxUnits = 8;      // copy units (4 rows x the slabs of one offset) per gather lane and stage, at most

struct WgtParams {
  const uint8_t *fsplit;       // [n_in][ci_eff * 4 B]
  const int32_t *nbr;          // [kvol][n_out]
  float *partial;              // [n_chunks][kvol][c_in][c_out]
  int n_in, n_out, c_in, c_out, kvol;
  int ci_eff, co_eff;          // channel counts of the operand images: rounded up to 32 / 64 / 128 (zero padded)
  int n_chunks, tiles_per_chunk, n_tiles;   // tiles of R rows
  int n_a, n_b;                // 128-byte slabs per row: ci_eff / 32, co_eff / 32
  int g;                       // kernel offsets per work item (their accumulators share the 512 TMEM columns)
  int n_kgroups;               // ceil(kvol / g)
  int s_a;                     // feature slabs per stage: g * n_a
  int m_blocks;                // accumulator row blocks (two feature slabs each): s_a / 2
  int stages, stage_bytes;
  int tmem_cols;
};

// UMMA shared-memory descriptor, MN-major, SWIZZLE_128B (cute/atom/mma_traits_sm100.hpp, canonical layout
// ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units): a reduction row is 128 B, eight rows form a 1024-byte swizzle
// atom (SBO = distance between 8-row groups), LBO = distance between 64-element atoms along M / N.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = (uint64_t)((smem_addr & 0x3ffff) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

__device__ __forceinline__ void wgt_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

__device__ __forceinline__ void wgt_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tma_tile_2d(uint32_t dst_smem, const CUtensorMap *map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst_smem), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}

// A work item = (chunk of row tiles, group of g kernel offsets).  A stage holds, for one tile of R rows, the
// feature slabs of the g offsets -- slab index = offset_in_group * n_a + slab_in_row -- followed by the n_b
// out-grad slabs, which are loaded ONCE per tile and multiplied against every offset of the group.  Accumulator
// block b (128 TMEM lanes x 2 co_eff columns) belongs to feature slabs 2 b and 2 b + 1: two offsets of 32
// channels, one offset of 64, or half an offset of 128.
template <int R, int U>
__global__ void __launch_bounds__(kWgtThreads, 1)
spconv_wgrad_tc_kernel(const WgtParams p, const __grid_constant__ CUtensorMap gmap) {
  constexpr int kWgtMaxUnits = U;        // copy units per gather lane and stage (shadows the global bound)
  constexpr int kSlab = R * 128;
  constexpr int kRowGroups = R / 4;      // a copy instruction covers 4 rows x 128 B of one slab
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;
  __shared__ uint64_t bars[2 * kWgtMaxStages + 2];
  __shared__ uint32_t tmem_base_s;
  const uint32_t full = smem_u32(&bars[0]), empty = smem_u32(&bars[kWgtMaxStages]);
  const uint32_t acc_full = smem_u32(&bars[2 * kWgtMaxStages]), acc_empty = smem_u32(&bars[2 * kWgtMaxStages + 1]);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int stages = p.stages, n_a = p.n_a, n_b = p.n_b, s_a = p.s_a;
  const uint32_t stage_bytes = (uint32_t)p.stage_bytes;

  if (tid == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(full + 8 * s, 8 + 1);      // eight gather warps + the out-grad loader's expect_tx arrive
      mbar_init(empty + 8 * s, 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 8);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(&tmem_base_s)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  const int n_items = p.n_chunks * p.n_kgroups;
  const int n2 = 2 * p.co_eff;           // accumulator columns per row block

  if (warp < 8) {
    // =============================== feature-row gather + epilogue ==========================
    const int m = lane >> 3, c = lane & 7;
    const uint32_t row_bytes = (uint32_t)p.ci_eff * 4u;
    const unsigned long long fbase = reinterpret_cast<unsigned long long>(p.fsplit);
    // The stage's copies are units u = offset_in_group * (R / 4) + row_group; warp w takes u = w, w + 8, ...  A unit
    // is 4 rows x the n_a slabs of one offset: lane (m, c) loads ONE neighbour index (row 4 row_group + m) and copies
    // that row's n_a 16-byte pieces: it writes physical chunk c and fetches the logical chunk c ^ (row & 7)
    // (lane-order stores, as in spconv_v6.cu).
    const int n_units = (p.g * kRowGroups + 7 - warp) >> 3;       // units of this warp (<= kWgtMaxUnits)
    // per-unit constants (the gather loop itself must stay lean: it is instruction-bound otherwise, ncu)
    int u_row[kWgtMaxUnits], u_kl[kWgtMaxUnits];
    uint32_t u_dst[kWgtMaxUnits], u_src[kWgtMaxUnits];
#pragma unroll
    for (int j = 0; j < kWgtMaxUnits; ++j) {
      const int u = warp + 8 * j;
      const int kl = u / kRowGroups, rg = u - kl * kRowGroups;
      const int r = 4 * rg + m;
      u_kl[j] = kl;
      u_row[j] = r;
      u_dst[j] = (uint32_t)(kl * n_a) * kSlab + (uint32_t)(r * 128 + (c << 4));
      u_src[j] = (uint32_t)((c ^ (r & 7)) << 4);
    }
    // software pipeline of the warp: the neighbour indices of a tile are loaded two tiles ahead and a stage is
    // signalled `deep` stages after its copies were issued (deep = 2 when the ring has >= 4 stages), so neither the
    // index load nor the copies' L2 latency sits on the per-stage critical path
    const bool deep2 = stages >= 4;
    int s = 0, pend0 = -1, pend1 = -1;     // stages whose copies are committed but not yet signalled (older, newer)
    uint32_t ph = 0, acc_ph = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int chunk = item / p.n_kgroups, kg = item - chunk * p.n_kgroups;
      const int k0 = kg * p.g;
      const int t_begin = chunk * p.tiles_per_chunk, t_end = min(p.n_tiles, t_begin + p.tiles_per_chunk);
      const int32_t *u_nbr[kWgtMaxUnits];               // this unit's row of the neighbour table (null: no such offset)
#pragma unroll
      for (int j = 0; j < kWgtMaxUnits; ++j)
        u_nbr[j] = (j < n_units && k0 + u_kl[j] < p.kvol) ? p.nbr + (long long)(k0 + u_kl[j]) * p.n_out + u_row[j] : nullptr;
      int idx0[kWgtMaxUnits], idx1[kWgtMaxUnits];      // indices of tile t, t + 1 (then refilled for t + 2)
      auto load_idx = [&](int t, int (&idx)[kWgtMaxUnits]) {
        const int o0 = t * R;
#pragma unroll
        for (int j = 0; j < kWgtMaxUnits; ++j) {
          idx[j] = -1;
          if (t < t_end && u_nbr[j] != nullptr && o0 + u_row[j] < p.n_out) idx[j] = __ldg(u_nbr[j] + o0);
        }
      };
      load_idx(t_begin, idx0);
      load_idx(t_begin + 1, idx1);
      for (int t = t_begin; t < t_end; ++t) {
        int cur[kWgtMaxUnits];
#pragma unroll
        for (int j = 0; j < kWgtMaxUnits; ++j) {
          cur[j] = idx0[j] >= p.n_in ? -1 : idx0[j];
          idx0[j] = idx1[j];
        }
        load_idx(t + 2, idx1);
        mbar_wait(empty + 8 * s, ph ^ 1u);
        const uint32_t a_stage = ring + (uint32_t)s * stage_bytes;
#pragma unroll
        for (int j = 0; j < kWgtMaxUnits; ++j) {
          if (j < n_units) {
            const uint32_t dst = a_stage + u_dst[j];
            const unsigned long long src = fbase + (unsigned long long)(uint32_t)max(cur[j], 0) * row_bytes + u_src[j];
            for (int i = 0; i < n_a; ++i) cp_async16_row(dst + (uint32_t)i * kSlab, src + (unsigned)(i * 128), cur[j]);
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        if (deep2) {
          if (pend0 >= 0) {              // the copies of two stages ago have had two stages' time
            asm volatile("cp.async.wait_group 2;" ::: "memory");
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(full + 8 * pend0);
          }
          pend0 = pend1;
          pend1 = s;
        } else {
          if (pend1 >= 0) {
            asm volatile("cp.async.wait_group 1;" ::: "memory");
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(full + 8 * pend1);
          }
          pend1 = s;
        }
        if (++s == stages) { s = 0; ph ^= 1u; }
      }
      if (pend0 >= 0 || pend1 >= 0) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (pend0 >= 0) mbar_arrive(full + 8 * pend0);
          if (pend1 >= 0) mbar_arrive(full + 8 * pend1);
        }
        pend0 = pend1 = -1;
      }
      // ------------------------------- epilogue of the item ---------------------------------
      mbar_wait(acc_full, acc_ph);
      acc_ph ^= 1u;
      tc_fence_after();
      const int q = warp & 3, half = warp >> 2;
      for (int mb = 0; mb < p.m_blocks; ++mb) {
        // TMEM lanes 32 q .. 32 q + 31 of block mb: feature slab 2 mb + (q >> 1), channels 16 (q & 1) + 0..15 of it,
        // lanes 0-15 the hi halves, 16-31 the lo halves
        const int slab = 2 * mb + (q >> 1);
        const int k = k0 + slab / n_a;
        const int ci = (slab % n_a) * 32 + (q & 1) * 16 + (lane & 15);
        float *dst_k = p.partial + (((long long)chunk * p.kvol + k) * p.c_in + ci) * p.c_out;
        const bool ok = lane < 16 && k < p.kvol && ci < p.c_in;
        for (int cg = half; cg < (p.c_out >> 4); cg += 2) {
          float v[32];
          wgt_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mb * n2 + cg * 32), v);
          float sum[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            sum[j] = v[j] + v[j + 16];                                   // hi.co + lo.co columns
            sum[j] += __shfl_down_sync(0xffffffffu, sum[j], 16);          // + the lo.ci accumulator row
          }
          if (ok) {
            float4 *dst = reinterpret_cast<float4 *>(dst_k + cg * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j) dst[j] = make_float4(sum[4 * j], sum[4 * j + 1], sum[4 * j + 2], sum[4 * j + 3]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
    }
  } else if (warp == 8) {
    // =============================== MMA issuer ==========================================
    const uint32_t idesc = umma_idesc_bf16(128, n2) | (1u << 15) | (1u << 16);      // A and B MN-major
    int s = 0;
    uint32_t ph = 0, pe = 0;
    bool first_item = true;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int chunk = item / p.n_kgroups;
      const int t_begin = chunk * p.tiles_per_chunk, t_end = min(p.n_tiles, t_begin + p.tiles_per_chunk);
      if (!first_item) {
        mbar_wait(acc_empty, pe);
        pe ^= 1u;
        tc_fence_after();
      }
      first_item = false;
      for (int t = t_begin; t < t_end; ++t) {
        mbar_wait(full + 8 * s, ph);
        tc_fence_after();
        if (elect_one_sync()) {
          const uint32_t a_stage = ring + (uint32_t)s * stage_bytes;
          const uint32_t b_stage = a_stage + (uint32_t)s_a * kSlab;
#pragma unroll
          for (int ks = 0; ks < R / 16; ++ks) {
            const uint64_t bdesc = umma_desc_mn_sw128(b_stage + (uint32_t)(ks * 2048), kSlab);
            for (int mb = 0; mb < p.m_blocks; ++mb) {
              const uint64_t adesc = umma_desc_mn_sw128(a_stage + (uint32_t)(2 * mb) * kSlab + (uint32_t)(ks * 2048), kSlab);
              wgt_mma(tmem_base + (uint32_t)(mb * n2), adesc, bdesc, idesc, (t == t_begin && ks == 0) ? 0u : 1u);
            }
          }
          tc_commit(empty + 8 * s);
          if (t == t_end - 1) tc_commit(acc_full);
        }
        __syncwarp();
        if (++s == stages) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // =============================== out-grad loader (TMA) ===============================
    // (lane 0 in a plain branch: the compiler's per-instruction ELECT loop issues a TMA in ~90 clk; an elect.sync
    // region measured ~190 clk per TMA, tools/gather4_probe.cu and profiles/r2_wgrad_tc.md)
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int chunk = item / p.n_kgroups;
        const int t_begin = chunk * p.tiles_per_chunk, t_end = min(p.n_tiles, t_begin + p.tiles_per_chunk);
        for (int t = t_begin; t < t_end; ++t) {
          mbar_wait(empty + 8 * s, ph ^ 1u);
          mbar_arrive_expect_tx(full + 8 * s, (uint32_t)n_b * kSlab);
          const uint32_t b_stage = ring + (uint32_t)s * stage_bytes + (uint32_t)s_a * kSlab;
          for (int sl = 0; sl < n_b; ++sl)
            tma_tile_2d(b_stage + (uint32_t)sl * kSlab, &gmap, sl * 64, t * R, full + 8 * s);
          if (++s == stages) { s = 0; ph ^= 1u; }
        }
      }
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)p.tmem_cols) : "memory");
  }
}

// dW[e] = sum over chunks (ascending) of partial[chunk][e]
__global__ void spconv_wgrad_tc_reduce_kernel(const float *__restrict__ partial, long long elems, int n_chunks,
                                              float *__restrict__ w_grad) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < elems; e += (long long)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int ch = 0; ch < n_chunks; ++ch) s += partial[(long long)ch * elems + e];
    w_grad[e] = s;
  }
}

typedef CUresult (*WgtEncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                   const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static WgtEncodeTiled wgt_encode_fn() {
  static WgtEncodeTiled fn = [] {
    void *f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      f = nullptr;
    return (WgtEncodeTiled)f;
  }();
  return fn;
}

bool spconv_wgrad_tc_ok(int c_in, int c_out, int kvol) {
  static const bool enabled = [] {
    const char *e = getenv("BEVB200_WGRAD_TC");
    return e == nullptr || atoi(e) != 0;
  }();
  return enabled && c_in >= 1 && c_in <= 128 && (c_out == 16 || c_out == 32 || c_out == 64 || c_out == 128) &&
         kvol >= 1 && kvol <= 27;
}

// channel count of an operand image: 128-byte slabs of 32 channels, 1 / 2 / 4 of them (zero padded)
static int wgt_eff(int c) { return c <= 32 ? 32 : (c <= 64 ? 64 : 128); }

// The shape of a launch: offsets per work item, rows per stage, row chunks.
struct WgtPlan {
  int ci_eff, co_eff, n_a, n_b;
  int g, n_kgroups, s_a, m_blocks, tmem_cols;
  int rows, stage_bytes, stages;
  int n_tiles, n_chunks, tiles_per_chunk;
};
static WgtPlan wgt_plan(int n_out, int c_in, int c_out, int kvol) {
  WgtPlan w;
  w.ci_eff = wgt_eff(c_in);
  w.co_eff = wgt_eff(c_out);
  w.n_a = w.ci_eff / 32;
  w.n_b = w.co_eff / 32;
  const int n2 = 2 * w.co_eff;
  // accumulator blocks (128 lanes x n2 columns, two feature slabs each) that fit the 512 TMEM columns
  int blocks = 512 / n2;
  int g = (2 * blocks) / w.n_a;                      // offsets whose slabs fill those blocks
  if (g < 1) g = 1;
  if (g > 16) g = 16;
  if (g > kvol) g = kvol;
  if (w.n_a == 1 && g > 4) g = 4;                    // measured: 4 offsets per item beat 8 / 16 for 32-channel slabs
  if (w.n_a == 1 && (g & 1)) ++g;                    // 32-channel slabs pair up two offsets per block
  w.g = g;
  w.n_kgroups = (kvol + g - 1) / g;
  w.s_a = g * w.n_a;
  w.m_blocks = (w.s_a + 1) / 2;
  w.tmem_cols = 32;
  while (w.tmem_cols < w.m_blocks * n2) w.tmem_cols <<= 1;
  // rows per stage: 16 / 32 / 64 / 128, a stage of at most 64 KB and at most 8 copy units per gather lane
  int rows = 128;
  while (rows > 16 && ((w.s_a + w.n_b) * rows * 128 > 64 * 1024 || g * (rows / 4) > 8 * kWgtMaxUnits)) rows >>= 1;
  w.rows = rows;
  w.stage_bytes = (w.s_a + w.n_b) * rows * 128;
  w.stages = (200 * 1024) / w.stage_bytes;
  if (w.stages > kWgtMaxStages) w.stages = kWgtMaxStages;
  // row chunks: ~3 work items per SM, every chunk non-empty
  w.n_tiles = (n_out + rows - 1) / rows;
  int n_chunks = (3 * kNumSMs) / w.n_kgroups;
  if (n_chunks < 1) n_chunks = 1;
  if (n_chunks > w.n_tiles) n_chunks = w.n_tiles > 0 ? w.n_tiles : 1;
  w.tiles_per_chunk = w.n_tiles > 0 ? (w.n_tiles + n_chunks - 1) / n_chunks : 1;
  w.n_chunks = w.n_tiles > 0 ? (w.n_tiles + w.tiles_per_chunk - 1) / w.tiles_per_chunk : 1;
  return w;
}

// where spconv_wgrad_tc() leaves the split image of out_grad inside its workspace; for c_out = 32 / 64 / 128 it is the
// generation-6 row image of out_grad, which the input gradient can gather from instead of splitting the rows again
const void *spconv_wgrad_tc_grad_image(const void *workspace, int n_in, int c_in) {
  return (const uint8_t *)workspace + align_up((size_t)n_in * wgt_eff(c_in) * 4);
}

size_t spconv_wgrad_tc_workspace_bytes(int n_in, int n_out, int c_in, int c_out, int kvol) {
  if (!spconv_wgrad_tc_ok(c_in, c_out, kvol) || n_in <= 0 || n_out <= 0) return 0;
  const WgtPlan w = wgt_plan(n_out, c_in, c_out, kvol);
  return align_up((size_t)n_in * w.ci_eff * 4) + align_up((size_t)n_out * w.co_eff * 4) +
         align_up((size_t)w.n_chunks * kvol * c_in * c_out * sizeof(float));
}

int spconv_wgrad_tc(const float *features, const float *out_grad, const int32_t *nbr, int n_in, int n_out,
                    int c_in, int c_out, int kvol, float *weight_grad, void *workspace, cudaStream_t st) {
  BEVB200_REQUIRE(spconv_wgrad_tc_ok(c_in, c_out, kvol), "shape has no tensor-core filter gradient");
  const WgtPlan w = wgt_plan(n_out, c_in, c_out, kvol);
  const int ci_eff = w.ci_eff, co_eff = w.co_eff, rows = w.rows;
  uint8_t *fsplit = (uint8_t *)workspace;
  uint8_t *gsplit = fsplit + align_up((size_t)n_in * ci_eff * 4);
  float *partial = (float *)(gsplit + align_up((size_t)n_out * co_eff * 4));
  int rc = spconv_v6_split_rows_padded(features, n_in, c_in, ci_eff, fsplit, st);
  if (!rc) rc = spconv_v6_split_rows_padded(out_grad, n_out, c_out, co_eff, gsplit, st);
  if (rc) return rc;
  WgtParams p;
  memset(&p, 0, sizeof(p));
  p.fsplit = fsplit;
  p.nbr = nbr;
  p.partial = partial;
  p.n_in = n_in; p.n_out = n_out; p.c_in = c_in; p.c_out = c_out; p.kvol = kvol;
  p.ci_eff = ci_eff; p.co_eff = co_eff;
  p.n_tiles = w.n_tiles; p.n_chunks = w.n_chunks; p.tiles_per_chunk = w.tiles_per_chunk;
  p.n_a = w.n_a; p.n_b = w.n_b;
  p.g = w.g; p.n_kgroups = w.n_kgroups; p.s_a = w.s_a; p.m_blocks = w.m_blocks;
  p.stage_bytes = w.stage_bytes; p.stages = w.stages;
  p.tmem_cols = w.tmem_cols;
  BEVB200_REQUIRE(p.tmem_cols <= 512 && p.stages >= 2, "filter gradient tile does not fit");
  // out-grad split image as a 2-D bf16 tensor [n_out][co_eff * 2]; one box = `rows` rows x 128 B
  WgtEncodeTiled enc = wgt_encode_fn();
  BEVB200_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available");
  CUtensorMap gmap;
  const cuuint64_t dims[2] = {(cuuint64_t)co_eff * 2, (cuuint64_t)n_out};
  const cuuint64_t strides[1] = {(cuuint64_t)co_eff * 4};
  const cuuint32_t box[2] = {64, (cuuint32_t)rows};
  const cuuint32_t estr[2] = {1, 1};
  BEVB200_REQUIRE(enc(&gmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, gsplit, dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS,
                  "cuTensorMapEncodeTiled failed for the out-grad image");
  const size_t smem = (size_t)p.stages * p.stage_bytes + 1024;
  const int n_items = p.n_chunks * p.n_kgroups;
  const int grid = n_items < kNumSMs ? n_items : kNumSMs;
  const int units = (w.g * (rows / 4) + 7) / 8;       // per gather lane
  const int ucap = units <= 2 ? 2 : (units <= 4 ? 4 : 8);
#define WGT_LAUNCH(R, U)                                                                                           \
  do {                                                                                                             \
    BEVB200_CUDA(cudaFuncSetAttribute(spconv_wgrad_tc_kernel<R, U>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    BEVB200_LAUNCH((spconv_wgrad_tc_kernel<R, U>), grid, kWgtThreads, smem, st, p, gmap);                          \
  } while (0)
#define WGT_ROWS(R)                                                                                                \
  do {                                                                                                             \
    if (ucap == 2) WGT_LAUNCH(R, 2);                                                                               \
    else if (ucap == 4) WGT_LAUNCH(R, 4);                                                                          \
    else WGT_LAUNCH(R, 8);                                                                                         \
  } while (0)
  if (rows == 128) WGT_ROWS(128);
  else if (rows == 64) WGT_ROWS(64);
  else if (rows == 32) WGT_ROWS(32);
  else WGT_ROWS(16);
#undef WGT_ROWS
#undef WGT_LAUNCH
  const long long elems = (long long)kvol * c_in * c_out;
  BEVB200_LAUNCH(spconv_wgrad_tc_reduce_kernel, grid_for(elems, 256), 256, 0, st, partial, elems, p.n_chunks, weight_grad);
  return BEVB200_OK;
}

}  // namespace bevb200
