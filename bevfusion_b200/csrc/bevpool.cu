// bev_pool for sm_100a: sorted-interval BEV pooling, forward / backward / precompute.
//
// Reference behaviour restated (not copied): mmdet3d/ops/bev_pool/src/bev_pool_cuda.cu:20-84
// (one thread per (interval, channel), serial loop over the interval) and the Python glue in
// mmdet3d/ops/bev_pool/bev_pool.py:38-98, mmdet3d/models/vtransforms/base.py:141-176.
//
// B200 design (HBM-bound, ~0.64 GB per launch at the C2 workload):
//   * the sorted row stream is cut into equal ranges, one per warp, so work per warp is uniform no
//     matter how skewed the interval lengths are (1 .. >1000); the forward streams each range
//     through a shared-memory ring (see "forward" below), the backward walks CHUNK_ROWS-row chunks
//   * an interval that crosses a range boundary leaves its pieces in a small partial buffer and a
//     second tiny kernel adds them in fixed order -> results are bit-reproducible run to run (no
//     float atomics)
//   * `perm` variants read rows of the ORIGINAL feature tensor through the sorted->original
//     map, which removes x[kept] / feats[indices] (2 x 0.6 GB of copies) from the frame
// The first forward kernel (one warp per 128-row chunk, 16-byte register loads, per-interval folds
// through shared memory) was removed after the TMA-staged kernel replaced it: DESIGN.md 4.1.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace bevb200 {

constexpr int kChunkRows = 128;            // rows of the sorted stream owned by one backward warp (and the
                                           // unit pool_partial_bytes sizes the forward's partial buffer in)
constexpr int kPoolWarps = 8;              // warps per CTA of the backward kernel

struct PoolDims {
  int b, d, h, w;
};

__device__ __forceinline__ long long cell_of(const int32_t *__restrict__ geom_feats, int row,
                                             const PoolDims dm) {
  // flat index into out[b][d][h][w] from (x, y, z, b) = geom_feats[row] (bev_pool_cuda.cu:34-36)
  int4 g = *reinterpret_cast<const int4 *>(geom_feats + 4ll * row);
  if ((unsigned)g.x >= (unsigned)dm.h || (unsigned)g.y >= (unsigned)dm.w ||
      (unsigned)g.z >= (unsigned)dm.d || (unsigned)g.w >= (unsigned)dm.b)
    return -1;
  return (((long long)g.w * dm.d + g.z) * dm.h + g.x) * dm.w + g.y;
}

// last index i in [0, n) with starts[i] <= row, or -1
__device__ __forceinline__ int find_interval(const int32_t *__restrict__ starts, int n, int row) {
  int lo = 0, hi = n;  // first index with starts[i] > row
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (__ldg(starts + mid) <= row) lo = mid + 1; else hi = mid;
  }
  return lo - 1;
}

// ---------------------------------------------------------------------------------------
// forward: TMA-staged streaming reduction (the tuned channel widths)
// ---------------------------------------------------------------------------------------
// Every warp owns a contiguous range of the sorted row stream and runs its own
// cp.async.bulk -> shared memory ring (32 rows per stage, mbarrier complete_tx), so the bytes in
// flight per SM (warps x stages x 32 rows x C x 4 B, ~120-180 KB) do not depend on registers or
// on the interval lengths.  Rows are gathered through `perm` with one 16*Q-byte bulk copy per
// row (one copy of the whole stage when the rows are already sorted).  The warp then walks the
// staged rows in order: lane q owns float4 column q, adds rows into a register accumulator and
// flushes it at interval boundaries (bitmask per stage built from the interval table) with a
// coalesced 16-byte-per-lane store.  An interval that crosses a warp-range boundary leaves its
// pieces in `partial` (2 slots per range: head = continuation from the previous range, tail =
// continues into the next) and the fix-up kernel adds them in range order: fixed summation
// order, bit-reproducible, no float atomics.  Requires the intervals to tile [0, n) in order,
// which is how QuickCumsumCuda (bev_pool.py:41-46) builds them; the host checks nothing else.
constexpr int kStageRows = 32;
constexpr int kPoolStages = 3;

__device__ __forceinline__ uint32_t pool_smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void pool_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "PW_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra PW_DONE;\n\t"
      "bra PW_LOOP;\n\t"
      "PW_DONE:\n\t}"
      ::"r"(bar), "r"(parity) : "memory");
}

__global__ void pool_interval_cells_kernel(const int32_t *__restrict__ geom_feats,
                                           const int32_t *__restrict__ starts, int n, int n_intervals,
                                           PoolDims dm, int32_t *__restrict__ cells) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_intervals; i += gridDim.x * blockDim.x) {
    int s = starts[i];
    long long c = (s >= 0 && s < n) ? cell_of(geom_feats, s, dm) : -1;
    cells[i] = (int32_t)c;  // host guarantees b*d*h*w < 2^31
  }
}

// MODE 0: rows already sorted (one TMA bulk copy per stage); MODE 1: rows gathered through perm;
// MODE 2: fused LSS lift -- row r is depth[perm[r]] * ctx[pixel(perm[r]), :] and is never materialised
// (x = ctx [n_pix, C] channels-last, `depth` = flattened [B*N, D, fH*fW] softmax volume).
struct LiftDims {
  int d_bins, hw;   // depth bins D and fH*fW: original index i -> pixel row (i / (D*hw)) * hw + i % hw
};
// (Gathering through perm with TMA tile::gather4, 4 rows per instruction, was measured no faster at C2 --
// 166 us vs 162 us: row-granular gathers cap near 3.9 TB/s with either mechanism -- and removed.)
template <int Q, int MODE>
__global__ void __launch_bounds__(256)
    bevpool_fwd_tma_kernel(const float4 *__restrict__ x,
                           const int32_t *__restrict__ perm, const float *__restrict__ depth, LiftDims lift,
                           const int32_t *__restrict__ starts, const int32_t *__restrict__ cells,
                           int n, int n_intervals, int rows_per_warp, int zfill, int total_cells,
                           float4 *__restrict__ out, float4 *__restrict__ partial) {
  constexpr int QPL = (Q + 31) / 32;              // float4 columns per lane
  constexpr uint32_t kRowBytes = Q * 16;
  constexpr bool PERM = MODE == 1 || MODE == 2;   // cp.async gather with commit groups
  constexpr uint32_t kStageBytes = kStageRows * kRowBytes + (MODE == 2 ? 128u : 0u);   // + 32 depth values
  extern __shared__ __align__(128) uint8_t pool_smem[];
  __shared__ uint64_t bars[8 * kPoolStages];
  const int warp = threadIdx.x >> 5, lane = lane_id(), nwarps = blockDim.x >> 5;
  const int j = blockIdx.x * nwarps + warp;       // warp-range index
  const long long R0l = (long long)j * rows_per_warp;
  if (R0l >= n) return;
  const int R0 = (int)R0l, R1 = min(n, R0 + rows_per_warp);
  uint8_t *my = pool_smem + (size_t)warp * kPoolStages * kStageBytes;
  const uint32_t my_u32 = pool_smem_u32(my);
  const uint32_t bar0 = pool_smem_u32(&bars[warp * kPoolStages]);
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kPoolStages; ++s)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8 * s));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  const int n_stages = (R1 - R0 + kStageRows - 1) / kStageRows;

  // Stage fill.  Sorted rows (PERM == false): ONE cp.async.bulk (TMA) of the whole stage,
  // completion on the stage's mbarrier.  Gathered rows (PERM == true): per-row bulk copies are
  // TMA-issue bound (measured: ~27 clk per 320-byte copy per SM), so the rows are gathered with
  // 16-byte cp.async (LDGSTS, no registers held) -- lane l holds the source row of stage row l,
  // float4 f of the stage comes from row f / Q -- and completion is tracked per commit group.
  auto issue = [&](int it) {
    const int s = it % kPoolStages;
    const int r0s = R0 + it * kStageRows;
    const int nrows = min(kStageRows, R1 - r0s);
    const uint32_t dst = my_u32 + (uint32_t)s * kStageBytes;
    if constexpr (PERM) {
      long long prow = lane < nrows ? (long long)__ldg(perm + r0s + lane) : 0ll;
      if constexpr (MODE == 2) {
        if (lane < nrows)   // the row's depth weight, staged behind the 32 feature rows
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + kStageRows * kRowBytes + (uint32_t)lane * 4u),
                       "l"(depth + prow) : "memory");
        const long long per_cam = (long long)lift.d_bins * lift.hw;
        prow = (prow / per_cam) * lift.hw + prow % lift.hw;     // pixel row of ctx
      }
#pragma unroll
      for (int t = 0; t < Q; ++t) {
        const int f = lane + 32 * t;
        const int row = f / Q, q = f - row * Q;
        const long long srow = __shfl_sync(0xffffffffu, prow, row);
        if (row < nrows)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (uint32_t)f * 16u),
                       "l"(x + srow * Q + q) : "memory");
      }
    } else {
      const uint32_t bar = bar0 + 8 * s;
      if (lane == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar),
                     "r"((uint32_t)nrows * kRowBytes) : "memory");
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
            ::"r"(dst), "l"(x + (long long)r0s * Q), "r"((uint32_t)nrows * kRowBytes), "r"(bar) : "memory");
      }
    }
  };
  auto commit = [&]() {
    if constexpr (PERM) asm volatile("cp.async.commit_group;" ::: "memory");
  };
  for (int it = 0; it < kPoolStages; ++it) {
    if (it < n_stages) issue(it);
    commit();                                     // one group per ring slot, even when empty
  }

  // interval bookkeeping: `ibase` = first interval whose start is >= the current stage's first row
  float4 acc[QPL];
#pragma unroll
  for (int u = 0; u < QPL; ++u) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
  bool open = false, head = false;   // an interval is being accumulated / it began before R0
  int cur_cell = -1;
  int ibase;
  {
    int i0 = find_interval(starts, n_intervals, R0);
    if (i0 >= 0 && __ldg(starts + i0) == R0) {
      ibase = i0;
    } else {
      ibase = i0 + 1;
      if (i0 >= 0) { open = true; head = true; }
    }
  }
  auto flush = [&](bool final_piece_continues) {
    if (!open) return;
    float4 *dst;
    if (head) dst = partial + (2ll * j) * Q;
    else if (final_piece_continues) dst = partial + (2ll * j + 1) * Q;
    else dst = cur_cell >= 0 ? out + (long long)cur_cell * Q : nullptr;
    if (dst) {
#pragma unroll
      for (int u = 0; u < QPL; ++u) {
        const int q = lane + 32 * u;
        if (q < Q) dst[q] = acc[u];
      }
    }
#pragma unroll
    for (int u = 0; u < QPL; ++u) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    open = false; head = false;
  };

  // with `zfill` (cells ascend with the interval index: plan tables, B*D == 1) the warp that
  // opens interval i also zeroes the empty cells between interval i-1 and i, so the grid needs
  // no separate memset pass
  auto zero_cells = [&](int lo, int hi) {        // cells [lo, hi)
    const long long cnt = (long long)(hi - lo) * Q;
    float4 *dst = out + (long long)lo * Q;
    for (long long i = lane; i < cnt; i += 32) dst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  };
  // interval table of the NEXT stage is fetched while the current one is reduced
  int st_n = ibase + lane < n_intervals ? __ldg(starts + ibase + lane) : 0x7fffffff;
  int cell_n = ibase + lane < n_intervals ? __ldg(cells + ibase + lane) : -1;
  int pc_n = ibase > 0 ? __ldg(cells + ibase - 1) : -1;
  for (int it = 0; it < n_stages; ++it) {
    const int s = it % kPoolStages;
    const int r0s = R0 + it * kStageRows;
    const int nrows = min(kStageRows, R1 - r0s);
    const int st = st_n, cellv = cell_n, prev_cell_base = pc_n;
    const bool in_stage = st < r0s + nrows;      // st >= r0s by construction of ibase
    const uint32_t mask = __reduce_or_sync(0xffffffffu, in_stage ? (1u << (st - r0s)) : 0u);
    const int ib_cur = ibase;
    ibase += __popc(mask);
    if (it + 1 < n_stages) {
      st_n = ibase + lane < n_intervals ? __ldg(starts + ibase + lane) : 0x7fffffff;
      cell_n = ibase + lane < n_intervals ? __ldg(cells + ibase + lane) : -1;
      pc_n = ibase > 0 ? __ldg(cells + ibase - 1) : -1;
    }
    if constexpr (PERM) {
      asm volatile("cp.async.wait_group %0;" ::"n"(kPoolStages - 1) : "memory");
      __syncwarp();                                // other lanes' copies are visible after their wait
    } else {
      pool_mbar_wait(bar0 + 8 * s, (uint32_t)(it / kPoolStages) & 1u);
    }
    const float4 *rows = reinterpret_cast<const float4 *>(my + (size_t)s * kStageBytes);
    const float *dvals = reinterpret_cast<const float *>(my + (size_t)s * kStageBytes + kStageRows * kRowBytes);
    int row = 0, iv = 0;   // iv = how many boundaries of this stage have been consumed
    while (row < nrows) {
      const uint32_t m = mask >> row;
      if (m & 1u) {        // `row` starts interval ib_cur + iv
        flush(false);
        cur_cell = __shfl_sync(0xffffffffu, cellv, iv);
        if (zfill) {
          const int prevc = iv > 0 ? __shfl_sync(0xffffffffu, cellv, iv - 1) : prev_cell_base;
          if (cur_cell > prevc + 1) zero_cells(prevc + 1, cur_cell);
          if (ib_cur + iv == n_intervals - 1 && cur_cell + 1 < total_cells) zero_cells(cur_cell + 1, total_cells);
        }
        ++iv;
        open = true;
      }
      const uint32_t rest = m >> 1;
      const int run = min(nrows - row, rest ? __ffs(rest) : 32);
      int rr = row;
      for (; rr + 4 <= row + run; rr += 4) {
#pragma unroll
        for (int u = 0; u < QPL; ++u) {
          const int q = lane + 32 * u;
          if (q < Q) {
            const float4 a = rows[(rr + 0) * Q + q], b = rows[(rr + 1) * Q + q];
            const float4 c = rows[(rr + 2) * Q + q], d = rows[(rr + 3) * Q + q];
            if constexpr (MODE == 2) {
              const float wa = dvals[rr], wb = dvals[rr + 1], wc = dvals[rr + 2], wd = dvals[rr + 3];
              // same arithmetic as the unfused path: product rounded to fp32, then added
              acc[u].x += __fmul_rn(wa, a.x); acc[u].y += __fmul_rn(wa, a.y); acc[u].z += __fmul_rn(wa, a.z); acc[u].w += __fmul_rn(wa, a.w);
              acc[u].x += __fmul_rn(wb, b.x); acc[u].y += __fmul_rn(wb, b.y); acc[u].z += __fmul_rn(wb, b.z); acc[u].w += __fmul_rn(wb, b.w);
              acc[u].x += __fmul_rn(wc, c.x); acc[u].y += __fmul_rn(wc, c.y); acc[u].z += __fmul_rn(wc, c.z); acc[u].w += __fmul_rn(wc, c.w);
              acc[u].x += __fmul_rn(wd, d.x); acc[u].y += __fmul_rn(wd, d.y); acc[u].z += __fmul_rn(wd, d.z); acc[u].w += __fmul_rn(wd, d.w);
            } else {
            acc[u].x += a.x; acc[u].y += a.y; acc[u].z += a.z; acc[u].w += a.w;
            acc[u].x += b.x; acc[u].y += b.y; acc[u].z += b.z; acc[u].w += b.w;
            acc[u].x += c.x; acc[u].y += c.y; acc[u].z += c.z; acc[u].w += c.w;
            acc[u].x += d.x; acc[u].y += d.y; acc[u].z += d.z; acc[u].w += d.w;
            }
          }
        }
      }
      for (; rr < row + run; ++rr) {
#pragma unroll
        for (int u = 0; u < QPL; ++u) {
          const int q = lane + 32 * u;
          if (q < Q) {
            const float4 a = rows[rr * Q + q];
            if constexpr (MODE == 2) {
              const float wa = dvals[rr];
              acc[u].x += __fmul_rn(wa, a.x); acc[u].y += __fmul_rn(wa, a.y); acc[u].z += __fmul_rn(wa, a.z); acc[u].w += __fmul_rn(wa, a.w);
            } else {
            acc[u].x += a.x; acc[u].y += a.y; acc[u].z += a.z; acc[u].w += a.w;
            }
          }
        }
      }
      row += run;
    }
    __syncwarp();                                  // all lanes are done reading this slot
    if (it + kPoolStages < n_stages) issue(it + kPoolStages);
    commit();
  }
  // does the open interval continue into the next warp range?
  const bool continues = R1 < n && !(ibase < n_intervals && __ldg(starts + ibase) == R1);
  flush(continues);
}

// one thread per warp range: if the interval holding the range's last row started inside the
// range and runs past its end, add its pieces (tail of this range + heads of the following ones)
template <int Q>
__global__ void bevpool_fwd_tma_fixup_kernel(const int32_t *__restrict__ starts,
                                             const int32_t *__restrict__ cells, int n,
                                             int n_intervals, int rows_per_warp, int n_ranges,
                                             float4 *__restrict__ out,
                                             const float4 *__restrict__ partial) {
  const int lane = lane_id();
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  for (int j = wid; j < n_ranges; j += nw) {
    const long long R0 = (long long)j * rows_per_warp, R1 = min((long long)n, R0 + rows_per_warp);
    if (R0 >= n || R1 >= n) continue;              // the last range has nothing after it
    const int iv = find_interval(starts, n_intervals, (int)R1 - 1);
    if (iv < 0) continue;
    const int s = __ldg(starts + iv);
    const int e = iv + 1 < n_intervals ? __ldg(starts + iv + 1) : n;   // intervals tile [0, n)
    if (s < R0 || e <= R1) continue;               // not the owner, or it ends inside the range
    const int cell = __ldg(cells + iv);
    if (cell < 0) continue;
    const int jl = (int)((e - 1) / rows_per_warp);
    for (int q = lane; q < Q; q += 32) {
      float4 r = partial[(2ll * j + 1) * Q + q];
      for (int jj = j + 1; jj <= jl; ++jj) {
        const float4 v = partial[(2ll * jj) * Q + q];
        r.x += v.x; r.y += v.y; r.z += v.z; r.w += v.w;
      }
      out[(long long)cell * Q + q] = r;
    }
  }
}

// [rows, C] -> [C, rows] tiled transpose (32 x 32 tiles through padded shared memory): turns the op
// layout [B, Z, X, Y, C] into the module output [B, Z*C, X, Y] (bev_pool.py:97 + base.py:174)
__global__ void __launch_bounds__(256)
    bev_channels_first_kernel(const float *__restrict__ in, float *__restrict__ out, int rows, int c,
                              int nz, long long out_batch_stride) {
  __shared__ float tile[32][33];
  const long long slab = blockIdx.z;                       // (b, z) slab of X*Y rows
  const float *src = in + slab * (long long)rows * c;
  float *dst = out + (slab / nz) * out_batch_stride + (slab % nz) * (long long)rows * c;
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int r = r0 + ty + i, cc = c0 + tx;
    tile[ty + i][tx] = (r < rows && cc < c) ? src[(long long)r * c + cc] : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int cc = c0 + ty + i, r = r0 + tx;
    if (cc < c && r < rows) dst[(long long)cc * rows + r] = tile[tx][ty + i];
  }
}

// any channel count: one thread per (interval, channel), like the reference kernel but on the
// caller's stream and with bounds checks.  Used only when C is not one of the tuned widths.
__global__ void bevpool_fwd_generic_kernel(const float *__restrict__ x,
                                           const int32_t *__restrict__ perm,
                                           const int32_t *__restrict__ geom_feats,
                                           const int32_t *__restrict__ starts,
                                           const int32_t *__restrict__ lengths, int n, int c,
                                           int n_intervals, PoolDims dm, float *__restrict__ out) {
  long long total = (long long)n_intervals * c;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int i = (int)(idx / c), ch = (int)(idx % c);
    int s = starts[i], L = lengths[i];
    if (L <= 0 || s < 0 || s >= n) continue;
    int e = min(s + L, n);
    long long cell = cell_of(geom_feats, s, dm);
    if (cell < 0) continue;
    float acc = 0.f;
    for (int r = s; r < e; ++r) {
      long long src = perm ? perm[r] : r;
      acc += x[src * c + ch];
    }
    out[cell * c + ch] = acc;
  }
}

// ---------------------------------------------------------------------------------------
// backward: x_grad[row, :] = out_grad[cell(interval(row)), :]
// ---------------------------------------------------------------------------------------
// Q = C/4 float4 per row, G rows per warp step, T = G*Q/32 float4 per lane per step.
template <int Q, int G>
struct PoolCfg {
  static constexpr int T = G * Q / 32;
  static_assert(G * Q % 32 == 0, "a warp step must be a whole number of float4 per lane");
  static_assert(32 % G == 0, "G must divide the 32-row perm block");
};

template <int Q, int G>
__global__ void __launch_bounds__(kPoolWarps * 32)
    bevpool_bwd_kernel(const float4 *__restrict__ out_grad, const int32_t *__restrict__ perm,
                       const int32_t *__restrict__ geom_feats,
                       const int32_t *__restrict__ starts, const int32_t *__restrict__ lengths,
                       int n, int n_total, int n_intervals, PoolDims dm,
                       float4 *__restrict__ x_grad) {
  constexpr int T = PoolCfg<Q, G>::T;
  const int lane = lane_id();
  int rig[T], qq[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    int f = lane + 32 * t;
    rig[t] = f / Q;
    qq[t] = f % Q;
  }
  const int nchunks = (n_total + kChunkRows - 1) / kChunkRows;
  const int warps_total = gridDim.x * kPoolWarps;
  for (int j = blockIdx.x * kPoolWarps + (threadIdx.x >> 5); j < nchunks; j += warps_total) {
    const int c0 = j * kChunkRows, c1 = min(n_total, c0 + kChunkRows);
    int i = c0 < n ? find_interval(starts, n_intervals, c0) : n_intervals;
    int r = c0;
    while (r < c1) {
      // next piece [r, pe): rows of interval i, or a gap of rows owned by no interval
      // (filtered-out rows at the tail of perm, or holes between malformed intervals)
      float4 g[T];
      int pe;
      bool have = false;
      if (i >= 0 && i < n_intervals) {
        int s = __ldg(starts + i), L = __ldg(lengths + i);
        int e = min(s + max(L, 0), n);
        if (r >= e) { ++i; continue; }
        if (r >= s) {
          pe = min(e, c1);
          long long cell = cell_of(geom_feats, s, dm);
          if (cell >= 0) {
            have = true;
#pragma unroll
            for (int t = 0; t < T; ++t) g[t] = __ldg(out_grad + cell * Q + qq[t]);
          }
        } else {
          pe = min(s, c1);
        }
      } else if (i < 0) {
        int s0 = n_intervals > 0 ? __ldg(starts) : n_total;
        pe = min(max(s0, r + 1), c1);
        if (s0 <= r) { i = 0; continue; }
      } else {
        pe = c1;
      }
      if (!have) {
#pragma unroll
        for (int t = 0; t < T; ++t) g[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      for (int r0 = r; r0 < pe; r0 += 32) {
        int row = r0 + lane;
        int src = row < pe ? (perm ? __ldg(perm + row) : row) : 0;
        const int nrows = min(32, pe - r0);
        for (int g0 = 0; g0 < nrows; g0 += G) {
#pragma unroll
          for (int t = 0; t < T; ++t) {
            int ra = g0 + rig[t];
            int sa = __shfl_sync(0xffffffffu, src, ra & 31);
            if (ra < nrows) stg_stream_f4(x_grad + (long long)sa * Q + qq[t], g[t]);
          }
        }
      }
      r = pe;
    }
  }
}

__global__ void bevpool_bwd_generic_kernel(const float *__restrict__ out_grad,
                                           const int32_t *__restrict__ perm,
                                           const int32_t *__restrict__ geom_feats,
                                           const int32_t *__restrict__ starts,
                                           const int32_t *__restrict__ lengths, int n, int c,
                                           int n_intervals, PoolDims dm,
                                           float *__restrict__ x_grad) {
  long long total = (long long)n_intervals * c;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int i = (int)(idx / c), ch = (int)(idx % c);
    int s = starts[i], L = lengths[i];
    if (L <= 0 || s < 0 || s >= n) continue;
    int e = min(s + L, n);
    long long cell = cell_of(geom_feats, s, dm);
    if (cell < 0) continue;
    float g = out_grad[cell * c + ch];
    for (int r = s; r < e; ++r) {
      long long src = perm ? perm[r] : r;
      x_grad[src * c + ch] = g;
    }
  }
}

// ---------------------------------------------------------------------------------------
// host dispatch
// ---------------------------------------------------------------------------------------
constexpr int kTmaMaxRanges = kNumSMs * 8;   // warp ranges of the TMA-staged kernel (<= 8 warps per SM)
static size_t pool_partial_bytes(int n, int c) {
  size_t nchunks = ((size_t)n + kChunkRows - 1) / kChunkRows;
  if (nchunks < (size_t)kTmaMaxRanges) nchunks = kTmaMaxRanges;
  // partial rows (2 per chunk / warp range) + one int32 cell id per interval (<= n of them)
  return align_up(2 * nchunks * (size_t)c * sizeof(float)) + align_up((size_t)n * sizeof(int32_t));
}

template <int Q>
static int launch_fwd_tma(const float *x, const int32_t *perm, const int32_t *geom,
                          const int32_t *starts, int n, int c, int n_intervals, PoolDims dm, float *out,
                          void *ws, int zfill, cudaStream_t st, const float *depth = nullptr,
                          LiftDims lift = LiftDims{1, 1}) {
  size_t nchunks = ((size_t)n + kChunkRows - 1) / kChunkRows;
  if (nchunks < (size_t)kTmaMaxRanges) nchunks = kTmaMaxRanges;
  float *partial = (float *)ws;
  int32_t *cells = (int32_t *)((char *)ws + align_up(2 * nchunks * (size_t)c * sizeof(float)));
  BEVB200_LAUNCH(pool_interval_cells_kernel, grid_for(n_intervals, 256), 256, 0, st, geom, starts, n,
                 n_intervals, dm, cells);
  const size_t stage_bytes = (size_t)kStageRows * Q * 16 + (depth ? 128 : 0);
  int warps = (int)((200 * 1024) / (kPoolStages * stage_bytes));
  if (warps > 8) warps = 8;
  if (warps < 1) warps = 1;
  const size_t smem = (size_t)warps * kPoolStages * stage_bytes;
  const int n_ranges_max = kNumSMs * warps;
  int rpw = (int)(((long long)n + n_ranges_max - 1) / n_ranges_max);
  rpw = (rpw + kStageRows - 1) / kStageRows * kStageRows;
  const int n_ranges = (n + rpw - 1) / rpw;
  const int grid = (n_ranges + warps - 1) / warps;
#define BEVB200_POOL_TMA_LAUNCH(MODE)                                                             \
  do {                                                                                              \
    BEVB200_CUDA(cudaFuncSetAttribute(bevpool_fwd_tma_kernel<Q, MODE>,                              \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));      \
    BEVB200_LAUNCH((bevpool_fwd_tma_kernel<Q, MODE>), grid, warps * 32, smem, st,                    \
                   (const float4 *)x, perm, depth, lift, starts, cells, n, n_intervals, rpw, zfill,  \
                   dm.b * dm.d * dm.h * dm.w, (float4 *)out, (float4 *)partial);                     \
  } while (0)
  if (depth) BEVB200_POOL_TMA_LAUNCH(2);
  else if (perm) BEVB200_POOL_TMA_LAUNCH(1);
  else BEVB200_POOL_TMA_LAUNCH(0);
#undef BEVB200_POOL_TMA_LAUNCH
  BEVB200_LAUNCH((bevpool_fwd_tma_fixup_kernel<Q>), (n_ranges * 32 + 255) / 256, 256, 0, st, starts, cells, n,
                 n_intervals, rpw, n_ranges, (float4 *)out, (const float4 *)partial);
  return BEVB200_OK;
}

template <int Q, int G>
static int launch_bwd(const float *og, const int32_t *perm, const int32_t *geom,
                      const int32_t *starts, const int32_t *lengths, int n, int n_total,
                      int n_intervals, PoolDims dm, float *xg, cudaStream_t st) {
  int nchunks = (n_total + kChunkRows - 1) / kChunkRows;
  int grid = min((nchunks + kPoolWarps - 1) / kPoolWarps, kNumSMs * 4);
  BEVB200_LAUNCH((bevpool_bwd_kernel<Q, G>), grid, kPoolWarps * 32, 0, st, (const float4 *)og, perm,
                 geom, starts, lengths, n, n_total, n_intervals, dm, (float4 *)xg);
  return BEVB200_OK;
}

#define BEVB200_POOL_DISPATCH(C, CALL, FALLBACK) \
  switch (C) {                                   \
    case 16: CALL(4, 32); break;                 \
    case 32: CALL(8, 16); break;                 \
    case 64: CALL(16, 8); break;                 \
    case 80: CALL(20, 8); break;                 \
    case 96: CALL(24, 4); break;                 \
    case 128: CALL(32, 4); break;                \
    case 160: CALL(40, 4); break;                \
    case 256: CALL(64, 2); break;                \
    default: FALLBACK; break;                    \
  }

static int pool_forward(int b, int d, int h, int w, int n, int c, int n_intervals, const float *x,
                        const int32_t *perm, const int32_t *geom, const int32_t *starts,
                        const int32_t *lengths, float *out, void *ws, size_t ws_bytes,
                        void *stream, bool trust_tables) {
  BEVB200_REQUIRE(b > 0 && d > 0 && h > 0 && w > 0 && c > 0, "bad output shape");
  BEVB200_REQUIRE(n >= 0 && n_intervals >= 0, "negative size");
  BEVB200_REQUIRE(out != nullptr, "null out");
  BEVB200_REQUIRE((long long)b * d * h * w * c < (1ll << 40), "output too large");
  BEVB200_REQUIRE((long long)b * d * h * w < (1ll << 31), "grid has too many cells");
  cudaStream_t st = (cudaStream_t)stream;
  size_t out_bytes = (size_t)b * d * h * w * c * sizeof(float);
  // plan tables (perm != null) with B*D == 1 are in ascending cell order: the pooling kernel
  // zero-fills the empty cells itself; every other case pre-zeroes the grid
  bool tuned = false;
  switch (c) { case 16: case 32: case 64: case 80: case 96: case 128: case 160: case 256: tuned = true; }
  const bool aligned16 = ((uintptr_t)x % 16 == 0) && ((uintptr_t)out % 16 == 0);
  const int zfill = (perm != nullptr && b * d == 1 && n > 0 && n_intervals > 0 && tuned && aligned16 &&
                     trust_tables) ? 1 : 0;
  if (!zfill) BEVB200_CUDA(cudaMemsetAsync(out, 0, out_bytes, st));
  if (n == 0 || n_intervals == 0) return BEVB200_OK;
  BEVB200_REQUIRE(x && geom && starts && lengths, "null input");
  PoolDims dm{b, d, h, w};
  int rc = BEVB200_OK;
  bool aligned = ((uintptr_t)x % 16 == 0) && ((uintptr_t)out % 16 == 0);
#define CALL_FWD(Q, G)                                                                         \
  do {                                                                                         \
    if (ws_bytes < pool_partial_bytes(n, c) || ws == nullptr) {                                \
      snprintf(g_last_error, sizeof(g_last_error), "bev_pool: workspace too small (%zu < %zu)", \
               ws_bytes, pool_partial_bytes(n, c));                                            \
      return BEVB200_EWORKSPACE;                                                               \
    }                                                                                          \
    rc = launch_fwd_tma<Q>(x, perm, geom, starts, n, c, n_intervals, dm, out, ws, zfill, st);    \
  } while (0)
#define CALL_FWD_GENERIC()                                                                     \
  do {                                                                                         \
    BEVB200_LAUNCH(bevpool_fwd_generic_kernel, grid_for((long long)n_intervals * c, 256), 256, 0, \
                   st, x, perm, geom, starts, lengths, n, c, n_intervals, dm, out);            \
  } while (0)
  if (!aligned) {
    CALL_FWD_GENERIC();
  } else {
    BEVB200_POOL_DISPATCH(c, CALL_FWD, CALL_FWD_GENERIC());
  }
#undef CALL_FWD
#undef CALL_FWD_GENERIC
  return rc;
}

static int pool_backward(int b, int d, int h, int w, int n, int n_total, int c, int n_intervals,
                         const float *og, const int32_t *perm, const int32_t *geom,
                         const int32_t *starts, const int32_t *lengths, float *xg, void *stream) {
  BEVB200_REQUIRE(b > 0 && d > 0 && h > 0 && w > 0 && c > 0, "bad grid shape");
  BEVB200_REQUIRE(n >= 0 && n_total >= n && n_intervals >= 0, "bad sizes");
  if (n_total == 0) return BEVB200_OK;
  BEVB200_REQUIRE(xg != nullptr, "null x_grad");
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0 || n_intervals == 0) {
    BEVB200_CUDA(cudaMemsetAsync(xg, 0, (size_t)n_total * c * sizeof(float), st));
    return BEVB200_OK;
  }
  BEVB200_REQUIRE(og && geom && starts && lengths, "null input");
  PoolDims dm{b, d, h, w};
  int rc = BEVB200_OK;
  bool aligned = ((uintptr_t)og % 16 == 0) && ((uintptr_t)xg % 16 == 0);
#define CALL_BWD(Q, G) \
  rc = launch_bwd<Q, G>(og, perm, geom, starts, lengths, n, n_total, n_intervals, dm, xg, st)
#define CALL_BWD_GENERIC()                                                                     \
  do {                                                                                         \
    BEVB200_CUDA(cudaMemsetAsync(xg, 0, (size_t)n_total * c * sizeof(float), st));             \
    BEVB200_LAUNCH(bevpool_bwd_generic_kernel, grid_for((long long)n_intervals * c, 256), 256, 0, \
                   st, og, perm, geom, starts, lengths, n, c, n_intervals, dm, xg);            \
  } while (0)
  if (!aligned) {
    CALL_BWD_GENERIC();
  } else {
    BEVB200_POOL_DISPATCH(c, CALL_BWD, CALL_BWD_GENERIC());
  }
#undef CALL_BWD
#undef CALL_BWD_GENERIC
  return rc;
}

// ---------------------------------------------------------------------------------------
// precompute: quantise / filter / rank / sort / interval table
// ---------------------------------------------------------------------------------------
struct QuantParams {
  float lower[3], dx[3];
  int nx[3];
  int B, n_per_batch;
};

// rank of a lidar-frame point, or `dropped_key` (one past the largest rank) when filtered out
__device__ __forceinline__ uint32_t pool_rank_of_xyz(const float xyz[3], int i, const QuantParams &p, uint32_t dropped_key) {
  // base.py:149: ((geom - (bx - dx/2)) / dx).long()  -- fp32 sub, fp32 IEEE div, trunc to 0
  long long idx[3];
  bool kept = true;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float v = __fdiv_rn(__fsub_rn(xyz[k], p.lower[k]), p.dx[k]);
    long long q = (long long)v;  // cvt.rzi.s64.f32 (NaN -> 0x8000.. : dropped below)
    idx[k] = q;
    kept = kept && q >= 0 && q < p.nx[k] && (v == v);
  }
  if (!kept) return dropped_key;
  int b = i / p.n_per_batch;
  // bev_pool.py:87-92 with (B, D, H, W) = (B, nz, nx, ny): x*(W*D*B) + y*(D*B) + z*B + b
  long long W = p.nx[1], D = p.nx[2], Bn = p.B;
  return (uint32_t)(idx[0] * (W * D * Bn) + idx[1] * (D * Bn) + idx[2] * Bn + b);
}

// keys[i] = rank of point i, or `dropped_key`
__global__ void pool_rank_from_geom_kernel(const float *__restrict__ geom, int n, QuantParams p,
                                           uint32_t dropped_key, uint32_t *__restrict__ keys,
                                           uint32_t *__restrict__ vals) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float xyz[3] = {geom[3ll * i], geom[3ll * i + 1], geom[3ll * i + 2]};
    keys[i] = pool_rank_of_xyz(xyz, i, p, dropped_key);
    vals[i] = (uint32_t)i;
  }
}

// BaseTransform.get_geometry (base.py:92-135) fused into the rank pass: the 96 MB [B, N, D, fH, fW, 3] tensor of
// lidar-frame frustum points is never written.  Explicit fp32, no FMA contraction, products summed left to right:
//   p = f - post_trans;  q = inv(post_rot) . p;  u = (q.x * q.z, q.y * q.z, q.z);  v = (R . inv(K)) . u + t
//   [v = extra_R . v] [v += extra_t]
// cam[c] = {inv(post_rot) 9, post_trans 3, R.inv(K) 9, t 3} (24 floats, the 3x3 inverses / product come from the
// caller exactly as the reference computes them with torch); extra[b] = {extra_R 9, extra_t 3} or null.
__device__ __forceinline__ void mat3_vec(const float *m, const float in[3], float out[3]) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
    out[r] = __fadd_rn(__fadd_rn(__fmul_rn(m[3 * r], in[0]), __fmul_rn(m[3 * r + 1], in[1])), __fmul_rn(m[3 * r + 2], in[2]));
}
__global__ void pool_rank_from_cameras_kernel(const float *__restrict__ frustum, int n_frustum, int cams_per_batch,
                                              const float *__restrict__ cam, const float *__restrict__ extra, int n,
                                              QuantParams p, uint32_t dropped_key, uint32_t *__restrict__ keys,
                                              uint32_t *__restrict__ vals, float *__restrict__ geom_out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int c = i / n_frustum, f = i - c * n_frustum;
    const float *m = cam + 24 * c;
    float a[3], q[3], v[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) a[k] = __fsub_rn(__ldg(frustum + 3 * f + k), __ldg(m + 9 + k));
    mat3_vec(m, a, q);
    const float u[3] = {__fmul_rn(q[0], q[2]), __fmul_rn(q[1], q[2]), q[2]};
    mat3_vec(m + 12, u, v);
#pragma unroll
    for (int k = 0; k < 3; ++k) v[k] = __fadd_rn(v[k], __ldg(m + 21 + k));
    if (extra) {
      const float *e = extra + 12 * (c / cams_per_batch);
      float w[3];
      mat3_vec(e, v, w);
#pragma unroll
      for (int k = 0; k < 3; ++k) v[k] = __fadd_rn(w[k], __ldg(e + 9 + k));
    }
    if (geom_out) {
      geom_out[3ll * i] = v[0]; geom_out[3ll * i + 1] = v[1]; geom_out[3ll * i + 2] = v[2];
    }
    keys[i] = pool_rank_of_xyz(v, i, p, dropped_key);
    vals[i] = (uint32_t)i;
  }
}

__global__ void pool_rank_from_coords_kernel(const long long *__restrict__ coords, int n, int B,
                                             int D, int H, int W, uint32_t dropped_key,
                                             uint32_t *__restrict__ keys,
                                             uint32_t *__restrict__ vals) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    long long cx = coords[4ll * i], cy = coords[4ll * i + 1], cz = coords[4ll * i + 2],
              cb = coords[4ll * i + 3];
    bool kept = cx >= 0 && cx < H && cy >= 0 && cy < W && cz >= 0 && cz < D && cb >= 0 && cb < B;
    keys[i] = kept ? (uint32_t)(cx * ((long long)W * D * B) + cy * ((long long)D * B) + cz * B + cb)
                   : dropped_key;
    vals[i] = (uint32_t)i;
  }
}

// after the sort: decode ranks into (x, y, z, b), flag interval heads
__global__ void pool_heads_kernel(const uint32_t *__restrict__ keys_sorted, int n,
                                  uint32_t dropped_key, int B, int D, int W,
                                  int32_t *__restrict__ ranks_sorted,
                                  int32_t *__restrict__ geom_sorted,
                                  uint32_t *__restrict__ head_flags, int32_t *__restrict__ counts) {
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
    uint32_t key = keys_sorted[r];
    bool kept = key < dropped_key;
    uint32_t prev = r > 0 ? keys_sorted[r - 1] : 0xffffffffu;
    head_flags[r] = (kept && (r == 0 || key != prev)) ? 1u : 0u;
    ranks_sorted[r] = (int32_t)key;
    int4 g = make_int4(0, 0, 0, 0);
    if (kept) {
      uint32_t rem = key;
      g.w = rem % B; rem /= B;
      g.z = rem % D; rem /= D;
      g.y = rem % W; rem /= W;
      g.x = rem;
      uint32_t next = r + 1 < n ? keys_sorted[r + 1] : dropped_key;
      if (next >= dropped_key) counts[0] = r + 1;  // n_kept (exactly one thread hits this)
    }
    *reinterpret_cast<int4 *>(geom_sorted + 4ll * r) = g;
  }
}

__global__ void pool_starts_kernel(const uint32_t *__restrict__ head_flags,
                                   const uint32_t *__restrict__ head_pos, int n,
                                   int32_t *__restrict__ starts) {
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x)
    if (head_flags[r]) starts[head_pos[r]] = r;
}

__global__ void pool_lengths_kernel(const int32_t *__restrict__ starts,
                                    const int32_t *__restrict__ counts,
                                    int32_t *__restrict__ lengths) {
  const int n_kept = counts[0], n_int = counts[1];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_int; i += gridDim.x * blockDim.x)
    lengths[i] = (i + 1 < n_int ? starts[i + 1] : n_kept) - starts[i];
}

struct PrepareWs {
  uint32_t *keys_a, *keys_b, *vals_a, *flags, *pos, *tiles;
  void *cub_tmp;
  size_t cub_bytes;
};

static size_t prepare_layout(int n, void *ws, size_t ws_bytes, PrepareWs *out) {
  Arena a(ws, ws_bytes);
  PrepareWs w;
  w.keys_a = a.take<uint32_t>(n);
  w.keys_b = a.take<uint32_t>(n);
  w.vals_a = a.take<uint32_t>(n);
  w.flags = a.take<uint32_t>(n);
  w.pos = a.take<uint32_t>(n);
  w.tiles = a.take<uint32_t>(scan_scratch_elems(n));
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const uint32_t *)nullptr,
                                  (uint32_t *)nullptr, (const uint32_t *)nullptr,
                                  (uint32_t *)nullptr, n > 0 ? n : 1, 0, 32, (cudaStream_t)0);
  w.cub_bytes = cub_bytes;
  w.cub_tmp = a.take<char>(cub_bytes);
  if (out) *out = w;
  return a.off;
}

static int prepare_finish(PrepareWs &w, int n, long long total_cells, int B, int D, int W,
                          int32_t *ranks_sorted, int32_t *perm, int32_t *geom_sorted,
                          int32_t *starts, int32_t *lengths, int32_t *counts, cudaStream_t st) {
  int end_bit = 1;
  while ((1ll << end_bit) <= total_cells && end_bit < 32) ++end_bit;  // keys in [0, total_cells]
  size_t cub_bytes = w.cub_bytes;
  // stable LSD radix sort: equal ranks keep ascending original index
  BEVB200_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, cub_bytes, (const uint32_t *)w.keys_a,
                                               w.keys_b, (const uint32_t *)w.vals_a,
                                               (uint32_t *)perm, n, 0, end_bit, st));
  g_launch_count += (end_bit + 7) / 8 + 2;  // cub: histogram + one onesweep pass per 8 bits
  BEVB200_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), st));
  BEVB200_LAUNCH(pool_heads_kernel, grid_for(n, 256), 256, 0, st, w.keys_b, n,
                 (uint32_t)total_cells, B, D, W, ranks_sorted, geom_sorted, w.flags, counts);
  int rc = exclusive_scan_u32(w.flags, w.pos, n, w.tiles, (uint32_t *)(counts + 1), false, st);
  if (rc) return rc;
  BEVB200_LAUNCH(pool_starts_kernel, grid_for(n, 256), 256, 0, st, w.flags, w.pos, n, starts);
  BEVB200_LAUNCH(pool_lengths_kernel, grid_for(n, 256), 256, 0, st, starts, counts, lengths);
  return BEVB200_OK;
}

}  // namespace bevb200

using namespace bevb200;

extern "C" {

size_t bevb200_bev_pool_workspace_bytes(int n, int c) {
  if (n < 0 || c <= 0) return 0;
  return pool_partial_bytes(n, c);
}

int bevb200_bev_pool(int b, int d, int h, int w, int n, int c, int n_intervals, const float *x,
                     const int32_t *geom_feats, const int32_t *interval_starts,
                     const int32_t *interval_lengths, float *out, void *workspace,
                     size_t workspace_bytes, void *stream) {
  return pool_forward(b, d, h, w, n, c, n_intervals, x, nullptr, geom_feats, interval_starts,
                      interval_lengths, out, workspace, workspace_bytes, stream, false);
}

int bevb200_bev_pool_perm(int b, int d, int h, int w, int n, int c, int n_intervals,
                          const float *x, const int32_t *perm, const int32_t *geom_feats,
                          const int32_t *interval_starts, const int32_t *interval_lengths,
                          float *out, void *workspace, size_t workspace_bytes, void *stream) {
  BEVB200_REQUIRE(perm != nullptr || n == 0, "null perm");
  return pool_forward(b, d, h, w, n, c, n_intervals, x, perm, geom_feats, interval_starts,
                      interval_lengths, out, workspace, workspace_bytes, stream, true);
}

int bevb200_bev_pool_grad(int b, int d, int h, int w, int n, int c, int n_intervals,
                          const float *out_grad, const int32_t *geom_feats,
                          const int32_t *interval_starts, const int32_t *interval_lengths,
                          float *x_grad, void *stream) {
  return pool_backward(b, d, h, w, n, n, c, n_intervals, out_grad, nullptr, geom_feats,
                       interval_starts, interval_lengths, x_grad, stream);
}

int bevb200_bev_pool_grad_perm(int b, int d, int h, int w, int n, int n_total, int c,
                               int n_intervals, const float *out_grad, const int32_t *perm,
                               const int32_t *geom_feats, const int32_t *interval_starts,
                               const int32_t *interval_lengths, float *x_grad, void *stream) {
  BEVB200_REQUIRE(perm != nullptr || n_total == 0, "null perm");
  return pool_backward(b, d, h, w, n, n_total, c, n_intervals, out_grad, perm, geom_feats,
                       interval_starts, interval_lengths, x_grad, stream);
}

int bevb200_bev_pool_lift(int b, int d, int h, int w, int n, int c, int n_intervals, const float *depth,
                          const float *ctx, int depth_bins, int pixels_per_camera, const int32_t *perm,
                          const int32_t *geom_feats, const int32_t *interval_starts,
                          const int32_t *interval_lengths, float *out, void *workspace,
                          size_t workspace_bytes, void *stream) {
  (void)interval_lengths;
  BEVB200_REQUIRE(b > 0 && d > 0 && h > 0 && w > 0 && c > 0 && n >= 0 && n_intervals >= 0, "bad sizes");
  BEVB200_REQUIRE(out != nullptr, "null out");
  BEVB200_REQUIRE(depth_bins > 0 && pixels_per_camera > 0, "bad lift dims");
  BEVB200_REQUIRE((long long)b * d * h * w < (1ll << 31), "grid has too many cells");
  cudaStream_t st = (cudaStream_t)stream;
  const int zfill = (b * d == 1 && n > 0 && n_intervals > 0) ? 1 : 0;
  if (!zfill) BEVB200_CUDA(cudaMemsetAsync(out, 0, (size_t)b * d * h * w * c * sizeof(float), st));
  if (n == 0 || n_intervals == 0) return BEVB200_OK;
  BEVB200_REQUIRE(depth && ctx && perm && geom_feats && interval_starts, "null input");
  BEVB200_REQUIRE(((uintptr_t)ctx % 16 == 0) && ((uintptr_t)out % 16 == 0), "ctx / out must be 16-byte aligned");
  if (workspace == nullptr || workspace_bytes < pool_partial_bytes(n, c)) {
    snprintf(g_last_error, sizeof(g_last_error), "bev_pool_lift: workspace too small");
    return BEVB200_EWORKSPACE;
  }
  PoolDims dm{b, d, h, w};
  LiftDims lift{depth_bins, pixels_per_camera};
#define CALL_LIFT(Q, G) return launch_fwd_tma<Q>(ctx, perm, geom_feats, interval_starts, n, c, n_intervals, dm, \
                                                 out, workspace, zfill, st, depth, lift)
  BEVB200_POOL_DISPATCH(c, CALL_LIFT, BEVB200_REQUIRE(false, "bev_pool_lift: channel count not in {16,32,64,80,96,128,160,256}"));
#undef CALL_LIFT
  return BEVB200_OK;
}

int bevb200_bev_channels_first(const float *in, float *out, int batch, int nz, int rows, int c,
                               long long out_batch_stride, void *stream) {
  BEVB200_REQUIRE(batch > 0 && nz > 0 && rows > 0 && c > 0 && in && out, "bad argument");
  BEVB200_REQUIRE((long long)batch * nz <= 65535, "too many (batch, z) slabs");
  if (out_batch_stride == 0) out_batch_stride = (long long)nz * rows * c;
  BEVB200_REQUIRE(out_batch_stride >= (long long)nz * rows * c, "output batch stride too small");
  dim3 grid((rows + 31) / 32, (c + 31) / 32, batch * nz);
  BEVB200_LAUNCH(bev_channels_first_kernel, grid, 256, 0, (cudaStream_t)stream, in, out, rows, c, nz,
                 out_batch_stride);
  return BEVB200_OK;
}

size_t bevb200_bev_pool_prepare_workspace_bytes(int n_total) {
  if (n_total < 0) return 0;
  return prepare_layout(n_total, nullptr, 0, nullptr);
}

int bevb200_bev_pool_prepare_geom(const float *geom_xyz, int n_total, int n_per_batch,
                                  const float *lower_host, const float *dx_host,
                                  const int32_t *nx_host, int B, int32_t *ranks_sorted,
                                  int32_t *perm, int32_t *geom_sorted, int32_t *interval_starts,
                                  int32_t *interval_lengths, int32_t *counts, void *workspace,
                                  size_t workspace_bytes, void *stream) {
  BEVB200_REQUIRE(n_total >= 0 && B > 0 && n_per_batch > 0, "bad sizes");
  BEVB200_REQUIRE(lower_host && dx_host && nx_host && counts, "null argument");
  BEVB200_REQUIRE((long long)n_per_batch * B >= n_total, "n_per_batch * B < n_total");
  long long total_cells = (long long)nx_host[0] * nx_host[1] * nx_host[2] * B;
  BEVB200_REQUIRE(nx_host[0] > 0 && nx_host[1] > 0 && nx_host[2] > 0, "bad grid");
  BEVB200_REQUIRE(total_cells < 0xfffffff0ll, "grid too large for 32-bit ranks");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_total == 0) {
    BEVB200_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), st));
    return BEVB200_OK;
  }
  BEVB200_REQUIRE(geom_xyz && ranks_sorted && perm && geom_sorted && interval_starts &&
                      interval_lengths, "null argument");
  PrepareWs w;
  size_t need = prepare_layout(n_total, workspace, workspace_bytes, &w);
  if (workspace == nullptr || workspace_bytes < need) {
    snprintf(g_last_error, sizeof(g_last_error), "bev_pool_prepare: workspace too small (%zu < %zu)",
             workspace_bytes, need);
    return BEVB200_EWORKSPACE;
  }
  QuantParams p;
  for (int k = 0; k < 3; ++k) {
    p.lower[k] = lower_host[k];
    p.dx[k] = dx_host[k];
    p.nx[k] = nx_host[k];
  }
  p.B = B;
  p.n_per_batch = n_per_batch;
  BEVB200_LAUNCH(pool_rank_from_geom_kernel, grid_for(n_total, 256), 256, 0, st, geom_xyz, n_total,
                 p, (uint32_t)total_cells, w.keys_a, w.vals_a);
  // (B, D, H, W) = (B, nz, nx, ny)
  return prepare_finish(w, n_total, total_cells, B, nx_host[2], nx_host[1], ranks_sorted, perm,
                        geom_sorted, interval_starts, interval_lengths, counts, st);
}

int bevb200_bev_pool_prepare_cameras(const float *frustum, int n_frustum, int cameras, int cams_per_batch,
                                     const float *cam_params, const float *extra_params, const float *lower_host,
                                     const float *dx_host, const int32_t *nx_host, int B, float *geom_out,
                                     int32_t *ranks_sorted, int32_t *perm, int32_t *geom_sorted,
                                     int32_t *interval_starts, int32_t *interval_lengths, int32_t *counts,
                                     void *workspace, size_t workspace_bytes, void *stream) {
  BEVB200_REQUIRE(n_frustum > 0 && cameras > 0 && cams_per_batch > 0 && B > 0 && cameras == B * cams_per_batch, "bad sizes");
  BEVB200_REQUIRE((long long)n_frustum * cameras < (1ll << 31), "too many frustum points");
  BEVB200_REQUIRE(frustum && cam_params && lower_host && dx_host && nx_host && counts, "null argument");
  const int n_total = n_frustum * cameras;
  long long total_cells = (long long)nx_host[0] * nx_host[1] * nx_host[2] * B;
  BEVB200_REQUIRE(nx_host[0] > 0 && nx_host[1] > 0 && nx_host[2] > 0, "bad grid");
  BEVB200_REQUIRE(total_cells < 0xfffffff0ll, "grid too large for 32-bit ranks");
  BEVB200_REQUIRE(ranks_sorted && perm && geom_sorted && interval_starts && interval_lengths, "null argument");
  cudaStream_t st = (cudaStream_t)stream;
  PrepareWs w;
  size_t need = prepare_layout(n_total, workspace, workspace_bytes, &w);
  if (workspace == nullptr || workspace_bytes < need) {
    snprintf(g_last_error, sizeof(g_last_error), "bev_pool_prepare: workspace too small (%zu < %zu)",
             workspace_bytes, need);
    return BEVB200_EWORKSPACE;
  }
  QuantParams p;
  for (int k = 0; k < 3; ++k) {
    p.lower[k] = lower_host[k];
    p.dx[k] = dx_host[k];
    p.nx[k] = nx_host[k];
  }
  p.B = B;
  p.n_per_batch = n_frustum * cams_per_batch;
  BEVB200_LAUNCH(pool_rank_from_cameras_kernel, grid_for(n_total, 256), 256, 0, st, frustum, n_frustum, cams_per_batch,
                 cam_params, extra_params, n_total, p, (uint32_t)total_cells, w.keys_a, w.vals_a, geom_out);
  return prepare_finish(w, n_total, total_cells, B, nx_host[2], nx_host[1], ranks_sorted, perm, geom_sorted,
                        interval_starts, interval_lengths, counts, st);
}

int bevb200_bev_pool_prepare_coords(const int64_t *coords, int n, int B, int D, int H, int W,
                                    int32_t *ranks_sorted, int32_t *perm, int32_t *geom_sorted,
                                    int32_t *interval_starts, int32_t *interval_lengths,
                                    int32_t *counts, void *workspace, size_t workspace_bytes,
                                    void *stream) {
  BEVB200_REQUIRE(n >= 0 && B > 0 && D > 0 && H > 0 && W > 0, "bad sizes");
  BEVB200_REQUIRE(counts != nullptr, "null counts");
  long long total_cells = (long long)B * D * H * W;
  BEVB200_REQUIRE(total_cells < 0xfffffff0ll, "grid too large for 32-bit ranks");
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    BEVB200_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), st));
    return BEVB200_OK;
  }
  BEVB200_REQUIRE(coords && ranks_sorted && perm && geom_sorted && interval_starts &&
                      interval_lengths, "null argument");
  PrepareWs w;
  size_t need = prepare_layout(n, workspace, workspace_bytes, &w);
  if (workspace == nullptr || workspace_bytes < need) {
    snprintf(g_last_error, sizeof(g_last_error), "bev_pool_prepare: workspace too small (%zu < %zu)",
             workspace_bytes, need);
    return BEVB200_EWORKSPACE;
  }
  BEVB200_LAUNCH(pool_rank_from_coords_kernel, grid_for(n, 256), 256, 0, st,
                 (const long long *)coords, n, B, D, H, W, (uint32_t)total_cells, w.keys_a, w.vals_a);
  return prepare_finish(w, n, total_cells, B, D, W, ranks_sorted, perm, geom_sorted,
                        interval_starts, interval_lengths, counts, st);
}

}  // extern "C"
