// Sparse convolution forward, generation 6 (BF16x3 precision): pre-split operands, no register stage.
//
//   out[o, :] = epilogue( sum_k features[nbr[k, o], :] @ W[k] )          (spconv_ops.h:260-361)
//
// What bounded generation 5 (profiles/r1_ncu_full_v5.md, r1_conv_v5_ablation.txt): every K block went
// gather -> staging slot -> ONE convert warp per row quarter (8 LDS.128, the fp32 -> bf16 hi/lo split,
// two tcgen05.st, wait::st) -> MMA, i.e. four mbarrier hand-offs and a serial ~130-instruction register
// chain per 128x32 block, and every CTA re-streamed the layer's whole weight tensor through L2 for its
// single 128-row tile (the L2 -> SM crossbar ran at 8 TB/s, half of it weights).  Here:
//   * PRE-SPLIT FEATURES.  A feature row is stored as the bf16 image the tensor core consumes: per
//     group of 16 channels 32 B of bf16 "hi" followed by 32 B of bf16 "lo" (hi = rn(x), lo = rn(x - hi);
//     4 bytes per element, like fp32).  The producing conv writes that image from its epilogue (and
//     fp32 rows only where dense() needs them; a residual is read from a split image too); the split is done once per row instead
//     of once per (row, kernel offset) visit.
//   * NO CONVERT WARPS, NO A RING IN TMEM.  Gather warps copy the rows with cp.async.cg straight into
//     the K-major SWIZZLE_128B tile the UMMA descriptor describes (row r at r*128 B, 16-byte chunk c at
//     (c ^ (r & 7))); the copies signal the stage's mbarrier themselves (cp.async.mbarrier.arrive.noinc)
//     and the MMA warp multiplies out of shared memory (SS form).  Two hand-offs per K block.
//   * A_hi x [W_hi | W_lo] as ONE N = 2*Cout MMA (Cout <= 64) + A_lo x W_hi: every A byte is read from
//     shared memory once.  Cout = 128 runs the three-product form out of a [W_hi | W_lo]-per-row image.
//   * R ROW TILES PER WEIGHT STAGE.  A CTA owns a contiguous range of 128-row tiles and walks it R
//     tiles at a time (R accumulators in its 256 TMEM columns: 4 / 4 / 2 / 2 for Cout 16 / 32 / 64 /
//     128); a weight stage is fetched once per R tiles, which divides the weight stream by R.
//   * PERSISTENT, DEVICE-SIDE COUNTS.  The grid is 2 CTAs per SM; the number of output rows is read
//     from device memory (n_out_dev), so a strided conv needs no host round trip for its output count
//     and the whole encoder can be captured in a CUDA graph.
// Warp roles (10 warps): 0-7 gather (row quarter = warp & 3; the two halves take alternate items) and
// epilogue (TMEM lane quarter = warp & 3, the halves split the columns); 8 MMA issuer (one elected
// lane) + TMEM allocation; 9 weight stream (cp.async.bulk ring).
// A TMA row gather (cp.async.bulk.tensor ... tile::gather4, four rows per instruction, from an eleventh warp)
// was measured 2x slower than the cp.async gather and removed: the TMA unit's gather4 rate is lower than what
// the LDGSTS gather sustains; measurement in profiles/r2_gather4_probe.txt.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace bevb200 {

constexpr int kV6Threads = 10 * 32;
constexpr int kV6TileM = 128;
constexpr int kV6AStageBytes = kV6TileM * 128;   // 128 rows x 128 B
constexpr int kV6MaxA = 12, kV6MaxB = 4;

struct V6Params {
  const uint8_t *fsplit;        // split image of the input rows, c_in * 4 bytes per row
  const uint8_t *wpacked;
  const int32_t *nbr;           // [kvol][nbr_stride]
  long long nbr_stride;
  const int32_t *n_out_dev;     // optional device-side row count (<= n_out)
  const float *scale, *shift, *residual;
  const uint8_t *residual_split; // residual rows as a split image (x = hi + lo, exact to 2^-17 |x|): lets a producer
                                 // skip its fp32 copy; may alias out_split (a lane reads its chunk before writing it)
  float *out;                   // optional fp32 rows [n_out, c_out]
  uint8_t *out_split;           // optional split image [n_out, c_out * 4 B]
  int n_in, n_out;
  int c_in, c_out, kvol, relu;
  int nkb, cin_shift;
  int r_shift;                  // log2(max row tiles per weight stage)
  int acc_cols;                 // TMEM columns per row tile
  int merged;                   // 1: A_hi x [W_hi | W_lo] (Cout <= 64); 0: three products (Cout = 128)
  int nsa, nsb, b_stage_bytes;
  int tmem_cols;
};

__device__ __forceinline__ void tc_mma_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16u(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_ld8u(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// hi = rn_bf16(x), lo = rn_bf16(x - hi) for a pair of values, packed (first value in the low half)
__device__ __forceinline__ void split_pair(float x0, float x1, uint32_t &hi, uint32_t &lo) {
  const uint32_t h = cvt_bf16x2(x1, x0);
  const float h0 = __uint_as_float(h << 16), h1 = __uint_as_float(h & 0xffff0000u);
  hi = h;
  lo = cvt_bf16x2(x1 - h1, x0 - h0);
}

// Epilogue of NC (8 or 16) consecutive channels [c0, c0 + NC) of one row: folded BN, residual, ReLU,
// then the fp32 row and / or its split image.  NC channels = NC/8 16-byte chunks of hi and of lo.
template <int NC>
__device__ __forceinline__ void v6_store_chunk(const V6Params &p, float (&acc)[NC], int orow, int c0) {
  const int c_out = p.c_out;
  float y[NC];
#pragma unroll
  for (int e = 0; e < NC; ++e) {
    float t = acc[e];
    if (p.scale) t *= __ldg(p.scale + c0 + e);
    if (p.shift) t += __ldg(p.shift + c0 + e);
    y[e] = t;
  }
  if (p.residual) {
    const float4 *res = reinterpret_cast<const float4 *>(p.residual + (long long)orow * c_out + c0);
#pragma unroll
    for (int j = 0; j < NC / 4; ++j) {
      const float4 rv = __ldg(res + j);
      y[4 * j] += rv.x; y[4 * j + 1] += rv.y; y[4 * j + 2] += rv.z; y[4 * j + 3] += rv.w;
    }
  } else if (p.residual_split) {
    // plain loads (the image may be this launch's own out_split, rewritten below by the same lane)
    const uint8_t *row = p.residual_split + (long long)orow * (c_out * 4) + (c0 >> 4) * 64 + (c0 & 15) * 2;
#pragma unroll
    for (int j = 0; j < NC / 8; ++j) {
      const uint4 h = *reinterpret_cast<const uint4 *>(row + 16 * j);
      const uint4 l = *reinterpret_cast<const uint4 *>(row + 32 + 16 * j);
      const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        y[8 * j + 2 * e] += __uint_as_float(hw[e] << 16) + __uint_as_float(lw[e] << 16);
        y[8 * j + 2 * e + 1] += __uint_as_float(hw[e] & 0xffff0000u) + __uint_as_float(lw[e] & 0xffff0000u);
      }
    }
  }
  if (p.relu) {
#pragma unroll
    for (int e = 0; e < NC; ++e) y[e] = fmaxf(y[e], 0.f);
  }
  if (p.out) {
    float4 *dst = reinterpret_cast<float4 *>(p.out + (long long)orow * c_out + c0);
#pragma unroll
    for (int j = 0; j < NC / 4; ++j) dst[j] = make_float4(y[4 * j], y[4 * j + 1], y[4 * j + 2], y[4 * j + 3]);
  }
  if (p.out_split) {
    uint32_t hi[NC / 2], lo[NC / 2];
#pragma unroll
    for (int e = 0; e < NC; e += 2) split_pair(y[e], y[e + 1], hi[e / 2], lo[e / 2]);
    // group g = c0 / 16 starts at g * 64 B: [hi 32 B | lo 32 B]; c0 % 16 is 0 or 8
    uint8_t *row = p.out_split + (long long)orow * (c_out * 4) + (c0 >> 4) * 64 + (c0 & 15) * 2;
#pragma unroll
    for (int j = 0; j < NC / 8; ++j) {
      *reinterpret_cast<uint4 *>(row + 16 * j) = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
      *reinterpret_cast<uint4 *>(row + 32 + 16 * j) = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
    }
  }
}

__global__ void __launch_bounds__(kV6Threads, 2) spconv_v6_kernel(const V6Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  __shared__ uint64_t bars[2 * kV6MaxA + 2 * kV6MaxB + 2];
  __shared__ uint32_t tmem_base_s;
  const uint32_t a_full = smem_u32(&bars[0]), a_empty = smem_u32(&bars[kV6MaxA]);
  const uint32_t b_full = smem_u32(&bars[2 * kV6MaxA]), b_empty = smem_u32(&bars[2 * kV6MaxA + kV6MaxB]);
  const uint32_t acc_full = smem_u32(&bars[2 * kV6MaxA + 2 * kV6MaxB]);
  const uint32_t acc_empty = smem_u32(&bars[2 * kV6MaxA + 2 * kV6MaxB + 1]);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nsa = p.nsa, nsb = p.nsb, nkb = p.nkb, c_out = p.c_out;
  const uint32_t b_ring = smem_base;                                           // nsb weight stages
  const uint32_t a_ring = smem_base + (uint32_t)nsb * (uint32_t)p.b_stage_bytes;   // nsa tiles of 16 KB

  if (tid == 0) {
    for (int s = 0; s < nsa; ++s) {
      mbar_init(a_full + 8 * s, 4);   // one arrival per gather warp of the stage
      mbar_init(a_empty + 8 * s, 1);
    }
    for (int s = 0; s < nsb; ++s) {
      mbar_init(b_full + 8 * s, 1);
      mbar_init(b_empty + 8 * s, 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 8);            // one arrival per gather / epilogue warp
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

  // Programmatic dependent launch: everything above (barriers, TMEM) ran while the previous kernel of the stream was
  // still draining; its results (feature image, row count) are only touched below.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  // this CTA's contiguous range of 128-row tiles (balanced to +-1 tile over the grid)
  int n_out = p.n_out;
  if (p.n_out_dev) n_out = min(n_out, __ldg(p.n_out_dev));
  const int n_tiles = (n_out + kV6TileM - 1) / kV6TileM;
  const int t_begin = (int)((long long)n_tiles * blockIdx.x / gridDim.x);
  const int t_end = (int)((long long)n_tiles * (blockIdx.x + 1) / gridDim.x);

  if (warp < 8) {
    // =============================== gather + epilogue ===================================
    const int q = warp & 3, par = warp >> 2;
    const int m = lane >> 3, c = lane & 7;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const uint32_t row_bytes = (uint32_t)p.c_in * 4u;
    const unsigned long long fbase = reinterpret_cast<unsigned long long>(p.fsplit);
    const int cin_shift = p.cin_shift, cin_mask = p.c_in - 1, kvol = p.kvol, n_in = p.n_in;
    const bool two_offsets = p.c_in == 16;     // a K block then spans two kernel offsets (chunks 0-3 / 4-7)
    const long long nbr_stride = p.nbr_stride;
    // Lane (m, c) of copy instruction t writes PHYSICAL chunk c of row 32 q + 8 m + t -- the eight lanes of a row
    // store 128 contiguous bytes in lane order -- and fetches the LOGICAL chunk c ^ t that the SWIZZLE_128B layout
    // keeps there.  (Permuting the destination instead -- lane c writes chunk c ^ t -- costs a fifth shared-memory
    // wavefront per instruction for every t != 0: ncu, profiles/r2_conv_v6_iterations.md.)
    uint32_t dst_off[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) dst_off[t] = (uint32_t)((q * 32 + 8 * m + t) * 128 + (c << 4));
    // an item is signalled one of this warp's items later (see the hand-off below): that needs a spare stage
    const bool lag = nsa >= 3;
    int pend = -1;          // stage whose copies are committed but not yet signalled
    int gs = 0;             // A ring stage / phase of the first item of the current group
    uint32_t gph = 0, acc_ph = 0;
    for (int tb = t_begin; tb < t_end;) {
      int rs = p.r_shift;
      while ((1 << rs) > t_end - tb) --rs;
      const int r_cur = 1 << rs, n_items = nkb << rs;
      int s = gs + par;     // ... of this warp's first item of the group (nsa >= 2)
      uint32_t ph = gph;
      if (s >= nsa) { s -= nsa; ph ^= 1u; }
      {
        const int tot = gs + n_items;
        gph ^= (uint32_t)(tot / nsa) & 1u;
        gs = tot % nsa;
      }
      // neighbour indices of one item: lane l holds the input row of output row (quarter base + l);
      // they are fetched one item ahead so that the L2 latency hides behind the stage wait
      // (the values are NOT touched here -- not even compared -- so the loads stay in flight across the
      // stage wait; the range check happens where they are consumed)
      auto load_idx = [&](int i, int &v0, int &v1) {
        const int kb = i >> rs, r = i & (r_cur - 1);
        const int row = (tb + r) * kV6TileM + q * 32 + lane;
        const int k0 = two_offsets ? 2 * kb : ((kb * 32) >> cin_shift);
        v0 = v1 = -1;
        if (k0 < kvol && row < n_out) v0 = __ldg(p.nbr + (long long)k0 * nbr_stride + row);
        if (two_offsets && 2 * kb + 1 < kvol && row < n_out)
          v1 = __ldg(p.nbr + (long long)(2 * kb + 1) * nbr_stride + row);
      };
      // A ring of PF index registers per lane: the indices of the warp's item j are loaded while it works on
      // item j - PF.  (One item ahead was not enough: the L1 queue in front of the loads is full of this
      // kernel's own cp.async traffic and ncu showed the warps parked on the index load, not on a stage.)
      constexpr int PF = 4;
      int v0q[PF], v1q[PF];
#pragma unroll
      for (int j = 0; j < PF; ++j) {
        v0q[j] = v1q[j] = -1;
        if (par + 2 * j < n_items) load_idx(par + 2 * j, v0q[j], v1q[j]);
      }
      for (int ibase = par; ibase < n_items; ibase += 2 * PF) {
#pragma unroll
        for (int j = 0; j < PF; ++j) {
        const int i = ibase + 2 * j;
        if (i >= n_items) break;
        const int kb = i >> rs;
        // the 8 source rows of this lane's copies: all shuffles first, then all copies
        int src[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          src[t] = __shfl_sync(0xffffffffu, v0q[j], 8 * m + t);
          if (two_offsets) {
            const int src1 = __shfl_sync(0xffffffffu, v1q[j], 8 * m + t);
            src[t] = ((c ^ t) & 4) ? src1 : src[t];      // logical chunks 4-7 belong to the second offset
          }
          if (src[t] >= n_in) src[t] = -1;
        }
        v0q[j] = v1q[j] = -1;
        if (i + 2 * PF < n_items) load_idx(i + 2 * PF, v0q[j], v1q[j]);     // refill the slot
        mbar_wait(a_empty + 8 * s, ph ^ 1u);
        const uint32_t stage = a_ring + (uint32_t)s * (uint32_t)kV6AStageBytes;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          // byte offset of logical chunk c ^ t inside the source row
          const unsigned long long base = fbase + (unsigned)(((kb * 32 + 4 * (c ^ t)) & cin_mask) << 2);
          cp_async16_row(stage + dst_off[t], base + (unsigned long long)(uint32_t)max(src[t], 0) * row_bytes, src[t]);
        }
        // Completion hand-off.  cp.async.mbarrier.arrive.noinc would signal from every LANE: 32 shared-memory
        // atomics per warp and item -- ncu counted them as 43 % of the LSU's shared-memory wavefronts of this
        // kernel.  Instead the warp commits the item as a cp.async group and signals the PREVIOUS item with ONE
        // arrive once that group has landed (wait_group 1): by then its copies have had a whole item's time.
        asm volatile("cp.async.commit_group;" ::: "memory");
        if (lag) {
          if (pend >= 0) {
            asm volatile("cp.async.wait_group 1;" ::: "memory");
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(a_full + 8 * pend);
          }
          pend = s;
        } else {
          asm volatile("cp.async.wait_group 0;" ::: "memory");
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(a_full + 8 * s);
        }
        s += 2;
        if (s >= nsa) { s -= nsa; ph ^= 1u; }
        }
      }
      if (pend >= 0) {                      // the last item of the group
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(a_full + 8 * pend);
        pend = -1;
      }
      // ------------------------------- epilogue of the group --------------------------------
      mbar_wait(acc_full, acc_ph);
      acc_ph ^= 1u;
      tc_fence_after();
      const int ncol_half = c_out >> 1, col_begin = par * ncol_half;
      for (int r = 0; r < r_cur; ++r) {
        const int orow = (tb + r) * kV6TileM + q * 32 + lane;
        const bool row_ok = orow < n_out;
        const uint32_t tacc = tmem_base + lane_base + (uint32_t)(r * p.acc_cols);
        if (ncol_half >= 16) {
          for (int c0 = col_begin; c0 < col_begin + ncol_half; c0 += 16) {
            float acc[16];
            tc_ld16u(tacc + (uint32_t)c0, acc);
            if (p.merged) {   // columns [c_out, 2 c_out) hold the hi x lo partial sums
              float more[16];
              tc_ld16u(tacc + (uint32_t)(c_out + c0), more);
#pragma unroll
              for (int e = 0; e < 16; ++e) acc[e] += more[e];
            }
            if (row_ok) v6_store_chunk<16>(p, acc, orow, c0);
          }
        } else {              // c_out == 16: 8 columns per half
          float acc[8], more[8];
          tc_ld8u(tacc + (uint32_t)col_begin, acc);
          tc_ld8u(tacc + (uint32_t)(c_out + col_begin), more);
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[e] += more[e];
          if (row_ok) v6_store_chunk<8>(p, acc, orow, col_begin);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
      tb += r_cur;
    }
  } else if (warp == 8) {
    // =============================== MMA issuer ==========================================
    // (A leaner issue loop -- running descriptors, ~50 instead of ~110 SASS instructions per item -- was measured
    // SLOWER at C = 64 / 128 (2.85 vs 2.69 ms for the 21 convs, profiles/r2_conv_v6_iterations.md): this warp is
    // not what paces the CTA once the shared-memory pipe is ~85 % busy, and its denser barrier polling costs
    // shared-memory wavefronts.)
    const uint32_t idesc_n = umma_idesc_bf16(kV6TileM, c_out);
    const uint32_t idesc_2n = umma_idesc_bf16(kV6TileM, 2 * c_out);
    const int merged = p.merged;
    int sa = 0, sb = 0;
    uint32_t pa = 0, pb = 0, pe = 0;
    bool first_group = true;
    for (int tb = t_begin; tb < t_end;) {
      int rs = p.r_shift;
      while ((1 << rs) > t_end - tb) --rs;
      const int r_cur = 1 << rs, n_items = nkb << rs;
      if (!first_group) {                 // the epilogue warps have drained the accumulators
        mbar_wait(acc_empty, pe);
        pe ^= 1u;
        tc_fence_after();
      }
      first_group = false;
      for (int i = 0; i < n_items; ++i) {
        const int kb = i >> rs, r = i & (r_cur - 1);
        // merged image: one weight stage = two K blocks; three-product image: one K block
        const bool b_new = r == 0 && (!merged || (kb & 1) == 0);
        const bool b_done = r == r_cur - 1 && (!merged || (kb & 1) || kb == nkb - 1);
        if (b_new) mbar_wait(b_full + 8 * sb, pb);
        mbar_wait(a_full + 8 * sa, pa);
        tc_fence_after();
        if (elect_one_sync()) {
          const uint32_t a_base = a_ring + (uint32_t)sa * (uint32_t)kV6AStageBytes;
          const uint32_t bstage = b_ring + (uint32_t)sb * (uint32_t)p.b_stage_bytes;
          const uint32_t d = tmem_base + (uint32_t)(r * p.acc_cols);
          const uint64_t bdesc = umma_desc_sw128(bstage);
#pragma unroll
          for (int g = 0; g < 2; ++g) {   // the two 16-channel groups of the K block
            const uint64_t a_hi = umma_desc_sw128(a_base + (uint32_t)(g * 64));
            const uint64_t a_lo = umma_desc_sw128(a_base + (uint32_t)(g * 64 + 32));
            const uint32_t acc0 = (kb == 0 && g == 0) ? 0u : 1u;
            if (merged) {
              const uint64_t b = bdesc + (uint64_t)((kb & 1) * 4 + g * 2);   // 16-byte units along K
              tc_mma_bf16_ss(d, a_hi, b, idesc_2n, acc0);    // hi*hi -> cols [0, c), hi*lo -> [c, 2c)
              tc_mma_bf16_ss(d, a_lo, b, idesc_n, 1u);       // lo*hi -> cols [0, c)
            } else {
              const uint64_t b_hi = bdesc + (uint64_t)(g * 2), b_lo = bdesc + (uint64_t)(4 + g * 2);
              tc_mma_bf16_ss(d, a_lo, b_hi, idesc_n, acc0);
              tc_mma_bf16_ss(d, a_hi, b_lo, idesc_n, 1u);
              tc_mma_bf16_ss(d, a_hi, b_hi, idesc_n, 1u);
            }
          }
          tc_commit(a_empty + 8 * sa);
          if (b_done) tc_commit(b_empty + 8 * sb);
          if (i == n_items - 1) tc_commit(acc_full);
        }
        __syncwarp();
        if (++sa == nsa) { sa = 0; pa ^= 1u; }
        if (b_done && ++sb == nsb) { sb = 0; pb ^= 1u; }
      }
      tb += r_cur;
    }
  } else if (warp == 9) {
    // =============================== weight stream =======================================
    if (lane == 0) {
      const int n_bstages = p.merged ? (nkb + 1) / 2 : nkb;
      const uint32_t bytes = (uint32_t)p.b_stage_bytes;
      int sb = 0;
      uint32_t pb = 1;   // an untouched stage counts as released
      for (int tb = t_begin; tb < t_end;) {
        int rs = p.r_shift;
        while ((1 << rs) > t_end - tb) --rs;
        const uint8_t *src = p.wpacked;
        for (int it = 0; it < n_bstages; ++it) {
          mbar_wait(b_empty + 8 * sb, pb);
          mbar_arrive_expect_tx(b_full + 8 * sb, bytes);
          bulk_copy_g2s(b_ring + (uint32_t)sb * bytes, src, bytes, b_full + 8 * sb);
          src += bytes;
          if (++sb == nsb) { sb = 0; pb ^= 1u; }
        }
        tb += 1 << rs;
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

// ---- operand images --------------------------------------------------------------------------
// fp32 rows [n, c_in] -> split image [n, c_eff * 4 B], c_eff = c_in rounded up to 16 (zero padded).
// One thread per (row, 8 channels): 16 B of hi and 16 B of lo.
__global__ void spconv_v6_split_rows_kernel(const float *__restrict__ in, int n_cap,
                                            const int32_t *__restrict__ n_dev, int c_in, int c_eff,
                                            uint8_t *__restrict__ out) {
  int n = n_cap;
  if (n_dev) n = min(n, __ldg(n_dev));
  const int per_row = c_eff >> 3;
  const long long total = (long long)n * per_row;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
       t += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(t % per_row);
    const long long r = t / per_row;
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = 8 * j + e < c_in ? in[r * c_in + 8 * j + e] : 0.f;
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 8; e += 2) split_pair(x[e], x[e + 1], hi[e / 2], lo[e / 2]);
    uint8_t *dst = out + r * ((long long)c_eff * 4) + (j >> 1) * 64 + (j & 1) * 16;
    *reinterpret_cast<uint4 *>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4 *>(dst + 32) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// Weight image of the three-product form (Cout = 128): one stage per 32-wide K block, row n =
// [W_hi kk 0-15 | W_hi kk 16-31 | W_lo kk 0-15 | W_lo kk 16-31] (32 B each), SWIZZLE_128B.
__global__ void spconv_v6_pack_rows_kernel(const float *__restrict__ w, int kvol, int c_in, int c_in_eff,
                                           int c_out, int nkb, uint16_t *__restrict__ packed) {
  const long long total = (long long)nkb * c_out * 32;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
       t += (long long)gridDim.x * blockDim.x) {
    const int cc = (int)(t % 32);
    const int n = (int)((t / 32) % c_out);
    const int kb = (int)(t / (32ll * c_out));
    const int kk = kb * 32 + cc;
    const int k = kk / c_in_eff, ci = kk % c_in_eff;
    const float v = (k < kvol && ci < c_in) ? w[((long long)k * c_in + ci) * c_out + n] : 0.f;
    uint32_t u = __float_as_uint(v);
    u += 0x7fffu + ((u >> 16) & 1u);
    const uint32_t hb = u >> 16;
    const float lo = v - __uint_as_float(hb << 16);
    uint32_t ul = __float_as_uint(lo);
    ul += 0x7fffu + ((ul >> 16) & 1u);
    // logical 16-byte chunk: hi -> cc / 8 (0..3), lo -> 4 + cc / 8; physical chunk = logical ^ (n & 7)
    uint16_t *row = packed + ((long long)kb * c_out + n) * 64;
    row[(((cc >> 3) ^ (n & 7)) << 3) | (cc & 7)] = (uint16_t)hb;
    row[((((cc >> 3) + 4) ^ (n & 7)) << 3) | (cc & 7)] = (uint16_t)(ul >> 16);
  }
}

// Merged weight image (Cout <= 64), the layout generation 5 uses: [nb64][hi | lo][Cout][64 bf16]; K index
// kk = kb64*64 + c, 16-byte chunk (c / 8) XOR (n & 7), element (c % 8) inside the chunk.  One stage
// (hi image then lo image, 2 * Cout rows of 128 B) serves two 32-wide K blocks.
__global__ void spconv_v6_pack_merged_kernel(const float *__restrict__ w, int kvol, int c_in, int c_in_eff,
                                             int c_out, int nb64, uint16_t *__restrict__ packed) {
  const long long total = (long long)nb64 * c_out * 64;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
       t += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(t % 64);
    const int n = (int)((t / 64) % c_out);
    const int kb = (int)(t / (64ll * c_out));
    const int kk = kb * 64 + c;
    const int k = kk / c_in_eff, ci = kk % c_in_eff;
    const float v = (k < kvol && ci < c_in) ? w[((long long)k * c_in + ci) * c_out + n] : 0.f;
    uint32_t u = __float_as_uint(v);
    u += 0x7fffu + ((u >> 16) & 1u);
    const uint32_t hb = u >> 16;
    const float lo = v - __uint_as_float(hb << 16);
    uint32_t ul = __float_as_uint(lo);
    ul += 0x7fffu + ((ul >> 16) & 1u);
    const int pos = n * 64 + ((((c >> 3) ^ (n & 7)) << 3) | (c & 7));
    packed[((long long)kb * 2 + 0) * c_out * 64 + pos] = (uint16_t)hb;
    packed[((long long)kb * 2 + 1) * c_out * 64 + pos] = (uint16_t)(ul >> 16);
  }
}

int spconv_v6_cin_eff(int c_in) {
  for (int e = 16; e <= 128; e <<= 1)
    if (c_in <= e) return e;
  return 0;
}
bool spconv_v6_shape_ok(int c_in, int c_out, int kvol) {
  return (c_out == 16 || c_out == 32 || c_out == 64 || c_out == 128) && c_in >= 1 &&
         spconv_v6_cin_eff(c_in) != 0 && kvol >= 1 && kvol <= 27;
}
static int v6_nkb(int c_eff, int kvol) { return (kvol * c_eff + 31) / 32; }

size_t spconv_v6_packed_bytes(int c_in, int c_out, int kvol) {
  if (!spconv_v6_shape_ok(c_in, c_out, kvol)) return 0;
  const int nkb = v6_nkb(spconv_v6_cin_eff(c_in), kvol);
  if (c_out <= 64) return (size_t)((nkb + 1) / 2) * 2 * c_out * 128;
  return (size_t)nkb * c_out * 128;
}

int spconv_v6_pack_weights(const float *weight, int c_in, int c_out, int kvol, void *packed, cudaStream_t st) {
  const int ce = spconv_v6_cin_eff(c_in);
  const int nkb = v6_nkb(ce, kvol);
  if (c_out <= 64) {
    const int nb64 = (nkb + 1) / 2;
    BEVB200_LAUNCH(spconv_v6_pack_merged_kernel, grid_for((long long)nb64 * c_out * 64, 256), 256, 0, st,
                   weight, kvol, c_in, ce, c_out, nb64, (uint16_t *)packed);
  } else {
    BEVB200_LAUNCH(spconv_v6_pack_rows_kernel, grid_for((long long)nkb * c_out * 32, 256), 256, 0, st, weight,
                   kvol, c_in, ce, c_out, nkb, (uint16_t *)packed);
  }
  return BEVB200_OK;
}

int spconv_v6_split_rows(const float *features, int n_cap, const int32_t *n_dev, int c_in, void *split,
                         cudaStream_t st) {
  const int ce = spconv_v6_cin_eff(c_in);
  if (n_cap <= 0) return BEVB200_OK;
  BEVB200_LAUNCH(spconv_v6_split_rows_kernel, grid_for((long long)n_cap * (ce / 8), 256), 256, 0, st, features,
                 n_cap, n_dev, c_in, ce, (uint8_t *)split);
  return BEVB200_OK;
}

// split image with an explicit padded channel count (multiple of 16, >= c_in): the filter-gradient kernel wants
// whole 128-byte slabs (spconv_wgrad_tc.cu)
int spconv_v6_split_rows_padded(const float *features, int n, int c_in, int c_eff, void *split, cudaStream_t st) {
  BEVB200_REQUIRE(c_eff >= c_in && c_eff % 16 == 0 && c_in >= 1, "bad padded channel count");
  if (n <= 0) return BEVB200_OK;
  BEVB200_LAUNCH(spconv_v6_split_rows_kernel, grid_for((long long)n * (c_eff / 8), 256), 256, 0, st, features, n,
                 (const int32_t *)nullptr, c_in, c_eff, (uint8_t *)split);
  return BEVB200_OK;
}

// features_split: split image with c_in (multiple of 16, <= 128) channels per row.
int spconv_v6_forward_ex(const void *features_split, const void *packed, const int32_t *nbr, long long nbr_stride,
                         int n_in, int n_out, const int32_t *n_out_dev, int c_in, int c_out, int kvol,
                         const float *scale, const float *shift, const float *residual, const void *residual_split,
                         int relu, float *out, void *out_split, cudaStream_t st);
int spconv_v6_forward(const void *features_split, const void *packed, const int32_t *nbr, long long nbr_stride,
                      int n_in, int n_out, const int32_t *n_out_dev, int c_in, int c_out, int kvol,
                      const float *scale, const float *shift, const float *residual, int relu, float *out,
                      void *out_split, cudaStream_t st) {
  return spconv_v6_forward_ex(features_split, packed, nbr, nbr_stride, n_in, n_out, n_out_dev, c_in, c_out, kvol, scale,
                              shift, residual, nullptr, relu, out, out_split, st);
}
// residual_split: the residual rows as a split image instead of fp32 rows (at most one of the two)
int spconv_v6_forward_ex(const void *features_split, const void *packed, const int32_t *nbr, long long nbr_stride,
                         int n_in, int n_out, const int32_t *n_out_dev, int c_in, int c_out, int kvol,
                         const float *scale, const float *shift, const float *residual, const void *residual_split,
                         int relu, float *out, void *out_split, cudaStream_t st) {
  BEVB200_REQUIRE(!(residual && residual_split), "residual given twice");
  BEVB200_REQUIRE(residual_split == nullptr || (uintptr_t)residual_split % 16 == 0, "residual image must be 16-byte aligned");
  BEVB200_REQUIRE(c_in == spconv_v6_cin_eff(c_in) && spconv_v6_shape_ok(c_in, c_out, kvol), "shape has no tensor-core form");
  BEVB200_REQUIRE(features_split && packed && nbr, "null argument");
  BEVB200_REQUIRE((uintptr_t)features_split % 16 == 0 && (out == nullptr || (uintptr_t)out % 16 == 0) &&
                      (out_split == nullptr || (uintptr_t)out_split % 16 == 0) &&
                      (residual == nullptr || (uintptr_t)residual % 16 == 0) && (uintptr_t)packed % 16 == 0,
                  "operands must be 16-byte aligned");
  if (n_out <= 0) return BEVB200_OK;
  V6Params p;
  memset(&p, 0, sizeof(p));
  p.fsplit = (const uint8_t *)features_split;
  p.wpacked = (const uint8_t *)packed;
  p.nbr = nbr;
  p.nbr_stride = nbr_stride;
  p.n_out_dev = n_out_dev;
  p.scale = scale; p.shift = shift; p.residual = residual;
  p.residual_split = (const uint8_t *)residual_split;
  p.out = out;
  p.out_split = (uint8_t *)out_split;
  p.n_in = n_in; p.n_out = n_out; p.c_in = c_in; p.c_out = c_out; p.kvol = kvol; p.relu = relu;
  p.nkb = v6_nkb(c_in, kvol);
  p.cin_shift = 0;
  while ((1 << p.cin_shift) < c_in) ++p.cin_shift;
  p.merged = c_out <= 64 ? 1 : 0;
  p.acc_cols = p.merged ? (2 * c_out < 32 ? 32 : 2 * c_out) : c_out;
  // two persistent CTAs per SM, each with half of the 512 TMEM columns and of the shared memory
  p.tmem_cols = 256;
  int r = p.tmem_cols / p.acc_cols;
  if (r > 4) r = 4;
  p.r_shift = 0;
  while ((2 << p.r_shift) <= r) ++p.r_shift;
  p.b_stage_bytes = p.merged ? 2 * c_out * 128 : c_out * 128;
  // per CTA: 1 KB alignment slack + weight ring + A ring
  const int budget = 111 * 1024 - 1024;
  p.nsb = (!p.merged || p.b_stage_bytes <= 8192) ? 3 : 2;
  p.nsa = (budget - p.nsb * p.b_stage_bytes) / kV6AStageBytes;
  if (p.nsa > kV6MaxA) p.nsa = kV6MaxA;
  BEVB200_REQUIRE(p.nsa >= 2, "shared memory budget: no room for two A stages");
  const size_t smem = (size_t)p.nsb * p.b_stage_bytes + (size_t)p.nsa * kV6AStageBytes + 1024;
  const int n_tiles = (n_out + kV6TileM - 1) / kV6TileM;
  int grid = 2 * kNumSMs;
  if (grid > n_tiles) grid = n_tiles;
  BEVB200_CUDA(cudaFuncSetAttribute(spconv_v6_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // programmatic stream serialisation: the kernel's prologue overlaps the tail of the previous kernel in the
  // stream (21 back-to-back convs per frame)
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)kV6Threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  BEVB200_CUDA(cudaLaunchKernelEx(&cfg, spconv_v6_kernel, p));
  ++g_launch_count;
  return BEVB200_OK;
}

}  // namespace bevb200

using namespace bevb200;

extern "C" {

int bevb200_spconv_split_channels(int c_in) { return spconv_v6_cin_eff(c_in); }

int bevb200_spconv_split_rows(const float *features, int n, const int32_t *n_dev, int c_in, void *split,
                              void *stream) {
  BEVB200_REQUIRE(n >= 0 && c_in >= 1 && spconv_v6_cin_eff(c_in) != 0, "bad sizes");
  if (n == 0) return BEVB200_OK;
  BEVB200_REQUIRE(features && split && (uintptr_t)split % 16 == 0, "null / unaligned argument");
  return spconv_v6_split_rows(features, n, n_dev, c_in, split, (cudaStream_t)stream);
}

size_t bevb200_spconv_split_weight_bytes(int c_in, int c_out, int kernel_volume) {
  return spconv_v6_packed_bytes(c_in, c_out, kernel_volume);
}

int bevb200_spconv_pack_split_weights(const float *weight, int c_in, int c_out, int kernel_volume, void *packed,
                                      void *stream) {
  BEVB200_REQUIRE(spconv_v6_shape_ok(c_in, c_out, kernel_volume), "shape has no tensor-core form");
  BEVB200_REQUIRE(weight && packed, "null argument");
  return spconv_v6_pack_weights(weight, c_in, c_out, kernel_volume, packed, (cudaStream_t)stream);
}

int bevb200_spconv_forward_split(const void *features_split, const void *packed_weight, const int32_t *nbr,
                                 long long nbr_stride, int n_in, int n_out, const int32_t *n_out_dev, int c_in,
                                 int c_out, int kernel_volume, const float *scale, const float *shift,
                                 const float *residual, int relu, float *out, void *out_split, void *stream) {
  BEVB200_REQUIRE(n_in >= 0 && n_out >= 0 && nbr_stride >= n_out, "bad sizes");
  BEVB200_REQUIRE(out != nullptr || out_split != nullptr, "no output requested");
  return spconv_v6_forward(features_split, packed_weight, nbr, nbr_stride, n_in, n_out, n_out_dev, c_in, c_out,
                           kernel_volume, scale, shift, residual, relu, out, out_split, (cudaStream_t)stream);
}

}  // extern "C"
