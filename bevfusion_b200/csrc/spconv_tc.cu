// Sparse convolution forward on the 5th-gen tensor cores (tcgen05 / TMEM), sm_100a only: the TF32 modes
// (generation 5) and the host dispatch of every precision.  BF16X3 runs generation 6 (spconv_v6.cu).
//
//   out[o, :] = epilogue( sum_k features[nbr[k, o], :] @ W[k] )          (spconv_ops.h:260-361)
//
// One CTA owns 128 output rows (UMMA M = 128, cta_group::1) and all Cout <= 128 columns; the fp32
// accumulator lives in TMEM across all kernel offsets, so every output row is written exactly
// once, after the fused BN / residual / ReLU epilogue.  The GEMM K axis is the concatenation over
// the kernel offsets of the Cin channels, cut into blocks of 32 floats (one 128-byte swizzle row).
//
// Kernel (spconv_tc_kernel_v5, two CTAs per SM, 10 warps each; see the comment above it):
//   warps 0-3  GATHER: cp.async.cg 16-byte copies of the neighbour feature rows, 8 lanes per row =
//              whole 128-byte lines, zero fill (ignore-src) for missing neighbours, into XOR-swizzled
//              4 KB shared-memory staging slots; completion is signalled on an mbarrier by the
//              copies themselves (cp.async.mbarrier.arrive.noinc).
//   warps 4-7  CONVERT: lane = row; 8 conflict-free LDS.128 fetch the row's 32 floats, which are
//              split into two parts (3xTF32: tf32 hi + lo) in registers and written into TENSOR
//              MEMORY with tcgen05.st (A ring of 2-4 stages).
//   warp 8     one elected lane issues tcgen05.mma (kind::tf32) with A from TMEM and B from shared
//              memory (M128 x N=Cout x 32 B of K; per K step lo*hi + hi*lo + hi*hi, or
//              A_hi x [W_hi | W_lo] + A_lo x W_hi as two MMAs when Cout <= 64; fp32 accumulate),
//              tcgen05.commit's the A / B ring slots back and finally the accumulator.
//   warp 9     streams the weights: pre-packed in global memory as the exact K-major SWIZZLE_128B
//              shared-memory image [hi | lo][Cout][128 B] and fetched with one cp.async.bulk
//              (TMA 1-D) per stage into a ring.
//   epilogue   warps 0-7 read the accumulator with tcgen05.ld (32 lanes x 16 columns; warps w and
//              w+4 share TMEM lane quarter w and split the columns), apply scale / shift (folded
//              BatchNorm1d), residual and ReLU, and store the row.
// Earlier generations were removed after their measurements (DESIGN.md 4.6):
//   v2, both operands in shared memory (see below): profiles/r1_conv_layers_v2.txt.
//   v4, 8 producer warps gathering into registers (4 lanes per row) + quad transposes: profiles/
//   r1_conv_layers_v4.txt.  v5's own BF16x3 mode lost to generation 6: profiles/r1_conv_layers_v5_bf16x3.txt,
//   r2_conv_v6_iterations.md.  Multicasting the weight stages across a thread-block cluster: no gain.
//
// Precision (all fp32 in, fp32 accumulate, fp32 out): BEVB200_PREC_BF16X3 (default, generation 6;
// 5e-6 .. 8e-6 of max|out| vs the float64 oracle), BEVB200_PREC_TF32X3 (1e-6 .. 1e-5), BEVB200_PREC_TF32
// (single pass, ~8e-4: below the 1e-4 parity bar, measurement only).
#include "common.cuh"
#include "tc_ptx.cuh"

namespace bevb200 {

constexpr int kTcProducerThreads = 256;
constexpr int kTileM = 128;
constexpr int kKBlock = 32;                       // floats per K block = one 128-byte swizzle row


constexpr int kMaxStages = 8;

// ---- A operand in TENSOR MEMORY (tcgen05.mma TS form) ----------------------------------------
// Measured on v2 (removed): with both operands in shared memory the M128 x N x K8 tf32 MMA re-reads the
// 4 KB A tile from smem on every instruction (3 per K step with the 3xTF32 split), which on top
// of the producers' stores saturates the 128 B/clk shared-memory port -- the kernel was smem
// bound, not tensor bound.  Here the producers write the split A rows straight from registers
// into TMEM (tcgen05.st 32x32b.x16: thread = row = TMEM lane, 16 K values = 16 columns), the MMA
// takes A from TMEM, and shared memory only carries the weights (B): a deep cp.async.bulk ring
// fed by its own warp.  Layout of the 256 TMEM columns of a CTA (two CTAs per SM):
//   [0, acc_cols)            fp32 accumulator, 128 lanes x Cout
//   [acc_cols + 64*s ...)    A ring stage s: 32 columns hi | 32 columns lo   (K block of 32)
constexpr int kTcThreads = 10 * 32;   // warps 0-7 producers/epilogue, 8 MMA issuer, 9 weight loader

struct TcParams {
  const float *features;
  const float *wpacked;
  const int32_t *nbr;
  const float *scale, *shift, *residual;
  float *out;
  int n_in, n_out, c_in, c_out, kvol, relu;
  int nkb, cin_shift;
  int nsa, nsb;       // TMEM A-ring stages, smem B-ring stages
  int acc_cols;       // accumulator columns (>= 32)
  int tmem_cols;      // allocation (power of two >= acc_cols + nsa * nsplit * 32)
  int nmerge;         // A_hi x [W_hi | W_lo] as ONE N = 2*c_out MMA (see the MMA issuer)
  int nsg;            // gather staging slots per row quarter (2..4, 4 KB each)
  int nbr_bytes;      // bytes of the neighbour table in shared memory (multiple of 128)
};

__device__ __forceinline__ void tc_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

// ---------------------------------------------------------------------------------------
// v5: the gather goes through shared memory with cp.async, in WHOLE 128-byte lines.
//
// What bounded v4 (register gather, since removed) after its instruction stream was trimmed: (1) a
// warp-level LDG is processed by the L1 one 128-byte line at a time, ~2 clk per line whatever part of the
// line is used; v4's 4-lanes-per-row loads touch 8 lines per instruction for 64 B each, 256 line-visits
// per K block per CTA, ~530 clk with two CTAs sharing the SM's L1; (2) the 4x4 register transposes
// (16 SHFL + as many selects per 16 floats) that turn "4 lanes per row" into "lane = row" for tcgen05.st.
// v5 splits the producers into four GATHER warps and four CONVERT warps (one of each per TMEM lane
// quarter):
//   gather   lane (m, c) = (lane >> 3, lane & 7) copies the 16-byte chunk c of rows 8m+t, t = 0..7,
//            of its quarter's 32 rows with cp.async.cg (LDGSTS, 16 B, src-size 0 = zero fill for
//            missing neighbours): one instruction = 4 rows x 128 B = 4 whole lines, 128 line-visits
//            per K block per CTA.  The chunk lands at row*128 + ((c ^ (row & 7)) << 4) of a 4 KB
//            staging slot (XOR swizzle: writes and reads are both bank-conflict free);
//            cp.async.mbarrier.arrive.noinc signals the slot's `full` barrier when the bytes landed.
//   convert  lane = row: 8 LDS.128 fetch the row's 32 floats (the transpose is free: it is just the
//            shared-memory addressing), the slot is released, the floats are split hi/lo and
//            written to the TMEM A stage with tcgen05.st; arrive on a_full.
// No data registers are held across the global-load latency (the slots are the prefetch buffer),
// there is no shuffle, and each role's loop is ~55 / ~135 instructions per K block.
// ---------------------------------------------------------------------------------------
constexpr int kStageSlotBytes = 32 * 128;   // one quarter's rows of one K block
constexpr int kMaxGatherSlots = 4;

__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

// NSPLIT: 1 = single-pass TF32, 2 = 3xTF32 (hi/lo tf32 parts)
template <int NSPLIT>
__global__ void __launch_bounds__(kTcThreads, 2) spconv_tc_kernel_v5(const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));
  const int c_out = p.c_out, nsa = p.nsa, nsb = p.nsb, nsg = p.nsg, n_iters = p.nkb;
  const int b_part_bytes = c_out * 128;
  const int b_stage_bytes = NSPLIT * b_part_bytes;
  __shared__ uint64_t bars[4 * kMaxStages + 1 + 8 * kMaxGatherSlots];
  __shared__ uint32_t tmem_base_s;
  const uint32_t a_full = smem_u32(&bars[0]), a_empty = smem_u32(&bars[kMaxStages]);
  const uint32_t b_full = smem_u32(&bars[2 * kMaxStages]), b_empty = smem_u32(&bars[3 * kMaxStages]);
  const uint32_t accbar = smem_u32(&bars[4 * kMaxStages]);
  const uint32_t g_full = smem_u32(&bars[4 * kMaxStages + 1]);                          // [quarter][slot]
  const uint32_t g_empty = smem_u32(&bars[4 * kMaxStages + 1 + 4 * kMaxGatherSlots]);
  const uint32_t ring_bytes = (uint32_t)nsb * (uint32_t)b_stage_bytes;
  int32_t *nbr_s = reinterpret_cast<int32_t *>(smem + ring_bytes);
  const uint32_t slots_base = smem_base + ring_bytes + (uint32_t)p.nbr_bytes;   // 128-byte aligned

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row0 = blockIdx.x * kTileM;

  if (tid == 0) {
    for (int s = 0; s < nsa; ++s) {
      mbar_init(a_full + 8 * s, 4);   // one arrival per convert warp
      mbar_init(a_empty + 8 * s, 1);
    }
    for (int s = 0; s < nsb; ++s) {
      mbar_init(b_full + 8 * s, 1);
      mbar_init(b_empty + 8 * s, 1);
    }
    for (int s = 0; s < 4 * kMaxGatherSlots; ++s) {
      mbar_init(g_full + 8 * s, 32);   // every lane of the gather warp: cp.async arrive (noinc)
      mbar_init(g_empty + 8 * s, 1);
    }
    mbar_init(accbar, 1);
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
  const uint32_t a_ring = tmem_base + (uint32_t)p.acc_cols;            // column offset of A stage 0
  constexpr uint32_t kAStageCols = (uint32_t)NSPLIT * 32u;

  if (warp < 8) {
    const int q = warp & 3;                      // TMEM lane quarter == row quarter of the tile
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    {
      // neighbour table of the tile: all (<= 14) loads of a thread are issued before any is used
      constexpr int kPer = (28 * kTileM + kTcProducerThreads - 1) / kTcProducerThreads;
      const int n_real = p.kvol * kTileM, n_tab = n_real + kTileM, n_out = p.n_out, n_in = p.n_in;   // + a row of -1
      int tv[kPer];
#pragma unroll
      for (int u = 0; u < kPer; ++u) {
        const int i = tid + u * kTcProducerThreads;
        const int k = i >> 7, rr = i & 127, o = row0 + rr;
        tv[u] = (i < n_real && o < n_out) ? __ldg(p.nbr + (long long)k * n_out + o) : -1;
      }
#pragma unroll
      for (int u = 0; u < kPer; ++u) {
        const int i = tid + u * kTcProducerThreads;
        if (i < n_tab) nbr_s[i] = tv[u] >= n_in ? -1 : tv[u];
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kTcProducerThreads) : "memory");
    const uint32_t my_slots = slots_base + (uint32_t)(q * nsg) * (uint32_t)kStageSlotBytes;
    const uint32_t my_full = g_full + 8u * (uint32_t)(q * kMaxGatherSlots);
    const uint32_t my_empty = g_empty + 8u * (uint32_t)(q * kMaxGatherSlots);

    if (warp < 4) {
      // =============================== gather ==============================================
      const int m = lane >> 3, c = lane & 7;
      const uint32_t row_bytes = (uint32_t)p.c_in * 4u;
      const char *features = reinterpret_cast<const char *>(p.features);
      const int32_t *nb_oct = nbr_s + q * 32 + 8 * m;      // the 8 rows of this lane's octet: two int4
      const int cin_shift = p.cin_shift, cin_mask = p.c_in - 1;
      uint32_t dst_off[8];                                  // row (8m + t), swizzled chunk c ^ t
#pragma unroll
      for (int t = 0; t < 8; ++t) dst_off[t] = (uint32_t)((8 * m + t) * 128 + ((c ^ t) << 4));
      int sg = 0;
      uint32_t pg = 0;
      for (int it = 0; it < n_iters; ++it) {
        const int kk = it * kKBlock + 4 * c;               // first K index of this lane's chunk
        const int k = kk >> cin_shift;                     // <= kvol: row kvol of the table is all -1
        // features + channel offset as ONE opaque 64-bit value, so that each gather address below is a
        // single IMAD.WIDE (row * row_bytes + base) instead of a multiply plus a 64-bit add
        unsigned long long base = reinterpret_cast<unsigned long long>(features) + (unsigned)((kk & cin_mask) << 2);
        asm volatile("" : "+l"(base));
        const int4 *nb = reinterpret_cast<const int4 *>(nb_oct + k * kTileM);
        const int4 i0 = nb[0], i1 = nb[1];
        const int src[8] = {i0.x, i0.y, i0.z, i0.w, i1.x, i1.y, i1.z, i1.w};
        mbar_wait(my_empty + 8 * sg, pg ^ 1u);             // slot released by the convert warp
        const uint32_t slot = my_slots + (uint32_t)sg * (uint32_t)kStageSlotBytes;
#pragma unroll
        for (int t = 0; t < 8; ++t)
          cp_async16_row(slot + dst_off[t], base + (unsigned long long)(uint32_t)max(src[t], 0) * row_bytes, src[t]);
        cp_async_mbar_arrive_noinc(my_full + 8 * sg);
        if (++sg == nsg) { sg = 0; pg ^= 1u; }
      }
    } else {
      // =============================== convert =============================================
      uint32_t src_off[8];                                  // row = lane, chunk j at j ^ (lane & 7)
#pragma unroll
      for (int j = 0; j < 8; ++j) src_off[j] = (uint32_t)(lane * 128 + ((j ^ (lane & 7)) << 4));
      int sg = 0, sa = 0;
      uint32_t pg = 0, pa = 0;
      for (int it = 0; it < n_iters; ++it) {
        mbar_wait(my_full + 8 * sg, pg);
        const uint32_t slot = my_slots + (uint32_t)sg * (uint32_t)kStageSlotBytes;
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = lds128(slot + src_off[j]);
        __syncwarp();
        if (lane == 0) mbar_arrive(my_empty + 8 * sg);     // release: the reads above are ordered before it
        if (++sg == nsg) { sg = 0; pg ^= 1u; }
        mbar_wait(a_empty + 8 * sa, pa ^ 1u);
        tc_fence_after();
        const uint32_t col = lane_base + a_ring + (uint32_t)sa * kAStageCols;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {   // two 16-float halves keep the live registers down
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 fv = v[4 * hh + j];
            const float f[4] = {fv.x, fv.y, fv.z, fv.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              hi[4 * j + e] = __float_as_uint(f[e]) & 0xffffe000u;
              lo[4 * j + e] = __float_as_uint(f[e] - __uint_as_float(hi[4 * j + e]));
            }
          }
          tc_st16(col + (uint32_t)(16 * hh), hi);
          if (NSPLIT == 2) tc_st16(col + 32u + (uint32_t)(16 * hh), lo);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(a_full + 8 * sa);       // 4 arrivals per K block
        if (++sa == nsa) { sa = 0; pa ^= 1u; }
      }
    }
    // =============================== epilogue ============================================
    const int half = warp >> 2;
    mbar_wait(accbar, 0);
    tc_fence_after();
    const int orow = row0 + q * 32 + lane;
    const int ncol_half = c_out / 2;
    const int col_begin = half * ncol_half;
    const bool row_ok = orow < p.n_out;
    const float *scale = p.scale, *shift = p.shift;
    const int relu = p.relu;
    for (int c0 = col_begin; c0 < col_begin + ncol_half; c0 += 16) {
      float acc[16];
      tc_ld16(tmem_base + lane_base + (uint32_t)c0, acc);
      if (p.nmerge) {   // columns [c_out, 2 c_out) hold the hi x lo partial sums
        float more[16];
        tc_ld16(tmem_base + lane_base + (uint32_t)(c_out + c0), more);
#pragma unroll
        for (int e = 0; e < 16; ++e) acc[e] += more[e];
      }
      if (row_ok) {
        float *dst = p.out + (long long)orow * c_out + c0;
        const float *res = p.residual ? p.residual + (long long)orow * c_out + c0 : nullptr;
        const int ncols = min(16, col_begin + ncol_half - c0);
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          if (j < ncols) {
            float y[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float t = acc[j + e];
              if (scale) t *= __ldg(scale + c0 + j + e);
              if (shift) t += __ldg(shift + c0 + j + e);
              y[e] = t;
            }
            if (res) {
              const float4 rv = __ldg(reinterpret_cast<const float4 *>(res + j));
              y[0] += rv.x; y[1] += rv.y; y[2] += rv.z; y[3] += rv.w;
            }
            if (relu) {
#pragma unroll
              for (int e = 0; e < 4; ++e) y[e] = fmaxf(y[e], 0.f);
            }
            *reinterpret_cast<float4 *>(dst + j) = make_float4(y[0], y[1], y[2], y[3]);
          }
        }
      }
    }
  } else if (warp == 8) {
    // =============================== MMA issuer ==========================================
    const uint32_t idesc = umma_idesc_tf32(kTileM, c_out);
    const uint32_t idesc2 = umma_idesc_tf32(kTileM, 2 * c_out);   // merged [W_hi | W_lo] operand
    const int nmerge = p.nmerge;
    int sa = 0, sb = 0;
    uint32_t pa = 0, pb = 0;
    for (int it = 0; it < n_iters; ++it) {
      mbar_wait(a_full + 8 * sa, pa);
      mbar_wait(b_full + 8 * sb, pb);
      tc_fence_after();
      if (elect_one_sync()) {
        const uint32_t a_hi = a_ring + (uint32_t)sa * kAStageCols;   // lane 0, column offset
        const uint32_t a_lo = a_hi + 32u;
        const uint32_t bstage = smem_base + (uint32_t)sb * (uint32_t)b_stage_bytes;
        const uint64_t b_hi = umma_desc_sw128(bstage);
        const uint64_t b_lo = umma_desc_sw128(bstage + b_part_bytes);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {   // 8 tf32 per MMA = 32 B of K
          const uint64_t badv = (uint64_t)(ks * 2);     // +32 B along K inside the 128-byte swizzled weight row
          const uint32_t aadv = (uint32_t)(ks * 8);     // 8 TMEM columns per K step
          const uint32_t d = tmem_base;
          const uint32_t first = (it == 0 && ks == 0) ? 0u : 1u;
          if (nmerge) {
            // The hi and lo weight images are adjacent in the stage (same swizzle atoms), so one
            // descriptor with N = 2*c_out multiplies A_hi by both: columns [0, c_out) collect
            // hi*hi (+ lo*hi below), columns [c_out, 2 c_out) collect hi*lo.  2 MMAs, not 3; the
            // epilogue adds the two column groups.
            tc_mma_tf32_ts(d, a_hi + aadv, b_hi + badv, idesc2, first);
            tc_mma_tf32_ts(d, a_lo + aadv, b_hi + badv, idesc, 1u);
          } else if (NSPLIT == 2) {
            tc_mma_tf32_ts(d, a_lo + aadv, b_hi + badv, idesc, first);
            tc_mma_tf32_ts(d, a_hi + aadv, b_lo + badv, idesc, 1u);
            tc_mma_tf32_ts(d, a_hi + aadv, b_hi + badv, idesc, 1u);
          } else {
            tc_mma_tf32_ts(d, a_hi + aadv, b_hi + badv, idesc, first);
          }
        }
        tc_commit(a_empty + 8 * sa);
        tc_commit(b_empty + 8 * sb);
        if (it == n_iters - 1) tc_commit(accbar);
      }
      __syncwarp();
      if (++sa == nsa) { sa = 0; pa ^= 1u; }
      if (++sb == nsb) { sb = 0; pb ^= 1u; }
    }
  } else {
    // =============================== weight loader =======================================
    // Every CTA streams the whole weight tensor once per tile (515 tiles x 1.77 MB at C = 128): with the
    // gather, the staging reads and the MMAs all disabled the kernel still took 72 % of its time (`dbg 7` of
    // the since-removed timing-diagnostic build, profiles/r1_conv_v5_ablation.txt), i.e. the floor is the per-K-block synchronisation skeleton plus
    // what every SM must ingest (weights: 16 KB per K block per CTA at C = 128, as much as the features).
    // Multicasting the stages across a thread-block cluster halved the L2 reads but not the per-SM ingest
    // and measured slower (DESIGN.md 4.6).
    if (lane == 0) {
      const char *src = reinterpret_cast<const char *>(p.wpacked);
      int sb = 0;
      uint32_t pb = 1;   // an untouched stage counts as released
      for (int it = 0; it < n_iters; ++it) {
        mbar_wait(b_empty + 8 * sb, pb);
        mbar_arrive_expect_tx(b_full + 8 * sb, (uint32_t)b_stage_bytes);
        bulk_copy_g2s(smem_base + (uint32_t)sb * (uint32_t)b_stage_bytes, src, (uint32_t)b_stage_bytes,
                      b_full + 8 * sb);
        src += b_stage_bytes;
        if (++sb == nsb) { sb = 0; pb ^= 1u; }
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

// weight [K][Cin][Cout] fp32 -> packed [nkb][nsplit][Cout][32] in the swizzled smem image.  The K
// axis is the concatenation over kernel offsets of the Cin channels (kk = k*Cin + ci), cut into
// blocks of 32; element (n, c) of block kb sits at float index n*32 + (((c/4) ^ (n&7)) * 4) + (c%4).
// c_in_eff >= c_in is the (zero-padded) channel count the kernel runs with.
__global__ void spconv_pack_weights_kernel(const float *__restrict__ w, int kvol, int c_in, int c_in_eff,
                                           int c_out, int nkb, int nsplit, float *__restrict__ packed) {
  const long long total = (long long)nkb * c_out * 32;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
       t += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(t % 32);
    const int n = (int)((t / 32) % c_out);
    const int kb = (int)(t / (32ll * c_out));
    const int kk = kb * 32 + c;
    const int k = kk / c_in_eff, ci = kk % c_in_eff;
    const float v = (k < kvol && ci < c_in) ? w[((long long)k * c_in + ci) * c_out + n] : 0.f;
    const float hi = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
    const long long blk = (long long)kb * nsplit;
    const int pos = n * 32 + ((((c >> 2) ^ (n & 7)) << 2) | (c & 3));
    packed[(blk + 0) * c_out * 32 + pos] = hi;
    if (nsplit == 2) packed[(blk + 1) * c_out * 32 + pos] = v - hi;
  }
}

int spconv_forward_simt(const float *features, const float *weight, const int32_t *nbr, int n_in,
                        int n_out, int c_in, int c_out, int kvol, const float *scale,
                        const float *shift, const float *residual, int relu, float *out,
                        cudaStream_t st);

// Generation 6 (spconv_v6.cu: pre-split operands gathered straight into UMMA tiles, R row tiles per weight
// stage, persistent CTAs) runs BF16X3; generation 5 (above) runs the TF32 modes.
int spconv_v6_cin_eff(int c_in);
bool spconv_v6_shape_ok(int c_in, int c_out, int kvol);
size_t spconv_v6_packed_bytes(int c_in, int c_out, int kvol);
int spconv_v6_pack_weights(const float *weight, int c_in, int c_out, int kvol, void *packed, cudaStream_t st);
int spconv_v6_split_rows(const float *features, int n_cap, const int32_t *n_dev, int c_in, void *split,
                         cudaStream_t st);
int spconv_v6_forward(const void *features_split, const void *packed, const int32_t *nbr, long long nbr_stride,
                      int n_in, int n_out, const int32_t *n_out_dev, int c_in, int c_out, int kvol,
                      const float *scale, const float *shift, const float *residual, int relu, float *out,
                      void *out_split, cudaStream_t st);

static bool use_v6(int c_in, int c_out, int kvol, int precision) {
  return precision == BEVB200_PREC_BF16X3 && spconv_v6_shape_ok(c_in, c_out, kvol);
}
// for spconv_bwd.cu: does this (shape, precision) run on generation 6, i.e. on split row images?
bool spconv_tc_runs_on_split_images(int c_in, int c_out, int kvol, int precision) {
  return use_v6(c_in, c_out, kvol, precision);
}

// Input channels the TF32 kernel runs with: narrow inputs (conv_input: Cin = 5) are zero-padded to 8,
// other counts to the next power of two up to 128.  0 = no tensor-core form.
static int tc_cin_eff(int c_in) {
  for (int e = 8; e <= 128; e <<= 1)
    if (c_in <= e) return e;
  return 0;
}

static bool tc_shape_ok(int c_in, int c_out, int kvol) {
  return (c_out == 16 || c_out == 32 || c_out == 64 || c_out == 128) && c_in >= 1 && tc_cin_eff(c_in) != 0 &&
         kvol >= 1 && kvol <= 27;
}

int spconv_padded_channels(int c_in, int precision) {
  if (precision == BEVB200_PREC_FP32 || c_in < 1) return c_in;
  if (precision == BEVB200_PREC_BF16X3) return c_in;   // the split pass pads
  const int e = tc_cin_eff(c_in);
  return e ? e : c_in;
}

static int tc_nkb(int c_in_eff, int kvol) { return (kvol * c_in_eff + kKBlock - 1) / kKBlock; }

size_t spconv_packed_bytes(int c_in, int c_out, int kvol, int precision) {
  if (precision == BEVB200_PREC_BF16X3) return spconv_v6_packed_bytes(c_in, c_out, kvol);
  if (!tc_shape_ok(c_in, c_out, kvol)) return 0;
  const int nsplit = precision == BEVB200_PREC_TF32X3 ? 2 : 1;
  return (size_t)tc_nkb(tc_cin_eff(c_in), kvol) * nsplit * c_out * 32 * sizeof(float);
}

int spconv_pack_weights(const float *weight, int c_in, int c_out, int kvol, int precision,
                        float *packed, cudaStream_t st) {
  if (precision == BEVB200_PREC_BF16X3) return spconv_v6_pack_weights(weight, c_in, c_out, kvol, packed, st);
  const int ce = tc_cin_eff(c_in);
  const int nsplit = precision == BEVB200_PREC_TF32X3 ? 2 : 1;
  const int nkb = tc_nkb(ce, kvol);
  BEVB200_LAUNCH(spconv_pack_weights_kernel, grid_for((long long)nkb * c_out * 32, 256), 256, 0, st,
                 weight, kvol, c_in, ce, c_out, nkb, nsplit, packed);
  return BEVB200_OK;
}

// [n, c_in] -> [n, c_eff] rows, zero padded (c_eff a multiple of 4: 16-byte aligned rows)
__global__ void spconv_pad_rows_kernel(const float *__restrict__ in, int n, int c_in, int c_eff,
                                       float *__restrict__ out) {
  const long long total = (long long)n * (c_eff / 4);
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
       t += (long long)gridDim.x * blockDim.x) {
    const int g4 = (int)(t % (c_eff / 4));
    const long long r = t / (c_eff / 4);
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = 4 * g4 + e < c_in ? in[r * c_in + 4 * g4 + e] : 0.f;
    *reinterpret_cast<float4 *>(out + r * c_eff + 4 * g4) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// `packed` may be null: the weights are then packed into a stream-ordered temporary.
int spconv_forward_tc(const float *features, const float *weight, const float *packed_in,
                      const int32_t *nbr, int n_in, int n_out, int c_in, int c_out, int kvol,
                      const float *scale, const float *shift, const float *residual, int relu,
                      int precision, float *out, cudaStream_t st) {
  if (use_v6(c_in, c_out, kvol, precision) && (uintptr_t)out % 16 == 0 &&
      (residual == nullptr || (uintptr_t)residual % 16 == 0)) {
    // generation 6 consumes the bf16 hi|lo image of the rows: build it (and, without pre-packed weights,
    // the weight image) in stream-ordered temporaries.  SparseEncoder's fused path never comes here: its
    // convs hand the image to each other (bevb200_encoder_forward).
    const int ce = spconv_v6_cin_eff(c_in);
    void *split = nullptr, *wtmp = nullptr;
    int rc = BEVB200_OK;
    if (cudaMallocAsync(&split, (size_t)(n_in > 0 ? n_in : 1) * ce * 4, st) != cudaSuccess) rc = BEVB200_ECUDA;
    if (!rc && packed_in == nullptr) {
      if (weight == nullptr) {
        snprintf(g_last_error, sizeof(g_last_error), "spconv_forward: null weights");
        rc = BEVB200_EINVAL;
      } else if (cudaMallocAsync(&wtmp, spconv_v6_packed_bytes(c_in, c_out, kvol), st) != cudaSuccess) {
        rc = BEVB200_ECUDA;
      } else {
        rc = spconv_v6_pack_weights(weight, c_in, c_out, kvol, wtmp, st);
      }
    }
    if (!rc) rc = spconv_v6_split_rows(features, n_in, nullptr, c_in, split, st);
    if (!rc)
      rc = spconv_v6_forward(split, packed_in ? (const void *)packed_in : wtmp, nbr, n_out, n_in, n_out, nullptr, ce,
                             c_out, kvol, scale, shift, residual, relu, out, nullptr, st);
    if (rc == BEVB200_ECUDA && g_last_error[0] == 0)
      snprintf(g_last_error, sizeof(g_last_error), "spconv_forward: stream-ordered allocation failed");
    if (split) cudaFreeAsync(split, st);
    if (wtmp) cudaFreeAsync(wtmp, st);
    return rc;
  }
  // BF16X3 shapes generation 6 cannot take (unaligned out / residual) and shapes / alignments the UMMA path
  // cannot take: exact-fp32 SIMT kernel
  const int c_in_real = c_in;
  const int c_eff = precision != BEVB200_PREC_BF16X3 && tc_shape_ok(c_in, c_out, kvol) ? tc_cin_eff(c_in) : 0;
  const bool ok = c_eff != 0 && (c_eff != c_in || (uintptr_t)features % 16 == 0) &&
                  ((uintptr_t)out % 16 == 0) && (residual == nullptr || (uintptr_t)residual % 16 == 0);
  if (!ok) {
    if (weight == nullptr) {
      snprintf(g_last_error, sizeof(g_last_error), "spconv_forward: shape needs the unpacked weights");
      return BEVB200_EINVAL;
    }
    return spconv_forward_simt(features, weight, nbr, n_in, n_out, c_in, c_out, kvol, scale, shift,
                               residual, relu, out, st);
  }
  // stream-ordered temporaries, released on every exit path
  struct Temps {
    cudaStream_t st;
    float *padded = nullptr, *packed = nullptr;
    ~Temps() {
      if (packed) cudaFreeAsync(packed, st);
      if (padded) cudaFreeAsync(padded, st);
    }
  } tmp;
  tmp.st = st;
  float *&padded = tmp.padded;
  if (c_eff != c_in) {   // e.g. conv_input (Cin = 5 -> 8): zero-padded copy of the rows, padded weights
    BEVB200_CUDA(cudaMallocAsync((void **)&padded, (size_t)(n_in > 0 ? n_in : 1) * c_eff * sizeof(float), st));
    if (n_in > 0)
      BEVB200_LAUNCH(spconv_pad_rows_kernel, grid_for((long long)n_in * (c_eff / 4), 256), 256, 0, st, features,
                     n_in, c_in, c_eff, padded);
    features = padded;
    c_in = c_eff;
  }
  const int nsplit = precision == BEVB200_PREC_TF32X3 ? 2 : 1;   // tf32 parts
  int cin_shift = 0;
  while ((1 << cin_shift) < c_in) ++cin_shift;

  float *&packed = tmp.packed;
  const float *wpacked = packed_in;
  if (packed_in == nullptr) {
    BEVB200_CUDA(cudaMallocAsync((void **)&packed, spconv_packed_bytes(c_in_real, c_out, kvol, precision), st));
    int rc = spconv_pack_weights(weight, c_in_real, c_out, kvol, precision, packed, st);
    if (rc) return rc;
    wpacked = packed;
  }

  TcParams p;
  p.features = features; p.nbr = nbr; p.scale = scale; p.shift = shift; p.residual = residual;
  p.out = out; p.n_in = n_in; p.n_out = n_out; p.c_in = c_in; p.c_out = c_out; p.kvol = kvol;
  p.relu = relu; p.nkb = tc_nkb(c_in, kvol); p.cin_shift = cin_shift; p.wpacked = wpacked;
  p.nmerge = (nsplit == 2 && c_out <= 64) ? 1 : 0;
  p.acc_cols = p.nmerge ? (2 * c_out < 32 ? 32 : 2 * c_out) : (c_out < 32 ? 32 : c_out);
  // 256 TMEM columns per CTA (two CTAs per SM): accumulator + A ring (>= 2 stages)
  p.nsa = (256 - p.acc_cols) / (nsplit * 32);
  if (p.nsa > 4) p.nsa = 4;
  p.tmem_cols = 256;
  // per CTA (two per SM): 1 KB alignment slack + weight ring + neighbour table + 4 quarters x nsg
  // staging slots of 4 KB.  As many slots as fit beside a 2-stage weight ring, then the ring
  // takes what is left.
  const int b_stage = nsplit * c_out * 128;
  const int budget = 111 * 1024;
  p.nbr_bytes = ((kvol + 1) * kTileM * 4 + 127) / 128 * 128;   // + one all -1 row (K tail padding)
  const int avail = budget - 1024 - p.nbr_bytes;
  p.nsg = (avail - 2 * b_stage) / (4 * kStageSlotBytes);
  if (p.nsg > kMaxGatherSlots) p.nsg = kMaxGatherSlots;
  BEVB200_REQUIRE(p.nsg >= 2, "shared memory budget: no room for two gather slots");
  p.nsb = (avail - p.nsg * 4 * kStageSlotBytes) / b_stage;
  if (p.nsb > kMaxStages) p.nsb = kMaxStages;
  const size_t smem = (size_t)p.nsb * b_stage + p.nbr_bytes + (size_t)p.nsg * 4 * kStageSlotBytes + 1024;
  const int grid = (n_out + kTileM - 1) / kTileM;
  if (nsplit == 2) {
    BEVB200_CUDA(cudaFuncSetAttribute(spconv_tc_kernel_v5<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    BEVB200_LAUNCH(spconv_tc_kernel_v5<2>, grid, kTcThreads, smem, st, p);
  } else {
    BEVB200_CUDA(cudaFuncSetAttribute(spconv_tc_kernel_v5<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    BEVB200_LAUNCH(spconv_tc_kernel_v5<1>, grid, kTcThreads, smem, st, p);
  }
  return BEVB200_OK;
}

}  // namespace bevb200
