// SparseEncoder as ONE native, sync-free call (replaces the per-conv python loop of
// mmdet3d/models/backbones/sparse_encoder.py:99-132 + spconv/conv.py:114-223 + spconv_ops.h:27-141,260-361).
//
// The reference (and generation 5 of this library) is host paced: every strided conv returns its output
// count to the host (`.item()` / indiceNum.to(kCPU), spconv_ops.h:271) before the next buffer can be
// sized and the next kernel launched.  Here every row count stays on the device:
//   * buffers are sized by CAPS known on the host (level 0: max_voxels; a strided conv can create at most
//     prod(ceil(k/s)) outputs per input and at most one per output site; the caller may pass tighter caps,
//     an overflow flag reports truncation),
//   * kernels take their row count from device memory (grid-stride loops / persistent CTAs),
//   * so the whole encoder -- operand split, 8 rulebooks, 21 convs with folded BN / residual / ReLU
//     epilogues, dense() -- is ~45 launches with no host round trip and can be captured in a CUDA graph.
// Rulebooks depend on the voxel coordinates only; they are built on `rulebook_stream` (when given) and the
// convs wait on one event per rulebook, so they hide behind the convolutions already queued.
//
// Rulebook = offset-major neighbour table nbr[k][row] over a site BITMAP of each level's dense grid with
// a popcount prefix per word ({bits, prefix} interleaved: one 8-byte load per lookup), built by a
// single-pass decoupled-look-back scan.  Strided convs are built output-side: the outputs of level l+1
// look their <= K inputs up in level l's bitmap (no scatter, no -1 fill pass, coalesced writes); one
// thread walks the kz column of one (kx, ky) so consecutive lookups hit the same word.
#include <stdlib.h>

#include <algorithm>
#include <new>
#include <vector>

#include "common.cuh"

namespace bevb200 {

int spconv_v6_cin_eff(int c_in);
bool spconv_v6_shape_ok(int c_in, int c_out, int kvol);
size_t spconv_v6_packed_bytes(int c_in, int c_out, int kvol);
int spconv_v6_pack_weights(const float *weight, int c_in, int c_out, int kvol, void *packed, cudaStream_t st);
int spconv_v6_split_rows(const float *features, int n_cap, const int32_t *n_dev, int c_in, void *split,
                         cudaStream_t st);
int spconv_v6_forward_ex(const void *features_split, const void *packed, const int32_t *nbr, long long nbr_stride,
                         int n_in, int n_out, const int32_t *n_out_dev, int c_in, int c_out, int kvol,
                         const float *scale, const float *shift, const float *residual, const void *residual_split,
                         int relu, float *out, void *out_split, cudaStream_t st);
int spconv_v6_forward(const void *features_split, const void *packed, const int32_t *nbr, long long nbr_stride,
                      int n_in, int n_out, const int32_t *n_out_dev, int c_in, int c_out, int kvol,
                      const float *scale, const float *shift, const float *residual, int relu, float *out,
                      void *out_split, cudaStream_t st);

struct EGeom {
  int in_shape[3], q_shape[3], ksize[3], stride[3], pad[3], dil[3];
  int batch;
};

__device__ __forceinline__ int enc_count(const int32_t *n_dev, int cap) {
  const int n = n_dev ? __ldg(n_dev) : cap;
  return min(max(n, 0), cap);
}
__device__ __forceinline__ long long enc_site(int b, int x, int y, int z, const int shape[3]) {
  return (((long long)b * shape[0] + x) * shape[1] + y) * shape[2] + z;   // tensorview.h:453-464
}

__global__ void enc_set_count_kernel(int32_t *dst, int value) { *dst = value; }

// active sites of a level <- its rows
__global__ void enc_mark_rows_kernel(const int32_t *__restrict__ idx, int cap, const int32_t *__restrict__ n_dev,
                                     EGeom g, uint2 *__restrict__ cells) {
  const int n = enc_count(n_dev, cap);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int4 c = *reinterpret_cast<const int4 *>(idx + 4ll * i);   // (b, x, y, z)
    if ((unsigned)c.x >= (unsigned)g.batch || (unsigned)c.y >= (unsigned)g.in_shape[0] ||
        (unsigned)c.z >= (unsigned)g.in_shape[1] || (unsigned)c.w >= (unsigned)g.in_shape[2])
      continue;
    const long long s = enc_site(c.x, c.y, c.z, c.w, g.in_shape);
    atomicOr(&cells[s >> 5].x, 1u << (s & 31));
  }
}

// output sites of a strided conv <- input rows: p = (q + pad - k*dil) / stride where divisible
// (the set getValidOutPos enumerates, geometry.h:24-85)
__global__ void enc_mark_outputs_kernel(const int32_t *__restrict__ idx, int cap, const int32_t *__restrict__ n_dev,
                                        EGeom g, uint2 *__restrict__ cells_out) {
  const int n = enc_count(n_dev, cap);
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const int4 c = *reinterpret_cast<const int4 *>(idx + 4ll * j);
    if ((unsigned)c.x >= (unsigned)g.batch) continue;
    const int q[3] = {c.y, c.z, c.w};
    for (int kx = 0; kx < g.ksize[0]; ++kx) {
      int vx = q[0] + g.pad[0] - kx * g.dil[0];
      if (vx < 0 || vx % g.stride[0]) continue;
      vx /= g.stride[0];
      if (vx >= g.q_shape[0]) continue;
      for (int ky = 0; ky < g.ksize[1]; ++ky) {
        int vy = q[1] + g.pad[1] - ky * g.dil[1];
        if (vy < 0 || vy % g.stride[1]) continue;
        vy /= g.stride[1];
        if (vy >= g.q_shape[1]) continue;
        for (int kz = 0; kz < g.ksize[2]; ++kz) {
          int vz = q[2] + g.pad[2] - kz * g.dil[2];
          if (vz < 0 || vz % g.stride[2]) continue;
          vz /= g.stride[2];
          if (vz >= g.q_shape[2]) continue;
          const long long s = enc_site(c.x, vx, vy, vz, g.q_shape);
          const uint32_t bit = 1u << (s & 31);
          if (!(cells_out[s >> 5].x & bit)) atomicOr(&cells_out[s >> 5].x, bit);
        }
      }
    }
  }
}

// ---- single-pass scan (decoupled look-back): cells[w].y = sum_{v < w} popc(cells[v].x) ----------
constexpr int kEncScanThreads = 256, kEncScanPer = 16, kEncScanTile = kEncScanThreads * kEncScanPer;
constexpr unsigned long long kFlagAgg = 1ull << 32, kFlagIncl = 2ull << 32;

__global__ void __launch_bounds__(kEncScanThreads)
    enc_scan_kernel(uint2 *__restrict__ cells, size_t nwords, unsigned long long *status, uint32_t *ticket,
                    uint32_t *total) {
  __shared__ uint32_t s_warp[kEncScanThreads / 32];
  __shared__ uint32_t s_tile, s_excl;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);     // tiles are taken in launch order: forward progress
  __syncthreads();
  const uint32_t tile = s_tile;
  const size_t base = (size_t)tile * kEncScanTile + (size_t)tid * kEncScanPer;
  uint32_t v[kEncScanPer], sum = 0;
#pragma unroll
  for (int j = 0; j < kEncScanPer; ++j) {
    v[j] = base + j < nwords ? (uint32_t)__popc(cells[base + j].x) : 0u;
    sum += v[j];
  }
  uint32_t incl = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += t;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  uint32_t woff = 0, tile_total = 0;
#pragma unroll
  for (int w = 0; w < kEncScanThreads / 32; ++w) {
    const uint32_t x = s_warp[w];
    if (w < warp) woff += x;
    tile_total += x;
  }
  if (tid == 0) {
    uint32_t excl = 0;
    if (tile == 0) {
      atomicExch(status + 0, kFlagIncl | tile_total);
    } else {
      atomicExch(status + tile, kFlagAgg | tile_total);
      for (int j = (int)tile - 1; j >= 0; --j) {
        unsigned long long st;
        do {
          st = *reinterpret_cast<volatile unsigned long long *>(status + j);
        } while ((st >> 32) == 0);
        excl += (uint32_t)st;
        if ((st >> 32) == 2) break;
      }
      atomicExch(status + tile, kFlagIncl | (unsigned long long)(excl + tile_total));
    }
    s_excl = excl;
    if ((size_t)(tile + 1) * kEncScanTile >= nwords) *total = excl + tile_total;
  }
  __syncthreads();
  uint32_t run = s_excl + woff + (incl - sum);
#pragma unroll
  for (int j = 0; j < kEncScanPer; ++j) {
    if (base + j < nwords) cells[base + j].y = run;
    run += v[j];
  }
}

__device__ __forceinline__ int enc_rank(const uint2 cell, uint32_t bit) {
  if (!(cell.x & bit)) return -1;
  return (int)(cell.y + __popc(cell.x & (bit - 1)));
}

// level 0 keeps the caller's row order: rank (ascending site) -> row
__global__ void enc_rank2row_kernel(const int32_t *__restrict__ idx, int cap, const int32_t *__restrict__ n_dev,
                                    EGeom g, const uint2 *__restrict__ cells, int32_t *__restrict__ rank2row) {
  const int n = enc_count(n_dev, cap);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int4 c = *reinterpret_cast<const int4 *>(idx + 4ll * i);
    if ((unsigned)c.x >= (unsigned)g.batch || (unsigned)c.y >= (unsigned)g.in_shape[0] ||
        (unsigned)c.z >= (unsigned)g.in_shape[1] || (unsigned)c.w >= (unsigned)g.in_shape[2])
      continue;
    const long long s = enc_site(c.x, c.y, c.z, c.w, g.in_shape);
    const int r = enc_rank(__ldg(cells + (s >> 5)), 1u << (s & 31));
    if (r >= 0 && r < cap) rank2row[r] = i;   // duplicate coordinates: any one row wins (reference: last)
  }
}

// n_out = min(total, cap); overflow flag when the cap truncates
__global__ void enc_count_kernel(const uint32_t *total, int cap, int32_t *n_out, int32_t *overflow) {
  const uint32_t t = *total;
  *n_out = t > (uint32_t)cap ? cap : (int)t;
  if (t > (uint32_t)cap) atomicOr(overflow, 1);
}

// rows of a level built from its bitmap: ascending flat index = the reference's GPU order after
// torch::_unique (spconv_ops.h:130-136, indice.cu.h:112-127)
__global__ void enc_out_indices_kernel(const uint2 *__restrict__ cells, size_t nwords, int X, int Y, int Z,
                                       int cap, int32_t *__restrict__ out_idx) {
  for (size_t w = blockIdx.x * (size_t)blockDim.x + threadIdx.x; w < nwords; w += (size_t)gridDim.x * blockDim.x) {
    const uint2 cell = cells[w];
    uint32_t m = cell.x;
    if (!m) continue;
    int r = (int)cell.y;
    while (m) {
      const int bit = __ffs(m) - 1;
      m &= m - 1;
      long long s = ((long long)w << 5) + bit;
      const int z = (int)(s % Z); s /= Z;
      const int y = (int)(s % Y); s /= Y;
      const int x = (int)(s % X); s /= X;
      if (r < cap) *reinterpret_cast<int4 *>(out_idx + 4ll * r) = make_int4((int)s, x, y, z);
      ++r;
    }
  }
}

// nbr[k][o] = row of the input site (o * stride - pad + k * dil), or -1.  grid (row tiles, kx * ky): a
// thread walks the kz column of one (kx, ky); consecutive z are consecutive bits, so the column usually
// costs ONE 8-byte cell load.
__global__ void __launch_bounds__(256)
    enc_nbr_kernel(const int32_t *__restrict__ qidx, int qcap, const int32_t *__restrict__ nq_dev, EGeom g,
                   const uint2 *__restrict__ cells_in, const int32_t *__restrict__ rank2row, int in_cap,
                   int32_t *__restrict__ nbr, long long nbr_stride) {
  const int n = enc_count(nq_dev, qcap);
  const int kxy = blockIdx.y, ky = kxy % g.ksize[1], kx = kxy / g.ksize[1];
  for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < n; o += gridDim.x * blockDim.x) {
    const int4 c = *reinterpret_cast<const int4 *>(qidx + 4ll * o);
    const int x = c.y * g.stride[0] - g.pad[0] + kx * g.dil[0];
    const int y = c.z * g.stride[1] - g.pad[1] + ky * g.dil[1];
    const bool ok_xy = (unsigned)c.x < (unsigned)g.batch && (unsigned)x < (unsigned)g.in_shape[0] &&
                       (unsigned)y < (unsigned)g.in_shape[1];
    const long long col = ok_xy ? enc_site(c.x, x, y, 0, g.in_shape) : 0;
    long long cur_w = -1;
    uint2 cell = make_uint2(0u, 0u);
    for (int kz = 0; kz < g.ksize[2]; ++kz) {
      const int z = c.w * g.stride[2] - g.pad[2] + kz * g.dil[2];
      int row = -1;
      if (ok_xy && (unsigned)z < (unsigned)g.in_shape[2]) {
        const long long s = col + z;
        if ((s >> 5) != cur_w) {
          cur_w = s >> 5;
          cell = __ldg(cells_in + cur_w);
        }
        const int r = enc_rank(cell, 1u << (s & 31));
        if (r >= 0 && r < in_cap) row = rank2row ? __ldg(rank2row + r) : r;
      }
      nbr[(long long)(kxy * g.ksize[2] + kz) * nbr_stride + o] = row;
    }
  }
}

// dense() + permute(0,1,4,2,3) + view(N, C*D, H, W) (structure.py:49-59, sparse_encoder.py:126-130)
__global__ void __launch_bounds__(256)
    enc_dense_kernel(const float *__restrict__ features, const int32_t *__restrict__ idx, int cap,
                     const int32_t *__restrict__ n_dev, int c, int batch, int X, int Y, int Z, int z_major,
                     long long out_batch_stride, float *__restrict__ out) {
  const int n = enc_count(n_dev, cap);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int4 p = *reinterpret_cast<const int4 *>(idx + 4ll * i);
    if ((unsigned)p.x >= (unsigned)batch || (unsigned)p.y >= (unsigned)X || (unsigned)p.z >= (unsigned)Y ||
        (unsigned)p.w >= (unsigned)Z)
      continue;
    const long long site = z_major ? ((long long)p.w * X + p.y) * Y + p.z : ((long long)p.y * Y + p.z) * Z + p.w;
    const long long plane = (long long)X * Y * Z;
    float *o = out + p.x * out_batch_stride + site;
    for (int ch = blockIdx.y; ch < c; ch += gridDim.y) o[ch * plane] = features[(long long)i * c + ch];
  }
}

// ---- the plan -----------------------------------------------------------------------------------
struct EConv {
  bevb200_encoder_conv_t d;
  int kvol, c_in_eff;
  int level_in, level_out, rulebook;
  bool want_fp32;
  size_t packed_off, scale_off, shift_off;   // offsets into the parameter buffer
  bool has_scale, has_shift;
};
struct ELevel {
  int shape[3];
  int c_max;           // widest tensor living on this level
};
struct ERulebook {
  int level_q, level_in;   // query (output) level, input level
  int ksize[3], stride[3], pad[3], dil[3];
  int kvol;
};

}  // namespace bevb200

using namespace bevb200;

struct bevb200_encoder {
  int in_channels, c0_eff;
  std::vector<EConv> convs;
  std::vector<ELevel> levels;
  std::vector<ERulebook> rulebooks;
  size_t param_bytes;
  std::vector<cudaEvent_t> events;   // [0] fork, [1..] one per rulebook, last: join
  int event_device;
};

namespace bevb200 {

static long long level_sites(const ELevel &l, int batch) {
  return (long long)batch * l.shape[0] * l.shape[1] * l.shape[2];
}

// row caps per level: [0] = max_voxels; a strided conv makes <= prod(ceil(k/s)) outputs per input and
// <= 1 per output site; user caps (> 0) may only tighten
static void level_caps(const bevb200_encoder *e, int max_voxels, int batch, const int32_t *user, std::vector<int> *caps) {
  caps->assign(e->levels.size(), 0);
  (*caps)[0] = max_voxels;
  for (const EConv &cv : e->convs) {
    if (cv.level_out == cv.level_in) continue;
    long long fan = 1;
    for (int d = 0; d < 3; ++d) fan *= (cv.d.ksize[d] + cv.d.stride[d] - 1) / cv.d.stride[d];
    long long cap = fan * (*caps)[cv.level_in];
    const long long sites = level_sites(e->levels[cv.level_out], batch);
    if (cap > sites) cap = sites;
    if (user && user[cv.level_out] > 0 && user[cv.level_out] < cap) cap = user[cv.level_out];
    if (cap > 0x7fffff00ll) cap = 0x7fffff00ll;
    (*caps)[cv.level_out] = (int)cap;
  }
}

struct EWs {
  std::vector<uint2 *> cells;
  std::vector<int32_t *> indices, counts;
  std::vector<unsigned long long *> status;
  std::vector<uint32_t *> ticket, total;
  int32_t *rank2row;
  std::vector<int32_t *> nbr;
  std::vector<uint8_t *> split[2];
  std::vector<float *> f32[2];
  char *zero_begin, *zero_end;
  size_t bytes;
};

static size_t enc_layout(const bevb200_encoder *e, const std::vector<int> &caps, int batch, void *ws, size_t ws_bytes,
                         EWs *w) {
  Arena a(ws, ws_bytes);
  const size_t nl = e->levels.size();
  w->cells.resize(nl); w->indices.resize(nl); w->counts.resize(nl); w->status.resize(nl);
  w->ticket.resize(nl); w->total.resize(nl);
  // --- region zeroed at the start of every forward: bitmaps, scan state ---
  w->zero_begin = a.base ? a.base + a.off : nullptr;
  for (size_t l = 0; l < nl; ++l) {
    const size_t nwords = (size_t)((level_sites(e->levels[l], batch) + 31) / 32);
    w->cells[l] = a.take<uint2>(nwords);
    w->status[l] = a.take<unsigned long long>((nwords + kEncScanTile - 1) / kEncScanTile + 1);
    w->ticket[l] = a.take<uint32_t>(4);
    w->total[l] = a.take<uint32_t>(4);
  }
  w->zero_end = a.base ? a.base + a.off : nullptr;
  for (size_t l = 0; l < nl; ++l) {
    w->indices[l] = l == 0 ? nullptr : a.take<int32_t>((size_t)caps[l] * 4);
    w->counts[l] = a.take<int32_t>(4);
  }
  w->rank2row = a.take<int32_t>((size_t)caps[0]);
  w->nbr.resize(e->rulebooks.size());
  for (size_t r = 0; r < e->rulebooks.size(); ++r)
    w->nbr[r] = a.take<int32_t>((size_t)e->rulebooks[r].kvol * caps[e->rulebooks[r].level_q]);
  for (int s = 0; s < 2; ++s) {
    w->split[s].resize(nl);
    w->f32[s].resize(nl);
    for (size_t l = 0; l < nl; ++l) {
      const size_t row = (size_t)e->levels[l].c_max * 4;
      w->split[s][l] = a.take<uint8_t>((size_t)caps[l] * row);
      w->f32[s][l] = a.take<float>((size_t)caps[l] * e->levels[l].c_max);
    }
  }
  w->bytes = a.off;
  return a.off;
}

}  // namespace bevb200

extern "C" {

int bevb200_encoder_create(int in_channels, const int32_t *sparse_shape_host, const bevb200_encoder_conv_t *convs,
                           int n_convs, bevb200_encoder_t **out) {
  BEVB200_REQUIRE(out && convs && sparse_shape_host && n_convs > 0 && in_channels > 0, "bad argument");
  bevb200_encoder *e = new (std::nothrow) bevb200_encoder();
  BEVB200_REQUIRE(e != nullptr, "out of host memory");
  e->in_channels = in_channels;
  e->c0_eff = spconv_v6_cin_eff(in_channels);
  e->event_device = -1;
  ELevel l0;
  for (int d = 0; d < 3; ++d) l0.shape[d] = sparse_shape_host[d];
  l0.c_max = e->c0_eff;
  e->levels.push_back(l0);
  int level = 0, c_prev = in_channels;
  size_t poff = 0;
  auto fail = [&](const char *msg) {
    snprintf(g_last_error, sizeof(g_last_error), "bevb200_encoder_create: %s", msg);
    delete e;
    return BEVB200_EINVAL;
  };
  if (e->c0_eff == 0) return fail("in_channels > 128");
  for (int i = 0; i < n_convs; ++i) {
    EConv cv;
    cv.d = convs[i];
    if (cv.d.c_in != c_prev) return fail("conv c_in does not match the previous conv's c_out");
    cv.kvol = cv.d.ksize[0] * cv.d.ksize[1] * cv.d.ksize[2];
    for (int d = 0; d < 3; ++d) {
      if (cv.d.ksize[d] <= 0 || cv.d.dilation[d] <= 0) return fail("bad kernel geometry");
      if (cv.d.subm) {   // spconv_ops.h:74-83: SubM forces stride 1 and padding k/2
        cv.d.stride[d] = 1;
        cv.d.padding[d] = cv.d.ksize[d] / 2;
      }
      if (cv.d.stride[d] <= 0 || cv.d.padding[d] < 0) return fail("bad stride / padding");
    }
    if (!spconv_v6_shape_ok(cv.d.c_in, cv.d.c_out, cv.kvol)) return fail("conv shape has no tensor-core form");
    cv.c_in_eff = spconv_v6_cin_eff(cv.d.c_in);
    if (i > 0 && cv.c_in_eff != cv.d.c_in) return fail("inner channel counts must be multiples of 16");
    if (cv.d.residual_from >= i) return fail("residual_from must name an earlier conv");
    cv.level_in = level;
    if (!cv.d.subm) {
      ELevel nl;
      for (int d = 0; d < 3; ++d) {   // ops.py:20-31
        const int num = e->levels[level].shape[d] + 2 * cv.d.padding[d] - cv.d.dilation[d] * (cv.d.ksize[d] - 1) - 1;
        if (num < 0) return fail("conv output shape is empty");
        nl.shape[d] = num / cv.d.stride[d] + 1;
      }
      nl.c_max = cv.d.c_out;
      e->levels.push_back(nl);
      ++level;
    }
    cv.level_out = level;
    if (cv.d.residual_from >= 0) {
      const EConv &src = e->convs[cv.d.residual_from];
      if (src.level_out != cv.level_out || src.d.c_out != cv.d.c_out) return fail("residual shape mismatch");
    }
    e->levels[cv.level_out].c_max = std::max(e->levels[cv.level_out].c_max, cv.d.c_out);
    // rulebook: shared by every conv with the same geometry on the same levels
    cv.rulebook = -1;
    for (size_t r = 0; r < e->rulebooks.size(); ++r) {
      const ERulebook &rb = e->rulebooks[r];
      bool same = rb.level_q == cv.level_out && rb.level_in == cv.level_in;
      for (int d = 0; d < 3 && same; ++d)
        same = rb.ksize[d] == cv.d.ksize[d] && rb.stride[d] == cv.d.stride[d] && rb.pad[d] == cv.d.padding[d] &&
               rb.dil[d] == cv.d.dilation[d];
      if (same) cv.rulebook = (int)r;
    }
    if (cv.rulebook < 0) {
      ERulebook rb;
      rb.level_q = cv.level_out;
      rb.level_in = cv.level_in;
      for (int d = 0; d < 3; ++d) {
        rb.ksize[d] = cv.d.ksize[d]; rb.stride[d] = cv.d.stride[d]; rb.pad[d] = cv.d.padding[d]; rb.dil[d] = cv.d.dilation[d];
      }
      rb.kvol = cv.kvol;
      cv.rulebook = (int)e->rulebooks.size();
      e->rulebooks.push_back(rb);
    }
    // A residual is read from the source conv's SPLIT image -- hi + lo is the value to 2^-17 -- so only the last
    // conv, whose rows dense() scatters, writes fp32 rows.
    cv.want_fp32 = i == n_convs - 1;
    cv.packed_off = poff; poff += align_up(spconv_v6_packed_bytes(cv.d.c_in, cv.d.c_out, cv.kvol));
    cv.scale_off = poff; poff += align_up((size_t)cv.d.c_out * 4);
    cv.shift_off = poff; poff += align_up((size_t)cv.d.c_out * 4);
    cv.has_scale = cv.has_shift = false;
    e->convs.push_back(cv);
    c_prev = cv.d.c_out;
  }
  e->param_bytes = poff;
  *out = e;
  return BEVB200_OK;
}

void bevb200_encoder_destroy(bevb200_encoder_t *e) {
  if (!e) return;
  for (cudaEvent_t ev : e->events) cudaEventDestroy(ev);
  delete e;
}

size_t bevb200_encoder_param_bytes(const bevb200_encoder_t *e) { return e ? e->param_bytes : 0; }

int bevb200_encoder_num_levels(const bevb200_encoder_t *e) { return e ? (int)e->levels.size() : 0; }

int bevb200_encoder_output_shape(const bevb200_encoder_t *e, int32_t *shape_out, int32_t *channels_out) {
  BEVB200_REQUIRE(e && shape_out && channels_out, "null argument");
  for (int d = 0; d < 3; ++d) shape_out[d] = e->levels.back().shape[d];
  *channels_out = e->convs.back().d.c_out;
  return BEVB200_OK;
}

int bevb200_encoder_set_conv(bevb200_encoder_t *e, int conv, const float *weight, const float *scale,
                             const float *shift, void *params, size_t params_bytes, void *stream) {
  BEVB200_REQUIRE(e && conv >= 0 && conv < (int)e->convs.size(), "bad conv index");
  BEVB200_REQUIRE(weight && params && params_bytes >= e->param_bytes, "null argument / parameter buffer too small");
  EConv &cv = e->convs[conv];
  cudaStream_t st = (cudaStream_t)stream;
  char *base = (char *)params;
  int rc = spconv_v6_pack_weights(weight, cv.d.c_in, cv.d.c_out, cv.kvol, base + cv.packed_off, st);
  if (rc) return rc;
  cv.has_scale = scale != nullptr;
  cv.has_shift = shift != nullptr;
  if (scale)
    BEVB200_CUDA(cudaMemcpyAsync(base + cv.scale_off, scale, (size_t)cv.d.c_out * 4, cudaMemcpyDeviceToDevice, st));
  if (shift)
    BEVB200_CUDA(cudaMemcpyAsync(base + cv.shift_off, shift, (size_t)cv.d.c_out * 4, cudaMemcpyDeviceToDevice, st));
  return BEVB200_OK;
}

int bevb200_encoder_level_caps(const bevb200_encoder_t *e, int max_voxels, int batch_size, const int32_t *user_caps,
                               int32_t *caps_out) {
  BEVB200_REQUIRE(e && caps_out && max_voxels > 0 && batch_size > 0, "bad argument");
  std::vector<int> caps;
  level_caps(e, max_voxels, batch_size, user_caps, &caps);
  for (size_t l = 0; l < caps.size(); ++l) caps_out[l] = caps[l];
  return BEVB200_OK;
}

size_t bevb200_encoder_workspace_bytes(const bevb200_encoder_t *e, int max_voxels, int batch_size,
                                       const int32_t *user_caps) {
  if (!e || max_voxels <= 0 || batch_size <= 0) return 0;
  std::vector<int> caps;
  level_caps(e, max_voxels, batch_size, user_caps, &caps);
  EWs w;
  return enc_layout(e, caps, batch_size, nullptr, 0, &w);
}

int bevb200_encoder_forward(bevb200_encoder_t *e, const void *params, const float *voxel_features,
                            const int32_t *coors, int max_voxels, const int32_t *n_voxels_dev, int batch_size,
                            const int32_t *user_caps, float *dense_out, long long out_batch_stride,
                            int32_t *status_dev, void *workspace, size_t workspace_bytes, void *stream,
                            void *rulebook_stream) {
  BEVB200_REQUIRE(e && params && dense_out && status_dev && max_voxels > 0 && batch_size > 0, "bad argument");
  BEVB200_REQUIRE(voxel_features && coors, "null input");
  cudaStream_t st = (cudaStream_t)stream, ss = rulebook_stream ? (cudaStream_t)rulebook_stream : st;
  const bool forked = ss != st;
  std::vector<int> caps;
  level_caps(e, max_voxels, batch_size, user_caps, &caps);
  EWs w;
  const size_t need = enc_layout(e, caps, batch_size, workspace, workspace_bytes, &w);
  if (workspace == nullptr || workspace_bytes < need) {
    snprintf(g_last_error, sizeof(g_last_error), "encoder_forward: workspace too small (%zu < %zu)", workspace_bytes, need);
    return BEVB200_EWORKSPACE;
  }
  const size_t nl = e->levels.size(), nr = e->rulebooks.size();
  if (forked) {
    int dev = 0;
    BEVB200_CUDA(cudaGetDevice(&dev));
    if (e->event_device != dev) {
      for (cudaEvent_t ev : e->events) cudaEventDestroy(ev);
      e->events.assign(nr + 2, nullptr);
      for (cudaEvent_t &ev : e->events) BEVB200_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      e->event_device = dev;
    }
    BEVB200_CUDA(cudaEventRecord(e->events[0], st));       // the coordinates are ready
    BEVB200_CUDA(cudaStreamWaitEvent(ss, e->events[0], 0));
  }
  const char *pbase = (const char *)params;
  auto geom_of = [&](const ERulebook &rb) {
    EGeom g;
    for (int d = 0; d < 3; ++d) {
      g.in_shape[d] = e->levels[rb.level_in].shape[d];
      g.q_shape[d] = e->levels[rb.level_q].shape[d];
      g.ksize[d] = rb.ksize[d]; g.stride[d] = rb.stride[d]; g.pad[d] = rb.pad[d]; g.dil[d] = rb.dil[d];
    }
    g.batch = batch_size;
    return g;
  };
  auto nwords_of = [&](size_t l) { return (size_t)((level_sites(e->levels[l], batch_size) + 31) / 32); };
  auto scan_level = [&](size_t l) -> int {
    const size_t nw = nwords_of(l);
    BEVB200_LAUNCH(enc_scan_kernel, (unsigned)((nw + kEncScanTile - 1) / kEncScanTile), kEncScanThreads, 0, ss,
                   w.cells[l], nw, w.status[l], w.ticket[l], w.total[l]);
    return BEVB200_OK;
  };

  // ------------------------------ rulebooks (stream ss) ------------------------------------
  BEVB200_CUDA(cudaMemsetAsync(w.zero_begin, 0, (size_t)(w.zero_end - w.zero_begin), ss));
  BEVB200_CUDA(cudaMemsetAsync(status_dev, 0, sizeof(int32_t) * (1 + nl), ss));
  // level 0: the caller's rows
  const int32_t *idx0 = coors;
  if (n_voxels_dev) {
    BEVB200_CUDA(cudaMemcpyAsync(w.counts[0], n_voxels_dev, sizeof(int32_t), cudaMemcpyDeviceToDevice, ss));
  } else {
    BEVB200_LAUNCH(enc_set_count_kernel, 1, 1, 0, ss, w.counts[0], max_voxels);
  }
  {
    EGeom g;
    memset(&g, 0, sizeof(g));
    for (int d = 0; d < 3; ++d) g.in_shape[d] = e->levels[0].shape[d];
    g.batch = batch_size;
    BEVB200_LAUNCH(enc_mark_rows_kernel, grid_for(caps[0], 256), 256, 0, ss, idx0, caps[0], w.counts[0], g, w.cells[0]);
    int rc = scan_level(0);
    if (rc) return rc;
    BEVB200_LAUNCH(enc_rank2row_kernel, grid_for(caps[0], 256), 256, 0, ss, idx0, caps[0], w.counts[0], g, w.cells[0],
                   w.rank2row);
  }
  std::vector<char> level_ready(nl, 0);
  level_ready[0] = 1;
  for (size_t r = 0; r < nr; ++r) {
    const ERulebook &rb = e->rulebooks[r];
    const EGeom g = geom_of(rb);
    const size_t lq = rb.level_q, li = rb.level_in;
    if (!level_ready[lq]) {
      // a new level: its sites are the outputs of this strided conv
      const int32_t *idx_in = li == 0 ? idx0 : w.indices[li];
      BEVB200_LAUNCH(enc_mark_outputs_kernel, grid_for(caps[li], 128), 128, 0, ss, idx_in, caps[li], w.counts[li], g,
                     w.cells[lq]);
      int rc = scan_level(lq);
      if (rc) return rc;
      BEVB200_LAUNCH(enc_count_kernel, 1, 1, 0, ss, w.total[lq], caps[lq], w.counts[lq], status_dev);
      const size_t nw = nwords_of(lq);
      BEVB200_LAUNCH(enc_out_indices_kernel, grid_for((long long)nw, 256), 256, 0, ss, w.cells[lq], nw,
                     e->levels[lq].shape[0], e->levels[lq].shape[1], e->levels[lq].shape[2], caps[lq], w.indices[lq]);
      level_ready[lq] = 1;
    }
    const int32_t *qidx = lq == 0 ? idx0 : w.indices[lq];
    BEVB200_LAUNCH(enc_nbr_kernel, dim3(grid_for(caps[lq], 256, kNumSMs * 4), rb.ksize[0] * rb.ksize[1]), 256, 0, ss,
                   qidx, caps[lq], w.counts[lq], g, w.cells[li], li == 0 ? w.rank2row : (const int32_t *)nullptr,
                   caps[li], w.nbr[r], (long long)caps[lq]);
    if (forked) BEVB200_CUDA(cudaEventRecord(e->events[1 + r], ss));
  }
  // row counts for the caller: status[1 + l]
  for (size_t l = 0; l < nl; ++l)
    BEVB200_CUDA(cudaMemcpyAsync(status_dev + 1 + l, w.counts[l], sizeof(int32_t), cudaMemcpyDeviceToDevice, ss));
  if (forked) BEVB200_CUDA(cudaEventRecord(e->events[1 + nr], ss));

  // ------------------------------ features (stream st) -------------------------------------
  int rc = spconv_v6_split_rows(voxel_features, caps[0], n_voxels_dev, e->in_channels, w.split[0][0], st);
  if (rc) return rc;
  std::vector<int> split_turn(nl, 0), f32_turn(nl, 0);
  split_turn[0] = 1;
  const uint8_t *cur_split = w.split[0][0];
  std::vector<const float *> f32_of(e->convs.size(), nullptr);
  std::vector<const uint8_t *> split_of(e->convs.size(), nullptr);
  std::vector<char> rb_waited(nr, 0);
  const float *last_f32 = nullptr;
  for (size_t i = 0; i < e->convs.size(); ++i) {
    const EConv &cv = e->convs[i];
    if (forked && !rb_waited[cv.rulebook]) {
      BEVB200_CUDA(cudaStreamWaitEvent(st, e->events[1 + cv.rulebook], 0));
      rb_waited[cv.rulebook] = 1;
    }
    const size_t lo = cv.level_out;
    const bool last = i + 1 == e->convs.size();
    uint8_t *osplit = nullptr;
    if (!last) {
      osplit = w.split[split_turn[lo]][lo];
      split_turn[lo] ^= 1;
    }
    float *of32 = nullptr;
    if (cv.want_fp32) {
      of32 = w.f32[f32_turn[lo]][lo];
      f32_turn[lo] ^= 1;
      f32_of[i] = of32;
    }
    // residual: the source conv's fp32 rows if it wrote them, else its split image (which may be the buffer this conv
    // writes: the two split buffers of a level alternate and a block's input is two convs back -- safe, see spconv_v6.cu)
    const float *res = cv.d.residual_from >= 0 ? f32_of[cv.d.residual_from] : nullptr;
    const uint8_t *res_split = (cv.d.residual_from >= 0 && res == nullptr) ? split_of[cv.d.residual_from] : nullptr;
    BEVB200_REQUIRE(cv.d.residual_from < 0 || res || res_split, "residual source has no rows");
    rc = spconv_v6_forward_ex(cur_split, pbase + cv.packed_off, w.nbr[cv.rulebook], (long long)caps[lo], caps[cv.level_in],
                              caps[lo], w.counts[lo], cv.c_in_eff, cv.d.c_out, cv.kvol,
                              cv.has_scale ? (const float *)(pbase + cv.scale_off) : nullptr,
                              cv.has_shift ? (const float *)(pbase + cv.shift_off) : nullptr, res, res_split, cv.d.relu,
                              of32, osplit, st);
    if (rc) return rc;
    split_of[i] = osplit;
    cur_split = osplit;
    last_f32 = of32;
  }
  // dense(): [B, C*Z, X, Y]
  {
    const ELevel &ll = e->levels.back();
    const int c = e->convs.back().d.c_out;
    const long long per_batch = (long long)c * ll.shape[0] * ll.shape[1] * ll.shape[2];
    if (out_batch_stride == 0) out_batch_stride = per_batch;
    BEVB200_REQUIRE(out_batch_stride >= per_batch, "output batch stride too small");
    if (out_batch_stride == per_batch) {
      BEVB200_CUDA(cudaMemsetAsync(dense_out, 0, (size_t)batch_size * per_batch * sizeof(float), st));
    } else {
      BEVB200_CUDA(cudaMemset2DAsync(dense_out, (size_t)out_batch_stride * sizeof(float), 0,
                                     (size_t)per_batch * sizeof(float), batch_size, st));
    }
    const size_t lo = nl - 1;
    BEVB200_LAUNCH(enc_dense_kernel, dim3(grid_for(caps[lo], 256, kNumSMs), c < 32 ? c : 32), 256, 0, st, last_f32,
                   w.indices[lo] ? w.indices[lo] : idx0, caps[lo], w.counts[lo], c, batch_size, ll.shape[0], ll.shape[1],
                   ll.shape[2], 1, out_batch_stride, dense_out);
  }
  if (forked) BEVB200_CUDA(cudaStreamWaitEvent(st, e->events[1 + nr], 0));   // join (also what a graph capture needs)
  return BEVB200_OK;
}

}  // extern "C"
