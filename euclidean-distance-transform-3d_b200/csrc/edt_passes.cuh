// edt_passes.cuh -- launchers of the axis-pass kernels, templated on the label width.
//
// Included by edt_passes_b{1,2,4,8}.cu, each of which instantiates launch_first / launch_later
// for ONE label width (the kernel templates are large; four translation units build in parallel).
// These launchers play the role of the per-axis loops of the reference's volume driver
// (pyedt::_edt3dsq, src/edt.hpp:428-475): which kernel variant, which tile shape, which grid.
// plan_first / plan_later make those choices in plain host code; the launchers carry them out.
#pragma once
#include "edt_host.h"

#include <cstdlib>

namespace edtb200 {
namespace host {

// An integer A/B switch of the environment, 0 when unset.  The launchers read each switch once per
// process and pass it to the plans; the tests force kernel variants with them.
inline int env_int(const char* name) { return getenv(name) ? atoi(getenv(name)) : 0; }

struct FirstPlan {
  int vec_k = 0;            // first_axis_vec_kernel<K> (rows of up to 128 K voxels); 0 = first_axis_kernel
  bool epilogue = false;    // flags != 0: the vector kernel's non-Plain instantiation
  size_t smem = 0;          // dynamic shared memory; above max_smem_optin the line does not fit
  int block = 0;
  int64_t grid = 0;
};

// x_grid: EDTB200_X_GRID, the vector kernel's CTAs per SM (0 = the built-in choice)
inline FirstPlan plan_first(int64_t nlines, int64_t sx, int label_bytes, uintptr_t labels_addr, uintptr_t f_addr,
                            int flags, int sm_count, int max_smem_optin, int x_grid) {
  FirstPlan p;
  p.epilogue = flags != 0;
  int64_t cap;
  // register-resident vector kernel when rows are short and 16-byte aligned
  if (sx % 4 == 0 && sx <= 1024 && labels_addr % (4 * label_bytes) == 0 && f_addr % 16 == 0) {
    p.vec_k = sx <= 128 ? 1 : sx <= 256 ? 2 : sx <= 512 ? 4 : 8;
    p.smem = sizeof(float) * (size_t)(sx + 2);
    p.block = 256;
    p.grid = (nlines + 7) / 8;
    cap = (int64_t)sm_count * (x_grid ? x_grid : (sx > 512 ? 12 : 15));   // whole waves at 5 (rows <= 512) / 3 CTAs per SM
  } else {
    const size_t per_warp = sizeof(uint32_t) * 4 * (size_t)((int)(sx >> 5) + 1);
    int warps = 8;
    while (warps > 1 && per_warp * warps > (size_t)max_smem_optin) warps >>= 1;
    p.smem = per_warp * warps;
    p.block = warps * 32;
    p.grid = (nlines + warps - 1) / warps;
    cap = (int64_t)sm_count * 16;
  }
  if (p.grid > cap) p.grid = cap;
  if (p.grid < 1) p.grid = 1;
  return p;
}

template <int Bytes, bool Plain, int K = 1>
auto first_vec_kernel(int k) {
  if constexpr (K < 8) {
    if (k > K) return first_vec_kernel<Bytes, Plain, K * 2>(k);
  }
  return first_axis_vec_kernel<Bytes, K, Plain>;
}

template <int Bytes>
int launch_first(const void* labels, float* f, int64_t nlines, int64_t sx, float w, int border, int flags,
                 DeviceCache& dc, cudaStream_t stream) {
  const float* table = nullptr;
  int trc = step_table(dc, w, (int)sx + 1, stream, &table);
  if (trc) return trc;
  const RunStat stat = {dc.stat_counter, dc.stat_ticket, dc.stat_publish_dev,
                        (unsigned long long)nlines * (unsigned long long)sx};

  static const int x_grid = env_int("EDTB200_X_GRID");
  const FirstPlan p = plan_first(nlines, sx, Bytes, reinterpret_cast<uintptr_t>(labels),
                                 reinterpret_cast<uintptr_t>(f), flags, dc.sm_count, dc.max_smem_optin, x_grid);
  if (p.smem > (size_t)dc.max_smem_optin)
    return fail(EDTB200_ELIMIT, "first axis of %lld voxels exceeds the shared-memory line buffer", (long long)sx);
  auto kern = first_axis_kernel<Bytes>;
  if (p.vec_k)
    kern = p.epilogue ? first_vec_kernel<Bytes, false>(p.vec_k) : first_vec_kernel<Bytes, true>(p.vec_k);
  else
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  kern<<<(unsigned)p.grid, p.block, p.smem, stream>>>(static_cast<const typename LabelOf<Bytes>::type*>(labels), f,
                                                      nlines, (int)sx, table, border, flags, stat);
  CUDA_TRY(cudaGetLastError());
  return step_table_used(dc, table, stream);
}

// Did the first-axis pass of the PREVIOUS transform on this device see label noise (at least nine
// runs per ten voxels along x)?  A prediction for the current volume, read from mapped host memory
// without any synchronisation; a wrong guess only costs speed (both kernel variants are complete).
inline bool noise_seen(const DeviceCache& dc) {
  const volatile unsigned long long* p = dc.stat_publish_host;
  if (!p) return false;
  const unsigned long long starts = p[0], voxels = p[1];
  return voxels > 0 && starts * 10ull >= voxels * 9ull;
}

// Tensor map over the distance volume for one later-axis pass: dims (adjacent lines, line
// length, outer), box = tx lines x box_rows.
inline bool make_tile_map(CUtensorMap* map, float* f, const LineGeom& g, int tx, int box_rows) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)g.inner_count, (cuuint64_t)g.n, (cuuint64_t)g.outer_count};
  const cuuint64_t strides[2] = {(cuuint64_t)g.line_stride * sizeof(float),
                                 (cuuint64_t)(g.outer_count > 1 ? g.outer_stride : g.line_stride * (int64_t)g.n) *
                                     sizeof(float)};
  const cuuint32_t box[3] = {(cuuint32_t)tx, (cuuint32_t)box_rows, 1u};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, f, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

inline void tile_boxes(int n, TileBoxes* tb) {
  tb->nboxes = (n + 255) / 256;
  tb->box_rows = (n + tb->nboxes - 1) / tb->nboxes;
  if (tb->nboxes > 1) tb->box_rows = (tb->box_rows + 3) & ~3;      // keeps every box 128-byte aligned
}

// Shared memory of one tile of `tx` lines (see later_axis_tile_kernel).
inline size_t tile_smem_bytes(int n, int tx, int rows_alloc) {
  const int nchunks = (n + 31) >> 5;
  return (size_t)rows_alloc * tx * 4 + (size_t)nchunks * tx * 12 + (size_t)((n + 3) & ~1) * 4 + 16 +
         (size_t)nchunks * tx +    // + one flag byte per (chunk, line)
         (size_t)tx * 4 + 4;       // + one word per line: chunks holding a run start
}

struct LaterPlan {
  bool tile = false;        // shared-memory tile kernel; false = later_axis_long_kernel
  int tx = 0;               // tile width in lines: 32, 16 or 8
  bool tma = false;         // TMA staging of the tile
  bool wide = false;        // long lines: one tile per SM with up to 32 warps
  int ctas = 3;             // CTAs per SM the kernel is built for: 2 = the noise variant
  bool int_hull = false;    // integer hull tests
  bool epilogue = false;    // flags != 0
  TileBoxes tb = {0, 0};
  int rows_alloc = 0;
  size_t smem = 0;
  int warps = 0;            // tile kernel: warps per CTA (the long kernel runs 128 threads)
  int64_t grid = 0;         // tiles, or blocks of 128 lines for the long kernel
  LineGeom g;               // the pass's geometry, tiles_per_outer set for the tile kernel
};

// fmax >= 0: the caller vouches that every finite sample of f is an integer not above fmax.
// tile_ctas: EDTB200_TILE_CTAS (2 / 3 forces the noise / normal variant); no_int_hull: EDTB200_NO_INT_HULL.
// tma_ok = false: the tensor map could not be encoded, so the tile is loaded without TMA.
inline LaterPlan plan_later(const LineGeom& g, uintptr_t f_addr, float w2, int flags, double fmax, bool noise_hint,
                            int max_smem_optin, int tile_ctas, bool no_int_hull, bool tma_ok) {
  LaterPlan p;
  p.g = g;
  p.epilogue = flags != 0;
  // ---- shared-memory tile kernel: whole lines x TX adjacent lines per CTA ----
  const bool fits32 = (int64_t)g.n * g.line_stride + 64 < (1LL << 32);
  if (fits32 && g.n <= 4096 && g.inner_count < (1LL << 31)) {
    tile_boxes(g.n, &p.tb);
    // Tile width: 128-byte rows (TX = 32) keep DRAM pages and L2 lines whole and measured
    // fastest even at one CTA per SM; narrower tiles only when a 32-wide tile cannot fit.
    // The width is chosen for TMA staging whether or not TMA is used.
    for (int cand = 32; cand >= 8 && !p.tx; cand >>= 1)
      if (tile_smem_bytes(g.n, cand, p.tb.box_rows * p.tb.nboxes) <= (size_t)max_smem_optin) p.tx = cand;
  }
  if (!p.tx) {
    p.grid = (g.inner_count * g.outer_count + 127) / 128;
    return p;
  }
  p.tile = true;
  const bool aligned = f_addr % 16 == 0 && g.line_stride % 4 == 0 && (g.outer_count <= 1 || g.outer_stride % 4 == 0);
  p.tma = tma_ok && aligned && g.inner_count >= p.tx;
  p.rows_alloc = p.tma ? p.tb.box_rows * p.tb.nboxes : g.n;
  p.smem = tile_smem_bytes(g.n, p.tx, p.rows_alloc);
  const int subs = 32 / p.tx;
  p.warps = (((g.n + 31) >> 5) + subs - 1) / subs;
  p.wide = p.warps > 16;
  if (p.warps > 32) p.warps = 32;
  p.g.tiles_per_outer = (int)((g.inner_count + p.tx - 1) / p.tx);
  p.grid = (int64_t)p.g.tiles_per_outer * g.outer_count;
  // the noise variant and the integer hull tests are instantiated for the hot shape only
  // (128-byte rows, TMA staging)
  const bool hot = p.tx == 32 && p.tma;
  if (hot && !p.wide && (tile_ctas == 2 || (tile_ctas != 3 && noise_hint))) p.ctas = 2;
  // Integer hull tests: with an integer w2 and fmax + w2 * n^2 < 2^31 every g = f + w2 v^2 is an
  // exact 32-bit integer.  fmax < 0 = unknown -> double.
  p.int_hull = hot && !no_int_hull && fmax >= 0.0 && w2 == floorf(w2) && w2 >= 1.0f && w2 < 1048576.0f &&
               fmax + (double)w2 * (double)g.n * (double)g.n < 2147483000.0;
  return p;
}

// Only the hot shape (TX = 32, TMA) has the noise and integer-hull variants.
template <int Bytes, int TX, bool Epi, bool TMA, bool IH = false>
auto tile_variant(const LaterPlan& p) {
  constexpr bool hot = TX == 32 && TMA;
  if constexpr (hot && !IH) {
    if (p.int_hull) return tile_variant<Bytes, TX, Epi, TMA, true>(p);
  }
  if (p.wide) return later_axis_tile_kernel<Bytes, TX, Epi, TMA, true, 3, IH>;
  if constexpr (hot) {
    if (p.ctas == 2) return later_axis_tile_kernel<Bytes, TX, Epi, TMA, false, 2, IH>;
  }
  return later_axis_tile_kernel<Bytes, TX, Epi, TMA, false, 3, IH>;
}

// The tile kernel a plan asks for.
template <int Bytes, int TX = 32>
auto tile_kernel(const LaterPlan& p) {
  if constexpr (TX > 8) {
    if (p.tx < TX) return tile_kernel<Bytes, TX / 2>(p);
  }
  if (p.epilogue) return p.tma ? tile_variant<Bytes, TX, true, true>(p) : tile_variant<Bytes, TX, true, false>(p);
  return p.tma ? tile_variant<Bytes, TX, false, true>(p) : tile_variant<Bytes, TX, false, false>(p);
}

template <int Bytes>
int launch_later(const void* labels, float* f, const LineGeom& g0, float w, int border_lo, int border_hi,
                 int flags, DeviceCache& dc, cudaStream_t stream, bool pdl, double fmax) {
  const auto* lab = static_cast<const typename LabelOf<Bytes>::type*>(labels);
  const float w2 = w * w;                       // float product, as src/edt.hpp:181
  static const int tile_ctas = env_int("EDTB200_TILE_CTAS");
  static const bool no_pdl = getenv("EDTB200_NO_PDL") != nullptr;
  static const bool no_int_hull = getenv("EDTB200_NO_INT_HULL") != nullptr;
  const bool noise = noise_seen(dc);
  auto plan = [&](bool tma_ok) {
    return plan_later(g0, reinterpret_cast<uintptr_t>(f), w2, flags, fmax, noise, dc.max_smem_optin, tile_ctas,
                      no_int_hull, tma_ok);
  };
  LaterPlan p = plan(true);
  if (p.grid > 0x7fffffffLL) return fail(EDTB200_ELIMIT, p.tile ? "too many line tiles" : "too many lines");
  if (p.tile) {
    CUtensorMap map = {};
    if (p.tma && !make_tile_map(&map, f, p.g, p.tx, p.tb.box_rows)) p = plan(false);
    const auto kern = tile_kernel<Bytes>(p);
    // Programmatic dependent launch: this pass may begin (label staging) while the previous pass of
    // the stream drains its last wave; the kernel itself waits before touching the distances.  Only
    // when the previous kernel of the stream is our own pass.
    cudaLaunchAttribute pdl_attr;
    pdl_attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl_attr.val.programmaticStreamSerializationAllowed = 1;
    const cudaLaunchConfig_t cfg = {dim3((unsigned)p.grid), dim3((unsigned)(p.warps * 32)), p.smem, stream,
                                    &pdl_attr, (pdl && !no_pdl) ? 1u : 0u};
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, map, lab, f, p.g, p.tb, w2, border_lo, border_hi, flags,
                                p.int_hull ? (int)w2 : 0));
    CUDA_TRY(cudaGetLastError());
    return 0;
  }
  // ---- long lines: out of place through a temporary volume ----
  const size_t bytes = sizeof(float) * (size_t)(g0.inner_count * g0.outer_count) * (size_t)g0.n;
  float* tmp = nullptr;
  int* hull = nullptr;
  CUDA_TRY(scratch_alloc(dc, reinterpret_cast<void**>(&tmp), bytes, stream));
  if (scratch_alloc(dc, reinterpret_cast<void**>(&hull), bytes, stream) != cudaSuccess) {
    cudaGetLastError();
    cudaFreeAsync(tmp, stream);
    return fail(EDTB200_ENOMEM, "no device memory for the long-line scratch volumes");
  }
  later_axis_long_kernel<Bytes><<<(unsigned)p.grid, 128, 0, stream>>>(lab, f, tmp, hull, g0, w2, border_lo,
                                                                      border_hi, flags);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(f, tmp, bytes, cudaMemcpyDeviceToDevice, stream));
  CUDA_TRY(cudaFreeAsync(hull, stream));
  CUDA_TRY(cudaFreeAsync(tmp, stream));
  return 0;
}

}  // namespace host
}  // namespace edtb200

#define EDT_INSTANTIATE_PASSES(B)                                                                        \
  template int edtb200::host::launch_first<B>(const void*, float*, int64_t, int64_t, float, int, int,    \
                                              edtb200::host::DeviceCache&, cudaStream_t);                \
  template int edtb200::host::launch_later<B>(const void*, float*, const edtb200::LineGeom&, float, int, \
                                              int, int, edtb200::host::DeviceCache&, cudaStream_t, bool, \
                                              double);
