// K3 -- fused clamp + normalise + colormap-LUT rasteriser.
//
// csg_panel_prepare restates make_spectrogram's z handling (CS/plotting.py:259-279 log branch,
// :307-315 linear branch) per panel on the device, from the region stats of K2a.
// csg_rasterise restates what imshow(matrix, cmap=, norm=LogNorm(..) | vmin=,vmax=) colours at
// cell resolution (CS/plotting.py:280-287,316-324): matplotlib 3.11 Normalize.__call__ /
// LogNorm (make_norm_from_scale(LogScale, nonpositive="mask")) and Colormap._get_rgba_and_mask.
// matplotlib is not installable in the build image, so this boundary is restated from the
// published algorithm (parity unpinned, see DESIGN.md):
//   x  = D(f64(v) - vmin);  x = D(f64(x) / (vmax - vmin))          [in-place ops, f64 scalars]
//   log: v -> log10_D(v) first, vmin/vmax -> log10 in f64
//   xa = x * 256 (in D); xa == 256 -> 255; xa < 0 -> under(256); xa >= 256 -> over(257);
//   NaN / masked -> bad(258); else trunc(xa).
// log10_D for float32 is defined as the correctly rounded float32 of the float64 logarithm
// (numpy's own float32 log10 is libm/SVML dependent).
#include "common.cuh"

namespace {

constexpr int I_UNDER = 256, I_OVER = 257, I_BAD = 258;

template <typename T>
__device__ __forceinline__ T round_to(double v) {
  return (T)v;
}

template <typename T>
__device__ __forceinline__ T log10_d(T v);
template <>
__device__ __forceinline__ float log10_d<float>(float v) {
  return (float)log10((double)v);
}
template <>
__device__ __forceinline__ double log10_d<double>(double v) {
  return log10(v);
}

// the reference's clamps before imshow: CS/plotting.py:278 (log), :310-312 (linear)
template <typename T>
__device__ __forceinline__ T substitute(T v, const csg_panel_norm& nm, bool log_scale) {
  if (log_scale) {
    if (!is_finite(v) || v <= T(0)) v = (T)nm.fill_lo;  // np.where(~isfinite(m) | (m <= 0), z_axis_min, m)
  } else {
    if (is_nan(v)) v = (T)nm.fill_lo;
    if (v == (T)(-CUDART_INF)) v = (T)nm.fill_lo;
    if (v == (T)CUDART_INF) v = (T)nm.fill_hi;
  }
  return v;
}

// matplotlib's index for an (already substituted) value, evaluated directly
template <typename T>
__device__ __forceinline__ int cmap_index_direct(T v, const csg_panel_norm& nm, bool log_scale) {
  if (nm.degenerate == 1) return 0;  // vmin == vmax: result.fill(0) / np.full_like(value, 0)
  T x;
  if (log_scale) {
    const T t = log10_d<T>(v);
    x = (T)((double)t - nm.t_vmin);
    x = (T)((double)x / nm.t_range);
    if (!is_finite(x)) return I_BAD;  // np.ma.masked_invalid
  } else {
    x = (T)((double)v - nm.t_vmin);
    x = (T)((double)x / nm.t_range);
  }
  T xa = mul_rn(x, T(256));
  if (xa == T(256)) xa = T(255);
  if (is_nan(xa)) return I_BAD;
  if (xa < T(0)) return I_UNDER;
  if (xa >= T(256)) return I_OVER;
  return (int)xa;
}

// The index is a monotone step function of the value, so a panel needs at most 257
// thresholds: thr[k] = smallest value whose "monotone code" (under = -1, 0..255, over = 256)
// is >= k.  The rasteriser then only counts thresholds <= value -- exact by construction
// (the thresholds come from the direct formula) and free of per-pixel float64 log10.
template <typename T>
__device__ __forceinline__ int monotone_code(T v, const csg_panel_norm& nm, bool log_scale) {
  const int idx = cmap_index_direct<T>(v, nm, log_scale);
  return idx == I_UNDER ? -1 : (idx == I_OVER ? 256 : idx);  // I_BAD cannot occur for ordered finite input
}

constexpr int kThr = 257;
constexpr int kThrPitch = 264;  // padded row length of the threshold table

template <typename T>
__global__ void __launch_bounds__(288)
    panel_threshold_kernel(const csg_panel* __restrict__ panels, const csg_panel_norm* __restrict__ norms, int n_panels,
                           T* __restrict__ thresholds) {
  typedef typename Key<T>::U U;
  const int pi = blockIdx.x;
  const int k = threadIdx.x;
  if (k >= kThr) return;
  const csg_panel_norm nm = norms[pi];
  T* out = thresholds + (size_t)pi * kThrPitch;
  if (nm.status != CSG_NORM_OK || nm.degenerate != 0) {
    out[k] = (T)CUDART_INF;
    return;
  }
  const bool log_scale = panels[pi].log_scale != 0;
  // ordered domain of substituted values: finite positives (log) or [-inf, +inf] (linear)
  const U dom_lo = log_scale ? Key<T>::key((T)0) + 1 : Key<T>::key((T)(-CUDART_INF));
  const U dom_hi = log_scale ? Key<T>::key((T)CUDART_INF) - 1 : Key<T>::key((T)CUDART_INF);
  auto code = [&](U key) { return monotone_code<T>(Key<T>::val(key), nm, log_scale); };
  // start from the analytic inverse, then gallop to a bracket and bisect
  const double frac = (double)k / 256.0;
  double guess = log_scale ? exp10(nm.t_vmin + frac * nm.t_range) : nm.t_vmin + frac * nm.t_range;
  T gT = (T)guess;
  if (is_nan(gT)) gT = T(1);
  U g = Key<T>::key(gT);
  if (g < dom_lo) g = dom_lo;
  if (g > dom_hi) g = dom_hi;
  U lo, hi;  // invariant once bracketed: code(lo) < k <= code(hi)
  U step = 2;
  constexpr U kMaxStep = (U)1 << (Key<T>::BITS - 2);  // the gallop saturates: a step that wrapped to 0 would never move
  bool found = true;
  if (code(g) >= k) {
    hi = g;
    while (true) {
      if (hi == dom_lo) {  // even the smallest value reaches k
        lo = hi;
        break;
      }
      lo = (hi - dom_lo > step) ? hi - step : dom_lo;
      if (code(lo) < k) break;
      hi = lo;
      if (step < kMaxStep) step <<= 2;
    }
  } else {
    lo = g;
    while (true) {
      if (lo == dom_hi) {  // no value reaches k
        found = false;
        break;
      }
      hi = (dom_hi - lo > step) ? lo + step : dom_hi;
      if (code(hi) >= k) break;
      lo = hi;
      if (step < kMaxStep) step <<= 2;
    }
  }
  if (!found) {
    out[k] = (T)CUDART_INF;
    return;
  }
  while (hi - lo > 1) {
    const U mid = lo + ((hi - lo) >> 1);
    if (code(mid) >= k)
      hi = mid;
    else
      lo = mid;
  }
  out[k] = Key<T>::val(hi);
}

template <typename T>
__global__ void panel_prepare_kernel(const csg_panel* __restrict__ panels, int n_panels,
                                     const csg_region_stats* __restrict__ stats, const double* __restrict__ zvals,
                                     csg_panel_norm* __restrict__ norms) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_panels) return;
  const csg_panel p = panels[i];
  const csg_region_stats own = stats[p.stat_region >= 0 ? p.stat_region : p.region];
  const csg_region_stats pct = stats[p.pct_region >= 0 ? p.pct_region : p.region];
  // compute_percentile_bounds(matrix, 1, 99, z_min, z_max)   CS/plotting.py:259
  const double given_lo = (p.zmin_slot >= 0 && zvals) ? zvals[p.zmin_slot] : p.z_min;
  const double given_hi = (p.zmax_slot >= 0 && zvals) ? zvals[p.zmax_slot] : p.z_max;
  double zmin = is_nan(given_lo) ? pct.p_lo : given_lo;
  double zmax = is_nan(given_hi) ? pct.p_hi : given_hi;
  csg_panel_norm nm;
  nm.status = CSG_NORM_OK;
  nm.degenerate = 0;
  nm.c0 = nm.c1 = 0.f;
  if (p.log_scale) {
    // safe_vmin = nanmin(finite positive) or 1e-10; z_min = float(max(z_min, safe_vmin, 1e-10))  :261-276
    const double safe = own.n_pos > 0 ? own.min_pos : 1e-10;
    double m = zmin;  // Python max(): keep the first unless a later one compares greater
    if (safe > m) m = safe;
    if (1e-10 > m) m = 1e-10;
    zmin = m;
    nm.vmin = zmin, nm.vmax = zmax;
    nm.fill_lo = (double)(T)zmin;
    nm.fill_hi = (double)(T)zmax;
    // LogNorm.__call__ checks, in matplotlib's order
    if (zmin > zmax) {
      nm.status = CSG_NORM_VMIN_GT_VMAX;
    } else if (zmin == zmax) {
      nm.degenerate = 1;
    }
    const double tlo = log10(zmin), thi = log10(zmax);
    nm.t_vmin = tlo;
    nm.t_range = thi - tlo;
    if (nm.status == CSG_NORM_OK && !nm.degenerate && !(is_finite(tlo) && is_finite(thi)))
      nm.status = CSG_NORM_INVALID;
    // vmin < vmax a few ulps apart, but log10 rounds both to the same double: every normalised value is
    // (t - t_vmin) / 0 = +-inf or NaN, which LogNorm masks -> "bad", like a NaN bound
    if (nm.status == CSG_NORM_OK && !nm.degenerate && nm.t_range == 0.0) nm.degenerate = 2;
  } else {
    nm.fill_lo = (double)(T)zmin;
    nm.fill_hi = (double)(T)zmax;
    if (!(is_finite(zmin) && is_finite(zmax) && zmax > zmin)) {
      // z_min = nanmin(matrix), z_max = nanmax(matrix) over the substituted matrix   :313-315
      double lo = CUDART_INF, hi = -CUDART_INF;
      bool any = false;
      if (own.fin_min <= own.fin_max) {
        lo = own.fin_min, hi = own.fin_max, any = true;
      }
      if ((own.n_nan > 0 || own.n_neginf > 0) && !is_nan(nm.fill_lo)) {
        lo = fmin(lo, nm.fill_lo), hi = fmax(hi, nm.fill_lo), any = true;
      }
      if (own.n_posinf > 0 && !is_nan(nm.fill_hi)) {
        lo = fmin(lo, nm.fill_hi), hi = fmax(hi, nm.fill_hi), any = true;
      }
      zmin = any ? lo : CUDART_NAN;
      zmax = any ? hi : CUDART_NAN;
    }
    nm.vmin = zmin, nm.vmax = zmax;
    nm.t_vmin = zmin;
    nm.t_range = zmax - zmin;
    if (zmin == zmax)
      nm.degenerate = 1;
    else if (zmin > zmax)
      nm.status = CSG_NORM_VMIN_GT_VMAX;
    else if (is_nan(zmin) || is_nan(zmax))
      nm.degenerate = 2;  // every normalised value is NaN -> "bad" colour
    else if (!is_finite(nm.t_range))
      // vmax - vmin = inf (an infinite percentile bound, or finite bounds whose difference overflows):
      // (v - vmin) / inf is NaN ("bad") where v - vmin is infinite -- every cell when vmin = -inf -- and 0
      // elsewhere.  Not a monotone step function of v, so no threshold table: the rasteriser tests each cell.
      nm.degenerate = is_finite(zmin) ? 3 : 2;
  }
  // first-guess coefficients of the rasteriser: #{thresholds <= v} ~ c1 * (log2 v | v) + c0
  nm.c1 = p.log_scale ? (float)(256.0 * 0.30102999566398120 / nm.t_range) : (float)(256.0 / nm.t_range);
  nm.c0 = (float)(-256.0 * nm.t_vmin / nm.t_range) + 1.0f;
  norms[i] = nm;
}

// A chunk = kPixPerBlock consecutive pixels of one panel's (E', T') image.  The collapsed matrices
// are energy-major, so consecutive pixels of an image row are consecutive cells of one matrix row:
// reads and writes are both fully coalesced and there is no transpose.  A thread owns groups of four
// consecutive pixels (one 128-bit RGBA store; one 128-bit load when the four cells are an aligned
// run of one matrix row).  Each cell is mapped to its LUT index through the panel's threshold table:
// a fast float guess of the count, verified against the two exact thresholds around it (exact by
// construction).
//
// The per-pixel table lookups are random, and at one or two table reads plus one LUT read per
// pixel the shared-memory pipe -- not HBM -- bounds the kernel when lanes collide on banks.  So
// both tables are kept BANK-REPLICATED: row k of a table is 32 words, one per lane, and a lane
// only ever reads its own column -- every lookup is a single conflict-free wavefront.  Blocks
// are persistent (a contiguous range of chunks each), so the replicated LUT is built once per
// block and the thresholds once per panel the block meets.
constexpr int kRasterThreads = 512;
constexpr int kPixPerThread = 16;
constexpr int kPixPerBlock = kRasterThreads * kPixPerThread;
constexpr int kRows = kThr + 2;       // thr[-1] = -inf, thr[0..256], thr[257] = +inf
constexpr int kLutRows = 260;

__device__ __forceinline__ float fast_log2(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));  // only a first guess: verified against the table
  return r;
}

__device__ __forceinline__ void lds(float& v, unsigned addr) { asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr)); }
__device__ __forceinline__ void lds(double& v, unsigned addr) { asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr)); }

// The out-of-line half of the rasteriser's value -> threshold-count lookup: walk the lane's own table
// column from a wrong first guess; NaN (it fails every comparison) counts as 258 = "bad".
template <typename T>
__device__ __noinline__ int recount(T v, int n, unsigned thr_col) {
  if (is_nan(v)) return 258;
  auto thr_at = [&](int row) -> T {
    T t;
    lds(t, thr_col + (unsigned)row * (32u * (unsigned)sizeof(T)));
    return t;
  };
  while (n > 0 && !(thr_at(n) <= v)) --n;
  while (n < kThr && thr_at(n + 1) <= v) ++n;
  return n;
}

template <bool B>
struct Flag {
  static constexpr bool value = B;
};

template <typename T>
constexpr size_t raster_smem_bytes() {
  return (size_t)kLutRows * 32 * sizeof(uint32_t) + (size_t)kRows * 32 * sizeof(T);
}

template <typename T>
__global__ void __launch_bounds__(kRasterThreads, sizeof(T) == 4 ? 3 : 2)
    rasterise_kernel(const T* __restrict__ mats, const csg_region* __restrict__ regions,
                     const int32_t* __restrict__ pool, const csg_panel* __restrict__ panels,
                     const csg_panel_norm* __restrict__ norms, int chunk_offset, int n_chunks,
                     const int32_t* __restrict__ block_panel, const T* __restrict__ thresholds,
                     const uint32_t* __restrict__ lut, uint32_t* __restrict__ rgba, uint16_t* __restrict__ index) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  T* s_thr = reinterpret_cast<T*>(s_raw);                                             // [kRows][32]
  uint32_t* s_lut = reinterpret_cast<uint32_t*>(s_raw + (size_t)kRows * 32 * sizeof(T));  // [kLutRows][32]

  const int tid = threadIdx.x, lane = tid & 31;
  // this block's contiguous range of chunks
  const int per = (n_chunks + (int)gridDim.x - 1) / (int)gridDim.x;
  const int c_begin = (int)blockIdx.x * per, c_end = min(n_chunks, c_begin + per);
  if (c_begin >= c_end) return;
  // LUT rows are keyed by the threshold COUNT n (what the lookup produces): 0 = under, 1..256 = colours
  // 0..255, 257 = over, 258 = bad -- the colormap index itself is only formed for the index plane
  for (int w = tid; w < kLutRows * 32; w += kRasterThreads) {
    const int n = w >> 5;
    const int idx = n == 0 ? I_UNDER : (n == kThr ? I_OVER : (n <= 256 ? n - 1 : I_BAD));
    s_lut[w] = (lut && n < 259) ? __ldg(lut + idx) : 0u;
  }
  // explicit shared-window addresses of this lane's table columns: row r of a table is 32 words
  // (128 bytes for float32 / the LUT) further on -- one add and one ld.shared per lookup
  unsigned thr_col = (unsigned)__cvta_generic_to_shared(s_thr + lane);  // row r (threshold k = r - 1)
  unsigned lut_col = (unsigned)__cvta_generic_to_shared(s_lut + lane);
  // opaque to the optimiser: otherwise both addresses are re-derived from %tid (seven instructions each)
  // at every lookup instead of living in a register
  asm volatile("" : "+r"(thr_col), "+r"(lut_col));
  auto thr_at = [&](int row) -> T {
    T v;
    lds(v, thr_col + (unsigned)row * (32u * (unsigned)sizeof(T)));
    return v;
  };
  auto lut_at = [&](int row) -> uint32_t {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(lut_col + (unsigned)row * 128u));
    return v;
  };

  int cur_panel = -1;
  // panel state (reloaded when the block crosses into another panel)
  bool skip = false, log_scale = false;
  int degenerate = 0;
  unsigned nt = 1, n_pix = 0;
  int first_block = 0, ld = 0, t0 = 0, rows_off = -1;
  long long out_off = 0;
  float c1 = 0.f, c0 = 0.f;
  T fill_lo = T(0), fill_hi = T(0);
  const T* mat = mats;
  const int32_t *cols = pool, *rows = pool;
  bool in_vec = false;

  for (int chunk = c_begin; chunk < c_end; ++chunk) {
    const int blk = chunk + chunk_offset;
    const int pi = __ldg(block_panel + blk);
    if (pi != cur_panel) {
      cur_panel = pi;
      const csg_panel* pn = panels + pi;
      const csg_region* rg = regions + __ldg(&pn->region);
      const csg_panel_norm* nm = norms + pi;
      skip = __ldg(&nm->status) != CSG_NORM_OK;  // the host raises matplotlib's ValueError for this panel
      degenerate = __ldg(&nm->degenerate);
      log_scale = __ldg(&pn->log_scale) != 0;
      nt = (unsigned)__ldg(&rg->nt);
      n_pix = (unsigned)__ldg(&rg->ne) * nt;
      first_block = __ldg(&pn->first_block);
      out_off = __ldg(&pn->out_off);
      c1 = __ldg(&nm->c1), c0 = __ldg(&nm->c0);
      fill_lo = (T)__ldg(&nm->fill_lo), fill_hi = (T)__ldg(&nm->fill_hi);
      mat = mats + __ldg(&rg->mat_off);
      cols = pool + __ldg(&rg->cols_off);
      rows_off = __ldg(&rg->rows_off);
      rows = pool + (rows_off < 0 ? 0 : rows_off);
      ld = __ldg(&rg->ld), t0 = __ldg(&rg->t0);
      in_vec = sizeof(T) == 4 && rows_off < 0 && (ld & 3) == 0 && (__ldg(&rg->mat_off) & 3) == 0 &&
               (reinterpret_cast<uintptr_t>(mats) & 15) == 0;
      __syncthreads();  // every lane is done with the previous panel's thresholds
      if (!skip && degenerate == 0) {
        const T* thr = thresholds + (size_t)pi * kThrPitch;
        for (int w = tid; w < kRows * 32; w += kRasterThreads) {
          const int k = (w >> 5) - 1;
          s_thr[w] = k < 0 ? (T)(-CUDART_INF) : (k >= kThr ? (T)CUDART_INF : __ldg(thr + k));
        }
      }
      __syncthreads();
    }
    if (skip) continue;
    const unsigned first = (unsigned)(blk - first_block) * kPixPerBlock;
    const unsigned last = first + kPixPerBlock < n_pix ? first + kPixPerBlock : n_pix;
    uint32_t* out_rgba = rgba ? rgba + out_off : nullptr;
    uint16_t* out_idx = index ? index + out_off : nullptr;
    if (degenerate != 0) {
      // 1: vmin == vmax, every cell maps to index 0; 2: NaN bound, every cell is "bad"; 3 (linear, vmax - vmin
      // = inf): index 0, or "bad" where the in-place subtraction v - vmin is infinite (inf / inf = NaN)
      const csg_panel_norm* nm = norms + cur_panel;
      const double vmin = degenerate == 3 ? __ldg(&nm->t_vmin) : 0.0;
      for (unsigned i = first + tid; i < last; i += kRasterThreads) {
        bool bad = degenerate == 2;
        if (degenerate == 3) {
          const unsigned jj = i / nt, t = i - jj * nt;
          T v = __ldg(mat + __ldg(cols + jj) * ld + (rows_off < 0 ? t0 + (int)t : __ldg(rows + t)));
          v = (is_nan(v) || v == (T)(-CUDART_INF)) ? fill_lo : (v == (T)CUDART_INF ? fill_hi : v);
          bad = !is_finite((T)((double)v - vmin));
        }
        if (out_rgba) out_rgba[i] = lut_at(bad ? 258 : 1);
        if (out_idx) out_idx[i] = (uint16_t)(bad ? I_BAD : 0);
      }
      continue;
    }

    // value -> number of thresholds <= value (258 for NaN).  A fast float guess n of the count is verified
    // against the two exact thresholds around it: n thresholds are <= v  <=>  thr[n-1] <= v < thr[n] (table
    // rows are offset by one: thr[k] = row k + 1).  The common path of a pixel is ~15 instructions: clamp
    // (2 compares + select), lg2 + fma, 2 x fmnmx + convert, one address, two ld.shared, two compares whose
    // verdict is only accumulated; a group of four pixels branches ONCE, and only when some guess was off or
    // some value is NaN (it fails every comparison) does the out-of-line walk (recount) run.
    auto substituted = [&](T v, auto log_c) -> T {
      constexpr bool LOG = decltype(log_c)::value;
      // the reference's clamps before imshow: CS/plotting.py:278 (log), :310-312 (linear)
      if (LOG) return (v > T(0)) & is_finite(v) ? v : fill_lo;
      v = (is_nan(v) || v == (T)(-CUDART_INF)) ? fill_lo : v;
      return (v == (T)CUDART_INF) ? fill_hi : v;
    };
    auto guess = [&](T v, auto log_c, bool& ok) -> int {
      constexpr bool LOG = decltype(log_c)::value;
      const float fv = (float)v;
      float gf = __fmaf_rn(LOG ? fast_log2(fv) : fv, c1, c0);
      gf = fminf(fmaxf(gf, 0.f), (float)kThr);  // NaN -> 0
      const int n = (int)gf;
      const unsigned row = thr_col + (unsigned)n * (32u * (unsigned)sizeof(T));
      T lo_thr, hi_thr;
      lds(lo_thr, row);
      lds(hi_thr, row + 32u * (unsigned)sizeof(T));
      ok = ok & (lo_thr <= v) & !(hi_thr <= v);
      return n;
    };
    auto to_count = [&](T raw, auto log_c) -> int {  // single pixels (panel tails)
      const T v = substituted(raw, log_c);
      bool ok = true;
      const int n = guess(v, log_c, ok);
      return ok ? n : recount<T>(v, n, thr_col);
    };
    auto count_to_index = [](int n) -> int { return n == 0 ? I_UNDER : (n == kThr ? I_OVER : (n == 258 ? I_BAD : n - 1)); };

    // the pixel loop, specialised on the scale, on how time steps are addressed and on what is written
    // (RGBA / index plane; 128-bit stores when the panel's output is aligned -- it always is for buffers
    // laid out by the host wrapper); 32-bit index math; a thread takes four consecutive pixels per step
    const bool out_vec = (out_off & 3) == 0 && (!out_rgba || (reinterpret_cast<uintptr_t>(rgba) & 15) == 0) &&
                         (!out_idx || (reinterpret_cast<uintptr_t>(index) & 7) == 0);
    auto pixels = [&](auto log_c, auto rowlist_c, auto rgba_c, auto idx_c, auto vec_c) {
      constexpr bool ROWLIST = decltype(rowlist_c)::value;
      constexpr bool RGBA = decltype(rgba_c)::value, INDEX = decltype(idx_c)::value, VEC = decltype(vec_c)::value;
      constexpr unsigned G = 4, STEP = G * kRasterThreads;
      unsigned i = first + G * tid;
      unsigned j = i / nt, tt = i - j * nt;
      const unsigned dq = STEP / nt, dr = STEP - dq * nt;
      auto address = [&](unsigned jj, unsigned t) -> unsigned {
        return (unsigned)(__ldg(cols + jj) * ld + (ROWLIST ? __ldg(rows + t) : t0 + (int)t));
      };
      auto load4 = [&](unsigned jj, unsigned t, T* v) {  // cells of pixels i..i+3 (the caller checked i + 3 < last)
        if (t + (G - 1) < nt) {
          const unsigned a0 = address(jj, t);
          if (!ROWLIST && in_vec && (a0 & 3u) == 0) {
            if constexpr (sizeof(T) == 4) {
              const float4 q = __ldg(reinterpret_cast<const float4*>(mat + a0));
              v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
            }
          } else if (!ROWLIST) {
#pragma unroll
            for (unsigned u = 0; u < G; ++u) v[u] = __ldg(mat + a0 + u);
          } else {
            const unsigned c = (unsigned)(__ldg(cols + jj) * ld);
#pragma unroll
            for (unsigned u = 0; u < G; ++u) v[u] = __ldg(mat + c + __ldg(rows + t + u));
          }
        } else {  // the group straddles two image rows
#pragma unroll
          for (unsigned u = 0; u < G; ++u) {
            v[u] = __ldg(mat + address(jj, t));
            if (++t == nt) t = 0, ++jj;
          }
        }
      };
      auto store4 = [&](unsigned at, const int* n) {
        if constexpr (RGBA) {
          if constexpr (VEC)
            *reinterpret_cast<uint4*>(out_rgba + at) = make_uint4(lut_at(n[0]), lut_at(n[1]), lut_at(n[2]), lut_at(n[3]));
          else {
#pragma unroll
            for (unsigned u = 0; u < G; ++u) out_rgba[at + u] = lut_at(n[u]);
          }
        }
        if constexpr (INDEX) {
          int idx[G];
#pragma unroll
          for (unsigned u = 0; u < G; ++u) idx[u] = count_to_index(n[u]);
          if constexpr (VEC)
            *reinterpret_cast<uint2*>(out_idx + at) =
                make_uint2((unsigned)idx[0] | ((unsigned)idx[1] << 16), (unsigned)idx[2] | ((unsigned)idx[3] << 16));
          else {
#pragma unroll
            for (unsigned u = 0; u < G; ++u) out_idx[at + u] = (uint16_t)idx[u];
          }
        }
      };
      auto advance = [&]() {
        i += STEP, j += dq, tt += dr;
        if (tt >= nt) tt -= nt, ++j;
      };
      auto classify_store = [&](unsigned at, T* v) {
        int x[G];
        bool ok = true;
#pragma unroll
        for (unsigned u = 0; u < G; ++u) {
          v[u] = substituted(v[u], log_c);
          x[u] = guess(v[u], log_c, ok);
        }
        if (!ok) {  // rare (fully unrolled: a dynamic index would push x[] / v[] into local memory)
#pragma unroll
          for (unsigned u = 0; u < G; ++u) x[u] = recount<T>(v[u], x[u], thr_col);
        }
        store4(at, x);
      };
      // full groups, two per trip: both loads are in flight before either group is classified (the kernel is
      // bound by the latency of these loads, not by issue slots: ncu long-scoreboard stall 10-12 per issue)
      while (i + STEP + (G - 1) < last) {
        T a[G], b[G];
        const unsigned ia = i;
        load4(j, tt, a);
        advance();
        const unsigned ib = i;
        load4(j, tt, b);
        advance();
        classify_store(ia, a);
        classify_store(ib, b);
      }
      while (i + (G - 1) < last) {
        T cur[G];
        load4(j, tt, cur);
        classify_store(i, cur);
        advance();
      }
      if (i < last) {  // the last, partial group of the panel (i was advanced past every full group)
        unsigned jj = j, t = tt;
        for (unsigned p = i; p < last; ++p) {
          const int n = to_count(__ldg(mat + address(jj, t)), log_c);
          if constexpr (RGBA) out_rgba[p] = lut_at(n);
          if constexpr (INDEX) out_idx[p] = (uint16_t)count_to_index(n);
          if (++t == nt) t = 0, ++jj;
        }
      }
    };
    auto by_output = [&](auto log_c, auto rowlist_c) {
      // the two configurations the batch path runs get their own instantiation with 128-bit stores; everything
      // else (index plane only, unaligned output) shares the scalar-store variants
      if (out_rgba && !out_idx && out_vec)
        pixels(log_c, rowlist_c, Flag<true>{}, Flag<false>{}, Flag<true>{});
      else if (out_rgba && out_idx && out_vec)
        pixels(log_c, rowlist_c, Flag<true>{}, Flag<true>{}, Flag<true>{});
      else if (out_rgba && out_idx)
        pixels(log_c, rowlist_c, Flag<true>{}, Flag<true>{}, Flag<false>{});
      else if (out_rgba)
        pixels(log_c, rowlist_c, Flag<true>{}, Flag<false>{}, Flag<false>{});
      else if (out_idx)
        pixels(log_c, rowlist_c, Flag<false>{}, Flag<true>{}, Flag<false>{});
    };
    if (log_scale) {
      if (rows_off < 0)
        by_output(Flag<true>{}, Flag<false>{});
      else
        by_output(Flag<true>{}, Flag<true>{});
    } else {
      if (rows_off < 0)
        by_output(Flag<false>{}, Flag<false>{});
      else
        by_output(Flag<false>{}, Flag<true>{});
    }
  }
}

}  // namespace

extern "C" {

int32_t csg_raster_blocks(int32_t ne, int32_t nt) {
  if (ne <= 0 || nt <= 0) return 0;
  return (int32_t)(((long long)ne * nt + kPixPerBlock - 1) / kPixPerBlock);
}

size_t csg_threshold_bytes(int n_panels, int dtype) {
  return (size_t)(n_panels > 0 ? n_panels : 0) * kThrPitch * (dtype == CSG_F64 ? 8 : 4);
}

int csg_panel_prepare(csg_ctx* ctx, const csg_panel* d_panels, int n_panels, const csg_region* d_regions,
                      const csg_region_stats* d_stats, int dtype, const double* d_zvals, csg_panel_norm* d_norms,
                      void* d_thresholds) {
  (void)d_regions;
  if (!ctx) return CSG_ERR_ARG;
  if (n_panels <= 0) return CSG_OK;
  if (!d_panels || !d_stats || !d_norms || !d_thresholds) return csg_fail(ctx, CSG_ERR_ARG, "NULL argument");
  const int blocks = (n_panels + 127) / 128;
  if (dtype == CSG_F32) {
    panel_prepare_kernel<float><<<blocks, 128, 0, ctx->stream>>>(d_panels, n_panels, d_stats, d_zvals, d_norms);
    CSG_LAUNCH_CHECK(ctx, "panel_prepare_kernel");
    panel_threshold_kernel<float><<<n_panels, 288, 0, ctx->stream>>>(d_panels, d_norms, n_panels, (float*)d_thresholds);
  } else if (dtype == CSG_F64) {
    panel_prepare_kernel<double><<<blocks, 128, 0, ctx->stream>>>(d_panels, n_panels, d_stats, d_zvals, d_norms);
    CSG_LAUNCH_CHECK(ctx, "panel_prepare_kernel");
    panel_threshold_kernel<double><<<n_panels, 288, 0, ctx->stream>>>(d_panels, d_norms, n_panels, (double*)d_thresholds);
  } else {
    return csg_fail(ctx, CSG_ERR_ARG, "bad dtype %d", dtype);
  }
  CSG_LAUNCH_CHECK(ctx, "panel_threshold_kernel");
  return CSG_OK;
}

int csg_rasterise(csg_ctx* ctx, const void* d_mats, int dtype, const csg_region* d_regions,
                  const int32_t* d_index_pool, const csg_panel* d_panels, const csg_panel_norm* d_norms,
                  const void* d_thresholds, int n_panels, int total_blocks, int block_offset,
                  const int32_t* d_block_panel, const uint8_t* d_lut, uint8_t* d_rgba, uint16_t* d_index) {
  if (!ctx) return CSG_ERR_ARG;
  if (n_panels <= 0 || total_blocks <= 0) return CSG_OK;
  if (!d_mats || !d_regions || !d_index_pool || !d_panels || !d_norms || !d_thresholds || !d_block_panel)
    return csg_fail(ctx, CSG_ERR_ARG, "NULL argument");
  if (d_rgba && !d_lut) return csg_fail(ctx, CSG_ERR_ARG, "d_rgba requested without d_lut");
  // persistent blocks: as many as fit the SMs at once (shared memory allows 2-3 per SM), each a contiguous chunk range
  static bool configured_dev[64] = {false};
  bool& configured = configured_dev[ctx->device & 63];
  if (!configured) {
    CSG_CUDA(ctx, cudaFuncSetAttribute(rasterise_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)raster_smem_bytes<float>()));
    CSG_CUDA(ctx, cudaFuncSetAttribute(rasterise_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)raster_smem_bytes<double>()));
    configured = true;
  }
  int per_sm = dtype == CSG_F32 ? 3 : 2;
  if (ctx->raster_blocks_per_sm > 0 && ctx->raster_blocks_per_sm < per_sm) per_sm = ctx->raster_blocks_per_sm;
  int grid = ctx->sm_count * per_sm;
  if (grid > total_blocks) grid = total_blocks;
  if (dtype == CSG_F32)
    rasterise_kernel<float><<<grid, kRasterThreads, raster_smem_bytes<float>(), ctx->stream>>>(
        (const float*)d_mats, d_regions, d_index_pool, d_panels, d_norms, block_offset, total_blocks, d_block_panel,
        (const float*)d_thresholds, (const uint32_t*)d_lut, (uint32_t*)d_rgba, d_index);
  else if (dtype == CSG_F64)
    rasterise_kernel<double><<<grid, kRasterThreads, raster_smem_bytes<double>(), ctx->stream>>>(
        (const double*)d_mats, d_regions, d_index_pool, d_panels, d_norms, block_offset, total_blocks, d_block_panel,
        (const double*)d_thresholds, (const uint32_t*)d_lut, (uint32_t*)d_rgba, d_index);
  else
    return csg_fail(ctx, CSG_ERR_ARG, "bad dtype %d", dtype);
  CSG_LAUNCH_CHECK(ctx, "rasterise_kernel");
  return CSG_OK;
}

int csg_rasterise_blocks_per_sm(csg_ctx* ctx, int blocks_per_sm) {
  if (!ctx || blocks_per_sm < 0) return CSG_ERR_ARG;
  ctx->raster_blocks_per_sm = blocks_per_sm;
  return CSG_OK;
}

}  // extern "C"
