// K4 -- figure mosaics composed and DEFLATE-encoded on the device (the PNG hand-off of the path).
//
// The reference's product is one PNG per figure (CS/fast/process_orbit.py:98-117 ->
// fig.savefig, CS/generic_batch.py:108-113); there nearly all wall time goes into Agg and zlib.
// Here the colour-mapped panels (K3) already sit in HBM, so a figure never exists as raw pixels
// anywhere: one kernel evaluates the mosaic for the scanline it encodes -- every tile is a source
// raster (a K3 panel in d_rgba, flipped to origin="lower" -- or, on a log energy axis, placed row by row
// through the host's row map; or a host-drawn annotation sprite in the
// overlay atlas) resampled nearest-neighbour into its rectangle on the canvas, the way
// imshow(aspect="auto") fills an axes box at display resolution (CS/plotting.py:280-287,606-611:
// 4800 x 2400 pixels for the FAST grids); cusp lines burnt in; background in the gaps -- the
// arithmetic of figure.SpectrogramFigure.compose -- and writes finished DEFLATE blocks:
//
//   segment   = up to 1024 pixels of one scanline = one warp = one Huffman block that ends
//               with an empty stored block (the zlib "sync flush": byte aligned, so segments
//               concatenate bytewise into a valid stream in any quantity)
//   rows      = only scanlines with NEW content are encoded: the host lists them per canvas from the
//               geometry alone (a resampled panel repeats every raster row several times; gaps
//               repeat the background).  They take filter 2 ("Up") like every other line: what a
//               listed line shares with the one above -- often all but one sprite or one step of a
//               colour bar -- turns into zeros.  Runs of repeated lines are Up lines of nothing but
//               zeros, a constant the host splices in between the segments (png.py)
//   tokens    = per pixel: equal to its left neighbour -> it extends a distance-4 match; else equal
//               to one of the 128 pixels before it -> a match at that distance (extended while the
//               following pixels keep matching); else four literals.
//   lanes     = 32 pixels each, encoded into private bit buffers; a warp prefix sum over the bit
//               counts places them in the segment's stream (shared-memory atomicOr)
//   adler32   = per segment (sum, weighted sum) of the filtered bytes, combined in order on the host
//
// The host adds the 2-byte zlib header, the final empty block, the Adler-32 and the PNG chunk
// framing (png.py).  A decoder sees an ordinary 8-bit RGBA, non-interlaced PNG.
#include <string.h>

#include "common.cuh"

namespace {

constexpr int kSegPixels = 1024;
constexpr int kMatchWindow = 128;    // pixels a match may reach back (distance <= 512 bytes)
constexpr int kShortWindow = 8;      // ... while the lane's recent pixels found nothing (noise: see the tokeniser)
constexpr int kPieces = 32;          // lanes
constexpr int kPiecePixels = 32;     // pixels per lane
constexpr int kPixStride = 33;       // padded piece stride (words): conflict-free column reads
constexpr int kTokWords = 37;        // per-lane token buffer: 32 pixels x 36 bits + header / trailer bits
constexpr int kHeaderWords = 40;     // block header (BFINAL/BTYPE + a dynamic block's code lengths): <= 160 bytes
constexpr int kMergedWords = kPieces * kTokWords + kHeaderWords + 4;
#ifndef CSG_K4_WARPS
#define CSG_K4_WARPS 1
#endif
// One warp = one segment = one block: segments differ a lot in work (a dismissed one ends at once, a line of new
// spectrogram cells takes the full tokeniser), and a block lives as long as its slowest warp.  Measured on 320
// figures of 4800x2400: 115.6 / 96.8 / 85.5 ms with 4 / 2 / 1 warps per block (achieved occupancy was 13.7 % of a
// theoretical 25 % with 4).
constexpr int kWarpsPerBlock = CSG_K4_WARPS;
constexpr int kTileRowMap = 4;       // csg_png_tile.flags: rows come from d_row_maps (TILE_ROW_MAP in csgpu.h)

// The code tables of one batch of figures (csg_png_tables in csgpu.h): either RFC 1951's fixed codes
// or a custom (dynamic-block) code built by the host from the batch's own symbol counts.  Codes are
// stored bit-reversed, ready to be OR-ed into the LSB-first stream; match entries hold the Huffman
// code followed by the extra bits.  Literal / length codes are limited to 9 bits, so a pixel never
// costs more than with the fixed code and the buffer sizes below hold for both.
typedef csg_png_tables HuffTables;
__constant__ HuffTables c_huff;

__device__ __forceinline__ unsigned sub4(unsigned a, unsigned b) { return __vsub4(a, b); }

// A tile as one segment sees it: the columns it covers on this scanline and the source row they read.
struct SegTile {
  const uint32_t* row;          // first pixel of the source row this scanline shows
  float xs;                     // source columns per canvas pixel
  int vline_first;
  int nt_minus_1;               // last source column (the nearest-neighbour index is clamped to it)
  unsigned short x0, x1;        // canvas columns [x0, x1) inside the segment's range (canvases are < 65536 wide)
  unsigned short tx;            // the tile's left edge on the canvas
  unsigned short vline_count;
  int pad;
};                              // 32 bytes
constexpr int kSegTiles = 48;   // tiles one 1024-pixel segment may intersect on one scanline (the device flags more)
// dynamic shared memory of png_encode_kernel: symbol counts | pixels / merged stream | lane token buffers | tile lists
constexpr size_t kOffPix = (size_t)kWarpsPerBlock * (286 + 30) * sizeof(unsigned);
constexpr size_t kOffTok = kOffPix + (size_t)kWarpsPerBlock * kMergedWords * sizeof(unsigned);
constexpr size_t kOffSeg = (kOffTok + (size_t)kWarpsPerBlock * kPieces * kTokWords * sizeof(unsigned) + 15) / 16 * 16;
constexpr size_t kEncodeSmem = kOffSeg + (size_t)kWarpsPerBlock * 2 * kSegTiles * sizeof(SegTile);
static_assert(sizeof(SegTile) == 32, "SegTile layout");

// source index of destination pixel d (0-based) of `n_dst`, nearest neighbour, pixel centres:
// floor((d + 0.5) * n_src / n_dst) in float32 -- figure.py evaluates the same float32 expression
__device__ __forceinline__ int nearest(int d, float scale, int last) {
  const int k = (int)(__fmul_rn(__fadd_rn((float)d, 0.5f), scale));
  return k > last ? last : k;
}

// One pixel of a figure's mosaic: the first listed tile that covers column x, else the background.
__device__ __forceinline__ unsigned mosaic_pixel(const SegTile* __restrict__ list, int n_list,
                                                 const csg_png_vline* __restrict__ vlines, int x, unsigned background) {
  for (int k = 0; k < n_list; ++k) {
    const SegTile& t = list[k];
    if (x < (int)t.x0 || x >= (int)t.x1) continue;
    const int dx = x - (int)t.tx;
    unsigned px = __ldg(t.row + nearest(dx, t.xs, t.nt_minus_1));
    for (int v = 0; v < (int)t.vline_count; ++v) {  // later lines overwrite earlier ones
      const csg_png_vline ln = vlines[t.vline_first + v];
      if (dx >= ln.col - ln.half && dx <= ln.col + ln.half) px = ln.rgba;
    }
    return px;
  }
  return background;
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
    png_encode_kernel(const uint32_t* __restrict__ rgba, const uint32_t* __restrict__ overlay,
                      const csg_png_canvas* __restrict__ canvases, int n_canvases, const csg_png_tile* __restrict__ tiles,
                      const csg_png_vline* __restrict__ vlines, const int32_t* __restrict__ rows, int n_segments,
                      unsigned char* __restrict__ slots, int slot_bytes, int32_t* __restrict__ sizes,
                      uint32_t* __restrict__ adler, unsigned* __restrict__ counts, int count_stride, int* __restrict__ error,
                      const csg_png_zero_segment* __restrict__ zero_table, int n_zero, const int32_t* __restrict__ row_maps) {
  // counts != NULL: no output, only the symbol statistics of every count_stride-th segment
  // (literal / length symbols 0..285, then distance symbols 0..29) for the host's custom code
  extern __shared__ __align__(16) unsigned char s_dyn[];
  unsigned(*s_counts)[286 + 30] = reinterpret_cast<unsigned(*)[286 + 30]>(s_dyn);
  unsigned(*s_pix)[kMergedWords] = reinterpret_cast<unsigned(*)[kMergedWords]>(s_dyn + kOffPix);
  unsigned(*s_tok)[kPieces * kTokWords] = reinterpret_cast<unsigned(*)[kPieces * kTokWords]>(s_dyn + kOffTok);
  SegTile(*s_seg)[2 * kSegTiles] = reinterpret_cast<SegTile(*)[2 * kSegTiles]>(s_dyn + kOffSeg);
  if (counts) {
    for (int i = threadIdx.x; i < kWarpsPerBlock * (286 + 30); i += blockDim.x) (&s_counts[0][0])[i] = 0;
    __syncthreads();
  }
  // s_pix: filtered pixels (padded pieces), then the merged stream; s_seg: the tile lists of this scanline and the one above
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int seg = (blockIdx.x * kWarpsPerBlock + warp) * (counts ? count_stride : 1);
  const bool active = seg < n_segments;
  if (!active && !counts) return;
  if (active) {
  // ---- which canvas / scanline / chunk
  int lo = 0, hi = n_canvases - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&canvases[mid].seg_first) <= seg)
      lo = mid;
    else
      hi = mid - 1;
  }
  const csg_png_canvas cv = canvases[lo];
  const int local = seg - cv.seg_first;
  const int k_row = local / cv.segs_per_row, chunk = local - k_row * cv.segs_per_row;
  const int row = __ldg(rows + cv.row_first + k_row);  // the k-th scanline of this canvas that has new content
  const int x0 = chunk * kSegPixels;
  const int npx = min(kSegPixels, cv.W - x0);
  const bool has_filter = chunk == 0;
  const int n_raw = (has_filter ? 1 : 0) + 4 * npx;  // filtered bytes this segment feeds to DEFLATE
  // Up filter on every listed scanline but the first of the canvas: what a listed line shares with the line
  // above (it may differ from it in one text sprite or one step of a colour bar only) becomes zeros
  const unsigned filter_type = row > 0 ? 2u : 0u;
  // ---- the tiles crossing this scanline (and the one above) inside [x0, x0 + npx), in table order (first match wins)
  SegTile* list = s_seg[warp];
  SegTile* list_up = s_seg[warp] + kSegTiles;
  int n_list = 0, n_up = 0;
  for (int which = 0; which < (row > 0 ? 2 : 1); ++which) {
    const int r = row - which;
    SegTile* dst = which ? list_up : list;
    int n = 0;
    for (int base = 0; base < cv.tile_count; base += 32) {
      const int ti = base + lane;
      bool hit = false;
      csg_png_tile t;
      if (ti < cv.tile_count) {
        t = tiles[cv.tile_first + ti];
        hit = t.w > 0 && t.h > 0 && r >= t.y && r < t.y + t.h && t.x < x0 + npx && t.x + t.w > x0;
      }
      const unsigned m = __ballot_sync(0xffffffffu, hit);
      if (hit) {
        const int at = n + __popc(m & ((1u << lane) - 1u));
        if (at < kSegTiles) {
          int src_row;
          if (t.flags & kTileRowMap) {  // a panel on a log energy axis: the host lists the storage row of every canvas row
            int k = 0;
            if (row_maps)
              k = __ldg(row_maps + t.row_map + (r - t.y));
            else if (error)
              atomicExch(error, -(1 + lo));  // the host raises: the tile's map table is missing
            src_row = min(max(k, 0), t.ne - 1);
          } else {
            const int r_top = nearest(r - t.y, __fdiv_rn((float)t.ne, (float)t.h), t.ne - 1);  // source row, counted from the top
            src_row = (t.flags & 2) ? r_top : t.ne - 1 - r_top;  // rasters store the lowest energy first
          }
          SegTile e;
          e.x0 = (unsigned short)max(t.x, x0), e.x1 = (unsigned short)min(t.x + t.w, x0 + npx);
          e.tx = (unsigned short)t.x, e.nt_minus_1 = t.nt - 1;
          e.xs = __fdiv_rn((float)t.nt, (float)t.w);
          e.vline_first = t.vline_first, e.vline_count = (unsigned short)t.vline_count, e.pad = 0;
          e.row = ((t.flags & 1) ? overlay : rgba) + t.rgba_off + (long long)src_row * t.nt;
          dst[at] = e;
        }
      }
      n += __popc(m);
    }
    if (n > kSegTiles) {
      if (lane == 0 && error) atomicExch(error, 1 + lo);  // the host raises: too many tiles meet in one segment
      n = kSegTiles;
    }
    if (which) n_up = n; else n_list = n;
  }
  __syncwarp();
  // ---- where can this scanline differ from the one above?  When both cross the same tiles in the same order,
  // a pixel's winner is the same tile on both lines and only a tile whose SOURCE row moved on can change it:
  // everything outside those tiles' columns is zero after the Up filter and is never evaluated (a colour bar
  // stepping to its next colour dirties 60 of 4800 pixels; a segment it does not touch is dismissed here).
  int dirty0 = x0, dirty1 = x0 + npx;
  if (row > 0 && n_list == n_up) {
    bool structural = false;
    int d0 = 0x7fffffff, d1 = -1;
    for (int i = lane; i < n_list; i += 32) {
      const SegTile a = list[i], b = list_up[i];
      if (a.tx != b.tx || a.x0 != b.x0 || a.x1 != b.x1 || a.xs != b.xs || a.nt_minus_1 != b.nt_minus_1 ||
          a.vline_first != b.vline_first || a.vline_count != b.vline_count)
        structural = true;  // another tile: the line starts or ends something
      else if (a.row != b.row)
        d0 = min(d0, (int)a.x0), d1 = max(d1, (int)a.x1);
    }
    structural = __any_sync(0xffffffffu, structural);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      d0 = min(d0, __shfl_xor_sync(0xffffffffu, d0, o));
      d1 = max(d1, __shfl_xor_sync(0xffffffffu, d1, o));
    }
    if (!structural) dirty0 = d0, dirty1 = d1;  // empty when d1 < d0
  }

  // ---- phase 1: compose + Up filter (coalesced), Adler partial sums
  unsigned* pix = s_pix[warp];
  unsigned long long sa = 0, sb = 0;
  unsigned nonzero = 0;
  for (int p = lane; p < npx; p += 32) {
    const int x = x0 + p;
    if (x < dirty0 || x >= dirty1) {  // same winner, same source row as above
      pix[(p >> 5) * kPixStride + (p & 31)] = 0u;
      continue;
    }
    const unsigned cur = mosaic_pixel(list, n_list, vlines, x, cv.background);
    const unsigned f = filter_type ? sub4(cur, mosaic_pixel(list_up, n_up, vlines, x, cv.background)) : cur;
    pix[(p >> 5) * kPixStride + (p & 31)] = f;
    nonzero |= f;
    const unsigned b0 = f & 255u, b1 = (f >> 8) & 255u, b2 = (f >> 16) & 255u, b3 = f >> 24;
    const unsigned t0 = (has_filter ? 1u : 0u) + 4u * (unsigned)p;  // position of b0 inside the segment
    sa += b0 + b1 + b2 + b3;
    sb += (unsigned long long)(n_raw - t0) * b0 + (unsigned long long)(n_raw - t0 - 1) * b1 +
          (unsigned long long)(n_raw - t0 - 2) * b2 + (unsigned long long)(n_raw - t0 - 3) * b3;
  }
  if (lane == 0 && has_filter) sa += filter_type, sb += (unsigned long long)filter_type * (unsigned long long)n_raw;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sa += __shfl_xor_sync(0xffffffffu, sa, o);
    sb += __shfl_xor_sync(0xffffffffu, sb, o);
  }
  __syncwarp();
  // A segment that only repeats the line above -- all zeros after the Up filter: most segments of a scanline
  // on which just one colour bar or one label moved on -- is a constant of its length: the host supplies it
  // ready made (zlib's encoding of the zeros, byte aligned like every segment) and no token is formed.
  const csg_png_zero_segment* canned = nullptr;
  if (filter_type == 2u && !__any_sync(0xffffffffu, nonzero != 0u))
    for (int z = 0; z < n_zero; ++z)
      if (zero_table[z].n_raw == n_raw) canned = zero_table + z;
  const int npx_tok = canned ? 0 : npx;  // pixels that go through the tokeniser

  // ---- phase 2: every lane turns its 32 pixels into tokens in a private bit buffer
  unsigned* tok = s_tok[warp] + lane * kTokWords;
  unsigned long long acc = 0;
  int nacc = 0, nwords = 0;
  auto put = [&](unsigned long long bits, int n) {  // n <= 32
    acc |= bits << nacc;
    nacc += n;
    if (nacc >= 32) {
      tok[nwords++] = (unsigned)acc;
      acc >>= 32;
      nacc -= 32;
    }
  };
  unsigned* cnt = counts ? s_counts[warp] : nullptr;
  // (the block header -- BFINAL / BTYPE and, for a custom code, its code lengths -- is the same bit
  // string for every segment: it is copied in front of the lanes' bits in the merge phase)
  if (lane == 0 && has_filter && !canned) {
    if (cnt) atomicAdd(&cnt[filter_type], 1u);
    put(c_huff.lit_code[filter_type], c_huff.lit_len[filter_type]);
  }
  const int p_begin = lane * kPiecePixels, p_end = min(npx_tok, p_begin + kPiecePixels);
  if (p_begin < npx_tok) {
    // pixel q of the segment (any lane's piece): matches may reach back into earlier pieces
    static_assert(kPixStride == 33 && kPiecePixels == 32, "at(): q + (q >> 5) is the padded index");
    auto at = [&](int q) { return pix[q + (q >> 5)]; };
    int run = 0, dist = 0;  // an open match of `run` pixels at distance `dist` pixels
    // The backward search was 62 % of this kernel's instructions (ncu, profiles/r2_ncu_full_png.txt): a pixel
    // of a line with new content (the difference of two neighbouring spectrogram rows) usually has no equal
    // within reach and pays for all 128 probes.  After two misses in a row the lane only looks 8 pixels
    // back until something matches again: noise costs 16x less, structure keeps the full window.
    int misses = 0;
    auto flush = [&]() {
      if (run) {
        if (cnt) {
          atomicAdd(&cnt[c_huff.len_sym[run]], 1u);
          atomicAdd(&cnt[286 + c_huff.dist_sym[dist]], 1u);
        }
        put(c_huff.len_code[run], c_huff.len_len[run]);   // <= 14 bits
        put(c_huff.dist_code[dist], c_huff.dist_len[dist]);  // <= 14 bits
        run = 0;
      }
    };
    for (int p = p_begin; p < p_end; ++p) {
      const unsigned x = at(p);
      if (run && x == at(p - dist)) {  // the open match goes on (run <= 32 pixels = 128 bytes)
        ++run;
        continue;
      }
      flush();
      int k = 0;
      const int reach = min(p, misses >= 2 ? kShortWindow : kMatchWindow);
      for (int d = 1; d <= reach; ++d)
        if (at(p - d) == x) {
          k = d;
          break;
        }
      if (k) {
        run = 1, dist = k, misses = 0;
        continue;
      }
      ++misses;
      const unsigned b0 = x & 255u, b1 = (x >> 8) & 255u, b2 = (x >> 16) & 255u, b3 = x >> 24;
      if (cnt) {
        atomicAdd(&cnt[b0], 1u);
        atomicAdd(&cnt[b1], 1u);
        atomicAdd(&cnt[b2], 1u);
        atomicAdd(&cnt[b3], 1u);
      }
      // two puts of <= 18 bits: the 64-bit accumulator holds < 32 pending bits
      put(c_huff.lit_code[b0] | ((unsigned)c_huff.lit_code[b1] << c_huff.lit_len[b0]), c_huff.lit_len[b0] + c_huff.lit_len[b1]);
      put(c_huff.lit_code[b2] | ((unsigned)c_huff.lit_code[b3] << c_huff.lit_len[b2]), c_huff.lit_len[b2] + c_huff.lit_len[b3]);
    }
    flush();
  }
  const bool last_lane = p_begin < npx_tok && p_end == npx_tok;
  if (last_lane) {
    if (cnt) atomicAdd(&cnt[256], 1u);
    put(c_huff.eob_code, c_huff.eob_len + 3);  // end-of-block, then the header of the empty stored block (000)
  }
  if (nacc) tok[nwords] = (unsigned)acc;
  const int my_bits = nwords * 32 + nacc;

  // ---- phase 3: place the lanes' bit strings one after the other
  int incl = my_bits;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int hdr_bits = c_huff.header_bits;
  const int total_bits = hdr_bits + __shfl_sync(0xffffffffu, incl, 31);
  const int off = hdr_bits + incl - my_bits;
  if (!counts && canned) {
    unsigned char* dst = slots + (size_t)seg * slot_bytes;
    for (int i = lane; i < canned->len; i += 32) dst[i] = canned->bytes[i];
    if (lane == 0) {
      sizes[seg] = canned->len;
      adler[2 * seg] = (unsigned)(sa % 65521ull);
      adler[2 * seg + 1] = (unsigned)(sb % 65521ull);
    }
  } else if (!counts) {
  __syncwarp();  // every lane is done reading pixels: the buffer becomes the merged stream
  unsigned* out = s_pix[warp];
  const int total_bytes = (total_bits + 7) / 8 + 4;  // pad to a byte, then LEN = 0000, NLEN = FFFF
  const int total_words = (total_bytes + 3) / 4;
  // the block header first (same bits for every segment), zeros behind it
  const int hdr_words = (hdr_bits + 31) / 32;
  for (int w = lane; w < total_words; w += 32) out[w] = w < hdr_words ? c_huff.header[w] : 0u;
  __syncwarp();
  const int my_words = (my_bits + 31) / 32;
  const int w0 = off >> 5, sh = off & 31;
  for (int k = 0; k < my_words; ++k) {
    const unsigned v = tok[k];
    atomicOr(&out[w0 + k], v << sh);
    if (sh) atomicOr(&out[w0 + k + 1], v >> (32 - sh));
  }
  __syncwarp();
  if (lane == 0) {  // NLEN = 0xFFFF after the (zero) LEN
    const int at = (total_bits + 7) / 8 + 2;
    atomicOr(&out[at >> 2], 0xffu << (8 * (at & 3)));
    atomicOr(&out[(at + 1) >> 2], 0xffu << (8 * ((at + 1) & 3)));
  }
  __syncwarp();
  unsigned* dst = reinterpret_cast<unsigned*>(slots + (size_t)seg * slot_bytes);
  for (int w = lane; w < total_words; w += 32) dst[w] = out[w];
  if (lane == 0) {
    sizes[seg] = total_bytes;
    adler[2 * seg] = (unsigned)(sa % 65521ull);
    adler[2 * seg + 1] = (unsigned)(sb % 65521ull);
  }
  }  // output mode
  }  // active
  if (counts) {
    __syncthreads();
    for (int i = threadIdx.x; i < 286 + 30; i += blockDim.x) {
      unsigned n = 0;
      for (int w = 0; w < kWarpsPerBlock; ++w) n += s_counts[w][i];
      if (n) atomicAdd(&counts[i], n);
    }
  }
}

// warp per segment: slot -> its place in the packed stream
__global__ void __launch_bounds__(256)
    png_compact_kernel(const unsigned char* __restrict__ slots, int slot_bytes, const int32_t* __restrict__ sizes,
                       const long long* __restrict__ offsets, int n_segments, unsigned char* __restrict__ packed) {
  const int seg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (seg >= n_segments) return;
  const unsigned char* src = slots + (size_t)seg * slot_bytes;
  unsigned char* dst = packed + offsets[seg];
  const int n = sizes[seg];
  for (int i = lane; i < n; i += 32) dst[i] = src[i];
}

unsigned reverse_bits(unsigned v, int n) {
  unsigned r = 0;
  for (int i = 0; i < n; ++i) r |= ((v >> i) & 1u) << (n - 1 - i);
  return r;
}

void build_fixed_tables(HuffTables* t) {
  memset(t, 0, sizeof(*t));
  for (int v = 0; v < 256; ++v) {
    if (v < 144) {
      t->lit_code[v] = (unsigned short)reverse_bits(0x30u + v, 8);
      t->lit_len[v] = 8;
    } else {
      t->lit_code[v] = (unsigned short)reverse_bits(0x190u + (v - 144), 9);
      t->lit_len[v] = 9;
    }
  }
  // RFC 1951 3.2.5: length codes 257..285 (base length, extra bits)
  static const int base[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
  static const int extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
  for (int n = 1; n <= 64; ++n) {
    const int len = 4 * n;
    int c = 28;
    while (c > 0 && base[c] > len) --c;
    const int sym = 257 + c;
    unsigned bits;
    int nb;
    if (sym < 280) {
      bits = reverse_bits((unsigned)(sym - 256), 7);
      nb = 7;
    } else {
      bits = reverse_bits(0xC0u + (unsigned)(sym - 280), 8);
      nb = 8;
    }
    bits |= (unsigned)(len - base[c]) << nb;  // extra bits: plain binary, LSB first
    nb += extra[c];
    t->len_code[n] = bits;
    t->len_len[n] = (unsigned char)nb;
    t->len_sym[n] = (unsigned short)sym;
  }
  // RFC 1951 3.2.5: distance codes 0..29 (base distance, extra bits); fixed code = 5 bits, reversed
  static const int dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
  static const int dextra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
  for (int k = 1; k <= kMatchWindow; ++k) {
    const int d = 4 * k;
    int c = 29;
    while (c > 0 && dbase[c] > d) --c;
    unsigned bits = reverse_bits((unsigned)c, 5);
    bits |= (unsigned)(d - dbase[c]) << 5;
    t->dist_code[k] = bits;
    t->dist_len[k] = (unsigned char)(5 + dextra[c]);
    t->dist_sym[k] = (unsigned char)c;
  }
  t->eob_code = 0, t->eob_len = 7;
  t->header[0] = 2u, t->header_bits = 3;  // BFINAL = 0, BTYPE = 01 (fixed Huffman)
}

bool g_tables_ready[64] = {false};
bool ctx_tables_ready(csg_ctx* ctx) { return g_tables_ready[ctx->device & 63]; }
void ctx_tables_set(csg_ctx* ctx) { g_tables_ready[ctx->device & 63] = true; }

}  // namespace

extern "C" {

int32_t csg_png_slot_bytes(void) {
  // 3 header bits + filter literal + 1024 pixels x 36 bits + EOB + stored header, padded, + LEN/NLEN, word rounded
  return (int32_t)(((kHeaderWords * 32 + 9 + kSegPixels * 36 + 15 + 3 + 7) / 8 + 4 + 15) / 16 * 16);
}

int32_t csg_png_segments(int32_t W, int32_t n_rows) {
  if (W <= 0 || n_rows <= 0) return 0;
  return (int32_t)(((long long)(W + kSegPixels - 1) / kSegPixels) * n_rows);
}

int32_t csg_png_max_segment_tiles(void) { return kSegTiles; }

int csg_png_fixed_tables(csg_png_tables* out) {
  if (!out) return CSG_ERR_ARG;
  build_fixed_tables(out);
  return CSG_OK;
}

int csg_png_set_tables(csg_ctx* ctx, const csg_png_tables* tables) {
  if (!ctx) return CSG_ERR_ARG;
  HuffTables h;
  if (tables)
    h = *tables;
  else
    build_fixed_tables(&h);
  if (h.header_bits < 3 || h.header_bits > kHeaderWords * 32 || h.eob_len < 1 || h.eob_len > 15)
    return csg_fail(ctx, CSG_ERR_ARG, "bad PNG code tables (header %d bits, end-of-block %d bits)", h.header_bits, (int)h.eob_len);
  for (int v = 0; v < 256; ++v)
    if (h.lit_len[v] < 1 || h.lit_len[v] > 9) return csg_fail(ctx, CSG_ERR_ARG, "literal %d has a %d-bit code (1..9 allowed)", v, (int)h.lit_len[v]);
  // stream-ordered: segments already enqueued keep the tables they were launched with
  CSG_CUDA(ctx, cudaMemcpyToSymbolAsync(c_huff, &h, sizeof(h), 0, cudaMemcpyHostToDevice, ctx->stream));
  CSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // `h` lives on this stack frame
  ctx_tables_set(ctx);
  return CSG_OK;
}

static int png_launch(csg_ctx* ctx, const uint8_t* d_rgba, const uint8_t* d_overlay, const csg_png_canvas* d_canvases,
                      int n_canvases, const csg_png_tile* d_tiles, const csg_png_vline* d_vlines, const int32_t* d_rows,
                      int n_segments, uint8_t* d_slots, int32_t* d_sizes, uint32_t* d_adler, uint32_t* d_counts,
                      int count_stride, int32_t* d_error, const csg_png_zero_segment* d_zero, int n_zero,
                      const int32_t* d_row_maps) {
  if (!ctx_tables_ready(ctx)) {
    const int st = csg_png_set_tables(ctx, nullptr);
    if (st != CSG_OK) return st;
  }
  const int work = d_counts ? (n_segments + count_stride - 1) / count_stride : n_segments;
  const int blocks = (work + kWarpsPerBlock - 1) / kWarpsPerBlock;
  static bool configured_dev[64] = {false};
  if (!configured_dev[ctx->device & 63]) {
    CSG_CUDA(ctx, cudaFuncSetAttribute(png_encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEncodeSmem));
    configured_dev[ctx->device & 63] = true;
  }
  png_encode_kernel<<<blocks, kWarpsPerBlock * 32, kEncodeSmem, ctx->stream>>>(
      (const uint32_t*)d_rgba, (const uint32_t*)d_overlay, d_canvases, n_canvases, d_tiles, d_vlines, d_rows, n_segments, d_slots,
      csg_png_slot_bytes(), d_sizes, d_adler, d_counts, count_stride, d_error, d_zero, d_zero ? n_zero : 0, d_row_maps);
  CSG_LAUNCH_CHECK(ctx, "png_encode_kernel");
  return CSG_OK;
}

int csg_png_encode(csg_ctx* ctx, const uint8_t* d_rgba, const uint8_t* d_overlay, const csg_png_canvas* d_canvases,
                   int n_canvases, const csg_png_tile* d_tiles, const csg_png_vline* d_vlines, const int32_t* d_rows,
                   int n_segments, uint8_t* d_slots, int32_t* d_sizes, uint32_t* d_adler, int32_t* d_error,
                   const csg_png_zero_segment* d_zero, int n_zero, const int32_t* d_row_maps) {
  if (!ctx) return CSG_ERR_ARG;
  if (n_canvases <= 0 || n_segments <= 0) return CSG_OK;
  if (!d_rgba || !d_canvases || !d_tiles || !d_rows || !d_slots || !d_sizes || !d_adler)
    return csg_fail(ctx, CSG_ERR_ARG, "NULL argument");
  return png_launch(ctx, d_rgba, d_overlay, d_canvases, n_canvases, d_tiles, d_vlines, d_rows, n_segments, d_slots, d_sizes,
                    d_adler, nullptr, 1, d_error, d_zero, n_zero, d_row_maps);
}

int csg_png_count(csg_ctx* ctx, const uint8_t* d_rgba, const uint8_t* d_overlay, const csg_png_canvas* d_canvases,
                  int n_canvases, const csg_png_tile* d_tiles, const csg_png_vline* d_vlines, const int32_t* d_rows,
                  int n_segments, int stride, uint32_t* d_counts, const csg_png_zero_segment* d_zero, int n_zero,
                  const int32_t* d_row_maps) {
  if (!ctx) return CSG_ERR_ARG;
  if (n_canvases <= 0 || n_segments <= 0) return CSG_OK;
  if (!d_rgba || !d_canvases || !d_tiles || !d_rows || !d_counts || stride < 1) return csg_fail(ctx, CSG_ERR_ARG, "bad argument");
  return png_launch(ctx, d_rgba, d_overlay, d_canvases, n_canvases, d_tiles, d_vlines, d_rows, n_segments, nullptr, nullptr,
                    nullptr, d_counts, stride, nullptr, d_zero, n_zero, d_row_maps);
}

int csg_png_compact(csg_ctx* ctx, const uint8_t* d_slots, const int32_t* d_sizes, const int64_t* d_offsets, int n_segments,
                    uint8_t* d_packed) {
  if (!ctx) return CSG_ERR_ARG;
  if (n_segments <= 0) return CSG_OK;
  if (!d_slots || !d_sizes || !d_offsets || !d_packed) return csg_fail(ctx, CSG_ERR_ARG, "NULL argument");
  const long long threads = (long long)n_segments * 32;
  png_compact_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>(d_slots, csg_png_slot_bytes(), d_sizes,
                                                                                 (const long long*)d_offsets, n_segments,
                                                                                 d_packed);
  CSG_LAUNCH_CHECK(ctx, "png_compact_kernel");
  return CSG_OK;
}

}  // extern "C"
