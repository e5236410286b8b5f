// K1 -- masked pitch-angle-range segmented reduction.
//
// Replaces np.nansum(cube, axis=1) (CS/constants.py:12; call sites CS/plotting.py:188,
// CS/fast/plotting.py:128,278, CS/fast/extrema.py:259) plus the pitch-angle gather
// (CS/fast/plotting.py:121-127) and the zoom "any non-NaN" probe (CS/plotting.py:597-603):
// one pass over the cube emits the unmasked sum, every pitch-angle group sum and the
// per-time-row non-NaN flags.  HBM-bound: T*P*E*s bytes in, (G+1)*T*E*s out.
//
// Output layout is ENERGY-MAJOR: sums[file][g][e][t] with row pitch Tp = T rounded up to a
// multiple of 4 -- the orientation of matrix_plot = collapsed.T (CS/plotting.py:236) that
// imshow draws, so K2a / K2b / K3 stream contiguous time runs and the rasteriser needs no
// transpose.
//
// Summation order is numpy's, bit for bit (SURVEY.md Appendix B):
//   layout TPE : ascending-p chain seeded with +0.0, NaN -> +0.0
//   layout TEP : (total) 8-accumulator pairwise over the contiguous pitch axis, then "+0.0";
//                (groups) the gather copies to C order, so the ascending-p chain again.
//
// Kernels
//   collapse_stream_kernel (TPE, the FAST shapes) block = 16 time rows x all energy chunks; the pitch
//       axis is walked in host-built runs of constant group membership with a loop body
//       specialised per membership mask.  Blocks of up to 384 threads (E = 96 float32 / 48 float64,
//       the FAST tables) take the PIPE body: every thread keeps a two-stage cp.async pipeline
//       of its own 16-byte chunks (8 pitch bins per stage) in shared memory, so loads stay in
//       flight while the previous bins are summed (6.7 TB/s).  Larger blocks, whose load slots
//       would not leave room for two blocks per SM, take the register-staged body with eight
//       128-bit streaming loads per batch (5.7 TB/s on the same shapes).  The transposed 16-row tile
//       leaves through shared memory as 64-byte row segments.  The tile loads are per-thread
//       cp.async (LDGSTS), not TMA: every thread consumes exactly the bytes it requested, so there
//       is no block-wide tile to hand around and no mbarrier to wait on; the kernel sits at the
//       measured copy bandwidth with 99.8 % useful DRAM traffic (profiles/r1_k1_traffic.json), so a
//       bulk-tensor variant has nothing left to win here and none is kept in the tree.
//   collapse_tpe_kernel      (TPE, any shape/alignment) register-staged generic path.
//   collapse_tep_rows_kernel (stored (T,E,P) view, no groups, 8 <= P <= 128, P % 8 == 0) two lanes
//       per (t,e) row own numpy's eight pairwise accumulators; P/8 vector loads in flight.
//   collapse_tep_kernel      (stored (T,E,P) view, general) rows staged in shared memory.
//   collapse_int_stream_kernel / collapse_int_tpe_kernel / collapse_int_tep_kernel: the same three
//       roles for integer cubes (CSG_I8 .. CSG_U32), read at their stored width into integer
//       accumulators, float64 sums out (see the section "Integer cubes" below).
#include <string.h>

#include <vector>

#include "common.cuh"

namespace {

constexpr int kBlock = 256;

template <typename T>
struct VecOf;
template <>
struct VecOf<float> {
  static constexpr int N = 4;
};
template <>
struct VecOf<double> {
  static constexpr int N = 2;
};

template <typename T, int VEC>
struct Chunk {
  T v[VEC];
};

__device__ __forceinline__ void load_chunk(Chunk<float, 4>& c, const float* p, bool aligned, int valid) {
  if (aligned) {
    float4 r = ld_stream4(p);
    c.v[0] = r.x, c.v[1] = r.y, c.v[2] = r.z, c.v[3] = r.w;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) c.v[i] = i < valid ? ld_stream1(p + i) : CUDART_NAN_F;  // padding lanes: ignored like NaN
  }
}
__device__ __forceinline__ void load_chunk(Chunk<double, 2>& c, const double* p, bool aligned, int valid) {
  if (aligned) {
    double2 r = ld_stream2(p);
    c.v[0] = r.x, c.v[1] = r.y;
  } else {
    c.v[0] = ld_stream1(p);
    c.v[1] = valid > 1 ? ld_stream1(p + 1) : CUDART_NAN;
  }
}

__device__ __forceinline__ int find_file(const csg_file_desc* files, int n_files, int block) {
  int lo = 0, hi = n_files - 1;
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if (__ldg(&files[mid].first_block) <= block)
      lo = mid;
    else
      hi = mid - 1;
  }
  return lo;
}

__device__ __forceinline__ int pitch_of(int T) { return (T + 3) & ~3; }

__device__ __forceinline__ void or_flag_byte(uint8_t* dst, unsigned fl) {
  // byte-wide OR through the containing aligned word
  const uintptr_t a = reinterpret_cast<uintptr_t>(dst);
  atomicOr(reinterpret_cast<unsigned*>(a & ~uintptr_t(3)), (fl & 0xffu) << (8 * (a & 3)));
}

// ---------------------------------------------------------------------------------
// stream kernel (TPE, the FAST shapes): block = 16 consecutive time rows x every energy chunk,
// thread = (time row, VEC consecutive energies), all lanes busy.  The pitch axis is walked in
// RUNS of constant group membership (host-built table: a handful per file) with a loop body
// specialised per membership mask -- no per-bin predicate work, only the adds a bin needs --
// eight 128-bit streaming loads in flight per thread.  Groups that contain every pitch bin are
// not summed at all: they equal the unmasked total (same elements, same order) and are copied.
// The transposed 16-row tile is staged in shared memory and leaves as 64-byte row segments.
// ---------------------------------------------------------------------------------
constexpr int kTileRows = 16;
constexpr int kOutPitch = kTileRows + 1;

// Two-stage cp.async pipeline private to a thread: the 16-byte chunks of pitch bins 8b .. 8b+7
// land in the thread's own shared-memory slots (slot s of thread t at (s * TPB + t) * 16 bytes:
// consecutive lanes, conflict-free) while the bins of batch b-1 are being summed.  Loads stay in
// flight during the arithmetic and cost no registers while they wait -- the register-staged
// variant below alternates "eight loads" and "a few hundred adds" and leaves the memory system
// idle during the adds (5.7 TB/s against 7.5 TB/s for the same access pattern without arithmetic).
template <typename T, int TPB>
struct Pipe {
  unsigned base;  // shared-window address of this thread's slot 0
  const T* ptr;
  long long E;
  int P;
  __device__ __forceinline__ void issue(int b) const {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int p = 8 * b + u;
      if (p < P)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(base + (unsigned)(((p & 15) * TPB) * 16)),
                     "l"(ptr + (long long)p * E)
                     : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  __device__ __forceinline__ void start() const {
    issue(0);
    issue(1);
  }
  // called before bin p is read: at a batch boundary, refill the stage just drained and wait for this one
  __device__ __forceinline__ void arrive(int p) const {
    if ((p & 7) == 0) {
      if (p >= 8) issue((p >> 3) + 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    }
  }
  __device__ __forceinline__ void get(Chunk<float, 4>& c, int p) const {
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(c.v[0]), "=f"(c.v[1]), "=f"(c.v[2]), "=f"(c.v[3])
                 : "r"(base + (unsigned)(((p & 15) * TPB) * 16)));
  }
  __device__ __forceinline__ void get(Chunk<double, 2>& c, int p) const {
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(c.v[0]), "=d"(c.v[1]) : "r"(base + (unsigned)(((p & 15) * TPB) * 16)));
  }
};

template <typename T, int NG, int MASK, int TPB, bool PIPE>
__device__ __forceinline__ void stream_run(const T* __restrict__ ptr, long long E, int p0, int p1,
                                           const uint8_t* __restrict__ bits_p, unsigned keep,
                                           T (&acc)[NG + 1][VecOf<T>::N], unsigned& flag, const Pipe<T, TPB>& pipe) {
  constexpr int V = VecOf<T>::N;
  constexpr int U = 8;
  bool any = false;
  unsigned any_bits = 0;
  auto one = [&](const Chunk<T, V>& x, int p) {
    const unsigned bits = MASK < 0 ? (__ldg(bits_p + p) & keep) : (unsigned)MASK;
    bool ok_any = false;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const bool ok = !is_nan(x.v[v]);
      const T z = ok ? x.v[v] : T(0);
      ok_any |= ok;
      acc[0][v] = add_rn(acc[0][v], z);
#pragma unroll
      for (int g = 0; g < NG; ++g)
        if ((bits >> g) & 1u) acc[g + 1][v] = add_rn(acc[g + 1][v], z);
    }
    any |= ok_any;
    if (MASK < 0) any_bits |= ok_any ? ((bits << 1) | 1u) : 0u;
  };
  int p = p0;
  if (PIPE) {
#pragma unroll 4
    for (; p < p1; ++p) {
      pipe.arrive(p);
      Chunk<T, V> x;
      pipe.get(x, p);
      one(x, p);
    }
  } else {
    for (; p + U <= p1; p += U) {
      Chunk<T, V> x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) load_chunk(x[u], ptr + (long long)(p + u) * E, true, V);
#pragma unroll
      for (int u = 0; u < U; ++u) one(x[u], p + u);
    }
    if (p + 4 <= p1) {
      Chunk<T, V> x[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) load_chunk(x[u], ptr + (long long)(p + u) * E, true, V);
#pragma unroll
      for (int u = 0; u < 4; ++u) one(x[u], p + u);
      p += 4;
    }
    for (; p < p1; ++p) {
      Chunk<T, V> x;
      load_chunk(x, ptr + (long long)p * E, true, V);
      one(x, p);
    }
  }
  if (MASK < 0)
    flag |= any_bits;
  else
    flag |= any ? (((unsigned)MASK << 1) | 1u) : 0u;
}

template <typename T, int NG, int TPB, bool PIPE>
__global__ void __launch_bounds__(TPB, (TPB <= 512 ? 2 : 1))
    collapse_stream_kernel(const csg_file_desc* __restrict__ files, int n_files, const int32_t* __restrict__ runs,
                           const uint8_t* __restrict__ pa_bits, int n_groups, T* __restrict__ sums,
                           uint8_t* __restrict__ row_flags) {
  constexpr int V = VecOf<T>::N;
  constexpr int EV = TPB / kTileRows;  // energy chunks per row
  constexpr int E = EV * V;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* s_out = reinterpret_cast<T*>(smem_raw);  // [(NG+1)][E][kOutPitch]; PIPE: first the threads' load slots [16][TPB] x 16 B
  __shared__ unsigned s_flags[kTileRows];

  const int fi = find_file(files, n_files, blockIdx.x);
  const csg_file_desc f = files[fi];
  const int t0 = (blockIdx.x - f.first_block) * kTileRows;
  const int rows_here = min(kTileRows, f.T - t0);
  const int r = threadIdx.x / EV, c = threadIdx.x - r * EV;
  if (threadIdx.x < kTileRows) s_flags[threadIdx.x] = 0;
  __syncthreads();

  const unsigned alias = (unsigned)f.reserved[2];  // groups holding every pitch bin
  T acc[NG + 1][V];
  unsigned flag = 0;
  if (r < rows_here) {
    const T* ptr = static_cast<const T*>(f.d_cube) + ((long long)(t0 + r) * f.P) * E + c * V;
    const int32_t* run = runs + 3 * (long long)f.reserved[0];
    const int n_runs = f.reserved[1];
    const uint8_t* bits_p = pa_bits + f.bits_off;
    Pipe<T, TPB> pipe;
    pipe.base = (unsigned)__cvta_generic_to_shared(smem_raw) + threadIdx.x * 16u;
    pipe.ptr = ptr, pipe.E = E, pipe.P = f.P;
    if (PIPE) pipe.start();
#pragma unroll
    for (int g = 0; g <= NG; ++g)
#pragma unroll
      for (int v = 0; v < V; ++v) acc[g][v] = T(0);
    for (int k = 0; k < n_runs; ++k) {
      const int p0 = __ldg(run + 3 * k), p1 = __ldg(run + 3 * k + 1), mask = __ldg(run + 3 * k + 2);
      if (NG == 4) {
        switch (mask & 15) {
#define CSG_RUN(M)                                                         \
  case M:                                                                  \
    stream_run<T, NG, M, TPB, PIPE>(ptr, E, p0, p1, bits_p, ~alias, acc, flag, pipe); \
    break;
          CSG_RUN(0)
          CSG_RUN(1)
          CSG_RUN(2)
          CSG_RUN(3)
          CSG_RUN(4)
          CSG_RUN(5)
          CSG_RUN(6)
          CSG_RUN(7)
          CSG_RUN(8)
          CSG_RUN(9)
          CSG_RUN(10)
          CSG_RUN(11)
          CSG_RUN(12)
          CSG_RUN(13)
          CSG_RUN(14)
          CSG_RUN(15)
#undef CSG_RUN
        }
      } else if (NG == 0) {
        stream_run<T, NG, 0, TPB, PIPE>(ptr, E, p0, p1, bits_p, ~alias, acc, flag, pipe);
      } else {
        stream_run<T, NG, -1, TPB, PIPE>(ptr, E, p0, p1, bits_p, ~alias, acc, flag, pipe);
      }
    }
    if (flag & 1u) flag |= alias << 1;
  }
  if (PIPE) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();  // every thread has drained its load slots: the staging tile may overwrite them
  }
  if (r < rows_here) {
#pragma unroll
    for (int g = 0; g <= NG; ++g) {
      const bool copy = g > 0 && ((alias >> (g - 1)) & 1u);
#pragma unroll
      for (int v = 0; v < V; ++v) s_out[((size_t)g * E + c * V + v) * kOutPitch + r] = copy ? acc[0][v] : acc[g][v];
    }
    if (flag) atomicOr(&s_flags[r], flag);
  }
  __syncthreads();
  // ---- transposed tile -> sums[g][e][t0 .. t0+rows_here): 64-byte segments
  const int Tp = pitch_of(f.T);
  const long long plane = (long long)E * Tp;
  T* out = sums + f.sums_off + t0;
  const int rr = threadIdx.x & (kTileRows - 1);
  constexpr int step = TPB / kTileRows;
  const int n_ge = (n_groups + 1) * E;
  if (rr < rows_here) {
    for (int ge = threadIdx.x / kTileRows; ge < n_ge; ge += step) {
      const int g = ge / E, e = ge - g * E;  // E is a compile-time constant
      out[g * plane + (long long)e * Tp + rr] = s_out[(size_t)ge * kOutPitch + rr];
    }
  }
  if (row_flags != nullptr && threadIdx.x < rows_here)
    row_flags[f.flags_off + t0 + threadIdx.x] = (uint8_t)s_flags[threadIdx.x];  // the block owns these rows
}

// ---------------------------------------------------------------------------------
// layout TPE, generic: thread = (time row, VEC consecutive energies); loop over pitch bins.
// Consecutive threads read consecutive 16-byte pieces of one (t,p) energy row, so every
// warp request covers whole 128-byte lines; P independent 128-bit loads per thread.
// ---------------------------------------------------------------------------------
template <typename T, int NG>
__global__ void __launch_bounds__(kBlock)
    collapse_tpe_kernel(const csg_file_desc* __restrict__ files, int n_files,
                        const uint8_t* __restrict__ pa_bits, int n_groups, T* __restrict__ sums,
                        uint8_t* __restrict__ row_flags) {
  extern __shared__ unsigned char smem_raw[];
  unsigned* s_flags = reinterpret_cast<unsigned*>(smem_raw);  // [kBlock + 1]
  uint8_t* s_bits = smem_raw + (kBlock + 1) * sizeof(unsigned);  // [P]

  const int fi = find_file(files, n_files, blockIdx.x);
  const csg_file_desc f = files[fi];
  constexpr int VEC = VecOf<T>::N;
  const int P = f.P, E = f.E;
  const int EV = (E + VEC - 1) / VEC;  // energy chunks per row (the last one may be partial)
  const long long n_items = (long long)f.T * EV;
  const long long item0 = (long long)(blockIdx.x - f.first_block) * kBlock;
  const long long item = item0 + threadIdx.x;
  const int t_first = (int)(item0 / EV);

  for (int p = threadIdx.x; p < P; p += kBlock) s_bits[p] = NG ? pa_bits[f.bits_off + p] : 0;
  for (int i = threadIdx.x; i <= kBlock; i += kBlock) s_flags[i] = 0;
  __syncthreads();

  if (item < n_items) {
    const int t = (int)(item / EV);
    const int c = (int)(item - (long long)t * EV);
    const T* cube = static_cast<const T*>(f.d_cube);
    const T* ptr = cube + ((long long)t * P) * E + (long long)c * VEC;
    const int valid = (E - c * VEC) < VEC ? (E - c * VEC) : VEC;
    const bool aligned = (E % VEC == 0) && ((reinterpret_cast<uintptr_t>(cube) & 15) == 0);

    T acc[NG + 1][VEC];
#pragma unroll
    for (int g = 0; g <= NG; ++g)
#pragma unroll
      for (int v = 0; v < VEC; ++v) acc[g][v] = T(0);
    unsigned flag = 0;

    constexpr int U = 8;
    int p = 0;
    for (; p + U <= P; p += U) {
      Chunk<T, VEC> x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) load_chunk(x[u], ptr + (long long)(p + u) * E, aligned, valid);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const unsigned bits = s_bits[p + u];
        const unsigned member = (bits << 1) | 1u;
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          const T xv = x[u].v[v];
          const bool ok = !is_nan(xv);
          const T z = ok ? xv : T(0);
          flag |= ok ? member : 0u;
          acc[0][v] = add_rn(acc[0][v], z);
#pragma unroll
          for (int g = 0; g < NG; ++g)
            if ((bits >> g) & 1u) acc[g + 1][v] = add_rn(acc[g + 1][v], z);
        }
      }
    }
    for (; p < P; ++p) {
      Chunk<T, VEC> x;
      load_chunk(x, ptr + (long long)p * E, aligned, valid);
      const unsigned bits = s_bits[p];
      const unsigned member = (bits << 1) | 1u;
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const T xv = x.v[v];
        const bool ok = !is_nan(xv);
        const T z = ok ? xv : T(0);
        flag |= ok ? member : 0u;
        acc[0][v] = add_rn(acc[0][v], z);
#pragma unroll
        for (int g = 0; g < NG; ++g)
          if ((bits >> g) & 1u) acc[g + 1][v] = add_rn(acc[g + 1][v], z);
      }
    }

    // energy-major output: element (e, t) at e*Tp + t (uncoalesced here; the stream kernel is the fast path)
    const int Tp = pitch_of(f.T);
    const long long plane = (long long)E * Tp;
    T* out = sums + f.sums_off + t;
#pragma unroll
    for (int g = 0; g <= NG; ++g)
      if (g <= n_groups)
#pragma unroll
        for (int v = 0; v < VEC; ++v)
          if (v < valid) out[g * plane + (long long)(c * VEC + v) * Tp] = acc[g][v];
    if (flag) atomicOr(&s_flags[t - t_first], flag);
  }
  __syncthreads();
  if (row_flags != nullptr) {
    // rows touched by this block: t_first .. t_last (a row can straddle two blocks)
    const long long last_item = (item0 + kBlock < n_items ? item0 + kBlock : n_items) - 1;
    const int n_rows = (int)(last_item / EV) - t_first + 1;
    for (int r = threadIdx.x; r < n_rows; r += kBlock) {
      const unsigned fl = s_flags[r];
      if (fl) or_flag_byte(row_flags + f.flags_off + t_first + r, fl);
    }
  }
}

// numpy pairwise_sum over n contiguous values (NaN already treated as 0), n >= 0
template <typename T, typename Load>
__device__ T pairwise_sum(Load load, int first, int n) {
  if (n < 8) {
    T r = T(-0.0);
    for (int i = 0; i < n; ++i) r = add_rn(r, load(first + i));
    return r;
  }
  if (n <= 128) {
    T r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = load(first + k);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
      for (int k = 0; k < 8; ++k) r[k] = add_rn(r[k], load(first + i + k));
    }
    T res = add_rn(add_rn(add_rn(r[0], r[1]), add_rn(r[2], r[3])),
                   add_rn(add_rn(r[4], r[5]), add_rn(r[6], r[7])));
    for (; i < n; ++i) res = add_rn(res, load(first + i));
    return res;
  }
  int n2 = n / 2;
  n2 -= n2 % 8;
  return add_rn(pairwise_sum<T>(load, first, n2), pairwise_sum<T>(load, first + n2, n - n2));
}

// ---------------------------------------------------------------------------------
// layout TEP: rows of P contiguous pitch samples.  A block stages ROWS rows in shared
// memory with coalesced 128-bit loads (row pitch P+1 words -> conflict-free row walks),
// then one thread per (t,e) row runs numpy's pairwise order for the total and the
// ascending-p chain for each pitch-angle group.
// ---------------------------------------------------------------------------------
template <typename T, int NG>
__global__ void collapse_tep_kernel(const csg_file_desc* __restrict__ files, int n_files,
                                    const uint8_t* __restrict__ pa_bits, int n_groups,
                                    T* __restrict__ sums, uint8_t* __restrict__ row_flags, int rows_per_block,
                                    int max_P) {
  extern __shared__ unsigned char smem_raw[];
  T* s_rows = reinterpret_cast<T*>(smem_raw);  // [rows_per_block][max_P + 1]
  uint8_t* s_bits = smem_raw + (size_t)rows_per_block * (max_P + 1) * sizeof(T);

  const int fi = find_file(files, n_files, blockIdx.x);
  const csg_file_desc f = files[fi];
  const int P = f.P, E = f.E;
  const long long n_rows = (long long)f.T * E;
  const long long row0 = (long long)(blockIdx.x - f.first_block) * rows_per_block;
  const int rows_here = (int)(n_rows - row0 < rows_per_block ? n_rows - row0 : rows_per_block);
  const T* cube = static_cast<const T*>(f.d_cube) + row0 * P;
  const int pitch = P + 1;

  for (int p = threadIdx.x; p < P; p += blockDim.x) s_bits[p] = NG ? pa_bits[f.bits_off + p] : 0;
  const long long n_elem = (long long)rows_here * P;
  constexpr int VEC = VecOf<T>::N;
  const bool aligned = ((reinterpret_cast<uintptr_t>(cube) & 15) == 0);
  if (aligned) {
    const long long n_vec = n_elem / VEC;
    for (long long i = threadIdx.x; i < n_vec; i += blockDim.x) {
      Chunk<T, VEC> x;
      load_chunk(x, cube + i * VEC, true, VEC);
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const long long j = i * VEC + v;
        const int r = (int)(j / P), p = (int)(j - (long long)r * P);
        s_rows[r * pitch + p] = x.v[v];
      }
    }
    for (long long j = n_vec * VEC + threadIdx.x; j < n_elem; j += blockDim.x) {
      const int r = (int)(j / P), p = (int)(j - (long long)r * P);
      s_rows[r * pitch + p] = ld_stream1(cube + j);
    }
  } else {
    for (long long j = threadIdx.x; j < n_elem; j += blockDim.x) {
      const int r = (int)(j / P), p = (int)(j - (long long)r * P);
      s_rows[r * pitch + p] = ld_stream1(cube + j);
    }
  }
  __syncthreads();

  const int r = threadIdx.x;
  if (r < rows_here) {
    const T* row = s_rows + r * pitch;
    unsigned flag = 0;
    T acc[NG + 1];
#pragma unroll
    for (int g = 0; g <= NG; ++g) acc[g] = T(0);
    for (int p = 0; p < P; ++p) {
      const T xv = row[p];
      const bool ok = !is_nan(xv);
      const unsigned bits = s_bits[p];
      flag |= ok ? ((bits << 1) | 1u) : 0u;
      const T z = ok ? xv : T(0);
#pragma unroll
      for (int g = 0; g < NG; ++g)
        if ((bits >> g) & 1u) acc[g + 1] = add_rn(acc[g + 1], z);
    }
    auto load = [row](int i) {
      const T xv = row[i];
      return is_nan(xv) ? T(0) : xv;
    };
    acc[0] = add_rn(T(0), pairwise_sum<T>(load, 0, P));  // reduction seeded with +0.0

    const long long grow = row0 + r;  // = t*E + e
    const int t = (int)(grow / E), e = (int)(grow - (long long)t * E);
    const int Tp = pitch_of(f.T);
    const long long plane = (long long)E * Tp;
    T* out = sums + f.sums_off + (long long)e * Tp + t;
#pragma unroll
    for (int g = 0; g <= NG; ++g)
      if (g <= n_groups) out[g * plane] = acc[g];
    if (row_flags != nullptr && flag) or_flag_byte(row_flags + f.flags_off + t, flag);
  }
}

// ---------------------------------------------------------------------------------
// layout TEP, total only (no pitch-angle groups), 8 <= P <= 128, P % 8 == 0: the generic stress cubes
// of BASELINE config 5.  numpy sums a contiguous axis of n <= 128 elements with eight interleaved
// accumulators r[k] += a[8j + k] and combines them as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)).  Two
// lanes share a (t, e) row: lane h owns r[4h .. 4h+3], i.e. the float4 at 8j + 4h of every group of
// eight -- P/8 independent 128-bit loads per lane, all in flight, 32-byte segments of 16 rows per
// warp instruction.  A block owns 32 consecutive time steps x every energy (one contiguous slab
// of the cube), stages the sums [e][t] in shared memory and writes 128-byte rows of the
// energy-major output; it also owns the zoom flags of its time steps.
// ---------------------------------------------------------------------------------
constexpr int kTepTile = 32;

template <typename T>
__global__ void __launch_bounds__(256)
    collapse_tep_rows_kernel(const csg_file_desc* __restrict__ files, int n_files, T* __restrict__ sums,
                             uint8_t* __restrict__ row_flags) {
  constexpr int V = VecOf<T>::N;       // elements per 16-byte load
  constexpr int LPR = 8 / V;           // lanes per row: each lane owns V of the eight accumulators
  constexpr int RPW = 32 / LPR;        // rows per warp pass
  constexpr int MAXJ = 16;             // P <= 128
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* s_out = reinterpret_cast<T*>(smem_raw);  // [E][kTepTile + 1]
  __shared__ unsigned s_flags[kTepTile];

  const int fi = find_file(files, n_files, blockIdx.x);
  const csg_file_desc f = files[fi];
  const int P = f.P, E = f.E, nj = P / 8;
  const int t0 = (blockIdx.x - f.first_block) * kTepTile;
  const int nt = min(kTepTile, f.T - t0);
  const long long n_rows = (long long)nt * E;  // rows (t, e) of this tile: one contiguous slab
  const T* slab = static_cast<const T*>(f.d_cube) + (long long)t0 * E * P;
  if (threadIdx.x < kTepTile) s_flags[threadIdx.x] = 0;
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
  const int sub = lane / LPR, h = lane % LPR;
  for (long long base = (long long)warp * RPW; base < n_rows; base += (long long)n_warps * RPW) {
    const long long row = base + sub;
    const bool in = row < n_rows;
    const T* q = slab + (in ? row : 0) * P + h * V;
    Chunk<T, V> x[MAXJ];
#pragma unroll
    for (int j = 0; j < MAXJ; ++j)
      if (j < nj) load_chunk(x[j], q + 8 * j, true, V);
    T r[V];
    bool any = false;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const bool ok = !is_nan(x[0].v[v]);
      any |= ok;
      r[v] = ok ? x[0].v[v] : T(0);
    }
#pragma unroll
    for (int j = 1; j < MAXJ; ++j)
      if (j < nj) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const bool ok = !is_nan(x[j].v[v]);
          any |= ok;
          r[v] = add_rn(r[v], ok ? x[j].v[v] : T(0));
        }
      }
    // ((r0+r1)+(r2+r3)) + ((r4+r5)+(r6+r7)): pairs inside the lane first, then across the row's lanes
    T s;
    if (V == 4) {
      s = add_rn(add_rn(r[0], r[1]), add_rn(r[V - 2], r[V - 1]));
      s = add_rn(s, __shfl_down_sync(0xffffffffu, s, 1));  // lane h=0 holds left + right
    } else {  // V == 2: four lanes per row own (r0,r1) (r2,r3) (r4,r5) (r6,r7)
      s = add_rn(r[0], r[V - 1]);
      s = add_rn(s, __shfl_down_sync(0xffffffffu, s, 1));  // h=0: (r0+r1)+(r2+r3); h=2: (r4+r5)+(r6+r7)
      s = add_rn(s, __shfl_down_sync(0xffffffffu, s, 2));  // h=0: left + right
    }
    unsigned okmask = __ballot_sync(0xffffffffu, any);
    if (in && h == 0) {
      const int tl = (int)(row / E), e = (int)(row - (long long)tl * E);
      s_out[e * (kTepTile + 1) + tl] = add_rn(T(0), s);  // the reduction is seeded with +0.0
      if ((okmask >> (lane & ~(LPR - 1))) & ((1u << LPR) - 1u)) atomicOr(&s_flags[tl], 1u);
    }
  }
  __syncthreads();
  const int Tp = pitch_of(f.T);
  T* out = sums + f.sums_off + t0;
  const int tl = threadIdx.x & (kTepTile - 1);
  if (tl < nt)
    for (int e = threadIdx.x / kTepTile; e < E; e += blockDim.x / kTepTile) out[(long long)e * Tp + tl] = s_out[e * (kTepTile + 1) + tl];
  if (row_flags != nullptr && threadIdx.x < nt && s_flags[threadIdx.x])
    row_flags[f.flags_off + t0 + threadIdx.x] = (uint8_t)s_flags[threadIdx.x];  // the block owns these time steps
}

inline bool tep_rows_ok(int32_t T, int32_t P, int32_t E, const void* d_cube, int n_groups) {
  return n_groups == 0 && T > 0 && P >= 8 && P <= 128 && P % 8 == 0 && E > 0 && E <= 1024 &&
         (reinterpret_cast<uintptr_t>(d_cube) & 15) == 0;
}

// warp = one zoom window: any row with the group's bit set?
__global__ void window_any_kernel(const uint8_t* __restrict__ row_flags, const csg_flag_window* __restrict__ windows,
                                  int n_windows, const int32_t* __restrict__ pool, uint8_t* __restrict__ out) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= n_windows) return;
  const csg_flag_window win = windows[w];
  const uint8_t* fl = row_flags + win.flags_off;
  bool any = false;
  for (int i = lane; i < win.nt; i += 32) {
    const int row = win.rows_off < 0 ? win.t0 + i : __ldg(pool + win.rows_off + i);
    any |= ((fl[row] >> win.bit) & 1u) != 0;
  }
  any = __any_sync(0xffffffffu, any);
  if (lane == 0) out[w] = any ? 1 : 0;
}

inline int tep_rows_per_block(int P, int dtype) {
  const size_t es = dtype == CSG_F64 ? 8 : 4;
  int rows = 256;
  while (rows > 32 && (size_t)rows * (P + 1) * es > 96 * 1024) rows >>= 1;
  return rows;
}

// ---- stream kernel eligibility: 16 x (E / VEC) threads per block must be a supported block size
inline int stream_tpb(int E, int dtype) {
  const int V = dtype == CSG_F64 ? 2 : 4;
  if (E <= 0 || E % V != 0) return 0;
  const int tpb = kTileRows * (E / V);
  return (tpb == 256 || tpb == 384 || tpb == 512 || tpb == 768 || tpb == 1024) ? tpb : 0;
}
inline size_t stream_smem(int E, int n_groups, int dtype) {
  const int NG = n_groups == 0 ? 0 : (n_groups <= 4 ? 4 : CSG_MAX_GROUPS);
  return (size_t)(NG + 1) * E * kOutPitch * (dtype == CSG_F64 ? 8 : 4);
}
inline bool stream_file_ok(int32_t T, int32_t P, int32_t E, int dtype, const void* d_cube) {
  if (T <= 0 || P <= 0 || stream_tpb(E, dtype) == 0) return false;
  return (reinterpret_cast<uintptr_t>(d_cube) & 15) == 0;
}

template <typename T>
int launch_tpe(csg_ctx* ctx, const csg_file_desc* d_files, int n_files, int total_blocks,
               const uint8_t* d_pa_bits, int n_groups, int max_P, T* d_sums, uint8_t* d_row_flags) {
  const size_t smem = (kBlock + 1) * sizeof(unsigned) + (size_t)max_P;
  auto go = [&](auto kern) {
    kern<<<total_blocks, kBlock, smem, ctx->stream>>>(d_files, n_files, d_pa_bits, n_groups, d_sums, d_row_flags);
  };
  if (n_groups == 0)
    go(collapse_tpe_kernel<T, 0>);
  else if (n_groups <= 4)
    go(collapse_tpe_kernel<T, 4>);
  else
    go(collapse_tpe_kernel<T, CSG_MAX_GROUPS>);
  CSG_LAUNCH_CHECK(ctx, "collapse_tpe_kernel");
  return CSG_OK;
}

// The cp.async pipeline needs 256 bytes of shared memory per thread; two blocks per SM must still
// fit, so blocks of up to 384 threads (E = 96 float32 / 48 float64 -- the FAST tables) take it and
// larger blocks (e.g. E = 96 float64) the register-staged body.  The block size fixes the body, so
// only that one is instantiated.
template <typename T, int NG, int TPB>
int launch_stream_one(csg_ctx* ctx, size_t smem, const csg_file_desc* d_files, int n_files, int total_blocks,
                      const int32_t* d_runs, const uint8_t* d_pa_bits, int n_groups, T* d_sums, uint8_t* d_row_flags) {
  if constexpr (TPB * 256 <= 100 * 1024) {
    auto kern = collapse_stream_kernel<T, NG, TPB, true>;
    const size_t need = smem > (size_t)TPB * 256 ? smem : (size_t)TPB * 256;
    CSG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
    kern<<<total_blocks, TPB, need, ctx->stream>>>(d_files, n_files, d_runs, d_pa_bits, n_groups, d_sums, d_row_flags);
  } else {
    auto kern = collapse_stream_kernel<T, NG, TPB, false>;
    CSG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<total_blocks, TPB, smem, ctx->stream>>>(d_files, n_files, d_runs, d_pa_bits, n_groups, d_sums, d_row_flags);
  }
  CSG_LAUNCH_CHECK(ctx, "collapse_stream_kernel");
  return CSG_OK;
}

template <typename T, int NG>
int launch_stream_ng(csg_ctx* ctx, int tpb, size_t smem, const csg_file_desc* d_files, int n_files, int total_blocks,
                     const int32_t* d_runs, const uint8_t* d_pa_bits, int n_groups, T* d_sums, uint8_t* d_row_flags) {
#define CSG_GO(TPB)                                                                                                   \
  case TPB:                                                                                                           \
    return launch_stream_one<T, NG, TPB>(ctx, smem, d_files, n_files, total_blocks, d_runs, d_pa_bits, n_groups, d_sums, \
                                         d_row_flags);
  switch (tpb) {
    CSG_GO(256)
    CSG_GO(384)
    CSG_GO(512)
    CSG_GO(768)
    CSG_GO(1024)
  }
#undef CSG_GO
  return csg_fail(ctx, CSG_ERR_ARG, "stream kernel: unsupported block size %d", tpb);
}

template <typename T>
int launch_stream(csg_ctx* ctx, int E, int dtype, const csg_file_desc* d_files, int n_files, int total_blocks,
                  const int32_t* d_runs, const uint8_t* d_pa_bits, int n_groups, T* d_sums, uint8_t* d_row_flags) {
  const int tpb = stream_tpb(E, dtype);
  const size_t smem = stream_smem(E, n_groups, dtype);
  if (tpb == 0 || smem > 200 * 1024)
    return csg_fail(ctx, CSG_ERR_ARG, "stream kernel cannot handle E=%d: use CSG_K1_GENERIC for this table", E);
  if (n_groups == 0)
    return launch_stream_ng<T, 0>(ctx, tpb, smem, d_files, n_files, total_blocks, d_runs, d_pa_bits, n_groups, d_sums,
                                  d_row_flags);
  if (n_groups <= 4)
    return launch_stream_ng<T, 4>(ctx, tpb, smem, d_files, n_files, total_blocks, d_runs, d_pa_bits, n_groups, d_sums,
                                  d_row_flags);
  return launch_stream_ng<T, CSG_MAX_GROUPS>(ctx, tpb, smem, d_files, n_files, total_blocks, d_runs, d_pa_bits, n_groups,
                                             d_sums, d_row_flags);
}

template <typename T>
int launch_tep(csg_ctx* ctx, const csg_file_desc* d_files, int n_files, int total_blocks,
               const uint8_t* d_pa_bits, int n_groups, int max_P, int dtype, T* d_sums, uint8_t* d_row_flags) {
  const int rows = tep_rows_per_block(max_P, dtype);
  const size_t smem = (size_t)rows * (max_P + 1) * sizeof(T) + (size_t)max_P;
  if (smem > 200 * 1024)
    return csg_fail(ctx, CSG_ERR_ARG, "layout TEP supports at most %d pitch bins per row for this dtype (got %d)",
                    (int)(200 * 1024 / (32 * sizeof(T))) - 2, max_P);
  auto go = [&](auto kern) {
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<total_blocks, rows, smem, ctx->stream>>>(d_files, n_files, d_pa_bits, n_groups, d_sums, d_row_flags, rows, max_P);
  };
  if (n_groups == 0)
    go(collapse_tep_kernel<T, 0>);
  else if (n_groups <= 4)
    go(collapse_tep_kernel<T, 4>);
  else
    go(collapse_tep_kernel<T, CSG_MAX_GROUPS>);
  CSG_LAUNCH_CHECK(ctx, "collapse_tep_kernel");
  return CSG_OK;
}

// =================================================================================
// Integer cubes (CSG_I8 .. CSG_U32): numpy sums them in int64 / uint64, and integer addition is
// associative, so any order gives the same bits -- there is no numpy order to copy.  The kernels
// read the stored type and accumulate in 32 bits (8- and 16-bit input: |sum| <= 65535 * 32768 < 2^31
// at the largest P csg_collapse accepts) or 64 bits (32-bit input: |sum| <= 2^32 * 2^15 = 2^47), then
// write float64 sums -- exact, since every such sum is below 2^53 -- the dtype every later stage
// reads.  There is no NaN: the row flags of row t are bit 0 and bit 1+k for every group k with a
// member bin, as the widened float64 path sets them.
// =================================================================================
template <typename I>
struct IntAcc {
  typedef int32_t A;
};
template <>
struct IntAcc<int32_t> {
  typedef long long A;
};
template <>
struct IntAcc<uint32_t> {
  typedef long long A;
};

// value v of the 16 bytes w of stored integers (v is a constant after unrolling: a shift and a convert)
template <typename I>
__device__ __forceinline__ typename IntAcc<I>::A int_elem(const uint4& w, int v) {
  constexpr int PER = 4 / sizeof(I);
  const int k = v / PER, j = v % PER;
  const unsigned word = k == 0 ? w.x : k == 1 ? w.y : k == 2 ? w.z : w.w;
  return (typename IntAcc<I>::A)(I)(word >> (8 * sizeof(I) * j));
}

__device__ __forceinline__ uint4 ld_stream_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

inline size_t int_itemsize(int dtype) {
  switch (dtype) {
    case CSG_I8:
    case CSG_U8:
      return 1;
    case CSG_I16:
    case CSG_U16:
      return 2;
    case CSG_I32:
    case CSG_U32:
      return 4;
  }
  return 0;
}
inline bool is_int_dtype(int dtype) { return int_itemsize(dtype) != 0; }
inline size_t cube_itemsize(int dtype) { return dtype == CSG_F64 ? 8 : (dtype == CSG_F32 ? 4 : int_itemsize(dtype)); }
inline size_t sums_itemsize(int dtype) { return dtype == CSG_F32 ? 4 : 8; }

// ---- stream kernel (TPE, 16-byte aligned, E * itemsize a multiple of 16): block = 16 time rows x the
// EV = E * itemsize / 16 chunks of a row, thread = (row, 16 bytes of consecutive energies).  The pitch
// axis is walked in the runs of constant group membership of the float stream kernel, eight 128-bit
// streaming loads in flight per thread.  The transposed tile leaves through shared memory one group at
// a time (the shared tile is E x 17 doubles whatever the number of groups).
constexpr int kIntStreamMaxEV = 32;  // blocks of at most 16 x 32 = 512 threads

inline int int_stream_ev(int E, int dtype) {
  const size_t es = int_itemsize(dtype);
  if (es == 0 || E <= 0 || (E * es) % 16 != 0) return 0;
  const int ev = (int)(E * es / 16);
  return ev <= kIntStreamMaxEV ? ev : 0;
}

template <typename I, int NG, int MASK>
__device__ __forceinline__ void int_stream_run(const I* __restrict__ ptr, long long E, int p0, int p1,
                                               const uint8_t* __restrict__ bits_p, unsigned keep,
                                               typename IntAcc<I>::A (&acc)[NG + 1][16 / sizeof(I)], unsigned& flag) {
  using A = typename IntAcc<I>::A;
  constexpr int V = 16 / sizeof(I);
  // eight loads in flight; four where the accumulators alone take 64 registers (they would spill)
  constexpr int U = (NG + 1) * V * sizeof(A) >= 256 ? 4 : 8;
  auto one = [&](const uint4& w, int p) {
    const unsigned bits = MASK < 0 ? (__ldg(bits_p + p) & keep) : (unsigned)MASK;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const A z = int_elem<I>(w, v);
      acc[0][v] += z;
#pragma unroll
      for (int g = 0; g < NG; ++g)
        if ((bits >> g) & 1u) acc[g + 1][v] += z;
    }
    if (MASK < 0) flag |= (bits << 1) | 1u;
  };
  int p = p0;
  for (; p + U <= p1; p += U) {
    uint4 x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) x[u] = ld_stream_u4(ptr + (long long)(p + u) * E);
#pragma unroll
    for (int u = 0; u < U; ++u) one(x[u], p + u);
  }
  for (; p < p1; ++p) one(ld_stream_u4(ptr + (long long)p * E), p);
  if (MASK >= 0 && p1 > p0) flag |= ((unsigned)MASK << 1) | 1u;
}

template <typename I, int NG>
__global__ void __launch_bounds__(kTileRows* kIntStreamMaxEV, 1)
    collapse_int_stream_kernel(const csg_file_desc* __restrict__ files, int n_files, const int32_t* __restrict__ runs,
                               const uint8_t* __restrict__ pa_bits, int n_groups, double* __restrict__ sums,
                               uint8_t* __restrict__ row_flags) {
  using A = typename IntAcc<I>::A;
  constexpr int V = 16 / sizeof(I);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* s_out = reinterpret_cast<double*>(smem_raw);  // [E][kOutPitch], one group at a time

  const int fi = find_file(files, n_files, blockIdx.x);
  const csg_file_desc f = files[fi];
  const int EV = blockDim.x / kTileRows;  // every file of the launch has E = EV * V
  const int E = EV * V;
  const int t0 = (blockIdx.x - f.first_block) * kTileRows;
  const int rows_here = min(kTileRows, f.T - t0);
  const int r = threadIdx.x / EV, c = threadIdx.x - r * EV;

  const unsigned alias = (unsigned)f.reserved[2];  // groups holding every pitch bin
  A acc[NG + 1][V];
#pragma unroll
  for (int g = 0; g <= NG; ++g)
#pragma unroll
    for (int v = 0; v < V; ++v) acc[g][v] = A(0);
  unsigned flag = 0;
  if (r < rows_here) {
    const I* ptr = static_cast<const I*>(f.d_cube) + ((long long)(t0 + r) * f.P) * E + c * V;
    const int32_t* run = runs + 3 * (long long)f.reserved[0];
    const int n_runs = f.reserved[1];
    const uint8_t* bits_p = pa_bits + f.bits_off;
    for (int k = 0; k < n_runs; ++k) {
      const int p0 = __ldg(run + 3 * k), p1 = __ldg(run + 3 * k + 1), mask = __ldg(run + 3 * k + 2);
      if (NG == 4) {
        switch (mask & 15) {
#define CSG_RUN(M)                                                             \
  case M:                                                                      \
    int_stream_run<I, NG, M>(ptr, E, p0, p1, bits_p, ~alias, acc, flag); \
    break;
          CSG_RUN(0)
          CSG_RUN(1)
          CSG_RUN(2)
          CSG_RUN(3)
          CSG_RUN(4)
          CSG_RUN(5)
          CSG_RUN(6)
          CSG_RUN(7)
          CSG_RUN(8)
          CSG_RUN(9)
          CSG_RUN(10)
          CSG_RUN(11)
          CSG_RUN(12)
          CSG_RUN(13)
          CSG_RUN(14)
          CSG_RUN(15)
#undef CSG_RUN
        }
      } else if (NG == 0) {
        int_stream_run<I, NG, 0>(ptr, E, p0, p1, bits_p, ~alias, acc, flag);
      } else {
        int_stream_run<I, NG, -1>(ptr, E, p0, p1, bits_p, ~alias, acc, flag);
      }
    }
    if (flag & 1u) flag |= alias << 1;
  }
  // every thread of a row walked every pitch bin: its flag is the row's
  if (row_flags != nullptr && r < rows_here && c == 0) row_flags[f.flags_off + t0 + r] = (uint8_t)flag;

  const int Tp = pitch_of(f.T);
  const long long plane = (long long)E * Tp;
  double* out = sums + f.sums_off + t0;
  const int rr = threadIdx.x & (kTileRows - 1);
  const int step = blockDim.x / kTileRows;
#pragma unroll
  for (int g = 0; g <= NG; ++g) {
    if (g > n_groups) break;
    if (g > 0) __syncthreads();  // the previous group's tile has left
    if (r < rows_here) {
      const bool copy = g > 0 && ((alias >> (g - 1)) & 1u);
#pragma unroll
      for (int v = 0; v < V; ++v) s_out[(c * V + v) * kOutPitch + r] = (double)(copy ? acc[0][v] : acc[g][v]);
    }
    __syncthreads();
    if (rr < rows_here)
      for (int e = threadIdx.x / kTileRows; e < E; e += step) out[g * plane + (long long)e * Tp + rr] = s_out[e * kOutPitch + rr];
  }
}

// ---- generic (TPE, any E or alignment): thread = one (t, e) cell column, consecutive threads read
// consecutive energies of a (t, p) row.
template <typename I, int NG>
__global__ void __launch_bounds__(kBlock)
    collapse_int_tpe_kernel(const csg_file_desc* __restrict__ files, int n_files, const uint8_t* __restrict__ pa_bits,
                            int n_groups, double* __restrict__ sums, uint8_t* __restrict__ row_flags) {
  using A = typename IntAcc<I>::A;
  extern __shared__ unsigned char smem_raw[];
  uint8_t* s_bits = smem_raw;  // [P]
  const int fi = find_file(files, n_files, blockIdx.x);
  const csg_file_desc f = files[fi];
  const int P = f.P, E = f.E;
  const long long item = (long long)(blockIdx.x - f.first_block) * kBlock + threadIdx.x;
  for (int p = threadIdx.x; p < P; p += kBlock) s_bits[p] = NG ? pa_bits[f.bits_off + p] : 0;
  __syncthreads();
  if (item >= (long long)f.T * E) return;
  const int t = (int)(item / E), e = (int)(item - (long long)t * E);
  const I* ptr = static_cast<const I*>(f.d_cube) + (long long)t * P * E + e;
  A acc[NG + 1];
#pragma unroll
  for (int g = 0; g <= NG; ++g) acc[g] = A(0);
  unsigned flag = 0;
  auto one = [&](I x, int p) {
    const unsigned bits = s_bits[p];
    const A z = (A)x;
    acc[0] += z;
#pragma unroll
    for (int g = 0; g < NG; ++g)
      if ((bits >> g) & 1u) acc[g + 1] += z;
    flag |= (bits << 1) | 1u;
  };
  constexpr int U = 8;
  int p = 0;
  for (; p + U <= P; p += U) {
    I x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) x[u] = __ldg(ptr + (long long)(p + u) * E);
#pragma unroll
    for (int u = 0; u < U; ++u) one(x[u], p + u);
  }
  for (; p < P; ++p) one(__ldg(ptr + (long long)p * E), p);
  const int Tp = pitch_of(f.T);
  const long long plane = (long long)E * Tp;
  double* out = sums + f.sums_off + (long long)e * Tp + t;
#pragma unroll
  for (int g = 0; g <= NG; ++g)
    if (g <= n_groups) out[g * plane] = (double)acc[g];
  if (row_flags != nullptr && e == 0) row_flags[f.flags_off + t] = (uint8_t)flag;  // the same for every e
}

// ---- stored (T,E,P) view: rows of P contiguous pitch samples, L = int_tep_lanes(P) lanes per (t, e)
// row (about four samples a lane for short rows), consecutive lanes read consecutive samples; the
// lanes' partial sums meet through shuffles.  Any P, any alignment, any number of groups.
__host__ __device__ inline int int_tep_lanes(int P) {
  return P >= 128 ? 32 : P >= 64 ? 16 : P >= 32 ? 8 : P >= 16 ? 4 : P >= 8 ? 2 : 1;
}

template <typename I, int NG>
__global__ void __launch_bounds__(kBlock)
    collapse_int_tep_kernel(const csg_file_desc* __restrict__ files, int n_files, const uint8_t* __restrict__ pa_bits,
                            int n_groups, double* __restrict__ sums, uint8_t* __restrict__ row_flags) {
  using A = typename IntAcc<I>::A;
  extern __shared__ unsigned char smem_raw[];
  uint8_t* s_bits = smem_raw;  // [P]
  const int fi = find_file(files, n_files, blockIdx.x);
  const csg_file_desc f = files[fi];
  const int P = f.P, E = f.E;
  const int L = int_tep_lanes(P);
  const long long row = (long long)(blockIdx.x - f.first_block) * (kBlock / L) + threadIdx.x / L;
  const int h = threadIdx.x & (L - 1);
  for (int p = threadIdx.x; p < P; p += kBlock) s_bits[p] = NG ? pa_bits[f.bits_off + p] : 0;
  __syncthreads();
  const bool in = row < (long long)f.T * E;
  A acc[NG + 1];
#pragma unroll
  for (int g = 0; g <= NG; ++g) acc[g] = A(0);
  unsigned flag = 0;
  if (in) {
    const I* q = static_cast<const I*>(f.d_cube) + row * P;
    for (int p = h; p < P; p += L) {
      const unsigned bits = s_bits[p];
      const A z = (A)__ldg(q + p);
      acc[0] += z;
#pragma unroll
      for (int g = 0; g < NG; ++g)
        if ((bits >> g) & 1u) acc[g + 1] += z;
      flag |= (bits << 1) | 1u;
    }
  }
  for (int o = 1; o < L; o <<= 1) {  // L is uniform in the block: every lane of the warp takes part
#pragma unroll
    for (int g = 0; g <= NG; ++g) acc[g] += __shfl_xor_sync(0xffffffffu, acc[g], o);
    flag |= __shfl_xor_sync(0xffffffffu, flag, o);
  }
  if (!in || h != 0) return;
  const int t = (int)(row / E), e = (int)(row - (long long)t * E);
  const int Tp = pitch_of(f.T);
  const long long plane = (long long)E * Tp;
  double* out = sums + f.sums_off + (long long)e * Tp + t;
#pragma unroll
  for (int g = 0; g <= NG; ++g)
    if (g <= n_groups) out[g * plane] = (double)acc[g];
  if (row_flags != nullptr && e == 0) row_flags[f.flags_off + t] = (uint8_t)flag;  // the same for every e
}

// 8-bit input with more than 4 groups would keep 8 x 16 accumulators per thread: the generic kernel
inline bool int_stream_file_ok(int32_t T, int32_t P, int32_t E, int dtype, const void* d_cube, int n_groups) {
  if (int_itemsize(dtype) == 1 && n_groups > 4) return false;
  return T > 0 && P > 0 && int_stream_ev(E, dtype) > 0 && (reinterpret_cast<uintptr_t>(d_cube) & 15) == 0;
}

template <typename I>
int launch_int(csg_ctx* ctx, int layout, int kernel, const csg_file_desc* d_files, int n_files, int total_blocks,
               const uint8_t* d_pa_bits, const int32_t* d_runs, int n_groups, int max_P, int max_E, int dtype,
               double* d_sums, uint8_t* d_row_flags) {
  auto go = [&](auto kern, int threads, size_t smem) -> int {
    if (smem > 48 * 1024) CSG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<total_blocks, threads, smem, ctx->stream>>>(d_files, n_files, d_pa_bits, n_groups, d_sums, d_row_flags);
    return CSG_OK;
  };
  auto by_groups = [&](auto k0, auto k4, auto k7, int threads, size_t smem) -> int {
    return n_groups == 0 ? go(k0, threads, smem) : n_groups <= 4 ? go(k4, threads, smem) : go(k7, threads, smem);
  };
  int st;
  if (layout == CSG_LAYOUT_TEP) {
    st = by_groups(collapse_int_tep_kernel<I, 0>, collapse_int_tep_kernel<I, 4>, collapse_int_tep_kernel<I, CSG_MAX_GROUPS>,
                   kBlock, (size_t)max_P);
    if (st != CSG_OK) return st;
    CSG_LAUNCH_CHECK(ctx, "collapse_int_tep_kernel");
    return CSG_OK;
  }
  if (kernel != CSG_K1_STREAM) {
    st = by_groups(collapse_int_tpe_kernel<I, 0>, collapse_int_tpe_kernel<I, 4>, collapse_int_tpe_kernel<I, CSG_MAX_GROUPS>,
                   kBlock, (size_t)max_P);
    if (st != CSG_OK) return st;
    CSG_LAUNCH_CHECK(ctx, "collapse_int_tpe_kernel");
    return CSG_OK;
  }
  const int ev = int_stream_ev(max_E, dtype);
  if (ev == 0)
    return csg_fail(ctx, CSG_ERR_ARG, "integer stream kernel cannot handle E=%d: use CSG_K1_GENERIC for this table", max_E);
  if (!d_runs) return csg_fail(ctx, CSG_ERR_ARG, "d_runs is NULL for the stream kernel");
  const int threads = kTileRows * ev;
  const size_t smem = (size_t)max_E * kOutPitch * sizeof(double);
  auto stream = [&](auto kern) -> int {
    if (smem > 48 * 1024) CSG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<total_blocks, threads, smem, ctx->stream>>>(d_files, n_files, d_runs, d_pa_bits, n_groups, d_sums, d_row_flags);
    return CSG_OK;
  };
  if constexpr (sizeof(I) == 1) {
    if (n_groups > 4) return csg_fail(ctx, CSG_ERR_ARG, "8-bit cubes with more than 4 groups take CSG_K1_GENERIC");
    st = n_groups == 0 ? stream(collapse_int_stream_kernel<I, 0>) : stream(collapse_int_stream_kernel<I, 4>);
  } else {
    st = n_groups == 0   ? stream(collapse_int_stream_kernel<I, 0>)
         : n_groups <= 4 ? stream(collapse_int_stream_kernel<I, 4>)
                         : stream(collapse_int_stream_kernel<I, CSG_MAX_GROUPS>);
  }
  if (st != CSG_OK) return st;
  CSG_LAUNCH_CHECK(ctx, "collapse_int_stream_kernel");
  return CSG_OK;
}

int launch_int_dtype(csg_ctx* ctx, int dtype, int layout, int kernel, const csg_file_desc* d_files, int n_files,
                     int total_blocks, const uint8_t* d_pa_bits, const int32_t* d_runs, int n_groups, int max_P, int max_E,
                     double* d_sums, uint8_t* d_row_flags) {
#define CSG_INT(CODE, TYPE) \
  case CODE:                \
    return launch_int<TYPE>(ctx, layout, kernel, d_files, n_files, total_blocks, d_pa_bits, d_runs, n_groups, max_P, max_E, dtype, d_sums, d_row_flags);
  switch (dtype) {
    CSG_INT(CSG_I8, int8_t)
    CSG_INT(CSG_U8, uint8_t)
    CSG_INT(CSG_I16, int16_t)
    CSG_INT(CSG_U16, uint16_t)
    CSG_INT(CSG_I32, int32_t)
    CSG_INT(CSG_U32, uint32_t)
  }
#undef CSG_INT
  return csg_fail(ctx, CSG_ERR_ARG, "bad dtype %d", dtype);
}

}  // namespace

extern "C" {

int csg_collapse_kernel(int32_t T, int32_t P, int32_t E, int dtype, int layout, const void* d_cube) {
  return csg_collapse_kernel_for(T, P, E, dtype, layout, d_cube, /*n_groups: unknown, assume some*/ 1);
}

int csg_collapse_kernel_for(int32_t T, int32_t P, int32_t E, int dtype, int layout, const void* d_cube, int n_groups) {
  if (is_int_dtype(dtype))  // stored (T,E,P) integer views always take the row kernel
    return layout == CSG_LAYOUT_TEP || int_stream_file_ok(T, P, E, dtype, d_cube, n_groups) ? CSG_K1_STREAM : CSG_K1_GENERIC;
  if (layout == CSG_LAYOUT_TEP) return tep_rows_ok(T, P, E, d_cube, n_groups) ? CSG_K1_STREAM : CSG_K1_GENERIC;
  return stream_file_ok(T, P, E, dtype, d_cube) ? CSG_K1_STREAM : CSG_K1_GENERIC;
}

// runs of constant group membership along the pitch axis: {p0, p1, mask} triples with the
// groups that hold every bin (returned in *alias) cleared from the masks
int csg_pitch_runs(const uint8_t* h_pa_bits, int P, int n_groups, int32_t* h_runs, int32_t* alias) {
  unsigned all = n_groups > 0 ? ((1u << n_groups) - 1u) : 0u;
  for (int p = 0; p < P; ++p) all &= h_pa_bits ? h_pa_bits[p] : 0u;
  auto bits = [&](int p) { return (unsigned)((h_pa_bits && n_groups > 0) ? h_pa_bits[p] : 0u) & ((1u << n_groups) - 1u); };
  int n = 0, start = 0;
  for (int p = 1; p <= P; ++p)
    if (p == P || bits(p) != bits(start)) {
      h_runs[3 * n] = start, h_runs[3 * n + 1] = p, h_runs[3 * n + 2] = (int32_t)(bits(start) & ~all);
      ++n, start = p;
    }
  if (alias) *alias = (int32_t)all;
  return n;
}

int32_t csg_collapse_blocks(int32_t T, int32_t P, int32_t E, int dtype, int layout, int kernel) {
  if (T <= 0 || E <= 0) return 0;
  if (is_int_dtype(dtype)) {
    if (layout == CSG_LAYOUT_TEP) {
      const int rows = kBlock / int_tep_lanes(P);
      return (int32_t)(((long long)T * E + rows - 1) / rows);
    }
    if (kernel == CSG_K1_STREAM) return (T + kTileRows - 1) / kTileRows;
    return (int32_t)(((long long)T * E + kBlock - 1) / kBlock);
  }
  if (layout == CSG_LAYOUT_TEP) {
    if (kernel == CSG_K1_STREAM) return (T + kTepTile - 1) / kTepTile;
    const int rows = tep_rows_per_block(P, dtype);
    return (int32_t)(((long long)T * E + rows - 1) / rows);
  }
  if (kernel == CSG_K1_STREAM) return (T + kTileRows - 1) / kTileRows;
  const int vec = dtype == CSG_F64 ? 2 : 4;
  const long long items = (long long)T * ((E + vec - 1) / vec);
  return (int32_t)((items + kBlock - 1) / kBlock);
}

int64_t csg_sums_elems(int32_t T, int32_t E, int n_groups) {
  if (T <= 0 || E <= 0) return 0;
  return (int64_t)(n_groups + 1) * E * ((T + 3) & ~3);
}

int csg_collapse(csg_ctx* ctx, const csg_file_desc* d_files, int n_files, int total_blocks,
                 const uint8_t* d_pa_bits, const int32_t* d_runs, int n_groups, int max_P, int max_E, int dtype,
                 int layout, int kernel, void* d_sums, uint8_t* d_row_flags) {
  if (!ctx) return CSG_ERR_ARG;
  if (n_groups < 0 || n_groups > CSG_MAX_GROUPS) return csg_fail(ctx, CSG_ERR_ARG, "n_groups %d out of range", n_groups);
  if (n_groups > 0 && !d_pa_bits) return csg_fail(ctx, CSG_ERR_ARG, "d_pa_bits is NULL with n_groups > 0");
  if (dtype != CSG_F32 && dtype != CSG_F64 && !is_int_dtype(dtype)) return csg_fail(ctx, CSG_ERR_ARG, "bad dtype %d", dtype);
  if (layout != CSG_LAYOUT_TPE && layout != CSG_LAYOUT_TEP) return csg_fail(ctx, CSG_ERR_ARG, "bad layout %d", layout);
  if (n_files <= 0 || total_blocks <= 0) return CSG_OK;
  if (!d_files || !d_sums) return csg_fail(ctx, CSG_ERR_ARG, "NULL table or output");
  if (max_P <= 0 || max_P > 32768) return csg_fail(ctx, CSG_ERR_ARG, "max_P %d out of range (1..32768)", max_P);
  if (is_int_dtype(dtype))
    return launch_int_dtype(ctx, dtype, layout, kernel, d_files, n_files, total_blocks, d_pa_bits, d_runs, n_groups, max_P,
                            max_E, (double*)d_sums, d_row_flags);
  if (layout == CSG_LAYOUT_TPE) {
    if (kernel == CSG_K1_STREAM) {
      if (!d_runs) return csg_fail(ctx, CSG_ERR_ARG, "d_runs is NULL for the stream kernel");
      if (dtype == CSG_F32)
        return launch_stream<float>(ctx, max_E, dtype, d_files, n_files, total_blocks, d_runs, d_pa_bits, n_groups,
                                    (float*)d_sums, d_row_flags);
      return launch_stream<double>(ctx, max_E, dtype, d_files, n_files, total_blocks, d_runs, d_pa_bits, n_groups,
                                   (double*)d_sums, d_row_flags);
    }
    if (dtype == CSG_F32)
      return launch_tpe<float>(ctx, d_files, n_files, total_blocks, d_pa_bits, n_groups, max_P, (float*)d_sums, d_row_flags);
    return launch_tpe<double>(ctx, d_files, n_files, total_blocks, d_pa_bits, n_groups, max_P, (double*)d_sums, d_row_flags);
  }
  if (kernel == CSG_K1_STREAM) {  // the row kernel: total only, 8 <= P <= 128, P % 8 == 0 (csg_collapse_kernel_for)
    if (n_groups != 0 || max_P > 128 || max_P % 8 != 0)
      return csg_fail(ctx, CSG_ERR_ARG, "the TEP row kernel needs n_groups = 0 and P a multiple of 8 up to 128");
    const size_t smem = (size_t)max_E * (kTepTile + 1) * (dtype == CSG_F64 ? 8 : 4);
    if (dtype == CSG_F32) {
      cudaFuncSetAttribute(collapse_tep_rows_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      collapse_tep_rows_kernel<float><<<total_blocks, 256, smem, ctx->stream>>>(d_files, n_files, (float*)d_sums, d_row_flags);
    } else {
      cudaFuncSetAttribute(collapse_tep_rows_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      collapse_tep_rows_kernel<double><<<total_blocks, 256, smem, ctx->stream>>>(d_files, n_files, (double*)d_sums, d_row_flags);
    }
    CSG_LAUNCH_CHECK(ctx, "collapse_tep_rows_kernel");
    return CSG_OK;
  }
  if (dtype == CSG_F32)
    return launch_tep<float>(ctx, d_files, n_files, total_blocks, d_pa_bits, n_groups, max_P, dtype, (float*)d_sums, d_row_flags);
  return launch_tep<double>(ctx, d_files, n_files, total_blocks, d_pa_bits, n_groups, max_P, dtype, (double*)d_sums, d_row_flags);
}

int csg_window_any(csg_ctx* ctx, const uint8_t* d_row_flags, const csg_flag_window* d_windows, int n_windows,
                   const int32_t* d_index_pool, uint8_t* d_out) {
  if (!ctx) return CSG_ERR_ARG;
  if (n_windows <= 0) return CSG_OK;
  if (!d_row_flags || !d_windows || !d_out) return csg_fail(ctx, CSG_ERR_ARG, "NULL argument");
  const int blocks = (n_windows * 32 + 255) / 256;
  window_any_kernel<<<blocks, 256, 0, ctx->stream>>>(d_row_flags, d_windows, n_windows, d_index_pool, d_out);
  CSG_LAUNCH_CHECK(ctx, "window_any_kernel");
  return CSG_OK;
}

int csg_collapse_host(csg_ctx* ctx, const void* h_cube, int32_t T, int32_t P, int32_t E, int dtype, int layout,
                      const uint8_t* h_pa_bits, int n_groups, void* h_sums, uint8_t* h_row_flags) {
  if (!ctx) return CSG_ERR_ARG;
  if (T < 0 || P <= 0 || E <= 0) return csg_fail(ctx, CSG_ERR_ARG, "bad cube shape (%d,%d,%d)", T, P, E);
  if (dtype != CSG_F32 && dtype != CSG_F64 && !is_int_dtype(dtype)) return csg_fail(ctx, CSG_ERR_ARG, "bad dtype %d", dtype);
  if (T == 0) return CSG_OK;
  const size_t es = sums_itemsize(dtype);  // an integer cube's sums are float64
  const size_t cube_bytes = (size_t)T * P * E * cube_itemsize(dtype);
  const int Tp = (T + 3) & ~3;
  const size_t sums_bytes = (size_t)csg_sums_elems(T, E, n_groups) * es;
  const size_t flag_bytes = ((size_t)T + 3) & ~size_t(3);
  void *d_cube = nullptr, *d_sums = nullptr, *d_flags = nullptr, *d_bits = nullptr, *d_desc = nullptr, *d_runs = nullptr;
  int st = CSG_OK;
  auto cleanup = [&]() {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(d_cube), cudaFree(d_sums), cudaFree(d_flags), cudaFree(d_bits), cudaFree(d_desc), cudaFree(d_runs);
  };
#define CSG_TRY(x)            \
  if ((st = (x)) != CSG_OK) { \
    cleanup();                \
    return st;                \
  }
  CSG_TRY(csg_dev_alloc(ctx, cube_bytes, &d_cube));
  CSG_TRY(csg_dev_alloc(ctx, sums_bytes, &d_sums));
  CSG_TRY(csg_dev_alloc(ctx, flag_bytes, &d_flags));
  CSG_TRY(csg_dev_alloc(ctx, (size_t)P, &d_bits));
  CSG_TRY(csg_dev_alloc(ctx, sizeof(csg_file_desc), &d_desc));
  CSG_TRY(csg_dev_alloc(ctx, (size_t)(3 * P + 3) * sizeof(int32_t), &d_runs));
  csg_file_desc desc;
  memset(&desc, 0, sizeof(desc));
  desc.d_cube = d_cube;
  desc.T = T, desc.P = P, desc.E = E;
  std::vector<int32_t> h_runs((size_t)3 * P + 3);
  int32_t alias = 0;
  desc.reserved[0] = 0;
  desc.reserved[1] = csg_pitch_runs(h_pa_bits, P, n_groups, h_runs.data(), &alias);
  desc.reserved[2] = alias;
  CSG_TRY(csg_h2d(ctx, d_runs, h_runs.data(), h_runs.size() * sizeof(int32_t)));
  const int kernel = csg_collapse_kernel_for(T, P, E, dtype, layout, d_cube, is_int_dtype(dtype) ? n_groups : 1);
  const int blocks = csg_collapse_blocks(T, P, E, dtype, layout, kernel);
  CSG_TRY(csg_h2d(ctx, d_cube, h_cube, cube_bytes));
  CSG_TRY(csg_h2d(ctx, d_desc, &desc, sizeof(desc)));
  if (n_groups > 0) CSG_TRY(csg_h2d(ctx, d_bits, h_pa_bits, (size_t)P));
  CSG_TRY(csg_memset(ctx, d_flags, 0, flag_bytes));
  CSG_TRY(csg_collapse(ctx, (const csg_file_desc*)d_desc, 1, blocks, (const uint8_t*)d_bits, (const int32_t*)d_runs,
                       n_groups, P, E, dtype, layout, kernel, d_sums, (uint8_t*)d_flags));
  // the device keeps sums energy-major [g][e][Tp]; the host entry hands back numpy's (T, E)
  std::vector<unsigned char> tmp(sums_bytes);
  CSG_TRY(csg_d2h(ctx, tmp.data(), d_sums, sums_bytes));
  if (h_row_flags) CSG_TRY(csg_d2h(ctx, h_row_flags, d_flags, (size_t)T));
  CSG_TRY(csg_sync(ctx));
#undef CSG_TRY
  for (int g = 0; g <= n_groups; ++g)
    for (int e = 0; e < E; ++e) {
      const unsigned char* src = tmp.data() + ((size_t)g * E + e) * Tp * es;
      unsigned char* dst = (unsigned char*)h_sums + ((size_t)g * T * E + e) * es;
      for (int t = 0; t < T; ++t) memcpy(dst + (size_t)t * E * es, src + (size_t)t * es, es);
    }
  cleanup();
  return CSG_OK;
}

}  // extern "C"
