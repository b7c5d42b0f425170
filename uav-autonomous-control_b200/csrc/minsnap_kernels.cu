// minsnap_kernels.cu -- K1 (batched minimum-snap solve), table geometry, K3 (sampled table) and the
// sampled-point AABB test of the correction loop.  All fp64, sm_100a.
//
// K1 is one thread per mission: ~2.5 k fp64 flops against 928 B of HBM traffic for S = 4
// (SURVEY 8(d)), i.e. HBM-bound.  For S <= 8 the per-mission output (8 S x 3 doubles, contiguous) is staged in
// shared memory one or two splines at a time and leaves the CTA as whole 32-byte sectors:
//   minsnap_solve_kernel<MAXS, kStageCopy1 | kStageCopy2>  by a copy loop over the CTA's threads (any output alignment);
//   minsnap_solve_kernel<MAXS, kStageTma>                  by 2-D tensor stores (16-byte aligned output);
//   minsnap_solve_stream_kernel                            the same stores from a persistent grid that bulk-loads its inputs (S = 4).
// S > 8 stores straight from registers (kDirect), as does the ragged-S kernel of the correction loop.
#include <mutex>

#include "minsnap_core.cuh"
#include "rollout_core.cuh"
#include "tma.cuh"
#include "uavb_common.cuh"

namespace uavb {

constexpr int kSolveThreads = 64;                          // missions per CTA (per tile of the streaming kernel)
constexpr int kTmaSubTileBytes = kSolveThreads * 128;     // 64 rows x 16 doubles

// K1's tensor-store staging: the 64 x 48-double tile of two splines leaves the CTA as three 2-D tensor stores
// (cp.async.bulk.tensor.2d, boxes of 64 missions x 16 doubles over the [B][24 S] coefficient matrix) issued by one thread; it is
// staged in the 128-byte swizzle the tensor map declares (16-byte chunk c of row r at chunk c ^ (r & 7)), and rows past the end of
// the batch and the unused half of an odd last flush are clipped by the map.  NT staging tiles: splines 2k and 2k+1 are staged in
// tile k % NT.  With one tile, the flush waits until the store has read it; with two, it waits for the store that read the OTHER
// tile (a whole tile ago), and the kernel waits for the last stores itself before its shared memory goes.
template <int NT>
struct SwizzledTiles {
  char* tiles;                                            // 1024-byte aligned (the swizzle period), NT x 3 sub-tiles
  char* row;
  unsigned sw;
  __device__ __forceinline__ explicit SwizzledTiles(char* t) : tiles(t), row(t + threadIdx.x * 128), sw((threadIdx.x & 7u) << 4) {}
  __device__ __forceinline__ void store(int seg, int j, int ax, double val) const {
    const int off = (seg & 1) * 24 + j * 3 + ax, q = off >> 4, d = off & 15, tile = (seg >> 1) % NT;   // sub-tile, double within the 128-byte row
    *reinterpret_cast<double*>(row + (tile * 3 + q) * kTmaSubTileBytes + ((((unsigned)d >> 1) << 4) ^ sw) + (d & 1) * 8) = val;
  }
  __device__ __forceinline__ void flush(const CUtensorMap* tmap, int seg, int S, long long base) const {
    const bool last = seg == S - 1;
    if (!(seg & 1) && !last) return;                      // uniform: S is the same for the whole launch
    const int first = (seg & 1) ? seg - 1 : seg, n_sub = (seg & 1) ? 3 : 2, tile = (seg >> 1) % NT;   // a lone last spline fills 24 of the 48 columns
    fence_proxy_async_smem();
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int q = 0; q < n_sub; ++q) tensor_store_2d(tmap, first * 24 + q * 16, (int)base, tiles + (tile * 3 + q) * kTmaSubTileBytes);
      bulk_commit();
      if (NT == 1) bulk_wait_read<0>();                   // the tile may be overwritten (or the CTA may end) once it has been read
      else if (!last) bulk_wait_read<1>();
    }
    if (!last) __syncthreads();
  }
};

// ---------------------------------------------------------------------------------------------
// K1, uniform S.  Output staging (MODE):
//   kStageCopy1, kStageCopy2  the 24 coefficients of MODE (one or two) splines per thread go to shared memory [thread][24 MODE + 1]
//                 (odd pitch in doubles: a warp's 64-bit stores need the minimal 2 wavefronts) and leave the CTA by a copy loop after
//                 every MODE splines, consecutive threads writing consecutive doubles of each mission's 192-byte (6-sector) or
//                 384-byte (three whole 128-byte lines) chunk.  12.8 / 25 KB per CTA, so residency is limited by registers only.
//   kStageTma     two splines per flush like kStageCopy2, but the tile leaves by tensor stores (SwizzledTiles<1>).
//   kDirect       per-thread stores straight from registers (S > 8: work arrays in local memory anyway).
// Threads past the end of the batch run the solve on the last mission (they must reach the barriers) and store nothing.
enum { kDirect = 0, kStageCopy1 = 1, kStageCopy2 = 2, kStageTma = 3 };

template <int MAXS, int MODE, int MINB>
__global__ void __launch_bounds__(kSolveThreads, MINB) minsnap_solve_kernel(
    const double* __restrict__ waypoints, const double* __restrict__ velocity, int B, int S, double factor,
    double* __restrict__ coeffs_out, double* __restrict__ times_out, int* __restrict__ status_out, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ double s_out[];
  const int per = 24 * S;              // doubles per mission
  const long long base = (long long)blockIdx.x * kSolveThreads;
  const long long b = base + threadIdx.x;
  const bool live = b < B;
  const long long bb = live ? b : (long long)B - 1;
  const int n_here = (int)((B - base) < kSolveThreads ? (B - base) : kSolveThreads);
  const double* w = waypoints + (size_t)bb * (S + 1) * 3;
  double* tout = times_out + (size_t)bb * S;
  auto loadw = [w](int i, int ax) { return __ldg(w + 3 * i + ax); };
  auto storet = [tout, live](int seg, double t) { if (live) tout[seg] = t; };
  int st;
  if constexpr (MODE == kStageCopy1 || MODE == kStageCopy2) {
    constexpr int P = MODE, pitch = 24 * P + 1;          // splines per flush
    double* mine = s_out + (size_t)threadIdx.x * pitch;
    double* gout = coeffs_out + (size_t)base * per;
    st = minsnap_solve_one<MAXS>(
        S, velocity[bb], factor, loadw, [mine](int seg, int j, int ax, double val) { mine[(seg % P) * 24 + j * 3 + ax] = val; }, storet,
        [&](int seg) {
          if (seg % P != P - 1 && seg != S - 1) return;    // uniform: S is the same for the whole launch
          const int first = seg - seg % P, cnt = (seg % P + 1) * 24;
          __syncthreads();
          for (int e = threadIdx.x; e < n_here * cnt; e += kSolveThreads) {
            const int m = e / cnt, off = e - m * cnt;
            gout[(size_t)m * per + first * 24 + off] = s_out[m * pitch + off];
          }
          __syncthreads();
        });
  } else if constexpr (MODE == kStageTma) {
    const SwizzledTiles<1> tiles(reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(s_out) + 1023) & ~(uintptr_t)1023));   // 1024-byte aligned
    st = minsnap_solve_one<MAXS>(
        S, velocity[bb], factor, loadw, [tiles](int seg, int j, int ax, double val) { tiles.store(seg, j, ax, val); }, storet,
        [&](int seg) { tiles.flush(&tmap, seg, S, base); });
  } else {
    double* mine = coeffs_out + (size_t)bb * per;
    st = minsnap_solve_one<MAXS>(S, velocity[bb], factor, loadw, [mine, live](int seg, int j, int ax, double val) { if (live) mine[seg * 24 + j * 3 + ax] = val; },
                                 storet);
  }
  if (live && status_out) status_out[b] = st;
}

// K1, streaming form (S <= 8, tensor-map output): a persistent grid of CTAs walks the 64-mission tiles.  Every global access of
// the tile is asynchronous: the NEXT tile's waypoints and velocities (64 x 24 (S+1) + 512 contiguous bytes) arrive by bulk copy
// (cp.async.bulk, completion on an mbarrier) while the current tile is solved, and the coefficients leave by tensor stores as in
// kStageTma.  The one-shot kernels above start every CTA with a dependent global load of its waypoints (ncu: 4.2 long-scoreboard
// stall cycles per issued instruction at 11 warps per SM); here a CTA waits for memory once, at its first tile.
constexpr int kStreamCtasPerSm = 4;
template <int MAXS, int MINB>
__global__ void __launch_bounds__(kSolveThreads, MINB) minsnap_solve_stream_kernel(
    const double* __restrict__ waypoints, const double* __restrict__ velocity, int B, int S, double factor, double* __restrict__ times_out,
    int* __restrict__ status_out, const __grid_constant__ CUtensorMap tmap) {
  // Dynamic shared memory only (so that it starts 1024-byte aligned, as the 128-byte swizzle of the tensor stores needs): TWO staging
  // tiles of three 8 KB sub-tiles -- splines 0-1 and 2-3 of a tile leave from different ones, so nobody waits for the TMA unit to
  // drain a tile before the next pair of splines is staged (the kernel is bound by HBM writes: that read-out waits for the write
  // queue) --, then the waypoints of the next tile, then the mbarrier: 56 840 bytes at S = 4, four CTAs per SM.
  extern __shared__ __align__(1024) double s_out[];
  const SwizzledTiles<2> tiles(reinterpret_cast<char*>(s_out));
  double* s_wp = reinterpret_cast<double*>(tiles.tiles + 6 * kTmaSubTileBytes);       // [64][3 (S+1)]
  const int wpd = 3 * (S + 1);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_wp + kSolveThreads * 3 * (MAXS + 1));   // (a fixed place: behind the largest waypoint tile)
  if ((smem_u32(tiles.tiles) & 1023u) != 0u) __trap();     // the staging tiles must sit on the swizzle period
  const int n_tiles = (B + kSolveThreads - 1) / kSolveThreads;
  // the waypoints of tile t: one bulk copy when the tile is whole, a cooperative copy for the ragged last tile (a bulk copy
  // needs a multiple of 16 bytes, 64 missions always are); the velocity of a thread's next mission travels in a register
  auto prefetch = [&](int tile) {                         // thread 0
    if ((long long)(tile + 1) * kSolveThreads > B) return;
    const uint32_t wp_bytes = (uint32_t)(kSolveThreads * wpd * 8);
    mbar_expect_tx(s_bar, wp_bytes);
    bulk_load_1d(s_wp, waypoints + (size_t)tile * kSolveThreads * wpd, wp_bytes, s_bar);
  };
  auto velocity_of = [&](int tile) {                      // this thread's mission of `tile` (the tile's first one past the end of the batch)
    if (tile >= n_tiles) return 0.0;
    const long long m = (long long)tile * kSolveThreads + threadIdx.x;
    return __ldg(velocity + (m < B ? m : (long long)tile * kSolveThreads));
  };
  if (threadIdx.x == 0) {
    mbar_init(s_bar, 1);
    if ((int)blockIdx.x < n_tiles) prefetch(blockIdx.x);
  }
  double vel_next = velocity_of(blockIdx.x);
  __syncthreads();
  unsigned phase = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long base = (long long)tile * kSolveThreads;
    const int n_here = (int)((B - base) < kSolveThreads ? (B - base) : kSolveThreads);
    const bool live = (int)threadIdx.x < n_here;
    if (n_here == kSolveThreads) {
      mbar_wait(s_bar, phase);
      phase ^= 1u;
    } else {                                              // ragged last tile (the last iteration of one CTA)
      for (int e = threadIdx.x; e < n_here * wpd; e += kSolveThreads) s_wp[e] = __ldg(waypoints + (size_t)base * wpd + e);
      __syncthreads();
    }
    // this thread's mission into registers (threads past the end of the batch solve the tile's first mission and store nothing)
    const int src = live ? threadIdx.x : 0;
    double wreg[3 * (MAXS + 1)];
#pragma unroll
    for (int k = 0; k < 3 * (MAXS + 1); ++k)
      if (k < wpd) wreg[k] = s_wp[src * wpd + k];
    const double vel = vel_next;
    vel_next = velocity_of(tile + (int)gridDim.x);        // in flight during this tile's solve
    if (threadIdx.x == 0) bulk_wait_read<1>();            // ... and the store that last read the FIRST staging tile (two stores ago) is done with it
    __syncthreads();                                      // the input buffer is free: fetch the tile this CTA solves next
    if (threadIdx.x == 0 && tile + (int)gridDim.x < n_tiles) prefetch(tile + gridDim.x);
    double* tout = times_out + (size_t)(base + src) * S;
    const int st = minsnap_solve_one<MAXS>(
        S, vel, factor, [&wreg](int i, int ax) { return wreg[3 * i + ax]; },
        [tiles](int seg, int j, int ax, double val) { tiles.store(seg, j, ax, val); },
        [tout, live](int seg, double t) { if (live) tout[seg] = t; },
        [&](int seg) { tiles.flush(&tmap, seg, S, base); });
    if (live && status_out) status_out[base + threadIdx.x] = st;
  }
  if (threadIdx.x == 0) bulk_wait_read<0>();              // shared memory must outlive the last store's read
}

// K1, ragged S (obstacle-correction loop): per-thread direct stores, packed segments.
template <int MAXS>
__global__ void __launch_bounds__(kSolveThreads) minsnap_solve_ragged_kernel(
    const double* __restrict__ waypoints, const int* __restrict__ wp_offsets, const double* __restrict__ velocity, int B,
    double factor, double* __restrict__ coeffs_out, double* __restrict__ times_out, int* __restrict__ status_out) {
  const long long b = (long long)blockIdx.x * kSolveThreads + threadIdx.x;
  if (b >= B) return;
  const int w0 = wp_offsets[b], w1 = wp_offsets[b + 1];
  const int S = w1 - w0 - 1;
  const int seg0 = w0 - (int)b;
  if (S < 1 || S > MAXS) {
    if (status_out) status_out[b] = UAVB_SOLVE_DEGENERATE;
    return;
  }
  const double* w = waypoints + (size_t)w0 * 3;
  double* cout = coeffs_out + (size_t)seg0 * 24;
  double* tout = times_out + seg0;
  const int st = minsnap_solve_one<MAXS>(
      S, velocity[b], factor, [w](int i, int ax) { return __ldg(w + 3 * i + ax); },
      [cout](int seg, int j, int ax, double val) { cout[seg * 24 + j * 3 + ax] = val; },
      [tout](int seg, double t) { tout[seg] = t; });
  if (status_out) status_out[b] = st;
}

// ---------------------------------------------------------------------------------------------
// Table geometry: rows per segment and the look-ahead yaw of every table (minimum_snap.py:104,126-136).
// len(np.arange(0, T, dt)): arange_len (minsnap_core.cuh).

// Horizontal velocity of a table row by the nested Horner recurrence of eval_row (flight_core.cuh): the same operations on the
// same values, so every kernel that decides "is this row's yaw valid" (table geometry, K3, the set-point table of K2 and K2's
// on-the-fly evaluation) sees the same bits.  Validity is the exact squared-speed form of rollout_core.cuh.
__device__ __forceinline__ void eval_vel_xy(const double* __restrict__ c, double t, double* vx, double* vy) {
  double v[2];
#pragma unroll
  for (int ax = 0; ax < 2; ++ax) {
    double pp = __ldg(c + 21 + ax), d1 = 0.0;
#pragma unroll
    for (int k = 6; k >= 0; --k) {
      d1 = fma(d1, t, pp);
      pp = fma(pp, t, __ldg(c + 3 * k + ax));
    }
    v[ax] = d1;
  }
  *vx = v[0]; *vy = v[1];
}

__device__ __forceinline__ bool yaw_valid(double vx, double vy) { return speed2_unfused(vx, vy) >= kSpeed2Min; }

// atan2 for the heading of a table row (np.arctan2(vy, vx), minimum_snap.py:133), for inputs that passed yaw_valid (never both zero).
// The library atan2 costs K3 a fifth of its instructions in 32-bit moves that materialise its polynomial constants (ncu: UMOV +
// IMAD.MOV 22 % of the kernel); here the coefficients are constant-bank operands of the DFMAs and the quotient comes from one
// reciprocal: with m = min(|x|,|y|), M = max(|x|,|y|):  w = m / M if 2 m <= M, else (m - M) / (m + M) and atan(m / M) = pi/4 + atan(w);
// |w| <= 1/2, atan(w) = w P(w^2) with a degree-12 Chebyshev fit on [0, 1/4] (max error 4e-18, generated with mpmath); then the octant
// and quadrant reflections.  Within 2 ulp of the correctly rounded result.
__constant__ double kAtanPoly[13] = {0.010030841489968486489,  -0.027302779603074175199, 0.041775850326747944004, -0.05118531938647954336,
                                     0.058574357651656937953,  -0.066636678441838564357, 0.076920579899766187704, -0.090908950580923122328,
                                     0.11111110602305970347,   -0.14285714274692063502,  0.19999999999875543348,  -0.33333333333332779631,
                                     1.0};
__device__ __forceinline__ double rcp_f64(double d) {       // d > 0, normal range
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));     // ~20 bits, two Newton steps
  double e = fma(-d, r, 1.0);
  r = fma(r, e, r);
  e = fma(-d, r, 1.0);
  return fma(r, e, r);
}
__device__ __forceinline__ double atan2_row(double y, double x) {
  const double ax = fabs(x), ay = fabs(y);
  const double mx = fmax(ax, ay), mn = fmin(ax, ay);
  const bool upper = mn + mn > mx;
  const double num = upper ? mn - mx : mn, den = upper ? mn + mx : mx;
  const double r = rcp_f64(den);
  double w = num * r;
  w = fma(fma(-w, den, num), r, w);                          // the quotient to ~1 ulp
  const double z = w * w;
  double p = kAtanPoly[0];
#pragma unroll
  for (int k = 1; k < 13; ++k) p = fma(p, z, kAtanPoly[k]);
  double a = fma(w, p, upper ? 0.78539816339744830962 : 0.0);
  a = (ay > ax) ? 1.57079632679489661923 - a : a;
  a = (x < 0.0) ? 3.14159265358979323846 - a : a;
  return copysign(a, y);
}

__global__ void __launch_bounds__(128) table_meta_kernel(const double* __restrict__ coeffs, const double* __restrict__ times,
                                                         const int* __restrict__ seg_offsets, int B, double dt,
                                                         int* __restrict__ rows_out, double* __restrict__ yaw0_out,
                                                         int* __restrict__ total_rows_out) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int s0 = seg_offsets[b], s1 = seg_offsets[b + 1];
  int total = 0;
  double yaw0 = 0.0;
  bool found = false;
  for (int s = s0; s < s1; ++s) {
    const int n = arange_len(times[s], dt);
    rows_out[s] = n;
    total += n;
    if (!found) {
      const double* c = coeffs + (size_t)s * 24;
      for (int j = 0; j < n; ++j) {
        double vx, vy;
        eval_vel_xy(c, (double)j * dt, &vx, &vy);
        if (yaw_valid(vx, vy)) { yaw0 = atan2_row(vy, vx); found = true; break; }
      }
    }
  }
  yaw0_out[b] = yaw0;
  if (total_rows_out) total_rows_out[b] = total;
}

// The same with one WARP per mission, for small batches (a shared mission's two tables): the thread-per-mission kernel walks a
// vertical take-off's rows one by one looking for a valid heading that never comes (~15 us for one mission); here the lanes take 32
// rows at a time.  Same values: the same row evaluation, the first valid row in row order.
__global__ void __launch_bounds__(128) table_meta_warp_kernel(const double* __restrict__ coeffs, const double* __restrict__ times,
                                                              const int* __restrict__ seg_offsets, int B, double dt,
                                                              int* __restrict__ rows_out, double* __restrict__ yaw0_out,
                                                              int* __restrict__ total_rows_out) {
  const int lane = threadIdx.x & 31;
  const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= B) return;
  const unsigned full = 0xffffffffu;
  const int s0 = seg_offsets[b], s1 = seg_offsets[b + 1];
  int total = 0;
  double yaw0 = 0.0;
  bool found = false;
  for (int s = s0; s < s1; ++s) {
    const int n = arange_len(times[s], dt);
    if (lane == 0) rows_out[s] = n;
    total += n;
    const double* c = coeffs + (size_t)s * 24;
    for (int base = 0; base < n && !found; base += 32) {
      const int j = base + lane;
      double vx = 0.0, vy = 0.0;
      bool valid = false;
      if (j < n) {
        eval_vel_xy(c, (double)j * dt, &vx, &vy);
        valid = yaw_valid(vx, vy);
      }
      const unsigned bal = __ballot_sync(full, valid);
      if (bal) {
        const int src = __ffs(bal) - 1;
        const double y = valid ? atan2_row(vy, vx) : 0.0;
        yaw0 = __shfl_sync(full, y, src);
        found = true;
      }
    }
  }
  if (lane == 0) {
    yaw0_out[b] = yaw0;
    if (total_rows_out) total_rows_out[b] = total;
  }
}

// ---------------------------------------------------------------------------------------------
// K3 sampled table, one pass, one warp per mission.  The lanes take 32 consecutive rows (across spline boundaries),
// evaluate position / velocity / acceleration, and resolve the yaw column with warp scans that carry their state from
// chunk to chunk: np.unwrap over the valid rows is raw + cumsum(correction) (a prefix sum), hold-last-valid is a
// fill-forward from the nearest valid lane, and rows before the first valid row take the first valid yaw, found by a
// short velocity-only pre-scan (minimum_snap.py:126-136).  Each 32 x 11 tile is staged in shared memory (two buffers per warp) and
// leaves as ONE bulk asynchronous copy (cp.async.bulk, 2 816 contiguous bytes) issued by lane 0 while the warp evaluates the next
// 32 rows; a bulk copy needs 16-byte alignment at both ends and rows are 88 bytes, so a mission that starts on an odd table row
// stages its tile 8 bytes up and writes its first row -- and a chunk with an odd row count its last row -- with plain stores.
constexpr int kSampleWarps = 1;
constexpr int kTileDoubles = 32 * 11 + 2;                  // + the 8-byte shift, rounded to 16 bytes

struct RowEval {
  double p[3], v[3], a[3];
};

__device__ __forceinline__ void eval_table_row(const double* __restrict__ c, double t, RowEval& r, bool vel_only) {
  if (vel_only) {
    eval_vel_xy(c, t, &r.v[0], &r.v[1]);
  } else {
    eval_row([c](int i) { return __ldg(c + i); }, t, r.p, r.v, r.a);
  }
}

__global__ void __launch_bounds__(32 * kSampleWarps, 32 / kSampleWarps) sample_table_kernel(const double* __restrict__ coeffs, const int* __restrict__ seg_offsets,
                                                                         const int* __restrict__ seg_rows, const int* __restrict__ row_offsets,
                                                                         int B, double dt, double* __restrict__ table) {
  __shared__ __align__(16) double s_tile[kSampleWarps][2][kTileDoubles];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= B) return;
  const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
  const double two_pi = 6.283185307179586476925286766559, pi = 3.141592653589793238462643383279;
  const int s0 = seg_offsets[b], s1 = seg_offsets[b + 1];
  const long long row0 = row_offsets[b];
  const int N = (int)(row_offsets[b + 1] - row0);
  // rows before the first 16-byte aligned one: a row is 11 doubles, so the parity of (table address / 8 + first row) decides
  const int head = (int)(((reinterpret_cast<uintptr_t>(table) >> 3) + (unsigned long long)row0) & 1ull);
  int buf = 0;

  // segment cursor shared by the warp: segment `cs` starts at mission row `cf`
  auto locate = [&](int g, int& s, int& f) {           // advance (s, f) until row g lies in segment s
    while (s < s1 - 1 && g >= f + seg_rows[s]) { f += seg_rows[s]; ++s; }
  };

  // ---- pre-scan: the first valid yaw (look-ahead value of the leading rows); zeros when no row is valid
  double first_yaw = 0.0;
  bool any_valid = false;
  {
    int cs = s0, cf = 0;
    for (int base = 0; base < N && !any_valid; base += 32) {
      int s = cs, f = cf;
      const int g = base + lane;
      bool valid = false;
      double raw = 0.0;
      if (g < N) {
        locate(g, s, f);
        RowEval r;
        eval_table_row(coeffs + (size_t)s * 24, (double)(g - f) * dt, r, true);
        valid = yaw_valid(r.v[0], r.v[1]);
        if (valid) raw = atan2_row(r.v[1], r.v[0]);
      }
      const unsigned bal = __ballot_sync(full, valid);
      if (bal) { first_yaw = __shfl_sync(full, raw, __ffs(bal) - 1); any_valid = true; }
      locate(base + 31 < N ? base + 31 : N - 1, cs, cf);   // warp-uniform cursor for the next chunk
    }
  }

  // ---- main pass.  The warp's cursor (segment cs starts at mission row cf and has cn rows) sits in registers: a chunk that lies
  // inside one segment -- most do, a spline has 100-250 rows -- walks no seg_rows (ncu: the cursor walk was 6 % of the kernel's
  // instructions and 10 % of its stall samples).  Caching the 24 coefficients per lane as well was measured slower (113 registers:
  // 16 instead of 28 warps per SM, 1.29 ms).
  int cs = s0, cf = 0, cn = N > 0 ? seg_rows[s0] : 0;
  bool have_prev = false;
  double prev_raw = 0.0, cum = 0.0, hold = first_yaw;
  for (int base = 0; base < N; base += 32) {
    int s = cs, f = cf;
    const int g = base + lane;
    const bool active = g < N;
    bool valid = false;
    double raw = 0.0;
    RowEval r;
    if (active) {
      if (g >= cf + cn) locate(g, s, f);                   // past the warp's segment (only in chunks that straddle a boundary)
      eval_table_row(coeffs + (size_t)s * 24, (double)(g - f) * dt, r, false);
      valid = yaw_valid(r.v[0], r.v[1]);
      if (valid) raw = atan2_row(r.v[1], r.v[0]);
    }
    const unsigned bal = __ballot_sync(full, valid);
    // np.unwrap on the valid rows: dd against the previous valid row (in this chunk or carried), correction where |dd| >= pi
    const unsigned before = bal & lt;
    const int pv = before ? 31 - __clz(before) : -1;
    const double pr_lane = __shfl_sync(full, raw, pv >= 0 ? pv : 0);
    double corr = 0.0;
    if (valid && (pv >= 0 || have_prev)) {
      const double dd = raw - (pv >= 0 ? pr_lane : prev_raw);
      if (fabs(dd) >= pi) {                                // the only rows np.unwrap corrects; rare, so is the division
        double ddmod = dd + pi;
        ddmod = ddmod - two_pi * floor(ddmod / two_pi) - pi;
        if (ddmod == -pi && dd > 0.0) ddmod = pi;
        corr = ddmod - dd;
      }
    }
    double incl = corr;                                  // inclusive prefix sum of the corrections over the lanes
    if (__any_sync(full, corr != 0.0)) {                   // most chunks have nothing to correct
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const double up = __shfl_up_sync(full, incl, off);
        if (lane >= off) incl += up;
      }
    }
    const double y_valid = raw + (cum + incl);
    // hold-last-valid: nearest valid lane at or before this one, else the value carried from earlier chunks
    const unsigned upto = bal & (lt | (1u << lane));
    const int lv = upto ? 31 - __clz(upto) : -1;
    const double y_lane = __shfl_sync(full, y_valid, lv >= 0 ? lv : 0);
    const double yaw = any_valid ? (lv >= 0 ? y_lane : hold) : 0.0;
    if (bal) {
      const int last = 31 - __clz(bal);
      prev_raw = __shfl_sync(full, raw, last);
      hold = __shfl_sync(full, y_valid, last);
      have_prev = true;
    }
    cum += __shfl_sync(full, incl, 31);
    // ---- stage the tile and send it off
    double* tile = s_tile[wib][buf] + head;
    if (lane == 0) bulk_wait_read<1>();                    // the copy that last read this buffer (two chunks ago) is done with it
    __syncwarp();
    if (active) {
      double* o = tile + lane * 11;
      o[0] = r.p[0]; o[1] = r.p[1]; o[2] = r.p[2]; o[3] = r.v[0]; o[4] = r.v[1]; o[5] = r.v[2];
      o[6] = r.a[0]; o[7] = r.a[1]; o[8] = r.a[2]; o[9] = yaw; o[10] = (double)(s - s0);
    }
    fence_proxy_async_smem();                              // every lane: its staged row before the async-proxy read
    __syncwarp();
    const int rows_here = N - base < 32 ? N - base : 32;
    const int first = head < rows_here ? head : rows_here;                 // plain-store rows in front ...
    const int bulk_rows = (rows_here - first) & ~1;                        // ... an even number of rows by the bulk copy ...
    double* out = table + (size_t)(row0 + base) * 11;
    if (lane == 0 && bulk_rows > 0) {
      bulk_store_1d(out + first * 11, tile + first * 11, (uint32_t)bulk_rows * 88u);
      bulk_commit();
    }
    if (lane < 11) {
      if (first) out[lane] = tile[lane];
      const int last = first + bulk_rows;                                  // ... and at most one row behind
      if (last < rows_here) out[last * 11 + lane] = tile[last * 11 + lane];
    }
    buf ^= 1;
    const int g_last = base + 31 < N ? base + 31 : N - 1;
    if (g_last >= cf + cn) {                               // the warp's cursor moves on (uniform)
      locate(g_last, cs, cf);
      cn = seg_rows[cs];
    }
  }
  if (lane == 0) bulk_wait_read<0>();                      // shared memory must outlive the copies that read it
}

// `col` points at the yaw entry of row 0 and consecutive rows are `stride` doubles apart (11 inside a table, 1 for a
// bare yaw vector).
__global__ void __launch_bounds__(128) sample_yaw_kernel(const int* __restrict__ row_offsets, int B, double* __restrict__ col, int stride) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const long long r0 = row_offsets[b], r1 = row_offsets[b + 1];
  const double two_pi = 6.283185307179586476925286766559, pi = 3.141592653589793238462643383279;
  // first valid yaw (look-ahead for the leading rows)
  double first = 0.0;
  long long rf = r1;
  for (long long r = r0; r < r1; ++r) {
    const double y = col[(size_t)r * stride];
    if (y == y) { first = y; rf = r; break; }
  }
  if (rf == r1) {                       // no valid row: all zeros (minimum_snap.py:130-131)
    for (long long r = r0; r < r1; ++r) col[(size_t)r * stride] = 0.0;
    return;
  }
  double prev_raw = first, hold = first;
  for (long long r = r0; r < r1; ++r) {
    double* y = col + (size_t)r * stride;
    const double raw = *y;
    if (r > rf && raw == raw) {
      // np.unwrap: dd = raw - prev_raw; ddmod = mod(dd + pi, 2 pi) - pi, with -pi -> +pi when dd > 0;
      // correction applied only where |dd| >= pi; cumulative.
      const double dd = raw - prev_raw;
      double ddmod = dd + pi;
      ddmod = ddmod - two_pi * floor(ddmod / two_pi) - pi;
      if (ddmod == -pi && dd > 0.0) ddmod = pi;
      double corr = ddmod - dd;
      if (fabs(dd) < pi) corr = 0.0;
      hold = hold + dd + corr;
      prev_raw = raw;
    }
    *y = hold;
  }
}

// Raw heading of every velocity row: atan2(vy, vx) where the horizontal speed reaches the threshold, NaN elsewhere.
__global__ void __launch_bounds__(256) yaw_raw_kernel(const double* __restrict__ vel, long long n, double* __restrict__ yaw) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const double vx = vel[3 * r], vy = vel[3 * r + 1];
  yaw[r] = (sqrt(__dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy))) >= 1e-3) ? atan2_row(vy, vx) : nan("");
}

// Sampled-point AABB test of the correction loop (minimum_snap.py:84-87): one warp per mission.
__global__ void __launch_bounds__(128) table_hits_kernel(const double* __restrict__ table, const int* __restrict__ row_offsets, int B,
                                                         const double* __restrict__ cuboid, int cuboid_stride,
                                                         unsigned long long* __restrict__ hit_mask) {
  const int lane = threadIdx.x & 31;
  const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= B) return;
  const double* q = cuboid + (size_t)cuboid_stride * b;
  const double x0 = q[0], x1 = q[1], y0 = q[2], y1 = q[3], z0 = q[4], z1 = q[5];
  unsigned long long m = 0ull;
  for (long long r = row_offsets[b] + lane; r < row_offsets[b + 1]; r += 32) {
    const double* o = table + (size_t)r * 11;
    const double x = o[0], y = o[1], z = o[2];
    if (x0 <= x && x <= x1 && y0 <= y && y <= y1 && z0 <= z && z <= z1) m |= 1ull << ((int)o[10] & 63);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, off);
  if (lane == 0) hit_mask[b] |= m;
}

// ---------------------------------------------------------------------------------------------
// The reference's constraint system A c = b (minimum_snap.py:171-255) in its own row order, one thread per (mission, row):
//   rows [0, S)        position of spline i at t = 0        = waypoint i          (:233-239)
//   rows [S, 2S)       position of spline i at t = T_i      = waypoint i+1        (:241-248)
//   rows 2S .. 2S+2    derivatives 1..3 of the first spline at t = 0   = 0        (:215-219)
//   rows 2S+3 .. 2S+5  derivatives 1..3 of the last spline at t = T    = 0        (:221-225)
//   then, for every interior waypoint s = 1 .. S-1 and k = 1..4: polynom(k, T_{s-1}) on spline s-1 minus polynom(k, 0) on spline s (:196-204)
// polynom(n, k, t)[i] = i! / (i-k)! t^(i-k) (:258-286).  K1 never forms this system (it solves the reduced problem); the kernel
// exists for the MinimumSnap.A / .b attributes of the reference API.
__device__ __forceinline__ double basis_entry(int i, int k, double t) {
  if (i < k) return 0.0;
  double f = 1.0;
  for (int m = 0; m < k; ++m) f *= (double)(i - m);
  double p = 1.0;
  for (int m = 0; m < i - k; ++m) p *= t;
  return f * p;
}

__global__ void __launch_bounds__(128) constraint_rows_kernel(const double* __restrict__ waypoints, const double* __restrict__ times, int B, int S,
                                                              double* __restrict__ A, double* __restrict__ b) {
  const int n_rows = 6 * S + 2, n_cols = 8 * S;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (long long)B * n_rows) return;
  const int m = (int)(g / n_rows), r = (int)(g - (long long)m * n_rows);
  const double* w = waypoints + (size_t)m * (S + 1) * 3;
  const double* T = times + (size_t)m * S;
  double* row = A + (size_t)g * n_cols;
  double* rhs = b + (size_t)g * 3;
  for (int c = 0; c < n_cols; ++c) row[c] = 0.0;
  rhs[0] = rhs[1] = rhs[2] = 0.0;
  if (r < 2 * S) {
    const int i = r < S ? r : r - S;
    const double t = r < S ? 0.0 : T[i];
    for (int c = 0; c < 8; ++c) row[8 * i + c] = basis_entry(c, 0, t);
    const double* p = w + 3 * (r < S ? i : i + 1);
    rhs[0] = p[0]; rhs[1] = p[1]; rhs[2] = p[2];
  } else if (r < 2 * S + 6) {
    const int q = r - 2 * S, k = q % 3 + 1;
    const int i = q < 3 ? 0 : S - 1;
    const double t = q < 3 ? 0.0 : T[S - 1];
    for (int c = 0; c < 8; ++c) row[8 * i + c] = basis_entry(c, k, t);
  } else {
    const int q = r - 2 * S - 6, s = q / 4 + 1, k = q % 4 + 1;
    for (int c = 0; c < 8; ++c) {
      row[8 * (s - 1) + c] = basis_entry(c, k, T[s - 1]);
      row[8 * s + c] = -1.0 * basis_entry(c, k, 0.0);
    }
  }
}

template <int MAXS, int MODE, int MINB>
static int launch_solve(const double* w, const double* vel, int B, int S, double factor, double* c, double* t, int* st, cudaStream_t stream,
                        const CUtensorMap* tmap = nullptr) {
  const size_t smem = MODE == kStageTma ? (size_t)3 * kTmaSubTileBytes + 1024
                                        : (MODE == kDirect ? 0 : sizeof(double) * (size_t)kSolveThreads * (24 * MODE + 1));   // kStageCopy1/2
  CUtensorMap none = {};
  minsnap_solve_kernel<MAXS, MODE, MINB><<<div_up(B, kSolveThreads), kSolveThreads, smem, stream>>>(w, vel, B, S, factor, c, t, st, tmap ? *tmap : none);
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

// The [B][24 S] coefficient matrix as a tensor map with boxes of 64 missions x 16 doubles in the 128-byte swizzle (SwizzledTiles).
static bool coeff_tensor_map(CUtensorMap* tm, double* coeffs, int B, int S) {
  return make_tensor_map_2d(tm, coeffs, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 24ull * S, (unsigned long long)B, 192ull * S, 16, kSolveThreads,
                            CU_TENSOR_MAP_SWIZZLE_128B);
}

}  // namespace uavb

using namespace uavb;

extern "C" int uavb_minsnap_solve_f64(const double* waypoints, const double* velocity, int B, int S, double factor,
                                      double* coeffs_out, double* times_out, int* status_out, void* stream) {
  UAVB_REQUIRE(waypoints && velocity && coeffs_out && times_out, "minsnap_solve: NULL pointer");
  UAVB_REQUIRE(B >= 0, "minsnap_solve: B must be >= 0");
  UAVB_REQUIRE(S >= 1 && S <= UAVB_MAX_SPLINES, "minsnap_solve: S must be in [1, UAVB_MAX_SPLINES]");
  int rc = require_device();
  if (rc) return rc;
  if (B == 0) return UAVB_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (S == 1) return launch_solve<1, kStageCopy1, 1>(waypoints, velocity, B, S, factor, coeffs_out, times_out, status_out, st);
  if (S == 2) return launch_solve<2, kStageCopy1, 1>(waypoints, velocity, B, S, factor, coeffs_out, times_out, status_out, st);
  // S <= 4 (BASELINE configs[1]): 6 CTAs per SM (168 registers) measured fastest -- 0.216 ms per 10^6 solves against 0.250 ms
  // unconstrained (198 registers, 5 CTAs) and 0.238 ms at 8 CTAs (128 registers, spills); DESIGN.md, K1
  // ... and staging two splines at a time (384-byte chunks = whole 128-byte lines, 25 KB per CTA) 0.198 ms against 0.2026 ms
  // ... and, where the driver gives a tensor map (16-byte aligned output), the tile leaves through the TMA unit instead of a copy loop
  CUtensorMap tm;
  const bool tma = S > 2 && S <= 8 && coeff_tensor_map(&tm, coeffs_out, B, S);
  const bool streaming = tma && S == 4 &&     // measured: S = 3 is 5 % faster one-shot (6 CTAs per SM), S = 4 14 % faster streaming
                         (reinterpret_cast<uintptr_t>(waypoints) & 15u) == 0 && (reinterpret_cast<uintptr_t>(velocity) & 15u) == 0;
  if (streaming) {
    int sms = 0;
    rc = sm_count_cached(&sms);
    if (rc) return rc;
    const size_t smem = (size_t)6 * kTmaSubTileBytes + sizeof(double) * kSolveThreads * 3 * (4 + 1) + sizeof(uint64_t);   // MAXS = 4
    const int n_tiles = div_up(B, kSolveThreads);
    const int grid = n_tiles < kStreamCtasPerSm * sms ? n_tiles : kStreamCtasPerSm * sms;
    static std::once_flag attr_once[kMaxDevices];          // > 48 KB of dynamic shared memory needs the opt-in, once per device
    int dev = 0;
    UAVB_CUDA_OK(cudaGetDevice(&dev));
    cudaError_t attr_err = cudaSuccess;
    std::call_once(attr_once[dev < kMaxDevices ? dev : kMaxDevices - 1], [&] {
      attr_err = cudaFuncSetAttribute(minsnap_solve_stream_kernel<4, kStreamCtasPerSm>, cudaFuncAttributeMaxDynamicSharedMemorySize, 60 * 1024);
      if (attr_err == cudaSuccess)
        attr_err = cudaFuncSetAttribute(minsnap_solve_stream_kernel<4, kStreamCtasPerSm>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    });
    UAVB_CUDA_OK(attr_err);
    minsnap_solve_stream_kernel<4, kStreamCtasPerSm><<<grid, kSolveThreads, smem, st>>>(waypoints, velocity, B, S, factor, times_out, status_out, tm);
    UAVB_CUDA_OK(cudaGetLastError());
    return UAVB_OK;
  }
  if (S <= 4) {
    if (tma) return launch_solve<4, kStageTma, 6>(waypoints, velocity, B, S, factor, coeffs_out, times_out, status_out, st, &tm);
    return launch_solve<4, kStageCopy2, 6>(waypoints, velocity, B, S, factor, coeffs_out, times_out, status_out, st);
  }
  if (S <= 8) {
    if (tma) return launch_solve<8, kStageTma, 1>(waypoints, velocity, B, S, factor, coeffs_out, times_out, status_out, st, &tm);
    return launch_solve<8, kStageCopy1, 1>(waypoints, velocity, B, S, factor, coeffs_out, times_out, status_out, st);
  }
  return launch_solve<UAVB_MAX_SPLINES, kDirect, 1>(waypoints, velocity, B, S, factor, coeffs_out, times_out, status_out, st);
}

extern "C" int uavb_minsnap_solve_ragged_f64(const double* waypoints, const int* wp_offsets, const double* velocity, int B,
                                             double factor, double* coeffs_out, double* times_out, int* status_out, void* stream) {
  UAVB_REQUIRE(waypoints && wp_offsets && velocity && coeffs_out && times_out, "minsnap_solve_ragged: NULL pointer");
  UAVB_REQUIRE(B >= 0, "minsnap_solve_ragged: B must be >= 0");
  int rc = require_device();
  if (rc) return rc;
  if (B == 0) return UAVB_OK;
  minsnap_solve_ragged_kernel<UAVB_MAX_SPLINES><<<div_up(B, kSolveThreads), kSolveThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      waypoints, wp_offsets, velocity, B, factor, coeffs_out, times_out, status_out);
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

extern "C" int uavb_minsnap_table_meta_f64(const double* coeffs, const double* times, const int* seg_offsets, int B, double dt,
                                           int* rows_out, double* yaw0_out, int* total_rows_out, void* stream) {
  UAVB_REQUIRE(coeffs && times && seg_offsets && rows_out && yaw0_out, "table_meta: NULL pointer");
  UAVB_REQUIRE(B >= 0 && dt > 0.0, "table_meta: B >= 0 and dt > 0 required");
  int rc = require_device();
  if (rc) return rc;
  if (B == 0) return UAVB_OK;
  if (B <= 2048)
    table_meta_warp_kernel<<<div_up((long long)B * 32, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(coeffs, times, seg_offsets, B, dt, rows_out,
                                                                                                          yaw0_out, total_rows_out);
  else
    table_meta_kernel<<<div_up(B, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(coeffs, times, seg_offsets, B, dt, rows_out,
                                                                                     yaw0_out, total_rows_out);
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

extern "C" int uavb_minsnap_sample_f64(const double* coeffs, const double* times, const int* seg_offsets, const int* seg_rows,
                                       const int* row_offsets, int B, double dt, double* table_out, void* stream) {
  (void)times;
  UAVB_REQUIRE(coeffs && seg_offsets && seg_rows && row_offsets && table_out, "minsnap_sample: NULL pointer");
  UAVB_REQUIRE(B >= 0 && dt > 0.0, "minsnap_sample: B >= 0 and dt > 0 required");
  int rc = require_device();
  if (rc) return rc;
  if (B == 0) return UAVB_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  sample_table_kernel<<<div_up((long long)B * 32, 32 * kSampleWarps), 32 * kSampleWarps, 0, st>>>(coeffs, seg_offsets, seg_rows, row_offsets, B, dt,
                                                                                                  table_out);
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

extern "C" int uavb_minsnap_yaw_profile_f64(const double* velocities, const int* row_offsets, int B, long long n_rows, double* yaws_out,
                                            void* stream) {
  UAVB_REQUIRE(velocities && row_offsets && yaws_out, "yaw_profile: NULL pointer");
  UAVB_REQUIRE(B >= 0 && n_rows >= 0, "yaw_profile: B and n_rows must be >= 0");
  int rc = require_device();
  if (rc) return rc;
  if (B == 0 || n_rows == 0) return UAVB_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  yaw_raw_kernel<<<div_up(n_rows, 256), 256, 0, st>>>(velocities, n_rows, yaws_out);
  UAVB_CUDA_OK(cudaGetLastError());
  sample_yaw_kernel<<<div_up(B, 128), 128, 0, st>>>(row_offsets, B, yaws_out, 1);
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

extern "C" int uavb_minsnap_table_hits_f64(const double* table, const int* row_offsets, int B, const double* cuboid,
                                           int cuboid_stride, unsigned long long* hit_mask_out, void* stream) {
  UAVB_REQUIRE(table && row_offsets && cuboid && hit_mask_out, "table_hits: NULL pointer");
  UAVB_REQUIRE(cuboid_stride == 0 || cuboid_stride == 6, "table_hits: cuboid_stride must be 0 or 6");
  UAVB_REQUIRE(B >= 0, "table_hits: B must be >= 0");
  int rc = require_device();
  if (rc) return rc;
  if (B == 0) return UAVB_OK;
  table_hits_kernel<<<div_up((long long)B * 32, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(table, row_offsets, B, cuboid,
                                                                                                 cuboid_stride, hit_mask_out);
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}

extern "C" int uavb_minsnap_constraints_f64(const double* waypoints, const double* times, int B, int S, double* A_out, double* b_out, void* stream) {
  UAVB_REQUIRE(waypoints && times && A_out && b_out, "minsnap_constraints: NULL pointer");
  UAVB_REQUIRE(B >= 0 && S >= 1 && S <= UAVB_MAX_SPLINES, "minsnap_constraints: B >= 0 and 1 <= S <= UAVB_MAX_SPLINES required");
  int rc = require_device();
  if (rc) return rc;
  if (B == 0) return UAVB_OK;
  const long long n = (long long)B * (6 * S + 2);
  constraint_rows_kernel<<<div_up(n, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(waypoints, times, B, S, A_out, b_out);
  UAVB_CUDA_OK(cudaGetLastError());
  return UAVB_OK;
}
