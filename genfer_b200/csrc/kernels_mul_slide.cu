// Sliding 1x2-blocked DFMA kernel for the truncated N-D product (multivariate_taylor.rs:984-1012) on dense cube
// slabs: X, Y and Z have the same (b1, b2, L) slab shape, b1 even, b2 divisible by 4, L = Lc chunks of LT doubles.
//
// A thread owns TWO adjacent output rows (k1; s, s+1; chunk kc) -- s even -- in registers and walks the x rows
// a = 0, 1, .., s+1 of one x plane j1.  Step a multiplies ONE x row with the two y rows (m1; s-a) and (m1; s+1-a):
//     z[s]   += x[a] (*) y[s-a]          z[s+1] += x[a] (*) y[s+1-a]
// The second y row of step a is the first y row of step a-1, so it is kept in registers: per step the thread loads
// one x row and ONE new y row (32 doubles) for two row convolutions (272 DFMA for LT = 16) -- the shared-memory
// economy of a 2x2 block with 2 instead of 3 accumulator rows and single-writer accumulators: ~60 fewer registers
// (3 CTAs per SM instead of 2) and a DFMA stream whose pure-register ceiling is 87 % of peak instead of 80 %
// (tools/probes.cu).  The two y buffers alternate roles with the parity of the thread's step counter (the step loop is
// unrolled by two), which is the same for every thread, so warps never diverge.  Row -1 and row b2 of every y plane
// are zero rows in shared memory: the first / last step of a run needs no special case.  As in kernels_mul_blk.cu:
// chunked last axes give `lo` and `hi` row convolutions run in two phases, slabs are staged with cp.async, lanes
// are folded (k <-> D-1-k on the plane axis and on the row pairs) so that every lane executes the same number of
// steps in lockstep with conflict-free LDS.128, work units are LPT-sorted chunks of the jA box, partial rows meet in
// HBM through RED.ADD.F64.
#include "kernels.cuh"

namespace gtp {

constexpr int ST = 128;   // maximum (and untiled) CTA size; tiled plans may launch fewer threads
constexpr int S_MAXA = 6;

struct SlideP {
  int na;
  unsigned xa[S_MAXA], ya[S_MAXA], ra[S_MAXA];
  long long xastr[S_MAXA], yastr[S_MAXA];
  unsigned rows_a0;
  unsigned planes, prow;          // planes (b1) and rows per plane (b2 * Lc) of a slab in HBM
  unsigned row;                   // doubles per row in shared memory
  unsigned x_plane_sm, y_plane_sm, x_slab_sm, y_slab_sm;
  unsigned y_first;               // offset of y row 0 inside a y plane (after the leading zero rows)
  unsigned y_up_off;              // distance from y row m2 to row m2+1 (Lc * row)
  unsigned z_rows, z_up;          // rows per output slab; rows between (s) and (s+1)
  int G;
  int nsteps_lo, nsteps;          // both even
  int tiled;                      // 1: the plane axis is tiled (last A axis = tile index); units on the last tile
                                  // sum skip the SE_UPPER steps (output planes beyond the truncation)
  const uint2* table;             // [nsteps][blockDim.x]
  const uint4* units;
  const double* x;
  const double* y;
  double* out;
};

// entry: .x = xoff (20) | g << 20 (4) | z1 valid << 25 | reload << 26 | valid << 31 ; .y = yoff (20) | zrow << 20 (12)
constexpr unsigned SE_VALID = 1u << 31;
constexpr unsigned SE_RELOAD = 1u << 26;
constexpr unsigned SE_Z1 = 1u << 25;
constexpr unsigned SE_UPPER = 1u << 27;   // tiled planes: the step feeds an output plane of the NEXT plane tile

template <int LT> __device__ __forceinline__ void sl_load(double (&r)[LT], const double* __restrict__ p) {
#pragma unroll
  for (int i = 0; i < LT; i += 2) {
    double2 v = *reinterpret_cast<const double2*>(p + i);
    r[i] = v.x;
    r[i + 1] = v.y;
  }
}
// RED.ADD the accumulator row into HBM and clear it IN PLACE: the "+d" operands pin every accumulator to its register
// across the (rare, divergent) flush branch, so the merge after it costs no register moves in the hot loop (with plain
// C++ here ptxas copied all 32 accumulators on every step to set up the merge: ~36 moves + 2 spills per 272 DFMA).
template <int LT> __device__ __forceinline__ void sl_flush(double (&z)[LT], double* __restrict__ dst, bool write) {
  const int w = write ? 1 : 0;
#pragma unroll
  for (int i = 0; i < LT; i += 2) {
    asm volatile(
        "{\n\t.reg .pred pw;\n\tsetp.ne.s32 pw, %3, 0;\n\t"
        "@pw red.global.add.f64 [%2], %0;\n\t"
        "@pw red.global.add.f64 [%2+8], %1;\n\t"
        "mov.f64 %0, 0d0000000000000000;\n\t"
        "mov.f64 %1, 0d0000000000000000;\n\t}"
        : "+d"(z[i]), "+d"(z[i + 1])
        : "l"(dst + i), "r"(w)
        : "memory");
  }
}
// z0 += x (*) ya ; z1 += x (*) yb   (both `lo` or both `hi`)
template <int LT, bool HI>
__device__ __forceinline__ void sl_col(double (&z0)[LT], double (&z1)[LT], const double (&ya)[LT], const double (&yb)[LT], const double xj,
                                       const int jj) {
  if (!HI) {
#pragma unroll
    for (int kk = jj; kk < LT; kk++) z0[kk] = fma(xj, ya[kk - jj], z0[kk]);
#pragma unroll
    for (int kk = jj; kk < LT; kk++) z1[kk] = fma(xj, yb[kk - jj], z1[kk]);
  } else {
#pragma unroll
    for (int kk = 0; kk < jj; kk++) z0[kk] = fma(xj, ya[LT + kk - jj], z0[kk]);
#pragma unroll
    for (int kk = 0; kk < jj; kk++) z1[kk] = fma(xj, yb[LT + kk - jj], z1[kk]);
  }
}
// A row convolution is a triangle: column j of x feeds LT - j (lo) or j (hi) accumulators, and every accumulator is a chain of
// dependent DFMAs over j.  Walking the columns in ascending order ends (lo) or starts (hi) with a run of narrow columns whose
// FMAs depend on each other at a distance below the DFMA latency.  The columns are therefore visited from both ends alternately
// (0, LT-1, 1, LT-2, ..): a narrow column is always followed by a wide one.  The summation order differs from the reference's;
// the DFMA kernels are tolerance-level anyway (contracted multiply-adds, RED.ADD meeting order).
template <int LT, bool HI>
__device__ __forceinline__ void sl_step(double (&z0)[LT], double (&z1)[LT], const double (&ya)[LT], const double (&yb)[LT],
                                        const double* __restrict__ xs) {
  static_assert(LT % 4 == 0 || LT % 4 == 2, "even chunk");
#pragma unroll
  for (int j = 0; j < LT / 2; j += 2) {
    const double2 xa = *reinterpret_cast<const double2*>(xs + j);             // columns j, j + 1
    const int jb = LT - 2 - j;                                                // columns jb, jb + 1
    if (jb > j) {
      const double2 xb = *reinterpret_cast<const double2*>(xs + jb);
      sl_col<LT, HI>(z0, z1, ya, yb, xa.x, j);
      sl_col<LT, HI>(z0, z1, ya, yb, xb.y, jb + 1);
      sl_col<LT, HI>(z0, z1, ya, yb, xa.y, j + 1);
      sl_col<LT, HI>(z0, z1, ya, yb, xb.x, jb);
    } else {   // the middle pair of a chunk whose half is odd (LT = 10, 14)
      sl_col<LT, HI>(z0, z1, ya, yb, xa.x, j);
      sl_col<LT, HI>(z0, z1, ya, yb, xa.y, j + 1);
    }
  }
}

template <int LT, bool CHUNKED>
__global__ void __launch_bounds__(ST, 3) k_mul_slide(const SlideP p) {
  constexpr int V2 = LT / 2;
  extern __shared__ __align__(16) double smem[];
  double* Xs = smem;
  double* Ys = smem + (size_t)p.G * p.x_slab_sm;
  const int tid = threadIdx.x;
  const int ST = blockDim.x;
  const uint4 unit = p.units[blockIdx.x];
  {  // zero fill once: the leading / trailing zero rows of the y planes are never overwritten
    const int total = p.G * (int)(p.x_slab_sm + p.y_slab_sm);
    for (int i = tid * 2; i < total; i += ST * 2) *reinterpret_cast<double2*>(smem + i) = make_double2(0.0, 0.0);
  }
  unsigned k[S_MAXA], lo[S_MAXA], ext[S_MAXA];
  unsigned skip_mask = 0u;   // steps with any of these bits set are skipped
  {
    unsigned rem = unit.x;
#pragma unroll
    for (int a = S_MAXA - 1; a >= 0; --a) {
      if (a < p.na) {
        unsigned len = (a == 0) ? p.rows_a0 : p.ra[a];
        unsigned idx = rem % len;
        rem /= len;
        k[a] = (a == 0) ? unit.w : idx;
        unsigned l = (k[a] + 1 > p.ya[a]) ? k[a] + 1 - p.ya[a] : 0;
        unsigned h = (k[a] + 1 < p.xa[a]) ? k[a] + 1 : p.xa[a];
        lo[a] = l;
        ext[a] = h > l ? h - l : 0;
        if (p.tiled && a == p.na - 1 && k[a] + 1 == p.ra[a]) skip_mask = SE_UPPER;   // last plane tile: no next tile
      } else {
        k[a] = lo[a] = 0;
        ext[a] = 1;
      }
    }
  }
  double* out_slab = p.out + (size_t)unit.x * p.z_rows * LT;

  double z0[LT], z1[LT], ya[LT], yb[LT];
#pragma unroll
  for (int i = 0; i < LT; i++) z0[i] = z1[i] = ya[i] = yb[i] = 0.0;
  unsigned cur = 0xffffffffu;   // zrow << 1 | z1 valid

  for (unsigned q = unit.y; q < unit.z; q += p.G) {
    const int ng = min((unsigned)p.G, unit.z - q);
    __syncthreads();
    for (int g = 0; g < ng; g++) {
      long long xo = 0, yo = 0;
      unsigned rem = q + g;
#pragma unroll
      for (int a = S_MAXA - 1; a >= 0; --a) {
        if (a < p.na) {
          unsigned j = lo[a] + rem % ext[a];
          rem /= ext[a];
          xo += (long long)j * p.xastr[a];
          yo += (long long)(k[a] - j) * p.yastr[a];
        }
      }
      const double2* gx = reinterpret_cast<const double2*>(p.x + xo);
      const double2* gy = reinterpret_cast<const double2*>(p.y + yo);
      double* xs = Xs + (size_t)g * p.x_slab_sm;
      double* ys = Ys + (size_t)g * p.y_slab_sm + p.y_first;
      const int n = (int)(p.planes * p.prow) * V2;
      for (int i = tid; i < n; i += ST) {
        int r = i / V2, c = i - r * V2;
        int pl = r / (int)p.prow, rr = r - pl * (int)p.prow;
        cp_async16(xs + pl * p.x_plane_sm + rr * p.row + 2 * c, gx + i);
        cp_async16(ys + pl * p.y_plane_sm + rr * p.row + 2 * c, gy + i);
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();

    // table entries are fetched one step pair ahead (the table carries two trailing zero rows): their L2 latency
    // is hidden behind 544 DFMA instead of being exposed at the top of every step pair
    uint2 n0 = p.table[tid], n1 = p.table[ST + tid];
#pragma unroll
    for (int ph = 0; ph < (CHUNKED ? 2 : 1); ph++) {
      const bool hi = CHUNKED && ph == 1;
      const int s_begin = hi ? p.nsteps_lo : 0, s_end = hi ? p.nsteps : p.nsteps_lo;
      for (int s = s_begin; s < s_end; s += 2) {
        const uint2 e0 = n0, e1 = n1;
        n0 = p.table[(s + 2) * ST + tid];
        n1 = p.table[(s + 3) * ST + tid];
#pragma unroll
        for (int par = 0; par < 2; par++) {
          const uint2 e = par ? e1 : e0;
          if ((e.x & SE_VALID) && !(e.x & skip_mask) && (int)((e.x >> 20) & 15u) < ng) {
            const unsigned zkey = ((e.y >> 20) << 1) | ((e.x >> 25) & 1u);
            if (zkey != cur) {
              if (cur != 0xffffffffu) {
                double* dst = out_slab + (size_t)(cur >> 1) * LT;
                sl_flush<LT>(z0, dst, true);
                sl_flush<LT>(z1, dst + (size_t)p.z_up * LT, (cur & 1u) != 0);
              }
              cur = zkey;
            }
            const double* xs = Xs + (e.x & 0xfffffu);
            const double* ys = Ys + (e.y & 0xfffffu);
            // even step: the new (lower) y row goes to ya and pairs with z0, yb keeps the previous step's new row
            if (par == 0) {
              sl_load<LT>(ya, ys);
              if (e.x & SE_RELOAD) sl_load<LT>(yb, ys + p.y_up_off);
              if (hi) sl_step<LT, true>(z0, z1, ya, yb, xs);
              else sl_step<LT, false>(z0, z1, ya, yb, xs);
            } else {
              sl_load<LT>(yb, ys);
              if (e.x & SE_RELOAD) sl_load<LT>(ya, ys + p.y_up_off);
              if (hi) sl_step<LT, true>(z0, z1, yb, ya, xs);
              else sl_step<LT, false>(z0, z1, yb, ya, xs);
            }
          }
        }
      }
    }
  }
  if (cur != 0xffffffffu) {
    double* dst = out_slab + (size_t)(cur >> 1) * LT;
    sl_flush<LT>(z0, dst, true);
    sl_flush<LT>(z1, dst + (size_t)p.z_up * LT, (cur & 1u) != 0);
  }
}

// k_mul_slide16's step: the columns of x in ascending order, each one's 2 (16 - j) DFMAs back to back.  In this kernel
// the order is 2 % faster than sl_step's alternating one on B200 (6 x 16: 492.5 against 502.6 ms,
// profiles/r03_step_order_variants.txt); ptxas then flags 604 instead of 536 of the kernel's 952 DFMAs with an operand
// .reuse.  Interleaving z0 / z1 per accumulator was slower (514 ms).
__device__ __forceinline__ void sl16_step(double (&z0)[16], double (&z1)[16], const double (&ya)[16], const double (&yb)[16],
                                          const double* __restrict__ xs) {
#pragma unroll
  for (int jq = 0; jq < 16; jq += 2) {
    const double2 xv = *reinterpret_cast<const double2*>(xs + jq);
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int j = jq + h;
      const double xj = h ? xv.y : xv.x;
#pragma unroll
      for (int kk = j; kk < 16; kk++) z0[kk] = fma(xj, ya[kk - j], z0[kk]);
#pragma unroll
      for (int kk = j; kk < 16; kk++) z1[kk] = fma(xj, yb[kk - j], z1[kk]);
    }
  }
}
// z1 += x (*) y: the last step of a run, whose z0 partner is the zero row y[-1] (columns from both ends, as sl_step; with
// ascending columns here ptxas allocates the kernel's registers differently and the pair loop loses .reuse flags)
__device__ __forceinline__ void sl16_col_z1(double (&z1)[16], const double (&y)[16], const double xj, const int jj) {
#pragma unroll
  for (int kk = jj; kk < 16; kk++) z1[kk] = fma(xj, y[kk - jj], z1[kk]);
}
__device__ __forceinline__ void sl16_step_z1(double (&z1)[16], const double (&y)[16], const double* __restrict__ xs) {
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    const double2 xa = *reinterpret_cast<const double2*>(xs + j);
    const double2 xb = *reinterpret_cast<const double2*>(xs + 14 - j);
    sl16_col_z1(z1, y, xa.x, j);
    sl16_col_z1(z1, y, xb.y, 15 - j);
    sl16_col_z1(z1, y, xa.y, j + 1);
    sl16_col_z1(z1, y, xb.x, 14 - j);
  }
}

// Whole 16^3 slabs (D1 = D2 = L = 16, one chunk, one staged pair): the schedule is a closed form of the thread index
// instead of a step table, and every warp walks whole runs in lockstep.
//   lane map: warp d = row fold (row pairs {d, 7-d}, s = 2d and 14-2d), quarter-warp = team, lane c1 of the quarter-warp =
//   plane fold (output planes {c1, 15-c1}).  All 32 lanes of a warp slide over the same row pair, so their runs have the
//   same lengths 2d+2 (phase 0) and 16-2d (phase 1); a run is the walk a = 0 .. s+1 of one (plane pair, row pair).
//   Each lane has 17 plane pairs t = 0..16 (t <= c1: planes (t, c1-t) -> c1, else (t-c1-1, 16-t) -> 15-c1), each with one
//   run per phase.  Team k takes t = 4k .. 4k+3 in phase 0 and back down in phase 1 (8 whole runs); the 9 step pairs of
//   t = 16's two runs are dealt 3 per team to teams 0..2, and team 3 multiplies zero rows instead (78 steps per team,
//   as the step table's 312 / 306).
// Per run the thread computes its x / y row bases once; inside it the x row moves by +L and the y row by -L.  The last
// step of a whole run pairs z0 with the zero row and runs as a z1-only body (136 DFMA).  The accumulators change their
// output rows only between runs, so the flush test is paid once per run.
__global__ void __launch_bounds__(ST, 3) k_mul_slide16(const SlideP p) {
  constexpr int LT = 16;
  extern __shared__ __align__(16) double smem[];
  double* Xs = smem;
  double* Ys = smem + p.x_slab_sm;
  const double* Zr = Ys + p.y_slab_sm;   // three zero rows: the operands of team 3's padding pairs
  const int tid = threadIdx.x;
  const uint4 unit = p.units[blockIdx.x];
  {
    const int total = (int)(p.x_slab_sm + p.y_slab_sm) + 3 * LT;
    for (int i = tid * 2; i < total; i += ST * 2) *reinterpret_cast<double2*>(smem + i) = make_double2(0.0, 0.0);
  }
  unsigned k[S_MAXA], lo[S_MAXA], ext[S_MAXA];
  {
    unsigned rem = unit.x;
#pragma unroll
    for (int a = S_MAXA - 1; a >= 0; --a) {
      if (a < p.na) {
        unsigned len = (a == 0) ? p.rows_a0 : p.ra[a];
        unsigned idx = rem % len;
        rem /= len;
        k[a] = (a == 0) ? unit.w : idx;
        unsigned l = (k[a] + 1 > p.ya[a]) ? k[a] + 1 - p.ya[a] : 0;
        unsigned h = (k[a] + 1 < p.xa[a]) ? k[a] + 1 : p.xa[a];
        lo[a] = l;
        ext[a] = h > l ? h - l : 0;
      } else {
        k[a] = lo[a] = 0;
        ext[a] = 1;
      }
    }
  }
  double* out_slab = p.out + (size_t)unit.x * p.z_rows * LT;
  const int d = tid >> 5, team = (tid >> 3) & 3, c1 = tid & 7;

  double z0[LT], z1[LT], ya[LT], yb[LT];
#pragma unroll
  for (int i = 0; i < LT; i++) z0[i] = z1[i] = ya[i] = yb[i] = 0.0;
  unsigned cur = 0xffffffffu;   // output row (r1 * 16 + s) of z0; z1 is the row after it

  for (unsigned q = unit.y; q < unit.z; q++) {
    __syncthreads();
    {
      long long xo = 0, yo = 0;
      unsigned rem = q;
#pragma unroll
      for (int a = S_MAXA - 1; a >= 0; --a) {
        if (a < p.na) {
          unsigned j = lo[a] + rem % ext[a];
          rem /= ext[a];
          xo += (long long)j * p.xastr[a];
          yo += (long long)(k[a] - j) * p.yastr[a];
        }
      }
      const double2* gx = reinterpret_cast<const double2*>(p.x + xo);
      const double2* gy = reinterpret_cast<const double2*>(p.y + yo);
      double* ys = Ys + p.y_first;
      constexpr int n = 16 * 16 * LT / 2;
      for (int i = tid; i < n; i += ST) {
        const int r = i >> 3, c = i & 7, pl = r >> 4, rr = r & 15;
        cp_async16(Xs + pl * p.x_plane_sm + rr * LT + 2 * c, gx + i);
        cp_async16(ys + pl * p.y_plane_sm + rr * LT + 2 * c, gy + i);
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();

#pragma unroll 1
    for (int i = 0; i < 11; i++) {
      int t, s, a0, npairs;
      bool pad = false;
      if (i < 8) {   // whole runs
        const int ph = i >> 2;
        t = 4 * team + (ph ? 3 - (i & 3) : (i & 3));
        s = ph ? 14 - 2 * d : 2 * d;
        a0 = 0;
        npairs = s / 2 + 1;
      } else {       // step pair pr of t = 16's runs: pairs 0..d belong to the phase-0 run, d+1..8 to the phase-1 run
        const int pr = 3 * team + (i - 8);
        t = 16;
        if (pr <= d) { s = 2 * d; a0 = 2 * pr; }
        else { s = 14 - 2 * d; a0 = 2 * (pr - d - 1); }
        pad = pr >= 9;
        npairs = 1;
      }
      const int r1 = t <= c1 ? c1 : 15 - c1;
      const int j1 = t <= c1 ? t : t - c1 - 1;
      const double* xs = Xs + j1 * p.x_plane_sm + a0 * LT;
      const double* ys = Ys + (r1 - j1) * p.y_plane_sm + (s - a0 + 1) * LT;   // y row s - a0 (row -1 is the zero row)
      unsigned zrow = (unsigned)(r1 * 16 + s);
      if (pad) { xs = Zr; ys = Zr + LT; zrow = cur; }
      if (zrow != cur) {
        if (cur != 0xffffffffu) {
          double* dst = out_slab + (size_t)cur * LT;
          sl_flush<LT>(z0, dst, true);
          sl_flush<LT>(z1, dst + LT, true);
        }
        cur = zrow;
      }
      sl_load<LT>(yb, ys + LT);
      const int whole = i < 8 ? npairs - 1 : npairs;
#pragma unroll 1   // one copy of the pair body: the four warps sit in runs of different lengths
      for (int m = 0; m < whole; m++) {
        sl_load<LT>(ya, ys);
        sl16_step(z0, z1, ya, yb, xs);
        sl_load<LT>(yb, ys - LT);
        sl16_step(z0, z1, yb, ya, xs + LT);
        xs += 2 * LT;
        ys -= 2 * LT;
      }
      if (i < 8) {   // a = s, s + 1
        sl_load<LT>(ya, ys);
        sl16_step(z0, z1, ya, yb, xs);
        sl16_step_z1(z1, ya, xs + LT);
      }
    }
  }
  if (cur != 0xffffffffu) {
    double* dst = out_slab + (size_t)cur * LT;
    sl_flush<LT>(z0, dst, true);
    sl_flush<LT>(z1, dst + LT, true);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct SlideGeom {
  int nd, na;      // na = real A axes (nd - 3); a tiled plan appends the plane-tile axis as one more A axis
  u64 lt, lc, D1, D2;
  u64 T1, nt;      // planes per staged slab and number of plane tiles (T1 == D1, nt == 1: untiled)
  int E;           // tiled: plane pairs of a class are interleaved over E lockstep lanes (T1 * E == 8)
  int threads;     // CTA size
  u64 row, xplane, yplane, xslab, yslab, yfirst;
  int G;
  int ctas;       // resident CTAs per SM the shared-memory footprint allows
  size_t smem;
};

static void slide_smem_layout(SlideGeom* g) {
  g->row = g->lt;                                         // lockstep lanes differ by plane, not by row: no row padding
  g->xplane = odd_groups(g->D2 * g->lc * g->row);
  g->yplane = odd_groups((g->D2 + 2) * g->lc * g->row);   // zero rows -1 and D2
  g->yfirst = g->lc * g->row;
  g->xslab = odd_groups(g->T1 * g->xplane);
  g->yslab = odd_groups(g->T1 * g->yplane);
}

static bool slide_geom(const Ctx& ctx, const MulArgs& a, SlideGeom* g) {
  const int nd = a.ndim;
  if (nd < 4 || a.accumulate) return false;
  const u64 ltt = a.rs[nd - 1], D1 = a.rs[nd - 3], D2 = a.rs[nd - 2];
  if (a.xs[nd - 1] != ltt || a.ys[nd - 1] != ltt) return false;
  if (a.xs[nd - 3] != D1 || a.ys[nd - 3] != D1 || a.xs[nd - 2] != D2 || a.ys[nd - 2] != D2) return false;
  if (D1 % 2 != 0 || D2 % 4 != 0) return false;
  const u64 lt = dfma_chunk(ltt);
  if (!lt) return false;
  for (int d = 0; d < nd; d++)
    if (a.xs[d] == 0 || a.ys[d] == 0 || a.rs[d] == 0) return false;
  g->nd = nd;
  g->na = nd - 3;
  if (g->na > S_MAXA) return false;
  g->lt = lt;
  g->lc = ltt / lt;
  g->D1 = D1;
  g->D2 = D2;
  const u64 budget3 = 74 * 1024, budget2 = 112 * 1024;
  // ---- untiled: the whole (D1, D2, L) slab of each operand is staged ----
  const u64 lanes = (D1 / 2) * (D2 / 4);
  if (ctx.slide_tile == 0 && lanes <= (u64)ST && lanes >= 16 && D1 * D2 * g->lc < 4096) {
    g->T1 = D1;
    g->nt = 1;
    g->E = 1;
    g->threads = ST;
    slide_smem_layout(g);
    const u64 pair = (g->xslab + g->yslab) * 8;
    bool ok = true;
    if (pair <= budget3) { g->ctas = 3; g->G = (int)std::min<u64>(8, budget3 / pair); }
    else if (pair <= budget2) { g->ctas = 2; g->G = 1; }
    else ok = false;
    if (ok && g->G * std::max(g->xslab, g->yslab) < (1u << 20)) {
      g->smem = (size_t)g->G * pair;
      return true;
    }
  }
  // ---- tiled plane axis: slabs of T1 planes, one more A axis over the D1 / T1 tiles ----
  if (g->na + 1 > S_MAXA) return false;
  for (u64 T1 : {4, 8}) {
    if (ctx.slide_tile != 0 && (u64)ctx.slide_tile != T1) continue;
    if (D1 % T1 != 0 || D1 / T1 < 2) continue;
    if (2 * T1 * D2 * g->lc >= 4096) continue;
    g->T1 = T1;
    g->nt = D1 / T1;
    g->E = (int)(8 / T1);
    g->threads = ST;
    g->G = 1;
    slide_smem_layout(g);
    const u64 pair = (g->xslab + g->yslab) * 8;
    if (pair > budget2 || std::max(g->xslab, g->yslab) >= (1u << 20)) continue;
    // 170 registers x 384 threads fill the register file: at most 384 / threads CTAs
    const u64 by_regs = std::max<u64>(1, 384 / (u64)((g->threads + 31) / 32 * 32));
    const u64 by_smem = (227 * 1024) / (pair + 1024);
    g->ctas = (int)std::max<u64>(1, std::min(by_regs, by_smem));
    g->smem = (size_t)pair;
    return true;
  }
  return false;
}

bool slide_mul_applicable(const Ctx& ctx, const MulArgs& a) {
  SlideGeom g;
  if (!slide_geom(ctx, a, &g)) return false;
  u64 slabs = a.row_count * g.nt;
  for (int d = 1; d < g.na; d++) slabs *= a.rs[d];
  return slabs >= 64 || (slabs >= 1 && (ctx.fast_mul == 2 || args_macs(a) >= DFMA_MIN_MACS));
}

// Folded lane sequences (see the header): lane (c1, d) owns planes {c1, D1-1-c1} and row pairs {d, P-1-d}.
static void build_slide_table(const SlideGeom& g, std::vector<uint2>* table, int* n_lo, int* n_hi) {
  const int D1 = (int)g.D1, D2 = (int)g.D2, P = D2 / 2, C1 = D1 / 2, DD = P / 2, LC = (int)g.lc;
  const int nl = C1 * DD, T = ST / nl;
  struct Step { unsigned xoff, yoff, zrow, z1ok, g; bool run_start; };
  std::vector<std::vector<Step>> seq_lo(nl), seq_hi(nl);
  for (int d = 0; d < DD; d++)
    for (int c1 = 0; c1 < C1; c1++) {
      const int lane = d * C1 + c1;
      int seam = 0;
      for (int phase = 0; phase < 2; phase++) {
        const int half = phase == 0 ? d : P - 1 - d;
        const int s = 2 * half;
        for (int kc = 0; kc < LC; kc++)
          for (int gi = 0; gi < g.G; gi++, seam++)
            for (int tt = 0; tt <= D1; tt++) {
              const int t = (seam & 1) ? D1 - tt : tt;
              const int r1 = t <= c1 ? c1 : D1 - 1 - c1;
              const int j1 = t <= c1 ? t : t - c1 - 1;
              const int m1 = r1 - j1;
              for (int jc = 0; jc < LC; jc++)
                for (int mc = 0; mc < LC; mc++) {
                  int kind;
                  if (jc + mc == kc) kind = 0;
                  else if (jc + mc + 1 == kc) kind = 1;
                  else continue;
                  const int a_hi = std::min(D2 - 1, s + 1);
                  for (int a = 0; a <= a_hi; a++) {
                    const int m2 = s - a;   // new (lower) y row; -1 is the leading zero row
                    Step st;
                    st.xoff = (unsigned)(gi * g.xslab + j1 * g.xplane + ((u64)a * LC + jc) * g.row);
                    st.yoff = (unsigned)(gi * g.yslab + m1 * g.yplane + ((u64)(m2 + 1) * LC + mc) * g.row);
                    st.zrow = (unsigned)(((u64)r1 * D2 + s) * LC + kc);
                    st.z1ok = s + 1 < D2 ? 1u : 0u;
                    st.g = (unsigned)gi;
                    st.run_start = a == 0;
                    (kind ? seq_hi : seq_lo)[lane].push_back(st);
                  }
                }
            }
      }
    }
  const size_t len_lo = seq_lo[0].size(), len_hi = seq_hi[0].size();
  auto steps_of = [&](size_t len) { int n = (int)((len + T - 1) / T); return (n + 1) / 2 * 2; };   // even
  *n_lo = steps_of(len_lo);
  *n_hi = steps_of(len_hi);
  table->assign((size_t)(std::max(*n_lo + *n_hi, 2) + 2) * ST, make_uint2(0u, 0u));
  auto emit = [&](const std::vector<Step>& seq, size_t b, size_t e, size_t row0, int tid) {
    for (size_t i = b; i < e; i++) {
      const Step& st = seq[i];
      const bool reload = st.run_start || i == b;   // first step of a share: nothing valid in the y registers yet
      uint2 en;
      en.x = st.xoff | (st.g << 20) | (st.z1ok << 25) | (reload ? SE_RELOAD : 0u) | SE_VALID;
      en.y = st.yoff | (st.zrow << 20);
      (*table)[(row0 + (i - b)) * ST + tid] = en;
    }
  };
  for (int team = 0; team < T; team++)
    for (int l = 0; l < nl; l++) {
      const int tid = team * nl + l;
      emit(seq_lo[l], len_lo * team / T, len_lo * (team + 1) / T, 0, tid);
      emit(seq_hi[l], len_hi * team / T, len_hi * (team + 1) / T, (size_t)*n_lo, tid);
    }
}

// Tiled plane axis (see slide_geom): a slab holds T1 planes of tile tp of X and of tile tq of Y; their plane pairs
// (j1, m1) feed the output planes r1 = j1 + m1 in 0 .. 2 T1 - 2 of output tile tp + tq (r1 >= T1: the next tile, SE_UPPER).
// Class c owns the output planes {c, c + T1}: exactly T1 plane pairs (j1 = t, m1 = (c - t) mod T1, t = 0 .. T1-1), which
// are dealt round-robin to E lockstep lanes (t = u E + tau).  The 8 lanes (c, tau) of a quarter-warp execute the same
// (row pair, chunk, step) on different planes: x rows are broadcast per tau, y rows sit in T1 different planes =>
// conflict-free LDS.128 (plane strides are odd numbers of 16-byte groups).  Lane d of the row-pair fold as untiled.
static void build_slide_table_tiled(const SlideGeom& g, std::vector<uint2>* table, int* n_lo, int* n_hi) {
  const int T1 = (int)g.T1, E = g.E, D2 = (int)g.D2, P = D2 / 2, DD = P / 2, LC = (int)g.lc;
  const int nl = 8 * DD, NT = g.threads, U = T1 / E;
  struct Step { unsigned xoff, yoff, zrow, z1ok, upper; bool run_start; };
  std::vector<std::vector<Step>> seq_lo(nl), seq_hi(nl);
  for (int d = 0; d < DD; d++)
    for (int tau = 0; tau < E; tau++)
      for (int c = 0; c < T1; c++) {
        const int lane = d * 8 + tau * T1 + c;
        int seam = 0;
        for (int phase = 0; phase < 2; phase++) {
          const int half = phase == 0 ? d : P - 1 - d;
          const int s = 2 * half;
          for (int kc = 0; kc < LC; kc++, seam++)
            for (int uu = 0; uu < U; uu++) {
              const int u = (seam & 1) ? U - 1 - uu : uu;
              const int t = u * E + tau;
              const int r1 = t <= c ? c : c + T1;
              const int j1 = t, m1 = r1 - j1;
              for (int jc = 0; jc < LC; jc++)
                for (int mc = 0; mc < LC; mc++) {
                  int kind;
                  if (jc + mc == kc) kind = 0;
                  else if (jc + mc + 1 == kc) kind = 1;
                  else continue;
                  const int a_hi = std::min(D2 - 1, s + 1);
                  for (int a = 0; a <= a_hi; a++) {
                    const int m2 = s - a;
                    Step st;
                    st.xoff = (unsigned)(j1 * g.xplane + ((u64)a * LC + jc) * g.row);
                    st.yoff = (unsigned)(m1 * g.yplane + ((u64)(m2 + 1) * LC + mc) * g.row);
                    st.zrow = (unsigned)(((u64)r1 * D2 + s) * LC + kc);
                    st.z1ok = s + 1 < D2 ? 1u : 0u;
                    st.upper = r1 >= T1 ? 1u : 0u;
                    st.run_start = a == 0;
                    (kind ? seq_hi : seq_lo)[lane].push_back(st);
                  }
                }
            }
        }
      }
  // The sequences of the DD row-fold lanes of one (c, tau) have the same length and structure.  Concatenated over d they
  // are cut into NT / 8 equal pieces, one per octet of threads: 128-thread CTAs for any D2 (a CTA of 3 warps leaves the
  // four schedulers of an SM unevenly loaded and its warps wait for each other at the round barrier: 21 % of the
  // stall samples on 5 x 24), every octet in lockstep on one d at a time.
  const int NO = NT / 8;
  const size_t len_lo = seq_lo[0].size() * DD, len_hi = seq_hi[0].size() * DD;
  auto steps_of = [&](size_t len) { int n = (int)((len + NO - 1) / NO); return (n + 1) / 2 * 2; };   // even
  *n_lo = steps_of(len_lo);
  *n_hi = steps_of(len_hi);
  table->assign((size_t)(std::max(*n_lo + *n_hi, 2) + 2) * NT, make_uint2(0u, 0u));
  auto emit = [&](const std::vector<std::vector<Step>>& seqs, int q8, size_t b, size_t e, size_t row0, int tid) {
    const size_t per = seqs[0].size();
    for (size_t i = b; i < e; i++) {
      const Step& st = seqs[(i / per) * 8 + q8][i % per];
      const bool reload = st.run_start || i == b;
      uint2 en;
      en.x = st.xoff | (st.z1ok << 25) | (reload ? SE_RELOAD : 0u) | (st.upper ? SE_UPPER : 0u) | SE_VALID;
      en.y = st.yoff | (st.zrow << 20);
      (*table)[(row0 + (i - b)) * NT + tid] = en;
    }
  };
  for (int o = 0; o < NO; o++)
    for (int q8 = 0; q8 < 8; q8++) {
      const int tid = o * 8 + q8;
      emit(seq_lo, q8, len_lo * o / NO, len_lo * (o + 1) / NO, 0, tid);
      emit(seq_hi, q8, len_hi * o / NO, len_hi * (o + 1) / NO, (size_t)*n_lo, tid);
    }
}

struct SlidePlan : DfmaPlan {
  bool runs = false;   // k_mul_slide16 (no step table)
  SlideP p;
  SlideGeom g;
};

template <int LT> static void slide_launch_lt(Ctx& ctx, const SlidePlan& pl, const SlideP& p) {
  if (pl.g.lc > 1) {
    allow_dyn_smem(k_mul_slide<LT, true>, ctx.device, pl.g.smem);
    GTP_LAUNCH(ctx, (k_mul_slide<LT, true>), pl.n_units, pl.g.threads, pl.g.smem, p);
  } else {
    allow_dyn_smem(k_mul_slide<LT, false>, ctx.device, pl.g.smem);
    GTP_LAUNCH(ctx, (k_mul_slide<LT, false>), pl.n_units, pl.g.threads, pl.g.smem, p);
  }
}

void launch_mul_slide(Ctx& ctx, const MulArgs& a) {
  SlideGeom g;
  GTP_CHECK(slide_geom(ctx, a, &g), GTP_ERR_ARG, "sliding product kernel not applicable");
  // whole 16^3 slabs run on k_mul_slide16 (ctx.slide_runs = false: the table-driven kernel, for A/B measurements)
  const bool runs = ctx.slide_runs && g.nt == 1 && g.D1 == 16 && g.D2 == 16 && g.lt == 16 && g.lc == 1 && g.G == 1 && g.threads == ST;
  if (runs) g.smem += 3 * 16 * sizeof(double);   // the zero rows of the padding pairs
  std::shared_ptr<void>& slot = dfma_plan_slot(ctx.slide_plans, a, g.T1 << 1 | (runs ? 1 : 0));
  if (!slot) {
    auto pl = std::make_shared<SlidePlan>();
    pl->g = g;
    pl->runs = runs;
    SlideP& p = pl->p;
    memset(&p, 0, sizeof(p));
    const int nd = g.nd, nr = g.na, tiled = g.nt > 1 ? 1 : 0, na = nr + tiled;
    Shape xst(nd, 1), yst(nd, 1);
    for (int i = nd - 2; i >= 0; --i) {
      xst[i] = xst[i + 1] * a.xs[i + 1];
      yst[i] = yst[i + 1] * a.ys[i + 1];
    }
    // extents of the A axes as the kernel and the unit builder see them (the plane-tile axis last)
    std::vector<u64> axs(na), ays(na), ars(na);
    for (int d = 0; d < nr; d++) { axs[d] = a.xs[d]; ays[d] = a.ys[d]; ars[d] = a.rs[d]; }
    p.na = na;
    for (int d = 0; d < nr; d++) {
      p.xastr[d] = (long long)xst[d];
      p.yastr[d] = (long long)yst[d];
    }
    if (tiled) {
      axs[nr] = ays[nr] = ars[nr] = g.nt;
      p.xastr[nr] = (long long)(g.T1 * xst[nd - 3]);
      p.yastr[nr] = (long long)(g.T1 * yst[nd - 3]);
    }
    for (int d = 0; d < na; d++) {
      p.xa[d] = (unsigned)axs[d];
      p.ya[d] = (unsigned)ays[d];
      p.ra[d] = (unsigned)ars[d];
    }
    p.tiled = tiled;
    p.rows_a0 = (unsigned)a.row_count;
    p.planes = (unsigned)g.T1;
    p.prow = (unsigned)(g.D2 * g.lc);
    p.row = (unsigned)g.row;
    p.x_plane_sm = (unsigned)g.xplane; p.y_plane_sm = (unsigned)g.yplane;
    p.x_slab_sm = (unsigned)g.xslab; p.y_slab_sm = (unsigned)g.yslab;
    p.y_first = (unsigned)g.yfirst;
    p.y_up_off = (unsigned)(g.lc * g.row);
    p.z_rows = (unsigned)(g.T1 * g.D2 * g.lc);
    p.z_up = (unsigned)g.lc;
    p.G = g.G;
    std::vector<uint2> table;
    if (runs) p.nsteps_lo = p.nsteps = 0;
    else if (tiled) build_slide_table_tiled(g, &table, &p.nsteps_lo, &p.nsteps);
    else build_slide_table(g, &table, &p.nsteps_lo, &p.nsteps);
    p.nsteps += p.nsteps_lo;
    dfma_upload(ctx, pl.get(), table, dfma_units(a, axs, ays, ars, g.G, (u64)ctx.sm_count * g.ctas));
    p.table = reinterpret_cast<const uint2*>(pl->table->d);
    p.units = reinterpret_cast<const uint4*>(pl->units->d);
    slot = pl;
  }
  const SlidePlan& pl = *std::static_pointer_cast<SlidePlan>(slot);
  SlideP p = pl.p;
  p.x = a.x;
  p.y = a.y;
  p.out = a.out;
  u64 row_elems = 1;
  for (int d = 1; d < a.ndim; d++) row_elems *= a.rs[d];
  GTP_CUDA(cudaMemsetAsync(a.out, 0, a.row_count * row_elems * sizeof(double), ctx.stream));
  if (pl.n_units == 0) return;
  if (pl.runs) {
    allow_dyn_smem(k_mul_slide16, ctx.device, pl.g.smem);
    GTP_LAUNCH(ctx, k_mul_slide16, pl.n_units, pl.g.threads, pl.g.smem, p);
    return;
  }
  if (p.nsteps == 0) return;
  switch ((int)pl.g.lt) {
    case 8: slide_launch_lt<8>(ctx, pl, p); break;
    case 10: slide_launch_lt<10>(ctx, pl, p); break;
    case 12: slide_launch_lt<12>(ctx, pl, p); break;
    case 14: slide_launch_lt<14>(ctx, pl, p); break;
    case 16: slide_launch_lt<16>(ctx, pl, p); break;
    default: throw Error(GTP_ERR_ARG, "unsupported chunk length");
  }
}

}  // namespace gtp
