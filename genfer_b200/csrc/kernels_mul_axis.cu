// Product of an N-D tensor with a 1-D operand (one non-unit axis `a`): a batched 1-d convolution along that axis,
//     Z[o, k, i] = sum_j  s[j] * B[o, k - j, i]            (views (outer, L, inner) of the axis)
// -- the compound-distribution / thinning products of multi-variable programs whose substitution has a long 1-d
// series (two_populations: [336] x [336, 336], 1.9e7 MACs each).  The reference-order kernel (one thread per output
// coefficient, 64-bit odometers, one dependent gather per MAC) ran these at ~0.15 TFLOP/s; the DFMA kernels need two dense
// operands of equal slab shape.  Here a thread owns KT consecutive outputs along the axis and keeps the sliding window
// B[k - j] in registers (one new load per step for KT multiply-adds, lanes along the contiguous inner axis), or -- when the
// axis is the contiguous one -- a CTA stages the row and the 1-d operand in shared memory.
//
// BIT-IDENTICAL to the reference (`mul` :984-1012): per output the terms are visited in ascending X index with a separate
// multiply and add; when the axis is the innermost non-unit axis of the result the sum runs from zero and is then added
// (mul_1d :972-982 + `*z += o` :998), otherwise every term arrives as its own 1-d leaf `0 + x*y` and is added to the
// running coefficient.  No FMA: these products keep the end-to-end reports byte-identical.
#include "kernels.cuh"

namespace gtp {

struct AxisP {
  const double* big;
  const double* small;
  double* out;
  unsigned outer, inner, Lb, Ls, Lr;   // big: (outer, Lb, inner); small: Ls; result: (outer, Lr, inner)
  int desc;                            // 1: visit the small operand's index descending (the small operand is Y)
};

// axis not innermost: lanes over the flattened (outer, inner) columns, KT outputs along the axis per thread
template <int KT>
__global__ void __launch_bounds__(128) k_mul_axis_cols(const AxisP p) {
  const unsigned ncol = p.outer * p.inner;
  const unsigned col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncol) return;
  const unsigned o = col / p.inner, i = col - o * p.inner;
  const unsigned k0 = blockIdx.y * KT;
  const double* bp = p.big + ((size_t)o * p.Lb) * p.inner + i;
  double acc[KT], w[KT];
#pragma unroll
  for (int q = 0; q < KT; q++) acc[q] = 0.0;
  // small indices that can pair with an output of this tile: m <= k, k - m < Lb, m < Ls
  const int m_lo = (int)k0 + 1 > (int)p.Lb ? (int)k0 + 1 - (int)p.Lb : 0;
  const int m_hi = min((int)k0 + KT - 1, (int)p.Ls - 1);   // inclusive
  if (m_hi < m_lo) {
#pragma unroll
    for (int q = 0; q < KT; q++)
      if (k0 + q < p.Lr) p.out[((size_t)o * p.Lr + k0 + q) * p.inner + i] = 0.0;
    return;
  }
  auto ldb = [&](int kb) -> double { return (kb >= 0 && kb < (int)p.Lb) ? bp[(size_t)kb * p.inner] : 0.0; };
  if (!p.desc) {
    // ascending m: window W_q(m) = B[k0 + q - m]; W_q(m + 1) = W_{q-1}(m), W_0(m + 1) is the one new load
#pragma unroll
    for (int q = 0; q < KT; q++) w[q] = ldb((int)k0 + q - m_lo);
    for (int m = m_lo; m <= m_hi; m += KT) {
#pragma unroll
      for (int u = 0; u < KT; u++) {
        const int mm = m + u;
        if (mm <= m_hi) {
          const double sv = p.small[mm];
#pragma unroll
          for (int q = 0; q < KT; q++) {
            const int kb = (int)k0 + q - mm;
            if (kb >= 0 && kb < (int)p.Lb) acc[q] = __dadd_rn(acc[q], __dadd_rn(0.0, __dmul_rn(sv, w[(q - u + KT) % KT])));
          }
          w[(KT - 1 - u + KT) % KT] = ldb((int)k0 - mm - 1);   // becomes W_0(mm + 1)
        }
      }
    }
  } else {
    // descending m: W_q(m - 1) = W_{q+1}(m), W_{KT-1}(m - 1) is the one new load
#pragma unroll
    for (int q = 0; q < KT; q++) w[q] = ldb((int)k0 + q - m_hi);
    for (int m = m_hi; m >= m_lo; m -= KT) {
#pragma unroll
      for (int u = 0; u < KT; u++) {
        const int mm = m - u;
        if (mm >= m_lo) {
          const double sv = p.small[mm];
#pragma unroll
          for (int q = 0; q < KT; q++) {
            const int kb = (int)k0 + q - mm;
            if (kb >= 0 && kb < (int)p.Lb) acc[q] = __dadd_rn(acc[q], __dadd_rn(0.0, __dmul_rn(sv, w[(q + u) % KT])));
          }
          w[u % KT] = ldb((int)k0 + KT - 1 - mm + 1);   // becomes W_{KT-1}(mm - 1)
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < KT; q++)
    if (k0 + q < p.Lr) p.out[((size_t)o * p.Lr + k0 + q) * p.inner + i] = acc[q];
}

// axis innermost (inner == 1): one CTA per (row o, tile of AX_TB outputs); the 1-d operand and the row window in shared memory
constexpr int AX_TB = 256;
__global__ void __launch_bounds__(AX_TB) k_mul_axis_row(const AxisP p) {
  extern __shared__ double ax_sm[];
  double* ss = ax_sm;              // Ls
  double* bw = ax_sm + p.Ls;       // window B[k0 - Ls + 1 .. k0 + AX_TB - 1]  (Ls + AX_TB - 1 values)
  const unsigned o = blockIdx.y, k0 = blockIdx.x * AX_TB;
  const double* bp = p.big + (size_t)o * p.Lb;
  for (unsigned t = threadIdx.x; t < p.Ls; t += AX_TB) ss[t] = p.small[t];
  const int w0 = (int)k0 - (int)p.Ls + 1;
  for (unsigned t = threadIdx.x; t < p.Ls + AX_TB - 1; t += AX_TB) {
    const int kb = w0 + (int)t;
    bw[t] = (kb >= 0 && kb < (int)p.Lb) ? bp[kb] : 0.0;
  }
  __syncthreads();
  const unsigned k = k0 + threadIdx.x;
  if (k >= p.Lr) return;
  const int m_lo = (int)k + 1 > (int)p.Lb ? (int)k + 1 - (int)p.Lb : 0;
  const int m_hi = min((int)k, (int)p.Ls - 1);
  double inner = 0.0;
  // B[k - m] = bw[k - m - w0]
  const double* bk = bw + ((int)k - w0);
  if (!p.desc) for (int m = m_lo; m <= m_hi; m++) inner = __dadd_rn(inner, __dmul_rn(ss[m], bk[-m]));
  else for (int m = m_hi; m >= m_lo; m--) inner = __dadd_rn(inner, __dmul_rn(ss[m], bk[-m]));
  p.out[(size_t)o * p.Lr + k] = __dadd_rn(0.0, inner);
}

// Returns false when the product is not of this form (the caller goes on to the reference-order kernel).
bool launch_mul_axis(Ctx& ctx, const MulArgs& a) {
  const int nd = a.ndim;
  if (nd < 1 || a.accumulate || !a.rows.empty() || a.row_begin != 0 || a.row_step != 1 || a.row_count != a.rs[0]) return false;
  auto one_axis = [&](const Shape& s, int* ax) {
    int n = 0;
    for (int d = 0; d < nd; d++)
      if (s[d] > 1) { n++; *ax = d; }
    return n == 1;
  };
  int ax = -1, ax2 = -1;
  const bool x1 = one_axis(a.xs, &ax), y1 = one_axis(a.ys, &ax2);
  bool small_is_x;
  if (x1 && y1) return false;                       // 1-d times 1-d: tiny or the reference-order kernel's business
  if (x1) small_is_x = true;
  else if (y1) { small_is_x = false; ax = ax2; }
  else return false;
  const Shape& ss = small_is_x ? a.xs : a.ys;
  const Shape& bs = small_is_x ? a.ys : a.xs;
  for (int d = 0; d < nd; d++) {
    if (d != ax && a.rs[d] != bs[d]) return false;  // the result keeps the big operand's extents off the axis (sum_shape)
    if (bs[d] == 0 || a.rs[d] == 0) return false;
  }
  const u64 Ls = ss[ax], Lb = bs[ax], Lr = a.rs[ax];
  if (Ls < 2 || Lr > Lb + Ls - 1) return false;
  u64 outer = 1, inner = 1;
  for (int d = 0; d < ax; d++) outer *= bs[d];
  for (int d = ax + 1; d < nd; d++) inner *= bs[d];
  if (outer * inner * std::max(Lb, Lr) >= (1ull << 31) || Ls >= (1u << 20)) return false;
  if ((double)outer * inner * Lr * std::min(Ls, Lb) < 16384.0) return false;   // launch-bound either way
  AxisP p;
  p.big = small_is_x ? a.y : a.x;
  p.small = small_is_x ? a.x : a.y;
  p.out = a.out;
  p.outer = (unsigned)outer;
  p.inner = (unsigned)inner;
  p.Lb = (unsigned)Lb;
  p.Ls = (unsigned)Ls;
  p.Lr = (unsigned)Lr;
  p.desc = small_is_x ? 0 : 1;   // ascending X index == descending index of a small Y
  if (inner == 1) {
    const size_t smem = (2 * Ls + AX_TB) * sizeof(double);
    if (smem > 200 * 1024 || outer > 65535) return false;
    allow_dyn_smem(k_mul_axis_row, ctx.device, std::max<size_t>(smem, 48 * 1024));
    dim3 grid((unsigned)((Lr + AX_TB - 1) / AX_TB), (unsigned)outer);
    GTP_LAUNCH(ctx, k_mul_axis_row, grid, AX_TB, smem, p);
    return true;
  }
  // outputs per thread along the axis: 8 when that still gives every SM a few hundred threads, fewer for small tensors
  // ([336] x [336, 336]: KT = 8 left 14 k threads, each a chain of 336 dependent steps: 95 us; latency-bound)
  const u64 ncol = outer * inner;
  int KT = 8;
  while (KT > 1 && ncol * ((Lr + KT - 1) / KT) < (u64)ctx.sm_count * 512) KT /= 2;
  const u64 ktiles = (Lr + KT - 1) / KT;
  if (ktiles > 65535) return false;
  dim3 grid((unsigned)((ncol + 127) / 128), (unsigned)ktiles);
  switch (KT) {
    case 8: GTP_LAUNCH(ctx, k_mul_axis_cols<8>, grid, 128, 0, p); break;
    case 4: GTP_LAUNCH(ctx, k_mul_axis_cols<4>, grid, 128, 0, p); break;
    case 2: GTP_LAUNCH(ctx, k_mul_axis_cols<2>, grid, 128, 0, p); break;
    default: GTP_LAUNCH(ctx, k_mul_axis_cols<1>, grid, 128, 0, p); break;
  }
  return true;
}

}  // namespace gtp
