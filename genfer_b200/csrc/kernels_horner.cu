// Fused Horner loop of subst_var (multivariate_taylor.rs:569-579) for a substitution of at most 32 coefficients:
//
//     for i in (0..len_v).rev():   res = res * subst + self.slice(v, i)
//
// The reference spends three whole-tensor operations per step (the slice copy, a general Mul, an Add); the per-operator
// device path mirrored that: 3 launches and 7 tensor passes per step, plus a classification of every intermediate.  Here
// the WHOLE remaining loop is ONE cooperative kernel: a step reads the previous result once (ld.global.cg: other CTAs
// wrote it), reads the slice straight out of `self` (no copy) and writes the next result -- 2 passes -- with a grid
// barrier between steps; results ping-pong between two buffers that stay L2-resident for small and mid-size tensors.
//
// Arithmetic per output coefficient is exactly the per-operator path's, i.e. the reference's:
//   * the product in the reference's nesting order (`mul` :984-1012 with Y = subst): outer axes ascending in the X index,
//     the innermost non-unit axis summed from zero and then added, multiply and add separate (== k_mul_stencil /
//     k_mul_ordered);
//   * Add's general path `(0 + a?) + b?` on zero-extended operands (:873-880), or its scalar path (`first += s`, :862-865)
//     when the slice is a single coefficient.
// The host enters the fused loop only once `res` has more than one coefficient and every axis that will ever be non-unit is
// non-unit in `res` (after at most two per-operator steps): from then on Mul's data-dependent fast paths (zero, one,
// constant) cannot fire, the set of non-unit axes -- which fixes the reference's summation nesting -- no longer changes, and
// the mul_linear fast path gives the same bits as the general product (two-term sums; DESIGN.md).
#include "device_sync.cuh"
#include "kernels.cuh"

namespace gtp {

constexpr int HN_MAXE = 8;
constexpr int HN_MAXT = 32;
constexpr int HN_T = 256;

struct HornerP {
  int ne, nt;
  unsigned d[HN_MAXE];          // degrees_p1 clip (UINT_MAX: unbounded)
  unsigned sshape[HN_MAXE];     // subst extents
  unsigned slice[HN_MAXE];      // slice extents (1 along v)
  long long selfstr[HN_MAXE];   // strides of `self` along the effective axes
  long long self_vstr;          // stride of axis v in `self`
  unsigned shape0[HN_MAXE];     // shape of the incoming res
  unsigned char m[HN_MAXT][HN_MAXE];
  unsigned char group_start[HN_MAXT];
  unsigned short sidx[HN_MAXT];
  const double* self;
  const double* subst;
  const double* res0;
  double* buf[2];
  unsigned i_top, nsteps;
  int slice_scalar;
  unsigned* bar;
};

// the term table of the substitution (or of a product's small operand)
static void set_terms(HornerP* p, const SmallTerms& st) {
  static_assert(sizeof(p->m) == sizeof(st.m), "HornerP holds the term table as it is built");
  p->nt = st.nt;
  memcpy(p->m, st.m, sizeof(p->m));
  memcpy(p->sidx, st.sidx, sizeof(p->sidx));
  memcpy(p->group_start, st.group_start, sizeof(p->group_start));
}

__global__ void __launch_bounds__(HN_T) k_horner(const __grid_constant__ HornerP p) {
  __shared__ double s_sv[HN_MAXT];
  __shared__ long long s_delta[HN_MAXT];   // offset of res[k - m_t] relative to res[k], for this step's strides
  if (threadIdx.x < (unsigned)p.nt) s_sv[threadIdx.x] = p.subst[p.sidx[threadIdx.x]];
  __syncthreads();
  const int ne = p.ne;
  unsigned cur[HN_MAXE], nxt[HN_MAXE], prodsh[HN_MAXE];
#pragma unroll
  for (int a = 0; a < HN_MAXE; a++) cur[a] = a < ne ? p.shape0[a] : 1u;
  unsigned phase = 0;
  const double* src = p.res0;
  for (unsigned step = 0; step < p.nsteps; step++) {
    double* dst = p.buf[step & 1u];
    const unsigned i = p.i_top - step;
    // shapes of this step: product (sum_shape :150-170), result of the Add (max_shape :129-148)
    unsigned total = 1;
    long long cstr[HN_MAXE];
#pragma unroll
    for (int a = 0; a < HN_MAXE; a++) {
      if (a < ne) {
        const unsigned long long s = (unsigned long long)cur[a] + p.sshape[a] - 1ull;
        prodsh[a] = (unsigned)min(s, (unsigned long long)p.d[a]);
        nxt[a] = max(prodsh[a], p.slice[a]);
        total *= nxt[a];
      } else {
        prodsh[a] = nxt[a] = 1u;
      }
    }
    {
      long long st = 1;
#pragma unroll
      for (int a = HN_MAXE - 1; a >= 0; --a) {
        if (a < ne) { cstr[a] = st; st *= (long long)cur[a]; } else cstr[a] = 0;
      }
    }
    __syncthreads();   // every thread is done with the previous step's deltas
    if (threadIdx.x < (unsigned)p.nt) {
      long long dl = 0;
#pragma unroll
      for (int a = 0; a < HN_MAXE; a++)
        if (a < ne) dl += (long long)p.m[threadIdx.x][a] * cstr[a];
      s_delta[threadIdx.x] = dl;
    }
    __syncthreads();
    const double* slice_base = p.self + (long long)i * p.self_vstr;
    for (unsigned lin = blockIdx.x * blockDim.x + threadIdx.x; lin < total; lin += gridDim.x * blockDim.x) {
      unsigned k[HN_MAXE];
      unsigned rem = lin;
      long long base = 0, so = 0;
      bool a_ok = true, b_ok = true;
#pragma unroll
      for (int a = HN_MAXE - 1; a >= 0; --a) {
        if (a < ne) {
          const unsigned q = rem / nxt[a];
          k[a] = rem - q * nxt[a];
          rem = q;
          base += (long long)k[a] * cstr[a];
          so += (long long)k[a] * p.selfstr[a];
          a_ok = a_ok && k[a] < prodsh[a];
          b_ok = b_ok && k[a] < p.slice[a];
        } else {
          k[a] = 0;
        }
      }
      double r = 0.0;
      double prod = 0.0;
      if (a_ok) {
        double total_v = 0.0, inner = 0.0;
        bool open = false;
        for (int t = 0; t < p.nt; t++) {
          if (p.group_start[t]) {
            if (open) total_v = __dadd_rn(total_v, inner);
            inner = 0.0;
            open = true;
#pragma unroll
            for (int a = 0; a < HN_MAXE - 1; a++)
              if (a < ne - 1) open = open && (k[a] - (unsigned)p.m[t][a]) < cur[a];   // unsigned: k >= m too
          }
          if (open) {
            const unsigned ml = p.m[t][ne - 1];
            if ((k[ne - 1] - ml) < cur[ne - 1]) inner = __dadd_rn(inner, __dmul_rn(ldcg(src + (base - s_delta[t])), s_sv[t]));
          }
        }
        if (open) total_v = __dadd_rn(total_v, inner);
        prod = total_v;
      }
      if (p.slice_scalar) {
        // Add's scalar path (:862-865): the product with `first += slice[0]`
        r = (lin == 0) ? __dadd_rn(prod, slice_base[0]) : prod;
      } else {
        if (a_ok) r = __dadd_rn(r, prod);
        if (b_ok) r = __dadd_rn(r, slice_base[so]);
      }
      dst[lin] = r;
    }
#pragma unroll
    for (int a = 0; a < HN_MAXE; a++) cur[a] = nxt[a];
    src = dst;
    if (step + 1 < p.nsteps) grid_barrier(p.bar, phase);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Row-staged variant for HBM-sized tensors (rows of 16..1024 coefficients along the last effective axis): the TMA engine
// streams whole source rows into shared memory with bulk asynchronous copies (cp.async.bulk + mbarrier complete_tx; SASS
// UBLKCP), two stages deep, while the CTA multiplies the previous batch out of shared memory.  One-thread-per-coefficient
// gathers (k_horner above, k_mul_stencil_v4) are latency-bound on these tensors: 45 % of HBM with 0.64 eligible warps per
// cycle (profiles/r01k_stencil_ncu.json); here address generation is per ROW (one elected thread), loads are 2-KB bulk
// transfers and the arithmetic reads conflict-free shared memory.
//   An output row (all effective axes but the last fixed) needs one source row per GROUP of terms (terms that share their
// outer offsets); a batch is HB_R consecutive output rows.  Source rows start at arbitrary element offsets: the copy
// starts at the 16-byte-aligned element below (shift 0 / 1) and the consumer indexes past the shift; the last-axis bounds
// are predicates, absent source rows (outer index out of range) skip their group exactly like the gather kernels do --
// per-coefficient arithmetic and its order are identical to k_horner's.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int HB_R = 8;          // output rows per batch
constexpr int HB_MAXG = 16;      // groups
constexpr int HB_T = 256;
constexpr int HB_NS = 4;         // ring stages

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

struct HornerBulkP {
  HornerP h;
  int ng;                                   // groups
  int ra;                                   // first axis of the row block: axes ra .. ne-1 form one contiguous block of the source
  int R;                                    // blocks per batch
  unsigned char gm[HB_MAXG][HN_MAXE];       // outer offsets of group g (axes < ra; zero on the block axes)
  unsigned char g_first[HB_MAXG], g_count[HB_MAXG];   // terms of group g: [g_first, g_first + g_count)
  unsigned slot;                            // doubles per staged block slot (even)
  int add_mode;                             // 0: product only (plain stencil product), 1: Add general path, 2: Add scalar path
};

__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// warp 0: producer (address generation + bulk copies, lanes over the (block, group) pairs of a batch);
// warps 1 .. 7: consumers.  full[st]: the producer's expect_tx arrival + the copies' bytes; empty[st]: one arrival per consumer.
__device__ __forceinline__ double lds_f64(unsigned addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f64(unsigned addr, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory"); }

// NT: compile-time bound on the number of terms (2, 4, 8, 16, 32): the term loop is fully unrolled, so the term offsets and
// group flags are immediate constant-bank operands and the substitution's coefficients live in registers (as in k_mul_stencil).
template <int NT>
__global__ void __launch_bounds__(HB_T) k_horner_rows(const __grid_constant__ HornerBulkP bp) {
  const HornerP& p = bp.h;
  extern __shared__ __align__(16) double hb_sm[];
  __shared__ __align__(8) unsigned long long s_full[HB_NS], s_empty[HB_NS];
  __shared__ unsigned char s_shift[HB_NS][HB_R * HB_MAXG];   // 0 / 1: element shift of the staged block; 255: absent
  __shared__ long long s_so[HB_NS][HB_R];                    // offset of the output block's slice coefficients in `self`
  __shared__ unsigned char s_rowok[HB_NS][HB_R];             // bit 0: block inside the product, bit 1: inside the slice (axes < ra)
  constexpr unsigned NCONS = HB_T - 32;
  const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  double sv[NT];
#pragma unroll
  for (int t = 0; t < NT; t++) sv[t] = t < p.nt ? p.subst[p.sidx[t]] : 0.0;
  const unsigned sm_base = smem_u32(hb_sm);
  if (threadIdx.x == 0) {
    for (int q = 0; q < HB_NS; q++) {
      mbar_init(&s_full[q], 1);
      mbar_init(&s_empty[q], NCONS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int ne = p.ne, ng = bp.ng, ra = bp.ra, R = bp.R;
  unsigned cur[HN_MAXE], nxt[HN_MAXE], prodsh[HN_MAXE];
#pragma unroll
  for (int a = 0; a < HN_MAXE; a++) cur[a] = a < ne ? p.shape0[a] : 1u;
  unsigned phase = 0;
  unsigned n_batches_done = 0;       // batches this CTA has pushed through the ring so far (same count on both sides)
  const double* src = p.res0;
  const unsigned stage_doubles = (unsigned)R * ng * bp.slot;
  for (unsigned step = 0; step < p.nsteps; step++) {
    double* dst = p.buf[step & 1u];
    const unsigned i = p.i_top - step;
    unsigned nsr = 1, QR = 1;          // super-rows (axes < ra) and rows per block (axes ra .. ne-2)
    long long cstr[HN_MAXE];
#pragma unroll
    for (int a = 0; a < HN_MAXE; a++) {
      if (a < ne) {
        const unsigned long long s = (unsigned long long)cur[a] + p.sshape[a] - 1ull;
        prodsh[a] = (unsigned)min(s, (unsigned long long)p.d[a]);
        nxt[a] = bp.add_mode ? max(prodsh[a], p.slice[a]) : prodsh[a];
        if (a < ra) nsr *= nxt[a];
        else if (a < ne - 1) QR *= nxt[a];
      } else {
        prodsh[a] = nxt[a] = 1u;
      }
    }
    {
      long long st = 1;
#pragma unroll
      for (int a = HN_MAXE - 1; a >= 0; --a) {
        if (a < ne) { cstr[a] = st; st *= (long long)cur[a]; } else cstr[a] = 0;
      }
    }
    const unsigned L_src = cur[ne - 1], L_out = nxt[ne - 1], L_prod = prodsh[ne - 1];
    const unsigned BS = QR * L_src, BO = QR * L_out;     // source / output elements of a block (rows per block equal: see host)
    const double* slice_base = p.self + (long long)i * p.self_vstr;
    const unsigned per_cta = (nsr + gridDim.x - 1) / gridDim.x;
    const unsigned row_lo = min(nsr, blockIdx.x * per_cta), row_hi = min(nsr, row_lo + per_cta);
    const unsigned nb = (row_hi - row_lo + R - 1) / R;

    if (warp == 0) {
      // ---------------- producer ----------------
      if (lane == 0) asm volatile("fence.proxy.async;" ::: "memory");   // other CTAs' generic-proxy stores (previous step)
      __syncwarp();
      for (unsigned b = 0; b < nb; b++) {
        const unsigned seq = n_batches_done + b, st = seq % HB_NS;
        if (seq >= HB_NS) mbar_wait(&s_empty[st], ((seq / HB_NS) - 1u) & 1u);   // the consumers released this stage's previous use
        double* base = hb_sm + (size_t)st * stage_doubles;
        const unsigned r0 = row_lo + b * R;
        unsigned bytes = 0;
        for (unsigned pr = lane; pr < (unsigned)(R * ng); pr += 32u) {
          const unsigned r = pr / ng, g = pr - r * ng;
          unsigned char sh = 255;
          if (r0 + r < row_hi) {
            unsigned rem = r0 + r;
            bool in_prod = true, in_slice = true, ok = true;
            long long so = 0, off = 0;
#pragma unroll
            for (int a = HN_MAXE - 2; a >= 0; --a) {
              if (a < ra) {
                const unsigned q = rem / nxt[a], ka = rem - q * nxt[a];
                rem = q;
                in_prod = in_prod && ka < prodsh[a];
                in_slice = in_slice && ka < p.slice[a];
                so += (long long)ka * p.selfstr[a];
                const unsigned idx = ka - (unsigned)bp.gm[g][a];
                ok = ok && idx < cur[a];
                off += (long long)idx * cstr[a];
              }
            }
            if (g == 0) {
              s_rowok[st][r] = (unsigned char)((in_prod ? 1 : 0) | (in_slice ? 2 : 0));
              s_so[st][r] = so;
            }
            if (ok && in_prod) {
              // copy [off - shift, off - shift + n): 16-byte aligned start, even length, never past the block's last element;
              // an odd tail element travels by an ordinary load and store of this lane (ordered before its arrival below)
              const unsigned shift = (unsigned)(off & 1ll);
              const unsigned n = (shift + BS) & ~1u;
              if (n) {
                bulk_g2s(base + (size_t)pr * bp.slot, src + (off - shift), n * 8u, &s_full[st]);
                bytes += n * 8u;
              }
              if (n < shift + BS) base[(size_t)pr * bp.slot + n] = ldcg(src + (off - shift) + n);
              sh = (unsigned char)shift;
            }
          }
          s_shift[st][pr] = sh;
        }
        __syncwarp();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) bytes += __shfl_xor_sync(0xffffffffu, bytes, o);
        __threadfence_block();
        __syncwarp();
        if (lane == 0) mbar_expect_tx(&s_full[st], bytes);   // release: the row tables and tail elements above are visible to whoever sees the phase
      }
    } else {
      // ---------------- consumers: a warp takes whole rows (no per-coefficient index decode), lanes along the row ----------------
      const unsigned cw = warp - 1u;
      constexpr unsigned NCW = NCONS / 32u;
      for (unsigned b = 0; b < nb; b++) {
        const unsigned seq = n_batches_done + b, st = seq % HB_NS;
        mbar_wait(&s_full[st], (seq / HB_NS) & 1u);
        const double* base = hb_sm + (size_t)st * stage_doubles;
        const unsigned r0 = row_lo + b * R;
        const unsigned rows_here = min((unsigned)R, row_hi - r0);
        for (unsigned rr = cw; rr < rows_here * QR; rr += NCW) {
          const unsigned r = rr / QR, q = rr - r * QR;
          const unsigned char rk = s_rowok[st][r];
          const unsigned sr = r0 + r;
          // slice row (Add general path): decode the block-axis indices of q once per row
          bool b_row = (rk & 2) != 0;
          long long so = s_so[st][r];
          if (bp.add_mode == 1) {
            unsigned rem = q;
#pragma unroll
            for (int a = HN_MAXE - 2; a >= 0; --a) {
              if (a >= ra && a < ne - 1) {
                const unsigned qq = rem / nxt[a], ka = rem - qq * nxt[a];
                rem = qq;
                b_row = b_row && ka < p.slice[a];
                so += (long long)ka * p.selfstr[a];
              }
            }
          }
          const unsigned qoff = q * L_src;
          double* drow = dst + (size_t)sr * BO + (size_t)q * L_out;
          // shared-space byte address of every group's block row (0: absent), once per row
          const unsigned stage_addr = sm_base + (unsigned)(st * stage_doubles) * 8u;
          for (unsigned c = lane; c < L_out; c += 32u) {
            const bool a_ok = (rk & 1) && c < L_prod;
            double prod = 0.0;
            if (a_ok) {
              double total_v = 0.0, inner = 0.0;
              bool open = false;
              unsigned gaddr = 0;
              int g = -1;
#pragma unroll
              for (int t = 0; t < NT; t++) {
                if (t < p.nt) {
                  if (p.group_start[t]) {
                    if (open) total_v = __dadd_rn(total_v, inner);
                    inner = 0.0;
                    g++;
                    const unsigned pr = r * ng + g;
                    const unsigned char sh = s_shift[st][pr];
                    open = sh != 255;                        // absent source block: the group is skipped
                    gaddr = stage_addr + (pr * bp.slot + sh + qoff) * 8u;
                  }
                  const unsigned cc = c - (unsigned)p.m[t][ne - 1];
                  if (open && cc < L_src) inner = __dadd_rn(inner, __dmul_rn(lds_f64(gaddr + cc * 8u), sv[t]));
                }
              }
              if (open) total_v = __dadd_rn(total_v, inner);
              prod = total_v;
            }
            double rv;
            if (bp.add_mode == 0) rv = prod;
            else if (bp.add_mode == 2) rv = (sr == 0 && q == 0 && c == 0) ? __dadd_rn(prod, slice_base[0]) : prod;
            else {
              rv = 0.0;
              if (a_ok) rv = __dadd_rn(rv, prod);
              if (b_row && c < p.slice[ne - 1]) rv = __dadd_rn(rv, slice_base[so + (long long)c * p.selfstr[ne - 1]]);
            }
            drow[c] = rv;
          }
        }
        mbar_arrive(&s_empty[st]);                           // this consumer is done with the stage
      }
    }
    n_batches_done += nb;
#pragma unroll
    for (int a = 0; a < HN_MAXE; a++) cur[a] = nxt[a];
    src = dst;
    if (step + 1 < p.nsteps) grid_barrier(p.bar, phase);
  }
}


// ---------------------------------------------------------------------------------------------------------------------
// Row-walking variant with plain coalesced loads.  A warp takes whole rows of the last effective axis (or 32 / W short rows
// at once, W = the row length rounded up to a power of two): the N-D index, the validity of every group of terms and the
// source offset of every term are computed ONCE PER ROW, so the element loop is NT back-to-back `ld.global.cg` (coalesced
// along the row, shifted re-reads of the same row are L2 hits), the reference-order multiply / add chain and one store --
// no integer division between loads, which is what keeps the per-coefficient gathers (k_horner, k_mul_stencil_v4) latency-
// bound at 45 % of HBM, and no staging ring whose small bulk copies complete too slowly (k_horner_rows as a single product).
// Arithmetic per coefficient and its order are k_horner's.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int HD_T = 256;
struct HornerDirectP {
  HornerP h;
  int add_mode;   // 0: product only, 1: Add general path, 2: Add scalar path
};

// MODE: 0 product only (plain stencil product), 1 Add general path, 2 Add scalar path (compile-time: no mode branches and no
// slice loads in the element loop of the other modes).
// Source rows are read with ordinary (L1-allocating) loads: the shifted re-read of a row by the next term of its group is an L1
// hit instead of a second trip to L2.  Data written by other CTAs in the previous step is ordered by the grid barrier (thread 0's
// acquire fence after the spin + bar.sync, the same protocol as cooperative-groups grid.sync(), after which plain loads are
// specified to observe it).
__device__ __forceinline__ double ld_row(const double* p) {
  double v;
  asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}
// GS: terms per group when every group has the same number (1 or 2: the substitution's extent along the last axis), else 0 --
// with it the group boundaries of the summation are compile-time and the arithmetic carries no selects.
template <int NT, int U, int MODE, int GS>
__global__ void __launch_bounds__(HD_T, (NT <= 4 ? (MODE == 0 ? 4 : 3) : (NT <= 8 ? 2 : 1))) k_horner_direct(const __grid_constant__ HornerDirectP dp) {
  const HornerP& p = dp.h;
  const int ne = p.ne;
  // step-constant extents and strides live in shared memory (they would cost ~50 registers as unrolled arrays)
  __shared__ unsigned s_cur[HN_MAXE], s_nxt[HN_MAXE], s_prodsh[HN_MAXE];
  __shared__ long long s_cstr[HN_MAXE];
  const unsigned lane = threadIdx.x & 31u;
  const unsigned warps_total = gridDim.x * (HD_T / 32), gw = blockIdx.x * (HD_T / 32) + (threadIdx.x >> 5);
  double sv[NT];
  unsigned gstart = 0;   // bit t: term t starts a group
  bool finite_sv = true;
#pragma unroll
  for (int t = 0; t < NT; t++) {
    sv[t] = t < p.nt ? p.subst[p.sidx[t]] : 0.0;
    if (t < p.nt && p.group_start[t]) gstart |= 1u << t;
    finite_sv = finite_sv && fabs(sv[t]) <= 1.7976931348623157e308;
  }
  if (threadIdx.x == 0)
    for (int a = 0; a < HN_MAXE; a++) s_nxt[a] = a < ne ? p.shape0[a] : 1u;
  unsigned phase = 0;
  const double* src = p.res0;
  for (unsigned step = 0; step < p.nsteps; step++) {
    double* dst = p.buf[step & 1u];
    const unsigned i = p.i_top - step;
    __syncthreads();
    if (threadIdx.x < HN_MAXE) {   // one lane per axis; the strides are a suffix product over the lanes
      const int a = (int)threadIdx.x;
      const unsigned ca = s_nxt[a];   // the previous step's result shape
      unsigned pa = 1u, na = 1u;
      if (a < ne) {
        const unsigned long long s = (unsigned long long)ca + p.sshape[a] - 1ull;
        pa = (unsigned)min(s, (unsigned long long)p.d[a]);
        na = MODE ? max(pa, p.slice[a]) : pa;
      }
      long long st = 1;
#pragma unroll
      for (int b = HN_MAXE - 1; b >= 1; --b) {
        const unsigned cb = __shfl_sync(0xffu, ca, b);
        if (b > a && b < ne) st *= (long long)cb;
      }
      s_cur[a] = ca;
      s_prodsh[a] = pa;
      s_nxt[a] = na;
      s_cstr[a] = a < ne ? st : 0;
    }
    __syncthreads();
    unsigned rows = 1;
    for (int a = 0; a < ne - 1; a++) rows *= s_nxt[a];
    const unsigned L_src = s_cur[ne - 1], L_out = s_nxt[ne - 1], L_prod = s_prodsh[ne - 1], L_slice = p.slice[ne - 1];
    unsigned W = 32;                       // lanes per row
    while (W > 1 && (W >> 1) >= L_out) W >>= 1;
    const unsigned G = 32u / W, sub = lane / W, c0 = lane & (W - 1u);
    const double* slice_base = p.self + (long long)i * p.self_vstr;
    const long long slice_cstr = p.selfstr[ne - 1];
    // Long rows (one row per warp at a time): every warp owns ONE contiguous range of rows -- balanced to within a row -- and
    // walks it: the first row is decoded in full, the following ones advance the index of the last row axis by one (pointers
    // move by one stride, no division) until that index wraps.  Short rows (several per warp): one group of rows per item.
    const unsigned n_items = G == 1u ? warps_total : (rows + G - 1) / G;
    const int al = ne - 2;   // the last row axis (>= 0: the kernel needs two effective axes)
    const unsigned n_last = s_nxt[al], c_last = s_cur[al], p_last = s_prodsh[al], sl_last = p.slice[al];
    const long long sa_last = s_cstr[al], self_last = p.selfstr[al];
    // ---- short rows (at most 32 coefficients) under at least two row axes: the last TWO axes are walked as one contiguous block
    // of the output (n_last rows of L_out), every lane busy; the row index inside the block comes from a multiply-high ----
    if (ne >= 3 && L_out <= 32u) {
      const unsigned BS = n_last * L_out, n_or = rows / n_last;
      const unsigned want = (warps_total + n_or - 1u) / n_or;                       // chunks per block that keep every warp busy
      const unsigned nchunk = max(1u, min((BS + 63u) / 64u, want));
      const unsigned CH = (((BS + nchunk - 1u) / nchunk) + 31u) & ~31u;
      const unsigned magic = (unsigned)(0x100000000ull / L_out) + 1u;                // e / L_out = umulhi(e, magic) for e < 2^32 / L_out
      unsigned mr[NT], ml[NT];
#pragma unroll
      for (int t = 0; t < NT; t++) { mr[t] = (unsigned)p.m[t][al]; ml[t] = (unsigned)p.m[t][ne - 1]; }
      for (unsigned item = gw; item < n_or * nchunk; item += warps_total) {
        const unsigned orow = item / nchunk, e_begin = (item - orow * nchunk) * CH, e_end = min(BS, e_begin + CH);
        bool in_prod_o = true, in_slice_o = true;
        unsigned open_o = (p.nt >= 32) ? 0xffffffffu : ((1u << p.nt) - 1u);
        long long so = 0, toff[NT];
#pragma unroll
        for (int t = 0; t < NT; t++) toff[t] = 0;
        {
          unsigned rem = orow;
          for (int a = al - 1; a >= 0; --a) {
            const unsigned na = s_nxt[a], ca = s_cur[a];
            const long long sa = s_cstr[a];
            const unsigned q = rem / na, ka = rem - q * na;
            rem = q;
            in_prod_o = in_prod_o && ka < s_prodsh[a];
            in_slice_o = in_slice_o && ka < p.slice[a];
            so += (long long)ka * p.selfstr[a];
#pragma unroll
            for (int t = 0; t < NT; t++) {
              const unsigned idx = ka - (unsigned)p.m[t][a];
              if (idx >= ca) open_o &= ~(1u << t);
              toff[t] += (long long)idx * sa;
            }
          }
        }
        if (!in_prod_o) open_o = 0;
        const unsigned pk = in_prod_o ? p_last : 0u, sk = (MODE == 1 && in_slice_o) ? sl_last : 0u;
        double* dblk = dst + (size_t)orow * BS;
        const double* sblk = slice_base + so;
        for (unsigned base = e_begin; base < e_end; base += U * 32u) {
          double xv[U][NT], sl[U];
          unsigned vm[U];
#pragma unroll
          for (int u = 0; u < U; u++) {
            const unsigned e = base + u * 32u + lane;
            const unsigned kk = __umulhi(e, magic), c = e - kk * L_out;
            const bool live = e < e_end && kk < pk && c < L_prod;
            vm[u] = 0;
#pragma unroll
            for (int t = 0; t < NT; t++) {
              const unsigned rk = kk - mr[t], rc = c - ml[t];
              const bool ok = live && ((open_o >> t) & 1u) && rk < c_last && rc < L_src;
              xv[u][t] = ok ? ld_row(src + (toff[t] + (long long)(int)(rk * L_src + rc))) : 0.0;
              vm[u] |= (ok ? 1u : 0u) << t;
            }
            if (MODE == 1) sl[u] = (e < e_end && kk < sk && c < L_slice) ? sblk[(long long)kk * self_last + (long long)c * slice_cstr] : 0.0;
          }
#pragma unroll
          for (int u = 0; u < U; u++) {
            const unsigned e = base + u * 32u + lane;
            if (e >= e_end) continue;
            const unsigned kk = __umulhi(e, magic), c = e - kk * L_out;
            double total_v = 0.0, inner = 0.0;
            if (finite_sv) {   // branch-free: see the long-row path below
#pragma unroll
              for (int t = 0; t < NT; t++) {
                if (t > 0 && (GS ? (t % (GS ? GS : 1)) == 0 : (((gstart >> t) & 1u) != 0u))) {
                  total_v = __dadd_rn(total_v, inner);
                  inner = 0.0;
                }
                inner = __dadd_rn(inner, __dmul_rn(xv[u][t], sv[t]));
              }
              total_v = __dadd_rn(total_v, inner);
            } else {
              bool open = false;
#pragma unroll
              for (int t = 0; t < NT; t++) {
                if (GS ? (t % (GS ? GS : 1)) == 0 && t < p.nt : (((gstart >> t) & 1u) != 0u)) {
                  if (open) total_v = __dadd_rn(total_v, inner);
                  inner = 0.0;
                  open = ((open_o >> t) & 1u) && (kk - mr[t]) < c_last;
                }
                if ((vm[u] >> t) & 1u) inner = __dadd_rn(inner, __dmul_rn(xv[u][t], sv[t]));
              }
              if (open) total_v = __dadd_rn(total_v, inner);
            }
            const bool a_ok = kk < pk && c < L_prod;
            const double prod = a_ok ? total_v : 0.0;
            double rv;
            if (MODE == 0) rv = prod;
            else if (MODE == 2) rv = (orow == 0 && e == 0) ? __dadd_rn(prod, slice_base[0]) : prod;
            else {
              rv = 0.0;
              if (a_ok) rv = __dadd_rn(rv, prod);
              if (kk < sk && c < L_slice) rv = __dadd_rn(rv, sl[u]);
            }
            dblk[e] = rv;
          }
        }
      }
      src = dst;
      if (step + 1 < p.nsteps) grid_barrier(p.bar, phase);
      continue;
    }
    for (unsigned item = gw; item < n_items; item += warps_total) {
      unsigned row, row_end;
      if (G == 1u) {
        row = (unsigned)(((unsigned long long)item * rows) / warps_total);
        row_end = (unsigned)(((unsigned long long)(item + 1u) * rows) / warps_total);
      } else {
        row = item * G + sub;
        row_end = row < rows ? row + 1u : row;
      }
      bool need_full = true;
      bool in_prod_o = true, in_slice_o = true;
      unsigned open_o = 0, k_last = 0;
      long long so = 0;
      int tp[NT];   // element offsets into `src` (tensors stay below 2^31 coefficients): one IMAD.WIDE per load, one register per term
      for (; row < row_end; row++) {
        if (need_full) {
          // ---- full decode: outer axes folded into flags / offsets, the last row axis kept as k_last ----
          in_prod_o = in_slice_o = true;
          so = 0;
          long long toff[NT];
          open_o = (p.nt >= 32) ? 0xffffffffu : ((1u << p.nt) - 1u);
#pragma unroll
          for (int t = 0; t < NT; t++) toff[t] = 0;
          unsigned rem = row;
          {
            const unsigned q = rem / n_last;
            k_last = rem - q * n_last;
            rem = q;
          }
          for (int a = al - 1; a >= 0; --a) {
            const unsigned na = s_nxt[a], ca = s_cur[a];
            const long long sa = s_cstr[a];
            const unsigned q = rem / na, ka = rem - q * na;
            rem = q;
            in_prod_o = in_prod_o && ka < s_prodsh[a];
            in_slice_o = in_slice_o && ka < p.slice[a];
            so += (long long)ka * p.selfstr[a];
#pragma unroll
            for (int t = 0; t < NT; t++) {
              const unsigned idx = ka - (unsigned)p.m[t][a];
              if (idx >= ca) open_o &= ~(1u << t);
              toff[t] += (long long)idx * sa;
            }
          }
          so += (long long)k_last * self_last;
#pragma unroll
          for (int t = 0; t < NT; t++)
            tp[t] = (int)(toff[t] + ((long long)k_last - (long long)p.m[t][al]) * sa_last - (long long)p.m[t][ne - 1] + (long long)c0);
          need_full = false;
        }
        // ---- per row: the last row axis ----
        const bool in_prod = in_prod_o && k_last < p_last, in_slice = in_slice_o && k_last < sl_last;
        unsigned openmask = open_o;
        unsigned lo[NT], span[NT];
#pragma unroll
        for (int t = 0; t < NT; t++) {
          if ((k_last - (unsigned)p.m[t][al]) >= c_last) openmask &= ~(1u << t);
          const unsigned ml = (unsigned)p.m[t][ne - 1];
          const bool ok = in_prod && ((openmask >> t) & 1u);
          const unsigned hi = min(L_prod, L_src + ml);
          lo[t] = ml;
          span[t] = (ok && hi > ml) ? hi - ml : 0u;
        }
        const unsigned drow = row * L_out + c0;   // element offset into `dst`
        const double* srow = slice_base + (so + (long long)c0 * slice_cstr);
        const unsigned prod_end = in_prod ? L_prod : 0u, slice_end = (MODE == 1 && in_slice) ? L_slice : 0u;
        // ---- the row: U chunks per trip, every load of all chunks issued before the first use ----
        for (unsigned base = 0; base < L_out; base += U * W) {
          double xv[U][NT], sl[U];
  #pragma unroll
          for (int u = 0; u < U; u++) {
            const unsigned idx = base + u * W, cu = idx + c0;
  #pragma unroll
            for (int t = 0; t < NT; t++) xv[u][t] = (cu - lo[t]) < span[t] ? ld_row(src + (tp[t] + (int)idx)) : 0.0;
            if (MODE == 1) sl[u] = cu < slice_end ? srow[(long long)idx * slice_cstr] : 0.0;
          }
          if (finite_sv) {
            // Branch-free arithmetic.  An absent term was loaded as +0.0 and contributes (+-0) to a sum that is never -0 (every
            // sum starts from +0.0), a closed group contributes +0.0 to the total, a coefficient outside the product / the slice
            // adds +0.0 to a value that is never -0: bit-identical to skipping them, as long as the substitution's coefficients
            // are finite (0 * inf would not be) -- checked once per launch; otherwise the predicated form below runs.
  #pragma unroll
            for (int u = 0; u < U; u++) {
              const unsigned idx = base + u * W, cu = idx + c0;
              double total_v = 0.0, inner = 0.0;
  #pragma unroll
              for (int t = 0; t < NT; t++) {
                if (t > 0 && (GS ? (t % (GS ? GS : 1)) == 0 : (((gstart >> t) & 1u) != 0u))) {
                  total_v = __dadd_rn(total_v, inner);
                  inner = 0.0;
                }
                inner = __dadd_rn(inner, __dmul_rn(xv[u][t], sv[t]));
              }
              total_v = __dadd_rn(total_v, inner);
              double rv;
              if (MODE == 0) rv = total_v;
              else if (MODE == 2) rv = (row == 0 && cu == 0) ? __dadd_rn(total_v, slice_base[0]) : total_v;
              else rv = __dadd_rn(__dadd_rn(0.0, total_v), sl[u]);
              if (cu < L_out) dst[drow + idx] = rv;
            }
            continue;
          }
  #pragma unroll
          for (int u = 0; u < U; u++) {
            const unsigned idx = base + u * W, cu = idx + c0;
            if (cu >= L_out) continue;
            // the product in the reference's order: groups ascending, the innermost axis summed from zero and then added
            double total_v = 0.0, inner = 0.0;
            bool open = false;
  #pragma unroll
            for (int t = 0; t < NT; t++) {
              if (GS ? (t % (GS ? GS : 1)) == 0 && t < p.nt : (((gstart >> t) & 1u) != 0u)) {
                if (open) total_v = __dadd_rn(total_v, inner);
                inner = 0.0;
                open = (openmask >> t) & 1u;
              }
              if ((cu - lo[t]) < span[t]) inner = __dadd_rn(inner, __dmul_rn(xv[u][t], sv[t]));
            }
            if (open) total_v = __dadd_rn(total_v, inner);
            const bool a_ok = cu < prod_end;
            const double prod = a_ok ? total_v : 0.0;
            double rv;
            if (MODE == 0) rv = prod;
            else if (MODE == 2) rv = (row == 0 && cu == 0) ? __dadd_rn(prod, slice_base[0]) : prod;
            else {
              rv = 0.0;
              if (a_ok) rv = __dadd_rn(rv, prod);
              if (cu < slice_end) rv = __dadd_rn(rv, sl[u]);
            }
            dst[drow + idx] = rv;
          }
        }
        // ---- advance to the next row of the block ----
        k_last++;
        if (k_last == n_last) {
          need_full = true;
        } else {
          so += self_last;
#pragma unroll
          for (int t = 0; t < NT; t++) tp[t] += (int)sa_last;
        }
      }
    }
    src = dst;
    if (step + 1 < p.nsteps) grid_barrier(p.bar, phase);
  }
}

// One cooperative launch of a Horner kernel: the kernel, its geometry and its parameters
struct HornerLaunch {
  const void* fn;
  unsigned grid;
  int block;
  size_t smem;
  const char* tag;   // its name in the GTP_LAUNCH_HIST census
  union {
    HornerP h;
    HornerDirectP direct;
    HornerBulkP bulk;
  } params;
};

void launch_horner_plan(Ctx& ctx, const HornerLaunch& pl) {
  coop_launch(ctx, pl.fn, pl.grid, pl.block, pl.smem, const_cast<void*>((const void*)&pl.params), pl.tag);
}

// Plans k_horner_direct for the steps of `p`; false: outside its domain.
static bool plan_direct_variant(const Ctx& ctx, const HornerP& p, int add_mode, const unsigned* final_shape, u64 final_total, const char* tag,
                                HornerLaunch* pl) {
  if (!ctx.use_direct || p.ne < 2) return false;
  const unsigned L_final = final_shape[p.ne - 1];
  if ((L_final < 48 && p.ne < 3) || final_total < ctx.direct_min) return false;   // short rows need a second row axis to walk blocks
  if (add_mode == 0 && L_final < 192 && !ctx.direct_products_all) return false;   // plain products: the gather kernel wins on shorter rows
  HornerDirectP& dp = pl->params.direct;
  memset(&dp, 0, sizeof(dp));
  dp.h = p;
  dp.add_mode = add_mode;
  const void* fn;
  // uniform group size (terms per group): 1 or 2 for the usual substitutions, else 0 = read the group starts at run time
  int gsz = 0;
  {
    int cnt = 0, first = -1;
    bool uniform = true;
    for (int t = 0; t <= p.nt; t++) {
      if (t == p.nt || p.group_start[t]) {
        if (t > 0) {
          if (first < 0) first = cnt;
          uniform = uniform && cnt == first;
        }
        cnt = 0;
      }
      cnt++;
    }
    if (uniform && (first == 1 || first == 2) && p.nt % first == 0) gsz = first;
  }
#define HD_PICK3(NT_, U_, GS_) (add_mode == 0 ? (const void*)k_horner_direct<NT_, U_, 0, GS_> : (add_mode == 1 ? (const void*)k_horner_direct<NT_, U_, 1, GS_> : (const void*)k_horner_direct<NT_, U_, 2, GS_>))
#define HD_PICK(NT_, U_) (gsz == 2 ? HD_PICK3(NT_, U_, 2) : (gsz == 1 ? HD_PICK3(NT_, U_, 1) : HD_PICK3(NT_, U_, 0)))
  if (p.nt <= 2) fn = HD_PICK(2, 4);
  else if (p.nt <= 4) fn = HD_PICK(4, 2);
  else if (p.nt <= 8) fn = HD_PICK(8, 2);
  else if (p.nt <= 16) fn = HD_PICK3(16, 1, 0);
  else fn = HD_PICK3(32, 1, 0);
#undef HD_PICK
#undef HD_PICK3
  const int per_sm = coop_ctas_per_sm(fn, ctx.device, HD_T, 0);
  if (per_sm == 0) return false;
  // rows per warp item at the final shape; mid-size tensors are barrier-bound (fewer CTAs), HBM-sized ones want loads in flight
  unsigned W = 32;
  while (W > 1 && (W >> 1) >= L_final) W >>= 1;
  const u64 items = (final_total / L_final + (32 / W) - 1) / (32 / W);
  const int want_per_sm = final_total >= (1u << 21) ? ctx.direct_ctas : (final_total >= (1u << 18) ? 2 : 1);
  const int ctas_per_sm = std::max(1, std::min(per_sm, want_per_sm));
  pl->fn = fn;
  pl->grid = (unsigned)std::max<u64>(1, std::min<u64>((items + HD_T / 32 - 1) / (HD_T / 32), (u64)ctas_per_sm * ctx.sm_count));
  pl->block = HD_T;
  pl->smem = 0;
  pl->tag = tag;
  return true;
}

// Fills the group tables from the (sorted) terms of `p` and plans k_horner_rows; false: outside its domain.
static bool plan_rows_variant(const Ctx& ctx, const HornerP& p, int add_mode, const unsigned* final_shape, u64 final_total, const char* tag,
                              HornerLaunch* pl) {
  if (!ctx.use_bulk || p.ne < 2) return false;
  const unsigned L_final = final_shape[p.ne - 1];
  if (L_final < 16 || L_final > 2048 || final_total < (1u << 18)) return false;
  if ((reinterpret_cast<uintptr_t>(p.res0) & 15u) || (reinterpret_cast<uintptr_t>(p.buf[0]) & 15u) || (reinterpret_cast<uintptr_t>(p.buf[1]) & 15u)) return false;
  HornerBulkP& bp = pl->params.bulk;
  memset(&bp, 0, sizeof(bp));
  bp.h = p;
  bp.add_mode = add_mode;
  int ng = 0;
  for (int t = 0; t < p.nt; t++) {
    if (p.group_start[t]) {
      if (ng == HB_MAXG) return false;
      for (int e = 0; e < p.ne - 1; e++) bp.gm[ng][e] = p.m[t][e];
      bp.g_first[ng] = (unsigned char)t;
      bp.g_count[ng] = 0;
      ng++;
    }
    bp.g_count[ng - 1]++;
  }
  bp.ng = ng;
  // Row block: trailing axes on which the substitution is constant and the slice is no longer than the incoming value are
  // merged with the last axis while the block stays <= 1024 coefficients -- one bulk copy then covers several short rows
  // (16^6 x [2,1,2,1,1,2]: 16 rows of 16).  On those axes product, result and source extents coincide at every step.
  int ra = p.ne - 1;
  u64 block = L_final;
  while (ra > 0) {
    const int a = ra - 1;
    if (p.sshape[a] != 1 || p.slice[a] > p.shape0[a] || final_shape[a] != p.shape0[a]) break;
    bool offs = false;
    for (int t = 0; t < p.nt; t++) offs |= p.m[t][a] != 0;
    if (offs || block * final_shape[a] > 1024) break;
    block *= final_shape[a];
    ra = a;
  }
  if (ra < 1 || block < 64) return false;       // short rows that cannot be merged: per-copy overhead dominates
  bp.ra = ra;
  bp.slot = (unsigned)((block + 3) & ~1ull);
  int R = (int)std::max<u64>(1, std::min<u64>(HB_R, (24 * 1024 / 8) / ((u64)ng * bp.slot)));   // <= 24 KB per stage
  bp.R = R;
  const size_t smem = (size_t)HB_NS * R * ng * bp.slot * sizeof(double);
  if (smem > 200 * 1024) return false;
  const void* fn;
  if (p.nt <= 2) fn = (const void*)k_horner_rows<2>;
  else if (p.nt <= 4) fn = (const void*)k_horner_rows<4>;
  else if (p.nt <= 8) fn = (const void*)k_horner_rows<8>;
  else if (p.nt <= 16) fn = (const void*)k_horner_rows<16>;
  else fn = (const void*)k_horner_rows<32>;
  const int per_sm = coop_ctas_per_sm(fn, ctx.device, HB_T, smem);
  if (per_sm == 0) return false;
  const u64 nsr = final_total / block;
  pl->fn = fn;
  pl->grid = (unsigned)std::max<u64>(1, std::min<u64>((nsr + R - 1) / R, (u64)std::min(per_sm, 4) * ctx.sm_count));
  pl->block = HB_T;
  pl->smem = smem;
  pl->tag = tag;
  return true;
}

// Host side.  `self`: the polynomial whose axis v is substituted (shape self_shape, already zero-extended to the common
// ndim), `d`: result degrees, `subst`: shape sshape (<= 32 coefficients, <= d), `res`: the running Horner value (shape
// rshape) BEFORE the step that adds slice i_top.  Runs the steps i_top, i_top-1, .., 0 and returns the final buffer and
// shape; false when the case is outside the kernel's domain (the caller continues with per-operator steps).
bool launch_horner(Ctx& ctx, const double* self, const Shape& self_shape, u64 v, const Shape& d, const double* subst,
                   const Shape& sshape, const double* res, const Shape& rshape, u64 i_top, BufP* out_buf, Shape* out_shape) {
  const int nd = (int)d.size();
  if ((int)self_shape.size() != nd || (int)sshape.size() != nd || (int)rshape.size() != nd) return false;
  const u64 ns = prod(sshape);
  if (ns < 2 || ns > (u64)HN_MAXT || prod(rshape) < 2) return false;
  Shape slice(nd);
  for (int a = 0; a < nd; a++) slice[a] = std::min(self_shape[a], d[a]);
  slice[v] = 1;
  // effective axes: the non-unit axes of res; every axis that can become non-unit must already be one
  int eff[HN_MAXE], ne = 0;
  for (int a = 0; a < nd; a++) {
    if (rshape[a] > 1) {
      if (ne == HN_MAXE) return false;
      eff[ne++] = a;
    } else if (sshape[a] > 1 || slice[a] > 1) {
      return false;
    }
    if (sshape[a] > d[a] || sshape[a] > 255) return false;
  }
  if (ne < 1) return false;
  // final shape (the same recurrence the kernel runs) and overflow checks
  Shape cur = rshape;
  const u64 nsteps = i_top + 1;
  for (u64 s = 0; s < nsteps; s++) {
    bool changed = false;
    for (int a = 0; a < nd; a++) {
      u64 pr = std::min<u64>(d[a], cur[a] + sshape[a] - 1);
      u64 nx = std::max<u64>(pr, slice[a]);
      changed |= nx != cur[a];
      cur[a] = nx;
    }
    if (!changed) break;
  }
  const u64 final_total = prod(cur);
  if (final_total >= (1ull << 31) || prod(self_shape) >= (1ull << 40)) return false;
  HornerP p;
  memset(&p, 0, sizeof(p));
  p.ne = ne;
  Shape selfst(nd, 1);
  for (int a = nd - 2; a >= 0; --a) selfst[a] = selfst[a + 1] * self_shape[a + 1];
  for (int e = 0; e < ne; e++) {
    const int a = eff[e];
    p.d[e] = d[a] >= 0xffffffffull ? 0xffffffffu : (unsigned)d[a];
    p.sshape[e] = (unsigned)sshape[a];
    p.slice[e] = (unsigned)slice[a];
    p.selfstr[e] = (long long)selfst[a];
    p.shape0[e] = (unsigned)rshape[a];
  }
  p.self_vstr = (long long)selfst[v];
  // terms of subst in the reference's visiting order: X = res index ascending <=> m descending
  set_terms(&p, small_terms(sshape, eff, ne, true));
  p.self = self;
  p.subst = subst;
  p.res0 = res;
  p.i_top = (unsigned)i_top;
  p.nsteps = (unsigned)nsteps;
  p.slice_scalar = prod(slice) == 1 ? 1 : 0;
  BufP b0 = ctx.alloc(final_total), b1 = nsteps > 1 ? ctx.alloc(final_total) : BufP();
  BufP bar = ctx.alloc(2);
  GTP_CUDA(cudaMemsetAsync(bar->d, 0, 16, ctx.stream));
  p.buf[0] = b0->d;
  p.buf[1] = b1 ? b1->d : b0->d;
  p.bar = reinterpret_cast<unsigned*>(bar->d);
  unsigned fs[HN_MAXE];
  for (int e = 0; e < ne; e++) fs[e] = (unsigned)cur[eff[e]];
  const int add_mode = p.slice_scalar ? 2 : 1;
  HornerLaunch pl;
  if (!plan_direct_variant(ctx, p, add_mode, fs, final_total, "k_horner_direct", &pl) &&
      !plan_rows_variant(ctx, p, add_mode, fs, final_total, "k_horner_rows", &pl)) {
    const int per_sm = coop_ctas_per_sm((const void*)k_horner, ctx.device, HN_T, 0);
    if (per_sm == 0) return false;
    const u64 want = (final_total + HN_T - 1) / HN_T;
    // small and mid-size tensors are barrier-bound (a step is ~1 us of L2 traffic): one CTA per SM keeps the barrier short;
    // HBM-sized tensors want every resident CTA for loads in flight
    const int ctas_per_sm = final_total >= (1u << 21) ? std::min(per_sm, 4) : (final_total >= (1u << 18) ? std::min(per_sm, 2) : 1);
    pl.params.h = p;
    pl.fn = (const void*)k_horner;
    pl.grid = (unsigned)std::max<u64>(1, std::min<u64>(want, (u64)ctas_per_sm * ctx.sm_count));
    pl.block = HN_T;
    pl.smem = 0;
    pl.tag = "k_horner";
  }
  launch_horner_plan(ctx, pl);
  *out_buf = ((nsteps - 1) & 1) ? b1 : b0;
  *out_shape = cur;
  return true;
}

// The plain small-operand product (the small-operand route of kernels_mul.cu) as one step of the Horner kernels without
// the Add.  Null: outside their domain (the caller goes on to the stencil kernels).
std::shared_ptr<const HornerLaunch> plan_small_rows(const Ctx& ctx, const MulArgs& a) {
  const int nd = a.ndim;
  if (a.accumulate || !a.rows.empty() || nd < 2 || a.row_begin != 0 || a.row_step != 1 || a.row_count != a.rs[0]) return nullptr;
  {  // cheap rejections first: this sits on the path of every small-operand product, most of them tiny
    u64 total = 1, last = 1;
    for (int d = 0; d < nd; d++) {
      total *= a.rs[d];
      if (a.rs[d] > 1) last = a.rs[d];
    }
    const bool direct = ctx.direct_products && ctx.use_direct && total >= ctx.direct_min && (last >= 192 || ctx.direct_products_all);
    const bool bulk = ctx.bulk_products && ctx.use_bulk && total >= (1u << 18);
    if (!direct && !bulk) return nullptr;
  }
  const u64 nx = prod(a.xs), ny = prod(a.ys);
  const bool small_is_x = nx <= ny;
  const Shape& ss = small_is_x ? a.xs : a.ys;
  const Shape& bs = small_is_x ? a.ys : a.xs;
  const u64 ns = std::min(nx, ny);
  if (ns < 1 || ns > (u64)HN_MAXT) return nullptr;
  int eff[HN_MAXE], ne = 0;
  for (int d = 0; d < nd; d++) {
    if (a.rs[d] == 1) {
      if (a.xs[d] != 1 || a.ys[d] != 1) return nullptr;
      continue;
    }
    if (a.rs[d] > bs[d] + ss[d] - 1 || ss[d] > 255) return nullptr;   // no rows / columns beyond the product's own extent
    if (ne == HN_MAXE) return nullptr;
    eff[ne++] = d;
  }
  if (ne < 2) return nullptr;
  const u64 total = prod(a.rs);
  if (total >= (1ull << 31) || prod(bs) >= (1ull << 31)) return nullptr;
  HornerP p;
  memset(&p, 0, sizeof(p));
  p.ne = ne;
  unsigned fs[HN_MAXE];
  for (int e = 0; e < ne; e++) {
    const int d = eff[e];
    p.d[e] = (unsigned)a.rs[d];
    p.sshape[e] = (unsigned)ss[d];
    p.slice[e] = 1;
    p.shape0[e] = (unsigned)bs[d];
    fs[e] = (unsigned)a.rs[d];
  }
  set_terms(&p, small_terms(ss, eff, ne, !small_is_x));   // ascending X index
  p.self = small_is_x ? a.y : a.x;    // unused (no Add), any valid pointer
  p.subst = small_is_x ? a.x : a.y;
  p.res0 = small_is_x ? a.y : a.x;
  p.buf[0] = p.buf[1] = a.out;
  p.i_top = 0;
  p.nsteps = 1;
  p.bar = nullptr;   // a single step never reaches the grid barrier
  HornerLaunch pl;
  if ((ctx.direct_products && plan_direct_variant(ctx, p, 0, fs, total, "k_horner_direct<product>", &pl)) ||
      (ctx.bulk_products && plan_rows_variant(ctx, p, 0, fs, total, "k_horner_rows<product>", &pl)))
    return std::make_shared<const HornerLaunch>(pl);
  return nullptr;
}

}  // namespace gtp
