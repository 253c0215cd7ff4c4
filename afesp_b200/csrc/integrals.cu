// Packed-ERI kernels: AO->MO transformation, MP2 energy, and the integral slices the CC drivers consume.
//
// Replaces src/mp2.f90:285-438 (four O(n^5) quarter transforms over dense n^4 temporaries, serial repack, MP2 sum)
// and the gathers of src/ccsd.f90:111-143,182-194 (spin-orbital <pq||rs>) and :496-512 (spin-free slices).
//
// Packing (src/integrals.f90:196-210, 0-based here): pair(i,j) = max(max+1)/2 + min; eri[pair(pair(i,j),pair(k,l))].
// 64-bit indices throughout (the reference's default-integer neri overflows at nbf = 400, SURVEY.md K8).
//
// AO->MO is done as two half transforms over *pair-packed* matrices instead of dense n^4 arrays:
//   phase 1:  H(kl, pq) = sum_ij C(p,i) C(q,j) (ij|kl)        (kl = spectator pair, p>=q packed)
//   phase 2:  (pq|rs)   = sum_kl C(r,k) C(s,l) H(kl, pq)      (pq = spectator pair, r>=s packed)
// Each phase processes spectator blocks:  unpack -> DMMA GEMM -> batched DMMA GEMM -> pack.  Flops 8 n^3 npair
// (half the dense 8 n^5), peak extra memory npair^2 doubles (51 GB at n=400 vs 2 x 205 GB dense).
#include "integrals.cuh"

#include <algorithm>

#include "kernels.cuh"

namespace afesp {
namespace {

__host__ __device__ __forceinline__ long long tri(long long i, long long j) {
  return i >= j ? i * (i + 1) / 2 + j : j * (j + 1) / 2 + i;
}

// X(xb, k, l) = src(x0+xb ; pair(k,l)),  xb fastest.
// mode 0: src is the packed triangular ERI array: src[tri(x, kl)]
// mode 1: src is a full matrix S[kl + ld * x]   (spectator is the *column*; used by phase 2 on H(kl,pq))
__global__ void k_unpack_pairs(double* __restrict__ X, const double* __restrict__ src, int mode, long long ld,
                               long long x0, int nb, int n) {
  const long long total = (long long)nb * n * n;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int xb = (int)(idx % nb);
    long long kl = idx / nb;
    int k = (int)(kl % n), l = (int)(kl / n);
    long long pr = tri(k, l);
    X[idx] = mode == 0 ? src[tri(x0 + xb, pr)] : src[pr + ld * (x0 + xb)];
  }
}

// Variant for mode 1 that reads S coalesced along kl and writes X coalesced along xb (32x32 smem transpose over
// (pair index, spectator)).  Grid: (ceil(npair/32), ceil(nb/32)).  Writes both X(xb,k,l) and X(xb,l,k).
// Only pairs pr in [pr_lo, npair) are handled (grid.x covers that range): with several GPUs the rows of S arrive in
// one chunk per source rank, each with its own base pointer and leading dimension.
__global__ void k_unpack_pairs_T(double* __restrict__ X, const double* __restrict__ S, long long ld, long long x0,
                                 int nb, int n, long long npair, long long pr_lo) {
  __shared__ double tile[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const long long pr0 = pr_lo + (long long)blockIdx.x * 32;
  const int xb0 = blockIdx.y * 32;
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    long long pr = pr0 + tx;
    int xb = xb0 + r;
    if (pr < npair && xb < nb) tile[r][tx] = S[(pr - pr_lo) + ld * (x0 + xb)];
  }
  __syncthreads();
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    long long pr = pr0 + r;
    int xb = xb0 + tx;
    if (pr < npair && xb < nb) {
      // invert pr -> (k >= l)
      long long k = (long long)((sqrt(8.0 * (double)pr + 1.0) - 1.0) * 0.5);
      while (k * (k + 1) / 2 > pr) --k;
      while ((k + 1) * (k + 2) / 2 <= pr) ++k;
      long long l = pr - k * (k + 1) / 2;
      double v = tile[tx][r];
      X[xb + (long long)nb * (k + n * l)] = v;
      X[xb + (long long)nb * (l + n * k)] = v;
    }
  }
}

// dest(x0+xb ; pair(r,s)) = Z(xb, r, s) for r >= s.
// mode 0: dest is a matrix D[(x - xoff) + ld * pair]   (phase 1: H(kl,pq), spectator = row, coalesced along xb;
//         xoff = first spectator this rank owns)
// mode 1: dest is the packed triangular array, only pair <= x is stored: D[tri(x, pair)]   (phase 2)
__global__ void k_pack_pairs(double* __restrict__ D, const double* __restrict__ Z, int mode, long long ld, long long x0,
                             int nb, int n, long long xoff) {
  const long long total = (long long)nb * n * n;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int xb = (int)(idx % nb);
    long long rs = idx / nb;
    int r = (int)(rs % n), s = (int)(rs / n);
    if (r < s) continue;
    long long pr = tri(r, s), x = x0 + xb;
    if (mode == 0) D[(x - xoff) + ld * pr] = Z[idx];
    else if (pr <= x) D[x * (x + 1) / 2 + pr] = Z[idx];
  }
}

// i, j run over the active occupied orbitals [k, o), a, b over the virtuals [o, n)
__global__ void __launch_bounds__(256) k_mp2(const double* __restrict__ g, const double* __restrict__ eps, int n, int o,
                                              int k, double* __restrict__ partials) {
  const int v = n - o, oa = o - k;
  const long long total = (long long)oa * oa * v * v;
  double acc = 0.0;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int b = (int)(idx % v) + o;
    long long t = idx / v;
    int a = (int)(t % v) + o;
    t /= v;
    int j = (int)(t % oa) + k, i = (int)(t / oa) + k;
    long long ia = tri(i, a), jb = tri(j, b), ib = tri(i, b), ja = tri(j, a);
    double iajb = g[tri(ia, jb)];
    acc += iajb * (2.0 * iajb - g[tri(ib, ja)]) / (eps[i] + eps[j] - eps[a] - eps[b]);
  }
  __shared__ double sh[8];
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += sh[w];
    partials[blockIdx.x] = s;
  }
}

struct SliceSpec { int lo[4], n[4]; };

// out(p,q,r,s) = <PQ|RS> = (PR|QS), P = lo0+p, ... (physicist order, src/ccsd.f90:500-501)
__global__ void k_slice_phys(double* __restrict__ out, const double* __restrict__ g, SliceSpec sp) {
  const long long total = (long long)sp.n[0] * sp.n[1] * sp.n[2] * sp.n[3];
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long t = idx;
    int p = (int)(t % sp.n[0]) + sp.lo[0]; t /= sp.n[0];
    int q = (int)(t % sp.n[1]) + sp.lo[1]; t /= sp.n[1];
    int r = (int)(t % sp.n[2]) + sp.lo[2]; t /= sp.n[2];
    int s = (int)t + sp.lo[3];
    out[idx] = g[tri(tri(p, r), tri(q, s))];
  }
}

__device__ __forceinline__ double asym_spinorb(const double* __restrict__ g, int P, int Q, int R, int S);
// out(P,Q,R,S) = <PQ||RS> over spin-orbitals (even = alpha, odd = beta of spatial orbital P/2), src/ccsd.f90:111-143
__global__ void k_slice_spinorb(double* __restrict__ out, const double* __restrict__ g, SliceSpec sp) {
  const long long total = (long long)sp.n[0] * sp.n[1] * sp.n[2] * sp.n[3];
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long t = idx;
    int P = (int)(t % sp.n[0]) + sp.lo[0]; t /= sp.n[0];
    int Q = (int)(t % sp.n[1]) + sp.lo[1]; t /= sp.n[1];
    int R = (int)(t % sp.n[2]) + sp.lo[2]; t /= sp.n[2];
    int S = (int)t + sp.lo[3];
    out[idx] = asym_spinorb(g, P, Q, R, S);
  }
}

// Permutational-symmetry self-check of the antisymmetrised spin-orbital integrals (src/ccsd.f90:150-167):
//   err = sum_{p, q<=p, r<=p, s<=r} |<pq||rs> + <pq||sr>| + |<pq||rs> - <rs||pq>| + |<pq||rs> + <sr||pq>| + |<pq||rs> - <sr||qp>|
// evaluated from the packed MO integrals through the same element function the slices are gathered with (the (2n)^4
// tensor of :108 is never formed).  One thread per (p,q,r,s) of the full (2n)^4 box, masked to the reference's range;
// warp-shuffle + per-block partial sums (fixed order: deterministic).
__device__ __forceinline__ double asym_spinorb(const double* __restrict__ g, int P, int Q, int R, int S) {
  const int p = P >> 1, q = Q >> 1, r = R >> 1, s = S >> 1;
  double val = 0.0;
  if ((P & 1) == (R & 1) && (Q & 1) == (S & 1)) val += g[tri(tri(p, r), tri(q, s))];
  if ((P & 1) == (S & 1) && (Q & 1) == (R & 1)) val -= g[tri(tri(p, s), tri(q, r))];
  return val;
}
// The box is the spin-orbitals [lo, lo + n2): lo = 2k when k core orbitals are frozen.
__global__ void k_spinorb_symmetry(const double* __restrict__ g, int lo, int n2, double* __restrict__ partials) {
  const long long total = (long long)n2 * n2 * n2 * n2;
  double err = 0.0;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long t = idx;
    const int s = (int)(t % n2) + lo; t /= n2;
    const int r = (int)(t % n2) + lo; t /= n2;
    const int q = (int)(t % n2) + lo;
    const int p = (int)(t / n2) + lo;
    if (q > p || r > p || s > r) continue;
    const double x = asym_spinorb(g, p, q, r, s);
    err += fabs(x + asym_spinorb(g, p, q, s, r)) + fabs(x - asym_spinorb(g, r, s, p, q)) +
           fabs(x + asym_spinorb(g, s, r, p, q)) + fabs(x - asym_spinorb(g, s, r, q, p));
  }
  __shared__ double red[8];
  for (int off = 16; off > 0; off >>= 1) err += __shfl_down_sync(0xffffffffu, err, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = err;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s2 = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s2 += red[w];
    partials[blockIdx.x] = s2;
  }
}

// (+/-)-symmetrised virtual-pair integrals for the particle-particle ladder:
//   Vp(ef, ab) = <ef|ab> + <ef|ba>,  e<=f, a<=b   (P+ = v(v+1)/2 pairs, pair(a,b) = b(b+1)/2 + a)
//   Vm(ef, ab) = <ef|ab> - <ef|ba>,  e<f,  a<b    (P- = v(v-1)/2 pairs, pair(a,b) = b(b-1)/2 + a)
// <ef|ab> = (ea|fb), virtual indices offset by voff (= nocc) in the packed MO array.
__global__ void k_build_vpm(double* __restrict__ V, const double* __restrict__ g, int voff, int v, int sign,
                            long long col0, long long ncols) {
  const long long P = sign > 0 ? (long long)v * (v + 1) / 2 : (long long)v * (v - 1) / 2;
  const long long total = P * ncols;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long ef = idx % P, ab = col0 + idx / P;
    long long f, e, b, a;
    if (sign > 0) {
      f = (long long)((sqrt(8.0 * (double)ef + 1.0) - 1.0) * 0.5);
      while (f * (f + 1) / 2 > ef) --f;
      while ((f + 1) * (f + 2) / 2 <= ef) ++f;
      e = ef - f * (f + 1) / 2;
      b = (long long)((sqrt(8.0 * (double)ab + 1.0) - 1.0) * 0.5);
      while (b * (b + 1) / 2 > ab) --b;
      while ((b + 1) * (b + 2) / 2 <= ab) ++b;
      a = ab - b * (b + 1) / 2;
    } else {
      f = (long long)((sqrt(8.0 * (double)ef + 1.0) + 1.0) * 0.5);
      while (f * (f - 1) / 2 > ef) --f;
      while ((f + 1) * f / 2 <= ef) ++f;
      e = ef - f * (f - 1) / 2;
      b = (long long)((sqrt(8.0 * (double)ab + 1.0) + 1.0) * 0.5);
      while (b * (b - 1) / 2 > ab) --b;
      while ((b + 1) * b / 2 <= ab) ++b;
      a = ab - b * (b - 1) / 2;
    }
    const long long E = e + voff, F = f + voff, A = a + voff, B = b + voff;
    const double x = g[tri(tri(E, A), tri(F, B))];   // <ef|ab>
    const double y = g[tri(tri(E, B), tri(F, A))];   // <ef|ba>
    V[idx] = sign > 0 ? x + y : x - y;
  }
}

// S(ij, e<=f) = c(ij,ef) + c(ij,fe) (e<f), c(ij,ee) (e==f);   A(ij, e<f) = c(ij,ef) - c(ij,fe)
__global__ void k_pack_c(double* __restrict__ S, double* __restrict__ A, const double* __restrict__ c, int oo, int v) {
  const long long Pp = (long long)v * (v + 1) / 2, Pm = (long long)v * (v - 1) / 2;
  const long long total = (long long)oo * v * v;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int ij = (int)(idx % oo);
    long long ef = idx / oo;
    int e = (int)(ef % v), f = (int)(ef / v);
    if (e > f) continue;
    double x = c[idx];
    if (e == f) {
      S[ij + (long long)oo * ((long long)f * (f + 1) / 2 + e)] = x;
    } else {
      double y = c[ij + (long long)oo * (f + (long long)v * e)];
      S[ij + (long long)oo * ((long long)f * (f + 1) / 2 + e)] = x + y;
      A[ij + (long long)oo * ((long long)f * (f - 1) / 2 + e)] = x - y;
    }
  }
  (void)Pp; (void)Pm;
}

// X(ij,a,b) += alpha/2 (Lp + Lm), X(ij,b,a) += alpha/2 (Lp - Lm) for a<b;  X(ij,a,a) += alpha/2 Lp
__global__ void k_unpack_ladder(double* __restrict__ X, const double* __restrict__ Lp, const double* __restrict__ Lm,
                                int oo, int v, double alpha) {
  const long long total = (long long)oo * v * v;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int ij = (int)(idx % oo);
    long long ab = idx / oo;
    int a = (int)(ab % v), b = (int)(ab / v);
    int lo = a < b ? a : b, hi = a < b ? b : a;
    double lp = Lp[ij + (long long)oo * ((long long)hi * (hi + 1) / 2 + lo)];
    double r = 0.5 * lp;
    if (a != b) {
      double lm = Lm[ij + (long long)oo * ((long long)hi * (hi - 1) / 2 + lo)];
      r += (a < b ? 0.5 : -0.5) * lm;
    }
    X[idx] += alpha * r;
  }
}

inline int grid_for(long long n) { return (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, 148LL * 16)); }

// Rows [pr_lo, pr_hi) of the half-transformed matrix as they sit in memory: element (pr, x) at
// p[(pr - pr_lo) + ld * (x - xoff)].  One chunk on a single GPU; one chunk per source rank after the exchange.
struct HChunk { const double* p; long long ld, pr_lo, pr_hi, xoff; };

// One half transform over the spectator range [xs0, xs1), in blocks (see file header).
//   src_mode 0: packed triangular source src[tri(x, pair)];  src_mode 1: matrix chunks (spectator = column)
//   dst_mode 0: matrix dst[(x - dst_xoff) + dst_ld * pair];  dst_mode 1: packed triangular dst[tri(x, pair)], pair <= x
void half_transform(Engine& e, int n, const double* C, const double* src, int src_mode, const std::vector<HChunk>& chunks,
                    double* dst, int dst_mode, long long dst_ld, long long dst_xoff, long long xs0, long long xs1,
                    long long max_block_bytes) {
  const long long n2 = (long long)n * n;
  const long long nspect = xs1 - xs0;
  if (nspect <= 0) return;
  long long nb = std::max<long long>(1, std::min<long long>(nspect, max_block_bytes / (3 * n2 * 8)));
  if (nb > 16) nb = nb / 16 * 16;
  Scratch X(e.pool, (size_t)(nb * n2)), Y(e.pool, (size_t)(nb * n2)), Z(e.pool, (size_t)(nb * n2));
  for (long long x0 = xs0; x0 < xs1; x0 += nb) {
    const int cb = (int)std::min<long long>(nb, xs1 - x0);
    if (src_mode == 0) {
      k_unpack_pairs<<<grid_for((long long)cb * n2), 256, 0, e.stream>>>(X.p, src, 0, 0, x0, cb, n);
      count_launch();
    } else {
      for (const HChunk& c : chunks) {
        if (c.pr_hi <= c.pr_lo) continue;
        dim3 grid((unsigned)((c.pr_hi - c.pr_lo + 31) / 32), (unsigned)((cb + 31) / 32));
        k_unpack_pairs_T<<<grid, dim3(32, 8), 0, e.stream>>>(X.p, c.p, c.ld, x0 - c.xoff, cb, n, c.pr_hi, c.pr_lo);
        count_launch();
      }
    }
    // Y(xb,k,s) = sum_l X(xb,k,l) C(s,l):  (cb*n x n) = X (cb*n x n) * C^T
    dgemm(e.stream, 'N', 'T', cb * n, n, n, 1.0, X.p, (long long)cb * n, C, n, 0.0, Y.p, (long long)cb * n);
    // Z(xb,r,s) = sum_k Y(xb,k,s) C(r,k):  for each s, (cb x n) = Y_s (cb x n) * C^T
    GemmBatch bt;
    bt.count = n; bt.strideA = (long long)cb * n; bt.strideB = 0; bt.strideC = (long long)cb * n;
    dgemm(e.stream, 'N', 'T', cb, n, n, 1.0, Y.p, cb, C, n, 0.0, Z.p, cb, &bt);
    k_pack_pairs<<<grid_for((long long)cb * n2), 256, 0, e.stream>>>(dst, Z.p, dst_mode, dst_ld, x0, cb, n, dst_xoff);
    count_launch();
    AFESP_CUDA_CHECK(cudaGetLastError());
  }
}

}  // namespace

namespace {
// eri[tri(ij,kl)] = G(ij, kl0 + c) for ij >= kl  (G block: npair x nb, ij fastest)
__global__ void k_pack_lower_block(double* __restrict__ eri, const double* __restrict__ G, long long npair, long long kl0,
                                   int nb) {
  const long long total = npair * nb;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long ij = idx % npair, kl = kl0 + idx / npair;
    if (ij >= kl) eri[ij * (ij + 1) / 2 + kl] = G[idx];
  }
}
}  // namespace

// Synthetic AO integrals on the device: eri[packed] = sum_P B(ij,P) B(kl,P), B is (npair x naux) column-major.
void synth_eri_from_factors(Engine& e, int n, int naux, const double* B, double* eri, long long block_bytes) {
  const long long npair = (long long)n * (n + 1) / 2;
  long long nb = std::max<long long>(1, std::min<long long>(npair, block_bytes / (npair * 8)));
  if (nb > 16) nb = nb / 16 * 16;
  Scratch G(e.pool, (size_t)(npair * nb));
  for (long long kl0 = 0; kl0 < npair; kl0 += nb) {
    const int cb = (int)std::min<long long>(nb, npair - kl0);
    // G(ij, c) = sum_P B(ij,P) B(kl0+c, P)
    dgemm(e.stream, 'N', 'T', (int)npair, cb, naux, 1.0, B, npair, B + kl0, npair, 0.0, G.p, npair);
    k_pack_lower_block<<<(int)std::min<long long>((npair * cb + 255) / 256, 148LL * 16), 256, 0, e.stream>>>(
        eri, G.p, npair, kl0, cb);
    count_launch();
  }
  AFESP_CUDA_CHECK(cudaGetLastError());
}

long long npair_of(int n) { return (long long)n * (n + 1) / 2; }
long long npacked_of(int n) { long long m = npair_of(n); return m * (m + 1) / 2; }

void ao2mo_packed(Engine& e, int n, const double* eri_ao, const double* C, double* eri_mo, long long block_bytes) {
  const long long npair = npair_of(n);
  Dist& d = e.dist;
  if (!d.active() || npair < 64LL * d.nranks) {
    Scratch H(e.pool, (size_t)(npair * npair));
    // phase 1: spectator = kl (AO pair), transform (ij) -> (pq): H(kl, pq), kl fastest
    half_transform(e, n, C, eri_ao, 0, {}, H.p, 0, npair, 0, 0, npair, block_bytes);
    // phase 2: spectator = pq (MO pair = column of H), transform (kl) -> (rs): eri_mo[tri(pq, rs)], rs <= pq
    half_transform(e, n, C, nullptr, 1, {HChunk{H.p, npair, 0, npair, 0}}, eri_mo, 1, 0, 0, 0, npair, block_bytes);
    return;
  }
  // ---- several GPUs: phase 1 over this rank's kl spectators, all-to-all of the half-transformed blocks, phase 2 over
  //      this rank's pq spectators, then every rank broadcasts its rows of the packed result (SURVEY.md §8e).
  const int R = d.nranks, me = d.rank;
  std::vector<long long> lo(R), hi(R);
  for (int r = 0; r < R; ++r) d.col_range(npair, r, &lo[r], &hi[r], 16);
  const long long mine = hi[me] - lo[me];
  Scratch Hloc(e.pool, (size_t)std::max<long long>(mine * npair, 1));   // H(kl in mine, all pq), ld = mine
  half_transform(e, n, C, eri_ao, 0, {}, Hloc.p, 0, mine, lo[me], lo[me], hi[me], block_bytes);
  Scratch Rcv(e.pool, (size_t)std::max<long long>(npair * mine, 1));    // chunk g: (hi[g]-lo[g]) x mine, kl fastest
  std::vector<HChunk> chunks;
  AFESP_REQUIRE(d.group_start() == 0, "ncclGroupStart failed");
  for (int g = 0; g < R; ++g) {
    const long long rows_g = hi[g] - lo[g];
    double* slot = Rcv.p + lo[g] * mine;
    chunks.push_back(HChunk{slot, rows_g, lo[g], hi[g], lo[me]});
    if (g == me) {
      if (mine > 0)
        AFESP_CUDA_CHECK(cudaMemcpyAsync(slot, Hloc.p + mine * lo[me], (size_t)(mine * mine) * 8,
                                         cudaMemcpyDeviceToDevice, e.stream));
      continue;
    }
    if (mine > 0 && rows_g > 0) {
      // my rows of the columns rank g owns: contiguous (mine x rows_g) block of Hloc
      AFESP_REQUIRE(d.send(Hloc.p + mine * lo[g], (size_t)(mine * rows_g), g, d.comm, e.stream) == 0, "ncclSend failed");
      AFESP_REQUIRE(d.recv(slot, (size_t)(rows_g * mine), g, d.comm, e.stream) == 0, "ncclRecv failed");
      d.exchanged_bytes += 8.0 * rows_g * mine;
    }
  }
  AFESP_REQUIRE(d.group_end() == 0, "ncclGroupEnd failed");
  half_transform(e, n, C, nullptr, 1, chunks, eri_mo, 1, 0, 0, lo[me], hi[me], block_bytes);
  std::vector<std::pair<long long, long long>> ranges(R);
  for (int r = 0; r < R; ++r) ranges[r] = {lo[r] * (lo[r] + 1) / 2, hi[r] * (hi[r] + 1) / 2};
  d.exchange(eri_mo, ranges, e.stream);
}

void mp2_energy(Engine& e, int n, int nocc, int nfrozen, const double* eri_mo, const double* eps, double* out_dev) {
  const long long total = (long long)(nocc - nfrozen) * (nocc - nfrozen) * (n - nocc) * (n - nocc);
  int nb = std::min(grid_for(total), 1024);
  double* part = reduce_scratch(e, nb);
  k_mp2<<<nb, 256, 0, e.stream>>>(eri_mo, eps, n, nocc, nfrozen, part);
  count_launch();
  finish_partials(e, part, nb, 1, out_dev);
}

void spinorb_symmetry_error(Engine& e, int n, int lo, const double* eri_mo, double* out_dev) {
  const int n2 = 2 * n - lo;
  const long long total = (long long)n2 * n2 * n2 * n2;
  const int nb = std::min(grid_for(total), 148 * 8);
  double* part = reduce_scratch(e, nb);
  k_spinorb_symmetry<<<nb, 256, 0, e.stream>>>(eri_mo, lo, n2, part);
  count_launch();
  AFESP_CUDA_CHECK(cudaGetLastError());
  finish_partials(e, part, nb, 1, out_dev);
}

void build_vpm(Engine& e, double* V, const double* eri_mo, int voff, int v, int sign, long long col0, long long ncols) {
  const long long P = sign > 0 ? (long long)v * (v + 1) / 2 : (long long)v * (v - 1) / 2;
  if (ncols < 0) ncols = P - col0;
  if (P == 0 || ncols <= 0) return;
  k_build_vpm<<<grid_for(P * ncols), 256, 0, e.stream>>>(V, eri_mo, voff, v, sign, col0, ncols);
  count_launch();
}

void pack_c(Engine& e, double* S, double* A, const double* c, int oo, int v) {
  k_pack_c<<<grid_for((long long)oo * v * v), 256, 0, e.stream>>>(S, A, c, oo, v);
  count_launch();
}

void unpack_ladder(Engine& e, double* X, const double* Lp, const double* Lm, int oo, int v, double alpha) {
  k_unpack_ladder<<<grid_for((long long)oo * v * v), 256, 0, e.stream>>>(X, Lp, Lm, oo, v, alpha);
  count_launch();
}

void slice_phys(Engine& e, double* out, const double* eri_mo, const int lo[4], const int cnt[4]) {
  SliceSpec sp;
  long long total = 1;
  for (int d = 0; d < 4; ++d) { sp.lo[d] = lo[d]; sp.n[d] = cnt[d]; total *= cnt[d]; }
  if (total == 0) return;
  k_slice_phys<<<grid_for(total), 256, 0, e.stream>>>(out, eri_mo, sp);
  count_launch();
}

void slice_spinorb(Engine& e, double* out, const double* eri_mo, const int lo[4], const int cnt[4]) {
  SliceSpec sp;
  long long total = 1;
  for (int d = 0; d < 4; ++d) { sp.lo[d] = lo[d]; sp.n[d] = cnt[d]; total *= cnt[d]; }
  if (total == 0) return;
  k_slice_spinorb<<<grid_for(total), 256, 0, e.stream>>>(out, eri_mo, sp);
  count_launch();
}

}  // namespace afesp
