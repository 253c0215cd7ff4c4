// Perturbative triples on the device: [T], (T), renormalised and completely renormalised variants (spin-free,
// src/ccsd.f90:2018-2336) and the spin-orbital (T) (src/ccsd.f90:1812-1922).
//
// The reference evaluates, for every ordered (i,j,k) and every (a,b,c), 12 (24 for CR) strided dot products
// (:2168-2173, :2188-2193).  Here each (i,j,k) block is built from FP64 DMMA GEMMs:
//     X_pqr(a,(b,c)) = sum_d t2(p,q,a,d) v_vovv(d,r,b,c)            [v x v^2 x v]
//                    - sum_l t2(l,p,b,a) v_ovoo(l,c,q,r)            [v^2 x v x o]   (accumulated into the same block)
//     W_ijk(a,b,c)   = sum over the six simultaneous permutations of X               (tiled combine kernel)
// batched over as many triples as fit the work buffer, followed by one fused epilogue kernel that forms the
// energy denominators, z3, y, the x-bar combinations and all six reductions in a single pass over W (and M3).
// Two permutations that share their first virtual label differ only by a swap of the other two, so with a second copy
// of the (n x v^2) operand stored (z,y)-transposed they are K-concatenated into ONE product of depth 2 nbf:
//     Y_s(x,(u,w)) = X_s(x,u,w) + X_{s+3}(x,w,u),  s = abc, bac, cba
// -- three GEMM outputs per triple instead of six, written once and read once by the epilogue.
//
// Occupied-triple symmetry: W, z3, y and M3 are covariant under simultaneous permutation of (i,a),(j,b),(k,c), so the
// sum over the orbit of an ordered triple equals  mult * sum_abc x~(abc) u(abc)  with the symmetrised
//     x~ = [8 x(abc) - 4 (x(acb) + x(cba) + x(bac)) + 2 (x(bca) + x(cab))] / 6
// (the group average of make_x_bar, :2314-2318; the same combination the GAMESS comment at :2320-2331 lists).  Only
// i <= j <= k is computed, weighted by mult = 6, 3 or 1.  Work is dealt round-robin over (rank, nranks): the unit of
// multi-GPU sharding (SURVEY.md §8e); the caller sums the six partial results across ranks.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>

#include "ccsd.cuh"

namespace afesp {
namespace {

constexpr int TS = 8;               // label tile edge
constexpr int TP = TS + 1;          // padded edge (bank spread)
constexpr int BOX = TS * TP * TP;   // doubles per staged box

__constant__ int c_perm[6][3] = {{0, 1, 2}, {1, 0, 2}, {2, 1, 0}, {0, 2, 1}, {1, 2, 0}, {2, 0, 1}};
__constant__ double c_coef[6] = {8.0 / 6.0, -4.0 / 6.0, -4.0 / 6.0, -4.0 / 6.0, 2.0 / 6.0, 2.0 / 6.0};

// One occupied triple of a (T) launch.  slot[s] = block of the batch buffer holding Y_s (s = abc, bac, cba).  Coincident
// occupied indices make blocks redundant (spin-free driver): i == j gives Y_bac = Y_abc (slot[1] = slot[0]); j == k
// gives Y_cba(x,u,w) = Y_bac(x,w,u) (flag bit 1: the epilogue takes the cba values from the bac gather, no block at all).
struct TripleDesc { int i, j, k, flags; double weight; int slot[3]; int pad; };
constexpr int kCbaFromBac = 2;

__device__ __forceinline__ int box_off(int x, int y, int z) { return (z * TP + y) * TP + x; }

// Compile-time permutation algebra (everything below constant-folds once the q/t/s loops are unrolled).
// perm t -> (p0,p1,p2) in the order of c_perm: abc, bac, cba, acb, bca, cab
__host__ __device__ constexpr int PM(int t, int m) {
  return t == 0 ? (m == 0 ? 0 : (m == 1 ? 1 : 2))
       : t == 1 ? (m == 0 ? 1 : (m == 1 ? 0 : 2))
       : t == 2 ? (m == 0 ? 2 : (m == 1 ? 1 : 0))
       : t == 3 ? (m == 0 ? 0 : (m == 1 ? 2 : 1))
       : t == 4 ? (m == 0 ? 1 : (m == 1 ? 2 : 0))
                : (m == 0 ? 2 : (m == 1 ? 0 : 1));
}
__host__ __device__ constexpr int perm_index(int r0, int r1, int r2) {
  return (r0 == 0 && r1 == 1) ? 0 : (r0 == 1 && r1 == 0) ? 1 : (r0 == 2 && r1 == 1) ? 2
       : (r0 == 0 && r1 == 2) ? 3 : (r0 == 1 && r1 == 2) ? 4 : 5;
}
// index of q o s, (q o s)[m] = q[s[m]]
__host__ __device__ constexpr int COMP(int q, int s) {
  return perm_index(PM(q, PM(s, 0)), PM(q, PM(s, 1)), PM(q, PM(s, 2)));
}
__host__ __device__ constexpr double COEF(int s) { return s == 0 ? 8.0 / 6.0 : (s <= 3 ? -4.0 / 6.0 : 2.0 / 6.0); }

struct FusedArgs {
  const double* X;    // [blocks][v^3]  pair-merged GEMM blocks Y_s (s = abc, bac, cba) for the W term, addressed through
                      //                TripleDesc::slot
  const double* XM;   // [blocks][v^3]  same for the M3 term (CR) or null
  const double* t1;   // (o,v)
  const double* t2;   // (o,o,v,v)
  const double* vo;   // v_oovv (o,o,v,v)
  const double* eo;
  const double* ev;
  const TripleDesc* tr;
  const int* tiles;   // [ntt][3] unordered label-tile triples A <= B <= C
  int o, v;
  double* partials;   // [gridDim.y * gridDim.x][6]
};

// ---- fused epilogue, "orbit form" -----------------------------------------------------------------------------------
// One CTA = one unordered triple of label tiles {A,B,C} (8 labels each) of one occupied triple (i,j,k); one THREAD = one
// label triple (a,b,c) = (A+tx, B+ty, C+tz) together with its six permutations P_u(a,b,c), u = abc, bac, cba, acb, bca,
// cab -- the "orbit".  Everything the reference evaluates per (a,b,c) couples only members of one orbit:
//   W(P_u abc)   = sum_s Y_s[P_{u o s} abc]                         (src/ccsd.f90:2168-2173; two of its six terms per Y_s)
//   x~(W)(P_u)   = sum_s c_s W(P_{u o s} abc)                       (make_x_bar, :2314-2318, group-averaged, see header)
//   D3 = e_i + e_j + e_k - e_a - e_b - e_c  is the SAME for all six members
// so after the gather below the six W (and M3, z3, y) values of the orbit sit in the thread's registers and the energy
// expressions (:2175-2233) need no further shared-memory traffic, one reciprocal, and no per-tile bookkeeping.
//
// Gather: V[s][w] = Y_s at tile origin (O o w), local position (l o w).  Each of the 18 boxes is read from global memory
// at the thread's NATURAL position (coalesced 64-byte rows, all 18 loads in flight), the 15 boxes with w != identity go
// through shared memory once: written at l, read back at l o w.  Each box is only ever read with its own permutation w,
// so it gets its own XOR-swizzled layout in which both the natural write and the permuted read of a half-warp
// (tx = 0..7, two consecutive ty) touch 16 distinct 8-byte banks (enumerated in tests/test_tma_layout.py).
constexpr int BOXW = TS * TS * TS;   // words per swizzled box (no padding)

__device__ __forceinline__ int swz(int w, int X, int Y, int Z) {   // w is a compile-time constant after unrolling
  switch (w) {
    case 1: return 64 * Z + 8 * Y + (X ^ Y);
    case 2: return 64 * Z + 8 * Y + (X ^ Z);
    case 3: return 64 * Z + 8 * (Y ^ (Z & 1)) + X;
    case 4: return 64 * Z + 8 * (Y ^ (X & 1)) + (X ^ Z);
    default: return 64 * Z + 8 * (Y ^ (Z & 1)) + (X ^ Y);
  }
}

template <bool USE_Z, bool DO_Y, bool DO_M>
constexpr size_t fused_smem_doubles() {
  return (size_t)15 * BOXW + ((USE_Z || DO_Y) ? (54 * TS * TS + 9 * TS) : 0);
}

template <bool USE_Z, bool DO_Y, bool DO_M, bool PAREN>
__global__ void __launch_bounds__(TS* TS* TS, 2) k_triples_fused(const FusedArgs g) {
  extern __shared__ double sm[];
  constexpr bool AUX = USE_Z || DO_Y;
  double* sS = sm;                                  // [3 s][5 w][BOXW] staged Y boxes with w != identity
  double* sV = sm + 15 * BOXW;                      // [3 pairs][3][3][TS*TS]  v_oovv(pair; R1, R2)
  double* sT = sV + (AUX ? 27 * TS * TS : 0);       // [3 occ][3 ranges][TS]    t1(occ; R)
  double* sY = sT + (AUX ? 9 * TS : 0);             // [3 pairs][3][3][TS*TS]  t2(pair; R1, R2)
  __shared__ double red[6][TS * TS * TS / 32];
  const int tx = threadIdx.x, ty = threadIdx.y, tz = threadIdx.z;
  const int tid = tx + TS * (ty + TS * tz);
  const int o = g.o, v = g.v;
  const TripleDesc td = g.tr[blockIdx.y];
  const int occ[3] = {td.i, td.j, td.k};
  const int T3[3] = {g.tiles[3 * blockIdx.x], g.tiles[3 * blockIdx.x + 1], g.tiles[3 * blockIdx.x + 2]};
  const int O[3] = {T3[0] * TS, T3[1] * TS, T3[2] * TS};
  const long long v3 = (long long)v * v * v, oo = (long long)o * o;
  const int l[3] = {tx, ty, tz};
  const bool full = (O[2] + TS <= v);               // tiles are ordered A <= B <= C: no edge tile involved
  const long long thr_off = tx + (long long)v * (ty + (long long)v * tz);
  // global offset of each box origin O o w and whether the thread's element of that box exists
  long long gorg[6];
  bool okb[6];
#pragma unroll
  for (int w = 0; w < 6; ++w) {
    gorg[w] = O[PM(w, 0)] + (long long)v * (O[PM(w, 1)] + (long long)v * O[PM(w, 2)]) + thr_off;
    okb[w] = full || ((O[PM(w, 0)] + tx < v) && (O[PM(w, 1)] + ty < v) && (O[PM(w, 2)] + tz < v));
  }
  int wr[6], rd[6];
#pragma unroll
  for (int w = 1; w < 6; ++w) {
    wr[w] = swz(w, tx, ty, tz);
    rd[w] = swz(w, l[PM(w, 0)], l[PM(w, 1)], l[PM(w, 2)]);
  }

  // out[u] = sum_s Y_s[P_{u o s}(a,b,c)], u = 0..5 (s = abc, bac, cba are involutions: V[s][w] lands in u = w o s).
  // Blocks that coincide for i == j (Y_bac = Y_abc: same slot, the L2 serves the second read) are simply read again;
  // for j == k (flag kCbaFromBac) Y_cba(x,u,w) = Y_bac(x,w,u), i.e. V[cba][w] = V[bac][w o acb]: no loads, no staging.
  const bool cba_from_bac = (td.flags & kCbaFromBac) != 0;   // CTA-uniform
  const int ns = cba_from_bac ? 2 : 3;
  auto gather = [&](const double* __restrict__ Ybase, double (&out)[6]) {
    double val[18];
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      if (s < ns) {
        const double* __restrict__ Yb = Ybase + (long long)td.slot[s] * v3;
#pragma unroll
        for (int w = 0; w < 6; ++w) val[s * 6 + w] = okb[w] ? __ldg(Yb + gorg[w]) : 0.0;
      }
    }
#pragma unroll
    for (int u = 0; u < 6; ++u) out[u] = 0.0;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      if (s < ns) {
        out[COMP(0, s)] += val[s * 6];
#pragma unroll
        for (int w = 1; w < 6; ++w) sS[(s * 5 + w - 1) * BOXW + wr[w]] = val[s * 6 + w];
      }
    }
    __syncthreads();
    double v1[6];   // the bac gather, kept for the j == k case
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      if (s < ns) {
#pragma unroll
        for (int w = 1; w < 6; ++w) {
          const double x = sS[(s * 5 + w - 1) * BOXW + rd[w]];
          out[COMP(w, s)] += x;
          if (s == 1) v1[w] = x;
        }
        if (s == 1) v1[0] = val[6];
      }
    }
    if (cba_from_bac) {
#pragma unroll
      for (int w = 0; w < 6; ++w) out[COMP(w, 2)] += v1[COMP(w, 3)];
    }
  };

  if (AUX) {
    for (int e = tid; e < 27 * TS * TS; e += TS * TS * TS) {
      int xy = e % (TS * TS), rr = (e / (TS * TS)) % 9, pr = e / (9 * TS * TS);
      int x = O[rr / 3] + xy % TS, y = O[rr % 3] + xy / TS;
      int p = pr == 0 ? occ[1] : occ[0], q = pr == 2 ? occ[1] : occ[2];  // pairs (j,k), (i,k), (i,j)
      bool ok = x < v && y < v;
      long long off = p + (long long)o * q + oo * (x + (long long)v * y);
      if (USE_Z) sV[e] = ok ? g.vo[off] : 0.0;
      if (DO_Y) sY[e] = ok ? g.t2[off] : 0.0;
    }
    for (int e = tid; e < 9 * TS; e += TS * TS * TS) {
      int x = O[(e / TS) % 3] + e % TS;
      sT[e] = x < v ? g.t1[occ[e / (3 * TS)] + (long long)o * x] : 0.0;
    }
  }
  double W[6], M[6];
  gather(g.X, W);
  if (DO_M) {
    __syncthreads();                                  // the staging boxes are reused
    gather(g.XM, M);
  }
  // energies of the orbit (:2175-2233)
  double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  const bool inside = full || ((O[0] + tx < v) && (O[1] + ty < v) && (O[2] + tz < v));
  if (inside) {
    const double D3 = g.eo[td.i] + g.eo[td.j] + g.eo[td.k] - g.ev[O[0] + tx] - g.ev[O[1] + ty] - g.ev[O[2] + tz];
    const double rD = 1.0 / D3;
    double z3[6], yv[6];
    if (USE_Z || DO_Y) {
#pragma unroll
      for (int w = 0; w < 6; ++w) {
        // labels (a',b',c') = P_w(a,b,c): component m lies in range w[m] with local index l[w[m]]
        const int w0 = PM(w, 0), w1 = PM(w, 1), w2 = PM(w, 2);
        const double ta = sT[(0 * 3 + w0) * TS + l[w0]], tb = sT[(1 * 3 + w1) * TS + l[w1]], tc = sT[(2 * 3 + w2) * TS + l[w2]];
        const int ibc = ((0 * 3 + w1) * 3 + w2) * TS * TS + l[w1] + TS * l[w2];
        const int iac = ((1 * 3 + w0) * 3 + w2) * TS * TS + l[w0] + TS * l[w2];
        const int iab = ((2 * 3 + w0) * 3 + w1) * TS * TS + l[w0] + TS * l[w1];
        if (USE_Z) z3[w] = ta * sV[ibc] + tb * sV[iac] + tc * sV[iab];                          // (:2178-2179), times rD below
        if (DO_Y) yv[w] = ta * tb * tc + ta * sY[ibc] + tb * sY[iac] + tc * sY[iab];            // (:2183-2184)
      }
    }
#pragma unroll
    for (int u = 0; u < 6; ++u) {
      double tt = 0.0, zt = 0.0;
#pragma unroll
      for (int s = 0; s < 6; ++s) {
        tt += COEF(s) * W[COMP(u, s)];
        if (USE_Z) zt += COEF(s) * z3[COMP(u, s)];
      }
      tt *= rD;
      zt *= rD;
      acc[0] += tt * W[u];
      if (PAREN) acc[1] += (tt + zt) * W[u];
      if (DO_Y) {
        acc[2] += tt * yv[u];
        if (PAREN) acc[3] += (tt + zt) * yv[u];
      }
      if (DO_M) {
        acc[4] += tt * M[u];
        if (PAREN) acc[5] += (tt + zt) * M[u];
      }
    }
  }
  // ordered tiles that coincide (A == B etc.) are visited more than once: weight each visit accordingly
  const double dup = (T3[0] == T3[1] && T3[1] == T3[2]) ? 1.0 / 6.0 : ((T3[0] == T3[1] || T3[1] == T3[2]) ? 0.5 : 1.0);
  const int lane = tid & 31, warp = tid >> 5;
  const double wgt = td.weight * dup;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const bool live = (k == 0) || (k == 1 && PAREN) || (k == 2 && DO_Y) || (k == 3 && DO_Y && PAREN) ||
                      (k == 4 && DO_M) || (k == 5 && DO_M && PAREN);
    if (!live) continue;
    double x = acc[k] * wgt;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_down_sync(0xffffffffu, x, off);
    if (lane == 0) red[k][warp] = x;
  }
  __syncthreads();
  if (tid < 6) {
    const int k = tid;
    const bool live = (k == 0) || (k == 1 && PAREN) || (k == 2 && DO_Y) || (k == 3 && DO_Y && PAREN) ||
                      (k == 4 && DO_M) || (k == 5 && DO_M && PAREN);
    double sacc = 0.0;
    if (live)
      for (int w2 = 0; w2 < TS * TS * TS / 32; ++w2) sacc += red[k][w2];
    g.partials[((long long)blockIdx.y * gridDim.x + blockIdx.x) * 6 + k] = sacc;
  }
}

// Spin-orbital epilogue (src/ccsd.f90:1873-1910): t3c = X - X(bac) - X(cba), same for the disconnected part,
// e_T += t3c (t3c / D + t3d) / 36, times the orbit weight.
struct EnergySoArgs {
  const double* X;   // [nb][v^3] connected block before P(a/bc)
  const double* t1;
  const double* vo;  // oovv (o,o,v,v)
  const double* eo;
  const double* ev;
  const TripleDesc* tr;
  int o, v, ntile;
  double* partials;  // [blocks][1]
};

__global__ void __launch_bounds__(TS* TS* TS) k_energy_spinorb_t(const EnergySoArgs g) {
  __shared__ double sX[3 * BOX];
  __shared__ double sV[27 * TS * TS];
  __shared__ double sT[9 * TS];
  __shared__ double red[TS * TS * TS / 32];
  const int tx = threadIdx.x, ty = threadIdx.y, tz = threadIdx.z;
  const int tid = tx + TS * (ty + TS * tz);
  const int o = g.o, v = g.v, ntile = g.ntile;
  const TripleDesc td = g.tr[blockIdx.y];
  const int occ[3] = {td.i, td.j, td.k};
  int tile = blockIdx.x;
  const int O[3] = {(tile % ntile) * TS, ((tile / ntile) % ntile) * TS, (tile / (ntile * ntile)) * TS};
  const long long v3 = (long long)v * v * v, oo = (long long)o * o;
  const double* Xb = g.X + (long long)blockIdx.y * v3;
  const int P3[3][3] = {{0, 1, 2}, {1, 0, 2}, {2, 1, 0}};  // abc, bac, cba
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    int x = O[P3[t][0]] + tx, y = O[P3[t][1]] + ty, z = O[P3[t][2]] + tz;
    double val = 0.0;
    if (x < v && y < v && z < v) val = Xb[x + (long long)v * (y + (long long)v * z)];
    sX[t * BOX + box_off(tx, ty, tz)] = val;
  }
  // oovv(p,q; x in R1, y in R2) for occupied pairs (j,k), (i,k), (j,i)                      (:1877-1878)
  for (int e = tid; e < 27 * TS * TS; e += TS * TS * TS) {
    int xy = e % (TS * TS), rr = (e / (TS * TS)) % 9, pr = e / (9 * TS * TS);
    int r1 = rr / 3, r2 = rr % 3;
    int x = O[r1] + xy % TS, y = O[r2] + xy / TS;
    int p = pr == 1 ? occ[0] : occ[1], q = pr == 2 ? occ[0] : occ[2];
    sV[e] = (x < v && y < v) ? g.vo[p + (long long)o * q + oo * (x + (long long)v * y)] : 0.0;
  }
  for (int e = tid; e < 9 * TS; e += TS * TS * TS) {
    int x = O[(e / TS) % 3] + e % TS;
    sT[e] = x < v ? g.t1[occ[e / (3 * TS)] + (long long)o * x] : 0.0;
  }
  __syncthreads();
  double acc = 0.0;
  const int l[3] = {tx, ty, tz};
  const int a = O[0] + tx, b = O[1] + ty, c = O[2] + tz;
  if (a < v && b < v && c < v) {
    const double D3 = g.eo[td.i] + g.eo[td.j] + g.eo[td.k] - g.ev[a] - g.ev[b] - g.ev[c];
    double t3c = 0.0, t3d = 0.0;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const int q0 = P3[t][0], q1 = P3[t][1], q2 = P3[t][2];
      const double sgn = t == 0 ? 1.0 : -1.0;
      t3c += sgn * sX[t * BOX + box_off(l[q0], l[q1], l[q2])];
      // disconnected part at labels (a',b',c'): t1(i,a') oovv(j,k,b',c') - t1(j,a') oovv(i,k,b',c') - t1(k,a') oovv(j,i,b',c')
      const int bc = l[q1] + TS * l[q2];
      double d = sT[(0 * 3 + q0) * TS + l[q0]] * sV[((0 * 3 + q1) * 3 + q2) * TS * TS + bc] -
                 sT[(1 * 3 + q0) * TS + l[q0]] * sV[((1 * 3 + q1) * 3 + q2) * TS * TS + bc] -
                 sT[(2 * 3 + q0) * TS + l[q0]] * sV[((2 * 3 + q1) * 3 + q2) * TS * TS + bc];
      t3d += sgn * d;
    }
    acc = t3c * (t3c / D3 + t3d / D3) / 36.0 * td.weight;
  }
  const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (tid == 0) {
    double sacc = 0.0;
    for (int w2 = 0; w2 < TS * TS * TS / 32; ++w2) sacc += red[w2];
    g.partials[(long long)blockIdx.y * gridDim.x + blockIdx.x] = sacc;
  }
}

struct DevPtrs {  // device pointer arrays for the batched GEMMs of one batch
  DBuf raw;       // reinterpret as const double*[]
  size_t cap = 0;
  void ensure(size_t nptr) {
    if (cap < nptr) { raw.alloc(nptr); cap = nptr; }  // sizeof(double) == sizeof(pointer)
  }
};

std::vector<TripleDesc> my_triples(int o, bool symmetric, bool strict, int rank, int nranks) {
  // symmetric: unique i<=j<=k with orbit multiplicity; strict: i<j<k only (spin-orbital, others vanish)
  std::vector<TripleDesc> all;
  if (symmetric) {
    for (int i = 0; i < o; ++i)
      for (int j = i; j < o; ++j)
        for (int k = j; k < o; ++k) {
          if (strict && (i == j || j == k)) continue;
          double w = (i == j && j == k) ? 1.0 : ((i == j || j == k) ? 3.0 : 6.0);
          all.push_back({i, j, k, 0, w, {0, 0, 0}, 0});
        }
  } else {
    for (int i = 0; i < o; ++i)
      for (int j = 0; j < o; ++j)
        for (int k = 0; k < o; ++k) all.push_back({i, j, k, 0, 1.0, {0, 0, 0}, 0});
  }
  std::vector<TripleDesc> mine;
  for (size_t t = 0; t < all.size(); ++t)
    if ((int)(t % (size_t)nranks) == rank) mine.push_back(all[t]);
  return mine;
}

static_assert(sizeof(double) == sizeof(void*), "pointer arrays are carried in double buffers");


}  // namespace

namespace {
// Developer check (AFESP_T_VERIFY=1): count elements of two X buffers that differ by more than rounding.
__global__ void k_count_mismatch(const double* __restrict__ a, const double* __restrict__ b, long long n, double tol,
                                 unsigned long long* __restrict__ out) {
  unsigned long long bad = 0;
  double worst = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double d = fabs(a[i] - b[i]);
    if (d > tol * fmax(fabs(b[i]), 1e-6)) { ++bad; worst = fmax(worst, d); }
  }
  if (bad) { atomicAdd(out, bad); atomicMax(out + 1, (unsigned long long)__double_as_longlong(worst)); }
}
}  // namespace

void triples_partition_counts(int o, bool symmetric, bool strict, int nranks, long long* counts) {
  for (int r = 0; r < nranks; ++r) counts[r] = (long long)my_triples(o, symmetric, strict, r, nranks).size();
}

double triples_denominator_constant(CCState& s) {
  // 1 + 2 sum t1^2 + sum asym_t2 * c  (src/ccsd.f90:2243), from the converged amplitudes (:2073-2105)
  Engine& e = s.eng;
  const int o = s.o, v = s.v;
  Scratch a(e.pool, (size_t)s.t2.size()), c(e.pool, (size_t)s.t2.size());
  TView A(a.p, s.t2.dims);
  transpose(e, "ijab->jiab", -1.0, s.t2.view(), 0.0, A);
  axpby(e.stream, s.t2.size(), 2.0, s.t2.p(), 1.0, a.p);
  t2_plus_t1t1(e.stream, c.p, s.t2.p(), s.t1.p(), o, v, 1.0, 0.0);
  if (s.red_out.n < 16) s.red_out.alloc(16);
  const double* pa[1] = {a.p};
  dotn(e, s.t2.size(), 1, pa, c.p, s.red_out.p);
  double h = 0.0;
  AFESP_CUDA_CHECK(cudaMemcpyAsync(&h, s.red_out.p, 8, cudaMemcpyDeviceToHost, e.stream));
  AFESP_CUDA_CHECK(cudaStreamSynchronize(e.stream));
  return 1.0 + 2.0 * cc_t1_norm2(s) + h;
}

void triples_spatial(CCState& s, bool paren, bool renorm, bool comp_renorm, int rank, int nranks, double sums[6]) {
  AFESP_REQUIRE(s.restricted, "triples_spatial needs a spin-free CCSD state");
  AFESP_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "triples: bad (rank, nranks)");
  Engine& e = s.eng;
  cudaStream_t st = e.stream;
  const int o = s.o, v = s.v;
  const long long v2 = (long long)v * v, v3 = v2 * v;
  const bool do_y = renorm || comp_renorm, do_m = comp_renorm;
  const bool use_z = paren && do_y;  // Q2: z3_bar is only formed for (T) *and* (R or CR)  (src/ccsd.f90:2211-2215)
  if (do_m) AFESP_REQUIRE(s.has("I_vovv_pp") && s.has("I_ooov_pp"), "CR triples need the CR intermediates");
  for (int k = 0; k < 6; ++k) sums[k] = 0.0;

  Trace tr(st);
  // K-concatenated GEMM operands (work arrays come from the engine's pool: cudaFree of GB-sized blocks is slow).
  // With the hole term written in the layout (c,b,a) it lands in the buffer of the permutation (r,q,p) as
  //     C_pqr(x,(y,z)) = sum_d t2(p,q,x,d) v_vovv(d,r,y,z) - sum_l v_ovoo(l,x,q,p) t2(l,r,y,z)
  // i.e. ONE product of depth K = v + o (= nbf without frozen core) per permutation:
  //     Acat(x, [d | l]; p,q) = [ t2(p,q,x,d) | -v_oovo(p,q,x,l) ]            (v x n) for each occupied pair
  //     Bcat([d | l], (y,z); r) = [ v_vvov(z,y,r,d) ; t2(l,r,y,z) ]           (n x v^2) for each occupied index
  //     BcatT(k, (y,z); r)      = Bcat(k, (z,y); r)
  // (the reference's reshapes at :2056-2066, re-aimed at GEMM blocks).  M3 uses I_ooov_pp / I_vovv_pp instead (:2188-2193).
  // The two permutations with the same first label are then one dual-segment GEMM (see the file header):
  //     Y_s(x,(u,w); i,j,k) = Acat(x,.; P0,P1) Bcat(.,(u,w); P2) + Acat(x,.; P0,P2) BcatT(.,(u,w); P1),  (P0,P1,P2) = p_s(i,j,k)
  // K = v + o is also the leading dimension of Bcat and the block stride of both operands.  With v even and o odd (e.g. an
  // odd number of frozen core orbitals) one zero column of Acat and one zero row of Bcat / BcatT make K even, so the
  // batches keep the 16-byte-aligned (TMA) kernel; the zero terms change only the grouping of the last k-tile.
  const int n = v + o + ((v % 2 == 0 && o % 2 == 1) ? 1 : 0);
  const size_t n_acat = (size_t)v * n * o * o, n_bcat = (size_t)n * v2 * o;
  Scratch sAcat(e.pool, n_acat + 16), sBcat(e.pool, n_bcat + 16), sBcatT(e.pool, n_bcat + 16);  // +16: TMA boxes over-read the last 16-row chunk
  std::unique_ptr<Scratch> sAcatM, sBcatM, sBcatMT;
  auto put = [&](const TView& in, const char* from, const char* to, double alpha, double* out, const long long* ostr) {
    int rank = (int)std::strlen(from), perm[4], dims[4];
    for (int d = 0; d < rank; ++d) {
      perm[d] = (int)(std::strchr(from, to[d]) - from);
      dims[d] = in.dims[d];
    }
    permute_strided(st, rank, dims, perm, alpha, in.p, 0.0, out, ostr);
  };
  const long long a_str[4] = {1, v, (long long)v * n, (long long)v * n * o};          // (x, k, p, q)
  const long long b_str[4] = {1, n, (long long)n * v, (long long)n * v2};             // (k, y, z, r)
  put(s.t2.view(), "pqxd", "xdpq", 1.0, sAcat.p, a_str);
  put(s.get("v_oovo").view(), "pqxl", "xlpq", -1.0, sAcat.p + (size_t)v * v, a_str);
  put(s.get("v_vvov").view(), "zyrd", "dyzr", 1.0, sBcat.p, b_str);
  put(s.t2.view(), "lryz", "lyzr", 1.0, sBcat.p + v, b_str);
  put(s.get("v_vvov").view(), "yzrd", "dyzr", 1.0, sBcatT.p, b_str);
  put(s.t2.view(), "lrzy", "lyzr", 1.0, sBcatT.p + v, b_str);
  auto zero_pad = [&](double* Acat, double* Bcat, double* BcatT) {   // pool scratch is not zeroed
    if (n == v + o) return;
    AFESP_CUDA_CHECK(cudaMemset2DAsync(Acat + (size_t)v * (v + o), (size_t)v * n * 8, 0, (size_t)v * 8, (size_t)o * o, st));
    AFESP_CUDA_CHECK(cudaMemset2DAsync(Bcat + (v + o), (size_t)n * 8, 0, 8, (size_t)v2 * o, st));
    AFESP_CUDA_CHECK(cudaMemset2DAsync(BcatT + (v + o), (size_t)n * 8, 0, 8, (size_t)v2 * o, st));
  };
  zero_pad(sAcat.p, sBcat.p, sBcatT.p);
  if (do_m) {
    sAcatM.reset(new Scratch(e.pool, n_acat + 16)); sBcatM.reset(new Scratch(e.pool, n_bcat + 16));
    sBcatMT.reset(new Scratch(e.pool, n_bcat + 16));
    put(s.t2.view(), "pqxd", "xdpq", 1.0, sAcatM->p, a_str);
    put(s.get("I_ooov_pp").view(), "qplx", "xlpq", -1.0, sAcatM->p + (size_t)v * v, a_str);
    put(s.get("I_vovv_pp").view(), "dryz", "dyzr", 1.0, sBcatM->p, b_str);
    put(s.t2.view(), "lryz", "lyzr", 1.0, sBcatM->p + v, b_str);
    put(s.get("I_vovv_pp").view(), "drzy", "dyzr", 1.0, sBcatMT->p, b_str);
    put(s.t2.view(), "lrzy", "lyzr", 1.0, sBcatMT->p + v, b_str);
    zero_pad(sAcatM->p, sBcatM->p, sBcatMT->p);
  }

  std::vector<TripleDesc> tri = my_triples(o, s.opt.triples_ijk_symmetry, false, rank, nranks);
  if (tri.empty()) return;
  tr.lap(0);
  // GEMM blocks per triple: 3, or fewer when occupied indices coincide (see TripleDesc): i == j -> {abc, cba},
  // j == k -> {abc, bac}, i == j == k -> {abc}.  At nocc = 20 / 40 that removes 8.7 % / 4.6 % of the (T) flop.
  const int perm3[3][3] = {{0, 1, 2}, {1, 0, 2}, {2, 1, 0}};   // s = abc, bac, cba (first three rows of c_perm)
  const long long cap_blocks = std::max<long long>(3, std::min<long long>(65535, s.opt.triples_batch_bytes / ((do_m ? 2 : 1) * v3 * 8)));
  struct Batch { size_t t0; int ntri; size_t b0; int nblk; };
  std::vector<Batch> batches;
  struct Blk { int pq, r, pq2, r2; long long slot; };
  std::vector<Blk> blks;                             // GEMM blocks of all batches, batch after batch
  {
    Batch cur{0, 0, 0, 0};
    for (size_t t = 0; t < tri.size(); ++t) {
      TripleDesc& td = tri[t];
      const bool same_ij = td.i == td.j, same_jk = td.j == td.k;
      const int need = 1 + (same_ij ? 0 : 1) + (same_jk ? 0 : 1);
      if (cur.nblk + need > cap_blocks) { batches.push_back(cur); cur = Batch{t, 0, blks.size(), 0}; }
      const int idx[3] = {td.i, td.j, td.k};
      td.flags = same_jk ? kCbaFromBac : 0;
      for (int sidx = 0; sidx < 3; ++sidx) {
        if (sidx == 1 && same_ij) { td.slot[1] = td.slot[0]; continue; }
        if (sidx == 2 && same_jk) { td.slot[2] = td.slot[1]; continue; }
        const int P0 = idx[perm3[sidx][0]], P1 = idx[perm3[sidx][1]], P2 = idx[perm3[sidx][2]];
        td.slot[sidx] = cur.nblk;
        blks.push_back({P0 + o * P1, P2, P0 + o * P2, P1, cur.nblk});   // Acat(P0,P1) Bcat(P2) + Acat(P0,P2) BcatT(P1)
        ++cur.nblk;
      }
      ++cur.ntri;
    }
    batches.push_back(cur);
  }
  const size_t nbatches = batches.size();
  long long max_blk = 0;
  for (const Batch& b : batches) max_blk = std::max<long long>(max_blk, b.nblk);
  Scratch X(e.pool, (size_t)max_blk * v3);
  std::unique_ptr<Scratch> XM;
  if (do_m) XM.reset(new Scratch(e.pool, (size_t)max_blk * v3));
  // unordered label-tile triples A <= B <= C
  const int ntile = (v + TS - 1) / TS;
  std::vector<int> tiles_h;
  for (int A = 0; A < ntile; ++A)
    for (int B = A; B < ntile; ++B)
      for (int C = B; C < ntile; ++C) { tiles_h.push_back(A); tiles_h.push_back(B); tiles_h.push_back(C); }
  const long long ntt = (long long)tiles_h.size() / 3;
  AFESP_REQUIRE(ntt < (1LL << 31), "triples: too many label tiles");
  Scratch tiles_d(e.pool, (tiles_h.size() + 1) / 2 + 1);
  AFESP_CUDA_CHECK(cudaMemcpyAsync(tiles_d.p, tiles_h.data(), tiles_h.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  static_assert(sizeof(TripleDesc) == 40, "TripleDesc layout");
  const bool al16 = (v % 2 == 0) && (n % 2 == 0);

  // Launch tables of ALL batches, built on the host and uploaded once (no per-batch synchronisation): the triple
  // descriptors, and per GEMM block the (A pair, B index) of both K segments as block indices (TMA gather form) and as
  // pointers (cp.async fallback).  Within a batch the blocks are sorted by their B blocks so that blocks reading the same
  // (n x v^2) operand block -- 52 MB at nbf=200, 0.4 GB at nbf=400 -- run back to back and find it in L2; each block
  // still writes its own slot of the output buffer (the epilogue addresses Y through TripleDesc::slot).
  const size_t ngt = blks.size();                    // GEMM blocks over all batches
  std::vector<int> hidx(ngt * 4);                    // [4][ngt]: Aidx, Bidx, Aidx2, Bidx2
  std::vector<long long> hslot(ngt);                 // output slot within the batch buffer
  for (const Batch& b : batches) {
    std::vector<int> order(b.nblk);
    for (int z = 0; z < b.nblk; ++z) order[z] = z;
    const Blk* bb = blks.data() + b.b0;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
      return bb[x].r != bb[y].r ? bb[x].r < bb[y].r : bb[x].r2 < bb[y].r2;
    });
    for (int z = 0; z < b.nblk; ++z) {
      const Blk& k = bb[order[z]];
      const size_t w = b.b0 + z;
      hidx[0 * ngt + w] = k.pq; hidx[1 * ngt + w] = k.r;
      hidx[2 * ngt + w] = k.pq2; hidx[3 * ngt + w] = k.r2;
      hslot[w] = k.slot;
    }
  }
  Scratch descs(e.pool, tri.size() * 5);             // TripleDesc is 40 bytes = 5 doubles
  Scratch idx_d(e.pool, ngt * 2 + 2);                // 4 * ngt int32
  AFESP_CUDA_CHECK(cudaMemcpyAsync(descs.p, tri.data(), tri.size() * sizeof(TripleDesc), cudaMemcpyHostToDevice, st));
  AFESP_CUDA_CHECK(cudaMemcpyAsync(idx_d.p, hidx.data(), hidx.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  const int* didx = reinterpret_cast<const int*>(idx_d.p);
  // pointer tables (5 per block: A, B, C, A2, B2) for one operand set; built once per set
  auto make_ptrs = [&](const double* Acat, const double* Bcat, const double* BcatT, double* out, Scratch& dst) {
    std::vector<const double*> hp(ngt * 5);
    for (size_t w = 0; w < ngt; ++w) {
      hp[0 * ngt + w] = Acat + (long long)hidx[0 * ngt + w] * v * n;
      hp[1 * ngt + w] = Bcat + (long long)hidx[1 * ngt + w] * n * v2;
      hp[2 * ngt + w] = out + hslot[w] * v3;
      hp[3 * ngt + w] = Acat + (long long)hidx[2 * ngt + w] * v * n;
      hp[4 * ngt + w] = BcatT + (long long)hidx[3 * ngt + w] * n * v2;
    }
    AFESP_CUDA_CHECK(cudaMemcpyAsync(dst.p, hp.data(), hp.size() * sizeof(void*), cudaMemcpyHostToDevice, st));
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));     // hp is a stack-scoped staging vector (once per (T) call)
  };
  Scratch ptrs_W(e.pool, ngt * 5);
  make_ptrs(sAcat.p, sBcat.p, sBcatT.p, X.p, ptrs_W);
  std::unique_ptr<Scratch> ptrs_M;
  if (do_m) {
    ptrs_M.reset(new Scratch(e.pool, ngt * 5));
    make_ptrs(sAcatM->p, sBcatM->p, sBcatMT->p, XM->p, *ptrs_M);
  }
  Scratch batch_sums(e.pool, nbatches * 6);

  // AFESP_T_VERIFY=1: every batch also through the cp.async kernel, compared on the device; =2: control experiment,
  // the cp.async kernel against itself (both passes with the TMA path switched off)
  static const int verify_mode = std::getenv("AFESP_T_VERIFY") ? std::atoi(std::getenv("AFESP_T_VERIFY")) : 0;
  const int scope_at_entry = gemm_tma_scope_get();
  if (verify_mode == 2) gemm_tma_scope(0);
  const bool verify_t = verify_mode == 2 || (verify_mode == 1 && gemm_tma_scope_get() != 0);
  std::unique_ptr<Scratch> verify_buf, verify_cnt, verify_ptrs;
  double verify_elems = 0.0;
  if (verify_t) {
    verify_buf.reset(new Scratch(e.pool, (size_t)max_blk * v3));
    verify_cnt.reset(new Scratch(e.pool, 2));
    verify_ptrs.reset(new Scratch(e.pool, ngt * 5));
    make_ptrs(sAcat.p, sBcat.p, sBcatT.p, verify_buf->p, *verify_ptrs);
    AFESP_CUDA_CHECK(cudaMemsetAsync(verify_cnt->p, 0, 16, st));
  }
  tr.lap(1);
  for (size_t bi = 0; bi < nbatches; ++bi) {
    const size_t t0 = batches[bi].t0, w0 = batches[bi].b0;
    const int cb = batches[bi].ntri;
    const int ng = batches[bi].nblk;
    auto run_gemms = [&](const double* Acat, const double* Bcat, const double* BcatT, const Scratch& ptrs) {
      const double* const* dp = reinterpret_cast<const double* const*>(ptrs.p);
      GemmBatch b1;
      b1.count = ng; b1.Aptr = dp + 0 * ngt + w0; b1.Bptr = dp + 1 * ngt + w0;
      b1.Cptr = (double* const*)(dp + 2 * ngt + w0); b1.ptr_aligned16 = al16;
      b1.Aptr2 = dp + 3 * ngt + w0; b1.Bptr2 = dp + 4 * ngt + w0;
      b1.Abase = Acat; b1.Ablock = (long long)v * n; b1.Anblocks = (long long)o * o; b1.Aidx = didx + 0 * ngt + w0;
      b1.Bbase = Bcat; b1.Bblock = (long long)n * v2; b1.Bnblocks = o; b1.Bidx = didx + 1 * ngt + w0;
      b1.Bbase2 = BcatT; b1.Aidx2 = didx + 2 * ngt + w0; b1.Bidx2 = didx + 3 * ngt + w0;
      dgemm(st, 'N', 'N', v, (int)v2, n, 1.0, nullptr, v, nullptr, n, 0.0, nullptr, v, &b1);
      tr.lap(4);
    };
    run_gemms(sAcat.p, sBcat.p, sBcatT.p, ptrs_W);
    if (verify_t) {
      // the same batch once more through the cp.async kernel, element-wise comparison on the device
      const int scope = gemm_tma_scope_get();
      gemm_tma_scope(0);
      run_gemms(sAcat.p, sBcat.p, sBcatT.p, *verify_ptrs);
      gemm_tma_scope(scope);
      k_count_mismatch<<<148 * 8, 256, 0, st>>>(X.p, verify_buf->p, (long long)ng * v3, 1e-11,
                                                reinterpret_cast<unsigned long long*>(verify_cnt->p));
      verify_elems += (double)ng * v3;
    }
    if (do_m) run_gemms(sAcatM->p, sBcatM->p, sBcatMT->p, *ptrs_M);
    FusedArgs fa{};
    fa.X = X.p; fa.XM = do_m ? XM->p : nullptr; fa.t1 = s.t1.p(); fa.t2 = s.t2.p(); fa.vo = s.get("v_oovv").p();
    fa.eo = s.eo.p(); fa.ev = s.ev.p(); fa.tr = reinterpret_cast<const TripleDesc*>(descs.p) + t0;
    fa.tiles = reinterpret_cast<const int*>(tiles_d.p);
    fa.o = o; fa.v = v;
    const long long nblocks = ntt * cb;
    fa.partials = reduce_scratch(e, (size_t)nblocks * 6);
    dim3 grid((unsigned)ntt, (unsigned)cb), block(TS, TS, TS);
    {
      auto go = [&](auto kern, size_t smem_doubles) {
        const size_t fsmem = smem_doubles * sizeof(double);
        AFESP_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));
        kern<<<grid, block, fsmem, st>>>(fa);
      };
      const int mode = (use_z ? 8 : 0) | (do_y ? 4 : 0) | (do_m ? 2 : 0) | (paren ? 1 : 0);
      switch (mode) {
        case 0: go(k_triples_fused<false, false, false, false>, fused_smem_doubles<false, false, false>()); break;   // CCSD[T]
        case 1: go(k_triples_fused<false, false, false, true>, fused_smem_doubles<false, false, false>()); break;    // CCSD(T) as coded (Q2: no z3_bar)
        case 4: go(k_triples_fused<false, true, false, false>, fused_smem_doubles<false, true, false>()); break;    // R-CCSD[T]
        case 13: go(k_triples_fused<true, true, false, true>, fused_smem_doubles<true, true, false>()); break;     // R-CCSD(T)
        case 6: go(k_triples_fused<false, true, true, false>, fused_smem_doubles<false, true, true>()); break;     // CR-CCSD[T]
        case 15: go(k_triples_fused<true, true, true, true>, fused_smem_doubles<true, true, true>()); break;      // CR-CCSD(T)
        default: throw Error(1, "triples: unsupported combination of calc_type flags");
      }
    }
    count_launch();
    AFESP_CUDA_CHECK(cudaGetLastError());
    tr.lap(5);
    finish_partials(e, fa.partials, (int)nblocks, 6, batch_sums.p + bi * 6);
    tr.lap(6);
  }
  {
    const char* names[] = {"operands", "setup", "-", "-", "gemm (K=2(v+o))", "fused epilogue", "finish"};
    tr.report(names, 7);
  }
  std::vector<double> h(nbatches * 6);
  AFESP_CUDA_CHECK(cudaMemcpyAsync(h.data(), batch_sums.p, h.size() * 8, cudaMemcpyDeviceToHost, st));
  AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
  if (verify_t) {
    unsigned long long cnt[2] = {0, 0};
    AFESP_CUDA_CHECK(cudaMemcpy(cnt, verify_cnt->p, 16, cudaMemcpyDeviceToHost));
    double worst;
    std::memcpy(&worst, &cnt[1], 8);
    if (verify_mode == 2) gemm_tma_scope(scope_at_entry);
    std::fprintf(stderr, verify_mode == 2 ? "[afesp T verify] CONTROL cp.async vs cp.async over %.3e X elements: %llu mismatches (worst |diff| %.3e)\n" :
                         "[afesp T verify] TMA vs cp.async over %.3e X elements: %llu mismatches (worst |diff| %.3e)\n",
                 verify_elems, cnt[0], cnt[0] ? worst : 0.0);
  }
  for (size_t bi = 0; bi < nbatches; ++bi)
    for (int k = 0; k < 6; ++k) sums[k] += h[bi * 6 + k];
  if (!paren) { sums[1] = 0.0; sums[3] = 0.0; sums[5] = 0.0; }
}

void triples_spinorb(CCState& s, int rank, int nranks, double* e_T) {
  AFESP_REQUIRE(!s.restricted, "triples_spinorb needs a spin-orbital CCSD state");
  AFESP_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "triples: bad (rank, nranks)");
  Engine& e = s.eng;
  cudaStream_t st = e.stream;
  const int o = s.o, v = s.v;
  const long long v2 = (long long)v * v, v3 = v2 * v;
  *e_T = 0.0;
  // X(a,b,c) = sum_f [ t2(j,k,a,f) vovv(f,i,b,c) - t2(i,k,a,f) vovv(f,j,b,c) - t2(j,i,a,f) vovv(f,k,b,c) ]
  //          + sum_m [ ovoo(m,a,j,k) t2(m,i,b,c) - ovoo(m,a,i,k) t2(m,j,b,c) - ovoo(m,a,j,i) t2(m,k,b,c) ]
  // (src/ccsd.f90:1881-1889 with t2(m,i,c,b) = -t2(m,i,b,c)); six DMMA GEMMs accumulate into one block.
  Tensor T2v({v, v, o, o}), Vv({v, v, v, o});
  transpose(e, "ijaf->afij", 1.0, s.t2.view(), 0.0, T2v.view());             // T2v(a,f;p,q) = t2(p,q,a,f)
  transpose(e, "fibc->fbci", 1.0, s.get("vovv").view(), 0.0, Vv.view());     // Vv(f,b,c;i) = vovv(f,i,b,c)
  Tensor& ovoo = s.get("ovoo");
  // i<j<k only: the summand is symmetric in (i,j,k) and vanishes when two occupied indices coincide.
  std::vector<TripleDesc> tri = my_triples(o, s.opt.triples_ijk_symmetry, s.opt.triples_ijk_symmetry, rank, nranks);
  if (tri.empty()) return;
  const long long per_triple = v3 * 8;
  int nb = (int)std::max<long long>(1, std::min<long long>((long long)tri.size(), s.opt.triples_batch_bytes / per_triple));
  nb = std::min(nb, 65535);
  Scratch X(e.pool, (size_t)nb * v3);
  const int ntile = (v + TS - 1) / TS;
  const long long blocks_per_triple = (long long)ntile * ntile * ntile;
  DBuf descs((size_t)nb * 5);   // TripleDesc is 40 bytes = 5 doubles
  DevPtrs ptrs;
  ptrs.ensure((size_t)nb * 13);
  const size_t nbatches = (tri.size() + nb - 1) / nb;
  DBuf batch_sums(nbatches);
  const bool al16 = (v % 2 == 0) && (o % 2 == 0);
  for (size_t bi = 0; bi < nbatches; ++bi) {
    const size_t t0 = bi * nb;
    const int cb = (int)std::min<size_t>(nb, tri.size() - t0);
    AFESP_CUDA_CHECK(cudaMemcpyAsync(descs.p, &tri[t0], (size_t)cb * sizeof(TripleDesc), cudaMemcpyHostToDevice, st));
    std::vector<const double*> hp((size_t)cb * 13);
    for (int tb = 0; tb < cb; ++tb) {
      const TripleDesc& td = tri[t0 + tb];
      const int i = td.i, j = td.j, k = td.k;
      // term s: (p,q | r) for the f-sum, (q',r' | p') for the m-sum
      const int pq[3][2] = {{j, k}, {i, k}, {j, i}};
      const int r[3] = {i, j, k};
      for (int t = 0; t < 3; ++t) {
        hp[(size_t)(0 + t) * cb + tb] = T2v.p() + ((long long)pq[t][0] + (long long)o * pq[t][1]) * v2;  // (a x f)
        hp[(size_t)(3 + t) * cb + tb] = Vv.p() + (long long)r[t] * v3;                                   // (f x bc)
        hp[(size_t)(6 + t) * cb + tb] = ovoo.p() + ((long long)pq[t][0] + (long long)o * pq[t][1]) * o * v;  // (m x a)
        hp[(size_t)(9 + t) * cb + tb] = s.t2.p() + (long long)o * r[t];                                  // (m x bc), ld o^2
      }
      hp[(size_t)12 * cb + tb] = X.p + (long long)tb * v3;
    }
    AFESP_CUDA_CHECK(cudaMemcpyAsync(ptrs.raw.p, hp.data(), hp.size() * sizeof(void*), cudaMemcpyHostToDevice, st));
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
    const double* const* dp = reinterpret_cast<const double* const*>(ptrs.raw.p);
    double* const* cp = (double* const*)(dp + (size_t)12 * cb);
    for (int t = 0; t < 3; ++t) {
      GemmBatch b1;
      b1.count = cb; b1.Aptr = dp + (size_t)(0 + t) * cb; b1.Bptr = dp + (size_t)(3 + t) * cb; b1.Cptr = cp;
      b1.ptr_aligned16 = al16;
      dgemm(st, 'N', 'N', v, (int)v2, v, t == 0 ? 1.0 : -1.0, nullptr, v, nullptr, v, t == 0 ? 0.0 : 1.0, nullptr, v, &b1);
    }
    for (int t = 0; t < 3; ++t) {
      GemmBatch b2;
      b2.count = cb; b2.Aptr = dp + (size_t)(6 + t) * cb; b2.Bptr = dp + (size_t)(9 + t) * cb; b2.Cptr = cp;
      b2.ptr_aligned16 = al16;
      dgemm(st, 'T', 'N', v, (int)v2, o, t == 0 ? 1.0 : -1.0, nullptr, o, nullptr, (long long)o * o, 1.0, nullptr, v, &b2);
    }
    EnergySoArgs ea{};
    ea.X = X.p; ea.t1 = s.t1.p(); ea.vo = s.get("oovv").p(); ea.eo = s.eo.p(); ea.ev = s.ev.p();
    ea.tr = reinterpret_cast<const TripleDesc*>(descs.p); ea.o = o; ea.v = v; ea.ntile = ntile;
    const long long nblocks = blocks_per_triple * cb;
    ea.partials = reduce_scratch(e, (size_t)nblocks);
    dim3 grid((unsigned)blocks_per_triple, (unsigned)cb), block(TS, TS, TS);
    k_energy_spinorb_t<<<grid, block, 0, st>>>(ea);
    count_launch();
    AFESP_CUDA_CHECK(cudaGetLastError());
    finish_partials(e, ea.partials, (int)nblocks, 1, batch_sums.p + bi);
  }
  std::vector<double> h(nbatches);
  AFESP_CUDA_CHECK(cudaMemcpyAsync(h.data(), batch_sums.p, h.size() * 8, cudaMemcpyDeviceToHost, st));
  AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
  for (double x : h) *e_T += x;
}

}  // namespace afesp
