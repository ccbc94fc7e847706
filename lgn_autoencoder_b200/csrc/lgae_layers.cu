// Remaining layer-level kernels of the reference's generic API (any maxdim, any width):
//   * complex scalar x irrep product with channel broadcast: edge features rad (x) zonal
//     (lgn/models/lgn_cg.py:167, lgn/g_lib/cplx_lib.py:54-72), forward + adjoint;
//   * RadPolyTrig: 2K Lorentzian bells of the pair norms, masked, followed by one Linear per zonal degree
//     (lgn/nn/position_levels.py:118-209), forward + adjoint with deterministic parameter gradients;
//   * Linear (+ bias, optional LeakyReLU) on rows, forward + adjoint: the CGMLP layers of widths the resident-weight
//     MLP kernel (lgae_mlp.cu) does not cover (lgn/models/lgn_levels.py:191-227).
#include <algorithm>

#include "lgae_common.cuh"

namespace lgae {

static int grid_for(int64_t work, int threads) {
    const int64_t need = (work + threads - 1) / threads, cap = (int64_t)sm_count() * 8;
    return (int)std::max<int64_t>(1, std::min(need, cap));
}

// ------------------------------------------------------------------------------------------------------------
// out[e, c, m] = s[e, c or 0] * v[e, c or 0, m]      (planar complex; cs, cv in {1, C})
// ------------------------------------------------------------------------------------------------------------
struct SvArgs {
    const double *s, *v, *g;
    double *out, *gs, *gv;
    int64_t E;
    int32_t cs, cv, C, d;
};
__global__ void __launch_bounds__(256) sv_fwd_kernel(const SvArgs a) {
    pdl_launch();
    pdl_wait();
    const int64_t per = (int64_t)a.C * a.d, total = a.E * per, sp = a.E * a.cs, vp = a.E * a.cv * a.d;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < total; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = it / per;
        const int w = (int)(it % per), c = w / a.d, m = w % a.d;
        const int64_t si = e * a.cs + (a.cs == 1 ? 0 : c), vi = (e * a.cv + (a.cv == 1 ? 0 : c)) * a.d + m;
        const cplx r = cmul(cmake(a.s[si], a.s[sp + si]), cmake(a.v[vi], a.v[vp + vi]));
        a.out[it] = r.x;
        a.out[total + it] = r.y;
    }
}
// gs[e, cs] = sum conj(v) g ; gv[e, cv, m] = sum conj(s) g   (sums over the broadcast axes, fixed order)
__global__ void __launch_bounds__(256) sv_bwd_kernel(const SvArgs a) {
    pdl_launch();
    pdl_wait();
    const int64_t gp = a.E * a.C * a.d, sp = a.E * a.cs, vp = a.E * a.cv * a.d;
    const int64_t n1 = a.gs ? sp : 0, n2 = a.gv ? vp : 0;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < n1 + n2; it += (int64_t)gridDim.x * blockDim.x) {
        cplx acc = czero();
        if (it < n1) {
            const int64_t e = it / a.cs;
            const int c0 = (int)(it % a.cs), c1 = a.cs == 1 ? a.C : c0 + 1;
            for (int c = c0; c < c1; ++c)
                for (int m = 0; m < a.d; ++m) {
                    const int64_t vi = (e * a.cv + (a.cv == 1 ? 0 : c)) * a.d + m, gi = (e * a.C + c) * a.d + m;
                    cfmac(acc, cmake(a.v[vi], a.v[vp + vi]), cmake(a.g[gi], a.g[gp + gi]));
                }
            a.gs[it] = acc.x;
            a.gs[sp + it] = acc.y;
        } else {
            const int64_t j = it - n1, e = j / ((int64_t)a.cv * a.d);
            const int w = (int)(j % ((int64_t)a.cv * a.d)), c0 = w / a.d, m = w % a.d, c1 = a.cv == 1 ? a.C : c0 + 1;
            for (int c = c0; c < c1; ++c) {
                const int64_t si = e * a.cs + (a.cs == 1 ? 0 : c), gi = (e * a.C + c) * a.d + m;
                cfmac(acc, cmake(a.s[si], a.s[sp + si]), cmake(a.g[gi], a.g[gp + gi]));
            }
            a.gv[j] = acc.x;
            a.gv[vp + j] = acc.y;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// RadPolyTrig.  x: E scalars (pair norms; the canonical basis passes its (2,B,N,N) re/im slices as 2*B*N*N scalars),
// mask: per edge, index e % n_mask.  bell_k = b_k / (1 + (c_k x)^2 + 1e-16) + a_k, zero on masked edges.
// For every zonal degree l: y_l = W_l bell + bias_l (W_l: nout x K2).  Output element (e, o):
//   planar != 0 (Cartesian): (2, E, nout/2) with o = 2c + re/im;   planar == 0 (canonical): (E, nout).
// ------------------------------------------------------------------------------------------------------------
#define RAD_MAX_L 4
struct RadArgs {
    const double *x, *a, *b, *c;
    const uint8_t* mask;
    const double* w[RAD_MAX_L];
    const double* bias[RAD_MAX_L];
    double* out[RAD_MAX_L];        // forward outputs / adjoint: their gradients
    double *gx, *part;             // adjoint: d/dx (E) and per-CTA parameter partial rows
    int64_t E, n_mask;
    int32_t K2, nout, L, planar, part_stride;
};
#ifndef LGAE_RAD_EB
#define LGAE_RAD_EB 64
#endif
#ifndef LGAE_RAD_CTAS
#define LGAE_RAD_CTAS 4
#endif
constexpr int RAD_EB = LGAE_RAD_EB;   // edges per block iteration
constexpr int RAD_T = 256;
// Row strides of the per-edge shared-memory tables, made odd: a warp that walks the edges at a fixed column then hits 16
// different bank pairs instead of 2-4 (K2 = 20) or one (n_l * n_out = 32).
__host__ __device__ inline int rad_odd(int n) { return n | 1; }

LGAE_DEV int64_t rad_out_index(const RadArgs& p, int64_t e, int o) {
    return p.planar ? (int64_t)(o & 1) * p.E * (p.nout / 2) + e * (p.nout / 2) + (o >> 1) : e * p.nout + o;
}
// bells (and optionally r = 1/(1+(cx)^2+1e-16)) of a block of edges -> shared memory [edge][K2]
LGAE_DEV void rad_bells(const RadArgs& p, int64_t e0, int ne, const double* pa, const double* pb, const double* pc, double* bell, double* rr) {
    for (int t = threadIdx.x; t < ne * p.K2; t += blockDim.x) {
        const int e = t / p.K2, k = t % p.K2;
        const int64_t ge = e0 + e;
        const bool on = p.mask[ge % p.n_mask] != 0;
        const double cx = pc[k] * p.x[ge];
        // same operation order as the reference: (1 + (c x)^2 + 1e-16)^-1, then b * (...) + a
        const double r = 1.0 / (__dadd_rn(__dadd_rn(1.0, __dmul_rn(cx, cx)), 1e-16));
        bell[e * rad_odd(p.K2) + k] = on ? __dadd_rn(__dmul_rn(pb[k], r), pa[k]) : 0.0;
        if (rr) rr[e * rad_odd(p.K2) + k] = on ? r : 0.0;
    }
}
__global__ void __launch_bounds__(RAD_T) rad_fwd_kernel(const RadArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int K2 = p.K2, nout = p.nout, L = p.L;
    double* pa = smem;
    double* pb = pa + K2;
    double* pc = pb + K2;
    double* ws = pc + K2;                    // L * nout * K2
    double* bs = ws + (size_t)L * nout * K2;  // L * nout
    double* bell = bs + (size_t)L * nout;     // RAD_EB * KS
    const int KS = rad_odd(K2);
    for (int t = threadIdx.x; t < K2; t += blockDim.x) { pa[t] = p.a[t]; pb[t] = p.b[t]; pc[t] = p.c[t]; }
    for (int l = 0; l < L; ++l) {
        for (int t = threadIdx.x; t < nout * K2; t += blockDim.x) ws[(size_t)l * nout * K2 + t] = p.w[l][t];
        for (int t = threadIdx.x; t < nout; t += blockDim.x) bs[l * nout + t] = p.bias[l][t];
    }
    pdl_wait();
    for (int64_t e0 = (int64_t)blockIdx.x * RAD_EB; e0 < p.E; e0 += (int64_t)gridDim.x * RAD_EB) {
        const int ne = (int)min((int64_t)RAD_EB, p.E - e0);
        __syncthreads();
        rad_bells(p, e0, ne, pa, pb, pc, bell, nullptr);
        __syncthreads();
        for (int t = threadIdx.x; t < ne * nout * L; t += blockDim.x) {
            // planar: consecutive threads walk the edges of one (l, o) => coalesced stores
            const int e = t % ne, o = (t / ne) % nout, l = t / (ne * nout);
            const double* w = ws + ((size_t)l * nout + o) * K2;
            const double* be = bell + (size_t)e * KS;
            double acc = 0.0;
            for (int k = 0; k < K2; ++k) acc = fma(be[k], w[k], acc);
            p.out[l][rad_out_index(p, e0 + e, o)] = acc + bs[l * nout + o];
        }
    }
}
// Adjoint.  Partial row per CTA: [l][nout][K2] dW, [l][nout] dbias, da[K2], db[K2], dc[K2].
__global__ void __launch_bounds__(RAD_T) rad_bwd_kernel(const RadArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int K2 = p.K2, nout = p.nout, L = p.L, LO = L * nout;
    double* pa = smem;
    double* pb = pa + K2;
    double* pc = pb + K2;
    double* ws = pc + K2;                     // LO * K2
    const int KS = rad_odd(K2), GS = rad_odd(LO);
    double* bell = ws + (size_t)LO * K2;      // RAD_EB * KS
    double* rr = bell + (size_t)RAD_EB * KS;  // RAD_EB * KS
    double* gb = rr + (size_t)RAD_EB * KS;    // RAD_EB * KS: d/dbell
    double* gy = gb + (size_t)RAD_EB * KS;    // RAD_EB * GS
    double* accs = gy + (size_t)RAD_EB * GS;  // LO*K2 + LO + 3*K2 accumulators (one owner thread each)
    const int n_w = LO * K2, n_acc = n_w + LO + 3 * K2;
    for (int t = threadIdx.x; t < K2; t += blockDim.x) { pa[t] = p.a[t]; pb[t] = p.b[t]; pc[t] = p.c[t]; }
    for (int l = 0; l < L; ++l)
        for (int t = threadIdx.x; t < nout * K2; t += blockDim.x) ws[(size_t)l * nout * K2 + t] = p.w[l][t];
    for (int t = threadIdx.x; t < n_acc; t += blockDim.x) accs[t] = 0.0;
    pdl_wait();
    for (int64_t e0 = (int64_t)blockIdx.x * RAD_EB; e0 < p.E; e0 += (int64_t)gridDim.x * RAD_EB) {
        const int ne = (int)min((int64_t)RAD_EB, p.E - e0);
        __syncthreads();
        rad_bells(p, e0, ne, pa, pb, pc, bell, rr);
        for (int t = threadIdx.x; t < ne * LO; t += blockDim.x) {
            const int e = t % ne, lo = t / ne;
            gy[(size_t)e * GS + lo] = p.out[lo / nout][rad_out_index(p, e0 + e, lo % nout)];
        }
        __syncthreads();
        // d/dbell[e, k] = sum_lo W[lo, k] gy[e, lo]   (zero on masked edges: rr == 0 there)
        for (int t = threadIdx.x; t < ne * K2; t += blockDim.x) {
            const int e = t / K2, k = t % K2;
            double acc = 0.0;
            for (int lo = 0; lo < LO; ++lo) acc = fma(ws[(size_t)lo * K2 + k], gy[(size_t)e * GS + lo], acc);
            gb[e * KS + k] = rr[e * KS + k] != 0.0 ? acc : 0.0;
        }
        // dW[lo, k] += sum_e gy[e, lo] bell[e, k];  dbias[lo] += sum_e gy[e, lo]
        for (int t = threadIdx.x; t < n_w + LO; t += blockDim.x) {
            double acc = 0.0;
            if (t < n_w) {
                const int lo = t / K2, k = t % K2;
                for (int e = 0; e < ne; ++e) acc = fma(gy[(size_t)e * GS + lo], bell[(size_t)e * KS + k], acc);
            } else {
                const int lo = t - n_w;
                for (int e = 0; e < ne; ++e) acc += gy[(size_t)e * GS + lo];
            }
            accs[t] += acc;
        }
        __syncthreads();
        // da, db, dc and d/dx from d/dbell
        for (int t = threadIdx.x; t < 3 * K2; t += blockDim.x) {
            const int which = t / K2, k = t % K2;
            double acc = 0.0;
            for (int e = 0; e < ne; ++e) {
                const double g = gb[(size_t)e * KS + k], r = rr[(size_t)e * KS + k];
                if (which == 0) acc += g;
                else if (which == 1) acc = fma(g, r, acc);
                else { const double x = p.x[e0 + e]; acc = fma(g, -2.0 * pb[k] * r * r * pc[k] * x * x, acc); }
            }
            accs[n_w + LO + t] += acc;
        }
        if (p.gx)
            for (int e = threadIdx.x; e < ne; e += blockDim.x) {
                const double x = p.x[e0 + e];
                double acc = 0.0;
                for (int k = 0; k < K2; ++k) {
                    const double r = rr[(size_t)e * KS + k];
                    acc = fma(gb[(size_t)e * KS + k], -2.0 * pb[k] * r * r * pc[k] * pc[k] * x, acc);
                }
                p.gx[e0 + e] = acc;
            }
    }
    __syncthreads();
    double* row = p.part + (int64_t)blockIdx.x * p.part_stride;
    for (int t = threadIdx.x; t < n_acc; t += blockDim.x) row[t] = accs[t];
}

// ------------------------------------------------------------------------------------------------------------
// Linear: tiled fp64 GEMM C[M, N] = A[M, K] B[K, N] with functor loads; 64 x 64 tile per CTA, 4 x 4 per thread.
// ------------------------------------------------------------------------------------------------------------
constexpr int GT = 64, GK = 16;
struct LinArgs {
    const double *x, *w, *b, *y, *gy;
    double *out, *part;
    int64_t rows;
    int32_t nin, nout, act;
    double slope;
    int64_t rows_per_split;
};
template <class LA, class LB, class ST>
LGAE_DEV void gemm_tile(int64_t M, int N, int64_t K0, int64_t K1, LA la, LB lb, ST store) {
    __shared__ double As[GK][GT + 1], Bs[GK][GT + 1];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const int64_t m0 = (int64_t)blockIdx.x * GT;
    const int n0 = blockIdx.y * GT;
    double acc[4][4] = {};
    for (int64_t k0 = K0; k0 < K1; k0 += GK) {
        __syncthreads();
        for (int t = threadIdx.x; t < GK * GT; t += blockDim.x) {
            const int kk = t % GK, mm = t / GK;
            As[kk][mm] = (m0 + mm < M && k0 + kk < K1) ? la(m0 + mm, k0 + kk) : 0.0;
        }
        for (int t = threadIdx.x; t < GK * GT; t += blockDim.x) {
            const int nn = t % GT, kk = t / GT;
            Bs[kk][nn] = (n0 + nn < N && k0 + kk < K1) ? lb(k0 + kk, n0 + nn) : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GK; ++kk) {
            double av[4], bv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { av[i] = As[kk][ty * 4 + i]; bv[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t m = m0 + ty * 4 + i;
            const int n = n0 + tx * 4 + j;
            if (m < M && n < N) store(m, n, acc[i][j]);
        }
}
LGAE_DEV double act_grad(const LinArgs& a, int64_t idx) {
    const double g = a.gy[idx];
    return a.act ? (a.y[idx] > 0.0 ? g : g * a.slope) : g;
}
// y = act(x W^T + b)
__global__ void __launch_bounds__(256) lin_fwd_kernel(const LinArgs a) {
    pdl_launch();
    pdl_wait();
    gemm_tile(a.rows, a.nout, 0, a.nin,
              [&](int64_t m, int64_t k) { return a.x[m * a.nin + k]; },
              [&](int64_t k, int n) { return a.w[(int64_t)n * a.nin + k]; },
              [&](int64_t m, int n, double v) {
                  v += a.b ? a.b[n] : 0.0;
                  a.out[m * a.nout + n] = a.act ? leaky(v, a.slope) : v;
              });
}
// gx = dZ W,  dZ = gy * act'(y)
__global__ void __launch_bounds__(256) lin_bwd_x_kernel(const LinArgs a) {
    pdl_launch();
    pdl_wait();
    gemm_tile(a.rows, a.nin, 0, a.nout,
              [&](int64_t m, int64_t k) { return act_grad(a, m * a.nout + k); },
              [&](int64_t k, int n) { return a.w[k * a.nin + n]; },
              [&](int64_t m, int n, double v) { a.out[m * a.nin + n] = v; });
}
// partial[z][o][i] = sum_{r in split z} dZ[r, o] x[r, i];  column i == nin holds the bias gradient
__global__ void __launch_bounds__(256) lin_bwd_w_kernel(const LinArgs a) {
    pdl_launch();
    pdl_wait();
    const int64_t r0 = (int64_t)blockIdx.z * a.rows_per_split, r1 = min(a.rows, r0 + a.rows_per_split);
    double* part = a.part + (int64_t)blockIdx.z * a.nout * (a.nin + 1);
    gemm_tile(a.nout, a.nin + 1, r0, r1,
              [&](int64_t m, int64_t k) { return act_grad(a, k * a.nout + m); },
              [&](int64_t k, int n) { return n < a.nin ? a.x[k * a.nin + n] : 1.0; },
              [&](int64_t m, int n, double v) { part[m * (a.nin + 1) + n] = v; });
}

// ------------------------------------------------------------------------------------------------------------
// Linear on the fp64 tensor-core MMA (DMMA m8n8k4) for layer widths <= 128 (the scalar MLPs of the generic path are
// (B N) x w x w GEMMs with w <= 96): the small operand lives in shared memory in fragment order, the row operand is
// streamed from global memory with a register prefetch, the accumulators never leave registers.
// ------------------------------------------------------------------------------------------------------------
constexpr int LMMA_MAX = 128;      // largest n_in / n_out of this path
constexpr int LMMA_THREADS = 256;
constexpr int LMMA_MT = 2;         // row groups (of 8 rows) a warp advances together
constexpr int LMMA_KC = 4;         // k-steps per prefetch chunk

// y = act(x W^T + b)  (BWDX = false: K = n_in, N = n_out)     gx = dZ W  (BWDX = true: K = n_out, N = n_in)
template <int NT, bool BWDX>
__global__ void __launch_bounds__(LMMA_THREADS, 1) lin_mma_kernel(const LinArgs a) {
    extern __shared__ __align__(16) double lin_smem[];
    double* Bs = lin_smem;   // Bs[(ks*NT + nt)*32 + lane] = B[4ks + q][8nt + g]
    const int K = BWDX ? a.nout : a.nin, N = BWDX ? a.nin : a.nout;
    const int KS = (K + 3) / 4;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, q = lane & 3;
    constexpr int MT = LMMA_MT, KC = LMMA_KC;
    pdl_launch();
    pdl_wait();
    // coalesced read of W (n_out x n_in, row-major), scattered into fragment order; padding entries are zero
    for (int t = threadIdx.x; t < KS * NT * 32; t += blockDim.x) Bs[t] = 0.0;
    __syncthreads();
    {
        const int total = a.nout * a.nin;
#pragma unroll 4
        for (int t = threadIdx.x; t < total; t += blockDim.x) {
            const int o = t / a.nin, i = t - o * a.nin;
            const int k = BWDX ? o : i, n = BWDX ? i : o;
            Bs[(((k >> 2) * NT + (n >> 3)) * 32) + ((n & 7) << 2) + (k & 3)] = a.w[t];
        }
    }
    __syncthreads();
    const bool pair_store = (N & 1) == 0;
    const int64_t units = (a.rows + 8 * MT - 1) / (8 * MT);
    for (int64_t u = (int64_t)blockIdx.x * (LMMA_THREADS / 32) + warp; u < units; u += (int64_t)gridDim.x * (LMMA_THREADS / 32)) {
        const int64_t r0 = u * 8 * MT;
        double acc[MT][NT][2];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            const int col = 8 * nt + 2 * q;
            const double b0 = (!BWDX && a.b && col < N) ? a.b[col] : 0.0, b1 = (!BWDX && a.b && col + 1 < N) ? a.b[col + 1] : 0.0;
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) { acc[mt][nt][0] = b0; acc[mt][nt][1] = b1; }
        }
        // raw operands only (no arithmetic on them here, so that the prefetch really stays in flight); BWDX: A = dZ = gy * act'(y)
        auto load_a = [&](int mt, int ks, double& v, double& yv) {
            const int64_t row = r0 + 8 * mt + g;
            const int k = 4 * ks + q;
            v = 0.0;
            yv = 1.0;
            if (row < a.rows && k < K) {
                const int64_t idx = row * K + k;
                v = BWDX ? a.gy[idx] : a.x[idx];
                if (BWDX && a.act) yv = a.y[idx];
            }
        };
        double cur[MT][KC], nxt[MT][KC], cy[MT][KC], ny[MT][KC];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int kc = 0; kc < KC; ++kc) { load_a(mt, kc, cur[mt][kc], cy[mt][kc]); nxt[mt][kc] = 0.0; ny[mt][kc] = 1.0; }
        for (int ks0 = 0; ks0 < KS; ks0 += KC) {
            if (ks0 + KC < KS) {
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                    for (int kc = 0; kc < KC; ++kc) load_a(mt, ks0 + KC + kc, nxt[mt][kc], ny[mt][kc]);
            }
#pragma unroll
            for (int kc = 0; kc < KC; ++kc) {
                const int ks = ks0 + kc;
                if (ks < KS) {
                    double av[MT];
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) av[mt] = (BWDX && !(cy[mt][kc] > 0.0)) ? cur[mt][kc] * a.slope : cur[mt][kc];
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        const double bv = Bs[(ks * NT + nt) * 32 + lane];
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) dmma(acc[mt][nt][0], acc[mt][nt][1], av[mt], bv);
                    }
                }
            }
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int kc = 0; kc < KC; ++kc) { cur[mt][kc] = nxt[mt][kc]; cy[mt][kc] = ny[mt][kc]; }
        }
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            const int64_t row = r0 + 8 * mt + g;
            if (row >= a.rows) continue;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int col = 8 * nt + 2 * q;
                if (col >= N) continue;
                double v0 = acc[mt][nt][0], v1 = acc[mt][nt][1];
                if (!BWDX && a.act) { v0 = leaky(v0, a.slope); v1 = leaky(v1, a.slope); }
                double* dst = a.out + row * N + col;
                if (pair_store) {
                    *reinterpret_cast<double2*>(dst) = make_double2(v0, v1);
                } else {
                    dst[0] = v0;
                    if (col + 1 < N) dst[1] = v1;
                }
            }
        }
    }
}

// partial[z][o][i] = sum_{r in split z} dZ[r, o] x[r, i]  (column i == nin: the bias gradient) as an MMA contraction over
// the rows of the split: A[o][r] = dZ[r][o], B[r][i] = x[r][i].  Warp (wm, wn) owns the output tiles (mt = wm + 4 i, nt = wn + 2 j)
// -- strided, so that the four schedulers of the SM carry the same number of tiles -- and fetches its operand fragments
// (L1-resident rows shared by the 8 warps) one k-step ahead.
constexpr int LW_TM = 4, LW_TN = 8;
__global__ void __launch_bounds__(LMMA_THREADS, 1) lin_bwd_w_mma_kernel(const LinArgs a) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, q = lane & 3;
    const int wm = warp & 3, wn = warp >> 2;
    const int MTt = (a.nout + 7) / 8, NTt = (a.nin + 1 + 7) / 8;
    pdl_launch();
    pdl_wait();
    const int64_t r0 = (int64_t)blockIdx.x * a.rows_per_split, r1 = min(a.rows, r0 + a.rows_per_split);
    double acc[LW_TM][LW_TN][2];
#pragma unroll
    for (int i = 0; i < LW_TM; ++i)
#pragma unroll
        for (int j = 0; j < LW_TN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    // raw operands of one k-step (4 rows); the activation derivative is applied when they are used, so that the loads of
    // the next k-step stay in flight during this one's MMAs
    auto fetch = [&](int64_t r, double (&av)[LW_TM], double (&yv)[LW_TM], double (&bv)[LW_TN]) {
        const int64_t rr = r + q;
        const bool ok = rr < r1;
#pragma unroll
        for (int i = 0; i < LW_TM; ++i) {
            const int o = 8 * (wm + 4 * i) + g;
            const bool in = ok && o < a.nout;
            av[i] = in ? a.gy[rr * a.nout + o] : 0.0;
            yv[i] = (in && a.act) ? a.y[rr * a.nout + o] : 1.0;
        }
#pragma unroll
        for (int j = 0; j < LW_TN; ++j) {
            const int c = 8 * (wn + 2 * j) + g;
            bv[j] = ok ? (c < a.nin ? a.x[rr * a.nin + c] : (c == a.nin ? 1.0 : 0.0)) : 0.0;
        }
    };
    double av[LW_TM], yv[LW_TM], bv[LW_TN], an[LW_TM], yn[LW_TM], bn[LW_TN];
#pragma unroll
    for (int i = 0; i < LW_TM; ++i) { av[i] = an[i] = 0.0; yv[i] = yn[i] = 1.0; }
#pragma unroll
    for (int j = 0; j < LW_TN; ++j) bv[j] = bn[j] = 0.0;
    if (r0 < r1) fetch(r0, av, yv, bv);
    for (int64_t r = r0; r < r1; r += 4) {
        if (r + 4 < r1) fetch(r + 4, an, yn, bn);
#pragma unroll
        for (int i = 0; i < LW_TM; ++i) {
            if (wm + 4 * i < MTt) {
                const double ai = yv[i] > 0.0 ? av[i] : av[i] * a.slope;
#pragma unroll
                for (int j = 0; j < LW_TN; ++j)
                    if (wn + 2 * j < NTt) dmma(acc[i][j][0], acc[i][j][1], ai, bv[j]);
            }
        }
#pragma unroll
        for (int i = 0; i < LW_TM; ++i) { av[i] = an[i]; yv[i] = yn[i]; }
#pragma unroll
        for (int j = 0; j < LW_TN; ++j) bv[j] = bn[j];
    }
    double* part = a.part + (int64_t)blockIdx.x * a.nout * (a.nin + 1);
#pragma unroll
    for (int i = 0; i < LW_TM; ++i) {
        const int o = 8 * (wm + 4 * i) + g;
        if (o >= a.nout) continue;
#pragma unroll
        for (int j = 0; j < LW_TN; ++j) {
            const int c = 8 * (wn + 2 * j) + 2 * q;
            if (c <= a.nin) part[(int64_t)o * (a.nin + 1) + c] = acc[i][j][0];
            if (c + 1 <= a.nin) part[(int64_t)o * (a.nin + 1) + c + 1] = acc[i][j][1];
        }
    }
}

// gw[o, i] / gb[o] = sum_z partial[z][o][i]
__global__ void __launch_bounds__(256) lin_reduce_kernel(const double* part, int splits, int nout, int nin, double* gw, double* gb) {
    pdl_launch();
    pdl_wait();
    const int n = nout * (nin + 1);
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int z = 0; z < splits; ++z) s += part[(int64_t)z * n + t];
        const int o = t / (nin + 1), i = t % (nin + 1);
        if (i < nin) { if (gw) gw[(int64_t)o * nin + i] = s; }
        else if (gb) gb[o] = s;
    }
}
__global__ void __launch_bounds__(256) rows_sum_kernel(const double* part, int rows, int64_t stride, int64_t n, double* out) {
    pdl_launch();
    pdl_wait();
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int r = 0; r < rows; ++r) s += part[(int64_t)r * stride + t];
        out[t] = s;
    }
}

static int lin_splits(int64_t rows) {
    const int64_t s = std::min<int64_t>((rows + 127) / 128, (int64_t)sm_count());
    return (int)std::max<int64_t>(1, s);
}
// Widths above LMMA_MAX use the plain tiled-FMA kernels.
static bool lin_use_mma(int n_in, int n_out) { return n_in <= LMMA_MAX && n_out <= LMMA_MAX; }
template <bool BWDX>
static int launch_lin_mma(const LinArgs& a, cudaStream_t st) {
    const int K = BWDX ? a.nout : a.nin, N = BWDX ? a.nin : a.nout;
    const int KS = (K + 3) / 4, nt = (N + 7) / 8;
    const int64_t units = (a.rows + 8 * LMMA_MT - 1) / (8 * LMMA_MT);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((units + LMMA_THREADS / 32 - 1) / (LMMA_THREADS / 32), sm_count()));
#define LGAE_LIN(NTV)                                                                      \
    {                                                                                      \
        auto kern = lin_mma_kernel<NTV, BWDX>;                                             \
        const size_t bytes = (size_t)KS * NTV * 32 * sizeof(double);                       \
        if (int rc = ensure_smem((const void*)kern, bytes)) return rc;                     \
        launch_k(kern, dim3(grid), dim3(LMMA_THREADS), bytes, st, a);                      \
    }
    if (nt <= 2) LGAE_LIN(2) else if (nt <= 4) LGAE_LIN(4) else if (nt <= 8) LGAE_LIN(8) else if (nt <= 12) LGAE_LIN(12) else LGAE_LIN(16)
#undef LGAE_LIN
    return LGAE_OK;
}
static int rad_ctas(int64_t E) {
    return (int)std::max<int64_t>(1, std::min<int64_t>((E + RAD_EB - 1) / RAD_EB, LGAE_RAD_CTAS * (int64_t)sm_count()));
}

}  // namespace lgae

using namespace lgae;

extern "C" {

int lgae_scalar_irrep_forward(const double* s, const double* v, int64_t edges, int32_t cs, int32_t cv, int32_t d, double* out, void* stream) {
    if (edges < 0 || cs < 1 || cv < 1 || d < 1 || (cs != cv && cs != 1 && cv != 1)) return LGAE_E_BADARG;
    if (edges == 0) return LGAE_OK;
    if (!s || !v || !out) return LGAE_E_BADARG;
    SvArgs a = {};
    a.s = s; a.v = v; a.out = out; a.E = edges; a.cs = cs; a.cv = cv; a.C = std::max(cs, cv); a.d = d;
    cudaStream_t st = (cudaStream_t)stream;
    LaunchScope ls_("scalar_irrep_fwd", st);
    launch_k(sv_fwd_kernel, dim3(grid_for(edges * a.C * d, 256)), dim3(256), 0, st, a);
    return check_launch("scalar_irrep_fwd");
}
int lgae_scalar_irrep_backward(const double* s, const double* v, const double* g_out, int64_t edges, int32_t cs, int32_t cv, int32_t d,
                               double* g_s, double* g_v, void* stream) {
    if (edges < 0 || cs < 1 || cv < 1 || d < 1 || (cs != cv && cs != 1 && cv != 1)) return LGAE_E_BADARG;
    if (edges == 0 || (!g_s && !g_v)) return LGAE_OK;
    if (!s || !v || !g_out) return LGAE_E_BADARG;
    SvArgs a = {};
    a.s = s; a.v = v; a.g = g_out; a.gs = g_s; a.gv = g_v; a.E = edges; a.cs = cs; a.cv = cv; a.C = std::max(cs, cv); a.d = d;
    cudaStream_t st = (cudaStream_t)stream;
    LaunchScope ls_("scalar_irrep_bwd", st);
    launch_k(sv_bwd_kernel, dim3(grid_for(edges * (cs + (int64_t)cv * d), 256)), dim3(256), 0, st, a);
    return check_launch("scalar_irrep_bwd");
}

static int rad_fill(RadArgs& p, const double* x, const uint8_t* mask, int64_t edges, int64_t n_mask, const double* a, const double* b,
                    const double* c, int32_t k2, int32_t n_out, int32_t n_l, const double* const* w, const double* const* bias,
                    double* const* outs, int32_t planar) {
    if (edges < 0 || n_mask < 1 || k2 < 1 || n_out < 1 || n_l < 1 || n_l > RAD_MAX_L || (planar && (n_out & 1))) return LGAE_E_BADARG;
    if (edges % n_mask) return LGAE_E_BADARG;
    if (!x || !mask || !a || !b || !c || !w || !bias || !outs) return LGAE_E_BADARG;
    p.x = x; p.mask = mask; p.a = a; p.b = b; p.c = c; p.E = edges; p.n_mask = n_mask; p.K2 = k2; p.nout = n_out; p.L = n_l; p.planar = planar;
    for (int l = 0; l < n_l; ++l) {
        if (!w[l] || !bias[l] || !outs[l]) return LGAE_E_BADARG;
        p.w[l] = w[l]; p.bias[l] = bias[l]; p.out[l] = outs[l];
    }
    return LGAE_OK;
}
int lgae_radial_functions_forward(const double* x, const uint8_t* mask, int64_t edges, int64_t n_mask, const double* a, const double* b,
                                  const double* c, int32_t k2, int32_t n_out, int32_t n_l, const double* const* w, const double* const* bias,
                                  double* const* outs, int32_t planar, void* stream) {
    RadArgs p = {};
    if (edges == 0) return LGAE_OK;
    if (int rc = rad_fill(p, x, mask, edges, n_mask, a, b, c, k2, n_out, n_l, w, bias, outs, planar)) return rc;
    const size_t bytes = ((size_t)3 * k2 + (size_t)n_l * n_out * (k2 + 1) + (size_t)RAD_EB * rad_odd(k2)) * sizeof(double);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = ensure_smem((const void*)rad_fwd_kernel, bytes)) return rc;
    LaunchScope ls_("radial_functions_fwd", st);
    launch_k(rad_fwd_kernel, dim3(std::max(1, std::min<int>((int)((edges + RAD_EB - 1) / RAD_EB), 8 * sm_count()))), dim3(RAD_T), bytes, st, p);
    return check_launch("radial_functions_fwd");
}
int64_t lgae_radial_functions_partials_doubles(int64_t edges, int32_t k2, int32_t n_out, int32_t n_l) {
    if (edges < 0 || k2 < 1 || n_out < 1 || n_l < 1) return -1;
    return (int64_t)rad_ctas(edges) * ((int64_t)n_l * n_out * (k2 + 1) + 3 * k2);
}
/* g_params: [l][n_out][k2] dW, [l][n_out] dbias, da[k2], db[k2], dc[k2] (contiguous, caller splits). */
int lgae_radial_functions_backward(const double* x, const uint8_t* mask, int64_t edges, int64_t n_mask, const double* a, const double* b,
                                   const double* c, int32_t k2, int32_t n_out, int32_t n_l, const double* const* w,
                                   const double* const* g_outs, int32_t planar, double* g_x, double* g_params, double* partials, void* stream) {
    RadArgs p = {};
    cudaStream_t st = (cudaStream_t)stream;
    if (k2 < 1 || n_out < 1 || n_l < 1 || !g_params) return LGAE_E_BADARG;
    const int64_t width = (int64_t)n_l * n_out * (k2 + 1) + 3 * k2;
    if (edges == 0) {
        if (cudaMemsetAsync(g_params, 0, (size_t)width * sizeof(double), st) != cudaSuccess) return check_launch("memset");
        return LGAE_OK;
    }
    if (!partials) return LGAE_E_BADARG;
    if (int rc = rad_fill(p, x, mask, edges, n_mask, a, b, c, k2, n_out, n_l, w, w /* bias unused */, (double* const*)g_outs, planar)) return rc;
    p.gx = g_x; p.part = partials; p.part_stride = (int32_t)width;
    const int lo = n_l * n_out;
    const size_t bytes = ((size_t)3 * k2 + (size_t)lo * k2 + (size_t)3 * RAD_EB * rad_odd(k2) + (size_t)RAD_EB * rad_odd(lo) + (size_t)width) * sizeof(double);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)rad_bwd_kernel, bytes)) return rc;
    const int ctas = rad_ctas(edges);
    {
        LaunchScope ls_("radial_functions_bwd", st);
        launch_k(rad_bwd_kernel, dim3(ctas), dim3(RAD_T), bytes, st, p);
        if (int rc = check_launch("radial_functions_bwd")) return rc;
    }
    LaunchScope ls_("radial_functions_bwd_sum", st);
    launch_k(rows_sum_kernel, dim3(grid_for(width, 256)), dim3(256), 0, st, (const double*)partials, ctas, width, width, g_params);
    return check_launch("radial_functions_bwd_sum");
}

int lgae_linear_forward(const double* x, const double* w, const double* b, int64_t rows, int32_t n_in, int32_t n_out, int32_t leaky_relu,
                        double slope, double* y, void* stream) {
    if (rows < 0 || n_in < 1 || n_out < 1) return LGAE_E_BADARG;
    if (rows == 0) return LGAE_OK;
    if (!x || !w || !y) return LGAE_E_BADARG;
    LinArgs a = {};
    a.x = x; a.w = w; a.b = b; a.out = y; a.rows = rows; a.nin = n_in; a.nout = n_out; a.act = leaky_relu; a.slope = slope;
    cudaStream_t st = (cudaStream_t)stream;
    LaunchScope ls_("linear_fwd", st);
    if (lin_use_mma(n_in, n_out)) {
        if (int rc = launch_lin_mma<false>(a, st)) return rc;
    } else {
        launch_k(lin_fwd_kernel, dim3((unsigned)((rows + GT - 1) / GT), (n_out + GT - 1) / GT), dim3(256), 0, st, a);
    }
    return check_launch("linear_fwd");
}
int64_t lgae_linear_partials_doubles(int64_t rows, int32_t n_in, int32_t n_out) {
    if (rows < 0 || n_in < 1 || n_out < 1) return -1;
    return (int64_t)lin_splits(rows) * n_out * (n_in + 1);
}
/* y: the forward output (needed when leaky_relu != 0 for the activation's derivative). */
int lgae_linear_backward(const double* x, const double* w, const double* y, const double* g_y, int64_t rows, int32_t n_in, int32_t n_out,
                         int32_t leaky_relu, double slope, double* g_x, double* g_w, double* g_b, double* partials, void* stream) {
    if (rows < 0 || n_in < 1 || n_out < 1) return LGAE_E_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (rows == 0) {
        if (g_w && cudaMemsetAsync(g_w, 0, (size_t)n_in * n_out * sizeof(double), st) != cudaSuccess) return check_launch("memset");
        if (g_b && cudaMemsetAsync(g_b, 0, (size_t)n_out * sizeof(double), st) != cudaSuccess) return check_launch("memset");
        return LGAE_OK;
    }
    if (!x || !w || !g_y || (leaky_relu && !y) || ((g_w || g_b) && !partials)) return LGAE_E_BADARG;
    LinArgs a = {};
    a.x = x; a.w = w; a.y = y; a.gy = g_y; a.rows = rows; a.nin = n_in; a.nout = n_out; a.act = leaky_relu; a.slope = slope;
    if (g_x) {
        a.out = g_x;
        LaunchScope ls_("linear_bwd_x", st);
        if (lin_use_mma(n_in, n_out)) {
            if (int rc = launch_lin_mma<true>(a, st)) return rc;
        } else {
            launch_k(lin_bwd_x_kernel, dim3((unsigned)((rows + GT - 1) / GT), (n_in + GT - 1) / GT), dim3(256), 0, st, a);
        }
        if (int rc = check_launch("linear_bwd_x")) return rc;
    }
    if (g_w || g_b) {
        const int splits = lin_splits(rows);
        a.part = partials;
        a.rows_per_split = (rows + splits - 1) / splits;
        {
            LaunchScope ls_("linear_bwd_w", st);
            if (lin_use_mma(n_in + 1, n_out))
                launch_k(lin_bwd_w_mma_kernel, dim3(splits), dim3(LMMA_THREADS), 0, st, a);
            else
                launch_k(lin_bwd_w_kernel, dim3((n_out + GT - 1) / GT, (n_in + 1 + GT - 1) / GT, splits), dim3(256), 0, st, a);
            if (int rc = check_launch("linear_bwd_w")) return rc;
        }
        LaunchScope ls_("linear_bwd_w_sum", st);
        launch_k(lin_reduce_kernel, dim3(grid_for((int64_t)n_out * (n_in + 1), 256)), dim3(256), 0, st, (const double*)partials, splits, (int)n_out,
                 (int)n_in, g_w, g_b);
        return check_launch("linear_bwd_w_sum");
    }
    return LGAE_OK;
}

}  // extern "C"
