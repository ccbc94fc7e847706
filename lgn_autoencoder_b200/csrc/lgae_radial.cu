// Radial functions of the encoder levels (N <= 32 path), forward and adjoint, as stand-alone kernels on the fp64
// tensor-core MMA (DMMA m8n8k4).  Replaces RadPolyTrig.forward / RadialFilters (lgn/nn/position_levels.py:118-209,
// 292-310) applied to the pair norms of zonal_functions_rel (lgn/cg_lib/zonal_functions.py:221-248):
//   n_ij   = s / sqrt|s|,  s = (p_i - p_j)^2 + 1e-16                          (Minkowski square, symmetric in i <-> j)
//   phi_k  = m_ij * ( b_k / (1 + (c_k n_ij)^2 + 1e-16) + a_k )                m_ij = mask_i mask_j [n_ij != 0]
//   R_ij   = W phi + bias   (4C outputs: level-0/1 radial weights, re/im interleaved per channel)
// Because n_ij == n_ji bit for bit, only the N(N+1)/2 unordered pairs are evaluated; the forward writes both
// (i,j) and (j,i) entries of the (B, N_j, C, 32_i, 4) tensor the level kernels stream through, and the adjoint first
// adds the two incoming gradients of a pair.
//
// Work decomposition: a warp owns a contiguous range of 16-pair units (two groups of 8 pairs = the M / K dimension of
// the MMA tiles) of the whole batch, so the grid is sized by the machine (CTAs per SM x 148), not by the batch.
#include <cstring>

#include "lgae_common.cuh"

namespace lgae {

struct RadialArgs {
    const double* theta;
    int64_t off_a, off_b, off_c, off_w0, off_b0, off_w1, off_b1;
    const double* p4;          // (B,N,4) real Cartesian
    const uint8_t* node_mask;  // (B,N) or nullptr (=> p4[...,0] != 0)
    double* r;                 // forward out: (B,N_j,C,32_i,4) = (R0.re, R0.im, R1.re, R1.im)
    double* nrm;               // forward out (optional) / adjoint in: (B, NPS) pair norms, NaN = masked edge or padding
    const double* g_r;         // adjoint in: same layout, dL/dR of the ORDERED pairs
    double* part;              // adjoint out: (gridDim.x, part_stride) rows of parameter-gradient partials
    int64_t part_stride;
    int64_t po_w0, po_b0, po_w1, po_b1, po_a, po_b, po_c;
    int B, N, C, K;
};

constexpr int RAD_MAXN = 32;
constexpr int RAD_MAXP = RAD_MAXN * (RAD_MAXN + 1) / 2;

LGAE_DEV double rad_pair_norm(const double* pi, const double* pj) {
    const double d0 = pi[0] - pj[0], d1 = pi[1] - pj[1], d2 = pi[2] - pj[2], d3 = pi[3] - pj[3];
    const double s = __dadd_rn(minkowski_sq(d0, d1, d2, d3), 1e-16);
    return s != 0.0 ? __ddiv_rn(s, __dsqrt_rn(fabs(s))) : s;
}
// The MMA columns are ordered channel-major, col = 4 c + 2 l + (re|im), i.e. exactly the (R0.re, R0.im, R1.re, R1.im) record
// of a channel: neighbouring lanes of a fragment then touch the same 32-byte sector of r / g_r.  Row 2c + (re|im) of
// linear.l (position_levels.py:171-176) is column col.
LGAE_DEV double rad_w(const RadialArgs& a, int col, int k) {
    if (k >= a.K || col >= 4 * a.C) return 0.0;
    const int o = 2 * (col >> 2) + (col & 1);
    return a.theta[(((col >> 1) & 1) ? a.off_w1 : a.off_w0) + (int64_t)o * a.K + k];
}
LGAE_DEV double rad_bias(const RadialArgs& a, int col) {
    if (col >= 4 * a.C) return 0.0;
    const int o = 2 * (col >> 2) + (col & 1);
    return a.theta[(((col >> 1) & 1) ? a.off_b1 : a.off_b0) + o];
}
// unordered pairs (i <= j) of one jet in the order p = j (j + 1) / 2 + i
LGAE_DEV void build_pair_table(int N, unsigned char* ti, unsigned char* tj) {
    for (int j = threadIdx.x; j < N; j += blockDim.x)
        for (int i = 0; i <= j; ++i) {
            ti[j * (j + 1) / 2 + i] = (unsigned char)i;
            tj[j * (j + 1) / 2 + i] = (unsigned char)j;
        }
}

// Reciprocal of x in [1, inf) to ~1 ulp: hardware seed (MUFU.RCP64H) + two Newton steps, no special cases (the argument
// 1 + (c n)^2 + 1e-16 is always finite and >= 1 for finite inputs).
LGAE_DEV double rcp_ge1(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
}

constexpr int RAD_UNIT = 16;   // pairs per work unit (two MMA groups of 8)
#ifndef LGAE_RFWD_CTAS
#define LGAE_RFWD_CTAS 4       // resident CTAs per SM the radial forward is launched with
#endif
#ifndef LGAE_RBWD_CTAS
#define LGAE_RBWD_CTAS 3       // ... and the radial adjoint (also its register cap: 3 -> 168, 4 -> 128)
#endif

// ------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------
// A warp owns a contiguous range of units; lanes 0..15 evaluate the norm of one pair each (no redundancy), the two
// MMA groups of the unit pick theirs up by shuffle.  Also writes nrm (B, NPS): n_ij, or NaN where the edge is masked,
// which is all the adjoint needs to re-evaluate the basis functions.
template <int NT, int KS>
LGAE_DEV void radial_fwd_body(const RadialArgs& a) {
    constexpr int KP = 4 * KS;
    __shared__ unsigned char ti[RAD_MAXP + RAD_UNIT], tj[RAD_MAXP + RAD_UNIT];
    __shared__ double abc_s[3 * KP];
    const int N = a.N, C = a.C, K = a.K;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    pdl_launch();
    build_pair_table(N, ti, tj);
    for (int k = threadIdx.x; k < KP; k += blockDim.x) {
        abc_s[k] = k < K ? a.theta[a.off_a + k] : 0.0;
        abc_s[KP + k] = k < K ? a.theta[a.off_b + k] : 0.0;
        abc_s[2 * KP + k] = k < K ? a.theta[a.off_c + k] : 0.0;
    }
    double wf[KS][NT], bf[NT][2];
#pragma unroll
    for (int s = 0; s < KS; ++s)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) wf[s][nt] = rad_w(a, 8 * nt + g, 4 * s + q);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        bf[nt][0] = rad_bias(a, 8 * nt + 2 * q);
        bf[nt][1] = rad_bias(a, 8 * nt + 2 * q + 1);
    }
    pdl_wait();   // p4 (normalised by an earlier kernel) is read below; r / nrm are written
    __syncthreads();
    const int NP = N * (N + 1) / 2, NU = (NP + RAD_UNIT - 1) / RAD_UNIT, NPS = NU * RAD_UNIT;
    const int total = a.B * NU, twarps = gridDim.x * nwarps;
    const int per = (total + twarps - 1) / twarps;
    const int u_begin = (blockIdx.x * nwarps + warp) * per, u_end = u_begin + per < total ? u_begin + per : total;
    for (int unit = u_begin; unit < u_end; ++unit) {
        const int b = unit / NU, p0 = (unit - b * NU) * RAD_UNIT;
        const double* pb = a.p4 + (int64_t)b * N * 4;
        double n = 0.0;
        int m = 0;
        {
            const int pid = p0 + (lane & 15);
            if (pid < NP) {
                const int i = ti[pid], j = tj[pid];
                const double4 pi = *reinterpret_cast<const double4*>(pb + 4 * i);
                const double4 pj = *reinterpret_cast<const double4*>(pb + 4 * j);
                const double vi[4] = {pi.x, pi.y, pi.z, pi.w}, vj[4] = {pj.x, pj.y, pj.z, pj.w};
                n = rad_pair_norm(vi, vj);
                const bool mi = a.node_mask ? a.node_mask[(int64_t)b * N + i] != 0 : pi.x != 0.0;
                const bool mj = a.node_mask ? a.node_mask[(int64_t)b * N + j] != 0 : pj.x != 0.0;
                m = (mi && mj && n != 0.0) ? 1 : 0;
            }
            if (lane < 16 && a.nrm) a.nrm[(int64_t)b * NPS + pid] = m ? n : __longlong_as_double(0x7ff8000000000000LL);
        }
        double acc[2][NT][2], nu[2];
        int mu[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            nu[u] = __shfl_sync(0xffffffffu, n, 8 * u + g);
            mu[u] = __shfl_sync(0xffffffffu, m, 8 * u + g);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) { acc[u][nt][0] = bf[nt][0]; acc[u][nt][1] = bf[nt][1]; }
        }
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            const int k = 4 * s + q;
            const double ak = abc_s[k], bk = abc_s[KP + k], ck = abc_s[2 * KP + k];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const double cn = ck * nu[u];
                const double phi = mu[u] ? fma(bk, rcp_ge1(1.0 + cn * cn + 1e-16), ak) : 0.0;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) dmma(acc[u][nt][0], acc[u][nt][1], phi, wf[s][nt]);
            }
        }
        double* rb = a.r + (int64_t)b * N * C * 128;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int pid = p0 + 8 * u + g;
            if (pid >= NP) continue;
            const int i = ti[pid], j = tj[pid];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int col = 8 * nt + 2 * q;
                if (col < 4 * C) {
                    const int l = (col >> 1) & 1, cc = col >> 2;
                    const double2 v = make_double2(acc[u][nt][0], acc[u][nt][1]);
                    *reinterpret_cast<double2*>(rb + ((int64_t)(j * C + cc) * 32 + i) * 4 + 2 * l) = v;
                    if (i != j) *reinterpret_cast<double2*>(rb + ((int64_t)(i * C + cc) * 32 + j) * 4 + 2 * l) = v;
                }
            }
        }
    }
}

template <int NT, int KS>
__global__ void __launch_bounds__(128, LGAE_RFWD_CTAS) radial_fwd_kernel(const RadialArgs a) {
    radial_fwd_body<NT, KS>(a);
}
// All encoder levels in one launch (blockIdx.y = level): the radial weights depend only on the momenta and on the level's own
// parameters, so the levels' launches need not be links of the step's dependency chain.
struct RadialMultiArgs {
    RadialArgs lv[LGAE_MAX_LEVELS];
};
template <int NT, int KS>
__global__ void __launch_bounds__(128, LGAE_RFWD_CTAS) radial_fwd_multi_kernel(const RadialMultiArgs m) {
    radial_fwd_body<NT, KS>(m.lv[blockIdx.y]);
}

// ------------------------------------------------------------------------------------------------------------
// adjoint
// ------------------------------------------------------------------------------------------------------------
// With G[col] the symmetrised incoming gradient of a pair (4C values), rd_k = 1 / (1 + (c_k n)^2 + 1e-16):
//   G1[col][k]   = sum_pairs G[col] * m rd_k          k < K ;   G1[col][K] = sum_pairs G[col] ;  G1[col][K+1] = sum_pairs G[col] m
//   G2[col][k]   = sum_pairs G[col] * m n^2 rd_k^2
// are two MMA-shaped contractions over the pairs; the parameter gradients are linear in them:
//   dW[col][k] = b_k G1[col][k] + a_k G1[col][K+1]      dbias[col] = G1[col][K]
//   da_k = sum_col W[col][k] G1[col][K+1]     db_k = sum_col W[col][k] G1[col][k]     dc_k = -2 b_k c_k sum_col W[col][k] G2[col][k]
// so every CTA applies that map to its own partial G1 / G2 and writes one row of partials.
// The operands of a unit (16 pairs: the two gradient entries of every pair, its norm) are fetched one unit ahead into
// registers, so the L2 latency of the scattered 8-byte reads overlaps the MMA work of the current unit.
template <int NT>
struct RadOperands {
    double g[2][2][NT][2];   // [group][k-step][m-tile][(i,j) | (j,i)]
    double n;                // norm of pair (lane & 15) of the unit, NaN = masked / invalid
};

template <int NT>
LGAE_DEV void rad_fetch(const RadialArgs& a, const unsigned char* ti, const unsigned char* tj, int unit, int NU, int NP, int NPS,
                        const int (&col_cc)[NT], const int (&col_x)[NT], int lane, RadOperands<NT>& op) {
    const int N = a.N, C = a.C, q = lane & 3;
    const int b = unit / NU, p0 = (unit - b * NU) * RAD_UNIT;
    const double* gb = a.g_r + (int64_t)b * N * C * 128;
    op.n = a.nrm[(int64_t)b * NPS + p0 + (lane & 15)];
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            const int pid = p0 + 8 * u + q + 4 * ks;
            const bool valid = pid < NP;
            const int i = valid ? ti[pid] : 0, j = valid ? tj[pid] : 0;
#pragma unroll
            for (int mt = 0; mt < NT; ++mt) {
                double v0 = 0.0, v1 = 0.0;
                if (valid && col_cc[mt] >= 0) {
                    v0 = gb[((int64_t)(j * C + col_cc[mt]) * 32 + i) * 4 + col_x[mt]];
                    if (i != j) v1 = gb[((int64_t)(i * C + col_cc[mt]) * 32 + j) * 4 + col_x[mt]];
                }
                op.g[u][ks][mt][0] = v0;
                op.g[u][ks][mt][1] = v1;
            }
        }
}

template <int NT, int KS>
__global__ void __launch_bounds__(128, LGAE_RBWD_CTAS) radial_bwd_kernel(const RadialArgs a) {
    constexpr int KP = 4 * KS;
    constexpr int NT2 = KS / 2 + 1;
    constexpr int NK = 8 * NT2, NCOL = 8 * NT;
    __shared__ unsigned char ti[RAD_MAXP + RAD_UNIT], tj[RAD_MAXP + RAD_UNIT];
    __shared__ double abc_s[3 * KP];
    __shared__ double w_s[NCOL * KP];
    __shared__ double red[2 * NCOL * NK];
    const int N = a.N, C = a.C, K = a.K;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    pdl_launch();
    build_pair_table(N, ti, tj);
    for (int k = threadIdx.x; k < KP; k += blockDim.x) {
        abc_s[k] = k < K ? a.theta[a.off_a + k] : 0.0;
        abc_s[KP + k] = k < K ? a.theta[a.off_b + k] : 0.0;
        abc_s[2 * KP + k] = k < K ? a.theta[a.off_c + k] : 0.0;
    }
    for (int t = threadIdx.x; t < NCOL * KP; t += blockDim.x) w_s[t] = rad_w(a, t / KP, t % KP);
    pdl_wait();   // g_r / nrm come from earlier kernels
    __syncthreads();
    double G1[NT][NT2][2], G2[NT][NT2][2];
#pragma unroll
    for (int mt = 0; mt < NT; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT2; ++nt) G1[mt][nt][0] = G1[mt][nt][1] = G2[mt][nt][0] = G2[mt][nt][1] = 0.0;
    // column (8 mt + g) of this lane's A fragments -> (channel, component) inside a (32_i, 4) record
    int col_cc[NT], col_x[NT];
#pragma unroll
    for (int mt = 0; mt < NT; ++mt) {
        const int col = 8 * mt + g;
        col_cc[mt] = col < 4 * C ? (col >> 2) : -1;
        col_x[mt] = col & 3;
    }
    // c_k of this lane's B-fragment columns k = 8 nt + g
    // and what that column is: a basis function (k < K), the bias column (k == K: 1), the mask column (k == K + 1: m)
    double ck[NT2], c_one[NT2], c_msk[NT2];
    bool isb[NT2];
#pragma unroll
    for (int nt = 0; nt < NT2; ++nt) {
        const int k = 8 * nt + g;
        isb[nt] = k < K;
        ck[nt] = isb[nt] ? abc_s[2 * KP + k] : 0.0;
        c_one[nt] = k == K ? 1.0 : 0.0;
        c_msk[nt] = k == K + 1 ? 1.0 : 0.0;
    }

    const int NP = N * (N + 1) / 2, NU = (NP + RAD_UNIT - 1) / RAD_UNIT, NPS = NU * RAD_UNIT;
    const int total = a.B * NU, twarps = gridDim.x * nwarps;
    const int per = (total + twarps - 1) / twarps;
    const int u_begin = (blockIdx.x * nwarps + warp) * per, u_end = u_begin + per < total ? u_begin + per : total;
    RadOperands<NT> cur, nxt;
    if (u_begin < u_end) rad_fetch<NT>(a, ti, tj, u_begin, NU, NP, NPS, col_cc, col_x, lane, cur);
    for (int unit = u_begin; unit < u_end; ++unit) {
        if (unit + 1 < u_end) rad_fetch<NT>(a, ti, tj, unit + 1, NU, NP, NPS, col_cc, col_x, lane, nxt);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                const double n2 = __shfl_sync(0xffffffffu, cur.n, 8 * u + q + 4 * ks);
                const bool m2 = n2 == n2;   // NaN marks a masked (or padding) pair
                double a3[NT];
#pragma unroll
                for (int mt = 0; mt < NT; ++mt) a3[mt] = cur.g[u][ks][mt][0] + cur.g[u][ks][mt][1];
                const double ns = m2 ? n2 : 0.0, nn = ns * ns;   // masked pair: every basis column is zero
                double b1[NT2], b2[NT2];
#pragma unroll
                for (int nt = 0; nt < NT2; ++nt) {   // branch-free: all reciprocal chains of the k-step in flight
                    const double cn = ck[nt] * ns;
                    const double rd = rcp_ge1(1.0 + cn * cn + 1e-16);
                    b1[nt] = isb[nt] ? (m2 ? rd : 0.0) : c_one[nt] + (m2 ? c_msk[nt] : 0.0);
                    b2[nt] = isb[nt] ? nn * rd * rd : 0.0;
                }
#pragma unroll
                for (int nt = 0; nt < NT2; ++nt)
#pragma unroll
                    for (int mt = 0; mt < NT; ++mt) {
                        dmma(G1[mt][nt][0], G1[mt][nt][1], a3[mt], b1[nt]);
                        dmma(G2[mt][nt][0], G2[mt][nt][1], a3[mt], b2[nt]);
                    }
            }
        }
        cur = nxt;
    }
    // ---- cross-warp reduction (warp after warp: fixed order), then this CTA's row of partials ----
    for (int w = 0; w < nwarps; ++w) {
        if (warp == w) {
#pragma unroll
            for (int mt = 0; mt < NT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT2; ++nt)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        double* d1 = &red[(8 * mt + g) * NK + 8 * nt + 2 * q + e];
                        double* d2 = d1 + NCOL * NK;
                        *d1 = w == 0 ? G1[mt][nt][e] : *d1 + G1[mt][nt][e];
                        *d2 = w == 0 ? G2[mt][nt][e] : *d2 + G2[mt][nt][e];
                    }
        }
        __syncthreads();
    }
    double* row = a.part + (int64_t)blockIdx.x * a.part_stride;
    const double* g1 = red;
    const double* g2 = red + NCOL * NK;
    for (int t = threadIdx.x; t < 4 * C * (K + 1); t += blockDim.x) {
        const int col = t / (K + 1), k = t % (K + 1);
        const int l = (col >> 1) & 1, o = 2 * (col >> 2) + (col & 1);
        if (k < K)
            row[(l ? a.po_w1 : a.po_w0) + (int64_t)o * K + k] = abc_s[KP + k] * g1[col * NK + k] + abc_s[k] * g1[col * NK + K + 1];
        else
            row[(l ? a.po_b1 : a.po_b0) + o] = g1[col * NK + K];
    }
    for (int t = threadIdx.x; t < 3 * K; t += blockDim.x) {
        const int x = t / K, k = t % K;
        double s = 0.0;
        for (int col = 0; col < 4 * C; ++col)
            s += w_s[col * KP + k] * (x == 0 ? g1[col * NK + K + 1] : x == 1 ? g1[col * NK + k] : g2[col * NK + k]);
        if (x == 2) s *= -2.0 * abc_s[KP + k] * abc_s[2 * KP + k];
        row[(x == 0 ? a.po_a : x == 1 ? a.po_b : a.po_c) + k] = s;
    }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
static int pick_ks(int K) { return K <= 12 ? 3 : (K <= 20 ? 5 : (K <= 32 ? 8 : -1)); }

int radial_fwd_grid() { return LGAE_RFWD_CTAS * sm_count(); }
int radial_grid() { return LGAE_RBWD_CTAS * sm_count(); }   // adjoint: CTAs = rows of partials
// doubles per jet of the pair-norm record (unordered pairs padded to whole units)
int64_t radial_nrm_stride(int n) { const int np = n * (n + 1) / 2; return (int64_t)((np + RAD_UNIT - 1) / RAD_UNIT) * RAD_UNIT; }

static void fill(RadialArgs& a, const LgaeModelDesc* d, int level, const double* theta, const double* p4, const uint8_t* node_mask, int batch) {
    memset(&a, 0, sizeof(a));
    a.theta = theta;
    a.off_a = d->off_rad_a[level]; a.off_b = d->off_rad_b[level]; a.off_c = d->off_rad_c[level];
    a.off_w0 = d->off_rad_w0[level]; a.off_b0 = d->off_rad_b0[level];
    a.off_w1 = d->off_rad_w1[level]; a.off_b1 = d->off_rad_b1[level];
    a.p4 = p4; a.node_mask = node_mask;
    a.B = batch; a.N = d->n_particles; a.C = d->channels[level]; a.K = d->n_basis;
}

template <int NT, int KS>
static int launch_radial(const RadialArgs& a, bool bwd, cudaStream_t st) {
    LaunchScope ls_(bwd ? "radial_bwd" : "radial_fwd", st);
    if (bwd)
        launch_k(radial_bwd_kernel<NT, KS>, dim3(radial_grid()), dim3(128), 0, st, a);
    else
        launch_k(radial_fwd_kernel<NT, KS>, dim3(radial_fwd_grid()), dim3(128), 0, st, a);
    return check_launch(bwd ? "radial_bwd" : "radial_fwd");
}

static int dispatch_radial(const RadialArgs& a, bool bwd, cudaStream_t st) {
    if (a.N > RAD_MAXN || a.C < 1 || a.C > LGAE_MAX_CHANNELS) return LGAE_E_UNSUPPORTED;
    const int nt = (4 * a.C + 7) / 8, ks = pick_ks(a.K);
    if (ks < 0) return LGAE_E_UNSUPPORTED;
#define LGAE_CASE(NTV, KSV) \
    if (nt == NTV && ks == KSV) return launch_radial<NTV, KSV>(a, bwd, st);
    LGAE_CASE(1, 3) LGAE_CASE(2, 3) LGAE_CASE(3, 3) LGAE_CASE(4, 3)
    LGAE_CASE(1, 5) LGAE_CASE(2, 5) LGAE_CASE(3, 5) LGAE_CASE(4, 5)
    LGAE_CASE(1, 8) LGAE_CASE(2, 8) LGAE_CASE(3, 8) LGAE_CASE(4, 8)
#undef LGAE_CASE
    return LGAE_E_UNSUPPORTED;
}

// R (B,N,C,32,4) of encoder level `level`.
int run_radial_fwd(const LgaeModelDesc* d, int level, const double* theta, const double* p4, const uint8_t* node_mask, int batch,
                   double* r, double* nrm, cudaStream_t st) {
    if (!d || d->is_decoder || level < 0 || level >= d->n_levels || !r) return LGAE_E_BADARG;
    if (batch <= 0) return LGAE_OK;
    RadialArgs a;
    fill(a, d, level, theta, p4, node_mask, batch);
    a.r = r;
    a.nrm = nrm;
    return dispatch_radial(a, false, st);
}

// R of ALL encoder levels in one launch; needs the same MMA tiling (ceil(4C/8), K) on every level, else LGAE_E_UNSUPPORTED
// (the caller then launches level by level).
int run_radial_fwd_all(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int batch,
                       double* const* r, double* nrm, cudaStream_t st) {
    if (!d || d->is_decoder || !r) return LGAE_E_BADARG;
    if (batch <= 0) return LGAE_OK;
    RadialMultiArgs m;
    int nt = -1;
    for (int l = 0; l < d->n_levels; ++l) {
        fill(m.lv[l], d, l, theta, p4, node_mask, batch);
        m.lv[l].r = r[l];
        m.lv[l].nrm = l == 0 ? nrm : nullptr;
        const int t = (4 * m.lv[l].C + 7) / 8;
        if (nt >= 0 && t != nt) return LGAE_E_UNSUPPORTED;
        nt = t;
        if (m.lv[l].N > RAD_MAXN || m.lv[l].C < 1 || m.lv[l].C > LGAE_MAX_CHANNELS) return LGAE_E_UNSUPPORTED;
    }
    const int ks = pick_ks(d->n_basis);
    if (ks < 0) return LGAE_E_UNSUPPORTED;
    LaunchScope ls_("radial_fwd", st);
#define LGAE_CASE(NTV, KSV) \
    if (nt == NTV && ks == KSV) { launch_k(radial_fwd_multi_kernel<NTV, KSV>, dim3(radial_fwd_grid(), d->n_levels), dim3(128), 0, st, m); return check_launch("radial_fwd"); }
    LGAE_CASE(1, 3) LGAE_CASE(2, 3) LGAE_CASE(3, 3) LGAE_CASE(4, 3)
    LGAE_CASE(1, 5) LGAE_CASE(2, 5) LGAE_CASE(3, 5) LGAE_CASE(4, 5)
    LGAE_CASE(1, 8) LGAE_CASE(2, 8) LGAE_CASE(3, 8) LGAE_CASE(4, 8)
#undef LGAE_CASE
    return LGAE_E_UNSUPPORTED;
}

static int dispatch_radial_bwd_tiled(const RadialArgs& a, cudaStream_t st);
int radial_tiled_grid();

int64_t radial_part_width(const LgaeModelDesc* d, int level) { return (int64_t)4 * d->channels[level] * (d->n_basis + 1) + 3 * d->n_basis; }

// Adjoint: g_r (B,N,C,32,4) -> partial rows for a, b, c, linear.{0,1}.{weight,bias} of the level.  nrm == NULL: any N, g_r in the
// tiled adjoint's blocked layout (B, nib, N, C, 32, 4), the norms recomputed from p4 (radial_bwd_tiled_kernel).
int run_radial_bwd(const LgaeModelDesc* d, int level, const double* theta, const double* p4, const uint8_t* node_mask, int batch,
                   const double* g_r, const double* nrm, PartPlan* plan, cudaStream_t st) {
    if (!d || d->is_decoder || level < 0 || level >= d->n_levels || !g_r || !plan) return LGAE_E_BADARG;
    if (batch <= 0) return LGAE_OK;
    RadialArgs a;
    fill(a, d, level, theta, p4, node_mask, batch);
    a.g_r = g_r;
    a.nrm = const_cast<double*>(nrm);
    const int C = a.C, K = a.K, grid = nrm ? radial_grid() : radial_tiled_grid();
    int64_t w = 0;
    a.po_w0 = w; w += (int64_t)2 * C * K;
    a.po_b0 = w; w += 2 * C;
    a.po_w1 = w; w += (int64_t)2 * C * K;
    a.po_b1 = w; w += 2 * C;
    a.po_a = w; w += K;
    a.po_b = w; w += K;
    a.po_c = w; w += K;
    const int64_t off = plan->block(grid, w);
    a.part = plan->base + off;
    a.part_stride = w;
    int rc = LGAE_OK;
    auto seg = [&](int64_t theta_off, int64_t col, int64_t len) { if (rc == LGAE_OK) rc = plan->seg(theta_off, off, w, col, len, grid); };
    seg(a.off_w0, a.po_w0, (int64_t)2 * C * K); seg(a.off_b0, a.po_b0, 2 * C);
    seg(a.off_w1, a.po_w1, (int64_t)2 * C * K); seg(a.off_b1, a.po_b1, 2 * C);
    seg(a.off_a, a.po_a, K); seg(a.off_b, a.po_b, K); seg(a.off_c, a.po_c, K);
    if (rc != LGAE_OK) return rc;
    return nrm ? dispatch_radial(a, true, st) : dispatch_radial_bwd_tiled(a, st);
}

}  // namespace lgae

// ============================================================================================================
// Adjoint for any N (tiled level adjoint): the math of radial_bwd_kernel, with three differences.  The pair index is decoded
// arithmetically (the unsigned char tables above hold 32 particles), the norms are recomputed from p4 (there is no nrm
// record past 32 particles), and dL/dR is read from the blocked layout (B, nib, N_o, C, 32_i, 4) of level_bwd_nbr_tiled.
// ============================================================================================================
namespace lgae {

// Resident CTAs per SM (register cap 255: at 3, i.e. 168 registers, the wider tilings spill the decoded pair indices).
constexpr int RAD_TILED_CTAS = 2;
int radial_tiled_grid() { return RAD_TILED_CTAS * sm_count(); }   // CTAs = rows of partials

// unordered pair p = j (j + 1) / 2 + i (i <= j) -> (i, j)
LGAE_DEV void pair_decode(int p, int& i, int& j) {
    int t = (int)((__dsqrt_rn(8.0 * p + 1.0) - 1.0) * 0.5);
    while (t * (t + 1) / 2 > p) --t;
    while ((t + 1) * (t + 2) / 2 <= p) ++t;
    j = t;
    i = p - t * (t + 1) / 2;
}

template <int NT>
LGAE_DEV void rad_fetch_tiled(const RadialArgs& a, int unit, int NU, int NP, const int (&col_cc)[NT], const int (&col_x)[NT], int lane,
                              RadOperands<NT>& op) {
    const int N = a.N, C = a.C, q = lane & 3, nib = (N + 31) / 32;
    const int b = unit / NU, p0 = (unit - b * NU) * RAD_UNIT;
    const double* gb = a.g_r + (int64_t)b * nib * N * C * 128;
    const double* pb = a.p4 + (int64_t)b * N * 4;
    {   // norm of pair p0 + (lane & 15) as the forward evaluates it; NaN = masked edge or padding
        const int pid = p0 + (lane & 15);
        double n = __longlong_as_double(0x7ff8000000000000LL);
        if (pid < NP) {
            int i, j;
            pair_decode(pid, i, j);
            const double4 pi = *reinterpret_cast<const double4*>(pb + 4 * i);
            const double4 pj = *reinterpret_cast<const double4*>(pb + 4 * j);
            const double vi[4] = {pi.x, pi.y, pi.z, pi.w}, vj[4] = {pj.x, pj.y, pj.z, pj.w};
            const double nn = rad_pair_norm(vi, vj);
            const bool mi = a.node_mask ? a.node_mask[(int64_t)b * N + i] != 0 : pi.x != 0.0;
            const bool mj = a.node_mask ? a.node_mask[(int64_t)b * N + j] != 0 : pj.x != 0.0;
            if (mi && mj && nn != 0.0) n = nn;
        }
        op.n = n;
    }
    // dL/dR of receiving node r, partner s
    auto at = [&](int r, int s, int cc, int x) { return gb[((((int64_t)(r >> 5) * N + s) * C + cc) * 32 + (r & 31)) * 4 + x]; };
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            const int pid = p0 + 8 * u + q + 4 * ks;
            const bool valid = pid < NP;
            int i = 0, j = 0;
            if (valid) pair_decode(pid, i, j);
#pragma unroll
            for (int mt = 0; mt < NT; ++mt) {
                double v0 = 0.0, v1 = 0.0;
                if (valid && col_cc[mt] >= 0) {
                    v0 = at(i, j, col_cc[mt], col_x[mt]);
                    if (i != j) v1 = at(j, i, col_cc[mt], col_x[mt]);
                }
                op.g[u][ks][mt][0] = v0;
                op.g[u][ks][mt][1] = v1;
            }
        }
}

template <int NT, int KS>
__global__ void __launch_bounds__(128, RAD_TILED_CTAS) radial_bwd_tiled_kernel(const RadialArgs a) {
    constexpr int KP = 4 * KS;
    constexpr int NT2 = KS / 2 + 1;
    constexpr int NK = 8 * NT2, NCOL = 8 * NT;
    __shared__ double abc_s[3 * KP];
    __shared__ double w_s[NCOL * KP];
    __shared__ double red[2 * NCOL * NK];
    const int N = a.N, C = a.C, K = a.K;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    pdl_launch();
    for (int k = threadIdx.x; k < KP; k += blockDim.x) {
        abc_s[k] = k < K ? a.theta[a.off_a + k] : 0.0;
        abc_s[KP + k] = k < K ? a.theta[a.off_b + k] : 0.0;
        abc_s[2 * KP + k] = k < K ? a.theta[a.off_c + k] : 0.0;
    }
    for (int t = threadIdx.x; t < NCOL * KP; t += blockDim.x) w_s[t] = rad_w(a, t / KP, t % KP);
    pdl_wait();
    __syncthreads();
    double G1[NT][NT2][2], G2[NT][NT2][2];
#pragma unroll
    for (int mt = 0; mt < NT; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT2; ++nt) G1[mt][nt][0] = G1[mt][nt][1] = G2[mt][nt][0] = G2[mt][nt][1] = 0.0;
    int col_cc[NT], col_x[NT];
#pragma unroll
    for (int mt = 0; mt < NT; ++mt) {
        const int col = 8 * mt + g;
        col_cc[mt] = col < 4 * C ? (col >> 2) : -1;
        col_x[mt] = col & 3;
    }
    double ck[NT2], c_one[NT2], c_msk[NT2];
    bool isb[NT2];
#pragma unroll
    for (int nt = 0; nt < NT2; ++nt) {
        const int k = 8 * nt + g;
        isb[nt] = k < K;
        ck[nt] = isb[nt] ? abc_s[2 * KP + k] : 0.0;
        c_one[nt] = k == K ? 1.0 : 0.0;
        c_msk[nt] = k == K + 1 ? 1.0 : 0.0;
    }
    const int NP = N * (N + 1) / 2, NU = (NP + RAD_UNIT - 1) / RAD_UNIT;
    const int64_t total = (int64_t)a.B * NU, twarps = (int64_t)gridDim.x * nwarps;
    const int64_t per = (total + twarps - 1) / twarps;
    const int64_t u_begin = ((int64_t)blockIdx.x * nwarps + warp) * per, u_end = u_begin + per < total ? u_begin + per : total;
    RadOperands<NT> cur, nxt;
    if (u_begin < u_end) rad_fetch_tiled<NT>(a, (int)u_begin, NU, NP, col_cc, col_x, lane, cur);
    for (int64_t unit = u_begin; unit < u_end; ++unit) {
        if (unit + 1 < u_end) rad_fetch_tiled<NT>(a, (int)(unit + 1), NU, NP, col_cc, col_x, lane, nxt);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                const double n2 = __shfl_sync(0xffffffffu, cur.n, 8 * u + q + 4 * ks);
                const bool m2 = n2 == n2;
                double a3[NT];
#pragma unroll
                for (int mt = 0; mt < NT; ++mt) a3[mt] = cur.g[u][ks][mt][0] + cur.g[u][ks][mt][1];
                const double ns = m2 ? n2 : 0.0, nn = ns * ns;
                double b1[NT2], b2[NT2];
#pragma unroll
                for (int nt = 0; nt < NT2; ++nt) {
                    const double cn = ck[nt] * ns;
                    const double rd = rcp_ge1(1.0 + cn * cn + 1e-16);
                    b1[nt] = isb[nt] ? (m2 ? rd : 0.0) : c_one[nt] + (m2 ? c_msk[nt] : 0.0);
                    b2[nt] = isb[nt] ? nn * rd * rd : 0.0;
                }
#pragma unroll
                for (int nt = 0; nt < NT2; ++nt)
#pragma unroll
                    for (int mt = 0; mt < NT; ++mt) {
                        dmma(G1[mt][nt][0], G1[mt][nt][1], a3[mt], b1[nt]);
                        dmma(G2[mt][nt][0], G2[mt][nt][1], a3[mt], b2[nt]);
                    }
            }
        }
        cur = nxt;
    }
    for (int w = 0; w < nwarps; ++w) {
        if (warp == w) {
#pragma unroll
            for (int mt = 0; mt < NT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT2; ++nt)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        double* d1 = &red[(8 * mt + g) * NK + 8 * nt + 2 * q + e];
                        double* d2 = d1 + NCOL * NK;
                        *d1 = w == 0 ? G1[mt][nt][e] : *d1 + G1[mt][nt][e];
                        *d2 = w == 0 ? G2[mt][nt][e] : *d2 + G2[mt][nt][e];
                    }
        }
        __syncthreads();
    }
    double* row = a.part + (int64_t)blockIdx.x * a.part_stride;
    const double* g1 = red;
    const double* g2 = red + NCOL * NK;
    for (int t = threadIdx.x; t < 4 * C * (K + 1); t += blockDim.x) {
        const int col = t / (K + 1), k = t % (K + 1);
        const int l = (col >> 1) & 1, o = 2 * (col >> 2) + (col & 1);
        if (k < K)
            row[(l ? a.po_w1 : a.po_w0) + (int64_t)o * K + k] = abc_s[KP + k] * g1[col * NK + k] + abc_s[k] * g1[col * NK + K + 1];
        else
            row[(l ? a.po_b1 : a.po_b0) + o] = g1[col * NK + K];
    }
    for (int t = threadIdx.x; t < 3 * K; t += blockDim.x) {
        const int x = t / K, k = t % K;
        double s = 0.0;
        for (int col = 0; col < 4 * C; ++col)
            s += w_s[col * KP + k] * (x == 0 ? g1[col * NK + K + 1] : x == 1 ? g1[col * NK + k] : g2[col * NK + k]);
        if (x == 2) s *= -2.0 * abc_s[KP + k] * abc_s[2 * KP + k];
        row[(x == 0 ? a.po_a : x == 1 ? a.po_b : a.po_c) + k] = s;
    }
}

static int dispatch_radial_bwd_tiled(const RadialArgs& a, cudaStream_t st) {
    if (a.C < 1 || a.C > LGAE_MAX_CHANNELS) return LGAE_E_UNSUPPORTED;
    const int nt = (4 * a.C + 7) / 8, ks = pick_ks(a.K);
    if (ks < 0) return LGAE_E_UNSUPPORTED;
    LaunchScope ls_("radial_bwd_tiled", st);
#define LGAE_CASE(NTV, KSV)                                                                                   \
    if (nt == NTV && ks == KSV) {                                                                             \
        launch_k(radial_bwd_tiled_kernel<NTV, KSV>, dim3(radial_tiled_grid()), dim3(128), 0, st, a);                \
        return check_launch("radial_bwd_tiled");                                                              \
    }
    LGAE_CASE(1, 3) LGAE_CASE(2, 3) LGAE_CASE(3, 3) LGAE_CASE(4, 3)
    LGAE_CASE(1, 5) LGAE_CASE(2, 5) LGAE_CASE(3, 5) LGAE_CASE(4, 5)
    LGAE_CASE(1, 8) LGAE_CASE(2, 8) LGAE_CASE(3, 8) LGAE_CASE(4, 8)
#undef LGAE_CASE
    return LGAE_E_UNSUPPORTED;
}

}  // namespace lgae
