// One LGN message-passing level at maxdim 2, fused per jet (SURVEY.md appendix A.2b):
//   radial functions -> edge features -> CG aggregation over the fully connected graph -> CG self product ->
//   concat [ag | node | sq] -> per-irrep complex channel mix,
// forward and hand-written adjoint.  Replaces LGNNodeLevel.forward (lgn/models/lgn_levels.py:96-121) and what
// it calls: cg_product / complex_kron_product (lgn/cg_lib/cg_ops.py:135-298), CatMixReps (lgn/nn/g_nn.py:260-278),
// RadPolyTrig.forward (lgn/nn/position_levels.py:118-209), the edge-feature product (lgn/models/lgn_cg.py:167)
// and the pairwise zonal functions / norms (lgn/cg_lib/zonal_functions.py:123-248).
//
// Thread mapping: lane = particle i (one warp covers a block of 32 particles), warp = channel c.  The radial
// weights R^l_ij[c] = Linear_l(phi(n_ij)) of a tile of neighbours j are produced with the fp64 tensor-core
// MMA (phi (pairs x K) times W^T (K x 4C)) into shared memory and consumed by the (i, c) threads; the neighbour
// sums stay in registers.  The only O(N^2) tensor that goes to HBM is the optional copy of the radial weights
// R_ij[c] (r_save) that the training forward keeps for the adjoint, which then does not re-evaluate them.
#include <cstring>

#include "lgae_common.cuh"

namespace lgae {

struct LevelArgs {
    const double* theta;
    int64_t off_a, off_b, off_c, off_w0, off_b0, off_w1, off_b1, off_m00, off_m11;
    const double* p;           // encoder: (B,N,4) real Cartesian ; decoder: (B,N,4,2) complex canonical
    const uint8_t* node_mask;  // encoder: (B,N) or nullptr
    const double* s_in;        // (B,N,C,2)
    const double* v_in;        // (B,N,C,4,2)
    double* sums;              // (B,N,C,10,2)   [A0V(4), A0S, A1Y(4), A1E]
    double* s_pre;             // (B,N,C',2)
    double* v_out;             // (B,N,C',4,2)
    double* r_save;            // encoder, N <= 32: (B,N_j,C,32_i,4) radial weights (R0.re, R0.im, R1.re, R1.im), produced by
                               // radial_fwd_kernel (lgae_radial.cu); input of the PRE forward and of the adjoint
    double* g_r;               // encoder adjoint out: dL/dR of the ordered pairs, same layout as r_save
    // backward only
    const double* g_s_pre;
    const double* g_v_out;
    double* g_s_in;
    double* g_v_in;
    double* g_y;               // decoder: (B,N,4,2), accumulated
    double* part;              // (gridDim.x, part_stride) per-CTA rows of parameter-gradient partials
    int64_t part_stride;
    int64_t po_w0, po_b0, po_w1, po_b1, po_a, po_b, po_c, po_m00, po_m11;   // column offsets inside a row
    int B, N, C, Cout, K;
};

#ifndef LGAE_BWD_UNROLL
#define LGAE_BWD_UNROLL 1   // unroll factor of the adjoint neighbour loop
#endif
#ifndef LGAE_FWD_UNROLL
#define LGAE_FWD_UNROLL 1   // ... and of the forward one
#endif
#ifndef LGAE_RPD_FWD
#define LGAE_RPD_FWD 2   // partners of radial weights in flight per thread in the forward neighbour loop
#endif
#ifndef LGAE_RPD_BWD
#define LGAE_RPD_BWD 2   // ... and in the adjoint
#endif
#ifndef LGAE_LBWD_CF_MINB
#define LGAE_LBWD_CF_MINB 3   // the same for the decoder's closed-form adjoint
#endif
#ifndef LGAE_LBWD_MINB_C4
#define LGAE_LBWD_MINB_C4 3   // same, launches with 4 channels (128 threads): 3 CTAs/SM = 444 slots < 512 jets, 4 => one wave but 128 registers
#endif
#ifndef LGAE_LBWD_CF_MINB_C4
#define LGAE_LBWD_CF_MINB_C4 3   // 4 = 128 registers (228 B of spills), one wave for 512 jets: 40.3 vs 40.5 us alone, but the step is 6 us slower
#endif
#ifndef LGAE_LBWD_MINB
#define LGAE_LBWD_MINB 3   // resident CTAs per SM the level adjoint is compiled for (register cap 168; 4 => 128 registers spills and is slower)
#endif
#ifndef LGAE_FWD_RING
#define LGAE_FWD_RING 1   // forward (PRE): radial weights arrive through a shared-memory ring of TMA bulk copies instead of per-thread loads
#endif
#ifndef LGAE_RING_PS
#define LGAE_RING_PS 3    // partners per ring stage
#endif
constexpr int kBwdUnroll = LGAE_BWD_UNROLL, kFwdUnroll = LGAE_FWD_UNROLL;
constexpr int kRingPS = LGAE_RING_PS, kRingMaxStages = 4;
#ifndef LGAE_TJ
#define LGAE_TJ 8   // with the component-wise mix and tile-wise partner features a 150-particle jet needs 43 KB per CTA (4: 8.74 vs 8.48 ms per 1024 jets)
#endif
constexpr int TJ = LGAE_TJ;  // neighbours per shared-memory tile of radial weights
constexpr int CAT_E = 21;  // entries per (channel, particle) of the concatenation staged for the channel mix

// Pair norm n_ij = s / sqrt|s|, s = (p_i - p_j)^2 + 1e-16, with the reference's rounding sequence
// (zonal_functions.py:142-144, 201-248).
LGAE_DEV double pair_norm(const double* pi, const double* pj) {
    const double d0 = pi[0] - pj[0], d1 = pi[1] - pj[1], d2 = pi[2] - pj[2], d3 = pi[3] - pj[3];
    const double s = __dadd_rn(minkowski_sq(d0, d1, d2, d3), 1e-16);
    return s != 0.0 ? __ddiv_rn(s, __dsqrt_rn(fabs(s))) : s;
}

LGAE_DEV double bell(double a, double b, double c, double n) {
    const double cn = c * n;
    const double d = 1.0 + cn * cn + 1e-16;
    return fma(b, 1.0 / d, a);
}

// Column `col` of the stacked radial linear maps: col = l*2C + 2c + (re|im)  (position_levels.py:171-176)
LGAE_DEV double radial_w(const LevelArgs& a, int col, int k) {
    if (k >= a.K || col >= 4 * a.C) return 0.0;
    return col < 2 * a.C ? a.theta[a.off_w0 + (int64_t)col * a.K + k] : a.theta[a.off_w1 + (int64_t)(col - 2 * a.C) * a.K + k];
}
LGAE_DEV double radial_bias(const LevelArgs& a, int col) {
    if (col >= 4 * a.C) return 0.0;
    return col < 2 * a.C ? a.theta[a.off_b0 + col] : a.theta[a.off_b1 + col - 2 * a.C];
}

// Radial weights of the pairs (i in block i0..i0+31, j in j0..j0+tj-1) -> Rs[((jj*C + c)*32 + il)*4 + 2l + ri].
template <int NT, int KS>
LGAE_DEV void radial_tile(const double* p_s, const uint8_t* msk_s, int N, int C, int i0, int j0, int tj,
                          const double* abc_s, const double (&wf)[KS][NT], const double (&bf)[NT][2], double* Rs) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    constexpr int KP = 4 * KS;
    for (int grp = warp; grp < 4 * tj; grp += nwarps) {
        const int jj = grp >> 2, il = (grp & 3) * 8 + g, i = i0 + il, j = j0 + jj;
        double n = 0.0;
        bool m = false;
        if (i < N) {
            n = pair_norm(p_s + 4 * i, p_s + 4 * j);
            m = msk_s[i] && msk_s[j] && n != 0.0;
        }
        double acc[NT][2];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) { acc[nt][0] = bf[nt][0]; acc[nt][1] = bf[nt][1]; }
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            const int k = 4 * s + q;
            const double phi = m ? bell(abc_s[k], abc_s[KP + k], abc_s[2 * KP + k], n) : 0.0;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) dmma(acc[nt][0], acc[nt][1], phi, wf[s][nt]);
        }
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            const int col = 8 * nt + 2 * q;
            if (col < 4 * C) {
                const int l = col >= 2 * C ? 1 : 0;
                const int cc = (col - l * 2 * C) >> 1;
                *reinterpret_cast<double2*>(Rs + ((size_t)((jj * C + cc) * 32 + il)) * 4 + 2 * l) = make_double2(acc[nt][0], acc[nt][1]);
            }
        }
    }
}

template <int NT, int KS>
LGAE_DEV void load_radial_frags(const LevelArgs& a, double (&wf)[KS][NT], double (&bf)[NT][2], double* abc_s) {
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
    constexpr int KP = 4 * KS;
#pragma unroll
    for (int s = 0; s < KS; ++s)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) wf[s][nt] = radial_w(a, 8 * nt + g, 4 * s + q);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        bf[nt][0] = radial_bias(a, 8 * nt + 2 * q);
        bf[nt][1] = radial_bias(a, 8 * nt + 2 * q + 1);
    }
    for (int k = threadIdx.x; k < KP; k += blockDim.x) {
        abc_s[k] = k < a.K ? a.theta[a.off_a + k] : 0.0;
        abc_s[KP + k] = k < a.K ? a.theta[a.off_b + k] : 0.0;
        abc_s[2 * KP + k] = k < a.K ? a.theta[a.off_c + k] : 0.0;
    }
}

// Shared-memory carve-up (in doubles) of the forward kernel.
struct LevelSmem {
    int p, msk, S, V, abc, m00, m11, big;  // offsets
    int total;
};
__host__ __device__ inline LevelSmem level_smem(bool enc, bool tiles, int N, int C, int Cout, int KS) {
    LevelSmem s;
    int o = 0;
    s.p = o; o += enc ? 4 * N : 8 * N;
    s.msk = o; o += ((N + 7) / 8 + 2) & ~1;
    // node features: the whole jet, or (radial weights evaluated in the kernel) only the partners of the current tile -- the
    // 10 N C doubles of a long jet would otherwise decide how many CTAs fit on an SM
    s.S = o; o += 2 * (tiles ? TJ : N) * C;
    s.V = o; o += 8 * (tiles ? TJ : N) * C;
    s.abc = o; o += (3 * 4 * KS + 1) & ~1;
    s.m00 = o; o += 2 * Cout * 5 * C;
    s.m11 = o; o += 2 * Cout * 5 * C;
    o = (o + 3) & ~3;
    s.big = o;
    // cat: [(c*21+e)][min(N,32)] complex; jets of more than 32 particles (several CTAs per jet, shared memory is what limits
    // their occupancy) mix component by component through a [(c*5+j)][32] buffer instead
    const int cat = N > 32 ? 2 * 5 * C * 32 : 2 * CAT_E * C * (N < 32 ? N : 32);
    const int tile = tiles ? TJ * C * 32 * 4 : 0;   // Rs (radial weights evaluated in the kernel)
    o += cat > tile ? cat : tile;
    s.total = o;
    return s;
}

// ------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------
// PRE (encoder, N <= 32): the radial weights were computed by radial_fwd_kernel and are streamed from r_save (one
// double4 per partner, prefetched one partner ahead); no radial tiles, no barriers inside the neighbour loop.
// The decoder is launched as <false, 1, 3, true> and takes the O(N) closed form.
template <bool ENC, int NT, int KS, bool PRE>
__global__ void __launch_bounds__(256) level_fwd_kernel(const LevelArgs a) {
    extern __shared__ __align__(128) double smem[];
    const int N = a.N, C = a.C, Cout = a.Cout;
    const int nib = (N + 31) / 32;
    const int b = blockIdx.x / nib, i0 = (blockIdx.x % nib) * 32;
    const int tid = threadIdx.x, lane = tid & 31, c = tid >> 5;
    const LevelSmem L = level_smem(ENC, ENC && !PRE, N, C, Cout, KS);
    double* p_s = smem + L.p;
    uint8_t* msk_s = reinterpret_cast<uint8_t*>(smem + L.msk);
    cplx* S_s = reinterpret_cast<cplx*>(smem + L.S);
    cplx* V_s = reinterpret_cast<cplx*>(smem + L.V);
    double* abc_s = smem + L.abc;
    cplx* m00_s = reinterpret_cast<cplx*>(smem + L.m00);
    cplx* m11_s = reinterpret_cast<cplx*>(smem + L.m11);
    double* Rs = smem + L.big;
    cplx* cat_s = reinterpret_cast<cplx*>(smem + L.big);
    const int NS = N < 32 ? N : 32;   // particle stride of cat_s

    // ---- stage the jet: momenta and node features by TMA bulk copies, weights by the threads meanwhile ----
    pdl_launch();
    __shared__ uint64_t mbar;
    __shared__ uint64_t rbar[kRingMaxStages];
    // PRE: the radial weights of this jet, (N_j, C, 32, 4) = pd doubles per partner, stream through a ring of `nst` stages of
    // kRingPS partners in the (still dead) cat buffer: one TMA bulk copy per stage, issued nst stages ahead of their use
    const int pd = C * 128;
    const int nst = (ENC && PRE && LGAE_FWD_RING) ? min((2 * CAT_E * C * NS) / pd / kRingPS, kRingMaxStages) : 0;
    const bool ring = nst >= 2;
    const int ngr = (N + kRingPS - 1) / kRingPS;
    auto ring_issue = [&](int g) {   // one thread
        const int s = g % nst, j0 = g * kRingPS, tj = min(kRingPS, N - j0);
        const unsigned bytes = (unsigned)(tj * pd * sizeof(double));
        mbar_expect_tx(&rbar[s], bytes);
        bulk_g2s(Rs + (size_t)s * kRingPS * pd, a.r_save + ((int64_t)b * N + j0) * pd, bytes, &rbar[s]);
    };
    if (tid == 0) {
        mbar_init(&mbar, 1);
        for (int s = 0; s < kRingMaxStages; ++s) mbar_init(&rbar[s], 1);
    }
    pdl_wait();   // everything below reads what earlier kernels of the step produced
    __syncthreads();
    {
        const int np = ENC ? 4 * N : 8 * N;
        const double* src = a.p + (int64_t)b * np;
        if (tid == 0) {
            constexpr bool kTiles = ENC && !PRE;   // node features of the partners arrive tile by tile
            mbar_expect_tx(&mbar, (unsigned)((np + (kTiles ? 0 : 10 * N * C)) * sizeof(double)));
            bulk_g2s(p_s, src, np * sizeof(double), &mbar);
            if (!kTiles) {
                bulk_g2s(smem + L.S, a.s_in + (int64_t)b * N * C * 2, 2 * N * C * sizeof(double), &mbar);
                bulk_g2s(smem + L.V, a.v_in + (int64_t)b * N * C * 8, 8 * N * C * sizeof(double), &mbar);
            }
            if (ring)
                for (int g = 0; g < nst && g < ngr; ++g) ring_issue(g);
        }
        if (ENC && !PRE)
            for (int t = tid; t < N; t += blockDim.x)
                msk_s[t] = a.node_mask ? a.node_mask[(int64_t)b * N + t] : (src[4 * t] != 0.0);
        const int nm = Cout * 5 * C;
        for (int t = tid; t < nm; t += blockDim.x) {
            m00_s[t] = cmake(a.theta[a.off_m00 + t], a.theta[a.off_m00 + nm + t]);
            m11_s[t] = cmake(a.theta[a.off_m11 + t], a.theta[a.off_m11 + nm + t]);
        }
    }
    double wf[KS][NT], bf[NT][2];
    cplx R0c = czero(), R1c = czero();
    if (ENC) {
        if (!PRE) load_radial_frags<NT, KS>(a, wf, bf, abc_s);
    } else {
        // decoder: all-zero edge mask => R^l[c] = bias_l[c] * (1+i)   (SURVEY.md appendix A.6)
        const double b0 = a.theta[a.off_b0 + c], b1 = a.theta[a.off_b1 + c];
        R0c = cmake(b0, b0);
        R1c = cmake(b1, b1);
    }
    mbar_wait(&mbar, 0);
    __syncthreads();

    const int i = i0 + lane;
    const bool live = i < N;
    double pi[4] = {0, 0, 0, 0};
    cplx yi[4] = {czero(), czero(), czero(), czero()};
    if (live) {
        if (ENC) {
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) pi[mu] = p_s[4 * i + mu];
        } else {
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) yi[mu] = reinterpret_cast<const cplx*>(p_s)[4 * i + mu];
        }
    }
    cplx A0V[4], A0S = czero(), A1Y[4], A1E = czero();
#pragma unroll
    for (int mu = 0; mu < 4; ++mu) { A0V[mu] = czero(); A1Y[mu] = czero(); }

    if (!ENC && PRE) {
        // Decoder, closed form (SURVEY.md appendix A.6): the radial weights are the constants R^l[c] = bias_l[c] (1+i), so
        // the neighbour sums factor through four jet-level moments of the node features, O(N) instead of O(N^2):
        //   SS = sum_j S_j   SV = sum_j V_j   SSY = sum_j S_j y_j   SVY = sum_j eta(V_j, y_j)
        //   A0V_i = R0 SV   A0S_i = R0 SS   A1Y_i = R1 (y_i SS - SSY)   A1E_i = R1 (eta(SV, y_i) - SVY)
        const cplx* y_s = reinterpret_cast<const cplx*>(p_s);
        double m[20];
#pragma unroll
        for (int t = 0; t < 20; ++t) m[t] = 0.0;
        for (int j = lane; j < N; j += 32) {
            const cplx Sj = S_s[j * C + c];
            cplx Vj[4], yj[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) { Vj[mu] = V_s[(j * C + c) * 4 + mu]; yj[mu] = y_s[4 * j + mu]; }
            m[0] += Sj.x; m[1] += Sj.y;
            const cplx e = ceta(Vj, yj);
            m[18] += e.x; m[19] += e.y;
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                m[2 + 2 * mu] += Vj[mu].x; m[3 + 2 * mu] += Vj[mu].y;
                const cplx sy = cmul(Sj, yj[mu]);
                m[10 + 2 * mu] += sy.x; m[11 + 2 * mu] += sy.y;
            }
        }
        warp_allsum_n<20>(m);
        const cplx SS = cmake(m[0], m[1]), SVY = cmake(m[18], m[19]);
        cplx SV[4], SSY[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) { SV[mu] = cmake(m[2 + 2 * mu], m[3 + 2 * mu]); SSY[mu] = cmake(m[10 + 2 * mu], m[11 + 2 * mu]); }
        A0S = cmul(R0c, SS);
        A1E = cmul(R1c, csub(ceta(SV, yi), SVY));
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) {
            A0V[mu] = cmul(R0c, SV[mu]);
            A1Y[mu] = cmul(R1c, csub(cmul(yi[mu], SS), SSY[mu]));
        }
    } else {
    // encoder: one neighbour j with its radial weights: the four neighbour sums of this (particle, channel)
    auto pair = [&](int j, int js, cplx R0, cplx R1) {   // js: where partner j's features lie in S_s / V_s
        const cplx Sj = S_s[js * C + c];
        cplx Vj[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) Vj[mu] = V_s[(js * C + c) * 4 + mu];
        cplx Y[4];
        double d[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) d[mu] = pi[mu] - p_s[4 * j + mu];
        canon_from_real(d, Y);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) cfma(A0V[mu], R0, Vj[mu]);
        cfma(A0S, R0, Sj);
        const cplx t = cmul(R1, Sj);
        // Y0, Y2 are real, Y3 = -conj... structured: saves a third of the multiplies
        cfmar(A1Y[0], t, Y[0].x);
        cfma(A1Y[1], t, Y[1]);
        cfmar(A1Y[2], t, Y[2].x);
        cfma(A1Y[3], t, Y[3]);
        cplx e = cscale(Vj[0], Y[0].x);
        cfma(e, Vj[1], Y[3]);
        cfmar(e, Vj[2], -Y[2].x);
        cfma(e, Vj[3], Y[1]);
        cfma(A1E, R1, e);
    };
    if (ring) {
        for (int g = 0; g < ngr; ++g) {
            const int s = g % nst, j0 = g * kRingPS, tj = min(kRingPS, N - j0);
            mbar_wait(&rbar[s], (unsigned)((g / nst) & 1));
            const double* rs = Rs + (size_t)s * kRingPS * pd + (c * 32 + lane) * 4;
#pragma unroll
            for (int jj = 0; jj < kRingPS; ++jj) {
                if (jj < tj) {
                    const double4 r = *reinterpret_cast<const double4*>(rs + (size_t)jj * pd);
                    pair(j0 + jj, j0 + jj, cmake(r.x, r.y), cmake(r.z, r.w));
                }
            }
            if (g + nst < ngr) {   // every warp is done with stage s: refill it
                __syncthreads();
                if (tid == 0) ring_issue(g + nst);
            }
        }
    } else {
    const double4* rsv = reinterpret_cast<const double4*>(a.r_save) + ((int64_t)b * N * C + c) * 32 + lane;
    constexpr int PDF = LGAE_RPD_FWD;
    double4 rq[PDF];
#pragma unroll
    for (int d = 0; d < PDF; ++d) {
        rq[d] = make_double4(0.0, 0.0, 0.0, 0.0);
        if (PRE && d < N) rq[d] = rsv[(int64_t)d * C * 32];
    }
    for (int j0 = 0; j0 < N; j0 += TJ) {
        const int tj = min(TJ, N - j0);
        if (!PRE) {
            // the tile's partner features: global loads in flight during the radial tile, then into shared memory
            constexpr int NPF = (TJ * 5 + 31) / 32;
            cplx pf[NPF];
            const int nsv = tj * C * 5;
            const cplx* sg = reinterpret_cast<const cplx*>(a.s_in) + ((int64_t)b * N + j0) * C;
            const cplx* vg = reinterpret_cast<const cplx*>(a.v_in) + ((int64_t)b * N + j0) * C * 4;
#pragma unroll
            for (int k = 0; k < NPF; ++k) {
                const int t = tid + k * blockDim.x;
                pf[k] = czero();
                if (t < nsv) pf[k] = t < tj * C ? sg[t] : vg[t - tj * C];
            }
            radial_tile<NT, KS>(p_s, msk_s, N, C, i0, j0, tj, abc_s, wf, bf, Rs);
#pragma unroll
            for (int k = 0; k < NPF; ++k) {
                const int t = tid + k * blockDim.x;
                if (t < nsv) { if (t < tj * C) S_s[t] = pf[k]; else V_s[t - tj * C] = pf[k]; }
            }
            __syncthreads();
        }
#pragma unroll kFwdUnroll
        for (int jj = 0; jj < tj; ++jj) {
            const int j = j0 + jj;
            cplx R0 = czero(), R1 = czero();
            if (PRE) {
                R0 = cmake(rq[0].x, rq[0].y);
                R1 = cmake(rq[0].z, rq[0].w);
#pragma unroll
                for (int d = 0; d + 1 < PDF; ++d) rq[d] = rq[d + 1];
                if (j + PDF < N) rq[PDF - 1] = rsv[(int64_t)(j + PDF) * C * 32];
            } else {
                const double4 r = *reinterpret_cast<const double4*>(Rs + ((size_t)((jj * C + c) * 32 + lane)) * 4);
                R0 = cmake(r.x, r.y);
                R1 = cmake(r.z, r.w);
            }
            pair(j, PRE ? j : jj, R0, R1);
        }
        if (!PRE) __syncthreads();
    }
    }
    }

    // ---- keep the neighbour sums for the backward pass; build cat = [ag | node | sq] in shared memory ----
    __syncthreads();  // Rs is dead, cat_s aliases it
    if (live) {
        cplx* dst = reinterpret_cast<cplx*>(a.sums) + ((int64_t)(b * N + i) * C + c) * 10;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) { dst[mu] = A0V[mu]; dst[5 + mu] = A1Y[mu]; }
        dst[4] = A0S;
        dst[9] = A1E;
    }
    cplx Si = czero(), Vi[4] = {czero(), czero(), czero(), czero()};
    if (live) {
        if (ENC && !PRE) {   // only the current tile's partners are in shared memory
            Si = reinterpret_cast<const cplx*>(a.s_in)[((int64_t)b * N + i) * C + c];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) Vi[mu] = reinterpret_cast<const cplx*>(a.v_in)[(((int64_t)b * N + i) * C + c) * 4 + mu];
        } else {
            Si = S_s[i * C + c];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) Vi[mu] = V_s[(i * C + c) * 4 + mu];
        }
    }
    if (N > 32) {
        // ---- component by component: the 5 (0,0) entries, then the 4 entries of each (1,1) component, through a small buffer
        // (same entries, weights and summation order as the one-shot form below) ----
#pragma unroll
        for (int comp = 0; comp < 5; ++comp) {
            if (comp) __syncthreads();   // the previous component's entries are consumed
            if (comp == 0) {
                cat_s[(c * 5 + 0) * 32 + lane] = cscale(A1E, 0.5);
                cat_s[(c * 5 + 1) * 32 + lane] = cmul_1pi(A0S);
                cat_s[(c * 5 + 2) * 32 + lane] = Si;
                cat_s[(c * 5 + 3) * 32 + lane] = cscale(ceta(Vi, Vi), 0.5);
                cat_s[(c * 5 + 4) * 32 + lane] = cmul(Si, Si);
            } else {
                const int mu = comp > 0 ? comp - 1 : 0;   // compile-time after unrolling
                const cplx a0 = A0V[mu], a1 = A1Y[mu], vi = Vi[mu];
                cat_s[(c * 5 + 0) * 32 + lane] = cmul_1pi(a0);
                cat_s[(c * 5 + 1) * 32 + lane] = a1;
                cat_s[(c * 5 + 2) * 32 + lane] = vi;
                cat_s[(c * 5 + 3) * 32 + lane] = cmul(vi, Si);
            }
            __syncthreads();
            for (int it = tid; it < 32 * Cout; it += blockDim.x) {
                const int il = it & 31, co = it >> 5, ii = i0 + il;
                if (ii >= N) continue;
                cplx acc = czero();
                if (comp == 0) {
                    const cplx* w = m00_s + co * 5 * C;
                    for (int cc = 0; cc < C; ++cc)
#pragma unroll
                        for (int j = 0; j < 5; ++j) cfma(acc, w[j * C + cc], cat_s[(cc * 5 + j) * 32 + il]);
                    reinterpret_cast<cplx*>(a.s_pre)[(int64_t)(b * N + ii) * Cout + co] = acc;
                } else {
                    const cplx* w = m11_s + co * 5 * C;
                    for (int cc = 0; cc < C; ++cc) {
#pragma unroll
                        for (int j = 0; j < 3; ++j) cfma(acc, w[j * C + cc], cat_s[(cc * 5 + j) * 32 + il]);
                        cfma(acc, cadd(w[3 * C + cc], w[4 * C + cc]), cat_s[(cc * 5 + 3) * 32 + il]);
                    }
                    reinterpret_cast<cplx*>(a.v_out)[((int64_t)(b * N + ii) * Cout + co) * 4 + comp - 1] = acc;
                }
            }
                    }
        return;
    }
    {
        // 21 entries per (channel, particle): the five (0,0) blocks [ag_a, ag_b, node, sq_a, sq_b], then the (1,1) components
        // of [ag_a, ag_b, node, sq]; the two self-product blocks share their (1,1) part V S, so it is stored once and
        // mixed with the sum of their weights.
        auto put = [&](int e, cplx v) { cat_s[(c * CAT_E + e) * NS + lane] = v; };
        if (lane < NS) {
            put(0, cscale(A1E, 0.5));
            put(1, cmul_1pi(A0S));
            put(2, Si);
            put(3, cscale(ceta(Vi, Vi), 0.5));
            put(4, cmul(Si, Si));
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                put(5 + mu, cmul_1pi(A0V[mu]));
                put(9 + mu, A1Y[mu]);
                put(13 + mu, Vi[mu]);
                put(17 + mu, cmul(Vi[mu], Si));
            }
        }
    }
    __syncthreads();
    // ---- complex channel mix (lgn/nn/g_nn.py:95-117): out[c'] = sum_k W[c'][k] cat[k] ----
    for (int it = tid; it < 32 * Cout * 5; it += blockDim.x) {
        const int il = it & 31, r = it >> 5, co = r / 5, comp = r % 5;
        const int ii = i0 + il;
        if (ii >= N) continue;
        cplx acc = czero();
        if (comp == 0) {
            const cplx* w = m00_s + co * 5 * C;
            for (int cc = 0; cc < C; ++cc)
#pragma unroll
                for (int j = 0; j < 5; ++j) cfma(acc, w[j * C + cc], cat_s[(cc * CAT_E + j) * NS + il]);
            reinterpret_cast<cplx*>(a.s_pre)[(int64_t)(b * N + ii) * Cout + co] = acc;
        } else {
            const cplx* w = m11_s + co * 5 * C;
            for (int cc = 0; cc < C; ++cc) {
#pragma unroll
                for (int j = 0; j < 3; ++j) cfma(acc, w[j * C + cc], cat_s[(cc * CAT_E + 5 + 4 * j + comp - 1) * NS + il]);
                cfma(acc, cadd(w[3 * C + cc], w[4 * C + cc]), cat_s[(cc * CAT_E + 17 + comp - 1) * NS + il]);
            }
            reinterpret_cast<cplx*>(a.v_out)[((int64_t)(b * N + ii) * Cout + co) * 4 + comp - 1] = acc;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------------------
// Shared-memory carve-up (in doubles) of the backward kernel.
struct LevelBwdSmem {
    int p, S, V, m00, m11, gm, gA, gy, gout, graw;
    int total;
};
__host__ __device__ inline LevelBwdSmem level_bwd_smem(bool enc, int N, int C, int Cout) {
    LevelBwdSmem s;
    int o = 0;
    s.p = o; o += enc ? 4 * N : 8 * N;
    s.S = o; o += 2 * N * C;
    s.V = o; o += 8 * N * C;
    s.m00 = o; o += 2 * Cout * 5 * C;
    s.m11 = o; o += 2 * Cout * 5 * C;
    s.gm = o; o += 2 * 2 * Cout * 5 * C;     // [irrep][c'][k] complex accumulators, live for the whole CTA
    s.gA = o; o += 2 * C * 10 * 32;          // [(c*10+e)][32] complex: adjoints of the neighbour sums
    o = (o + 3) & ~3;
    s.gout = o; o += 2 * Cout * 5 * 32;      // incoming gradients [(c'*5+comp)][32] complex
    s.graw = o; o += 2 * N * Cout * 5;       // the same as they lie in HBM: g_s_pre (N,C') | g_v_out (N,C',4), bulk-copied
    // decoder: per-channel dL/dy, summed over channels in a fixed order; written after the neighbour loop, when the two gradient
    // buffers are dead, so it lies on top of them
    s.gy = s.gout;
    const int gy = enc ? 0 : 2 * 4 * 32 * C;
    if (o - s.gout < gy) o = s.gout + gy;
    s.total = o;
    return s;
}

// Adjoint of "cat -> mix" for one block of the concatenation (k = blk*C + c), thread = (particle lane, channel c):
//   gm[irrep][c'][k] += sum_lanes conj(cat[comp]) gout[c'][comp]      (mix-weight gradient; lgn/nn/g_nn.py:95-117)
//   gc[comp]          = sum_c'   conj(W[c'][k])  gout[c'][comp]       (gradient wrt this thread's cat entries)
LGAE_DEV void mix_adjoint_block(int k, int Cout, int C5, int nm, int lane, const cplx (&cat5)[5], const cplx* gout_s,
                                const cplx* m00_s, const cplx* m11_s, double* gm_d, cplx (&gc)[5]) {
#pragma unroll
    for (int comp = 0; comp < 5; ++comp) gc[comp] = czero();
    for (int cb = 0; cb < Cout; cb += 4) {
        double v[16];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int co = cb + u;
            cplx a0 = czero(), a1 = czero();
            if (co < Cout) {
                const cplx* gp = gout_s + (co * 5) * 32 + lane;
                const cplx g0 = gp[0];
                a0 = cmulc(cat5[0], g0);
                cfmac(gc[0], m00_s[co * C5 + k], g0);
                const cplx w1 = m11_s[co * C5 + k];
#pragma unroll
                for (int comp = 1; comp < 5; ++comp) {
                    const cplx gv = gp[comp * 32];
                    cfmac(a1, cat5[comp], gv);
                    cfmac(gc[comp], w1, gv);
                }
            }
            v[4 * u] = a0.x; v[4 * u + 1] = a0.y; v[4 * u + 2] = a1.x; v[4 * u + 3] = a1.y;
        }
        const double tot = warp_sum16(v);
        const int idx = lane >> 1, co = cb + (idx >> 2), irr = (idx >> 1) & 1, ri = idx & 1;
        if (!(lane & 1) && co < Cout) gm_d[((size_t)(irr * nm + co * C5 + k)) * 2 + ri] += tot;
    }
}

// One CTA works on one jet at a time (persistent over jets); warp = channel c, lane = particle.
//   1. stage the jet, rebuild this thread's 25 cat entries from the saved neighbour sums, push the incoming gradients
//      through the adjoint of the channel mix (registers + warp butterflies, no cat buffer in shared memory);
//   2. encoder: neighbour loop over partners o, no barriers: role 1 (own = receiving node) yields dL/dR_{lane,o}, streamed to
//      g_r for radial_bwd_kernel; role 2 (own = neighbour) accumulates dL/dS_lane, dL/dV_lane in registers; R_{lane,o} is
//      streamed from r_save, prefetched.  Decoder: adjoint of the O(N) closed form (constant radial weights);
//   3. when the CTA runs out of jets: one compact row of parameter-gradient partials (mix weights, decoder biases).
// GA (encoder): also write gA, the adjoints of the neighbour sums, to g_a (B,N,C,10) complex for the input-gradient kernels
// (lgae_input_grad.cu).
template <bool ENC, bool GA>
LGAE_DEV void level_bwd_body(const LevelArgs& a, double* g_a) {
    extern __shared__ __align__(128) double smem[];
    const int N = a.N, C = a.C, Cout = a.Cout;
    const int tid = threadIdx.x, lane = tid & 31, c = tid >> 5;
    const LevelBwdSmem L = level_bwd_smem(ENC, N, C, Cout);
    double* p_s = smem + L.p;
    cplx* S_s = reinterpret_cast<cplx*>(smem + L.S);
    cplx* V_s = reinterpret_cast<cplx*>(smem + L.V);
    cplx* m00_s = reinterpret_cast<cplx*>(smem + L.m00);
    cplx* m11_s = reinterpret_cast<cplx*>(smem + L.m11);
    double* gm_d = smem + L.gm;
    cplx* gA_s = reinterpret_cast<cplx*>(smem + L.gA);
    cplx* gy_s = reinterpret_cast<cplx*>(smem + L.gy);
    cplx* gout_s = reinterpret_cast<cplx*>(smem + L.gout);
    const int nm = Cout * 5 * C, C5 = 5 * C;

    pdl_launch();
    for (int t = tid; t < nm; t += blockDim.x) {
        m00_s[t] = cmake(a.theta[a.off_m00 + t], a.theta[a.off_m00 + nm + t]);
        m11_s[t] = cmake(a.theta[a.off_m11 + t], a.theta[a.off_m11 + nm + t]);
    }
    for (int t = tid; t < 4 * nm; t += blockDim.x) gm_d[t] = 0.0;

    cplx R0c = czero(), R1c = czero(), gR0c = czero(), gR1c = czero();
    if (!ENC) {
        const double b0 = a.theta[a.off_b0 + c], b1 = a.theta[a.off_b1 + c];
        R0c = cmake(b0, b0);
        R1c = cmake(b1, b1);
    }

    const int i = lane;
    const bool live = i < N;
    __shared__ uint64_t mbar;
    if (tid == 0) mbar_init(&mbar, 1);
    unsigned phase = 0;
    pdl_wait();   // the weights above come from theta (constant during the step); everything below from earlier kernels
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        __syncthreads();
        // ---- 1a. stage the jet (TMA bulk copies) and the incoming gradients ----
        {
            const int np = ENC ? 4 * N : 8 * N;
            if (tid == 0) {
                // encoder: pull this jet's radial weights (written by the forward pass long ago) towards L2 while the mix
                // adjoint runs; the neighbour loop then streams them with a two-partner register prefetch
                if (ENC) bulk_prefetch_l2(a.r_save + (int64_t)b * N * C * 128, (unsigned)(N * C * 128 * sizeof(double)));
                const unsigned gs_bytes = a.g_s_pre ? 2 * N * Cout * sizeof(double) : 0u;
                mbar_expect_tx(&mbar, (unsigned)((np + 10 * N * C + 8 * N * Cout + 20 * N * C) * sizeof(double)) + gs_bytes);
                // saved neighbour sums (N,C,10) complex land in the gA buffer, which is only written after they are consumed
                bulk_g2s(smem + L.gA, a.sums + (int64_t)b * N * C * 20, 20 * N * C * sizeof(double), &mbar);
                bulk_g2s(p_s, a.p + (int64_t)b * np, np * sizeof(double), &mbar);
                bulk_g2s(smem + L.S, a.s_in + (int64_t)b * N * C * 2, 2 * N * C * sizeof(double), &mbar);
                bulk_g2s(smem + L.V, a.v_in + (int64_t)b * N * C * 8, 8 * N * C * sizeof(double), &mbar);
                if (a.g_s_pre) bulk_g2s(smem + L.graw, a.g_s_pre + (int64_t)b * N * Cout * 2, gs_bytes, &mbar);
                bulk_g2s(smem + L.graw + 2 * N * Cout, a.g_v_out + (int64_t)b * N * Cout * 8, 8 * N * Cout * sizeof(double), &mbar);
            }
        }
        // encoder: first radial weights of this jet, in flight while the mix adjoint runs
        const double4* rsv = reinterpret_cast<const double4*>(a.r_save) + ((int64_t)b * N * C + c) * 32 + lane;
        constexpr int PDB = LGAE_RPD_BWD;
        double4 rq[PDB];
#pragma unroll
        for (int d = 0; d < PDB; ++d) {
            rq[d] = make_double4(0.0, 0.0, 0.0, 0.0);
            if (ENC && d < N) rq[d] = rsv[(int64_t)d * C * 32];
        }
        mbar_wait(&mbar, phase);
        phase ^= 1;
        cplx A[10];
#pragma unroll
        for (int e = 0; e < 10; ++e) A[e] = live ? reinterpret_cast<const cplx*>(smem + L.gA)[(i * C + c) * 10 + e] : czero();
        {   // incoming gradients -> [(c'*5+comp)][lane] (conflict-free for the per-lane reads of the mix adjoint)
            const cplx* gs_raw = reinterpret_cast<const cplx*>(smem + L.graw);
            const cplx* gv_raw = gs_raw + N * Cout;
            for (int it = tid; it < 32 * Cout * 5; it += blockDim.x) {
                const int il = it & 31, r = it >> 5, co = r / 5, comp = r % 5;
                cplx v = czero();
                if (il < N) {
                    if (comp == 0) {
                        if (a.g_s_pre) v = gs_raw[il * Cout + co];
                    } else {
                        v = gv_raw[(il * Cout + co) * 4 + comp - 1];
                    }
                }
                gout_s[r * 32 + il] = v;
            }
        }
        __syncthreads();
        // ---- 1b. adjoint of cat -> mix, block by block, in registers ----
        cplx gS = czero(), gV[4] = {czero(), czero(), czero(), czero()};
        {
            const cplx Si = live ? S_s[i * C + c] : czero();
            cplx Vi[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) Vi[mu] = live ? V_s[(i * C + c) * 4 + mu] : czero();
            cplx cat5[5], gc[5];
            // block 0: [ (1/2) A1E | (1+i) A0V ]   -> adjoints of A1E, A0V
            cat5[0] = cscale(A[9], 0.5);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cat5[1 + mu] = cmul_1pi(A[mu]);
            mix_adjoint_block(c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
            gA_s[(c * 10 + 9) * 32 + lane] = cscale(gc[0], 0.5);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) gA_s[(c * 10 + mu) * 32 + lane] = cmul_1mi(gc[1 + mu]);
            // block 1: [ (1+i) A0S | A1Y ]
            cat5[0] = cmul_1pi(A[4]);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cat5[1 + mu] = A[5 + mu];
            mix_adjoint_block(C + c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
            gA_s[(c * 10 + 4) * 32 + lane] = cmul_1mi(gc[0]);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) gA_s[(c * 10 + 5 + mu) * 32 + lane] = gc[1 + mu];
            // block 2: the node itself
            cat5[0] = Si;
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cat5[1 + mu] = Vi[mu];
            mix_adjoint_block(2 * C + c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
            gS = gc[0];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) gV[mu] = gc[1 + mu];
            // block 3: self product, [ (1/2) eta(V,V) | V S ]
            cplx gh[4];
            cghat(Vi, gh);
            cat5[0] = cscale(ceta(Vi, Vi), 0.5);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cat5[1 + mu] = cmul(Vi[mu], Si);
            mix_adjoint_block(3 * C + c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                cfmac(gV[mu], gh[mu], gc[0]);
                cfmac(gV[mu], Si, gc[1 + mu]);
                cfmac(gS, Vi[mu], gc[1 + mu]);
            }
            // block 4: self product, [ S^2 | S V ]
            cat5[0] = cmul(Si, Si);
            mix_adjoint_block(4 * C + c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
            cfmac(gS, Si, cscale(gc[0], 2.0));
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                cfmac(gV[mu], Si, gc[1 + mu]);
                cfmac(gS, Vi[mu], gc[1 + mu]);
            }
        }
        __syncthreads();  // gA_s of every channel is complete (role 2 reads other lanes' entries)
        if (GA && live) {
            cplx* dst = reinterpret_cast<cplx*>(g_a) + ((int64_t)(b * N + i) * C + c) * 10;
#pragma unroll
            for (int e = 0; e < 10; ++e) dst[e] = gA_s[(c * 10 + e) * 32 + lane];
        }
        // ---- 2. adjoint of the neighbour sums ----
        cplx gy[4] = {czero(), czero(), czero(), czero()};
        if (!ENC) {
            // Decoder, closed form: adjoint of  A0V_i = R0 SV, A0S_i = R0 SS, A1Y_i = R1 (y_i SS - SSY), A1E_i = R1 (eta(SV, y_i) - SVY)
            // with the jet-level moments SS, SV, SSY, SVY of the forward (recomputed here), all O(N).
            const cplx* y_s = reinterpret_cast<const cplx*>(p_s);
            cplx ya[4], Va[4], gAa[10];
            const cplx Sa = live ? S_s[i * C + c] : czero();
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                ya[mu] = live ? y_s[4 * i + mu] : czero();
                Va[mu] = live ? V_s[(i * C + c) * 4 + mu] : czero();
            }
#pragma unroll
            for (int e = 0; e < 10; ++e) gAa[e] = live ? gA_s[(c * 10 + e) * 32 + lane] : czero();
            // moments (this lane's particle only: N <= 32 in the adjoint)
            double m[20];
            {
                const cplx e = ceta(Va, ya);
                m[0] = Sa.x; m[1] = Sa.y; m[18] = e.x; m[19] = e.y;
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) {
                    m[2 + 2 * mu] = Va[mu].x; m[3 + 2 * mu] = Va[mu].y;
                    const cplx sy = cmul(Sa, ya[mu]);
                    m[10 + 2 * mu] = sy.x; m[11 + 2 * mu] = sy.y;
                }
            }
            warp_allsum_n<20>(m);
            const cplx SS = cmake(m[0], m[1]), SVY = cmake(m[18], m[19]);
            cplx SV[4], SSY[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) { SV[mu] = cmake(m[2 + 2 * mu], m[3 + 2 * mu]); SSY[mu] = cmake(m[10 + 2 * mu], m[11 + 2 * mu]); }
            // per-particle pieces
            cplx gT[4], gU = cmulc(R1c, gAa[9]);          // conj(R1) gA1E_i
            cplx gr0 = cmulc(SS, gAa[4]);                 // conj(SS) gA0S_i
            const cplx U = csub(ceta(SV, ya), SVY);
            cplx gr1 = cmulc(U, gAa[9]);
            cplx yt = czero();                            // sum_mu conj(y_i) gT_i
            cplx ghy[4], ghsv[4], ghv[4];
            cghat(ya, ghy);
            cghat(SV, ghsv);
            cghat(Va, ghv);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                gT[mu] = cmulc(R1c, gAa[5 + mu]);
                cfmac(gr0, SV[mu], gAa[mu]);
                const cplx T = csub(cmul(ya[mu], SS), SSY[mu]);
                cfmac(gr1, T, gAa[5 + mu]);
                cfmac(yt, ya[mu], gT[mu]);
            }
            gR0c = cadd(gR0c, gr0);
            gR1c = cadd(gR1c, gr1);
            // jet-level sums: [sum gA0V (4) | sum gA0S | sum gT (4) | sum gU | sum conj(y) gT | sum conj(ghat(y)) gU (4)]
            double r[30];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                r[2 * mu] = gAa[mu].x; r[2 * mu + 1] = gAa[mu].y;
                r[10 + 2 * mu] = gT[mu].x; r[11 + 2 * mu] = gT[mu].y;
                const cplx t = cmulc(ghy[mu], gU);
                r[22 + 2 * mu] = t.x; r[23 + 2 * mu] = t.y;
            }
            r[8] = gAa[4].x; r[9] = gAa[4].y;
            r[18] = gU.x; r[19] = gU.y;
            r[20] = yt.x; r[21] = yt.y;
            warp_allsum_n<30>(r);
            cplx gSS = cmulc(R0c, cmake(r[8], r[9]));
            gSS = cadd(gSS, cmake(r[20], r[21]));
            const cplx gSVY = cneg(cmake(r[18], r[19]));
            cplx gSa = gSS;
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                cplx gSVm = cmulc(R0c, cmake(r[2 * mu], r[2 * mu + 1]));
                gSVm = cadd(gSVm, cmake(r[22 + 2 * mu], r[23 + 2 * mu]));
                const cplx gSSYm = cneg(cmake(r[10 + 2 * mu], r[11 + 2 * mu]));
                cfmac(gSa, ya[mu], gSSYm);
                cplx gv = gSVm;
                cfmac(gv, ghy[mu], gSVY);
                gV[mu] = cadd(gV[mu], gv);
                cplx g = cmulc(SS, gT[mu]);
                cfmac(g, ghsv[mu], gU);
                cfmac(g, Sa, gSSYm);
                cfmac(g, ghv[mu], gSVY);
                gy[mu] = g;
            }
            gS = cadd(gS, gSa);
        } else {
            // encoder: loop over the partners o
            double pa[4] = {0, 0, 0, 0};
            if (live) {
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) pa[mu] = p_s[4 * i + mu];
            }
            cplx gAa[10];
#ifndef LGAE_GAA_SMEM
#pragma unroll
            for (int e = 0; e < 10; ++e) gAa[e] = gA_s[(c * 10 + e) * 32 + lane];
#endif
            double4* grv = reinterpret_cast<double4*>(a.g_r) + ((int64_t)b * N * C + c) * 32 + lane;
#pragma unroll kBwdUnroll
            for (int o = 0; o < N; ++o) {
                const cplx R0 = cmake(rq[0].x, rq[0].y), R1 = cmake(rq[0].z, rq[0].w);
#pragma unroll
                for (int d = 0; d + 1 < PDB; ++d) rq[d] = rq[d + 1];
                if (o + PDB < N) rq[PDB - 1] = rsv[(int64_t)(o + PDB) * C * 32];
                const cplx So = S_s[o * C + c];
                cplx Vo[4], Y[4];
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) Vo[mu] = V_s[(o * C + c) * 4 + mu];
                // Y = canon(p_i - p_o) = (d0, (ya, -yb), d3, (-ya, -yb)) with real d0, d3, ya, yb -- the contractions
                // with Y below use that structure (12 instead of 16 multiply-adds each)
                double d[4];
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) d[mu] = pa[mu] - p_s[4 * o + mu];
                canon_from_real(d, Y);
                const double d0 = Y[0].x, d3 = Y[2].x, ya_ = Y[1].x, yb_ = -Y[1].y;
                // sum_mu conj(Y_mu) g_mu  and  eta(v, Y)
                auto ydot = [&](const cplx* gq) {
                    const cplx dm = csub(gq[1], gq[3]), sp = cadd(gq[1], gq[3]);
                    return cmake(fma(d0, gq[0].x, fma(d3, gq[2].x, fma(ya_, dm.x, -yb_ * sp.y))),
                                 fma(d0, gq[0].y, fma(d3, gq[2].y, fma(ya_, dm.y, yb_ * sp.x))));
                };
                auto yeta = [&](const cplx* v) {
                    const cplx vm = csub(v[3], v[1]), vp = cadd(v[1], v[3]);
                    return cmake(fma(d0, v[0].x, fma(-d3, v[2].x, fma(ya_, vm.x, yb_ * vp.y))),
                                 fma(d0, v[0].y, fma(-d3, v[2].y, fma(ya_, vm.y, -yb_ * vp.x))));
                };
                // role 1: own = receiving node i, other = neighbour j.  Y = Y_ij.
                {
#ifdef LGAE_GAA_SMEM
#pragma unroll
                    for (int e = 0; e < 10; ++e) gAa[e] = gA_s[(c * 10 + e) * 32 + lane];
#endif
                    cplx gR0 = czero();
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) cfmac(gR0, Vo[mu], gAa[mu]);
                    const cplx w = ydot(gAa + 5);
                    cfmac(gR0, So, gAa[4]);
                    const cplx e = yeta(Vo);
                    cplx gR1 = cmulc(So, w);
                    cfmac(gR1, e, gAa[9]);
                    grv[(int64_t)o * C * 32] = make_double4(gR0.x, gR0.y, gR1.x, gR1.y);
                }
                // role 2: own = neighbour j, other = receiving node i.  Y_ij = -Y ; R_ij = R_ji.
                {
                    cplx gAo[10];
#pragma unroll
                    for (int e = 0; e < 10; ++e) gAo[e] = gA_s[(c * 10 + e) * 32 + o];
                    cplx Yn[4], gh[4];
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) Yn[mu] = cneg(Y[mu]);
                    cghat(Yn, gh);
                    const cplx w = cneg(ydot(gAo + 5));   // sum_mu conj(-Y_mu) gA1Y_o
                    const cplx r1g = cmulc(R1, gAo[9]);   // conj(R1) gA1E_i
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) {
                        cfmac(gV[mu], R0, gAo[mu]);
                        cfmac(gV[mu], gh[mu], r1g);
                    }
                    cfmac(gS, R0, gAo[4]);
                    cfmac(gS, R1, w);
                }
            }
        }
        // ---- results for this jet ----
        if (live) {
            reinterpret_cast<cplx*>(a.g_s_in)[(int64_t)(b * N + i) * C + c] = gS;
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) reinterpret_cast<cplx*>(a.g_v_in)[((int64_t)(b * N + i) * C + c) * 4 + mu] = gV[mu];
        }
        if (!ENC) {
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) gy_s[(c * 4 + mu) * 32 + lane] = live ? gy[mu] : czero();
            __syncthreads();
            for (int t = tid; t < 4 * N; t += blockDim.x) {
                const int ii = t >> 2, mu = t & 3;
                cplx* dst = reinterpret_cast<cplx*>(a.g_y) + (int64_t)(b * N + ii) * 4 + mu;
                cplx acc = *dst;
                for (int cc = 0; cc < C; ++cc) acc = cadd(acc, gy_s[(cc * 4 + mu) * 32 + ii]);   // fixed order: deterministic
                *dst = acc;
            }
        }
    }

    // ---- 3. this CTA's row of parameter-gradient partials ----
    __syncthreads();
    double* row = a.part + (int64_t)blockIdx.x * a.part_stride;
    for (int t = tid; t < nm; t += blockDim.x) {
        row[a.po_m00 + t] = gm_d[2 * t];
        row[a.po_m00 + nm + t] = gm_d[2 * t + 1];
        row[a.po_m11 + t] = gm_d[2 * (nm + t)];
        row[a.po_m11 + nm + t] = gm_d[2 * (nm + t) + 1];
    }
    if (!ENC) {
        // decoder: only the biases learn; R^l[c] = bias (1+i)  =>  g_bias = Re(gR) + Im(gR)
        double v0 = warp_sum(gR0c.x + gR0c.y), v1 = warp_sum(gR1c.x + gR1c.y);
        if (lane == 0) {
            row[a.po_b0 + c] = v0;
            row[a.po_b1 + c] = v1;
        }
    }
}

template <bool ENC, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) level_bwd_kernel(const LevelArgs a) { level_bwd_body<ENC, false>(a, nullptr); }
template <int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) level_bwd_ga_kernel(const LevelArgs a, double* g_a) { level_bwd_body<true, true>(a, g_a); }

// ------------------------------------------------------------------------------------------------------------
// host-side launchers
// ------------------------------------------------------------------------------------------------------------
static int pick_ks(int K) { return K <= 12 ? 3 : (K <= 20 ? 5 : (K <= 32 ? 8 : -1)); }

template <bool ENC, int NT, int KS, bool PRE>
static int launch_level_fwd(const LevelArgs& a, cudaStream_t st) {
    const LevelSmem L = level_smem(ENC, ENC && !PRE, a.N, a.C, a.Cout, KS);
    const size_t bytes = (size_t)L.total * sizeof(double);
    if (bytes > 227 * 1024) return LGAE_E_UNSUPPORTED;
    auto kern = level_fwd_kernel<ENC, NT, KS, PRE>;
    if (int rc = ensure_smem((const void*)kern, bytes)) return rc;
    const int nib = (a.N + 31) / 32;
    LaunchScope ls_("level_fwd", st);
    launch_k(kern, dim3(a.B * nib), dim3(32 * a.C), bytes, st, a);
    return check_launch("level_fwd");
}

template <bool ENC>
static int launch_level_bwd(const LevelArgs& a, int grid, cudaStream_t st, double* g_a) {
    if (a.N > 32) return LGAE_E_UNSUPPORTED;
    const LevelBwdSmem L = level_bwd_smem(ENC, a.N, a.C, a.Cout);
    const size_t bytes = (size_t)L.total * sizeof(double);
    if (bytes > 227 * 1024) return LGAE_E_UNSUPPORTED;
    LaunchScope ls_("level_bwd", st);
#define LGAE_LAUNCH(MAXT, MINB)                                               \
    {                                                                         \
        if constexpr (ENC) {                                                  \
            if (g_a) {                                                        \
                auto kern = level_bwd_ga_kernel<MAXT, (MINB)>;                \
                if (int rc = ensure_smem((const void*)kern, bytes)) return rc; \
                launch_k(kern, dim3(grid), dim3(32 * a.C), bytes, st, a, g_a); \
                return check_launch("level_bwd");                             \
            }                                                                 \
        }                                                                     \
        auto kern = level_bwd_kernel<ENC, MAXT, (MINB)>;                      \
        if (int rc = ensure_smem((const void*)kern, bytes)) return rc;        \
        launch_k(kern, dim3(grid), dim3(32 * a.C), bytes, st, a);                               \
    }
    if (a.C <= 3)
        LGAE_LAUNCH(128, ENC ? LGAE_LBWD_MINB : LGAE_LBWD_CF_MINB)
    else if (a.C == 4)
        LGAE_LAUNCH(128, ENC ? LGAE_LBWD_MINB_C4 : LGAE_LBWD_CF_MINB_C4)
    else
        LGAE_LAUNCH(256, 1)
#undef LGAE_LAUNCH
    return check_launch("level_bwd");
}

// Number of CTAs (= rows of partials) the level adjoint uses for a batch.
int level_bwd_grid(int batch) {
    const int cap = 4 * sm_count();
    return batch < cap ? (batch > 0 ? batch : 1) : cap;
}

static int dispatch_level_fwd(const LevelArgs& a, bool enc, cudaStream_t st) {
    if (a.C < 1 || a.C > LGAE_MAX_CHANNELS || a.Cout < 1 || a.Cout > LGAE_MAX_CHANNELS) return LGAE_E_UNSUPPORTED;
    if (!enc) return launch_level_fwd<false, 1, 3, true>(a, st);   // closed form
    if (a.r_save) return launch_level_fwd<true, 1, 3, true>(a, st);   // radial weights precomputed (N <= 32)
    const int nt = (4 * a.C + 7) / 8, ks = pick_ks(a.K);
    if (ks < 0) return LGAE_E_UNSUPPORTED;
#define LGAE_CASE(NTV, KSV) \
    if (nt == NTV && ks == KSV) return launch_level_fwd<true, NTV, KSV, false>(a, st);
    LGAE_CASE(1, 3) LGAE_CASE(2, 3) LGAE_CASE(3, 3) LGAE_CASE(4, 3)
    LGAE_CASE(1, 5) LGAE_CASE(2, 5) LGAE_CASE(3, 5) LGAE_CASE(4, 5)
    LGAE_CASE(1, 8) LGAE_CASE(2, 8) LGAE_CASE(3, 8) LGAE_CASE(4, 8)
#undef LGAE_CASE
    return LGAE_E_UNSUPPORTED;
}

static void fill_level_args(LevelArgs& a, const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y,
                            const uint8_t* node_mask, int batch, const double* s_in, const double* v_in, double* sums, double* r_save) {
    memset(&a, 0, sizeof(a));
    a.theta = theta;
    a.off_a = d->off_rad_a[level]; a.off_b = d->off_rad_b[level]; a.off_c = d->off_rad_c[level];
    a.off_w0 = d->off_rad_w0[level]; a.off_b0 = d->off_rad_b0[level];
    a.off_w1 = d->off_rad_w1[level]; a.off_b1 = d->off_rad_b1[level];
    a.off_m00 = d->off_mix00[level]; a.off_m11 = d->off_mix11[level];
    a.p = p_or_y; a.node_mask = node_mask; a.s_in = s_in; a.v_in = v_in; a.sums = sums;
    a.r_save = (!d->is_decoder && d->n_particles <= 32) ? r_save : nullptr;
    a.B = batch; a.N = d->n_particles; a.C = d->channels[level]; a.Cout = d->channels[level + 1]; a.K = d->n_basis;
}

// Forward of one level.  Encoder with r_save != NULL (N <= 32): r_save must already hold the radial weights
// (run_radial_fwd); otherwise the radial functions are evaluated inside the kernel, tile by tile.
int run_level_fwd(const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y, const uint8_t* node_mask, int batch,
                  const double* s_in, const double* v_in, double* sums, double* r_save, double* s_pre, double* v_out, cudaStream_t st) {
    if (!d || level < 0 || level >= d->n_levels) return LGAE_E_BADARG;
    if (batch <= 0) return LGAE_OK;
    LevelArgs a;
    fill_level_args(a, d, level, theta, p_or_y, node_mask, batch, s_in, v_in, sums, r_save);
    a.s_pre = s_pre; a.v_out = v_out;
    return dispatch_level_fwd(a, !d->is_decoder, st);
}

// Adjoint of one level (without the adjoint of the radial functions: the encoder streams dL/dR to g_r for
// run_radial_bwd).  Reserves a block of `plan` for the per-CTA partial rows and declares its segments.  Encoder with g_a != NULL:
// also writes the adjoints of the neighbour sums to g_a (B,N,C,10) complex, for the input gradient.
int run_level_bwd(const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y, const uint8_t* node_mask, int batch,
                  const double* s_in, const double* v_in, const double* sums, const double* r_save, double* g_r, const double* g_s_pre,
                  const double* g_v_out, double* g_s_in, double* g_v_in, double* g_y, PartPlan* plan, cudaStream_t st, double* g_a) {
    if (!d || level < 0 || level >= d->n_levels || !plan) return LGAE_E_BADARG;
    if (batch <= 0) return LGAE_OK;
    LevelArgs a;
    fill_level_args(a, d, level, theta, p_or_y, node_mask, batch, s_in, v_in, const_cast<double*>(sums), const_cast<double*>(r_save));
    const bool enc = !d->is_decoder;
    if (enc && (!a.r_save || !g_r)) return LGAE_E_UNSUPPORTED;   // the encoder adjoint needs the saved radial weights (N <= 32)
    a.g_r = g_r;
    a.g_s_pre = g_s_pre; a.g_v_out = g_v_out; a.g_s_in = g_s_in; a.g_v_in = g_v_in; a.g_y = g_y;
    const int grid = level_bwd_grid(batch);
    const int C = a.C, nm2 = 2 * a.Cout * 5 * C;
    int64_t w = 0;
    if (!enc) {
        a.po_b0 = w; w += C;
        a.po_b1 = w; w += C;
    }
    a.po_m00 = w; w += nm2;
    a.po_m11 = w; w += nm2;
    const int64_t off = plan->block(grid, w);
    a.part = plan->base + off;
    a.part_stride = w;
    int rc = LGAE_OK;
    auto seg = [&](int64_t theta_off, int64_t col, int64_t len) { if (rc == LGAE_OK) rc = plan->seg(theta_off, off, w, col, len, grid); };
    if (!enc) { seg(a.off_b0, a.po_b0, C); seg(a.off_b1, a.po_b1, C); }
    seg(a.off_m00, a.po_m00, nm2); seg(a.off_m11, a.po_m11, nm2);
    if (rc != LGAE_OK) return rc;
    if (a.C < 1 || a.C > LGAE_MAX_CHANNELS || a.Cout < 1 || a.Cout > LGAE_MAX_CHANNELS) return LGAE_E_UNSUPPORTED;
    return enc ? launch_level_bwd<true>(a, grid, st, g_a) : launch_level_bwd<false>(a, grid, st, nullptr);
}

// Width (doubles) of one row of partials of the level adjoint.
int64_t level_part_width(const LgaeModelDesc* d, int level) {
    const int C = d->channels[level], Cout = d->channels[level + 1];
    const int64_t mix = (int64_t)4 * Cout * 5 * C;
    return d->is_decoder ? 2 * C + mix : mix;
}

}  // namespace lgae

// ============================================================================================================
// Tiled adjoint, any N (lgae_encoder_backward_tiled / lgae_decoder_backward_tiled).  The per-lane adjoint above holds
// one particle per lane and streams the saved radial weights of every pair, so it stops at 32 particles.  This one
// works like the N > 32 forward: a CTA of 32 C threads (warp = channel, lane = particle of a block of 32) takes one
// (jet, particle block) unit at a time, persistent over the units in a fixed order, and the encoder re-evaluates the
// radial weights tile by tile with radial_tile.  Three kernels per level:
//   level_bwd_mix_tiled  adjoint of the channel mix -> gA (the adjoints of the 10 neighbour sums, (B,N,C,10) complex) in
//                        scratch, node and self-product parts of dL/dS, dL/dV, one row of mix-weight partials per CTA;
//   level_bwd_nbr_tiled  encoder: neighbour loop over partner tiles.  Role 1 writes dL/dR_{i,o} to g_r, laid out as the
//                        per-lane adjoint's (B,N_o,C,32_i,4) with a block axis: (B, nib, N_o, C, 32_i, 4); role 2 adds the
//                        neighbour part of dL/dS_i, dL/dV_i (accumulated in partner order) to the mix kernel's values;
//   level_bwd_cf_tiled   decoder: adjoint of the O(N) closed form, one CTA per jet looping over the blocks.
// ============================================================================================================
namespace lgae {

struct TiledMixSmem {
    int m00, m11, gm, gout;
    int total;
};
__host__ __device__ inline TiledMixSmem tiled_mix_smem(int C, int Cout) {
    TiledMixSmem s;
    const int nm = Cout * 5 * C;
    int o = 0;
    s.m00 = o; o += 2 * nm;
    s.m11 = o; o += 2 * nm;
    s.gm = o; o += 4 * nm;               // [irrep][c'][k] complex accumulators, live for the whole CTA
    s.gout = o; o += 2 * Cout * 5 * 32;  // incoming gradients of the unit [(c'*5+comp)][32] complex
    s.total = o;
    return s;
}

__global__ void __launch_bounds__(256) level_bwd_mix_tiled(const LevelArgs a, double* gA) {
    extern __shared__ __align__(128) double smem[];
    const int N = a.N, C = a.C, Cout = a.Cout, nib = (N + 31) / 32;
    const int tid = threadIdx.x, lane = tid & 31, c = tid >> 5;
    const TiledMixSmem L = tiled_mix_smem(C, Cout);
    cplx* m00_s = reinterpret_cast<cplx*>(smem + L.m00);
    cplx* m11_s = reinterpret_cast<cplx*>(smem + L.m11);
    double* gm_d = smem + L.gm;
    cplx* gout_s = reinterpret_cast<cplx*>(smem + L.gout);
    const int nm = Cout * 5 * C, C5 = 5 * C;

    pdl_launch();
    for (int t = tid; t < nm; t += blockDim.x) {
        m00_s[t] = cmake(a.theta[a.off_m00 + t], a.theta[a.off_m00 + nm + t]);
        m11_s[t] = cmake(a.theta[a.off_m11 + t], a.theta[a.off_m11 + nm + t]);
    }
    for (int t = tid; t < 4 * nm; t += blockDim.x) gm_d[t] = 0.0;
    pdl_wait();
    const cplx* gsp = reinterpret_cast<const cplx*>(a.g_s_pre);
    const cplx* gvo = reinterpret_cast<const cplx*>(a.g_v_out);
    for (int u = blockIdx.x; u < a.B * nib; u += gridDim.x) {
        const int b = u / nib, i0 = (u % nib) * 32, i = i0 + lane;
        const bool live = i < N;
        const int64_t node = (int64_t)b * N + i;
        __syncthreads();   // the previous unit's gradients are consumed
        for (int it = tid; it < 32 * Cout * 5; it += blockDim.x) {
            const int il = it & 31, r = it >> 5, co = r / 5, comp = r % 5;
            const int64_t nd = (int64_t)b * N + i0 + il;
            cplx v = czero();
            if (i0 + il < N) {
                if (comp == 0) {
                    if (gsp) v = gsp[nd * Cout + co];
                } else {
                    v = gvo[(nd * Cout + co) * 4 + comp - 1];
                }
            }
            gout_s[r * 32 + il] = v;
        }
        cplx A[10], Si = czero(), Vi[4];
        const cplx* sums = reinterpret_cast<const cplx*>(a.sums) + (node * C + c) * 10;
#pragma unroll
        for (int e = 0; e < 10; ++e) A[e] = live ? sums[e] : czero();
        if (live) Si = reinterpret_cast<const cplx*>(a.s_in)[node * C + c];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) Vi[mu] = live ? reinterpret_cast<const cplx*>(a.v_in)[(node * C + c) * 4 + mu] : czero();
        __syncthreads();
        // the five blocks of the concatenation, as in level_bwd_kernel
        cplx gS = czero(), gV[4] = {czero(), czero(), czero(), czero()}, gAl[10];
        cplx cat5[5], gc[5];
        cat5[0] = cscale(A[9], 0.5);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) cat5[1 + mu] = cmul_1pi(A[mu]);
        mix_adjoint_block(c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
        gAl[9] = cscale(gc[0], 0.5);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) gAl[mu] = cmul_1mi(gc[1 + mu]);
        cat5[0] = cmul_1pi(A[4]);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) cat5[1 + mu] = A[5 + mu];
        mix_adjoint_block(C + c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
        gAl[4] = cmul_1mi(gc[0]);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) gAl[5 + mu] = gc[1 + mu];
        cat5[0] = Si;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) cat5[1 + mu] = Vi[mu];
        mix_adjoint_block(2 * C + c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
        gS = gc[0];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) gV[mu] = gc[1 + mu];
        cplx gh[4];
        cghat(Vi, gh);
        cat5[0] = cscale(ceta(Vi, Vi), 0.5);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) cat5[1 + mu] = cmul(Vi[mu], Si);
        mix_adjoint_block(3 * C + c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) {
            cfmac(gV[mu], gh[mu], gc[0]);
            cfmac(gV[mu], Si, gc[1 + mu]);
            cfmac(gS, Vi[mu], gc[1 + mu]);
        }
        cat5[0] = cmul(Si, Si);
        mix_adjoint_block(4 * C + c, Cout, C5, nm, lane, cat5, gout_s, m00_s, m11_s, gm_d, gc);
        cfmac(gS, Si, cscale(gc[0], 2.0));
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) {
            cfmac(gV[mu], Si, gc[1 + mu]);
            cfmac(gS, Vi[mu], gc[1 + mu]);
        }
        if (live) {
            cplx* dst = reinterpret_cast<cplx*>(gA) + (node * C + c) * 10;
#pragma unroll
            for (int e = 0; e < 10; ++e) dst[e] = gAl[e];
            reinterpret_cast<cplx*>(a.g_s_in)[node * C + c] = gS;
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) reinterpret_cast<cplx*>(a.g_v_in)[(node * C + c) * 4 + mu] = gV[mu];
        }
    }
    __syncthreads();
    double* row = a.part + (int64_t)blockIdx.x * a.part_stride;
    for (int t = tid; t < nm; t += blockDim.x) {
        row[a.po_m00 + t] = gm_d[2 * t];
        row[a.po_m00 + nm + t] = gm_d[2 * t + 1];
        row[a.po_m11 + t] = gm_d[2 * (nm + t)];
        row[a.po_m11 + nm + t] = gm_d[2 * (nm + t) + 1];
    }
}

struct TiledNbrSmem {
    int p, msk, abc, S, V, gA, Rs;
    int total;
};
__host__ __device__ inline TiledNbrSmem tiled_nbr_smem(int N, int C, int KS) {
    TiledNbrSmem s;
    int o = 0;
    s.p = o; o += 4 * N;
    s.msk = o; o += ((N + 7) / 8 + 2) & ~1;
    s.abc = o; o += (3 * 4 * KS + 1) & ~1;
    s.S = o; o += 2 * TJ * C;    // the partner tile's node features and neighbour-sum adjoints
    s.V = o; o += 8 * TJ * C;
    s.gA = o; o += 20 * TJ * C;
    o = (o + 3) & ~3;
    s.Rs = o; o += TJ * C * 32 * 4;   // radial weights of the tile, as radial_tile writes them
    s.total = o;
    return s;
}

template <int NT, int KS>
__global__ void __launch_bounds__(256) level_bwd_nbr_tiled(const LevelArgs a, const double* gA) {
    extern __shared__ __align__(128) double smem[];
    const int N = a.N, C = a.C, nib = (N + 31) / 32;
    const int tid = threadIdx.x, lane = tid & 31, c = tid >> 5;
    const TiledNbrSmem L = tiled_nbr_smem(N, C, KS);
    double* p_s = smem + L.p;
    uint8_t* msk_s = reinterpret_cast<uint8_t*>(smem + L.msk);
    double* abc_s = smem + L.abc;
    cplx* S_s = reinterpret_cast<cplx*>(smem + L.S);
    cplx* V_s = reinterpret_cast<cplx*>(smem + L.V);
    cplx* gA_s = reinterpret_cast<cplx*>(smem + L.gA);
    double* Rs = smem + L.Rs;

    pdl_launch();
    double wf[KS][NT], bf[NT][2];
    load_radial_frags<NT, KS>(a, wf, bf, abc_s);
    pdl_wait();
    const cplx* gAg = reinterpret_cast<const cplx*>(gA);
    for (int u = blockIdx.x; u < a.B * nib; u += gridDim.x) {
        const int b = u / nib, ib = u % nib, i0 = ib * 32, i = i0 + lane;
        const bool live = i < N;
        const int64_t node = (int64_t)b * N + i;
        __syncthreads();   // the previous unit is done with p_s / msk_s
        const double* pg = a.p + (int64_t)b * N * 4;
        for (int t = tid; t < 4 * N; t += blockDim.x) p_s[t] = pg[t];
        for (int t = tid; t < N; t += blockDim.x) msk_s[t] = a.node_mask ? a.node_mask[(int64_t)b * N + t] : (pg[4 * t] != 0.0);
        double pa[4] = {0, 0, 0, 0};
        cplx gAa[10], gS = czero(), gV[4];
#pragma unroll
        for (int e = 0; e < 10; ++e) gAa[e] = live ? gAg[(node * C + c) * 10 + e] : czero();
        if (live) {
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) pa[mu] = pg[4 * i + mu];
            gS = reinterpret_cast<const cplx*>(a.g_s_in)[node * C + c];
        }
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) gV[mu] = live ? reinterpret_cast<const cplx*>(a.g_v_in)[(node * C + c) * 4 + mu] : czero();
        double4* grv = reinterpret_cast<double4*>(a.g_r) + ((((int64_t)b * nib + ib) * N) * C + c) * 32 + lane;
        for (int j0 = 0; j0 < N; j0 += TJ) {
            const int tj = min(TJ, N - j0);
            __syncthreads();   // p_s / msk_s staged; the previous tile's buffers are consumed
            {
                const int64_t base = (int64_t)b * N + j0;
                const cplx* sg = reinterpret_cast<const cplx*>(a.s_in) + base * C;
                const cplx* vg = reinterpret_cast<const cplx*>(a.v_in) + base * C * 4;
                const cplx* ag = gAg + base * C * 10;
                const int ns = tj * C;
                for (int t = tid; t < 15 * ns; t += blockDim.x) {
                    if (t < ns) S_s[t] = sg[t];
                    else if (t < 5 * ns) V_s[t - ns] = vg[t - ns];
                    else gA_s[t - 5 * ns] = ag[t - 5 * ns];
                }
            }
            radial_tile<NT, KS>(p_s, msk_s, N, C, i0, j0, tj, abc_s, wf, bf, Rs);
            __syncthreads();
            for (int jj = 0; jj < tj; ++jj) {
                const int o = j0 + jj;
                const double4 r = *reinterpret_cast<const double4*>(Rs + ((size_t)((jj * C + c) * 32 + lane)) * 4);
                const cplx R0 = cmake(r.x, r.y), R1 = cmake(r.z, r.w);
                const cplx So = S_s[jj * C + c];
                cplx Vo[4], Y[4];
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) Vo[mu] = V_s[(jj * C + c) * 4 + mu];
                double d[4];
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) d[mu] = pa[mu] - p_s[4 * o + mu];
                canon_from_real(d, Y);
                const double d0 = Y[0].x, d3 = Y[2].x, ya_ = Y[1].x, yb_ = -Y[1].y;
                auto ydot = [&](const cplx* gq) {
                    const cplx dm = csub(gq[1], gq[3]), sp = cadd(gq[1], gq[3]);
                    return cmake(fma(d0, gq[0].x, fma(d3, gq[2].x, fma(ya_, dm.x, -yb_ * sp.y))),
                                 fma(d0, gq[0].y, fma(d3, gq[2].y, fma(ya_, dm.y, yb_ * sp.x))));
                };
                auto yeta = [&](const cplx* v) {
                    const cplx vm = csub(v[3], v[1]), vp = cadd(v[1], v[3]);
                    return cmake(fma(d0, v[0].x, fma(-d3, v[2].x, fma(ya_, vm.x, yb_ * vp.y))),
                                 fma(d0, v[0].y, fma(-d3, v[2].y, fma(ya_, vm.y, -yb_ * vp.x))));
                };
                // role 1: own = receiving node i, other = neighbour o
                if (live) {
                    cplx gR0 = czero();
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) cfmac(gR0, Vo[mu], gAa[mu]);
                    const cplx w = ydot(gAa + 5);
                    cfmac(gR0, So, gAa[4]);
                    const cplx e = yeta(Vo);
                    cplx gR1 = cmulc(So, w);
                    cfmac(gR1, e, gAa[9]);
                    grv[(int64_t)o * C * 32] = make_double4(gR0.x, gR0.y, gR1.x, gR1.y);
                }
                // role 2: own = neighbour i of the receiving node o.  Y_oi = -Y ; R_oi = R_io.
                {
                    const cplx* gAo = gA_s + (jj * C + c) * 10;
                    cplx Yn[4], gh[4];
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) Yn[mu] = cneg(Y[mu]);
                    cghat(Yn, gh);
                    const cplx w = cneg(ydot(gAo + 5));
                    const cplx r1g = cmulc(R1, gAo[9]);
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) {
                        cfmac(gV[mu], R0, gAo[mu]);
                        cfmac(gV[mu], gh[mu], r1g);
                    }
                    cfmac(gS, R0, gAo[4]);
                    cfmac(gS, R1, w);
                }
            }
        }
        if (live) {
            reinterpret_cast<cplx*>(a.g_s_in)[node * C + c] = gS;
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) reinterpret_cast<cplx*>(a.g_v_in)[(node * C + c) * 4 + mu] = gV[mu];
        }
    }
}

// Decoder: the closed form's adjoint (see level_bwd_kernel) with the jet-level moments and the 30 jet-level adjoint sums
// accumulated over the particles lane-strided (particle j in lane j % 32, in increasing j, then one warp butterfly: a
// fixed order), then the per-particle dL/dS, dL/dV (added to the mix kernel's values) and dL/dy block by block.
__global__ void __launch_bounds__(256) level_bwd_cf_tiled(const LevelArgs a, const double* gA) {
    extern __shared__ __align__(128) double smem[];
    const int N = a.N, C = a.C;
    const int tid = threadIdx.x, lane = tid & 31, c = tid >> 5;
    cplx* gy_s = reinterpret_cast<cplx*>(smem);   // [(c*4+mu)][32]
    pdl_launch();
    const double b0 = a.theta[a.off_b0 + c], b1 = a.theta[a.off_b1 + c];
    const cplx R0c = cmake(b0, b0), R1c = cmake(b1, b1);
    cplx gR0c = czero(), gR1c = czero();
    pdl_wait();
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        const cplx* y_g = reinterpret_cast<const cplx*>(a.p) + (int64_t)b * N * 4;
        const cplx* S_g = reinterpret_cast<const cplx*>(a.s_in) + (int64_t)b * N * C;
        const cplx* V_g = reinterpret_cast<const cplx*>(a.v_in) + (int64_t)b * N * C * 4;
        const cplx* gA_g = reinterpret_cast<const cplx*>(gA) + (int64_t)b * N * C * 10;
        // jet moments, summed as the forward sums them
        double m[20];
#pragma unroll
        for (int t = 0; t < 20; ++t) m[t] = 0.0;
        for (int j = lane; j < N; j += 32) {
            const cplx Sj = S_g[j * C + c];
            cplx Vj[4], yj[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) { Vj[mu] = V_g[(j * C + c) * 4 + mu]; yj[mu] = y_g[4 * j + mu]; }
            m[0] += Sj.x; m[1] += Sj.y;
            const cplx e = ceta(Vj, yj);
            m[18] += e.x; m[19] += e.y;
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                m[2 + 2 * mu] += Vj[mu].x; m[3 + 2 * mu] += Vj[mu].y;
                const cplx sy = cmul(Sj, yj[mu]);
                m[10 + 2 * mu] += sy.x; m[11 + 2 * mu] += sy.y;
            }
        }
        warp_allsum_n<20>(m);
        const cplx SS = cmake(m[0], m[1]), SVY = cmake(m[18], m[19]);
        cplx SV[4], SSY[4], ghsv[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) { SV[mu] = cmake(m[2 + 2 * mu], m[3 + 2 * mu]); SSY[mu] = cmake(m[10 + 2 * mu], m[11 + 2 * mu]); }
        cghat(SV, ghsv);
        // jet-level sums: [sum gA0V (4) | sum gA0S | sum gT (4) | sum gU | sum conj(y) gT | sum conj(ghat(y)) gU (4)]
        double r[30];
#pragma unroll
        for (int t = 0; t < 30; ++t) r[t] = 0.0;
        for (int i = lane; i < N; i += 32) {
            cplx ya[4], gAa[10];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) ya[mu] = y_g[4 * i + mu];
#pragma unroll
            for (int e = 0; e < 10; ++e) gAa[e] = gA_g[(i * C + c) * 10 + e];
            const cplx gU = cmulc(R1c, gAa[9]);
            cplx gr0 = cmulc(SS, gAa[4]);
            const cplx U = csub(ceta(SV, ya), SVY);
            cplx gr1 = cmulc(U, gAa[9]);
            cplx yt = czero();
            cplx ghy[4];
            cghat(ya, ghy);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                const cplx gT = cmulc(R1c, gAa[5 + mu]);
                cfmac(gr0, SV[mu], gAa[mu]);
                const cplx T = csub(cmul(ya[mu], SS), SSY[mu]);
                cfmac(gr1, T, gAa[5 + mu]);
                cfmac(yt, ya[mu], gT);
                r[2 * mu] += gAa[mu].x; r[2 * mu + 1] += gAa[mu].y;
                r[10 + 2 * mu] += gT.x; r[11 + 2 * mu] += gT.y;
                const cplx t = cmulc(ghy[mu], gU);
                r[22 + 2 * mu] += t.x; r[23 + 2 * mu] += t.y;
            }
            r[8] += gAa[4].x; r[9] += gAa[4].y;
            r[18] += gU.x; r[19] += gU.y;
            r[20] += yt.x; r[21] += yt.y;
            gR0c = cadd(gR0c, gr0);
            gR1c = cadd(gR1c, gr1);
        }
        warp_allsum_n<30>(r);
        cplx gSS = cmulc(R0c, cmake(r[8], r[9]));
        gSS = cadd(gSS, cmake(r[20], r[21]));
        const cplx gSVY = cneg(cmake(r[18], r[19]));
        cplx gSVm[4], gSSYm[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) {
            gSVm[mu] = cadd(cmulc(R0c, cmake(r[2 * mu], r[2 * mu + 1])), cmake(r[22 + 2 * mu], r[23 + 2 * mu]));
            gSSYm[mu] = cneg(cmake(r[10 + 2 * mu], r[11 + 2 * mu]));
        }
        for (int i0 = 0; i0 < N; i0 += 32) {
            const int i = i0 + lane;
            const bool live = i < N;
            cplx gy[4] = {czero(), czero(), czero(), czero()};
            if (live) {
                cplx ya[4], Va[4], ghy[4], ghv[4];
                const cplx Sa = S_g[i * C + c], gU = cmulc(R1c, gA_g[(i * C + c) * 10 + 9]);
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) { ya[mu] = y_g[4 * i + mu]; Va[mu] = V_g[(i * C + c) * 4 + mu]; }
                cghat(ya, ghy);
                cghat(Va, ghv);
                cplx* gs_d = reinterpret_cast<cplx*>(a.g_s_in) + ((int64_t)b * N + i) * C + c;
                cplx* gv_d = reinterpret_cast<cplx*>(a.g_v_in) + (((int64_t)b * N + i) * C + c) * 4;
                cplx gSa = gSS;
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) {
                    cfmac(gSa, ya[mu], gSSYm[mu]);
                    cplx gv = gSVm[mu];
                    cfmac(gv, ghy[mu], gSVY);
                    gv_d[mu] = cadd(gv_d[mu], gv);
                    cplx g = cmulc(SS, cmulc(R1c, gA_g[(i * C + c) * 10 + 5 + mu]));
                    cfmac(g, ghsv[mu], gU);
                    cfmac(g, Sa, gSSYm[mu]);
                    cfmac(g, ghv[mu], gSVY);
                    gy[mu] = g;
                }
                *gs_d = cadd(*gs_d, gSa);
            }
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) gy_s[(c * 4 + mu) * 32 + lane] = gy[mu];
            __syncthreads();
            const int nb = min(32, N - i0);
            for (int t = tid; t < 4 * nb; t += blockDim.x) {
                const int il = t >> 2, mu = t & 3;
                cplx* dst = reinterpret_cast<cplx*>(a.g_y) + ((int64_t)b * N + i0 + il) * 4 + mu;
                cplx acc = *dst;
                for (int cc = 0; cc < C; ++cc) acc = cadd(acc, gy_s[(cc * 4 + mu) * 32 + il]);   // fixed order: deterministic
                *dst = acc;
            }
            __syncthreads();
        }
    }
    double* row = a.part + (int64_t)blockIdx.x * a.part_stride;
    const double v0 = warp_sum(gR0c.x + gR0c.y), v1 = warp_sum(gR1c.x + gR1c.y);
    if (lane == 0) {
        row[a.po_b0 + c] = v0;
        row[a.po_b1 + c] = v1;
    }
}

// ---- host side of the tiled adjoint ----
#define LGAE_TRY(expr)                  \
    do {                                \
        const int rc_ = (expr);         \
        if (rc_ != LGAE_OK) return rc_; \
    } while (0)

static int level_tiled_check(const LevelArgs& a, bool enc, size_t* nbr_bytes) {
    if (a.C < 1 || a.C > LGAE_MAX_CHANNELS || a.Cout < 1 || a.Cout > LGAE_MAX_CHANNELS) return LGAE_E_UNSUPPORTED;
    if ((size_t)tiled_mix_smem(a.C, a.Cout).total * sizeof(double) > 227 * 1024) return LGAE_E_UNSUPPORTED;
    if (!enc) return 2 * 4 * 32 * a.C * sizeof(double) > 227 * 1024 ? LGAE_E_UNSUPPORTED : LGAE_OK;
    const int ks = pick_ks(a.K);
    if (ks < 0) return LGAE_E_UNSUPPORTED;
    const size_t bytes = (size_t)tiled_nbr_smem(a.N, a.C, ks).total * sizeof(double);
    if (bytes > 227 * 1024) return LGAE_E_UNSUPPORTED;
    if (nbr_bytes) *nbr_bytes = bytes;
    return LGAE_OK;
}

// LGAE_OK if the tiled adjoint runs every level of the model, else LGAE_E_UNSUPPORTED (no GPU needed).
int level_bwd_tiled_check(const LgaeModelDesc* d) {
    for (int l = 0; l < d->n_levels; ++l) {
        LevelArgs a;
        fill_level_args(a, d, l, nullptr, nullptr, nullptr, 1, nullptr, nullptr, nullptr, nullptr);
        if (int rc = level_tiled_check(a, !d->is_decoder, nullptr)) return rc;
    }
    return LGAE_OK;
}

// Width (doubles) of the partial rows of one level of the tiled adjoint, over all its kernels.
int64_t level_tiled_part_doubles(const LgaeModelDesc* d, int level, int batch) {
    const int C = d->channels[level], Cout = d->channels[level + 1], nib = (d->n_particles + 31) / 32;
    int64_t n = (int64_t)level_bwd_grid(batch * nib) * 4 * Cout * 5 * C;
    if (d->is_decoder) n += (int64_t)level_bwd_grid(batch) * 2 * C;
    return n;
}

// Adjoint of one level for any N.  gA: (B,N,C,10) complex scratch; g_r (encoder): (B, nib, N, C, 32, 4) scratch of dL/dR,
// for run_radial_bwd with nrm == NULL.  Reserves blocks of `plan` for the partial rows and declares their segments.
int run_level_bwd_tiled(const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y, const uint8_t* node_mask, int batch,
                        const double* s_in, const double* v_in, const double* sums, double* gA, double* g_r, const double* g_s_pre,
                        const double* g_v_out, double* g_s_in, double* g_v_in, double* g_y, PartPlan* plan, cudaStream_t st) {
    if (!d || level < 0 || level >= d->n_levels || !plan || !gA) return LGAE_E_BADARG;
    if (batch <= 0) return LGAE_OK;
    const bool enc = !d->is_decoder;
    if (enc ? !g_r : !g_y) return LGAE_E_BADARG;
    LevelArgs a;
    fill_level_args(a, d, level, theta, p_or_y, node_mask, batch, s_in, v_in, const_cast<double*>(sums), nullptr);
    a.r_save = nullptr;
    a.g_r = g_r;
    a.g_s_pre = g_s_pre; a.g_v_out = g_v_out; a.g_s_in = g_s_in; a.g_v_in = g_v_in; a.g_y = g_y;
    size_t nbr_bytes = 0;
    LGAE_TRY(level_tiled_check(a, enc, &nbr_bytes));
    const int C = a.C, nm2 = 2 * a.Cout * 5 * C, nib = (a.N + 31) / 32;
    const int grid = level_bwd_grid(batch * nib);
    {   // channel mix: rows [m00 | m11]
        const int64_t w = 2 * (int64_t)nm2, off = plan->block(grid, w);
        a.part = plan->base + off; a.part_stride = w; a.po_m00 = 0; a.po_m11 = nm2;
        LGAE_TRY(plan->seg(a.off_m00, off, w, 0, nm2, grid));
        LGAE_TRY(plan->seg(a.off_m11, off, w, nm2, nm2, grid));
        const size_t bytes = (size_t)tiled_mix_smem(C, a.Cout).total * sizeof(double);
        LGAE_TRY(ensure_smem((const void*)level_bwd_mix_tiled, bytes));
        LaunchScope ls_("level_bwd_mix_tiled", st);
        launch_k(level_bwd_mix_tiled, dim3(grid), dim3(32 * C), bytes, st, a, gA);
        LGAE_TRY(check_launch("level_bwd_mix_tiled"));
    }
    if (enc) {
        const int nt = (4 * C + 7) / 8, ks = pick_ks(a.K);
        LaunchScope ls_("level_bwd_nbr_tiled", st);
#define LGAE_CASE(NTV, KSV)                                                                      \
    if (nt == NTV && ks == KSV) {                                                                \
        auto kern = level_bwd_nbr_tiled<NTV, KSV>;                                               \
        LGAE_TRY(ensure_smem((const void*)kern, nbr_bytes));                               \
        launch_k(kern, dim3(grid), dim3(32 * C), nbr_bytes, st, a, (const double*)gA);           \
        return check_launch("level_bwd_nbr_tiled");                                              \
    }
        LGAE_CASE(1, 3) LGAE_CASE(2, 3) LGAE_CASE(3, 3) LGAE_CASE(4, 3)
        LGAE_CASE(1, 5) LGAE_CASE(2, 5) LGAE_CASE(3, 5) LGAE_CASE(4, 5)
        LGAE_CASE(1, 8) LGAE_CASE(2, 8) LGAE_CASE(3, 8) LGAE_CASE(4, 8)
#undef LGAE_CASE
        return LGAE_E_UNSUPPORTED;
    }
    {   // decoder closed form: rows [b0 | b1]
        const int gj = level_bwd_grid(batch);
        const int64_t w = 2 * C, off = plan->block(gj, w);
        a.part = plan->base + off; a.part_stride = w; a.po_b0 = 0; a.po_b1 = C;
        LGAE_TRY(plan->seg(a.off_b0, off, w, 0, C, gj));
        LGAE_TRY(plan->seg(a.off_b1, off, w, C, C, gj));
        const size_t bytes = (size_t)2 * 4 * 32 * C * sizeof(double);
        LGAE_TRY(ensure_smem((const void*)level_bwd_cf_tiled, bytes));
        LaunchScope ls_("level_bwd_cf_tiled", st);
        launch_k(level_bwd_cf_tiled, dim3(gj), dim3(32 * C), bytes, st, a, (const double*)gA);
        return check_launch("level_bwd_cf_tiled");
    }
}

}  // namespace lgae
