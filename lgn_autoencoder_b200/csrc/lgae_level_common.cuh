// Shared by the level kernels (lgae_level.cu: maxdim 2) and the maxdim-3 forward (lgae_md3.cu): the level arguments, the pair
// norms and Lorentzian bells of RadPolyTrig, and the tensor-core tile of radial weights R^l_ij[c].
#ifndef LGAE_LEVEL_COMMON_CUH
#define LGAE_LEVEL_COMMON_CUH

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

#ifndef LGAE_TJ
#define LGAE_TJ 8   // with the component-wise mix and tile-wise partner features a 150-particle jet needs 43 KB per CTA (4: 8.74 vs 8.48 ms per 1024 jets)
#endif
constexpr int TJ = LGAE_TJ;  // neighbours per shared-memory tile of radial weights

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

}  // namespace lgae
#endif  // LGAE_LEVEL_COMMON_CUH
