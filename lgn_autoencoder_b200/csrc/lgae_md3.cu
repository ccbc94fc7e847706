// Forward of one maxdim-3 LGN level (max_zf = 1): the same level as lgae_level.cu computes at maxdim 2 -- aggregation over the
// fully connected graph, CG self product, concatenation [ag | node | sq] and per-irrep complex channel mix -- with the node
// irreps (0,0), (1,1), (2,0), (0,2), (2,2): 20 complex components per channel instead of 5.  Forward only (no saved state for an
// adjoint).  The CG algebra comes from the generated lgae_md3_tables.h (tools/gen_md3_tables.py, md3_layout.py).
//
// Two launches per level:
//   md3_enc_nbr_kernel (encoder) / md3_dec_nbr_kernel (decoder): the neighbour sums of every (particle i, channel c)
//       S0[a] = sum_j R0_ij z_j[a]                 (20 complex)
//       T[4a+d] = sum_j R1_ij z_j[a] Y_ij[d]       (80 complex; Y_ij = canon(p_i - p_j), formed per pair)
//     into a (B,N,C,100) complex buffer.  The encoder evaluates the radial weights R_ij tile by tile with the tensor-core tile of
//     the maxdim-2 kernels (radial_tile); its node components are split over gridDim.y groups of 5 so that the 25 complex
//     accumulators of a thread stay in registers.  The decoder's radial weights are the constants bias (1+i) (all-zero edge mask),
//     so its sums come from per-jet moments M = sum_j z_j and P = sum_j z_j (x) y_j:  S0 = R0 M,  T = R1 (M (x) y_i - P).
//   md3_mix_kernel: per block of 256 / C particles, output component by output component: every cat entry of the component (node
//     component, CG-contracted neighbour sum or CG self product, as the generated term lists say) into shared memory, then the mix
//     with the level's weights, which every (persistent) CTA keeps in shared memory.  The concatenation of one output component of
//     one row block is all that exists.
// No atomics; every sum runs in a fixed order, so results are bit-identical from run to run and independent of the batch.
#include <cstring>

#include "lgae_level_common.cuh"
#include "lgae_md3_tables.h"

namespace lgae {

constexpr int kGroup = 5;       // node components per neighbour-sum group (one gridDim.y slice of the encoder kernel)
constexpr int kNbr = 100;       // complex neighbour sums per (particle, channel): S0[20] | T[80]

LGAE_DEV int irrep_dim(int t) { return t == 0 ? 1 : (t == 1 ? 4 : (t == 4 ? 9 : 3)); }
LGAE_DEV int irrep_off(int t) { return t == 0 ? 0 : (t == 1 ? 1 : (t == 2 ? 5 : (t == 3 ? 8 : 11))); }

// Component `k` (0..19) of channel c of node row `row`: S (rows,C) | V (rows,C,4) | H (rows,C,15) complex.
LGAE_DEV cplx node_comp(const double* s, const double* v, const double* h, int64_t row, int C, int c, int k) {
    const int64_t rc = row * C + c;
    if (k == 0) return reinterpret_cast<const cplx*>(s)[rc];
    if (k < 5) return reinterpret_cast<const cplx*>(v)[rc * 4 + k - 1];
    return reinterpret_cast<const cplx*>(h)[rc * 15 + k - 5];
}

// ------------------------------------------------------------------------------------------------------------
// encoder neighbour sums
// ------------------------------------------------------------------------------------------------------------
struct NbrSmem {
    int p, msk, z, abc, rs, total;
};
__host__ __device__ inline NbrSmem nbr_smem(int N, int C, int KS) {
    NbrSmem s;
    int o = 0;
    s.p = o; o += 4 * N;
    s.msk = o; o += ((N + 7) / 8 + 2) & ~1;
    s.z = o; o += 2 * kGroup * TJ * C;     // the current tile's partner components of this group
    s.abc = o; o += (3 * 4 * KS + 1) & ~1;
    o = (o + 3) & ~3;
    s.rs = o; o += TJ * C * 32 * 4;        // radial weights of the tile
    s.total = o;
    return s;
}

// grid (B * ceil(N/32), groups), block 32 C: lane = particle i of the block, warp = channel c, blockIdx.y = components 5g..5g+4.
template <int NT, int KS>
__global__ void __launch_bounds__(256) md3_enc_nbr_kernel(const LevelArgs a, const double* h_in, double* nbr) {
    extern __shared__ __align__(128) double smem[];
    const int N = a.N, C = a.C;
    const int nib = (N + 31) / 32;
    const int b = blockIdx.x / nib, i0 = (blockIdx.x % nib) * 32, g = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, c = tid >> 5;
    const NbrSmem L = nbr_smem(N, C, KS);
    double* p_s = smem + L.p;
    uint8_t* msk_s = reinterpret_cast<uint8_t*>(smem + L.msk);
    cplx* z_s = reinterpret_cast<cplx*>(smem + L.z);
    double* abc_s = smem + L.abc;
    double* Rs = smem + L.rs;

    pdl_launch();
    double wf[KS][NT], bf[NT][2];
    load_radial_frags<NT, KS>(a, wf, bf, abc_s);   // parameters only
    pdl_wait();
    const double* pg = a.p + (int64_t)b * N * 4;
    for (int t = tid; t < 4 * N; t += blockDim.x) p_s[t] = pg[t];
    for (int t = tid; t < N; t += blockDim.x) msk_s[t] = a.node_mask ? a.node_mask[(int64_t)b * N + t] : (pg[4 * t] != 0.0);
    __syncthreads();

    const int i = i0 + lane;
    const bool live = i < N;
    double pi[4] = {0.0, 0.0, 0.0, 0.0};
    if (live) {
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) pi[mu] = p_s[4 * i + mu];
    }
    cplx S0[kGroup], T[kGroup][4];
#pragma unroll
    for (int k = 0; k < kGroup; ++k) {
        S0[k] = czero();
#pragma unroll
        for (int d = 0; d < 4; ++d) T[k][d] = czero();
    }
    for (int j0 = 0; j0 < N; j0 += TJ) {
        const int tj = min(TJ, N - j0);
        for (int t = tid; t < tj * C * kGroup; t += blockDim.x) {
            const int k = t % kGroup, r = t / kGroup;   // r = jj * C + cc
            z_s[t] = node_comp(a.s_in, a.v_in, h_in, (int64_t)b * N + j0 + r / C, C, r % C, kGroup * g + k);
        }
        radial_tile<NT, KS>(p_s, msk_s, N, C, i0, j0, tj, abc_s, wf, bf, Rs);
        __syncthreads();
        for (int jj = 0; jj < tj; ++jj) {
            const int j = j0 + jj;
            const double4 r = *reinterpret_cast<const double4*>(Rs + ((size_t)((jj * C + c) * 32 + lane)) * 4);
            const cplx R0 = cmake(r.x, r.y), R1 = cmake(r.z, r.w);
            double dp[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) dp[mu] = pi[mu] - p_s[4 * j + mu];
            cplx Y[4];
            canon_from_real(dp, Y);   // Y[0], Y[2] are real
            const cplx* zj = z_s + (jj * C + c) * kGroup;
#pragma unroll
            for (int k = 0; k < kGroup; ++k) {
                const cplx z = zj[k];
                cfma(S0[k], R0, z);
                const cplx t = cmul(R1, z);
                cfmar(T[k][0], t, Y[0].x);
                cfma(T[k][1], t, Y[1]);
                cfmar(T[k][2], t, Y[2].x);
                cfma(T[k][3], t, Y[3]);
            }
        }
        __syncthreads();   // z_s and Rs are refilled by the next tile
    }
    if (live) {
        cplx* dst = reinterpret_cast<cplx*>(nbr) + ((int64_t)(b * N + i) * C + c) * kNbr;
#pragma unroll
        for (int k = 0; k < kGroup; ++k) {
            const int comp = kGroup * g + k;
            dst[comp] = S0[k];
#pragma unroll
            for (int d = 0; d < 4; ++d) dst[20 + 4 * comp + d] = T[k][d];
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// decoder neighbour sums (closed form, LGNDecoder._level_closed_form)
// ------------------------------------------------------------------------------------------------------------
// grid B, one CTA per jet: the jet moments M (20) and P (80) per channel in shared memory (each a sum over j in particle order),
// then the sums of every particle.  ncomp: node components present (5 at level 0, 20 later).
__global__ void __launch_bounds__(256) md3_dec_nbr_kernel(const LevelArgs a, const double* h_in, double* nbr, int ncomp) {
    extern __shared__ __align__(128) double smem[];
    cplx* mom = reinterpret_cast<cplx*>(smem);   // [C][100]
    const int N = a.N, C = a.C, b = blockIdx.x;
    pdl_launch();
    pdl_wait();
    const cplx* y = reinterpret_cast<const cplx*>(a.p) + (int64_t)b * N * 4;
    for (int e = threadIdx.x; e < C * kNbr; e += blockDim.x) {
        const int c = e / kNbr, x = e % kNbr;
        const int comp = x < 20 ? x : (x - 20) >> 2, d = (x - 20) & 3;
        cplx acc = czero();
        if (comp < ncomp) {
            for (int j = 0; j < N; ++j) {
                const cplx zj = node_comp(a.s_in, a.v_in, h_in, (int64_t)b * N + j, C, c, comp);
                if (x < 20) acc = cadd(acc, zj);
                else cfma(acc, zj, y[4 * j + d]);
            }
        }
        mom[e] = acc;
    }
    __syncthreads();
    const int per = C * kNbr;
    for (int e = threadIdx.x; e < N * per; e += blockDim.x) {
        const int i = e / per, r = e % per, c = r / kNbr, x = r % kNbr;
        cplx v;
        if (x < 20) {
            const double b0 = a.theta[a.off_b0 + c];
            v = cmul(cmake(b0, b0), mom[c * kNbr + x]);
        } else {
            const double b1 = a.theta[a.off_b1 + c];
            const int comp = (x - 20) >> 2, d = (x - 20) & 3;
            v = cmul(cmake(b1, b1), csub(cmul(mom[c * kNbr + comp], y[4 * i + d]), mom[c * kNbr + x]));
        }
        reinterpret_cast<cplx*>(nbr)[((int64_t)b * N + i) * per + r] = v;
    }
}

// ------------------------------------------------------------------------------------------------------------
// concatenation pieces and channel mix
// ------------------------------------------------------------------------------------------------------------
struct MixArgs {
    const double* theta;
    int64_t off_mix[md3::kIrreps];     // (2, C', nblk * C) planar complex per irrep
    const double* s_in;                // (rows, C) complex
    const double* v_in;                // (rows, C, 4)
    const double* h_in;                // (rows, C, 15) or nullptr (level 0: (0,0) and (1,1) only)
    const double* nbr;                 // (rows, C, 100)
    double* s_pre;                     // (rows, C')
    double* v_out;                     // (rows, C', 4)
    double* h_out;                     // (rows, C', 15)
    int64_t rows;
    int C, Cout, variant;
    int nblk[md3::kIrreps];
};
// Particles per row block: 256 (particle, channel) pairs, one per thread of the first half of the CTA.
constexpr int kMixThreads = 512, kMixPairs = 256;
__host__ __device__ inline int mix_rows(int C) { return kMixPairs / C; }
// Shared memory (complex): the mix weights of all irreps (rows padded to ncol + 1 against bank conflicts), the node components of
// one row block, and one output component's concatenation of the row block ([r][ncol + 1], ncol <= 14 C).
__host__ __device__ inline int mix_w_cplx(int C, int Cout, const int* nblk) {
    int n = 0;
#pragma unroll
    for (int t = 0; t < md3::kIrreps; ++t) n += Cout * (nblk[t] * C + 1);
    return n;
}
__host__ __device__ inline int mix_smem_doubles(int C, int Cout, const int* nblk) {
    return 2 * (mix_w_cplx(C, Cout, nblk) + mix_rows(C) * C * md3::kComp + mix_rows(C) * (md3::kMaxBlocks * C + 1));
}

// Persistent: grid <= one CTA per SM; each loads the weights once and walks row blocks blockIdx.x, + gridDim.x, ...  Output
// component by output component: the cat entries of a (piece, component) are the work of whole warps (thread = particle x channel),
// so the term loop is uniform within a warp; then one thread per (particle, c') sums its column.
__global__ void __launch_bounds__(kMixThreads) md3_mix_kernel(const MixArgs a) {
    extern __shared__ __align__(128) double smem[];
    const int C = a.C, Cout = a.Cout, tid = threadIdx.x;
    const int rows_blk = mix_rows(C);
    cplx* w_s = reinterpret_cast<cplx*>(smem);
    cplx* z_s = w_s + mix_w_cplx(C, Cout, a.nblk);   // [r][c][20]
    cplx* cat_s = z_s + rows_blk * C * md3::kComp;   // [r][ncol + 1]
    pdl_launch();
    {   // weights: parameters only
        int o = 0;
#pragma unroll
        for (int t = 0; t < md3::kIrreps; ++t) {
            const int ncol = a.nblk[t] * C, n = Cout * ncol;
            const double* w = a.theta + a.off_mix[t];
            for (int e = tid; e < n; e += blockDim.x) w_s[o + (e / ncol) * (ncol + 1) + e % ncol] = cmake(w[e], w[n + e]);
            o += Cout * (ncol + 1);
        }
    }
    pdl_wait();
    const int ncomp = a.h_in ? md3::kComp : 5;
    const cplx* nbr = reinterpret_cast<const cplx*>(a.nbr);
    const unsigned char* bp = md3::md3_block_piece + a.variant * md3::kIrreps * md3::kMaxBlocks;
    const int64_t nblocks = (a.rows + rows_blk - 1) / rows_blk;
    const int pr = tid % kMixPairs, r = pr / C, c = pr % C, half = tid / kMixPairs;
    for (int64_t rb = blockIdx.x; rb < nblocks; rb += gridDim.x) {
        const int64_t r0 = rb * rows_blk;
        const int nr = (int)min((int64_t)rows_blk, a.rows - r0);
        __syncthreads();   // the previous row block is done with z_s
        for (int t = tid; t < nr * C * md3::kComp; t += blockDim.x) {
            const int rr = t / (C * md3::kComp), q = t % (C * md3::kComp), cc = q / md3::kComp, k = q % md3::kComp;
            z_s[t] = k < ncomp ? node_comp(a.s_in, a.v_in, a.h_in, r0 + rr, C, cc, k) : czero();
        }
        __syncthreads();
        const bool live = r < nr;
        const cplx* z = z_s + pr * md3::kComp;
        const cplx* s = nbr + ((r0 + (live ? r : 0)) * C + c) * kNbr;
        int wo = 0;
#pragma unroll
        for (int t = 0; t < md3::kIrreps; ++t) {   // unrolled: a.nblk and off_mix are indexed at compile time
            const int dt = irrep_dim(t), nb = a.nblk[t], ncol = nb * C, ld = ncol + 1;
            for (int m = 0; m < dt; ++m) {
                if (live) {
                    for (int blk = half; blk < nb; blk += kMixThreads / kMixPairs) {
                        const int p = bp[t * md3::kMaxBlocks + blk];
                        const int kind = md3::md3_piece_kind[p];
                        cplx v = czero();
                        if (kind == 0) {
                            v = z[md3::md3_piece_src[p] + m];
                        } else {
                            const int f = md3::md3_piece_first[p] + m;
                            const int k0 = md3::md3_term_range[f], k1 = md3::md3_term_range[f + 1];
                            for (int k = k0; k < k1; ++k) {
                                const double cf = md3::md3_term_c[k];
                                const int x = md3::md3_term_x[k];
                                if (kind == 3) cfmar(v, cmul(z[x], z[md3::md3_term_y[k]]), cf);
                                else if (kind == 2) cfmar(v, s[20 + x], cf);
                                else cfmar(v, s[x], cf);
                            }
                            if (kind == 1) v = cmul_1pi(v);   // the (0,0) edge feature R0 (1+i)
                        }
                        cat_s[r * ld + blk * C + c] = v;
                    }
                }
                __syncthreads();
                for (int e = tid; e < nr * Cout; e += blockDim.x) {
                    const int co = e % Cout, rr = e / Cout;
                    const cplx* x = cat_s + rr * ld;
                    const cplx* w = w_s + wo + co * ld;
                    cplx acc = czero();
                    for (int k = 0; k < ncol; ++k) cfma(acc, w[k], x[k]);
                    const int64_t row = r0 + rr;
                    if (t == 0) reinterpret_cast<cplx*>(a.s_pre)[row * Cout + co] = acc;
                    else if (t == 1) reinterpret_cast<cplx*>(a.v_out)[(row * Cout + co) * 4 + m] = acc;
                    else reinterpret_cast<cplx*>(a.h_out)[(row * Cout + co) * 15 + irrep_off(t) - 5 + m] = acc;
                }
                __syncthreads();   // cat_s is refilled for the next component
            }
            wo += Cout * ld;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
static int md3_pick_ks(int K) { return K <= 12 ? 3 : (K <= 20 ? 5 : (K <= 32 ? 8 : -1)); }

template <int NT, int KS>
static int launch_enc_nbr(const LevelArgs& a, const double* h_in, double* nbr, int groups, cudaStream_t st) {
    const size_t bytes = (size_t)nbr_smem(a.N, a.C, KS).total * sizeof(double);
    if (bytes > 227 * 1024) return LGAE_E_UNSUPPORTED;
    auto kern = md3_enc_nbr_kernel<NT, KS>;
    if (int rc = ensure_smem((const void*)kern, bytes)) return rc;
    const int nib = (a.N + 31) / 32;
    LaunchScope ls_("md3_nbr", st);
    launch_k(kern, dim3(a.B * nib, groups), dim3(32 * a.C), bytes, st, a, h_in, nbr);
    return check_launch("md3_nbr");
}

// Shared memory the level needs, 0 if it fits (checked before anything is launched).
int md3_level_check(const LgaeModelDesc* d) {
    for (int l = 0; l < d->n_levels; ++l) {
        const int C = d->channels[l];
        if (!d->is_decoder) {
            const int ks = md3_pick_ks(d->n_basis);
            if (ks < 0 || (size_t)nbr_smem(d->n_particles, C, ks).total * sizeof(double) > 227 * 1024) return LGAE_E_UNSUPPORTED;
        }
        const int variant = l == 0 ? 0 : (d->has_mlp ? 1 : 2);
        if ((size_t)mix_smem_doubles(C, d->channels[l + 1], md3::kNBlocks[variant]) * sizeof(double) > 227 * 1024) return LGAE_E_UNSUPPORTED;
    }
    return LGAE_OK;
}

// Neighbour-sum doubles of one level: (B,N,C,100) complex.
int64_t md3_nbr_doubles(const LgaeModelDesc* d, int level, int64_t batch) {
    return batch * d->n_particles * d->channels[level] * kNbr * 2;
}

// One maxdim-3 level: s_in / v_in / h_in (h_in == nullptr at level 0) -> s_pre (0,0), v_out (1,1), h_out (2,0)|(0,2)|(2,2).
// nbr: md3_nbr_doubles(d, level, batch) doubles of scratch.
int run_md3_level_fwd(const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y, const uint8_t* node_mask, int batch,
                      const double* s_in, const double* v_in, const double* h_in, double* nbr, double* s_pre, double* v_out, double* h_out,
                      cudaStream_t st) {
    if (!d || level < 0 || level >= d->n_levels) return LGAE_E_BADARG;
    if (batch <= 0) return LGAE_OK;
    LevelArgs a;
    memset(&a, 0, sizeof(a));
    a.theta = theta;
    a.off_a = d->off_rad_a[level]; a.off_b = d->off_rad_b[level]; a.off_c = d->off_rad_c[level];
    a.off_w0 = d->off_rad_w0[level]; a.off_b0 = d->off_rad_b0[level];
    a.off_w1 = d->off_rad_w1[level]; a.off_b1 = d->off_rad_b1[level];
    a.p = p_or_y; a.node_mask = node_mask; a.s_in = s_in; a.v_in = v_in;
    a.B = batch; a.N = d->n_particles; a.C = d->channels[level]; a.Cout = d->channels[level + 1]; a.K = d->n_basis;
    if (a.C < 1 || a.C > LGAE_MAX_CHANNELS || a.Cout < 1 || a.Cout > LGAE_MAX_CHANNELS) return LGAE_E_UNSUPPORTED;
    const int ncomp = level == 0 ? 5 : md3::kComp;
    if (!d->is_decoder) {
        const int nt = (4 * a.C + 7) / 8, ks = md3_pick_ks(a.K);
        int rc = LGAE_E_UNSUPPORTED;
#define LGAE_CASE(NTV, KSV) \
        if (nt == NTV && ks == KSV) rc = launch_enc_nbr<NTV, KSV>(a, h_in, nbr, ncomp / kGroup, st);
        LGAE_CASE(1, 3) LGAE_CASE(2, 3) LGAE_CASE(3, 3) LGAE_CASE(4, 3)
        LGAE_CASE(1, 5) LGAE_CASE(2, 5) LGAE_CASE(3, 5) LGAE_CASE(4, 5)
        LGAE_CASE(1, 8) LGAE_CASE(2, 8) LGAE_CASE(3, 8) LGAE_CASE(4, 8)
#undef LGAE_CASE
        if (rc != LGAE_OK) return rc;
    } else {
        const size_t bytes = (size_t)a.C * kNbr * 2 * sizeof(double);
        if (int rc = ensure_smem((const void*)md3_dec_nbr_kernel, bytes)) return rc;
        LaunchScope ls_("md3_dec_nbr", st);
        launch_k(md3_dec_nbr_kernel, dim3(batch), dim3(256), bytes, st, a, h_in, nbr, ncomp);
        if (int rc = check_launch("md3_dec_nbr")) return rc;
    }
    MixArgs m;
    memset(&m, 0, sizeof(m));
    m.theta = theta;
    m.off_mix[0] = d->off_mix00[level]; m.off_mix[1] = d->off_mix11[level];
    m.off_mix[2] = d->off_mix20[level]; m.off_mix[3] = d->off_mix02[level]; m.off_mix[4] = d->off_mix22[level];
    m.s_in = s_in; m.v_in = v_in; m.h_in = level == 0 ? nullptr : h_in; m.nbr = nbr;
    m.s_pre = s_pre; m.v_out = v_out; m.h_out = h_out;
    m.rows = (int64_t)batch * d->n_particles;
    m.C = a.C; m.Cout = a.Cout;
    m.variant = level == 0 ? 0 : (d->has_mlp ? 1 : 2);
    for (int t = 0; t < md3::kIrreps; ++t) m.nblk[t] = md3::kNBlocks[m.variant][t];
    const size_t bytes = (size_t)mix_smem_doubles(a.C, a.Cout, m.nblk) * sizeof(double);
    if (int rc = ensure_smem((const void*)md3_mix_kernel, bytes)) return rc;
    const int64_t nblocks = (m.rows + mix_rows(a.C) - 1) / mix_rows(a.C);
    const int grid = (int)(nblocks < sm_count() ? nblocks : sm_count());
    LaunchScope ls_("md3_mix", st);
    launch_k(md3_mix_kernel, dim3(grid), dim3(kMixThreads), bytes, st, m);
    return check_launch("md3_mix");
}

}  // namespace lgae
