// Gradients with respect to the inputs of the fused maxdim-2 path (DESIGN.md section 4e):
//   pgrad_level_kernel    one encoder level's contribution to dL/dp: the edge features R^1_ij Y_ij (Y_ij = canon(p_i - p_j)) and
//                         the radial weights' dependence on the pair norms n_ij, from the level adjoint's gA (adjoints of the
//                         neighbour sums), added into a (B,N,4) accumulator in level order;
//   pgrad_input_kernel    the input map (mass scalar sqrt|p^2| and canon(p)), the accumulated level terms and the input scale ->
//                         dL/dp4, written once;
//   chamfer_target_kernel dL/dtarget of the chamfer loss;
//   normalize_bwd_kernel  adjoint of normalize_p4 (overall max).
// fp64 throughout, no atomics: every output element has one owning thread and sums run in a fixed order, so the results do not
// depend on the batch size or the grid.
#include "lgae_common.cuh"

namespace lgae {

struct PGradArgs {
    const double* theta;
    int64_t off_a, off_b, off_c, off_w0, off_b0, off_w1, off_b1;
    const double* p;           // (B,N,4) the momenta the encoder read (input scale applied)
    const uint8_t* node_mask;  // (B,N) or nullptr (=> p[...,0] != 0)
    const double* s_in;        // (B,N,C,2)   node features entering the level
    const double* v_in;        // (B,N,C,4,2)
    const double* gA;          // (B,N,C,10) complex: adjoints of [A0V(4), A0S, A1Y(4), A1E]
    double* gp;                // (B,N,4) accumulator of dL/dp
    int B, N, C, K, ns;        // ns: slices of the partner range per particle
};

constexpr int PGRAD_THREADS = 128;

struct PGradSmem {
    int w, bias, abc, p, part, phi, dphi, msk, total;
};
__host__ __device__ inline PGradSmem pgrad_smem(int N, int C, int K, int ns) {
    PGradSmem s;
    int o = 0;
    s.w = o; o += 4 * C * K;              // stacked radial linear maps [col][k], col = l*2C + 2c + (re|im)
    s.bias = o; o += 4 * C;
    s.abc = o; o += 3 * K;
    s.p = o; o += 4 * N;
    s.part = o; o += 4 * N * ns;          // per-slice partial sums [(i*ns + s)*4 + mu]
    s.phi = o; o += K * PGRAD_THREADS;    // per-thread basis values and derivatives of the current pair, [k][thread]
    s.dphi = o; o += K * PGRAD_THREADS;
    s.msk = o; o += (N + 7) / 8;
    s.total = o;
    return s;
}

// One CTA per jet (persistent over jets), one thread per (particle i, slice of partners j).  For every ordered pair it takes both
// orientations at once -- i receiving from j and j receiving from i -- so that particle i's thread owns all of its terms:
//   dL/dR^l_ij + dL/dR^l_ji (role 1 of the level adjoint for both orientations; R_ij = R_ji) -> dL/dn_ij through the bell functions,
//   times dn_ij/dp_i = eta (p_i - p_j) / sqrt|s_ij|, only where the edge is live (node masks and n_ij != 0, as in the forward);
//   dL/dY_ij - dL/dY_ji through canon, for every pair (masked edges keep the bias radial weights).
// Self pairs contribute nothing (p_i - p_i does not depend on p_i).
__global__ void __launch_bounds__(PGRAD_THREADS) pgrad_level_kernel(const PGradArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int N = a.N, C = a.C, K = a.K, ns = a.ns, tid = threadIdx.x;
    const PGradSmem L = pgrad_smem(N, C, K, ns);
    double* w_s = smem + L.w;
    double* bias_s = smem + L.bias;
    double* abc_s = smem + L.abc;
    double* p_s = smem + L.p;
    double* part_s = smem + L.part;
    double* phi_s = smem + L.phi + tid;
    double* dphi_s = smem + L.dphi + tid;
    uint8_t* msk_s = reinterpret_cast<uint8_t*>(smem + L.msk);

    pdl_launch();
    for (int t = tid; t < 4 * C * K; t += blockDim.x) {
        const int col = t / K, k = t % K;
        w_s[t] = col < 2 * C ? a.theta[a.off_w0 + (int64_t)col * K + k] : a.theta[a.off_w1 + (int64_t)(col - 2 * C) * K + k];
    }
    for (int t = tid; t < 4 * C; t += blockDim.x) bias_s[t] = t < 2 * C ? a.theta[a.off_b0 + t] : a.theta[a.off_b1 + t - 2 * C];
    for (int t = tid; t < K; t += blockDim.x) {
        abc_s[t] = a.theta[a.off_a + t];
        abc_s[K + t] = a.theta[a.off_b + t];
        abc_s[2 * K + t] = a.theta[a.off_c + t];
    }
    pdl_wait();
    const cplx* S = reinterpret_cast<const cplx*>(a.s_in);
    const cplx* V = reinterpret_cast<const cplx*>(a.v_in);
    const cplx* G = reinterpret_cast<const cplx*>(a.gA);
    const int len = (N + ns - 1) / ns;
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        __syncthreads();   // the previous jet's partials are consumed
        for (int t = tid; t < 4 * N; t += blockDim.x) p_s[t] = a.p[(int64_t)b * N * 4 + t];
        for (int t = tid; t < N; t += blockDim.x)
            msk_s[t] = a.node_mask ? a.node_mask[(int64_t)b * N + t] != 0 : a.p[((int64_t)b * N + t) * 4] != 0.0;
        __syncthreads();
        for (int it = tid; it < N * ns; it += blockDim.x) {
            const int i = it / ns, sl = it % ns;
            const int j0 = sl * len, j1 = min(N, j0 + len);
            const int64_t ni = (int64_t)b * N + i;
            double acc[4] = {0.0, 0.0, 0.0, 0.0};
            for (int j = j0; j < j1; ++j) {
                if (j == i) continue;
                const int64_t nj = (int64_t)b * N + j;
                double d[4];
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) d[mu] = p_s[4 * i + mu] - p_s[4 * j + mu];
                cplx Y[4];
                canon_from_real(d, Y);
                const double d0 = Y[0].x, d3 = Y[2].x, ya_ = Y[1].x, yb_ = -Y[1].y;
                // pair norm exactly as the forward's pair_norm (lgae_level.cu)
                const double s = __dadd_rn(minkowski_sq(d[0], d[1], d[2], d[3]), 1e-16);
                const double rs = s != 0.0 ? __dsqrt_rn(fabs(s)) : 0.0;
                const double n = s != 0.0 ? __ddiv_rn(s, rs) : s;
                const bool live = msk_s[i] && msk_s[j] && n != 0.0;
                if (live) {
                    for (int k = 0; k < K; ++k) {
                        const double cn = abc_s[2 * K + k] * n;
                        const double r = 1.0 / (1.0 + cn * cn + 1e-16);
                        phi_s[k * PGRAD_THREADS] = fma(abc_s[K + k], r, abc_s[k]);
                        dphi_s[k * PGRAD_THREADS] = -2.0 * abc_s[K + k] * abc_s[2 * K + k] * cn * r * r;
                    }
                }
                cplx gy[4] = {czero(), czero(), czero(), czero()};   // sum_c (dL/dY_ij - dL/dY_ji)
                double gn = 0.0;                                       // dL/dn_ij + dL/dn_ji
                for (int c = 0; c < C; ++c) {
                    const cplx* gi = G + (ni * C + c) * 10;
                    const cplx* gj = G + (nj * C + c) * 10;
                    const cplx Si = S[ni * C + c], Sj = S[nj * C + c];
                    cplx Vi[4], Vj[4], gai[10], gaj[10];
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) { Vi[mu] = V[(ni * C + c) * 4 + mu]; Vj[mu] = V[(nj * C + c) * 4 + mu]; }
#pragma unroll
                    for (int e = 0; e < 10; ++e) { gai[e] = gi[e]; gaj[e] = gj[e]; }
                    // sum_mu conj(Y_mu) g_mu and eta(v, Y), as in the level adjoint's role 1
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
                    // q_mu: dL/dY_ij - dL/dY_ji with conj(R1) factored out
                    cplx ghi[4], ghj[4], q[4];
                    cghat(Vi, ghi);
                    cghat(Vj, ghj);
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) {
                        cplx t = cmulc(Sj, gai[5 + mu]);
                        cfmac(t, ghj[mu], gai[9]);
                        cplx u = cmulc(Si, gaj[5 + mu]);
                        cfmac(u, ghi[mu], gaj[9]);
                        q[mu] = csub(t, u);
                    }
                    cplx R1 = cmake(bias_s[2 * C + 2 * c], bias_s[2 * C + 2 * c + 1]);
                    if (live) {
                        // dL/dR of both orientations (Y_ji = -Y_ij)
                        cplx gR0 = cmulc(Sj, gai[4]);
                        cfmac(gR0, Si, gaj[4]);
#pragma unroll
                        for (int mu = 0; mu < 4; ++mu) { cfmac(gR0, Vj[mu], gai[mu]); cfmac(gR0, Vi[mu], gaj[mu]); }
                        cplx gR1 = cmulc(Sj, ydot(gai + 5));
                        cfmac(gR1, yeta(Vj), gai[9]);
                        cfmac(gR1, Si, cneg(ydot(gaj + 5)));
                        cfmac(gR1, cneg(yeta(Vi)), gaj[9]);
                        const double* w0r = w_s + (2 * c) * K;
                        const double* w0i = w0r + K;
                        const double* w1r = w_s + (2 * C + 2 * c) * K;
                        const double* w1i = w1r + K;
                        for (int k = 0; k < K; ++k) {
                            const double ph = phi_s[k * PGRAD_THREADS];
                            R1.x = fma(w1r[k], ph, R1.x);
                            R1.y = fma(w1i[k], ph, R1.y);
                            const double h = fma(gR0.x, w0r[k], fma(gR0.y, w0i[k], fma(gR1.x, w1r[k], gR1.y * w1i[k])));
                            gn = fma(h, dphi_s[k * PGRAD_THREADS], gn);
                        }
                    }
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) cfmac(gy[mu], R1, q[mu]);
                }
                // canon(d) = (d0, r(d1 - i d2), d3, -r(d1 + i d2)), r = 1/sqrt2  =>  dL/dd
                acc[0] += gy[0].x;
                acc[1] += LGAE_RSQRT2 * (gy[1].x - gy[3].x);
                acc[2] -= LGAE_RSQRT2 * (gy[1].y + gy[3].y);
                acc[3] += gy[2].x;
                if (live) {   // dn/dd = eta d / sqrt|s|
                    const double f = gn / rs;
                    acc[0] += f * d[0];
                    acc[1] -= f * d[1];
                    acc[2] -= f * d[2];
                    acc[3] -= f * d[3];
                }
            }
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) part_s[(i * ns + sl) * 4 + mu] = acc[mu];
        }
        __syncthreads();
        for (int t = tid; t < 4 * N; t += blockDim.x) {
            const int i = t >> 2, mu = t & 3;
            double* dst = a.gp + ((int64_t)b * N + i) * 4 + mu;
            double v = *dst;
            for (int sl = 0; sl < ns; ++sl) v += part_s[(i * ns + sl) * 4 + mu];
            *dst = v;
        }
    }
}

// The input map S_0[c] = w00[c] m, V_0[c] = w11[c] canon(p), m = sqrt|p^2| (enc_input_node, lgae_glue.cu), plus the level terms
// in gp; dL/dp4 = scale * dL/dp.  Where p^2 == 0 exactly the mass term is dropped (its derivative is 0 * inf there; DESIGN 4e).
__global__ void __launch_bounds__(256) pgrad_input_kernel(const double* theta, int64_t off00, int64_t off11, const double* p4, int64_t nodes,
                                                          int C, const double* gS, const double* gV, const double* gp, double scale,
                                                          double* g_p4) {
    pdl_launch();
    pdl_wait();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nodes) return;
    const double* p = p4 + 4 * t;
    double gm = 0.0;
    cplx gy[4] = {czero(), czero(), czero(), czero()};
    for (int c = 0; c < C; ++c) {
        const cplx w0 = cmake(theta[off00 + c], theta[off00 + C + c]), w1 = cmake(theta[off11 + c], theta[off11 + C + c]);
        const cplx g = reinterpret_cast<const cplx*>(gS)[t * C + c];
        gm = fma(w0.x, g.x, fma(w0.y, g.y, gm));
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) cfmac(gy[mu], w1, reinterpret_cast<const cplx*>(gV)[(t * C + c) * 4 + mu]);
    }
    double g[4];
    g[0] = gp[4 * t] + gy[0].x;
    g[1] = gp[4 * t + 1] + LGAE_RSQRT2 * (gy[1].x - gy[3].x);
    g[2] = gp[4 * t + 2] - LGAE_RSQRT2 * (gy[1].y + gy[3].y);
    g[3] = gp[4 * t + 3] + gy[2].x;
    const double s = minkowski_sq(p[0], p[1], p[2], p[3]);
    if (s != 0.0) {   // dm/dp = sign(s) eta p / m
        const double f = (s > 0.0 ? gm : -gm) / __dsqrt_rn(fabs(s));
        g[0] += f * p[0];
        g[1] -= f * p[1];
        g[2] -= f * p[2];
        g[3] -= f * p[3];
    }
#pragma unroll
    for (int mu = 0; mu < 4; ++mu) g_p4[4 * t + mu] = scale * g[mu];
}

// ------------------------------------------------------------------------------------------------------------
// chamfer target adjoint
// ------------------------------------------------------------------------------------------------------------
LGAE_DEV double get_real_x(int mode, double re, double im) {
    switch (mode) {
        case LGAE_GET_REAL_IMAG: return im;
        case LGAE_GET_REAL_SUM: return re + im;
        case LGAE_GET_REAL_MEAN: return (re + im) / 2;
        case LGAE_GET_REAL_NORM: return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im)), 1e-16));
        default: return re;
    }
}
// One CTA per jet: the nearest-neighbour indices of both directions as chamfer_kernel (lgae_glue.cu) finds them -- the same
// distances, the first index of the minimum -- then per target particle j, in a fixed order over i:
//   dL/dt_j = g_loss * ( -(x_{i2[j]} - t_j) - sum_{i : j1[i] = j} (x_i - t_j) )
__global__ void __launch_bounds__(128) chamfer_target_kernel(const double* recon, const double* target, int B, int N, int M,
                                                             const double* g_loss, double* g_target, int mode) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    double* x = smem;            // N*4
    double* t = x + 4 * N;       // M*4
    int* j1 = reinterpret_cast<int*>(t + 4 * M);   // N
    int* i2 = j1 + N;                               // M
    const int b = blockIdx.x, tid = threadIdx.x;
    const int64_t plane = (int64_t)B * N * 4;
    for (int k = tid; k < 4 * N; k += blockDim.x) x[k] = get_real_x(mode, recon[(int64_t)b * N * 4 + k], recon[plane + (int64_t)b * N * 4 + k]);
    for (int k = tid; k < 4 * M; k += blockDim.x) t[k] = target[(int64_t)b * M * 4 + k];
    __syncthreads();
    auto dist = [&](int i, int j) {
        double s = 0.0;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) { const double d = x[4 * i + mu] - t[4 * j + mu]; s += d * d; }
        return s;
    };
    for (int i = tid; i < N; i += blockDim.x) {
        double best = dist(i, 0);
        int bj = 0;
        for (int j = 1; j < M; ++j) { const double d = dist(i, j); if (d < best) { best = d; bj = j; } }
        j1[i] = bj;
    }
    for (int j = tid; j < M; j += blockDim.x) {
        double best = dist(0, j);
        int bi = 0;
        for (int i = 1; i < N; ++i) { const double d = dist(i, j); if (d < best) { best = d; bi = i; } }
        i2[j] = bi;
    }
    __syncthreads();
    const double scale = g_loss ? *g_loss : 1.0;
    for (int j = tid; j < M; j += blockDim.x) {
        double g[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) g[mu] = t[4 * j + mu] - x[4 * i2[j] + mu];
        for (int i = 0; i < N; ++i)
            if (j1[i] == j) {
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) g[mu] -= x[4 * i + mu] - t[4 * j + mu];
            }
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) g_target[((int64_t)b * M + j) * 4 + mu] = g[mu] * scale;
    }
}

// ------------------------------------------------------------------------------------------------------------
// normalize_p4 adjoint
// ------------------------------------------------------------------------------------------------------------
// out = p4 / f, f = max_i max_mu |p4_i,mu| + 1e-16 (normalize_kernel, lgae_glue.cu).  dL/df = g_factor - sum g_out p4 / f^2 reaches
// the maxima as torch's amax adjoint routes it: split evenly between the tied particles of the outer max and, inside each, between
// the tied components of the inner max; |x|' = sign(x) (0 at 0).  One CTA per jet; per-particle maxima in shared memory (N doubles).
__global__ void __launch_bounds__(128) normalize_bwd_kernel(const double* p4, int N, const double* g_out, const double* g_factor,
                                                            double* g_p4) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(16) double pm[];   // N
    __shared__ double scratch[32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const double* p = p4 + (int64_t)b * N * 4;
    double m = 0.0;
    for (int i = tid; i < N; i += blockDim.x) {
        const double v = fmax(fmax(fabs(p[4 * i]), fabs(p[4 * i + 1])), fmax(fabs(p[4 * i + 2]), fabs(p[4 * i + 3])));
        pm[i] = v;
        m = fmax(m, v);
    }
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) scratch[tid >> 5] = m;
    __syncthreads();
    double M = 0.0;
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) M = fmax(M, scratch[w]);
    const double f = M + 1e-16;
    __syncthreads();   // scratch is reused by the sums below
    double cnt = 0.0, gs = 0.0;
    for (int i = tid; i < N; i += blockDim.x) cnt += pm[i] == M ? 1.0 : 0.0;
    if (g_out)
        for (int k = tid; k < 4 * N; k += blockDim.x) gs = fma(g_out[(int64_t)b * N * 4 + k], p[k], gs);
    cnt = block_sum(cnt, scratch);
    __syncthreads();
    gs = block_sum(gs, scratch);
    __shared__ double bc[2];
    if (tid == 0) {
        bc[0] = (g_factor ? g_factor[b] : 0.0) - gs / (f * f);   // dL/df
        bc[1] = cnt;
    }
    __syncthreads();
    const double gf = bc[0] / bc[1];   // per tied particle
    for (int i = tid; i < N; i += blockDim.x) {
        int ties = 0;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) ties += fabs(p[4 * i + mu]) == pm[i] ? 1 : 0;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) {
            const int64_t k = (int64_t)b * N * 4 + 4 * i + mu;
            const double x = p[4 * i + mu];
            double g = g_out ? g_out[k] / f : 0.0;
            if (pm[i] == M && fabs(x) == pm[i] && x != 0.0) g += (x > 0.0 ? gf : -gf) / ties;
            g_p4[k] = g;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
static int pgrad_slices(int N) { const int s = (2 * PGRAD_THREADS + N - 1) / N; return s < 1 ? 1 : (s > N ? N : s); }
static size_t pgrad_bytes(const LgaeModelDesc* d, int level) {
    const int N = d->n_particles;
    return (size_t)pgrad_smem(N, d->channels[level], d->n_basis, pgrad_slices(N)).total * sizeof(double);
}

// LGAE_OK if the input-gradient kernels run this encoder (no GPU needed).
int pgrad_check(const LgaeModelDesc* d) {
    if (d->is_decoder || d->n_basis < 1 || d->n_basis > 32) return LGAE_E_UNSUPPORTED;
    for (int l = 0; l < d->n_levels; ++l)
        if (pgrad_bytes(d, l) > 227 * 1024) return LGAE_E_UNSUPPORTED;
    return LGAE_OK;
}

int run_pgrad_level(const LgaeModelDesc* d, int level, const double* theta, const double* p, const uint8_t* node_mask, int batch,
                    const double* s_in, const double* v_in, const double* gA, double* gp, cudaStream_t st) {
    PGradArgs a;
    a.theta = theta;
    a.off_a = d->off_rad_a[level]; a.off_b = d->off_rad_b[level]; a.off_c = d->off_rad_c[level];
    a.off_w0 = d->off_rad_w0[level]; a.off_b0 = d->off_rad_b0[level];
    a.off_w1 = d->off_rad_w1[level]; a.off_b1 = d->off_rad_b1[level];
    a.p = p; a.node_mask = node_mask; a.s_in = s_in; a.v_in = v_in; a.gA = gA; a.gp = gp;
    a.B = batch; a.N = d->n_particles; a.C = d->channels[level]; a.K = d->n_basis; a.ns = pgrad_slices(a.N);
    const size_t bytes = pgrad_bytes(d, level);
    if (bytes > 227 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)pgrad_level_kernel, bytes)) return rc;
    const int cap = 4 * sm_count(), grid = batch < cap ? batch : cap;
    LaunchScope ls_("pgrad_level", st);
    launch_k(pgrad_level_kernel, dim3(grid), dim3(PGRAD_THREADS), bytes, st, a);
    return check_launch("pgrad_level");
}

int run_pgrad_input(const LgaeModelDesc* d, const double* theta, const double* p, int batch, const double* gS, const double* gV,
                    const double* gp, double scale, double* g_p4, cudaStream_t st) {
    const int64_t nodes = (int64_t)batch * d->n_particles;
    LaunchScope ls_("pgrad_input", st);
    launch_k(pgrad_input_kernel, dim3((unsigned)((nodes + 255) / 256)), dim3(256), 0, st, theta, d->off_in00, d->off_in11, p, nodes,
             d->channels[0], gS, gV, gp, scale, g_p4);
    return check_launch("pgrad_input");
}

int run_chamfer_target_grad(const double* recon, const double* target, int B, int N, int M, int mode, const double* g_loss,
                            double* g_target, cudaStream_t st) {
    const size_t bytes = (size_t)(4 * N + 4 * M) * sizeof(double) + (size_t)(N + M) * sizeof(int);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)chamfer_target_kernel, bytes)) return rc;
    LaunchScope ls_("chamfer_target_grad", st);
    launch_k(chamfer_target_kernel, dim3(B), dim3(128), bytes, st, recon, target, B, N, M, g_loss, g_target, mode);
    return check_launch("chamfer_target_grad");
}

int run_normalize_bwd(const double* p4, int B, int N, const double* g_out, const double* g_factor, double* g_p4, cudaStream_t st) {
    const size_t bytes = (size_t)N * sizeof(double);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)normalize_bwd_kernel, bytes)) return rc;
    LaunchScope ls_("normalize_p4_bwd", st);
    launch_k(normalize_bwd_kernel, dim3(B), dim3(128), bytes, st, p4, N, g_out, g_factor, g_p4);
    return check_launch("normalize_p4_bwd");
}

}  // namespace lgae
