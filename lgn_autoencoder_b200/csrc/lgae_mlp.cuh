// CGMLP (lgn/models/lgn_levels.py:191-227): the scalar MLP applied to every particle's (0,0) features,
// rows = B*N, re/im interleaved on the feature axis: Linear(2C'->w), [Linear(w->w)] x (hidden-1), Linear(w->2C'),
// an activation after all but the last (LGAE_ACT_*: LeakyReLU(0.01) by default).  This is the one genuinely dense GEMM
// chain of the LGAE ((B*N) x w x w, fp64), so it runs on the fp64 tensor-core MMA (DMMA m8n8k4).
//
// Both kernels keep the weights of ALL layers resident in shared memory (<= 98 KB at w = 48), staged once per CTA in
// MMA-fragment order, so the layer chain of a row group runs without any block-wide barrier.
//
// Forward: a warp owns 8 rows at a time and keeps them in registers through the whole chain.  The accumulator
// fragment of layer l (row g, columns 2q,2q+1 of every 8-column tile) is reused directly as the A operand of
// layer l+1 by enumerating the reduction index in the order the fragments already have (k-step (tile, e) <->
// column 8*tile + 2q + e), so no shuffles or shared-memory round trips are needed between layers.
// Backward: a CTA owns a contiguous slab of rows.  Per layer, the data gradient uses the same register trick with
// the transposed weights; the weight gradient dW = dZ^T H is a second MMA contraction over the slab's rows with dZ
// and H staged in shared memory, computed by dedicated warps as register-blocked tile blocks, and the result goes
// straight to the CTA's row of parameter-gradient partials.
//
// This header holds the kernels and their launchers; lgae_mlp.cu packs the weights and dispatches.
#pragma once

#include "lgae_common.cuh"

namespace lgae {

struct MlpArgs {
    const double* theta;
    const double* wpack;   // fragment-ordered weights of all layers (mlp_pack_kernel): [forward order | transposed order]
    int64_t off_w[LGAE_MAX_LINEAR], off_b[LGAE_MAX_LINEAR];
    int n_lin;   // number of Linear layers (hidden + 1)
    int nin;     // 2C'
    int width;   // hidden width w
    const double* x;  // (rows, nin)
    double* acts;     // (n_lin-1, rows, 8*NTW)
    double* y;        // (rows, nin)
    int64_t rows;
    int64_t rows_per_cta;  // backward: slab of rows owned by a CTA (multiple of 8)
    const double* g_y;
    double* g_x;
    double* part;          // (gridDim.x, part_stride) per-CTA rows of parameter-gradient partials
    int64_t part_stride;
    int64_t po_w[LGAE_MAX_LINEAR], po_b[LGAE_MAX_LINEAR];   // column offsets inside a row
    double slope;
};

constexpr int MLP_THREADS = 256;
#ifndef LGAE_MLP_FWD_MT
#define LGAE_MLP_FWD_MT 2     // row groups (of 8 rows) a warp of the forward kernel carries through the chain at a time
#endif
#ifndef LGAE_MLP_FWD_CTAS
#define LGAE_MLP_FWD_CTAS 1   // resident CTAs per SM the forward kernel is compiled and launched for
#endif
constexpr int MLP_BWD_ROWS = 128;   // rows of a slab processed at once by the backward kernel (16 row groups)

// Doubles of fragment-ordered weights of layer l (tiles padded to 8).
__host__ __device__ inline int mlp_layer_frag(int l, int n_lin, int NTW, int NTI) {
    const int kt = l == 0 ? NTI : NTW, no = l == n_lin - 1 ? NTI : NTW;
    return kt * 2 * no * 32;
}

// Hidden-layer activation (LGAE_ACT_*) and its derivative.  The derivative is taken from the activation's output y, which is
// what the forward saves in `acts`, so every activation shares one workspace layout.  Padded columns of a layer (beyond its
// width) may carry a non-zero activation (sigmoid(0) = 0.5); the zero-padded weights of the next layer cancel them.
template <int ACT>
LGAE_DEV double mlp_act(double x, double slope) {
    if constexpr (ACT == LGAE_ACT_LEAKYRELU) return leaky(x, slope);
    else if constexpr (ACT == LGAE_ACT_RELU) return x > 0.0 ? x : 0.0;
    else if constexpr (ACT == LGAE_ACT_ELU) return x > 0.0 ? x : expm1(x);
    else if constexpr (ACT == LGAE_ACT_SIGMOID) return 1.0 / (1.0 + exp(-x));
    else if constexpr (ACT == LGAE_ACT_LOGSIGMOID) return fmin(x, 0.0) - log1p(exp(-fabs(x)));   // no overflow for x << 0
    else if constexpr (ACT == LGAE_ACT_TANH) return tanh(x);
    else {
        static_assert(ACT == LGAE_ACT_ATAN, "unknown activation");
        return atan(x);
    }
}
template <int ACT>
LGAE_DEV double mlp_act_grad(double y, double slope) {
    if constexpr (ACT == LGAE_ACT_LEAKYRELU) return y > 0.0 ? 1.0 : slope;
    else if constexpr (ACT == LGAE_ACT_RELU) return y > 0.0 ? 1.0 : 0.0;
    else if constexpr (ACT == LGAE_ACT_ELU) return y > 0.0 ? 1.0 : y + 1.0;        // exp(x) = expm1(x) + 1
    else if constexpr (ACT == LGAE_ACT_SIGMOID) return y * (1.0 - y);
    else if constexpr (ACT == LGAE_ACT_LOGSIGMOID) return -expm1(y);               // sigmoid(-x) = 1 - exp(y)
    else if constexpr (ACT == LGAE_ACT_TANH) return 1.0 - y * y;
    else {
        static_assert(ACT == LGAE_ACT_ATAN, "unknown activation");
        // 1 / (1 + x^2) = cos^2(atan x).  cospi: |y| < pi/2, and cos's slow-path argument reduction would need a stack frame
        const double c = cospi(y * 0.31830988618379067154);
        return c * c;
    }
}

// MT row groups advance together so that MT * NO independent accumulator chains are in flight (the fp64 MMA has a long
// dependent-issue latency; a single group's NO chains leave the pipe idle).
template <int MT, int KT, int NO>
LGAE_DEV void layer_mma(const double (&act)[MT][KT][2], double (&acc)[MT][NO][2], const double* Wp, int q, int g) {
#pragma unroll
    for (int kt = 0; kt < KT; ++kt)
#pragma unroll
        for (int e = 0; e < 2; ++e)
#pragma unroll
            for (int nt = 0; nt < NO; ++nt) {
                const double bv = Wp[((kt * 2 + e) * NO + nt) * 32 + q * 8 + g];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) dmma(acc[mt][nt][0], acc[mt][nt][1], act[mt][kt][e], bv);
            }
}

// ------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------
template <int NTW, int NTI, int ACT>
__global__ void __launch_bounds__(MLP_THREADS, LGAE_MLP_FWD_CTAS) mlp_fwd_kernel(const MlpArgs a) {
    extern __shared__ __align__(128) double smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    constexpr int WP = 8 * NTW;
    const int last = a.n_lin - 1;
    // ---- all layers' weights and biases, once per CTA ----
    pdl_launch();
    double* bias_s = smem;                 // n_lin * WP
    double* w_s = smem + a.n_lin * WP;
    {
        int wtotal = 0;
        for (int l = 0; l <= last; ++l) {
            const int nout = l == last ? a.nin : a.width;
            wtotal += mlp_layer_frag(l, a.n_lin, NTW, NTI);
            for (int t = tid; t < WP; t += blockDim.x) bias_s[l * WP + t] = t < nout ? a.theta[a.off_b[l] + t] : 0.0;
        }
        // one TMA bulk copy brings all layers' fragments (<= 98 KB) into shared memory.  It is issued BEFORE the dependency
        // wait: the packed weights are written by mlp_pack_kernel, which never releases its dependents early, so they are
        // complete before any later kernel of the stream can start -- the copy overlaps the predecessor's tail
        __shared__ uint64_t mbar;
        if (tid == 0) mbar_init(&mbar, 1);
        __syncthreads();
        if (tid == 0) {
            mbar_expect_tx(&mbar, (unsigned)(wtotal * sizeof(double)));
            bulk_g2s(w_s, a.wpack, (unsigned)(wtotal * sizeof(double)), &mbar);
        }
        pdl_wait();   // the rows come from the previous kernel of the step
        mbar_wait(&mbar, 0);
    }
    __syncthreads();
    // ---- row groups of 8: a contiguous range per CTA, each warp takes MT = 2 consecutive groups at a time ----
    constexpr int MT = LGAE_MLP_FWD_MT;
    const int64_t ngroups = (a.rows + 7) / 8;
    const int64_t per_cta = (ngroups + gridDim.x - 1) / gridDim.x;
    const int64_t g_begin = (int64_t)blockIdx.x * per_cta, g_end = g_begin + per_cta < ngroups ? g_begin + per_cta : ngroups;
    for (int64_t grp = g_begin + MT * warp; grp < g_end; grp += MT * nwarps) {
        int64_t row[MT];
        bool ok[MT];
        double in0[MT][NTI][2];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            row[mt] = (grp + mt) * 8 + g;
            ok[mt] = grp + mt < g_end && row[mt] < a.rows;
#pragma unroll
            for (int nt = 0; nt < NTI; ++nt) {
                const int col = 8 * nt + 2 * q;
                double2 v = make_double2(0.0, 0.0);
                if (ok[mt] && col < a.nin) v = *reinterpret_cast<const double2*>(a.x + row[mt] * a.nin + col);
                in0[mt][nt][0] = v.x;
                in0[mt][nt][1] = v.y;
            }
        }
        double act[MT][NTW][2], acc[MT][NTW][2];
        const double* wl = w_s;
        // first layer: nin -> w
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) { acc[mt][nt][0] = bias_s[8 * nt + 2 * q]; acc[mt][nt][1] = bias_s[8 * nt + 2 * q + 1]; }
        layer_mma<MT, NTI, NTW>(in0, acc, wl, q, g);
        wl += NTI * 2 * NTW * 32;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) {
                act[mt][nt][0] = mlp_act<ACT>(acc[mt][nt][0], a.slope);
                act[mt][nt][1] = mlp_act<ACT>(acc[mt][nt][1], a.slope);
                if (ok[mt]) *reinterpret_cast<double2*>(a.acts + row[mt] * WP + 8 * nt + 2 * q) = make_double2(act[mt][nt][0], act[mt][nt][1]);
            }
        // hidden layers: w -> w
        for (int l = 1; l < last; ++l) {
            const double* bl = bias_s + l * WP;
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) { acc[mt][nt][0] = bl[8 * nt + 2 * q]; acc[mt][nt][1] = bl[8 * nt + 2 * q + 1]; }
            layer_mma<MT, NTW, NTW>(act, acc, wl, q, g);
            wl += NTW * 2 * NTW * 32;
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) {
                    act[mt][nt][0] = mlp_act<ACT>(acc[mt][nt][0], a.slope);
                    act[mt][nt][1] = mlp_act<ACT>(acc[mt][nt][1], a.slope);
                    if (ok[mt])
                        *reinterpret_cast<double2*>(a.acts + ((int64_t)l * a.rows + row[mt]) * WP + 8 * nt + 2 * q) =
                            make_double2(act[mt][nt][0], act[mt][nt][1]);
                }
        }
        // last layer: w -> nin, no activation
        double out[MT][NTI][2];
        const double* bl = bias_s + last * WP;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < NTI; ++nt) { out[mt][nt][0] = bl[8 * nt + 2 * q]; out[mt][nt][1] = bl[8 * nt + 2 * q + 1]; }
        layer_mma<MT, NTW, NTI>(act, out, wl, q, g);
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < NTI; ++nt) {
                const int col = 8 * nt + 2 * q;
                if (ok[mt] && col < a.nin) *reinterpret_cast<double2*>(a.y + row[mt] * a.nin + col) = make_double2(out[mt][nt][0], out[mt][nt][1]);
            }
    }
}

// ------------------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------------------
// Warp-specialised: warps 0-3 ("dW warps") own the weight-gradient tiles of a layer as register-blocked (<= 3 x 3) tile
// blocks -- each k-step loads 3 + 3 fragments for 9 MMAs instead of 2 per MMA, which is what keeps the contraction off the
// shared-memory bandwidth limit -- plus the bias gradient and the staging of the layer inputs H_l (prefetched one layer
// ahead); warps 4-7 ("row warps") own the slab's row groups: they carry dZ through the layer chain in registers (data
// gradient with the transposed weights) and publish it to shared memory for the dW warps.  Both run concurrently between
// the two barriers of a layer, one of each kind per SM sub-partition.
template <int NTW, int NTI, int ACT>
__global__ void __launch_bounds__(MLP_THREADS, 1) mlp_bwd_kernel(const MlpArgs a) {
    extern __shared__ __align__(128) double smem[];
    constexpr int WS = 8 * NTW + 4;                 // padded row stride of the staged tiles (conflict-free fragment loads)
    constexpr int WP = 8 * NTW;
    constexpr int NWH = 4;                          // warps per role
    constexpr int GMAX = MLP_BWD_ROWS / 8 / NWH;    // row groups per row warp per chunk (4)
    constexpr int MB = (NTW + 1) / 2;               // tile-block edge (3 for w = 48)
    constexpr int PERD = (MLP_BWD_ROWS * WP / 4 + 32 * NWH - 1) / (32 * NWH);   // double4 of H per dW-warp thread
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const bool dw_role = warp < NWH;
    const int wi = warp & (NWH - 1);
    const int last = a.n_lin - 1;
    double* w_s = smem;
    int wtotal = 0;
    for (int l = 0; l <= last; ++l) wtotal += mlp_layer_frag(l, a.n_lin, NTW, NTI);
    double* dz_s = w_s + wtotal;                    // MLP_BWD_ROWS * WS
    double* h_s = dz_s + MLP_BWD_ROWS * WS;         // MLP_BWD_ROWS * WS
    double* bred = h_s + MLP_BWD_ROWS * WS;         // 2 * NWH * WP : per-row-warp column sums of dZ, double-buffered by layer parity
    pdl_launch();
    {
        // (weights staged before the dependency wait: see mlp_fwd_kernel)
        __shared__ uint64_t mbar;
        if (tid == 0) mbar_init(&mbar, 1);
        __syncthreads();
        if (tid == 0) {
            mbar_expect_tx(&mbar, (unsigned)(wtotal * sizeof(double)));
            bulk_g2s(w_s, a.wpack + wtotal, (unsigned)(wtotal * sizeof(double)), &mbar);
        }
        pdl_wait();
        mbar_wait(&mbar, 0);
    }
    double* part = a.part + (int64_t)blockIdx.x * a.part_stride;
    const int64_t slab0 = (int64_t)blockIdx.x * a.rows_per_cta;
    const int64_t slab1 = slab0 + a.rows_per_cta < a.rows ? slab0 + a.rows_per_cta : a.rows;
    bool first = true;   // first chunk of the slab: partials are stored, later chunks accumulate
    // The two roles run separate copies of the chunk / layer loops (disjoint register live ranges) and meet at the same
    // two block-wide barriers per layer (bar.sync 0 from either branch).
    auto cta_sync = [] { asm volatile("bar.sync 0;" ::: "memory"); };
    if (dw_role) {
        for (int64_t r0 = slab0;; r0 += MLP_BWD_ROWS) {
            const int crows = (int)(slab1 - r0 < MLP_BWD_ROWS ? (slab1 > r0 ? slab1 - r0 : 0) : MLP_BWD_ROWS);
            const int ksteps = ((crows + 7) / 8) * 2;   // MMA k-steps (4 rows each) covering the chunk; even
            // the saved activations feeding layer l (its input H_l), fetched one layer ahead; the chunk's rows are one
            // contiguous run of crows * WP doubles
            double4 hv[PERD];
            auto fetch_h = [&](int layer) {
                const double4* src = reinterpret_cast<const double4*>(a.acts + ((int64_t)(layer - 1) * a.rows + r0) * WP);
#pragma unroll
                for (int j = 0; j < PERD; ++j) {
                    const int idx = wi * 32 + lane + 32 * NWH * j;
                    hv[j] = make_double4(0.0, 0.0, 0.0, 0.0);
                    if (idx < ksteps * 4 * (WP / 4) && r0 + idx / (WP / 4) < slab1) hv[j] = src[idx];
                }
            };
            if (last > 0) fetch_h(last);
            int nout_prev = 0, l_prev = -1;
            for (int l = last; l >= 0; --l) {
                const int nout = l == last ? a.nin : a.width, nink = l == 0 ? a.nin : a.width;
                const int NOt = l == last ? NTI : NTW, KIt = l == 0 ? NTI : NTW;
                cta_sync();   // the previous layer's readers of dz_s / h_s are done; its bias partials are complete
                if (l_prev >= 0)
                    for (int n = tid; n < nout_prev; n += 32 * NWH) {
                        double s = 0.0;
#pragma unroll
                        for (int w = 0; w < NWH; ++w) s += bred[((l_prev & 1) * NWH + w) * WP + n];
                        double* dst = part + a.po_b[l_prev] + n;
                        dst[0] = first ? s : dst[0] + s;
                    }
                // ---- stage the layer input H_l, then start fetching H_{l-1} ----
                if (l > 0) {
#pragma unroll
                    for (int j = 0; j < PERD; ++j) {
                        const int idx = wi * 32 + lane + 32 * NWH * j, rr = idx / (WP / 4), c4 = idx % (WP / 4);
                        if (idx < ksteps * 4 * (WP / 4)) *reinterpret_cast<double4*>(h_s + rr * WS + 4 * c4) = hv[j];
                    }
                    if (l > 1) fetch_h(l - 1);
                } else {
                    for (int idx = wi * 32 + lane; idx < ksteps * 4 * 8 * NTI; idx += 32 * NWH) {
                        const int rr = idx / (8 * NTI), cc = idx % (8 * NTI);
                        const int64_t row = r0 + rr;
                        h_s[rr * WS + cc] = (row < slab1 && cc < a.nin) ? a.x[row * a.nin + cc] : 0.0;
                    }
                }
                cta_sync();
                __syncwarp();
                // (the bias gradient -- column sums of dZ -- comes from the row warps, which hold dZ in registers: bred[l & 1])
                // ---- weight gradient dW[n][k] = sum_rows dZ[row][n] H[row][k]: this warp's (<= MB x MB) tile block ----
                const int MBo = (NOt + 1) / 2, NBo = (KIt + 1) / 2;
                const int m0 = (wi >> 1) * MBo, n0 = (wi & 1) * NBo;
                const int mcnt = NOt - m0 < MBo ? NOt - m0 : MBo, ncnt = KIt - n0 < NBo ? KIt - n0 : NBo;
                if (mcnt > 0 && ncnt > 0) {
                    double cw[2][MB][MB][2];   // even / odd k-steps: twice the independent MMA chains
#pragma unroll
                    for (int h = 0; h < 2; ++h)
#pragma unroll
                        for (int i = 0; i < MB; ++i)
#pragma unroll
                            for (int j = 0; j < MB; ++j) cw[h][i][j][0] = cw[h][i][j][1] = 0.0;
                    for (int ks = 0; ks < ksteps; ks += 2) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const double* dr = dz_s + (4 * (ks + h) + q) * WS + 8 * m0 + g;
                            const double* hr = h_s + (4 * (ks + h) + q) * WS + 8 * n0 + g;
                            double af[MB], bf[MB];
#pragma unroll
                            for (int i = 0; i < MB; ++i) af[i] = i < mcnt ? dr[8 * i] : 0.0;
#pragma unroll
                            for (int j = 0; j < MB; ++j) bf[j] = j < ncnt ? hr[8 * j] : 0.0;
#pragma unroll
                            for (int i = 0; i < MB; ++i)
#pragma unroll
                                for (int j = 0; j < MB; ++j)
                                    if (i < mcnt && j < ncnt) dmma(cw[h][i][j][0], cw[h][i][j][1], af[i], bf[j]);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < MB; ++i)
#pragma unroll
                        for (int j = 0; j < MB; ++j) {
                            if (i >= mcnt || j >= ncnt) continue;
                            const int n = 8 * (m0 + i) + g, k = 8 * (n0 + j) + 2 * q;
                            const double c0 = cw[0][i][j][0] + cw[1][i][j][0], c1 = cw[0][i][j][1] + cw[1][i][j][1];
                            if (n < nout) {
                                double* dst = part + a.po_w[l] + (int64_t)n * nink + k;
                                if (k < nink) dst[0] = first ? c0 : dst[0] + c0;
                                if (k + 1 < nink) dst[1] = first ? c1 : dst[1] + c1;
                            }
                        }
                }
                nout_prev = nout;
                l_prev = l;
            }
            cta_sync();   // bias partials of the first layer
            for (int n = tid; n < nout_prev; n += 32 * NWH) {
                double s = 0.0;
#pragma unroll
                for (int w = 0; w < NWH; ++w) s += bred[w * WP + n];   // layer 0: parity 0
                double* dst = part + a.po_b[0] + n;
                dst[0] = first ? s : dst[0] + s;
            }
            first = false;
            if (r0 + MLP_BWD_ROWS >= slab1) break;
        }
    } else {
        for (int64_t r0 = slab0;; r0 += MLP_BWD_ROWS) {
            const int crows = (int)(slab1 - r0 < MLP_BWD_ROWS ? (slab1 > r0 ? slab1 - r0 : 0) : MLP_BWD_ROWS);
            const int ksteps = ((crows + 7) / 8) * 2;
            // gradient wrt the output of the last layer, accumulator-fragment layout, for the warp's row groups
            double dz[GMAX][NTW][2];
#pragma unroll
            for (int u = 0; u < GMAX; ++u) {
                const int64_t row = r0 + (wi + NWH * u) * 8 + g;
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) {
                    dz[u][nt][0] = dz[u][nt][1] = 0.0;
                    if (nt < NTI) {
                        const int col = 8 * nt + 2 * q;
                        if (row < slab1 && col < a.nin) {
                            const double2 v = *reinterpret_cast<const double2*>(a.g_y + row * a.nin + col);
                            dz[u][nt][0] = v.x;
                            dz[u][nt][1] = v.y;
                        }
                    }
                }
            }
            const double* wl = w_s + wtotal;
            for (int l = last; l >= 0; --l) {
                const int NOt = l == last ? NTI : NTW, KIt = l == 0 ? NTI : NTW;
                wl -= mlp_layer_frag(l, a.n_lin, NTW, NTI);
                cta_sync();
                // ---- publish dZ_l of this warp's row groups ----
#pragma unroll
                for (int u = 0; u < GMAX; ++u) {
                    const int rl = (wi + NWH * u) * 8;
                    if (rl < ksteps * 4) {
#pragma unroll
                        for (int nt = 0; nt < NTW; ++nt)
                            if (nt < NOt)
                                *reinterpret_cast<double2*>(dz_s + (rl + g) * WS + 8 * nt + 2 * q) = make_double2(dz[u][nt][0], dz[u][nt][1]);
                    }
                }
                // ---- bias gradient of layer l: column sums of this warp's rows of dZ_l, straight from the registers (padding rows
                //      carry zeros): add the warp's row groups, then a butterfly over the 8 rows of the fragment ----
                {
                    double* bl = bred + ((l & 1) * NWH + wi) * WP;
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt) {
                        if (nt < NOt) {
                            double c0 = 0.0, c1 = 0.0;
#pragma unroll
                            for (int u = 0; u < GMAX; ++u) { c0 += dz[u][nt][0]; c1 += dz[u][nt][1]; }
#pragma unroll
                            for (int o = 4; o < 32; o <<= 1) {
                                c0 += __shfl_xor_sync(0xffffffffu, c0, o);
                                c1 += __shfl_xor_sync(0xffffffffu, c1, o);
                            }
                            if (g == 0) *reinterpret_cast<double2*>(bl + 8 * nt + 2 * q) = make_double2(c0, c1);
                        }
                    }
                }
                cta_sync();
                // ---- data gradient: Gin[row][k] = sum_n dZ[row][n] W[n][k], then through the activation of layer l-1; two row
                //      groups advance together (2 * KIt independent chains) ----
#pragma unroll
                for (int up = 0; up < GMAX; up += 2) {
                    if ((wi + NWH * up) * 8 >= ksteps * 4) continue;   // both groups of the pair are padding
                    double gin[2][NTW][2];
#pragma unroll
                    for (int u = 0; u < 2; ++u)
#pragma unroll
                        for (int kt = 0; kt < NTW; ++kt) gin[u][kt][0] = gin[u][kt][1] = 0.0;
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt) {
                        if (nt < NOt) {
#pragma unroll
                            for (int e = 0; e < 2; ++e)
#pragma unroll
                                for (int kt = 0; kt < NTW; ++kt)
                                    if (kt < KIt) {
                                        const double bv = wl[((nt * 2 + e) * KIt + kt) * 32 + q * 8 + g];
#pragma unroll
                                        for (int u = 0; u < 2; ++u) dmma(gin[u][kt][0], gin[u][kt][1], dz[up + u][nt][e], bv);   // padding groups carry zeros
                                    }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const int rl = (wi + NWH * (up + u)) * 8;
                        if (rl >= ksteps * 4) continue;
                        if (l > 0) {
#pragma unroll
                            for (int kt = 0; kt < NTW; ++kt) {
                                const double2 h = *reinterpret_cast<const double2*>(h_s + (rl + g) * WS + 8 * kt + 2 * q);
                                dz[up + u][kt][0] = gin[u][kt][0] * mlp_act_grad<ACT>(h.x, a.slope);
                                dz[up + u][kt][1] = gin[u][kt][1] * mlp_act_grad<ACT>(h.y, a.slope);
                            }
                        } else if (a.g_x) {
                            const int64_t row = r0 + rl + g;
#pragma unroll
                            for (int kt = 0; kt < NTI; ++kt) {
                                const int col = 8 * kt + 2 * q;
                                if (row < slab1 && col < a.nin)
                                    *reinterpret_cast<double2*>(a.g_x + row * a.nin + col) = make_double2(gin[u][kt][0], gin[u][kt][1]);
                            }
                        }
                    }
                }
            }
            cta_sync();   // pairs with the dW warps' barrier before the last bias reduction
            if (r0 + MLP_BWD_ROWS >= slab1) break;
        }
    }
}

inline int mlp_frag_total(int n_lin, int NTW, int NTI) {
    int t = 0;
    for (int l = 0; l < n_lin; ++l) t += mlp_layer_frag(l, n_lin, NTW, NTI);
    return t;
}

int mlp_bwd_grid();

template <int NTW, int NTI, int ACT>
int launch_mlp(MlpArgs& a, bool bwd, cudaStream_t st) {
    const int wtotal = mlp_frag_total(a.n_lin, NTW, NTI);
    if (!bwd) {
        const size_t bytes = (size_t)(wtotal + a.n_lin * 8 * NTW) * sizeof(double);
        if (bytes > 227 * 1024) return LGAE_E_UNSUPPORTED;
        auto kern = mlp_fwd_kernel<NTW, NTI, ACT>;
        if (int rc = ensure_smem((const void*)kern, bytes)) return rc;
        const int64_t ngroups = (a.rows + 7) / 8;
        const int cap = LGAE_MLP_FWD_CTAS * sm_count();
        const int grid = (int)(ngroups < cap ? ngroups : cap);
        LaunchScope ls_("mlp_fwd", st);
        launch_k(kern, dim3(grid), dim3(MLP_THREADS), bytes, st, a);
        return check_launch("mlp_fwd");
    }
    const size_t bytes = (size_t)(wtotal + 2 * MLP_BWD_ROWS * (8 * NTW + 4) + 2 * 4 * 8 * NTW) * sizeof(double);
    if (bytes > 227 * 1024) return LGAE_E_UNSUPPORTED;
    auto kern = mlp_bwd_kernel<NTW, NTI, ACT>;
    if (int rc = ensure_smem((const void*)kern, bytes)) return rc;
    const int grid = mlp_bwd_grid();
    const int64_t per = (a.rows + grid - 1) / grid;
    a.rows_per_cta = ((per + 7) / 8) * 8;
    LaunchScope ls_("mlp_bwd", st);
    launch_k(kern, dim3(grid), dim3(MLP_THREADS), bytes, st, a);
    return check_launch("mlp_bwd");
}

// launch_mlp<NTW, NTI, ACT> at every (NTW, NTI) of run_mlp's dispatch (LGAE_MLP_CASE in lgae_mlp.cu).  lgae_mlp.cu instantiates
// the LeakyReLU kernels; the other activations are instantiated in translation units of their own, two activations each, so
// that they compile in parallel (lgae_mlp_act_relu.cu, lgae_mlp_act_sigmoid.cu, lgae_mlp_act_tanh.cu).
#define LGAE_MLP_INSTANCE(EXT, W, I, ACT) EXT template int launch_mlp<W, I, ACT>(MlpArgs&, bool, cudaStream_t);
#define LGAE_MLP_INSTANCES(EXT, ACT)                                                                                          \
    LGAE_MLP_INSTANCE(EXT, 1, 1, ACT) LGAE_MLP_INSTANCE(EXT, 2, 1, ACT) LGAE_MLP_INSTANCE(EXT, 3, 1, ACT)                      \
    LGAE_MLP_INSTANCE(EXT, 4, 1, ACT) LGAE_MLP_INSTANCE(EXT, 5, 1, ACT) LGAE_MLP_INSTANCE(EXT, 6, 1, ACT)                      \
    LGAE_MLP_INSTANCE(EXT, 2, 2, ACT) LGAE_MLP_INSTANCE(EXT, 3, 2, ACT) LGAE_MLP_INSTANCE(EXT, 4, 2, ACT)                      \
    LGAE_MLP_INSTANCE(EXT, 5, 2, ACT) LGAE_MLP_INSTANCE(EXT, 6, 2, ACT) LGAE_MLP_INSTANCE(EXT, 8, 2, ACT)                      \
    LGAE_MLP_INSTANCE(EXT, 9, 2, ACT)

}  // namespace lgae
