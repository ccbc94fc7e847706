// CGMLP kernels for hidden widths the resident kernels (lgae_mlp.cuh) cannot hold: up to 96 (ntw <= 12).  Same inputs and
// outputs as mlp_fwd_kernel / mlp_bwd_kernel -- the packed weights of mlp_pack_kernel (both fragment orders, one contiguous
// block per layer), the saved activations `acts` (hidden, rows, 8 * NTW) and one row of parameter-gradient partials per CTA --
// so a level may run the resident forward and the streamed adjoint.  Instead of all layers' weights, shared memory holds two
// layer buffers: one TMA bulk copy brings a layer's fragments while the CTA computes with the other buffer's layer.
//
// Forward: layer-major over the CTA's contiguous slab of row groups.  For layer l a warp reads its row group's input
// fragments from acts[l-1] (or x) -- the same addresses the same lane wrote for layer l-1, so no barrier orders them -- and
// writes acts[l] (or y).  Each layer's weights are fetched once per CTA.
// Adjoint: chunks of MLP_STREAMED_ROWS rows as in mlp_bwd_kernel, dZ carried through the layer chain in registers by the row
// warps (one row group each); every chunk streams the transposed-order weights layer by layer.  The dW warps loop over tile
// blocks of at most 3 x 3 and accumulate into the CTA's partial row in a fixed order (no atomics).
//
// Weight buffer b = step & 1 of step s (the s-th layer the CTA streams) is refilled for step s + 2 only after a block-wide
// barrier that every reader of step s has passed; its mbarrier completes once per use, so step s waits for parity (s >> 1) & 1.
#pragma once

#include "lgae_mlp.cuh"

namespace lgae {

constexpr int MLP_STREAMED_ROWS = 32;   // rows of an adjoint chunk: one row group per row warp

// Doubles of the larger layer buffer: a hidden layer's fragments (the first and last layers are smaller).
__host__ __device__ constexpr int mlp_streamed_wbuf(int NTW) { return NTW * 2 * NTW * 32; }

// Offset (doubles) of layer l's fragments inside one fragment order of the packed weights (l = n_lin: the order's size).
LGAE_DEV int mlp_layer_off(int l, int n_lin, int NTW, int NTI) {
    int off = 0;
    for (int i = 0; i < l; ++i) off += mlp_layer_frag(i, n_lin, NTW, NTI);
    return off;
}

// ------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------
template <int NTW, int NTI, int ACT>
__global__ void __launch_bounds__(MLP_THREADS, 1) mlp_fwd_streamed_kernel(const MlpArgs a) {
    extern __shared__ __align__(128) double smem[];
    constexpr int WP = 8 * NTW, WB = mlp_streamed_wbuf(NTW);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int last = a.n_lin - 1;
    double* bias_s = smem + 2 * WB;   // n_lin * WP
    __shared__ uint64_t mbar[2];
    pdl_launch();
    auto fetch = [&](int l) {   // (one thread) layer l's fragments into buffer l & 1
        const unsigned bytes = (unsigned)(mlp_layer_frag(l, a.n_lin, NTW, NTI) * sizeof(double));
        mbar_expect_tx(&mbar[l & 1], bytes);
        bulk_g2s(smem + (l & 1) * WB, a.wpack + mlp_layer_off(l, a.n_lin, NTW, NTI), bytes, &mbar[l & 1]);
    };
    if (tid == 0) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); }
    __syncthreads();
    // the first two layers are fetched before the dependency wait (see mlp_fwd_kernel: mlp_pack_kernel never releases its
    // dependents early)
    if (tid == 0) { fetch(0); fetch(1); }
    for (int l = 0; l <= last; ++l) {
        const int nout = l == last ? a.nin : a.width;
        for (int t = tid; t < WP; t += blockDim.x) bias_s[l * WP + t] = t < nout ? a.theta[a.off_b[l] + t] : 0.0;
    }
    pdl_wait();   // the rows come from the previous kernel of the step
    __syncthreads();
    const int64_t ngroups = (a.rows + 7) / 8;
    const int64_t per_cta = (ngroups + gridDim.x - 1) / gridDim.x;
    const int64_t g_begin = (int64_t)blockIdx.x * per_cta, g_end = g_begin + per_cta < ngroups ? g_begin + per_cta : ngroups;
    for (int l = 0; l <= last; ++l) {
        mbar_wait(&mbar[l & 1], (l >> 1) & 1);
        const double* wl = smem + (l & 1) * WB;
        const double* bl = bias_s + l * WP;
        for (int64_t grp = g_begin + warp; grp < g_end; grp += nwarps) {
            const int64_t row = grp * 8 + g;
            const bool ok = row < a.rows;
            if (l == 0) {
                double in0[1][NTI][2], acc[1][NTW][2];
#pragma unroll
                for (int nt = 0; nt < NTI; ++nt) {
                    const int col = 8 * nt + 2 * q;
                    double2 v = make_double2(0.0, 0.0);
                    if (ok && col < a.nin) v = *reinterpret_cast<const double2*>(a.x + row * a.nin + col);
                    in0[0][nt][0] = v.x;
                    in0[0][nt][1] = v.y;
                }
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) { acc[0][nt][0] = bl[8 * nt + 2 * q]; acc[0][nt][1] = bl[8 * nt + 2 * q + 1]; }
                layer_mma<1, NTI, NTW>(in0, acc, wl, q, g);
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt)
                    if (ok)
                        *reinterpret_cast<double2*>(a.acts + row * WP + 8 * nt + 2 * q) =
                            make_double2(mlp_act<ACT>(acc[0][nt][0], a.slope), mlp_act<ACT>(acc[0][nt][1], a.slope));
                continue;
            }
            // the input fragments of a hidden or the last layer: row g, columns 8 kt + 2q, +1 of acts[l-1], as this lane
            // wrote them (rows past a.rows read as zero)
            double act[1][NTW][2];
            const double* src = a.acts + ((int64_t)(l - 1) * a.rows + row) * WP + 2 * q;
#pragma unroll
            for (int kt = 0; kt < NTW; ++kt) {
                double2 v = make_double2(0.0, 0.0);
                if (ok) v = *reinterpret_cast<const double2*>(src + 8 * kt);
                act[0][kt][0] = v.x;
                act[0][kt][1] = v.y;
            }
            if (l < last) {
                double acc[1][NTW][2];
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) { acc[0][nt][0] = bl[8 * nt + 2 * q]; acc[0][nt][1] = bl[8 * nt + 2 * q + 1]; }
                layer_mma<1, NTW, NTW>(act, acc, wl, q, g);
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt)
                    if (ok)
                        *reinterpret_cast<double2*>(a.acts + ((int64_t)l * a.rows + row) * WP + 8 * nt + 2 * q) =
                            make_double2(mlp_act<ACT>(acc[0][nt][0], a.slope), mlp_act<ACT>(acc[0][nt][1], a.slope));
            } else {
                double out[1][NTI][2];
#pragma unroll
                for (int nt = 0; nt < NTI; ++nt) { out[0][nt][0] = bl[8 * nt + 2 * q]; out[0][nt][1] = bl[8 * nt + 2 * q + 1]; }
                layer_mma<1, NTW, NTI>(act, out, wl, q, g);
#pragma unroll
                for (int nt = 0; nt < NTI; ++nt) {
                    const int col = 8 * nt + 2 * q;
                    if (ok && col < a.nin) *reinterpret_cast<double2*>(a.y + row * a.nin + col) = make_double2(out[0][nt][0], out[0][nt][1]);
                }
            }
        }
        if (l + 2 <= last) {
            __syncthreads();   // every warp is done with buffer l & 1
            if (tid == 0) fetch(l + 2);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// adjoint
// ------------------------------------------------------------------------------------------------------------
// Warp roles and the two block-wide barriers per layer as in mlp_bwd_kernel.  Step s = chunk * n_lin + (last - l); after the
// first barrier of step s >= 1 every row warp is done with step s - 1's buffer, and thread 0 refills it with step s + 1.
template <int NTW, int NTI, int ACT>
__global__ void __launch_bounds__(MLP_THREADS, 1) mlp_bwd_streamed_kernel(const MlpArgs a) {
    extern __shared__ __align__(128) double smem[];
    constexpr int WS = 8 * NTW + 4;                 // padded row stride of the staged tiles (conflict-free fragment loads)
    constexpr int WP = 8 * NTW, WB = mlp_streamed_wbuf(NTW);
    constexpr int NWH = 4;                          // warps per role
    constexpr int ROWS = MLP_STREAMED_ROWS;
    constexpr int PERD = (ROWS * WP / 4 + 32 * NWH - 1) / (32 * NWH);   // double4 of H per dW-warp thread
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const bool dw_role = warp < NWH;
    const int wi = warp & (NWH - 1);
    const int last = a.n_lin - 1;
    double* dz_s = smem + 2 * WB;                   // ROWS * WS
    double* h_s = dz_s + ROWS * WS;                 // ROWS * WS
    double* bred = h_s + ROWS * WS;                 // 2 * NWH * WP : per-row-warp column sums of dZ, double-buffered by layer parity
    const int64_t slab0 = (int64_t)blockIdx.x * a.rows_per_cta;
    const int64_t slab1 = slab0 + a.rows_per_cta < a.rows ? slab0 + a.rows_per_cta : a.rows;
    const int64_t nchunks = slab1 > slab0 ? (slab1 - slab0 + ROWS - 1) / ROWS : 1;   // an empty slab still writes its zero row
    const int64_t steps = nchunks * a.n_lin;
    const double* wq = a.wpack + mlp_layer_off(a.n_lin, a.n_lin, NTW, NTI);   // transposed order, behind the forward order
    __shared__ uint64_t mbar[2];
    auto fetch = [&](int64_t s) {   // (one thread) the weights of step s into buffer s & 1
        const int l = last - (int)(s % a.n_lin);
        const unsigned bytes = (unsigned)(mlp_layer_frag(l, a.n_lin, NTW, NTI) * sizeof(double));
        mbar_expect_tx(&mbar[s & 1], bytes);
        bulk_g2s(smem + (s & 1) * WB, wq + mlp_layer_off(l, a.n_lin, NTW, NTI), bytes, &mbar[s & 1]);
    };
    pdl_launch();
    if (tid == 0) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); }
    __syncthreads();
    if (tid == 0) { fetch(0); if (steps > 1) fetch(1); }   // before the dependency wait: see mlp_fwd_kernel
    pdl_wait();
    double* part = a.part + (int64_t)blockIdx.x * a.part_stride;
    bool first = true;   // first chunk of the slab: partials are stored, later chunks accumulate
    auto cta_sync = [] { asm volatile("bar.sync 0;" ::: "memory"); };
    if (dw_role) {
        int64_t s = 0;
        for (int64_t r0 = slab0;; r0 += ROWS) {
            const int crows = (int)(slab1 - r0 < ROWS ? (slab1 > r0 ? slab1 - r0 : 0) : ROWS);
            const int ksteps = ((crows + 7) / 8) * 2;   // MMA k-steps (4 rows each) covering the chunk; even
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
            for (int l = last; l >= 0; --l, ++s) {
                const int nout = l == last ? a.nin : a.width, nink = l == 0 ? a.nin : a.width;
                const int NOt = l == last ? NTI : NTW, KIt = l == 0 ? NTI : NTW;
                cta_sync();   // the previous layer's readers of dz_s / h_s / its weight buffer are done; its bias partials are complete
                if (tid == 0 && s >= 1 && s + 1 < steps) fetch(s + 1);
                if (l_prev >= 0)
                    for (int n = tid; n < nout_prev; n += 32 * NWH) {
                        double sum = 0.0;
#pragma unroll
                        for (int w = 0; w < NWH; ++w) sum += bred[((l_prev & 1) * NWH + w) * WP + n];
                        double* dst = part + a.po_b[l_prev] + n;
                        dst[0] = first ? sum : dst[0] + sum;
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
                // ---- weight gradient dW[n][k] = sum_rows dZ[row][n] H[row][k]: this warp's quadrant of tiles, in blocks of
                //      at most 3 x 3 tiles ----
                const int MBo = (NOt + 1) / 2, NBo = (KIt + 1) / 2;
                const int m0 = (wi >> 1) * MBo, n0 = (wi & 1) * NBo;
                const int mcnt = NOt - m0 < MBo ? NOt - m0 : MBo, ncnt = KIt - n0 < NBo ? KIt - n0 : NBo;
                for (int bi = 0; bi < mcnt; bi += 3)
                    for (int bj = 0; bj < ncnt; bj += 3) {
                        const int mc = mcnt - bi < 3 ? mcnt - bi : 3, nc = ncnt - bj < 3 ? ncnt - bj : 3;
                        double cw[2][3][3][2];   // even / odd k-steps: twice the independent MMA chains
#pragma unroll
                        for (int h = 0; h < 2; ++h)
#pragma unroll
                            for (int i = 0; i < 3; ++i)
#pragma unroll
                                for (int j = 0; j < 3; ++j) cw[h][i][j][0] = cw[h][i][j][1] = 0.0;
                        for (int ks = 0; ks < ksteps; ks += 2) {
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const double* dr = dz_s + (4 * (ks + h) + q) * WS + 8 * (m0 + bi) + g;
                                const double* hr = h_s + (4 * (ks + h) + q) * WS + 8 * (n0 + bj) + g;
                                double af[3], bf[3];
#pragma unroll
                                for (int i = 0; i < 3; ++i) af[i] = i < mc ? dr[8 * i] : 0.0;
#pragma unroll
                                for (int j = 0; j < 3; ++j) bf[j] = j < nc ? hr[8 * j] : 0.0;
#pragma unroll
                                for (int i = 0; i < 3; ++i)
#pragma unroll
                                    for (int j = 0; j < 3; ++j)
                                        if (i < mc && j < nc) dmma(cw[h][i][j][0], cw[h][i][j][1], af[i], bf[j]);
                            }
                        }
#pragma unroll
                        for (int i = 0; i < 3; ++i)
#pragma unroll
                            for (int j = 0; j < 3; ++j) {
                                if (i >= mc || j >= nc) continue;
                                const int n = 8 * (m0 + bi + i) + g, k = 8 * (n0 + bj + j) + 2 * q;
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
                double sum = 0.0;
#pragma unroll
                for (int w = 0; w < NWH; ++w) sum += bred[w * WP + n];   // layer 0: parity 0
                double* dst = part + a.po_b[0] + n;
                dst[0] = first ? sum : dst[0] + sum;
            }
            first = false;
            if (r0 + ROWS >= slab1) break;
        }
    } else {
        int64_t s = 0;
        for (int64_t r0 = slab0;; r0 += ROWS) {
            const int crows = (int)(slab1 - r0 < ROWS ? (slab1 > r0 ? slab1 - r0 : 0) : ROWS);
            const int rl = wi * 8;                         // this warp's row group inside the chunk
            const bool live = rl < ((crows + 7) / 8) * 8;  // a group holding at least one row of the slab
            const int64_t row = r0 + rl + g;
            // gradient wrt the output of the last layer, accumulator-fragment layout (rows past the slab carry zero dZ)
            double dz[NTW][2];
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) {
                dz[nt][0] = dz[nt][1] = 0.0;
                if (nt < NTI) {
                    const int col = 8 * nt + 2 * q;
                    if (row < slab1 && col < a.nin) {
                        const double2 v = *reinterpret_cast<const double2*>(a.g_y + row * a.nin + col);
                        dz[nt][0] = v.x;
                        dz[nt][1] = v.y;
                    }
                }
            }
            for (int l = last; l >= 0; --l, ++s) {
                const int NOt = l == last ? NTI : NTW, KIt = l == 0 ? NTI : NTW;
                cta_sync();
                // ---- publish dZ_l of this warp's row group ----
                if (live) {
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt)
                        if (nt < NOt) *reinterpret_cast<double2*>(dz_s + (rl + g) * WS + 8 * nt + 2 * q) = make_double2(dz[nt][0], dz[nt][1]);
                }
                // ---- bias gradient of layer l: column sums of this warp's rows of dZ_l, a butterfly over the 8 rows ----
                {
                    double* bl = bred + ((l & 1) * NWH + wi) * WP;
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt) {
                        if (nt < NOt) {
                            double c0 = dz[nt][0], c1 = dz[nt][1];
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
                // ---- data gradient: Gin[row][k] = sum_n dZ[row][n] W[n][k], then through the activation of layer l-1 ----
                mbar_wait(&mbar[s & 1], (unsigned)((s >> 1) & 1));
                if (!live) continue;
                const double* wl = smem + (s & 1) * WB;
                double gin[NTW][2];
#pragma unroll
                for (int kt = 0; kt < NTW; ++kt) gin[kt][0] = gin[kt][1] = 0.0;
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) {
                    if (nt < NOt) {
#pragma unroll
                        for (int e = 0; e < 2; ++e)
#pragma unroll
                            for (int kt = 0; kt < NTW; ++kt)
                                if (kt < KIt) dmma(gin[kt][0], gin[kt][1], dz[nt][e], wl[((nt * 2 + e) * KIt + kt) * 32 + q * 8 + g]);
                    }
                }
                if (l > 0) {
#pragma unroll
                    for (int kt = 0; kt < NTW; ++kt) {
                        const double2 h = *reinterpret_cast<const double2*>(h_s + (rl + g) * WS + 8 * kt + 2 * q);
                        dz[kt][0] = gin[kt][0] * mlp_act_grad<ACT>(h.x, a.slope);
                        dz[kt][1] = gin[kt][1] * mlp_act_grad<ACT>(h.y, a.slope);
                    }
                } else if (a.g_x) {
#pragma unroll
                    for (int kt = 0; kt < NTI; ++kt) {
                        const int col = 8 * kt + 2 * q;
                        if (row < slab1 && col < a.nin) *reinterpret_cast<double2*>(a.g_x + row * a.nin + col) = make_double2(gin[kt][0], gin[kt][1]);
                    }
                }
            }
            cta_sync();   // pairs with the dW warps' barrier before the last bias reduction
            if (r0 + ROWS >= slab1) break;
        }
    }
}

template <int NTW, int NTI, int ACT>
int launch_mlp_streamed(MlpArgs& a, bool bwd, cudaStream_t st) {
    constexpr int WP = 8 * NTW, WB = mlp_streamed_wbuf(NTW);
    if (!bwd) {
        const size_t bytes = (size_t)(2 * WB + a.n_lin * WP) * sizeof(double);
        auto kern = mlp_fwd_streamed_kernel<NTW, NTI, ACT>;
        if (int rc = ensure_smem((const void*)kern, bytes)) return rc;
        const int64_t ngroups = (a.rows + 7) / 8;
        const int cap = sm_count();
        const int grid = (int)(ngroups < cap ? ngroups : cap);
        LaunchScope ls_("mlp_fwd_streamed", st);
        launch_k(kern, dim3(grid), dim3(MLP_THREADS), bytes, st, a);
        return check_launch("mlp_fwd_streamed");
    }
    const size_t bytes = (size_t)(2 * WB + 2 * MLP_STREAMED_ROWS * (WP + 4) + 2 * 4 * WP) * sizeof(double);
    auto kern = mlp_bwd_streamed_kernel<NTW, NTI, ACT>;
    if (int rc = ensure_smem((const void*)kern, bytes)) return rc;
    const int grid = mlp_bwd_grid();
    const int64_t per = (a.rows + grid - 1) / grid;
    a.rows_per_cta = ((per + 7) / 8) * 8;
    LaunchScope ls_("mlp_bwd_streamed", st);
    launch_k(kern, dim3(grid), dim3(MLP_THREADS), bytes, st, a);
    return check_launch("mlp_bwd_streamed");
}

// launch_mlp_streamed<NTW, NTI, ACT> at every tiling of the streamed range, 7 <= NTW <= 12 (hidden widths 49..96), NTI = 1, 2.
// One translation unit per activation (lgae_mlp_streamed_*.cu).
#define LGAE_MLP_STREAMED_INSTANCE(EXT, W, I, ACT) EXT template int launch_mlp_streamed<W, I, ACT>(MlpArgs&, bool, cudaStream_t);
#define LGAE_MLP_STREAMED_INSTANCES(EXT, ACT)                                                                                                 \
    LGAE_MLP_STREAMED_INSTANCE(EXT, 7, 1, ACT) LGAE_MLP_STREAMED_INSTANCE(EXT, 8, 1, ACT) LGAE_MLP_STREAMED_INSTANCE(EXT, 9, 1, ACT)          \
    LGAE_MLP_STREAMED_INSTANCE(EXT, 10, 1, ACT) LGAE_MLP_STREAMED_INSTANCE(EXT, 11, 1, ACT) LGAE_MLP_STREAMED_INSTANCE(EXT, 12, 1, ACT)       \
    LGAE_MLP_STREAMED_INSTANCE(EXT, 7, 2, ACT) LGAE_MLP_STREAMED_INSTANCE(EXT, 8, 2, ACT) LGAE_MLP_STREAMED_INSTANCE(EXT, 9, 2, ACT)          \
    LGAE_MLP_STREAMED_INSTANCE(EXT, 10, 2, ACT) LGAE_MLP_STREAMED_INSTANCE(EXT, 11, 2, ACT) LGAE_MLP_STREAMED_INSTANCE(EXT, 12, 2, ACT)

}  // namespace lgae
