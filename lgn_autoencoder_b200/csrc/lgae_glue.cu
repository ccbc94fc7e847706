// Encoder / decoder glue around the LGN levels, and the caller-side ops of the training step:
//   enc_input   : LGNEncoder._prepare_input + input MixReps      (lgn/models/lgn_encoder.py:338-412, 290-296)
//   enc_latent  : latent MixReps + rep_to_p + pooling             (lgn_encoder.py:313-336, 419-583)
//   dec_input   : latent_to_graph + p_cplx_to_rep + input MixReps (lgn/models/lgn_decoder.py:305-345, 259-262)
//   dec_output  : mix_to_output + rep_to_p                        (lgn_decoder.py:286-296)
//   chamfer     : ChamferLoss over cdist                          (utils/losses/chamfer_loss/chamfer_loss.py:16-31)
//   normalize_p4, L1 regulariser, partial-gradient reduction.
// All of these are O(B*N*C) memory-trivial kernels; they exist so that a training step never leaves the
// library's node layout and launches ~35 kernels instead of the reference's several thousand ATen calls.
#include "lgae_common.cuh"

namespace lgae {

constexpr int MAXC = LGAE_MAX_CHANNELS;

// planar complex weight (2, R, Cc) at theta+off -> element [r][cc]
LGAE_DEV cplx wget(const double* theta, int64_t off, int rows, int cols, int r, int cc) {
    const int64_t idx = off + (int64_t)r * cols + cc;
    return cmake(theta[idx], theta[idx + (int64_t)rows * cols]);
}
// store element [r][cc] of a planar complex weight gradient into a row of partials (column offset `off`)
LGAE_DEV void pput(double* part, int64_t off, int rows, int cols, int r, int cc, cplx v) {
    const int64_t idx = off + (int64_t)r * cols + cc;
    part[idx] = v.x;
    part[idx + (int64_t)rows * cols] = v.y;
}

// ------------------------------------------------------------------------------------------------------------
// encoder input
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void enc_input_node(const double* theta, int64_t off00, int64_t off11, const double* p4, int64_t t, int C,
                                               double* mass, double* S, double* V) {
    const double* p = p4 + 4 * t;
    const double m = __dsqrt_rn(fabs(minkowski_sq(p[0], p[1], p[2], p[3])));   // lgn_encoder.py:376
    mass[t] = m;
    cplx y[4];
    canon_from_real(p, y);
    for (int c = 0; c < C; ++c) {
        const cplx w0 = wget(theta, off00, C, 1, c, 0), w1 = wget(theta, off11, C, 1, c, 0);
        reinterpret_cast<cplx*>(S)[t * C + c] = cscale(w0, m);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) reinterpret_cast<cplx*>(V)[(t * C + c) * 4 + mu] = cmul(w1, y[mu]);
    }
}
__global__ void enc_input_kernel(const double* theta, int64_t off00, int64_t off11, const double* p4, int64_t nodes, int C,
                                 double* mass, double* S, double* V) {
    pdl_launch();
    pdl_wait();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nodes) return;
    enc_input_node(theta, off00, off11, p4, t, C, mass, S, V);
}

__global__ void __launch_bounds__(256) enc_input_bwd_kernel(int64_t off00, int64_t off11, const double* p4, const double* mass, int64_t nodes,
                                                            int C, const double* gS, const double* gV, double* partials, int64_t part_stride) {
    pdl_launch();
    pdl_wait();
    __shared__ double scratch[32];
    double acc[MAXC][4];
#pragma unroll
    for (int c = 0; c < MAXC; ++c) acc[c][0] = acc[c][1] = acc[c][2] = acc[c][3] = 0.0;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nodes; t += (int64_t)gridDim.x * blockDim.x) {
        const double m = mass[t];
        cplx y[4];
        canon_from_real(p4 + 4 * t, y);
#pragma unroll
        for (int c = 0; c < MAXC; ++c) {
            if (c < C) {
                if (gS) {
                    const cplx g = reinterpret_cast<const cplx*>(gS)[t * C + c];
                    acc[c][0] = fma(m, g.x, acc[c][0]);
                    acc[c][1] = fma(m, g.y, acc[c][1]);
                }
                cplx s = czero();
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) cfmac(s, y[mu], reinterpret_cast<const cplx*>(gV)[(t * C + c) * 4 + mu]);
                acc[c][2] += s.x;
                acc[c][3] += s.y;
            }
        }
    }
    double* part = partials + (int64_t)blockIdx.x * part_stride;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
        if (c < C) {
#pragma unroll
            for (int x = 0; x < 4; ++x) {
                const double v = block_sum(acc[c][x], scratch);
                if (threadIdx.x == 0) {
                    const int64_t off = x < 2 ? off00 : off11;
                    part[off + (x & 1) * C + c] = v;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// encoder latent map
// ------------------------------------------------------------------------------------------------------------
struct LatentArgs {
    const double* theta;
    int64_t off00, off11;
    int B, N, C, tau_s, tau_v, mode;
    int parts;         // forward: 1 = latent scalars only, 2 = latent vectors only, 3 = both
    const double* S;   // (B,N,C,2)
    const double* V;   // (B,N,C,4,2)
    double* lat00;     // (2,B,1,Ts,1)
    double* lat11;     // (2,B,1,Tv,4)
    int32_t* sel;      // (4,2,B,tau_max)
    const double* g_lat00;
    const double* g_lat11;
    double* gS;
    double* gV;
    double* partials;       // (gridDim.x, part_stride) rows; columns [po00 ...), [po11 ...)
    int64_t part_stride, po00, po11;
};

LGAE_DEV double msq_of(const double* v) {   // get_msq, lgn_encoder.py:499-505 (sqrt, then square)
    const double nrm = __dsqrt_rn(v[1] * v[1] + v[2] * v[2] + v[3] * v[3]);
    return v[0] * v[0] - nrm * nrm;
}

// One CTA per jet.  Shared: L00 (N*tau_s complex), L11 Cartesian (N*tau_v*4 complex).
// `lat_out` (optional, shared memory, T_v * 4 complex): the jet's latent vectors, for a fused consumer (latent_bridge_kernel).
LGAE_DEV void enc_latent_body(const LatentArgs& a, double* smem, cplx* lat_out) {
    const int b = blockIdx.x, tid = threadIdx.x;
    const int N = a.N, C = a.C, ts = a.tau_s, tv = a.tau_v;
    const bool mix = a.mode == LGAE_LATENT_MIX;
    const int rows = mix ? 1 : N;        // 'mix' contracts particles and channels together
    const int cin = mix ? N * C : C;
    cplx* L00 = reinterpret_cast<cplx*>(smem);
    cplx* L11 = L00 + rows * ts;
    const cplx* S = reinterpret_cast<const cplx*>(a.S) + (int64_t)b * N * C;
    const cplx* V = reinterpret_cast<const cplx*>(a.V) + (int64_t)b * N * C * 4;
    const bool do_s = (a.parts & 1) != 0, do_v = (a.parts & 2) != 0;
    for (int it = tid; do_s && it < rows * ts; it += blockDim.x) {
        const int i = it / ts, t = it % ts;
        cplx acc = czero();
        for (int k = 0; k < cin; ++k) cfma(acc, wget(a.theta, a.off00, ts, cin, t, k), S[i * cin + k]);
        L00[it] = acc;
    }
    for (int it = tid; do_v && it < rows * tv; it += blockDim.x) {
        const int i = it / tv, t = it % tv;
        cplx acc[4] = {czero(), czero(), czero(), czero()};
        for (int k = 0; k < cin; ++k) {
            const cplx w = wget(a.theta, a.off11, tv, cin, t, k);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cfma(acc[mu], w, V[(i * cin + k) * 4 + mu]);
        }
        cplx cart[4];
        cart_from_canon(acc, cart);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) L11[it * 4 + mu] = cart[mu];
    }
    __syncthreads();
    const int B = a.B;
    const int mode = a.mode;
    if (mode == LGAE_LATENT_MEAN || mode == LGAE_LATENT_SUM || mix) {
        const double scale = mode == LGAE_LATENT_MEAN ? 1.0 / N : 1.0;
        for (int it = tid; do_s && it < ts; it += blockDim.x) {
            cplx acc = czero();
            for (int i = 0; i < rows; ++i) acc = cadd(acc, L00[i * ts + it]);
            a.lat00[(int64_t)(0 * B + b) * ts + it] = acc.x * scale;
            a.lat00[(int64_t)(1 * B + b) * ts + it] = acc.y * scale;
        }
        for (int it = tid; do_v && it < tv * 4; it += blockDim.x) {
            cplx acc = czero();
            for (int i = 0; i < rows; ++i) acc = cadd(acc, L11[i * tv * 4 + it]);
            a.lat11[(int64_t)(0 * B + b) * tv * 4 + it] = acc.x * scale;
            a.lat11[(int64_t)(1 * B + b) * tv * 4 + it] = acc.y * scale;
            if (lat_out) lat_out[it] = cscale(acc, scale);
        }
        return;
    }
    // min / max / min&max: arg-select per (re|im, tau), re and im parts independently (lgn_encoder.py:540-583)
    const bool both = mode == LGAE_LATENT_MINMAX;
    const int Ts = both ? 2 * ts : ts, Tv = both ? 2 * tv : tv;
    const int tmax = ts > tv ? ts : tv;
    for (int it = tid; do_s && it < 2 * 2 * ts; it += blockDim.x) {          // scalars: [kind][part][t]
        const int t = it % ts, part = (it / ts) & 1, kind = it / (2 * ts);   // kind 0 = min, 1 = max
        if (!both && kind != (mode == LGAE_LATENT_MAX ? 1 : 0)) continue;
        int best = 0;
        double bv = 0.0;
        for (int i = 0; i < N; ++i) {
            const cplx z = L00[i * ts + t];
            const double s = part ? z.y : z.x;
            const double key = kind ? s * s : s;                     // max selects on s^2 (get_msq of a scalar)
            if (i == 0 || (kind ? key > bv : key < bv)) { bv = key; best = i; }
        }
        const cplx z = L00[best * ts + t];
        const int T = (both && kind) ? ts + t : t;
        a.lat00[(int64_t)(part * B + b) * Ts + T] = part ? z.y : z.x;
        if (a.sel) a.sel[((int64_t)((kind)*2 + part) * B + b) * tmax + t] = best;
    }
    for (int it = tid; do_v && it < 2 * 2 * tv; it += blockDim.x) {          // vectors
        const int t = it % tv, part = (it / tv) & 1, kind = it / (2 * tv);
        if (!both && kind != (mode == LGAE_LATENT_MAX ? 1 : 0)) continue;
        int best = 0;
        double bv = 0.0;
        for (int i = 0; i < N; ++i) {
            double v[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) { const cplx z = L11[(i * tv + t) * 4 + mu]; v[mu] = part ? z.y : z.x; }
            const double key = msq_of(v);
            if (i == 0 || (kind ? key > bv : key < bv)) { bv = key; best = i; }
        }
        const int T = (both && kind) ? tv + t : t;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) {
            const cplx z = L11[(best * tv + t) * 4 + mu];
            a.lat11[((int64_t)(part * B + b) * Tv + T) * 4 + mu] = part ? z.y : z.x;
            if (lat_out) {   // re and im parts are selected independently: two threads fill the two halves
                if (part) lat_out[T * 4 + mu].y = z.y; else lat_out[T * 4 + mu].x = z.x;
            }
        }
        if (a.sel) a.sel[((int64_t)((2 + kind) * 2 + part) * B + b) * tmax + t] = best;
    }
}

__global__ void __launch_bounds__(256) enc_latent_kernel(const LatentArgs a) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    enc_latent_body(a, smem, nullptr);
}

// Adjoint of enc_latent.  Persistent CTAs over jets; latent-weight gradients accumulate in shared memory.
// Split into init / per-jet / flush pieces so that the training step can run it in one kernel with the decoder-input
// adjoint (latent_bridge_bwd_kernel), which hands the latent gradient over in shared memory.
struct EncLatBwdSm {
    cplx *gL00, *gL11, *gw00, *gw11, *w00_s, *w11_s, *S_s, *V_s;
    int rows, cin;
};
__device__ __forceinline__ EncLatBwdSm enc_latent_bwd_init(const LatentArgs& a, double* smem) {
    const int tid = threadIdx.x, N = a.N, C = a.C, ts = a.tau_s, tv = a.tau_v;
    const bool mix = a.mode == LGAE_LATENT_MIX;
    EncLatBwdSm m;
    m.rows = mix ? 1 : N; m.cin = mix ? N * C : C;
    const int rows = m.rows, cin = m.cin;
    m.gL00 = reinterpret_cast<cplx*>(smem);       // rows*ts
    m.gL11 = m.gL00 + rows * ts;                  // rows*tv*4 (canonical after the basis change)
    m.gw00 = m.gL11 + rows * tv * 4;              // ts*cin
    m.gw11 = m.gw00 + ts * cin;                   // tv*cin
    m.w00_s = m.gw11 + tv * cin;                  // ts*cin   latent weights, interleaved
    m.w11_s = m.w00_s + ts * cin;                 // tv*cin
    m.S_s = m.w11_s + tv * cin;                   // N*C      this jet's node features
    m.V_s = m.S_s + N * C;                        // N*C*4
    for (int t = tid; t < (ts + tv) * cin; t += blockDim.x) m.gw00[t] = czero();
    for (int t = tid; t < ts * cin; t += blockDim.x) m.w00_s[t] = wget(a.theta, a.off00, ts, cin, t / cin, t % cin);
    for (int t = tid; t < tv * cin; t += blockDim.x) m.w11_s[t] = wget(a.theta, a.off11, tv, cin, t / cin, t % cin);
    return m;
}
__host__ __device__ inline size_t enc_latent_bwd_smem_cplx(int N, int C, int ts, int tv, int mode) {
    const int mix = mode == LGAE_LATENT_MIX;
    const int rows = mix ? 1 : N, cin = mix ? N * C : C;
    return (size_t)rows * (ts + 4 * tv) + (size_t)2 * (ts + tv) * cin + (size_t)5 * N * C;
}
// GLAT_S: the latent-vector gradient of jet b is read from shared memory (Tv*4 interleaved complex) instead of a.g_lat11.
template <bool GLAT_S>
__device__ __forceinline__ void enc_latent_bwd_jet(const LatentArgs& a, const EncLatBwdSm& m, int b, const cplx* glat_s) {
    const int tid = threadIdx.x;
    const int N = a.N, C = a.C, ts = a.tau_s, tv = a.tau_v, B = a.B, mode = a.mode;
    const bool mix = mode == LGAE_LATENT_MIX;
    const int rows = m.rows, cin = m.cin;
    cplx *gL00 = m.gL00, *gL11 = m.gL11, *gw00 = m.gw00, *gw11 = m.gw11, *w00_s = m.w00_s, *w11_s = m.w11_s, *S_s = m.S_s, *V_s = m.V_s;
    const bool both = mode == LGAE_LATENT_MINMAX;
    const int Ts = both ? 2 * ts : ts, Tv = both ? 2 * tv : tv;
    const int tmax = ts > tv ? ts : tv;
    const bool have11 = GLAT_S || a.g_lat11;
    auto g11 = [&](int part, int width, int r) -> double {   // element r of the (width) latent-vector gradient, part re/im
        if (GLAT_S) return part ? glat_s[r].y : glat_s[r].x;
        return a.g_lat11[(int64_t)(part * B + b) * width + r];
    };
    {
        __syncthreads();
        for (int t = tid; t < rows * (ts + 4 * tv); t += blockDim.x) gL00[t] = czero();
        {   // node features of the jet -> shared memory (16-byte vector loads, all in flight)
            const double2* gs = reinterpret_cast<const double2*>(a.S) + (int64_t)b * N * C;
            const double2* gv = reinterpret_cast<const double2*>(a.V) + (int64_t)b * N * C * 4;
            for (int t = tid; t < N * C; t += blockDim.x) S_s[t] = gs[t];
            for (int t = tid; t < N * C * 4; t += blockDim.x) V_s[t] = gv[t];
        }
        __syncthreads();
        if (mode == LGAE_LATENT_MEAN || mode == LGAE_LATENT_SUM || mix) {
            const double scale = mode == LGAE_LATENT_MEAN ? 1.0 / N : 1.0;
            for (int it = tid; it < rows * ts; it += blockDim.x) {
                const int t = it % ts;
                if (a.g_lat00) gL00[it] = cmake(a.g_lat00[(int64_t)(0 * B + b) * ts + t] * scale, a.g_lat00[(int64_t)(1 * B + b) * ts + t] * scale);
            }
            for (int it = tid; it < rows * tv * 4; it += blockDim.x) {
                const int r = it % (tv * 4);
                if (have11) gL11[it] = cmake(g11(0, tv * 4, r) * scale, g11(1, tv * 4, r) * scale);
            }
        } else {
            // scatter: one thread per (tau) handles its 2 kinds x 2 parts sequentially => no write conflicts
            for (int t = tid; t < ts; t += blockDim.x) {
                if (!a.g_lat00) break;
                for (int kind = 0; kind < 2; ++kind) {
                    if (!both && kind != (mode == LGAE_LATENT_MAX ? 1 : 0)) continue;
                    const int T = (both && kind) ? ts + t : t;
                    for (int part = 0; part < 2; ++part) {
                        const int i = a.sel[((int64_t)(kind * 2 + part) * B + b) * tmax + t];
                        const double gv = a.g_lat00[(int64_t)(part * B + b) * Ts + T];
                        if (part) gL00[i * ts + t].y += gv; else gL00[i * ts + t].x += gv;
                    }
                }
            }
            for (int t = tid; t < tv; t += blockDim.x) {
                if (!have11) break;
                for (int kind = 0; kind < 2; ++kind) {
                    if (!both && kind != (mode == LGAE_LATENT_MAX ? 1 : 0)) continue;
                    const int T = (both && kind) ? tv + t : t;
                    for (int part = 0; part < 2; ++part) {
                        const int i = a.sel[((int64_t)((2 + kind) * 2 + part) * B + b) * tmax + t];
                        for (int mu = 0; mu < 4; ++mu) {
                            const double gv = g11(part, Tv * 4, T * 4 + mu);
                            if (part) gL11[(i * tv + t) * 4 + mu].y += gv; else gL11[(i * tv + t) * 4 + mu].x += gv;
                        }
                    }
                }
            }
        }
        __syncthreads();
        // adjoint of rep_to_p: Cartesian gradient -> canonical
        for (int it = tid; it < rows * tv; it += blockDim.x) {
            cplx gc[4], gy[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) gc[mu] = gL11[it * 4 + mu];
            canon_from_cplx(gc, gy);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) gL11[it * 4 + mu] = gy[mu];
        }
        __syncthreads();
        const cplx* S = S_s;
        const cplx* V = V_s;
        // feature gradients
        for (int it = tid; it < rows * cin; it += blockDim.x) {
            const int i = it / cin, k = it % cin;
            cplx gs = czero(), gv[4] = {czero(), czero(), czero(), czero()};
            for (int t = 0; t < ts; ++t) cfmac(gs, w00_s[t * cin + k], gL00[i * ts + t]);
            for (int t = 0; t < tv; ++t) {
                const cplx w = w11_s[t * cin + k];
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) cfmac(gv[mu], w, gL11[(i * tv + t) * 4 + mu]);
            }
            reinterpret_cast<cplx*>(a.gS)[(int64_t)b * N * C + it] = gs;
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) reinterpret_cast<cplx*>(a.gV)[((int64_t)b * N * C + it) * 4 + mu] = gv[mu];
        }
        // weight gradients: one thread per (t, k)
        for (int it = tid; it < ts * cin; it += blockDim.x) {
            const int t = it / cin, k = it % cin;
            cplx acc = czero();
            for (int i = 0; i < rows; ++i) cfmac(acc, S[i * cin + k], gL00[i * ts + t]);
            gw00[it] = cadd(gw00[it], acc);
        }
        for (int it = tid; it < tv * cin; it += blockDim.x) {
            const int t = it / cin, k = it % cin;
            cplx acc = czero();
            for (int i = 0; i < rows; ++i)
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) cfmac(acc, V[(i * cin + k) * 4 + mu], gL11[(i * tv + t) * 4 + mu]);
            gw11[it] = cadd(gw11[it], acc);
        }
    }
}
__device__ __forceinline__ void enc_latent_bwd_flush(const LatentArgs& a, const EncLatBwdSm& m) {
    const int tid = threadIdx.x, ts = a.tau_s, tv = a.tau_v, cin = m.cin;
    double* part = a.partials + (int64_t)blockIdx.x * a.part_stride;
    for (int it = tid; it < ts * cin; it += blockDim.x) pput(part, a.po00, ts, cin, it / cin, it % cin, m.gw00[it]);
    for (int it = tid; it < tv * cin; it += blockDim.x) pput(part, a.po11, tv, cin, it / cin, it % cin, m.gw11[it]);
}
__global__ void __launch_bounds__(256) enc_latent_bwd_kernel(const LatentArgs a) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    const EncLatBwdSm m = enc_latent_bwd_init(a, smem);
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) enc_latent_bwd_jet<false>(a, m, b, nullptr);
    __syncthreads();
    enc_latent_bwd_flush(a, m);
}

// ------------------------------------------------------------------------------------------------------------
// decoder input
// ------------------------------------------------------------------------------------------------------------
struct DecInArgs {
    const double* theta;
    int64_t off_g11, off_in00, off_in11;
    int B, N, C, tau;
    const double* lat11;   // (2,B,1,tau,4)
    double* y;             // (B,N,4,2)
    double* S;
    double* V;
    const double* gS;
    const double* gV;
    const double* gy;      // accumulated by the level adjoints
    double* g_lat11;
    double* partials;       // (gridDim.x, part_stride) rows
    int64_t part_stride, po_g11, po_in00, po_in11;
};

// latent_to_graph + p_cplx_to_rep + input MixReps of one jet from its latent vectors `lat` (tau * 4 complex, shared memory).
LGAE_DEV void dec_input_body(const DecInArgs& a, const cplx* lat) {
    const int b = blockIdx.x, tid = threadIdx.x, N = a.N, C = a.C, tau = a.tau;
    for (int i = tid; i < N; i += blockDim.x) {
        cplx P[4] = {czero(), czero(), czero(), czero()};
        for (int t = 0; t < tau; ++t) {
            const cplx w = wget(a.theta, a.off_g11, N, tau, i, t);
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cfma(P[mu], w, lat[t * 4 + mu]);
        }
        cplx y[4];
        canon_from_cplx(P, y);
        const int64_t node = (int64_t)b * N + i;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) reinterpret_cast<cplx*>(a.y)[node * 4 + mu] = y[mu];
        for (int c = 0; c < C; ++c) {
            const cplx w0 = wget(a.theta, a.off_in00, C, 1, c, 0), w1 = wget(a.theta, a.off_in11, C, 1, c, 0);
            reinterpret_cast<cplx*>(a.S)[node * C + c] = cmul_1pi(w0);     // zonal (0,0) = 1 + 1j (zonal_functions.py:150-154)
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) reinterpret_cast<cplx*>(a.V)[(node * C + c) * 4 + mu] = cmul(w1, y[mu]);
        }
    }
}
__global__ void __launch_bounds__(128) dec_input_kernel(const DecInArgs a) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    cplx* lat = reinterpret_cast<cplx*>(smem);   // tau*4
    const int b = blockIdx.x, tid = threadIdx.x, tau = a.tau, B = a.B;
    for (int t = tid; t < tau * 4; t += blockDim.x)
        lat[t] = cmake(a.lat11[(int64_t)(0 * B + b) * tau * 4 + t], a.lat11[(int64_t)(1 * B + b) * tau * 4 + t]);
    __syncthreads();
    dec_input_body(a, lat);
}
// Encoder latent map and decoder input of a jet in one launch (the latent never leaves the CTA between the two; it is still
// written to HBM as the step's output).  Shared memory: [enc_latent scratch | latent vectors (T_v * 4 complex)].
__global__ void __launch_bounds__(256) latent_bridge_kernel(const LatentArgs a, const DecInArgs d, int lat_off) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    cplx* lat = reinterpret_cast<cplx*>(smem + lat_off);
    enc_latent_body(a, smem, lat);
    __syncthreads();
    dec_input_body(d, lat);
}

// Persistent over jets; the threads loop over the particles.
struct DecInBwdSm { cplx *lat, *gP_s, *gwg, *gin; };
__device__ __forceinline__ DecInBwdSm dec_input_bwd_init(const DecInArgs& a, double* smem) {
    const int tid = threadIdx.x, N = a.N, C = a.C, tau = a.tau;
    DecInBwdSm m;
    m.lat = reinterpret_cast<cplx*>(smem);   // tau*4
    m.gP_s = m.lat + tau * 4;                // N*4
    m.gwg = m.gP_s + N * 4;                  // N*tau   accumulators
    m.gin = m.gwg + N * tau;                 // 2*C     accumulators (in00, in11)
    for (int t = tid; t < N * tau + 2 * C; t += blockDim.x) m.gwg[t] = czero();
    return m;
}
__host__ __device__ inline size_t dec_input_bwd_smem_cplx(int N, int C, int tau) { return (size_t)tau * 4 + (size_t)N * 4 + (size_t)N * tau + 2 * C; }
// glat_s (optional): also leaves the latent gradient of jet b in shared memory, tau*4 interleaved complex.
__device__ __forceinline__ void dec_input_bwd_jet(const DecInArgs& a, const DecInBwdSm& m, int b, cplx* glat_s) {
    const int tid = threadIdx.x, N = a.N, C = a.C, tau = a.tau, B = a.B;
    cplx *lat = m.lat, *gP_s = m.gP_s, *gwg = m.gwg, *gin = m.gin;
    {
        __syncthreads();
        for (int t = tid; t < tau * 4; t += blockDim.x)
            lat[t] = cmake(a.lat11[(int64_t)(0 * B + b) * tau * 4 + t], a.lat11[(int64_t)(1 * B + b) * tau * 4 + t]);
        for (int i = tid; i < N; i += blockDim.x) {
            const int64_t node = (int64_t)b * N + i;
            cplx gy[4], y[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                gy[mu] = reinterpret_cast<const cplx*>(a.gy)[node * 4 + mu];
                y[mu] = reinterpret_cast<const cplx*>(a.y)[node * 4 + mu];
            }
            for (int c = 0; c < C; ++c) {
                const cplx w1 = wget(a.theta, a.off_in11, C, 1, c, 0);
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) cfmac(gy[mu], w1, reinterpret_cast<const cplx*>(a.gV)[(node * C + c) * 4 + mu]);
            }
            cplx gP[4];
            cart_from_canon(gy, gP);   // adjoint of p_cplx_to_rep
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) gP_s[i * 4 + mu] = gP[mu];
        }
        __syncthreads();
        // input-mix weight gradients: one warp per (which, c), lanes over the particles, butterfly sum (fixed order)
        for (int it = tid >> 5; it < 2 * C; it += blockDim.x >> 5) {
            const int which = it / C, c = it % C, lane = tid & 31;
            cplx acc = czero();
            for (int i = lane; i < N; i += 32) {
                const int64_t node = (int64_t)b * N + i;
                if (which) {
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu)
                        cfmac(acc, reinterpret_cast<const cplx*>(a.y)[node * 4 + mu], reinterpret_cast<const cplx*>(a.gV)[(node * C + c) * 4 + mu]);
                } else if (a.gS) {
                    acc = cadd(acc, cmul_1mi(reinterpret_cast<const cplx*>(a.gS)[node * C + c]));
                }
            }
            acc.x = warp_sum(acc.x);
            acc.y = warp_sum(acc.y);
            if (lane == 0) gin[which * C + c] = cadd(gin[which * C + c], acc);
        }
        // latent_to_graph weight gradient and latent gradient
        for (int it = tid; it < N * tau; it += blockDim.x) {
            const int i = it / tau, t = it % tau;
            cplx acc = czero();
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cfmac(acc, lat[t * 4 + mu], gP_s[i * 4 + mu]);
            gwg[it] = cadd(gwg[it], acc);
        }
        for (int it = tid; it < tau * 4; it += blockDim.x) {
            const int t = it / 4, mu = it % 4;
            cplx acc = czero();
            for (int i = 0; i < N; ++i) cfmac(acc, wget(a.theta, a.off_g11, N, tau, i, t), gP_s[i * 4 + mu]);
            a.g_lat11[(int64_t)(0 * B + b) * tau * 4 + it] = acc.x;
            a.g_lat11[(int64_t)(1 * B + b) * tau * 4 + it] = acc.y;
            if (glat_s) glat_s[it] = acc;
        }
    }
}
__device__ __forceinline__ void dec_input_bwd_flush(const DecInArgs& a, const DecInBwdSm& m) {
    const int tid = threadIdx.x, N = a.N, C = a.C, tau = a.tau;
    double* part = a.partials + (int64_t)blockIdx.x * a.part_stride;
    for (int it = tid; it < N * tau; it += blockDim.x) pput(part, a.po_g11, N, tau, it / tau, it % tau, m.gwg[it]);
    for (int c = tid; c < C; c += blockDim.x) {
        pput(part, a.po_in00, C, 1, c, 0, m.gin[c]);
        pput(part, a.po_in11, C, 1, c, 0, m.gin[C + c]);
    }
}
__global__ void __launch_bounds__(128) dec_input_bwd_kernel(const DecInArgs a) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    const DecInBwdSm m = dec_input_bwd_init(a, smem);
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) dec_input_bwd_jet(a, m, b, nullptr);
    __syncthreads();
    dec_input_bwd_flush(a, m);
}
// Training step: decoder-input adjoint and encoder-latent adjoint of the same jets in one kernel; the latent gradient
// goes from one to the other through shared memory (and is still written to g_lat11 for the caller).
__global__ void __launch_bounds__(256) latent_bridge_bwd_kernel(const DecInArgs d, const LatentArgs a, int off_enc, int off_glat) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    const DecInBwdSm md = dec_input_bwd_init(d, smem);
    const EncLatBwdSm me = enc_latent_bwd_init(a, smem + off_enc);
    cplx* glat_s = reinterpret_cast<cplx*>(smem + off_glat);
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        dec_input_bwd_jet(d, md, b, glat_s);
        enc_latent_bwd_jet<true>(a, me, b, glat_s);   // starts with a barrier: glat_s is complete
    }
    __syncthreads();
    dec_input_bwd_flush(d, md);
    enc_latent_bwd_flush(a, me);
}

// ------------------------------------------------------------------------------------------------------------
// decoder output
// ------------------------------------------------------------------------------------------------------------
__global__ void dec_output_kernel(const double* theta, int64_t off00, int64_t off11, int B, int N, int C, const double* S,
                                  const double* V, double* recon, double* gen00) {
    pdl_launch();
    pdl_wait();
    const int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= (int64_t)B * N) return;
    cplx gen[4] = {czero(), czero(), czero(), czero()}, g0 = czero();
    for (int c = 0; c < C; ++c) {
        const cplx w1 = wget(theta, off11, 1, C, 0, c);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) cfma(gen[mu], w1, reinterpret_cast<const cplx*>(V)[(node * C + c) * 4 + mu]);
        if (gen00) cfma(g0, wget(theta, off00, 1, C, 0, c), reinterpret_cast<const cplx*>(S)[node * C + c]);
    }
    cplx p[4];
    cart_from_canon(gen, p);
#pragma unroll
    for (int mu = 0; mu < 4; ++mu) {
        recon[node * 4 + mu] = p[mu].x;
        recon[((int64_t)B * N + node) * 4 + mu] = p[mu].y;
    }
    if (gen00) {
        gen00[node] = g0.x;
        gen00[(int64_t)B * N + node] = g0.y;
    }
}

__global__ void __launch_bounds__(256) dec_output_bwd_kernel(const double* theta, int64_t off00, int64_t off11, int B, int N, int C,
                                                             const double* S, const double* V, const double* g_recon, const double* g_gen00,
                                                             double* gS, double* gV, double* partials, int64_t part_stride) {
    pdl_launch();
    pdl_wait();
    __shared__ double scratch[32];
    double acc[MAXC][4];
#pragma unroll
    for (int c = 0; c < MAXC; ++c) acc[c][0] = acc[c][1] = acc[c][2] = acc[c][3] = 0.0;
    const int64_t nodes = (int64_t)B * N;
    for (int64_t node = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; node < nodes; node += (int64_t)gridDim.x * blockDim.x) {
        cplx gp[4], gg[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) gp[mu] = cmake(g_recon[node * 4 + mu], g_recon[(nodes + node) * 4 + mu]);
        canon_from_cplx(gp, gg);    // adjoint of rep_to_p
        const cplx g0 = g_gen00 ? cmake(g_gen00[node], g_gen00[nodes + node]) : czero();
#pragma unroll
        for (int c = 0; c < MAXC; ++c) {
            if (c < C) {
                const cplx w1 = wget(theta, off11, 1, C, 0, c);
                cplx gw = czero();
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) {
                    reinterpret_cast<cplx*>(gV)[(node * C + c) * 4 + mu] = cmulc(w1, gg[mu]);
                    cfmac(gw, reinterpret_cast<const cplx*>(V)[(node * C + c) * 4 + mu], gg[mu]);
                }
                acc[c][2] += gw.x;
                acc[c][3] += gw.y;
                if (g_gen00) {
                    reinterpret_cast<cplx*>(gS)[node * C + c] = cmulc(wget(theta, off00, 1, C, 0, c), g0);
                    const cplx gw0 = cmulc(reinterpret_cast<const cplx*>(S)[node * C + c], g0);
                    acc[c][0] += gw0.x;
                    acc[c][1] += gw0.y;
                }
            }
        }
    }
    // row of partials: [out00 (2C) | out11 (2C)]
    double* part = partials + (int64_t)blockIdx.x * part_stride;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
        if (c < C) {
#pragma unroll
            for (int x = 0; x < 4; ++x) {
                const double v = block_sum(acc[c][x], scratch);
                if (threadIdx.x == 0) part[(x < 2 ? 0 : 2 * C) + (x & 1) * C + c] = v;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// chamfer loss (+ gradient), normalisation, L1, reductions
// ------------------------------------------------------------------------------------------------------------
// get_real (utils/utils.py:194-207): the real 4-momentum the loss sees, x = f(re, im), and its derivative (d_re, d_im).
LGAE_DEV double get_real_value(int mode, double re, double im) {
    switch (mode) {
        case LGAE_GET_REAL_IMAG: return im;
        case LGAE_GET_REAL_SUM: return re + im;
        case LGAE_GET_REAL_MEAN: return (re + im) / 2;
        case LGAE_GET_REAL_NORM: return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im)), 1e-16));
        default: return re;
    }
}
LGAE_DEV void get_real_grad(int mode, double re, double im, double x, double g, double& g_re, double& g_im) {
    switch (mode) {
        case LGAE_GET_REAL_IMAG: g_re = 0.0; g_im = g; break;
        case LGAE_GET_REAL_SUM: g_re = g; g_im = g; break;
        case LGAE_GET_REAL_MEAN: g_re = 0.5 * g; g_im = 0.5 * g; break;
        case LGAE_GET_REAL_NORM: g_re = g * (re / x); g_im = g * (im / x); break;
        default: g_re = g; g_im = 0.0; break;
    }
}
// One CTA per jet.  x_i = get_real(recon_i)  (utils/train.py:292).
__global__ void __launch_bounds__(128) chamfer_kernel(const double* recon, const double* target, int B, int N, int M, double* jet_loss,
                                                      const double* g_loss, double* g_recon, int mode) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    double* x = smem;            // N*4
    double* t = x + 4 * N;       // M*4
    double* m1 = t + 4 * M;      // N
    double* m2 = m1 + N;         // M
    int* j1 = reinterpret_cast<int*>(m2 + M);   // N
    int* i2 = j1 + N;                            // M
    const int b = blockIdx.x, tid = threadIdx.x;
    const int64_t plane = (int64_t)B * N * 4;
    for (int k = tid; k < 4 * N; k += blockDim.x) x[k] = get_real_value(mode, recon[(int64_t)b * N * 4 + k], recon[plane + (int64_t)b * N * 4 + k]);
    for (int k = tid; k < 4 * M; k += blockDim.x) t[k] = target[(int64_t)b * M * 4 + k];
    __syncthreads();
    auto dist = [&](int i, int j) {
        double s = 0.0;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) { const double d = x[4 * i + mu] - t[4 * j + mu]; s += d * d; }
        return s;
    };
    // the two directions run side by side: even warps take the reconstructed particles, odd warps the targets
    __shared__ double dir_sum[2];
    const int lane = tid & 31, warp = tid >> 5, nw2 = (blockDim.x >> 5) >> 1;   // blockDim is a multiple of 64
    if ((warp & 1) == 0) {
        for (int i = (warp >> 1) * 32 + lane; i < N; i += nw2 * 32) {
            double best = dist(i, 0);
            int bj = 0;
            for (int j = 1; j < M; ++j) { const double d = dist(i, j); if (d < best) { best = d; bj = j; } }
            m1[i] = best; j1[i] = bj;
        }
    } else {
        for (int j = (warp >> 1) * 32 + lane; j < M; j += nw2 * 32) {
            double best = dist(0, j);
            int bi = 0;
            for (int i = 1; i < N; ++i) { const double d = dist(i, j); if (d < best) { best = d; bi = i; } }
            m2[j] = best; i2[j] = bi;
        }
    }
    __syncthreads();
    if (warp < 2) {   // per-direction sums: lanes stride the particles, then a butterfly (fixed order)
        const double* mm = warp == 0 ? m1 : m2;
        const int n = warp == 0 ? N : M;
        double acc = 0.0;
        for (int k = lane; k < n; k += 32) acc += mm[k];
        acc = warp_sum(acc);
        if (lane == 0) dir_sum[warp] = acc;
    }
    __syncthreads();
    if (tid == 0) jet_loss[b] = 0.5 * (dir_sum[0] + dir_sum[1]);
    if (g_recon) {
        const double scale = g_loss ? *g_loss : 1.0;
        for (int i = tid; i < N; i += blockDim.x) {
            double g[4];
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) g[mu] = x[4 * i + mu] - t[4 * j1[i] + mu];
            for (int j = 0; j < M; ++j)
                if (i2[j] == i) {
#pragma unroll
                    for (int mu = 0; mu < 4; ++mu) g[mu] += x[4 * i + mu] - t[4 * j + mu];
                }
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) {
                const int64_t k = ((int64_t)b * N + i) * 4 + mu;
                double g_re, g_im;
                get_real_grad(mode, recon[k], recon[plane + k], x[4 * i + mu], g[mu] * scale, g_re, g_im);
                g_recon[k] = g_re;
                g_recon[plane + k] = g_im;
            }
        }
    }
}

// Per-jet anomaly scores of the Cartesian family (utils/jet_analysis/anomaly_detection.py:251-419), one CTA per jet:
//   x = scale * get_real(recon), t = scale * target (scale = factor[b] or 1: the reference scores both the un-normalised and the
//   normalised jets), N == M.  out[b] = [chamfer (Euclidean norm, :498-503: mean_i (min_j |x_i - t_j| + min_j |x_j - t_i|)),
//   mse (:473: mean_i |x_i - t_i|^2), chamfer_lorentz (:523-527, Minkowski square instead of the norm), mse_lorentz (:428-437),
//   jet mse (:405: |sum_i x_i - sum_i t_i|^2), jet mse_lorentz (:419)].
__global__ void __launch_bounds__(128) scores_kernel(const double* recon, const double* target, const double* factor, int B, int N, int mode,
                                                     double* out) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(128) double smem[];
    double* x = smem;          // N*4
    double* t = x + 4 * N;     // N*4
    double* red = t + 4 * N;   // 4 * N : per-particle terms
    __shared__ double scratch[32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int64_t plane = (int64_t)B * N * 4;
    const double sc = factor ? factor[b] : 1.0;
    for (int k = tid; k < 4 * N; k += blockDim.x) {
        x[k] = sc * get_real_value(mode, recon[(int64_t)b * N * 4 + k], recon[plane + (int64_t)b * N * 4 + k]);
        t[k] = sc * target[(int64_t)b * N * 4 + k];
    }
    __syncthreads();
    auto lor = [](double d0, double d1, double d2, double d3) { return d0 * d0 - d1 * d1 - d2 * d2 - d3 * d3; };
    for (int i = tid; i < N; i += blockDim.x) {
        double e_pq = INFINITY, e_qp = INFINITY, l_pq = INFINITY, l_qp = INFINITY;
        for (int j = 0; j < N; ++j) {
            // dist[i][j] = d(x_i, t_j): min over j (dim -1) and, for the other direction, min over the first index of dist[j][i]
            const double a0 = x[4 * i] - t[4 * j], a1 = x[4 * i + 1] - t[4 * j + 1], a2 = x[4 * i + 2] - t[4 * j + 2], a3 = x[4 * i + 3] - t[4 * j + 3];
            const double c0 = x[4 * j] - t[4 * i], c1 = x[4 * j + 1] - t[4 * i + 1], c2 = x[4 * j + 2] - t[4 * i + 2], c3 = x[4 * j + 3] - t[4 * i + 3];
            e_pq = fmin(e_pq, sqrt(a0 * a0 + a1 * a1 + a2 * a2 + a3 * a3));
            e_qp = fmin(e_qp, sqrt(c0 * c0 + c1 * c1 + c2 * c2 + c3 * c3));
            l_pq = fmin(l_pq, lor(a0, a1, a2, a3));
            l_qp = fmin(l_qp, lor(c0, c1, c2, c3));
        }
        const double d0 = x[4 * i] - t[4 * i], d1 = x[4 * i + 1] - t[4 * i + 1], d2 = x[4 * i + 2] - t[4 * i + 2], d3 = x[4 * i + 3] - t[4 * i + 3];
        red[i] = e_pq + e_qp;
        red[N + i] = d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
        red[2 * N + i] = l_pq + l_qp;
        red[3 * N + i] = lor(d0, d1, d2, d3);
    }
    __syncthreads();
    double res[4];
    for (int s = 0; s < 4; ++s) {
        double acc = 0.0;
        for (int i = tid; i < N; i += blockDim.x) acc += red[s * N + i];
        res[s] = block_sum(acc, scratch);
    }
    double jd[4];
    for (int mu = 0; mu < 4; ++mu) {
        double acc = 0.0;
        for (int i = tid; i < N; i += blockDim.x) acc += x[4 * i + mu] - t[4 * i + mu];
        jd[mu] = block_sum(acc, scratch);
    }
    if (tid == 0) {
        double* o = out + (int64_t)b * 6;
        o[0] = res[0] / N; o[1] = res[1] / N; o[2] = res[2] / N; o[3] = res[3] / N;
        o[4] = jd[0] * jd[0] + jd[1] * jd[1] + jd[2] * jd[2] + jd[3] * jd[3];
        o[5] = lor(jd[0], jd[1], jd[2], jd[3]);
    }
}

// Decoder tail of a training step, one CTA per jet: mix_to_output + rep_to_p (reconstruction), get_real('sum') + chamfer against
// the target jet, the loss gradient, and the adjoint of the output map -- dec_output, chamfer, chamfer_sum and dec_output_bwd
// in one launch.  The last CTA to finish adds up the per-jet losses in a fixed order (`counter` must be zero at launch; it is
// reset for the next one).  Row of partials per CTA: [out00 (2C, zero: the output scalars do not reach the loss) | out11 (2C)].
struct DecTailArgs {
    const double* theta;
    int64_t off11;
    int B, N, M, C;
    int mode;               // LGAE_GET_REAL_*
    const double* V;        // (B,N,C,4,2) node vectors after the last level
    const double* target;   // (B,M,4)
    double* recon;          // (2,B,N,4)
    double* g_recon;        // (2,B,N,4) or nullptr
    double* gV;             // (B,N,C,4,2) gradient wrt V
    double* jet_loss;       // (B)
    double* loss;           // (1)
    unsigned int* counter;
    double* partials;
    int64_t part_stride;
};
__global__ void __launch_bounds__(128) dec_tail_kernel(const DecTailArgs a) {
    pdl_launch();
    extern __shared__ __align__(128) double smem[];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = a.N, M = a.M, C = a.C, B = a.B;
    cplx* V_s = reinterpret_cast<cplx*>(smem);          // N*C*4
    cplx* gg_s = V_s + N * C * 4;                        // N*4   canonical gradient of the generated vectors
    cplx* w_s = gg_s + N * 4;                            // C
    double* x = reinterpret_cast<double*>(w_s + C);      // N*4
    double* t = x + 4 * N;                               // M*4
    double* m1 = t + 4 * M;                              // N
    double* m2 = m1 + N;                                 // M
    int* j1 = reinterpret_cast<int*>(m2 + M);            // N
    int* i2 = j1 + N;                                    // M
    __shared__ double dir_sum[2];
    __shared__ double scratch[32];
    __shared__ bool is_last;
    for (int c = tid; c < C; c += blockDim.x) w_s[c] = wget(a.theta, a.off11, 1, C, 0, c);
    pdl_wait();
    {
        const double2* gv = reinterpret_cast<const double2*>(a.V) + (int64_t)b * N * C * 4;
        for (int k = tid; k < N * C * 4; k += blockDim.x) V_s[k] = gv[k];
        for (int k = tid; k < 4 * M; k += blockDim.x) t[k] = a.target[(int64_t)b * M * 4 + k];
    }
    __syncthreads();
    const int64_t plane = (int64_t)B * N * 4;
    // ---- reconstruction (lgn_decoder.py:286-296) ----
    for (int i = tid; i < N; i += blockDim.x) {
        cplx gen[4] = {czero(), czero(), czero(), czero()};
        for (int c = 0; c < C; ++c)
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cfma(gen[mu], w_s[c], V_s[(i * C + c) * 4 + mu]);
        cplx pc[4];
        cart_from_canon(gen, pc);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) {
            a.recon[((int64_t)b * N + i) * 4 + mu] = pc[mu].x;
            a.recon[plane + ((int64_t)b * N + i) * 4 + mu] = pc[mu].y;
            x[4 * i + mu] = get_real_value(a.mode, pc[mu].x, pc[mu].y);   // get_real, utils/utils.py:194-207
        }
    }
    __syncthreads();
    // ---- chamfer (chamfer_loss.py:16-31): the two directions side by side on even / odd warps ----
    auto dist = [&](int i, int j) {
        double s = 0.0;
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) { const double d = x[4 * i + mu] - t[4 * j + mu]; s += d * d; }
        return s;
    };
    const int nw2 = (blockDim.x >> 5) >> 1;
    if ((warp & 1) == 0) {
        for (int i = (warp >> 1) * 32 + lane; i < N; i += nw2 * 32) {
            double best = dist(i, 0);
            int bj = 0;
            for (int j = 1; j < M; ++j) { const double d = dist(i, j); if (d < best) { best = d; bj = j; } }
            m1[i] = best; j1[i] = bj;
        }
    } else {
        for (int j = (warp >> 1) * 32 + lane; j < M; j += nw2 * 32) {
            double best = dist(0, j);
            int bi = 0;
            for (int i = 1; i < N; ++i) { const double d = dist(i, j); if (d < best) { best = d; bi = i; } }
            m2[j] = best; i2[j] = bi;
        }
    }
    __syncthreads();
    if (warp < 2) {
        const double* mm = warp == 0 ? m1 : m2;
        const int n = warp == 0 ? N : M;
        double acc = 0.0;
        for (int k = lane; k < n; k += 32) acc += mm[k];
        acc = warp_sum(acc);
        if (lane == 0) dir_sum[warp] = acc;
    }
    // ---- loss gradient and the adjoint of rep_to_p / mix_to_output ----
    for (int i = tid; i < N; i += blockDim.x) {
        double g[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) g[mu] = x[4 * i + mu] - t[4 * j1[i] + mu];
        for (int j = 0; j < M; ++j)
            if (i2[j] == i) {
#pragma unroll
                for (int mu = 0; mu < 4; ++mu) g[mu] += x[4 * i + mu] - t[4 * j + mu];
            }
        cplx gp[4], gg[4];
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) {
            const int64_t k = ((int64_t)b * N + i) * 4 + mu;
            double re = 0.0, im = 0.0;
            if (a.mode == LGAE_GET_REAL_NORM) { re = a.recon[k]; im = a.recon[plane + k]; }   // written by this thread above
            get_real_grad(a.mode, re, im, x[4 * i + mu], g[mu], gp[mu].x, gp[mu].y);
            if (a.g_recon) {
                a.g_recon[k] = gp[mu].x;
                a.g_recon[plane + k] = gp[mu].y;
            }
        }
        canon_from_cplx(gp, gg);   // adjoint of rep_to_p
        for (int c = 0; c < C; ++c)
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) reinterpret_cast<cplx*>(a.gV)[(((int64_t)b * N + i) * C + c) * 4 + mu] = cmulc(w_s[c], gg[mu]);
#pragma unroll
        for (int mu = 0; mu < 4; ++mu) gg_s[i * 4 + mu] = gg[mu];
    }
    __syncthreads();
    if (tid == 0) a.jet_loss[b] = 0.5 * (dir_sum[0] + dir_sum[1]);
    // ---- output-weight gradient: one warp per channel, lanes over the particles ----
    double* part = a.partials + (int64_t)b * a.part_stride;
    for (int c = warp; c < C; c += blockDim.x >> 5) {
        cplx acc = czero();
        for (int i = lane; i < N; i += 32)
#pragma unroll
            for (int mu = 0; mu < 4; ++mu) cfmac(acc, V_s[(i * C + c) * 4 + mu], gg_s[i * 4 + mu]);
        acc.x = warp_sum(acc.x);
        acc.y = warp_sum(acc.y);
        if (lane == 0) {
            part[c] = 0.0;
            part[C + c] = 0.0;
            part[2 * C + c] = acc.x;
            part[3 * C + c] = acc.y;
        }
    }
    // ---- the last CTA sums the per-jet losses (fixed order => deterministic) ----
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = atomicAdd(a.counter, 1u) == (unsigned)(B - 1);
    __syncthreads();
    if (is_last) {
        __threadfence();
        double s = 0.0;
        for (int k = tid; k < B; k += blockDim.x) s += __ldcg(a.jet_loss + k);
        s = block_sum(s, scratch);
        if (tid == 0) {
            a.loss[0] = s;
            *a.counter = 0u;
        }
    }
}

// Deterministic single-block sum of n values: out[0] = sum (or += when accumulate).
__global__ void __launch_bounds__(1024) sum_kernel(const double* v, int64_t n, double scale, double* out, int accumulate) {
    pdl_launch();
    pdl_wait();
    __shared__ double scratch[32];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += v[i];
    s = block_sum(s, scratch);
    if (threadIdx.x == 0) out[0] = (accumulate ? out[0] : 0.0) + scale * s;
}

__device__ __forceinline__ void normalize_jet(const double* p4, int N, double* out, double* factor, int b, double* scratch) {
    double m = 0.0;
    for (int k = threadIdx.x; k < 4 * N; k += blockDim.x) m = fmax(m, fabs(p4[(int64_t)b * N * 4 + k]));
    // block max via the sum helper's scratch
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = m;
    __syncthreads();
    double f = 0.0;
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) f = fmax(f, scratch[w]);
    f = f + 1e-16;
    if (threadIdx.x == 0 && factor) factor[b] = f;
    for (int k = threadIdx.x; k < 4 * N; k += blockDim.x) out[(int64_t)b * N * 4 + k] = p4[(int64_t)b * N * 4 + k] / f;
}
__global__ void __launch_bounds__(128) normalize_kernel(const double* p4, int N, double* out, double* factor) {
    pdl_launch();
    pdl_wait();
    __shared__ double scratch[32];
    normalize_jet(p4, N, out, factor, blockIdx.x, scratch);
}
// Training step: normalisation and the encoder's input map of one jet per CTA (the normalised momenta are re-read by the
// CTA that wrote them, after a barrier).
__global__ void __launch_bounds__(128) norm_input_kernel(const double* p4, int N, double* out, double* factor, const double* theta,
                                                         int64_t off00, int64_t off11, int C, double* mass, double* S, double* V) {
    pdl_launch();
    pdl_wait();
    __shared__ double scratch[32];
    normalize_jet(p4, N, out, factor, blockIdx.x, scratch);
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) enc_input_node(theta, off00, off11, out, (int64_t)blockIdx.x * N + i, C, mass, S, V);
}

// out = s * in (the encoder's input scale, lgn_encoder.py:371)
__global__ void __launch_bounds__(256) scale_kernel(const double* in, int64_t n, double s, double* out) {
    pdl_launch();
    pdl_wait();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = in[i] * s;
}

// Single block: the parameter vector has ~3e4..3e5 entries.  out[0] += lambda * sum|theta| ; gtheta += lambda * sign(theta).
__global__ void __launch_bounds__(1024) l1_kernel(const double* theta, int64_t n, double lambda, double* out, double* gtheta) {
    pdl_launch();
    pdl_wait();
    __shared__ double scratch[32];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        const double v = theta[i];
        s += fabs(v);
        if (gtheta) gtheta[i] += lambda * (v > 0.0 ? 1.0 : (v < 0.0 ? -1.0 : 0.0));
    }
    s = block_sum(s, scratch);
    if (threadIdx.x == 0 && out) out[0] += lambda * s;
}

// gtheta = lambda * sign(theta) (the L1 regulariser's gradient; zero when lambda == 0); psum[block] = sum |theta| of the block.
constexpr int L1_BLOCKS_MAX = 256;
__global__ void __launch_bounds__(256) grad_init_kernel(const double* theta, int64_t n, double lambda, double* gtheta, double* psum) {
    pdl_launch();
    pdl_wait();
    __shared__ double scratch[32];
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double g = 0.0;
        if (lambda != 0.0) {
            const double v = theta[i];
            s += fabs(v);
            g = lambda * (v > 0.0 ? 1.0 : (v < 0.0 ? -1.0 : 0.0));
        }
        gtheta[i] = g;
    }
    s = block_sum(s, scratch);
    if (threadIdx.x == 0 && psum) psum[blockIdx.x] = s;
}

// Two-model variant of grad_init_kernel for a shared gradient bucket: model A owns [0, na), model B owns [off_b, off_b + nb).
__global__ void __launch_bounds__(256) grad_init2_kernel(const double* theta_a, int64_t na, const double* theta_b, int64_t nb, int64_t off_b,
                                                         double lambda, double* gtheta, double* psum) {
    pdl_launch();
    pdl_wait();
    __shared__ double scratch[32];
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < na + nb; i += (int64_t)gridDim.x * blockDim.x) {
        const bool in_a = i < na;
        double g = 0.0;
        if (lambda != 0.0) {
            const double v = in_a ? theta_a[i] : theta_b[i - na];
            s += fabs(v);
            g = lambda * (v > 0.0 ? 1.0 : (v < 0.0 ? -1.0 : 0.0));
        }
        gtheta[in_a ? i : off_b + (i - na)] = g;
    }
    s = block_sum(s, scratch);
    if (threadIdx.x == 0 && psum) psum[blockIdx.x] = s;
}

// gtheta[seg] += sum over the rows of the segment's block.  blockIdx.y = segment, blockDim = (32 columns, 8 row groups);
// fixed summation order => deterministic gradients.  The extra y-block (blockIdx.y == t.n) adds the L1 term to the loss.
constexpr int RED_Y = 16;   // row lanes per 32-column chunk: a 512-row block of partials is 8 dependent rounds of 4 loads per thread
__global__ void __launch_bounds__(32 * RED_Y) reduce_segs_kernel(const SegTable t, const double* partials, double* gtheta, const double* psum,
                                                          int npsum, double lambda, double* loss) {
    pdl_launch();
    pdl_wait();
    __shared__ double sm[RED_Y][33];
    // blockIdx.x enumerates the 32-column chunks of all segments back to back (t.chunk0[s] = first chunk of segment s); the
    // block after the last chunk adds the L1 term to the loss
    if ((int)blockIdx.x == t.chunk0[t.n]) {
        if (threadIdx.x == 0 && threadIdx.y == 0 && loss) {
            double s = 0.0;
            for (int i = 0; i < npsum; ++i) s += psum[i];
            loss[0] += lambda * s;
        }
        return;
    }
    int si = 0;
    while (si + 1 < t.n && (int)blockIdx.x >= t.chunk0[si + 1]) ++si;
    const Seg sg = t.s[si];
    {
        const int x0 = ((int)blockIdx.x - t.chunk0[si]) * 32;
        const int x = x0 + threadIdx.x;
        double acc = 0.0;
        if (x < sg.len) {
            const double* src = partials + sg.part_off + x;
            int r = threadIdx.y;
            double a1 = 0.0, a2 = 0.0, a3 = 0.0;
            for (; r + 3 * RED_Y < sg.rows; r += 4 * RED_Y) {   // four independent loads in flight
                acc += src[(int64_t)r * sg.stride];
                a1 += src[(int64_t)(r + RED_Y) * sg.stride];
                a2 += src[(int64_t)(r + 2 * RED_Y) * sg.stride];
                a3 += src[(int64_t)(r + 3 * RED_Y) * sg.stride];
            }
            for (; r < sg.rows; r += RED_Y) acc += src[(int64_t)r * sg.stride];
            acc = (acc + a1) + (a2 + a3);
        }
        sm[threadIdx.y][threadIdx.x] = acc;
        __syncthreads();
        if (threadIdx.y == 0 && x < sg.len) {
            double v = 0.0;
#pragma unroll
            for (int y = 0; y < RED_Y; ++y) v += sm[y][threadIdx.x];
            gtheta[sg.theta_off + x] += v;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// host wrappers used by lgae_api.cu
// ------------------------------------------------------------------------------------------------------------
int run_enc_input(const LgaeModelDesc* d, const double* theta, const double* p4, int B, double* mass, double* S, double* V, cudaStream_t st) {
    const int64_t nodes = (int64_t)B * d->n_particles;
    LaunchScope ls_("enc_input", st);
    launch_k(enc_input_kernel, dim3((unsigned)((nodes + 127) / 128)), dim3(128), 0, st, theta, d->off_in00, d->off_in11, p4, nodes, d->channels[0], mass, S, V);
    return check_launch("enc_input");
}
int run_enc_input_bwd(const LgaeModelDesc* d, const double* p4, const double* mass, int B, const double* gS, const double* gV,
                      PartPlan* plan, cudaStream_t st) {
    const int64_t nodes = (int64_t)B * d->n_particles;
    const int C = d->channels[0], grid = sm_count();
    const int64_t w = 4 * C, off = plan->block(grid, w);   // row: [in00 (2C) | in11 (2C)]
    if (int rc = plan->seg(d->off_in00, off, w, 0, 2 * C, grid)) return rc;
    if (int rc = plan->seg(d->off_in11, off, w, 2 * C, 2 * C, grid)) return rc;
    LaunchScope ls_("enc_input_bwd", st);
    launch_k(enc_input_bwd_kernel, dim3(grid), dim3(256), 0, st, 0, 2 * C, p4, mass, nodes, C, gS, gV, plan->base + off, w);
    return check_launch("enc_input_bwd");
}

// CTAs (= rows of partials) of the per-jet glue adjoints: one jet per CTA up to four CTAs per SM.
int glue_grid(int B) {
    const int cap = 4 * sm_count();
    return B < cap ? (B > 0 ? B : 1) : cap;
}

static LatentArgs latent_args(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V) {
    LatentArgs a;
    a.theta = theta; a.off00 = d->off_lat00; a.off11 = d->off_lat11;
    a.B = B; a.N = d->n_particles; a.C = d->channels[d->n_levels]; a.tau_s = d->tau_s; a.tau_v = d->tau_v; a.mode = d->latent_mode;
    a.parts = 3;
    a.S = S; a.V = V; a.lat00 = nullptr; a.lat11 = nullptr; a.sel = nullptr; a.g_lat00 = nullptr; a.g_lat11 = nullptr;
    a.gS = nullptr; a.gV = nullptr; a.partials = nullptr; a.part_stride = 0; a.po00 = 0; a.po11 = 0;
    return a;
}
int run_enc_latent(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V, double* lat00, double* lat11,
                   int32_t* sel, cudaStream_t st, int parts) {
    LatentArgs a = latent_args(d, theta, B, S, V);
    a.lat00 = lat00; a.lat11 = lat11; a.sel = sel; a.parts = parts;
    const int rows = a.mode == LGAE_LATENT_MIX ? 1 : a.N;
    const size_t bytes = (size_t)rows * (a.tau_s + 4 * a.tau_v) * sizeof(cplx);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)enc_latent_kernel, bytes)) return rc;
    LaunchScope ls_("enc_latent", st);
    launch_k(enc_latent_kernel, dim3(B), dim3(256), bytes, st, a);
    return check_launch("enc_latent");
}
int run_enc_latent_bwd(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V, const int32_t* sel,
                       const double* g_lat00, const double* g_lat11, double* gS, double* gV, PartPlan* plan, cudaStream_t st) {
    LatentArgs a = latent_args(d, theta, B, S, V);
    a.sel = const_cast<int32_t*>(sel); a.g_lat00 = g_lat00; a.g_lat11 = g_lat11; a.gS = gS; a.gV = gV;
    const int mix = a.mode == LGAE_LATENT_MIX;
    const int rows = mix ? 1 : a.N, cin = mix ? a.N * a.C : a.C;
    const int grid = glue_grid(B);
    {
        const int64_t n00 = (int64_t)2 * a.tau_s * cin, n11 = (int64_t)2 * a.tau_v * cin, w = n00 + n11, off = plan->block(grid, w);
        if (int rc = plan->seg(a.off00, off, w, 0, n00, grid)) return rc;
        if (int rc = plan->seg(a.off11, off, w, n00, n11, grid)) return rc;
        a.partials = plan->base + off; a.part_stride = w; a.po00 = 0; a.po11 = n00;
    }
    const size_t bytes = ((size_t)rows * (a.tau_s + 4 * a.tau_v) + (size_t)2 * (a.tau_s + a.tau_v) * cin + (size_t)5 * a.N * a.C) * sizeof(cplx);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)enc_latent_bwd_kernel, bytes)) return rc;
    LaunchScope ls_("enc_latent_bwd", st);
    launch_k(enc_latent_bwd_kernel, dim3(grid), dim3(256), bytes, st, a);
    return check_launch("enc_latent_bwd");
}

static DecInArgs dec_in_args(const LgaeModelDesc* d, const double* theta, int B, const double* lat11, double* y, double* S, double* V) {
    DecInArgs a;
    a.theta = theta; a.off_g11 = d->off_graph11; a.off_in00 = d->off_in00; a.off_in11 = d->off_in11;
    a.B = B; a.N = d->n_particles; a.C = d->channels[0]; a.tau = d->tau_v; a.lat11 = lat11; a.y = y; a.S = S; a.V = V;
    a.gS = nullptr; a.gV = nullptr; a.gy = nullptr; a.g_lat11 = nullptr; a.partials = nullptr; a.part_stride = 0; a.po_g11 = a.po_in00 = a.po_in11 = 0;
    return a;
}
int run_dec_input(const LgaeModelDesc* d, const double* theta, int B, const double* lat11, double* y, double* S, double* V, cudaStream_t st) {
    DecInArgs a = dec_in_args(d, theta, B, lat11, y, S, V);
    const size_t bytes = (size_t)a.tau * 4 * sizeof(cplx);
    LaunchScope ls_("dec_input", st);
    launch_k(dec_input_kernel, dim3(B), dim3(128), bytes, st, a);
    return check_launch("dec_input");
}
// Shared memory of enc_latent_body (the first region of latent_bridge_kernel's).
static size_t latent_bridge_scratch_bytes(const LgaeModelDesc* de) {
    const int rows = de->latent_mode == LGAE_LATENT_MIX ? 1 : de->n_particles;
    return (size_t)rows * (de->tau_s + 4 * de->tau_v) * sizeof(cplx);
}
// enc_latent + dec_input fused (training step / inference of both models back to back).
int run_latent_bridge(const LgaeModelDesc* de, const double* theta_e, const LgaeModelDesc* dd, const double* theta_d, int B, const double* S,
                      const double* V, double* lat00, double* lat11, int32_t* sel, double* y, double* S0, double* V0, cudaStream_t st, int parts) {
    LatentArgs a = latent_args(de, theta_e, B, S, V);
    a.lat00 = lat00; a.lat11 = lat11; a.sel = sel; a.parts = parts;
    DecInArgs di = dec_in_args(dd, theta_d, B, lat11, y, S0, V0);
    const int mult = a.mode == LGAE_LATENT_MINMAX ? 2 : 1;
    if (di.tau != mult * a.tau_v) return LGAE_E_BADARG;   // decoder latent width must be the encoder's output width
    const size_t scratch = latent_bridge_scratch_bytes(de);
    const size_t bytes = scratch + (size_t)di.tau * 4 * sizeof(cplx);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)latent_bridge_kernel, bytes)) return rc;
    LaunchScope ls_("latent_bridge", st);
    launch_k(latent_bridge_kernel, dim3(B), dim3(256), bytes, st, a, di, (int)(scratch / sizeof(double)));
    return check_launch("latent_bridge");
}
int run_dec_input_bwd(const LgaeModelDesc* d, const double* theta, int B, const double* lat11, double* y, const double* gS, const double* gV,
                      const double* gy, double* g_lat11, PartPlan* plan, cudaStream_t st) {
    DecInArgs a = dec_in_args(d, theta, B, lat11, y, nullptr, nullptr);
    a.gS = gS; a.gV = gV; a.gy = gy; a.g_lat11 = g_lat11;
    const int grid = glue_grid(B);
    {
        const int64_t ng = (int64_t)2 * a.N * a.tau, w = ng + 4 * a.C, off = plan->block(grid, w);
        if (int rc = plan->seg(a.off_g11, off, w, 0, ng, grid)) return rc;
        if (int rc = plan->seg(a.off_in00, off, w, ng, 2 * a.C, grid)) return rc;
        if (int rc = plan->seg(a.off_in11, off, w, ng + 2 * a.C, 2 * a.C, grid)) return rc;
        a.partials = plan->base + off; a.part_stride = w; a.po_g11 = 0; a.po_in00 = ng; a.po_in11 = ng + 2 * a.C;
    }
    const size_t bytes = ((size_t)a.tau * 4 + (size_t)a.N * 4 + (size_t)a.N * a.tau + 2 * a.C) * sizeof(cplx);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)dec_input_bwd_kernel, bytes)) return rc;
    LaunchScope ls_("dec_input_bwd", st);
    launch_k(dec_input_bwd_kernel, dim3(grid), dim3(128), bytes, st, a);
    return check_launch("dec_input_bwd");
}
// Shared memory of latent_bridge_bwd_kernel: [dec_input_bwd | enc_latent_bwd | latent gradient], in complex numbers, each
// region rounded up to 8.  0 if the two models do not fit together (latent widths or particle counts differ).
static size_t latent_bridge_bwd_cd(const LgaeModelDesc* dd) {
    return (dec_input_bwd_smem_cplx(dd->n_particles, dd->channels[0], dd->tau_v) + 7) & ~(size_t)7;
}
static size_t latent_bridge_bwd_smem_cplx(const LgaeModelDesc* dd, const LgaeModelDesc* de) {
    const int mult = de->latent_mode == LGAE_LATENT_MINMAX ? 2 : 1;
    if (dd->tau_v != mult * de->tau_v || dd->n_particles != de->n_particles) return 0;
    const size_t ce = (enc_latent_bwd_smem_cplx(de->n_particles, de->channels[de->n_levels], de->tau_s, de->tau_v, de->latent_mode) + 7) &
                      ~(size_t)7;
    return latent_bridge_bwd_cd(dd) + ce + (size_t)dd->tau_v * 4;
}
// dec_input_bwd + enc_latent_bwd fused (training step).  g_lat11 is still written (API output).
int run_latent_bridge_bwd(const LgaeModelDesc* dd, const double* theta_d, const LgaeModelDesc* de, const double* theta_e, int B,
                          const double* lat11, double* y, const double* gS_d, const double* gV_d, const double* gy, double* g_lat11,
                          const double* S, const double* V, const int32_t* sel, double* gS_e, double* gV_e, PartPlan* plan_d,
                          PartPlan* plan_e, cudaStream_t st) {
    // plan_d / plan_e: the decoder's and the encoder's plans (they may be the same object); both allocate from one buffer,
    // the encoder's plan continues where the decoder's ends
    DecInArgs di = dec_in_args(dd, theta_d, B, lat11, y, nullptr, nullptr);
    di.gS = gS_d; di.gV = gV_d; di.gy = gy; di.g_lat11 = g_lat11;
    LatentArgs a = latent_args(de, theta_e, B, S, V);
    a.sel = const_cast<int32_t*>(sel); a.g_lat00 = nullptr; a.g_lat11 = nullptr; a.gS = gS_e; a.gV = gV_e;
    const size_t smem = latent_bridge_bwd_smem_cplx(dd, de);
    if (smem == 0) return LGAE_E_BADARG;
    const int mix = a.mode == LGAE_LATENT_MIX;
    const int cin = mix ? a.N * a.C : a.C;
    const int grid = glue_grid(B);
    {
        const int64_t ng = (int64_t)2 * di.N * di.tau, w = ng + 4 * di.C, off = plan_d->block(grid, w);
        if (int rc = plan_d->seg(di.off_g11, off, w, 0, ng, grid)) return rc;
        if (int rc = plan_d->seg(di.off_in00, off, w, ng, 2 * di.C, grid)) return rc;
        if (int rc = plan_d->seg(di.off_in11, off, w, ng + 2 * di.C, 2 * di.C, grid)) return rc;
        di.partials = plan_d->base + off; di.part_stride = w; di.po_g11 = 0; di.po_in00 = ng; di.po_in11 = ng + 2 * di.C;
    }
    if (plan_e != plan_d) plan_e->used = plan_d->used;
    {
        const int64_t n00 = (int64_t)2 * a.tau_s * cin, n11 = (int64_t)2 * a.tau_v * cin, w = n00 + n11, off = plan_e->block(grid, w);
        if (int rc = plan_e->seg(a.off00, off, w, 0, n00, grid)) return rc;
        if (int rc = plan_e->seg(a.off11, off, w, n00, n11, grid)) return rc;
        a.partials = plan_e->base + off; a.part_stride = w; a.po00 = 0; a.po11 = n00;
    }
    const size_t cd = latent_bridge_bwd_cd(dd), ce = smem - cd - (size_t)di.tau * 4;
    const size_t bytes = smem * sizeof(cplx);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)latent_bridge_bwd_kernel, bytes)) return rc;
    LaunchScope ls_("latent_bridge_bwd", st);
    launch_k(latent_bridge_bwd_kernel, dim3(grid), dim3(256), bytes, st, di, a, (int)(2 * cd), (int)(2 * (cd + ce)));
    return check_launch("latent_bridge_bwd");
}
int run_dec_output(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V, double* recon, double* gen00, cudaStream_t st) {
    const int64_t nodes = (int64_t)B * d->n_particles;
    LaunchScope ls_("dec_output", st);
    launch_k(dec_output_kernel, dim3((unsigned)((nodes + 127) / 128)), dim3(128), 0, st, theta, d->off_out00, d->off_out11, B, d->n_particles, d->channels[d->n_levels], S, V, recon, gen00);
    return check_launch("dec_output");
}
int run_dec_output_bwd(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V, const double* g_recon,
                       const double* g_gen00, double* gS, double* gV, PartPlan* plan, cudaStream_t st) {
    const int C = d->channels[d->n_levels], grid = sm_count();
    const int64_t w = 4 * C, off = plan->block(grid, w);
    if (int rc = plan->seg(d->off_out00, off, w, 0, 2 * C, grid)) return rc;
    if (int rc = plan->seg(d->off_out11, off, w, 2 * C, 2 * C, grid)) return rc;
    LaunchScope ls_("dec_output_bwd", st);
    launch_k(dec_output_bwd_kernel, dim3(grid), dim3(256), 0, st, theta, d->off_out00, d->off_out11, B, d->n_particles, C, S, V, g_recon, g_gen00, gS, gV, plan->base + off, w);
    return check_launch("dec_output_bwd");
}
// gtheta = lambda sign(theta) (0 when lambda == 0), then every segment of the plan is reduced over its rows and added;
// loss[0] += lambda |theta|_1 when loss != NULL.  Uses L1_BLOCKS_MAX doubles of scratch behind the plan's blocks.
int run_reduce_plan(PartPlan* plan, int64_t n_params, double* gtheta, const double* theta, double lambda, double* loss, cudaStream_t st) {
    const bool l1 = lambda != 0.0 && theta;
    int nb = (int)((n_params + 1023) / 1024);
    nb = nb < 1 ? 1 : (nb > L1_BLOCKS_MAX ? L1_BLOCKS_MAX : nb);
    double* psum = plan->base + plan->used;
    {
        LaunchScope ls_("grad_init", st);
        launch_k(grad_init_kernel, dim3(nb), dim3(256), 0, st, theta, n_params, l1 ? lambda : 0.0, gtheta, l1 ? psum : nullptr);
        if (int rc = check_launch("grad_init")) return rc;
    }
    if (plan->table.n == 0 && !l1) return LGAE_OK;
    int chunks = 0;
    for (int i = 0; i < plan->table.n; ++i) {
        plan->table.chunk0[i] = chunks;
        chunks += (plan->table.s[i].len + 31) / 32;
    }
    plan->table.chunk0[plan->table.n] = chunks;
    LaunchScope ls_("reduce_partials", st);
    launch_k(reduce_segs_kernel, dim3(chunks + 1), dim3(32, RED_Y), 0, st, plan->table, plan->base, gtheta, psum, nb, lambda, l1 ? loss : nullptr);
    return check_launch("reduce_partials");
}
int reduce_scratch_doubles() { return L1_BLOCKS_MAX; }

// The same for two models whose gradients share one bucket (segments of model B were declared with plan->theta_base = off_b).
// The two halves of run_reduce_plan2, so that a caller can run the gradient init early on another stream (it only needs
// theta): psum = L1_BLOCKS_MAX doubles of scratch that nothing else touches between the two launches.
int run_grad_init2(const double* theta_a, int64_t na, const double* theta_b, int64_t nb, int64_t off_b, double* gtheta, double lambda,
                   double* psum, cudaStream_t st) {
    const bool l1 = lambda != 0.0;
    int nblk = (int)((na + nb + 1023) / 1024);
    nblk = nblk < 1 ? 1 : (nblk > L1_BLOCKS_MAX ? L1_BLOCKS_MAX : nblk);
    LaunchScope ls_("grad_init", st);
    launch_k(grad_init2_kernel, dim3(nblk), dim3(256), 0, st, theta_a, na, theta_b, nb, off_b, l1 ? lambda : 0.0, gtheta, l1 ? psum : nullptr);
    return check_launch("grad_init");
}
int run_reduce_segs(PartPlan* plan, int64_t n_params, double* gtheta, const double* psum, double lambda, double* loss, cudaStream_t st) {
    const bool l1 = lambda != 0.0;
    int nblk = (int)((n_params + 1023) / 1024);
    nblk = nblk < 1 ? 1 : (nblk > L1_BLOCKS_MAX ? L1_BLOCKS_MAX : nblk);
    if (plan->table.n == 0 && !l1) return LGAE_OK;
    int chunks = 0;
    for (int i = 0; i < plan->table.n; ++i) {
        plan->table.chunk0[i] = chunks;
        chunks += (plan->table.s[i].len + 31) / 32;
    }
    plan->table.chunk0[plan->table.n] = chunks;
    LaunchScope ls_("reduce_partials", st);
    launch_k(reduce_segs_kernel, dim3(chunks + 1), dim3(32, RED_Y), 0, st, plan->table, plan->base, gtheta, psum, nblk, lambda, l1 ? loss : nullptr);
    return check_launch("reduce_partials");
}
int run_reduce_plan2(PartPlan* plan, const double* theta_a, int64_t na, const double* theta_b, int64_t nb, int64_t off_b, double* gtheta,
                     double lambda, double* loss, cudaStream_t st) {
    double* psum = plan->base + plan->used;
    if (int rc = run_grad_init2(theta_a, na, theta_b, nb, off_b, gtheta, lambda, psum, st)) return rc;
    return run_reduce_segs(plan, na + nb, gtheta, psum, lambda, loss, st);
}
// Doubles of partial rows used by the glue adjoints of a model.
int64_t glue_part_doubles(const LgaeModelDesc* d, int batch) {
    const int64_t g = sm_count(), gj = glue_grid(batch);
    if (d->is_decoder) return gj * ((int64_t)2 * d->n_particles * d->tau_v + 4 * d->channels[0]) + g * 4 * d->channels[d->n_levels];
    const int mix = d->latent_mode == LGAE_LATENT_MIX;
    const int64_t cin = mix ? (int64_t)d->n_particles * d->channels[d->n_levels] : d->channels[d->n_levels];
    return g * 4 * d->channels[0] + gj * 2 * (d->tau_s + d->tau_v) * cin;
}
int run_chamfer(const double* recon, const double* target, int B, int N, int M, double* loss, double* jet_loss, const double* g_loss,
                double* g_recon, int mode, cudaStream_t st) {
    const size_t bytes = (size_t)(4 * N + 4 * M + N + M) * sizeof(double) + (size_t)(N + M) * sizeof(int);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)chamfer_kernel, bytes)) return rc;
    LaunchScope ls_("chamfer", st);
    launch_k(chamfer_kernel, dim3(B), dim3(128), bytes, st, recon, target, B, N, M, jet_loss, g_loss, g_recon, mode);
    int rc = check_launch("chamfer");
    if (rc) return rc;
    if (loss) {
        LaunchScope ls_("chamfer_sum", st);
        launch_k(sum_kernel, dim3(1), dim3(1024), 0, st, jet_loss, B, 1.0, loss, 0);
        rc = check_launch("chamfer_sum");
    }
    return rc;
}
int run_scores(const double* recon, const double* target, const double* factor, int B, int N, int mode, double* out, cudaStream_t st) {
    const size_t bytes = (size_t)12 * N * sizeof(double);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)scores_kernel, bytes)) return rc;
    LaunchScope ls_("anomaly_scores", st);
    launch_k(scores_kernel, dim3(B), dim3(128), bytes, st, recon, target, factor, B, N, mode, out);
    return check_launch("anomaly_scores");
}
static size_t dec_tail_bytes(int N, int M, int C) {
    return ((size_t)N * C * 4 + N * 4 + C) * sizeof(cplx) + (size_t)(4 * N + 4 * M + N + M) * sizeof(double) + (size_t)(N + M) * sizeof(int);
}
// mix_to_output + chamfer + their adjoints for a training step (see dec_tail_kernel).  `counter`: 4 bytes of device scratch.
int run_dec_tail(const LgaeModelDesc* d, const double* theta, int B, int M, const double* V, const double* target, double* recon,
                 double* g_recon, double* gV, double* jet_loss, double* loss, unsigned int* counter, int mode, PartPlan* plan, cudaStream_t st) {
    DecTailArgs a;
    a.mode = mode;
    a.theta = theta; a.off11 = d->off_out11;
    a.B = B; a.N = d->n_particles; a.M = M; a.C = d->channels[d->n_levels];
    a.V = V; a.target = target; a.recon = recon; a.g_recon = g_recon; a.gV = gV; a.jet_loss = jet_loss; a.loss = loss; a.counter = counter;
    const int C = a.C, N = a.N;
    const int64_t w = 4 * C, off = plan->block(B, w);
    if (int rc = plan->seg(d->off_out00, off, w, 0, 2 * C, B)) return rc;
    if (int rc = plan->seg(d->off_out11, off, w, 2 * C, 2 * C, B)) return rc;
    a.partials = plan->base + off; a.part_stride = w;
    const size_t bytes = dec_tail_bytes(N, M, C);
    if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
    if (int rc = ensure_smem((const void*)dec_tail_kernel, bytes)) return rc;
    if (cudaMemsetAsync(counter, 0, sizeof(unsigned int), st) != cudaSuccess) return check_launch("memset counter");
    LaunchScope ls_("dec_tail", st);
    launch_k(dec_tail_kernel, dim3(B), dim3(128), bytes, st, a);
    return check_launch("dec_tail");
}
int run_norm_input(const LgaeModelDesc* d, const double* theta, const double* p4, int B, double* out, double* factor, double* mass, double* S,
                   double* V, cudaStream_t st) {
    LaunchScope ls_("norm_input", st);
    launch_k(norm_input_kernel, dim3(B), dim3(128), 0, st, p4, d->n_particles, out, factor, theta, d->off_in00, d->off_in11, d->channels[0], mass, S, V);
    return check_launch("norm_input");
}
int run_normalize(const double* p4, int B, int N, double* out, double* factor, cudaStream_t st) {
    LaunchScope ls_("normalize_p4", st);
    launch_k(normalize_kernel, dim3(B), dim3(128), 0, st, p4, N, out, factor);
    return check_launch("normalize_p4");
}
int run_scale(const double* in, int64_t n, double s, double* out, cudaStream_t st) {
    LaunchScope ls_("scale_input", st);
    const int grid = (int)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
    launch_k(scale_kernel, dim3(grid), dim3(256), 0, st, in, n, s, out);
    return check_launch("scale_input");
}
int run_l1(const double* theta, int64_t n, double lambda, double* out, double* gtheta, cudaStream_t st) {
    LaunchScope ls_("l1", st);
    launch_k(l1_kernel, dim3(1), dim3(1024), 0, st, theta, n, lambda, out, gtheta);
    return check_launch("l1");
}

}  // namespace lgae

namespace lgae {
// LGAE_OK if the adjoints of the model's input and output maps fit their kernels' shared memory at its particle count (the
// checks run_enc_latent_bwd / run_dec_input_bwd make before launching), else LGAE_E_UNSUPPORTED.  No GPU needed.
int glue_bwd_check(const LgaeModelDesc* d) {
    const size_t n = d->is_decoder ? dec_input_bwd_smem_cplx(d->n_particles, d->channels[0], d->tau_v)
                                   : enc_latent_bwd_smem_cplx(d->n_particles, d->channels[d->n_levels], d->tau_s, d->tau_v, d->latent_mode);
    return n * sizeof(cplx) > 200 * 1024 ? LGAE_E_UNSUPPORTED : LGAE_OK;
}
// The same for the fused glue kernels of the training step (latent_bridge, dec_tail, latent_bridge_bwd), with the checks their
// launchers make: LGAE_E_BADARG if the two models do not fit together, LGAE_E_UNSUPPORTED if a kernel's shared memory does not
// fit.  No GPU needed.
int train_step_glue_check(const LgaeModelDesc* de, const LgaeModelDesc* dd) {
    const size_t bridge_bwd = latent_bridge_bwd_smem_cplx(dd, de);
    if (bridge_bwd == 0) return LGAE_E_BADARG;
    const size_t lim = 200 * 1024;
    if (bridge_bwd * sizeof(cplx) > lim || latent_bridge_scratch_bytes(de) + (size_t)dd->tau_v * 4 * sizeof(cplx) > lim ||
        dec_tail_bytes(dd->n_particles, de->n_particles, dd->channels[dd->n_levels]) > lim)
        return LGAE_E_UNSUPPORTED;
    return LGAE_OK;
}
}  // namespace lgae
