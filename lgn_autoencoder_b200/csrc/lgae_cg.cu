// Layer-level kernels of the reference's generic API, for any maxdim:
//   * Clebsch-Gordan product of one (irrep1, irrep2) pair, channel-wise, point-wise or aggregated over the neighbour
//     axis, forward and adjoint  (lgn/cg_lib/cg_ops.py:135-298: cg_product / complex_kron_product);
//   * per-irrep complex channel mixing W.x, forward and adjoint  (lgn/nn/g_nn.py:95-121, lgn/g_lib/cplx_lib.py:7-25).
// The reference materialises the Kronecker product (4,B,N,N,C,d1*d2) and multiplies by the dense CG matrix; here the
// non-zero CG coefficients are a term list (out component, a, d, coefficient) staged in shared memory, the neighbour sum
// runs over shared-memory slabs of the jet and nothing of size N*N*d1*d2 is ever written.
//
// Tensors are the reference's planar complex layout: (2, ..., C, d) with the leading index re/im.
#include <algorithm>
#include <cstring>

#include "lgae_common.cuh"

namespace lgae {

struct CgOut {
    double* ptr;      // forward: output part; adjoint: its gradient
    int64_t plane;    // distance re -> im (doubles)
    int32_t d, comp0, ctot, coff;
};
struct CgArgs {
    const double *z1, *z2;
    double *g1, *g2;
    int64_t plane1, plane2;
    int32_t B, N, NJ, C, d1, d2, n_comp, n_terms, n_out, JT, acc1, acc2;
    int32_t JS;           // forward: lanes that share one output item and split the neighbour sum (power of two <= 32)
    const int32_t* tab;   // [3 orderings][n_terms][3] (comp, a, d), then comp_start[n_comp+1], a_start[d1+1], d_start[d2+1]
    const double* coef;   // [3 orderings][n_terms]
    CgOut out[LGAE_CG_MAX_OUT];
};

constexpr int CG_THREADS = 256;
constexpr int CG_ITEMS = 4;   // work items per thread held in registers
constexpr size_t CG_SMEM_MAX = 227 * 1024;   // dynamic shared memory one sm_100 CTA may opt in to

// Term list of one ordering (0: by output component, 1: by a, 2: by d) -> shared memory.
struct TermsSm {
    int32_t *comp, *a, *d, *start;
    double* coef;
};
LGAE_DEV int terms_start_len(const CgArgs& p, int ord) { return (ord == 0 ? p.n_comp : ord == 1 ? p.d1 : p.d2) + 1; }
LGAE_DEV const int32_t* terms_start_src(const CgArgs& p, int ord) {
    const int32_t* s = p.tab + (int64_t)9 * p.n_terms;
    if (ord >= 1) s += p.n_comp + 1;
    if (ord >= 2) s += p.d1 + 1;
    return s;
}
// carve `mem` (8-byte aligned); returns the number of doubles consumed
LGAE_DEV int terms_load(const CgArgs& p, int ord, double* mem, TermsSm& t) {
    const int n = p.n_terms, ns = terms_start_len(p, ord);
    t.coef = mem;
    t.comp = reinterpret_cast<int32_t*>(mem + n);
    t.a = t.comp + n;
    t.d = t.a + n;
    t.start = t.d + n;
    const int32_t* src = p.tab + (int64_t)ord * 3 * n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        t.coef[i] = p.coef[(int64_t)ord * n + i];
        t.comp[i] = src[3 * i];
        t.a[i] = src[3 * i + 1];
        t.d[i] = src[3 * i + 2];
    }
    const int32_t* ss = terms_start_src(p, ord);
    for (int i = threadIdx.x; i < ns; i += blockDim.x) t.start[i] = ss[i];
    return n + (3 * n + ns + 1) / 2;
}
static size_t terms_doubles(int n_terms, int n_start) { return (size_t)n_terms + (size_t)(3 * n_terms + n_start + 1) / 2; }

LGAE_DEV int out_of_comp(const CgArgs& p, int oc) {
    int o = 0;
    while (o + 1 < p.n_out && oc >= p.out[o + 1].comp0) ++o;
    return o;
}
LGAE_DEV void stage_planar(cplx* dst, const double* src, int64_t plane, int n) {
    for (int t = threadIdx.x; t < n; t += blockDim.x) dst[t] = cmake(src[t], src[plane + t]);
}
// The same with one row of `rowlen` complex numbers per neighbour, rows `stride` apart.  stride = rowlen | 1 (odd): lanes
// that split the neighbour sum of one item read the same column of consecutive rows, 16 bytes each, from different banks.
__host__ __device__ inline int cg_row_stride(int rowlen) { return rowlen | 1; }
LGAE_DEV void stage_rows(cplx* dst, const double* src, int64_t plane, int rows, int rowlen) {
    const int stride = cg_row_stride(rowlen), n = rows * rowlen;
    for (int t = threadIdx.x; t < n; t += blockDim.x) dst[(t / rowlen) * stride + t % rowlen] = cmake(src[t], src[plane + t]);
}

// ------------------------------------------------------------------------------------------------------------
// aggregated product: out_i = sum_j H (z1_j (x) z2_ij);  z1 (2,B,NJ,C,d1), z2 (2,B,N,NJ,C,d2)
// grid (B, i-split); the neighbour axis is processed in tiles of JT particles held in shared memory.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CG_THREADS) cg_agg_fwd_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, d1 = p.d1, d2 = p.d2, NJ = p.NJ, JT = p.JT;
    const int S1 = cg_row_stride(C * d1), S2 = cg_row_stride(C * d2);
    cplx* z1s = reinterpret_cast<cplx*>(smem);
    cplx* z2s = z1s + (size_t)JT * S1;
    TermsSm T;
    terms_load(p, 0, reinterpret_cast<double*>(z2s + (size_t)JT * S2), T);
    pdl_wait();
    const int b = blockIdx.x, items = C * p.n_comp;
    const bool single = JT >= NJ;
    if (single) stage_rows(z1s, p.z1 + (int64_t)b * NJ * C * d1, p.plane1, NJ, C * d1);
    const int JS = p.JS, jl = tid % JS, per_pass = CG_THREADS / JS;
    for (int i = blockIdx.y; i < p.N; i += gridDim.y) {
        cplx acc[CG_ITEMS];
#pragma unroll
        for (int k = 0; k < CG_ITEMS; ++k) acc[k] = czero();
        for (int j0 = 0; j0 < NJ; j0 += JT) {
            const int jt = min(JT, NJ - j0);
            __syncthreads();
            if (!single) stage_rows(z1s, p.z1 + ((int64_t)b * NJ + j0) * C * d1, p.plane1, jt, C * d1);
            stage_rows(z2s, p.z2 + (((int64_t)b * p.N + i) * NJ + j0) * C * d2, p.plane2, jt, C * d2);
            __syncthreads();
#pragma unroll
            for (int k = 0; k < CG_ITEMS; ++k) {
                const int it = tid / JS + k * per_pass;
                if (it < items) {
                    const int c = it % C, oc = it / C;
                    for (int t = T.start[oc]; t < T.start[oc + 1]; ++t) {
                        const cplx* x = z1s + c * d1 + T.a[t];
                        const cplx* y = z2s + c * d2 + T.d[t];
                        cplx s = czero();
                        for (int j = jl; j < jt; j += JS) cfma(s, x[j * S1], y[j * S2]);
                        cfmar(acc[k], s, T.coef[t]);
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < CG_ITEMS; ++k) {
            // butterfly over the JS lanes of the item (fixed order); every lane of the warp takes part in the shuffles
            for (int o = JS >> 1; o > 0; o >>= 1) {
                acc[k].x += __shfl_xor_sync(0xffffffffu, acc[k].x, o);
                acc[k].y += __shfl_xor_sync(0xffffffffu, acc[k].y, o);
            }
            const int it = tid / JS + k * per_pass;
            if (it < items && jl == 0) {
                const int c = it % C, oc = it / C;
                const CgOut& o = p.out[out_of_comp(p, oc)];
                const int64_t idx = (((int64_t)b * p.N + i) * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
                o.ptr[idx] = acc[k].x;
                o.ptr[o.plane + idx] = acc[k].y;
            }
        }
    }
}

// Whole-jet variant (the common case: the jet's node slab and IB rows of the edge tensor fit in shared memory):
// grid (B, ceil(N / IB)), no loop and no barrier after the single staging step; a thread owns one (i, channel, output
// component) and runs the whole neighbour sum.  p.JT holds IB.
__global__ void __launch_bounds__(CG_THREADS) cg_agg_fwd_block_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, d1 = p.d1, d2 = p.d2, NJ = p.NJ, IB = p.JT;
    cplx* z1s = reinterpret_cast<cplx*>(smem);
    cplx* z2s = z1s + (size_t)NJ * C * d1;
    TermsSm T;
    terms_load(p, 0, reinterpret_cast<double*>(z2s + (size_t)IB * NJ * C * d2), T);
    pdl_wait();
    const int b = blockIdx.x, i0 = blockIdx.y * IB, ib = min(IB, p.N - i0), items = C * p.n_comp;
    stage_planar(z1s, p.z1 + (int64_t)b * NJ * C * d1, p.plane1, NJ * C * d1);
    stage_planar(z2s, p.z2 + ((int64_t)b * p.N + i0) * NJ * C * d2, p.plane2, ib * NJ * C * d2);
    __syncthreads();
    for (int it = tid; it < ib * items; it += CG_THREADS) {
        const int il = it / items, w = it % items, c = w % C, oc = w / C;
        const cplx* xb = z1s + c * d1;
        const cplx* yb = z2s + ((size_t)il * NJ * C + c) * d2;
        cplx acc = czero();
        for (int t = T.start[oc]; t < T.start[oc + 1]; ++t) {
            const cplx* x = xb + T.a[t];
            const cplx* y = yb + T.d[t];
            cplx s = czero();
            for (int j = 0; j < NJ; ++j) cfma(s, x[(size_t)j * C * d1], y[(size_t)j * C * d2]);
            cfmar(acc, s, T.coef[t]);
        }
        const CgOut& o = p.out[out_of_comp(p, oc)];
        const int64_t idx = (((int64_t)b * p.N + i0 + il) * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
        o.ptr[idx] = acc.x;
        o.ptr[o.plane + idx] = acc.y;
    }
}

// Kronecker-sum form of the whole-jet variant for the common edge dimensions D2 (1, 3, 4, 9): phase 1 builds
// K[a][d] = sum_j z1_j[a] z2_ij[d] per (i, channel) with the d axis in registers (one z1 load + D2 z2 loads per D2 complex
// FMAs instead of two loads per FMA, and d1*d2 products instead of one per CG term); phase 2 applies the CG matrix,
// out[m] = sum_terms coef K[a][d].  Same grid, staging and p.JT = IB as cg_agg_fwd_block_kernel.
template <int D2>
__global__ void __launch_bounds__(CG_THREADS) cg_agg_fwd_kron_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, d1 = p.d1, NJ = p.NJ, IB = p.JT;
    cplx* z1s = reinterpret_cast<cplx*>(smem);
    cplx* z2s = z1s + (size_t)NJ * C * d1;
    cplx* ks = z2s + (size_t)IB * NJ * C * D2;   // IB * C * d1 * D2
    TermsSm T;
    terms_load(p, 0, reinterpret_cast<double*>(ks + (size_t)IB * C * d1 * D2), T);
    pdl_wait();
    const int b = blockIdx.x, i0 = blockIdx.y * IB, ib = min(IB, p.N - i0), items = C * p.n_comp;
    stage_planar(z1s, p.z1 + (int64_t)b * NJ * C * d1, p.plane1, NJ * C * d1);
    stage_planar(z2s, p.z2 + ((int64_t)b * p.N + i0) * NJ * C * D2, p.plane2, ib * NJ * C * D2);
    __syncthreads();
    for (int it = tid; it < ib * C * d1; it += CG_THREADS) {   // (il, c, a), a fastest
        const int a_ = it % d1, c = (it / d1) % C, il = it / (d1 * C);
        const cplx* x = z1s + c * d1 + a_;
        const cplx* y = z2s + ((size_t)il * NJ * C + c) * D2;
        cplx acc[D2];
#pragma unroll
        for (int d = 0; d < D2; ++d) acc[d] = czero();
        for (int j = 0; j < NJ; ++j) {
            const cplx xv = x[(size_t)j * C * d1];
#pragma unroll
            for (int d = 0; d < D2; ++d) cfma(acc[d], xv, y[(size_t)j * C * D2 + d]);
        }
#pragma unroll
        for (int d = 0; d < D2; ++d) ks[(size_t)it * D2 + d] = acc[d];
    }
    __syncthreads();
    for (int it = tid; it < ib * items; it += CG_THREADS) {
        const int il = it / items, w = it % items, c = w % C, oc = w / C;
        const cplx* k = ks + ((size_t)il * C + c) * d1 * D2;
        cplx acc = czero();
        for (int t = T.start[oc]; t < T.start[oc + 1]; ++t) cfmar(acc, k[T.a[t] * D2 + T.d[t]], T.coef[t]);
        const CgOut& o = p.out[out_of_comp(p, oc)];
        const int64_t idx = (((int64_t)b * p.N + i0 + il) * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
        o.ptr[idx] = acc.x;
        o.ptr[o.plane + idx] = acc.y;
    }
}

// All (node irrep, edge irrep) pairs of one aggregated cg_product call in ONE launch (Kronecker form): the rows of every edge
// part are staged once, interleaved per (i, j, channel); K[a][d] is built for all node components a (the node parts are read
// straight from global memory: every element is needed by exactly one thread per i) against all D2T edge components d in
// registers; the CG matrices of all pairs are then applied from one term list.  grid (B, ceil(N / IB)), p.JT = IB.
struct CgMultiArgs {
    const double* node[LGAE_CG_MAX_PARTS];
    const double* edge[LGAE_CG_MAX_PARTS];
    double* out[LGAE_CG_MAX_OUT];
    int32_t node_d[LGAE_CG_MAX_PARTS], node_off[LGAE_CG_MAX_PARTS + 1], edge_d[LGAE_CG_MAX_PARTS], edge_off[LGAE_CG_MAX_PARTS + 1];
    int32_t out_d[LGAE_CG_MAX_OUT], out_ctot[LGAE_CG_MAX_OUT];
    int32_t B, N, NJ, C, n_node, n_edge, n_comp, n_terms, IB;
    const int32_t* tab;    // [n_terms][3] = (component, a_all, d_all) sorted by component, then comp_start[n_comp + 1],
                           // then per component: output tensor, m, channel offset  ([n_comp][3])
    const double* coef;    // [n_terms]
    // adjoint: out[] holds the gradients of the outputs; terms sorted by cell = a_all * D2T + d_all
    const int32_t* tab_b;  // [n_terms] component of every term, then cell_start[D1T * D2T + 1], then the [n_comp][3] output map
    const double* coef_b;  // [n_terms]
    double* gnode[LGAE_CG_MAX_PARTS];
    double* gedge[LGAE_CG_MAX_PARTS];
};
// adjoint helpers: output gradients of IB particles -> shared memory, then gK[a_all][d_all] = sum_terms coef g[component]
LGAE_DEV void multi_stage_g(const CgMultiArgs& p, const int32_t* cinfo, cplx* gs, int b, int i0, int ib) {
    const int C = p.C, nc = p.n_comp;
    for (int t = threadIdx.x; t < ib * C * nc; t += blockDim.x) {
        const int oc = t % nc, c = (t / nc) % C, il = t / (nc * C);
        const int o = cinfo[3 * oc], m = cinfo[3 * oc + 1], coff = cinfo[3 * oc + 2];
        const int64_t rowsz = (int64_t)p.out_ctot[o] * p.out_d[o];
        const int64_t idx = ((int64_t)b * p.N + i0 + il) * rowsz + (int64_t)(coff + c) * p.out_d[o] + m;
        gs[t] = cmake(p.out[o][idx], p.out[o][(int64_t)p.B * p.N * rowsz + idx]);
    }
}
LGAE_DEV void multi_gk(const CgMultiArgs& p, const int32_t* toc, const int32_t* cstart, const double* coef_s, const cplx* gs, cplx* gk, int ib,
                       int ncell) {
    const int C = p.C, nc = p.n_comp;
    for (int it = threadIdx.x; it < ib * C * ncell; it += blockDim.x) {   // (il, c, cell)
        const int cell = it % ncell, ic = it / ncell;
        const cplx* g = gs + (size_t)ic * nc;
        cplx v = czero();
        for (int t = cstart[cell]; t < cstart[cell + 1]; ++t) cfmar(v, g[toc[t]], coef_s[t]);
        gk[it] = v;
    }
}
// carve the adjoint's tables out of shared memory (coef, component per term, cell starts, output map)
struct MultiBwdTabs {
    double* coef;
    int32_t *toc, *cstart, *cinfo;
};
LGAE_DEV MultiBwdTabs multi_load_bwd_tabs(const CgMultiArgs& p, double* mem, int ncell) {
    MultiBwdTabs T;
    const int nt = p.n_terms, nc = p.n_comp;
    T.coef = mem;
    T.toc = reinterpret_cast<int32_t*>(mem + nt);
    T.cstart = T.toc + nt;
    T.cinfo = T.cstart + ncell + 1;
    for (int t = threadIdx.x; t < nt; t += blockDim.x) T.coef[t] = p.coef_b[t];
    for (int t = threadIdx.x; t < nt + ncell + 1 + 3 * nc; t += blockDim.x) T.toc[t] = p.tab_b[t];
    return T;
}
static size_t multi_bwd_tab_bytes(int nt, int nc, int ncell) { return (size_t)nt * sizeof(double) + ((size_t)nt + ncell + 1 + 3 * nc) * sizeof(int32_t) + 16; }

#ifndef LGAE_AGG_FWD_MINB
#define LGAE_AGG_FWD_MINB 1
#endif
#ifndef LGAE_AGG_FWD_IB
#define LGAE_AGG_FWD_IB 3
#endif
#ifndef LGAE_AGG_EDGE_MINB
#define LGAE_AGG_EDGE_MINB 1
#endif
#ifndef LGAE_AGG_EDGE_IB
#define LGAE_AGG_EDGE_IB 4
#endif
template <int D2T>
__global__ void __launch_bounds__(CG_THREADS, LGAE_AGG_FWD_MINB) cg_agg_multi_fwd_kernel(const CgMultiArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, NJ = p.NJ, IB = p.IB, nc = p.n_comp, nt = p.n_terms;
    const int D1T = p.node_off[p.n_node];
    cplx* z2s = reinterpret_cast<cplx*>(smem);                 // IB * NJ * C * D2T
    cplx* ks = z2s + (size_t)IB * NJ * C * D2T;                  // IB * C * D1T * D2T
    double* coef_s = reinterpret_cast<double*>(ks + (size_t)IB * C * D1T * D2T);
    int32_t* ta = reinterpret_cast<int32_t*>(coef_s + nt);       // a_all
    int32_t* td = ta + nt;                                       // d_all
    int32_t* start = td + nt;                                    // n_comp + 1
    int32_t* cinfo = start + nc + 1;                             // n_comp * 3
    for (int t = tid; t < nt; t += blockDim.x) {
        coef_s[t] = p.coef[t];
        ta[t] = p.tab[3 * t + 1];
        td[t] = p.tab[3 * t + 2];
    }
    for (int t = tid; t < nc + 1 + 3 * nc; t += blockDim.x) start[t] = p.tab[3 * nt + t];
    pdl_wait();
    const int b = blockIdx.x, i0 = blockIdx.y * IB, ib = min(IB, p.N - i0);
    for (int q = 0; q < p.n_edge; ++q) {
        const int dq = p.edge_d[q], off = p.edge_off[q];
        const int64_t plane = (int64_t)p.B * p.N * NJ * C * dq;
        const double* src = p.edge[q] + ((int64_t)b * p.N + i0) * NJ * C * dq;
        for (int t = tid; t < ib * NJ * C * dq; t += blockDim.x)
            z2s[(size_t)(t / dq) * D2T + off + t % dq] = cmake(src[t], src[plane + t]);
    }
    __syncthreads();
    for (int it = tid; it < ib * C * D1T; it += CG_THREADS) {   // (il, c, a_all), a_all fastest
        const int a_all = it % D1T, c = (it / D1T) % C, il = it / (D1T * C);
        int pn = 0;
        while (pn + 1 < p.n_node && a_all >= p.node_off[pn + 1]) ++pn;
        const int dp = p.node_d[pn];
        const int64_t plane = (int64_t)p.B * NJ * C * dp, step = (int64_t)C * dp;
        const double* x = p.node[pn] + ((int64_t)b * NJ * C + c) * dp + (a_all - p.node_off[pn]);
        const cplx* y = z2s + ((size_t)il * NJ * C + c) * D2T;
        cplx acc[D2T];
#pragma unroll
        for (int d = 0; d < D2T; ++d) acc[d] = czero();
#pragma unroll 2
        for (int j = 0; j < NJ; ++j) {
            const cplx xv = cmake(x[j * step], x[plane + j * step]);
#pragma unroll
            for (int d = 0; d < D2T; ++d) cfma(acc[d], xv, y[(size_t)j * C * D2T + d]);
        }
#pragma unroll
        for (int d = 0; d < D2T; ++d) ks[(size_t)it * D2T + d] = acc[d];
    }
    __syncthreads();
    for (int it = tid; it < ib * C * nc; it += CG_THREADS) {   // (il, oc, c), c fastest
        const int c = it % C, oc = (it / C) % nc, il = it / (C * nc);
        const cplx* k = ks + ((size_t)il * C + c) * D1T * D2T;
        cplx acc = czero();
        for (int t = start[oc]; t < start[oc + 1]; ++t) cfmar(acc, k[ta[t] * D2T + td[t]], coef_s[t]);
        const int o = cinfo[3 * oc], m = cinfo[3 * oc + 1], coff = cinfo[3 * oc + 2];
        const int64_t rowsz = (int64_t)p.out_ctot[o] * p.out_d[o];
        const int64_t idx = ((int64_t)b * p.N + i0 + il) * rowsz + (int64_t)(coff + c) * p.out_d[o] + m;
        p.out[o][idx] = acc.x;
        p.out[o][(int64_t)p.B * p.N * rowsz + idx] = acc.y;
    }
}

// Adjoint of the one-launch aggregate, edge operand: dL/dz2_q[i, j][d] = sum_{a_all} conj(z1_j[a_all]) gK_i[a_all][d_all] for every
// edge part q at once; grid (B, ceil(N / IB)), fully parallel, node parts read from global memory.
template <int D2T>
__global__ void __launch_bounds__(CG_THREADS, LGAE_AGG_EDGE_MINB) cg_agg_multi_bwd_edge_kernel(const CgMultiArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, NJ = p.NJ, IB = p.IB, nc = p.n_comp;
    const int D1T = p.node_off[p.n_node], ncell = D1T * D2T;
    cplx* gs = reinterpret_cast<cplx*>(smem);             // IB * C * n_comp
    cplx* gk = gs + (size_t)IB * C * nc;                    // IB * C * D1T * D2T
    const MultiBwdTabs T = multi_load_bwd_tabs(p, reinterpret_cast<double*>(gk + (size_t)IB * C * ncell), ncell);
    pdl_wait();
    __syncthreads();
    const int b = blockIdx.x, i0 = blockIdx.y * IB, ib = min(IB, p.N - i0);
    multi_stage_g(p, T.cinfo, gs, b, i0, ib);
    __syncthreads();
    multi_gk(p, T.toc, T.cstart, T.coef, gs, gk, ib, ncell);
    __syncthreads();
    for (int it = tid; it < ib * NJ * C; it += CG_THREADS) {   // (il, j, c), c fastest
        const int c = it % C, j = (it / C) % NJ, il = it / (C * NJ);
        cplx acc[D2T];
#pragma unroll
        for (int d = 0; d < D2T; ++d) acc[d] = czero();
        for (int pn = 0; pn < p.n_node; ++pn) {
            const int dp = p.node_d[pn];
            const int64_t plane = (int64_t)p.B * NJ * C * dp;
            const double* x = p.node[pn] + (((int64_t)b * NJ + j) * C + c) * dp;
            const cplx* kk = gk + (((size_t)il * C + c) * D1T + p.node_off[pn]) * D2T;
            for (int a_ = 0; a_ < dp; ++a_) {
                const cplx xv = cmake(x[a_], x[plane + a_]);
#pragma unroll
                for (int d = 0; d < D2T; ++d) cfmac(acc[d], xv, kk[a_ * D2T + d]);
            }
        }
        for (int q = 0; q < p.n_edge; ++q) {
            if (!p.gedge[q]) continue;
            const int dq = p.edge_d[q];
            const int64_t plane = (int64_t)p.B * p.N * NJ * C * dq;
            double* g2 = p.gedge[q] + ((((int64_t)b * p.N + i0 + il) * NJ + j) * C + c) * dq;
#pragma unroll
            for (int d = 0; d < D2T; ++d) {
                const int dl = d - p.edge_off[q];
                if (dl >= 0 && dl < dq) {
                    g2[dl] = acc[d].x;
                    g2[plane + dl] = acc[d].y;
                }
            }
        }
    }
}
// Adjoint, node operands: dL/dz1_p[j][a] = sum_i sum_{d_all} conj(z2_ij[d_all]) gK_i[a_all][d_all]; one CTA per jet walks the particles
// i in blocks of IB, a thread owns one (j, channel) and all D1T accumulators in registers (fixed summation order).
#ifndef LGAE_AGG_NODE_MINB
#define LGAE_AGG_NODE_MINB 2   // 128 registers, no spills: 2 CTAs per SM (1.45 -> 1.13 ms per launch at cfg-4)
#endif
template <int D1T, int D2T>
__global__ void __launch_bounds__(CG_THREADS, LGAE_AGG_NODE_MINB) cg_agg_multi_bwd_node_kernel(const CgMultiArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, NJ = p.NJ, IB = p.IB, nc = p.n_comp;
    constexpr int ncell = D1T * D2T;
    cplx* z2s = reinterpret_cast<cplx*>(smem);              // IB * NJ * C * D2T
    cplx* gs = z2s + (size_t)IB * NJ * C * D2T;               // IB * C * n_comp
    cplx* gk = gs + (size_t)IB * C * nc;                      // IB * C * D1T * D2T
    const MultiBwdTabs T = multi_load_bwd_tabs(p, reinterpret_cast<double*>(gk + (size_t)IB * C * ncell), ncell);
    pdl_wait();
    const int b = blockIdx.x, per_i = NJ * C;
    cplx acc[D1T];
#pragma unroll
    for (int a_ = 0; a_ < D1T; ++a_) acc[a_] = czero();
    for (int i0 = 0; i0 < p.N; i0 += IB) {
        const int ib = min(IB, p.N - i0);
        __syncthreads();
        for (int q = 0; q < p.n_edge; ++q) {
            const int dq = p.edge_d[q], off = p.edge_off[q];
            const int64_t plane = (int64_t)p.B * p.N * NJ * C * dq;
            const double* src = p.edge[q] + ((int64_t)b * p.N + i0) * NJ * C * dq;
            for (int t = tid; t < ib * per_i * dq; t += blockDim.x) z2s[(size_t)(t / dq) * D2T + off + t % dq] = cmake(src[t], src[plane + t]);
        }
        multi_stage_g(p, T.cinfo, gs, b, i0, ib);
        __syncthreads();
        multi_gk(p, T.toc, T.cstart, T.coef, gs, gk, ib, ncell);
        __syncthreads();
        if (tid < per_i) {
            const int c = tid % C;
            for (int il = 0; il < ib; ++il) {
                const cplx* z = z2s + ((size_t)il * per_i + tid) * D2T;
                const cplx* kk = gk + ((size_t)il * C + c) * ncell;
                cplx zv[D2T];
#pragma unroll
                for (int d = 0; d < D2T; ++d) zv[d] = z[d];
#pragma unroll
                for (int a_ = 0; a_ < D1T; ++a_)
#pragma unroll
                    for (int d = 0; d < D2T; ++d) cfmac(acc[a_], zv[d], kk[a_ * D2T + d]);
            }
        }
    }
    if (tid < per_i) {
        int pn = 0;
#pragma unroll
        for (int a_ = 0; a_ < D1T; ++a_) {
            while (pn + 1 < p.n_node && a_ >= p.node_off[pn + 1]) ++pn;
            if (p.gnode[pn]) {
                const int dp = p.node_d[pn];
                const int64_t idx = ((int64_t)b * per_i + tid) * dp + (a_ - p.node_off[pn]);
                p.gnode[pn][idx] = acc[a_].x;
                p.gnode[pn][(int64_t)p.B * per_i * dp + idx] = acc[a_].y;
            }
        }
    }
}

// Adjoint.  grid (B, neighbour tiles): the CTA owns the gradient of its z1 tile (registers) and writes the gradient of
// the z2 entries (i, tile) for every i.  Every sum has a fixed order.
__global__ void __launch_bounds__(CG_THREADS) cg_agg_bwd_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, d1 = p.d1, d2 = p.d2, NJ = p.NJ, JT = p.JT, nc = p.n_comp;
    const int S1 = cg_row_stride(C * d1), S2 = cg_row_stride(C * d2);
    cplx* z1s = reinterpret_cast<cplx*>(smem);
    cplx* z2s = z1s + (size_t)JT * S1;
    cplx* gs = z2s + (size_t)JT * S2;   // C * n_comp
    double* rest = reinterpret_cast<double*>(gs + (size_t)C * nc);
    TermsSm Ta, Td;
    rest += terms_load(p, 1, rest, Ta);
    terms_load(p, 2, rest, Td);
    pdl_wait();
    const int b = blockIdx.x, j0 = blockIdx.y * JT, jt = min(JT, NJ - j0);
    stage_rows(z1s, p.z1 + ((int64_t)b * NJ + j0) * C * d1, p.plane1, jt, C * d1);
    const int items1 = p.g1 ? jt * C * d1 : 0, items2 = p.g2 ? jt * C * d2 : 0;
    cplx acc[CG_ITEMS];
#pragma unroll
    for (int k = 0; k < CG_ITEMS; ++k) acc[k] = czero();
    const int ng = C * nc;
    for (int i = 0; i < p.N; ++i) {
        __syncthreads();
        stage_rows(z2s, p.z2 + (((int64_t)b * p.N + i) * NJ + j0) * C * d2, p.plane2, jt, C * d2);
        for (int t = tid; t < ng; t += blockDim.x) {
            const int c = t / nc, oc = t % nc;
            const CgOut& o = p.out[out_of_comp(p, oc)];
            const int64_t idx = (((int64_t)b * p.N + i) * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
            gs[t] = cmake(o.ptr[idx], o.ptr[o.plane + idx]);
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < CG_ITEMS; ++k) {
            const int it = tid + k * CG_THREADS;
            if (it >= items1) break;
            const int a_ = it % d1, c = (it / d1) % C, j = it / (d1 * C);
            cplx s = czero();
            for (int t = Ta.start[a_]; t < Ta.start[a_ + 1]; ++t) {
                cplx v = czero();
                cfmac(v, z2s[j * S2 + c * d2 + Ta.d[t]], gs[c * nc + Ta.comp[t]]);
                cfmar(s, v, Ta.coef[t]);
            }
            acc[k] = cadd(acc[k], s);
        }
        for (int it = tid; it < items2; it += blockDim.x) {
            const int d_ = it % d2, c = (it / d2) % C, j = it / (d2 * C);
            cplx s = czero();
            for (int t = Td.start[d_]; t < Td.start[d_ + 1]; ++t) {
                cplx v = czero();
                cfmac(v, z1s[j * S1 + c * d1 + Td.a[t]], gs[c * nc + Td.comp[t]]);
                cfmar(s, v, Td.coef[t]);
            }
            const int64_t idx = (((int64_t)b * p.N + i) * NJ + j0) * C * d2 + it;
            if (p.acc2) {
                p.g2[idx] += s.x;
                p.g2[p.plane2 + idx] += s.y;
            } else {
                p.g2[idx] = s.x;
                p.g2[p.plane2 + idx] = s.y;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < CG_ITEMS; ++k) {
        const int it = tid + k * CG_THREADS;
        if (it >= items1) break;
        const int64_t idx = ((int64_t)b * NJ + j0) * C * d1 + it;
        if (p.acc1) {
            p.g1[idx] += acc[k].x;
            p.g1[p.plane1 + idx] += acc[k].y;
        } else {
            p.g1[idx] = acc[k].x;
            p.g1[p.plane1 + idx] = acc[k].y;
        }
    }
}

// Gradient of the edge operand alone: dL/dz2[i, j] = sum_terms coef conj(z1_j) g_i needs no neighbour sum and no z2, so it is
// a fully parallel kernel over (jet, block of IB particles i): node slab + IB rows of output gradients in shared memory,
// one thread per (i, j, c, d), stores contiguous in the edge tensor's layout.  p.JT holds IB.
__global__ void __launch_bounds__(CG_THREADS) cg_agg_bwd_edge_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, d1 = p.d1, d2 = p.d2, NJ = p.NJ, IB = p.JT, nc = p.n_comp;
    cplx* z1s = reinterpret_cast<cplx*>(smem);
    cplx* gs = z1s + (size_t)NJ * C * d1;   // IB * C * n_comp
    TermsSm Td;
    terms_load(p, 2, reinterpret_cast<double*>(gs + (size_t)IB * C * nc), Td);
    pdl_wait();
    const int b = blockIdx.x, i0 = blockIdx.y * IB, ib = min(IB, p.N - i0);
    stage_planar(z1s, p.z1 + (int64_t)b * NJ * C * d1, p.plane1, NJ * C * d1);
    for (int t = tid; t < ib * C * nc; t += blockDim.x) {
        const int il = t / (C * nc), w = t % (C * nc), c = w / nc, oc = w % nc;
        const CgOut& o = p.out[out_of_comp(p, oc)];
        const int64_t idx = (((int64_t)b * p.N + i0 + il) * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
        gs[t] = cmake(o.ptr[idx], o.ptr[o.plane + idx]);
    }
    __syncthreads();
    const int per_i = NJ * C * d2;
    double* g2 = p.g2 + ((int64_t)b * p.N + i0) * per_i;
    for (int it = tid; it < ib * per_i; it += CG_THREADS) {
        const int il = it / per_i, w = it % per_i, d_ = w % d2, c = (w / d2) % C, j = w / (d2 * C);
        const cplx* gi = gs + ((size_t)il * C + c) * nc;
        const cplx* zj = z1s + ((size_t)j * C + c) * d1;
        cplx sum = czero();
        for (int t = Td.start[d_]; t < Td.start[d_ + 1]; ++t) {
            cplx v = czero();
            cfmac(v, zj[Td.a[t]], gi[Td.comp[t]]);
            cfmar(sum, v, Td.coef[t]);
        }
        if (p.acc2) {
            g2[it] += sum.x;
            g2[p.plane2 + it] += sum.y;
        } else {
            g2[it] = sum.x;
            g2[p.plane2 + it] = sum.y;
        }
    }
}

// Kronecker form of the edge gradient: gK[a][d] = sum_terms coef g[m] (the transposed CG matrix applied to the output
// gradient) per (i, channel), then dL/dz2[i, j][d] = sum_a conj(z1_j[a]) gK[a][d] with the d axis in registers.
template <int D2>
__global__ void __launch_bounds__(CG_THREADS) cg_agg_bwd_edge_kron_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, d1 = p.d1, NJ = p.NJ, IB = p.JT, nc = p.n_comp;
    cplx* z1s = reinterpret_cast<cplx*>(smem);
    cplx* gs = z1s + (size_t)NJ * C * d1;        // IB * C * n_comp
    cplx* gk = gs + (size_t)IB * C * nc;         // IB * C * d1 * D2
    TermsSm Ta;
    terms_load(p, 1, reinterpret_cast<double*>(gk + (size_t)IB * C * d1 * D2), Ta);
    pdl_wait();
    const int b = blockIdx.x, i0 = blockIdx.y * IB, ib = min(IB, p.N - i0);
    stage_planar(z1s, p.z1 + (int64_t)b * NJ * C * d1, p.plane1, NJ * C * d1);
    for (int t = tid; t < ib * C * nc; t += blockDim.x) {
        const int il = t / (C * nc), w = t % (C * nc), c = w / nc, oc = w % nc;
        const CgOut& o = p.out[out_of_comp(p, oc)];
        const int64_t idx = (((int64_t)b * p.N + i0 + il) * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
        gs[t] = cmake(o.ptr[idx], o.ptr[o.plane + idx]);
    }
    __syncthreads();
    for (int it = tid; it < ib * C * d1 * D2; it += CG_THREADS) {   // (il, c, a, d)
        const int d_ = it % D2, a_ = (it / D2) % d1, ic = it / (D2 * d1);
        const cplx* g = gs + (size_t)ic * nc;
        cplx acc = czero();
        for (int t = Ta.start[a_]; t < Ta.start[a_ + 1]; ++t)
            if (Ta.d[t] == d_) cfmar(acc, g[Ta.comp[t]], Ta.coef[t]);
        gk[it] = acc;
    }
    __syncthreads();
    const int per_i = NJ * C;
    double* g2 = p.g2 + ((int64_t)b * p.N + i0) * per_i * D2;
    for (int it = tid; it < ib * per_i; it += CG_THREADS) {   // (il, j, c), c fastest
        const int il = it / per_i, w = it % per_i, c = w % C, j = w / C;
        const cplx* zj = z1s + ((size_t)j * C + c) * d1;
        const cplx* k = gk + ((size_t)il * C + c) * d1 * D2;
        cplx acc[D2];
#pragma unroll
        for (int d = 0; d < D2; ++d) acc[d] = czero();
        for (int a_ = 0; a_ < d1; ++a_) {
            const cplx xv = zj[a_];
#pragma unroll
            for (int d = 0; d < D2; ++d) cfmac(acc[d], xv, k[a_ * D2 + d]);
        }
#pragma unroll
        for (int d = 0; d < D2; ++d) {
            const int64_t o = (int64_t)it * D2 + d;
            if (p.acc2) {
                g2[o] += acc[d].x;
                g2[p.plane2 + o] += acc[d].y;
            } else {
                g2[o] = acc[d].x;
                g2[p.plane2 + o] = acc[d].y;
            }
        }
    }
}

// Kronecker form of the node gradient: dL/dz1[j][a] = sum_i sum_d conj(z2_ij[d]) gK_i[a][d].  One CTA per jet walks the
// particles i in blocks of IB (p.JT): IB rows of the edge tensor and the IB gK matrices in shared memory, a thread owns one
// (neighbour j, channel) and keeps its D1 accumulators in registers over the whole walk (fixed summation order).
template <int D1, int D2>
__global__ void __launch_bounds__(CG_THREADS) cg_agg_bwd_node_kron_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, C = p.C, NJ = p.NJ, IB = p.JT, nc = p.n_comp;
    cplx* z2s = reinterpret_cast<cplx*>(smem);          // IB * NJ * C * D2
    cplx* gs = z2s + (size_t)IB * NJ * C * D2;            // IB * C * n_comp
    cplx* gk = gs + (size_t)IB * C * nc;                  // IB * C * D1 * D2
    TermsSm Ta;
    terms_load(p, 1, reinterpret_cast<double*>(gk + (size_t)IB * C * D1 * D2), Ta);
    pdl_wait();
    const int b = blockIdx.x, per_i = NJ * C;
    constexpr int PASS = 2;   // (j, c) items per thread
    cplx acc[PASS][D1];
#pragma unroll
    for (int k = 0; k < PASS; ++k)
#pragma unroll
        for (int a_ = 0; a_ < D1; ++a_) acc[k][a_] = czero();
    for (int i0 = 0; i0 < p.N; i0 += IB) {
        const int ib = min(IB, p.N - i0);
        __syncthreads();
        stage_planar(z2s, p.z2 + ((int64_t)b * p.N + i0) * per_i * D2, p.plane2, ib * per_i * D2);
        for (int t = tid; t < ib * C * nc; t += blockDim.x) {
            const int il = t / (C * nc), w = t % (C * nc), c = w / nc, oc = w % nc;
            const CgOut& o = p.out[out_of_comp(p, oc)];
            const int64_t idx = (((int64_t)b * p.N + i0 + il) * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
            gs[t] = cmake(o.ptr[idx], o.ptr[o.plane + idx]);
        }
        __syncthreads();
        for (int it = tid; it < ib * C * D1 * D2; it += CG_THREADS) {   // gK (il, c, a, d)
            const int d_ = it % D2, a_ = (it / D2) % D1, ic = it / (D2 * D1);
            const cplx* g = gs + (size_t)ic * nc;
            cplx v = czero();
            for (int t = Ta.start[a_]; t < Ta.start[a_ + 1]; ++t)
                if (Ta.d[t] == d_) cfmar(v, g[Ta.comp[t]], Ta.coef[t]);
            gk[it] = v;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < PASS; ++k) {
            const int it = tid + k * CG_THREADS;
            if (it < per_i) {
                const int c = it % C;
                for (int il = 0; il < ib; ++il) {
                    const cplx* z = z2s + ((size_t)il * per_i + it) * D2;
                    const cplx* kk = gk + ((size_t)il * C + c) * D1 * D2;
                    cplx zv[D2];
#pragma unroll
                    for (int d = 0; d < D2; ++d) zv[d] = z[d];
#pragma unroll
                    for (int a_ = 0; a_ < D1; ++a_)
#pragma unroll
                        for (int d = 0; d < D2; ++d) cfmac(acc[k][a_], zv[d], kk[a_ * D2 + d]);
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < PASS; ++k) {
        const int it = tid + k * CG_THREADS;
        if (it < per_i) {
            double* g1 = p.g1 + ((int64_t)b * per_i + it) * D1;
#pragma unroll
            for (int a_ = 0; a_ < D1; ++a_) {
                if (p.acc1) {
                    g1[a_] += acc[k][a_].x;
                    g1[p.plane1 + a_] += acc[k][a_].y;
                } else {
                    g1[a_] = acc[k][a_].x;
                    g1[p.plane1 + a_] = acc[k][a_].y;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// point-wise product: out_r = H (z1_r (x) z2_r), rows r = 0..B-1 (p.B = number of rows, p.N = 1, p.NJ = 0)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CG_THREADS) cg_pt_fwd_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    TermsSm T;
    terms_load(p, 0, smem, T);
    pdl_wait();
    __syncthreads();
    const int C = p.C, d1 = p.d1, d2 = p.d2;
    const int64_t per_row = (int64_t)C * p.n_comp, total = (int64_t)p.B * per_row;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < total; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = it / per_row;
        const int w = (int)(it % per_row), c = w % C, oc = w / C;
        const double* x = p.z1 + (r * C + c) * d1;
        const double* y = p.z2 + (r * C + c) * d2;
        cplx acc = czero();
        for (int t = T.start[oc]; t < T.start[oc + 1]; ++t) {
            const int a_ = T.a[t], d_ = T.d[t];
            cfmar(acc, cmul(cmake(x[a_], x[p.plane1 + a_]), cmake(y[d_], y[p.plane2 + d_])), T.coef[t]);
        }
        const CgOut& o = p.out[out_of_comp(p, oc)];
        const int64_t idx = (r * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
        o.ptr[idx] = acc.x;
        o.ptr[o.plane + idx] = acc.y;
    }
}

__global__ void __launch_bounds__(CG_THREADS) cg_pt_bwd_kernel(const CgArgs p) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    TermsSm Ta, Td;
    double* rest = smem;
    rest += terms_load(p, 1, rest, Ta);
    terms_load(p, 2, rest, Td);
    pdl_wait();
    __syncthreads();
    const int C = p.C, d1 = p.d1, d2 = p.d2;
    const int64_t n1 = p.g1 ? (int64_t)p.B * C * d1 : 0, n2 = p.g2 ? (int64_t)p.B * C * d2 : 0;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < n1 + n2; it += (int64_t)gridDim.x * blockDim.x) {
        const bool first = it < n1;
        const int64_t e = first ? it : it - n1;
        const int dd = first ? d1 : d2, od = first ? d2 : d1;
        const int q = (int)(e % dd), c = (int)((e / dd) % C);
        const int64_t r = e / ((int64_t)dd * C);
        const TermsSm& T = first ? Ta : Td;
        const double* other = (first ? p.z2 : p.z1) + (r * C + c) * od;
        const int64_t oplane = first ? p.plane2 : p.plane1;
        cplx s = czero();
        for (int t = T.start[q]; t < T.start[q + 1]; ++t) {
            const int oc = T.comp[t], k = first ? T.d[t] : T.a[t];
            const CgOut& o = p.out[out_of_comp(p, oc)];
            const int64_t idx = (r * o.ctot + o.coff + c) * o.d + (oc - o.comp0);
            cplx v = czero();
            cfmac(v, cmake(other[k], other[oplane + k]), cmake(o.ptr[idx], o.ptr[o.plane + idx]));
            cfmar(s, v, T.coef[t]);
        }
        double* g = first ? p.g1 : p.g2;
        const int64_t gplane = first ? p.plane1 : p.plane2;
        if (first ? p.acc1 : p.acc2) {
            g[e] += s.x;
            g[gplane + e] += s.y;
        } else {
            g[e] = s.x;
            g[gplane + e] = s.y;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// channel mixing  out[r, co, m] = sum_ci W[co, ci] x[r, ci, m]      x (2,R,Cin,d), W (2,Cout,Cin), out (2,R,Cout,d)
// ------------------------------------------------------------------------------------------------------------
struct MixArgs {
    const double *x, *w, *g;
    double *out, *gx, *gw_part;
    int64_t R;
    int32_t cin, cout, d, rows_per_cta;
    int32_t co0;   // forward: first output channel of this launch (blocks of CO channels); weight gradient: rows per stage
    int32_t nsub;  // weight gradient: row lanes
};
constexpr int MIX_THREADS = 256;

LGAE_DEV void mix_stage_w(const MixArgs& a, cplx* ws) {
    const int n = a.cout * a.cin;
    for (int t = threadIdx.x; t < n; t += blockDim.x) ws[t] = cmake(a.w[t], a.w[n + t]);
}
// thread = one (row, component m): it reads x[r, :, m] once and keeps the accumulators of all CO output channels in registers
// (2 global loads + CO broadcast shared-memory loads per 4 CO multiply-adds)
template <int CO>
__global__ void __launch_bounds__(MIX_THREADS) mix_fwd_kernel(const MixArgs a) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    cplx* ws = reinterpret_cast<cplx*>(smem);   // [ci][CO], zero beyond cout
    {
        const int n = a.cout * a.cin;
        for (int t = threadIdx.x; t < a.cin * CO; t += blockDim.x) {
            const int ci = t / CO, co = a.co0 + t % CO;
            ws[t] = co < a.cout ? cmake(a.w[co * a.cin + ci], a.w[n + co * a.cin + ci]) : czero();
        }
    }
    pdl_wait();
    __syncthreads();
    const int64_t items = a.R * a.d, xplane = a.R * a.cin * a.d, oplane = a.R * a.cout * a.d;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = it / a.d;
        const int m = (int)(it - r * a.d);
        const double* x = a.x + r * a.cin * a.d + m;
        cplx acc[CO];
#pragma unroll
        for (int co = 0; co < CO; ++co) acc[co] = czero();
#pragma unroll 2
        for (int ci = 0; ci < a.cin; ++ci) {
            const cplx xv = cmake(x[(int64_t)ci * a.d], x[xplane + (int64_t)ci * a.d]);
#pragma unroll
            for (int co = 0; co < CO; ++co) cfma(acc[co], ws[ci * CO + co], xv);
        }
        double* o = a.out + (r * a.cout + a.co0) * a.d + m;
#pragma unroll
        for (int co = 0; co < CO; ++co)
            if (a.co0 + co < a.cout) {
                o[(int64_t)co * a.d] = acc[co].x;
                o[oplane + (int64_t)co * a.d] = acc[co].y;
            }
    }
}
// gx[r, ci, m] = sum_co conj(W[co, ci]) g[r, co, m]
__global__ void __launch_bounds__(MIX_THREADS) mix_bwd_x_kernel(const MixArgs a) {
    pdl_launch();
    extern __shared__ __align__(16) double smem[];
    cplx* ws = reinterpret_cast<cplx*>(smem);
    mix_stage_w(a, ws);
    pdl_wait();
    __syncthreads();
    const int64_t per_row = (int64_t)a.cin * a.d, total = a.R * per_row, gplane = a.R * a.cout * a.d;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < total; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = it / per_row;
        const int w = (int)(it % per_row), m = w % a.d, ci = w / a.d;
        const double* g = a.g + r * a.cout * a.d + m;
        cplx acc = czero();
        for (int co = 0; co < a.cout; ++co) cfmac(acc, ws[co * a.cin + ci], cmake(g[(int64_t)co * a.d], g[gplane + (int64_t)co * a.d]));
        a.gx[it] = acc.x;
        a.gx[total + it] = acc.y;
    }
}
// gW[co, ci] = sum_{r, m} conj(x[r, ci, m]) g[r, co, m]: one partial (2, cout*cin) per CTA over its rows, fixed order.
// Rows are staged `rows_per_stage` at a time; thread = (input channel ci, row lane): it reads its x entries once and keeps the
// accumulators of CO output channels in registers (the g entries are warp-wide broadcasts); the row lanes are then added
// in order through shared memory.
template <int CO>
__global__ void __launch_bounds__(MIX_THREADS) mix_bwd_w_kernel(const MixArgs a) {
    pdl_launch();
    pdl_wait();
    extern __shared__ __align__(16) double smem[];
    const int cin = a.cin, cout = a.cout, d = a.d, RB = a.co0;   // co0 carries the rows per stage here
    cplx* xs = reinterpret_cast<cplx*>(smem);            // RB * cin * d
    cplx* gs = xs + (size_t)RB * cin * d;                // RB * cout * d
    cplx* red = reinterpret_cast<cplx*>(smem);           // nsub * cb * CO, aliases the staging area after the row loop
    const int n = cout * cin;
    const int64_t xplane = a.R * cin * d, gplane = a.R * cout * d;
    const int64_t r0 = (int64_t)blockIdx.x * a.rows_per_cta, r1 = min(a.R, r0 + a.rows_per_cta);
    double* part = a.gw_part + (int64_t)blockIdx.x * 2 * n;
    const int cb = min(cin, MIX_THREADS);                // input channels per pass
    const int nsub = a.nsub;                             // row lanes (<= MIX_THREADS / cb)
    const int cl = threadIdx.x % cb, sub = threadIdx.x / cb;
    for (int ci0 = 0; ci0 < cin; ci0 += cb)
        for (int co0 = 0; co0 < cout; co0 += CO) {
            const int ci = ci0 + cl;
            const bool active = sub < nsub && ci < cin;
            cplx acc[CO];
#pragma unroll
            for (int co = 0; co < CO; ++co) acc[co] = czero();
            for (int64_t rb = r0; rb < r1; rb += RB) {
                const int nr = (int)min((int64_t)RB, r1 - rb);
                __syncthreads();
                stage_planar(xs, a.x + rb * cin * d, xplane, nr * cin * d);
                stage_planar(gs, a.g + rb * cout * d, gplane, nr * cout * d);
                __syncthreads();
                if (active)
                    for (int rr = sub; rr < nr; rr += nsub) {
                        const cplx* xr = xs + ((size_t)rr * cin + ci) * d;
                        const cplx* gr = gs + ((size_t)rr * cout + co0) * d;
                        for (int m = 0; m < d; ++m) {
                            const cplx xv = xr[m];
#pragma unroll
                            for (int co = 0; co < CO; ++co)
                                if (co0 + co < cout) cfmac(acc[co], xv, gr[co * d + m]);
                        }
                    }
            }
            __syncthreads();
            if (active) {
#pragma unroll
                for (int co = 0; co < CO; ++co) red[((size_t)sub * cb + cl) * CO + co] = acc[co];
            }
            __syncthreads();
            for (int t = threadIdx.x; t < cb * CO; t += blockDim.x) {
                const int c2 = t / CO, co = t % CO;
                if (ci0 + c2 >= cin || co0 + co >= cout) continue;
                cplx v = red[t];
                for (int sl = 1; sl < nsub; ++sl) v = cadd(v, red[(size_t)sl * cb * CO + t]);
                const int it = (co0 + co) * cin + ci0 + c2;
                part[it] = v.x;
                part[n + it] = v.y;
            }
        }
}
// out[t] = sum_rows part[row][t]: 32 columns x 8 row lanes per CTA, every lane walks its rows in order, then the lanes are
// added in order (fixed summation order: deterministic)
constexpr int COLSUM_Y = 8;
__global__ void __launch_bounds__(32 * COLSUM_Y) colsum_kernel(const double* part, int rows, int64_t n, double* out) {
    pdl_launch();
    pdl_wait();
    __shared__ double red[COLSUM_Y][33];
    const int64_t t = (int64_t)blockIdx.x * 32 + threadIdx.x;
    double s = 0.0;
    if (t < n)
        for (int r = threadIdx.y; r < rows; r += COLSUM_Y) s += part[(int64_t)r * n + t];
    red[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && t < n) {
        double acc = red[0][threadIdx.x];
#pragma unroll
        for (int y = 1; y < COLSUM_Y; ++y) acc += red[y][threadIdx.x];
        out[t] = acc;
    }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
static int grid_for(int64_t work, int threads) {
    const int64_t need = (work + threads - 1) / threads, cap = (int64_t)sm_count() * 8;
    return (int)std::max<int64_t>(1, std::min(need, cap));
}
static int cg_fill(const LgaeCgPairDesc* d, const int32_t* tab, const double* coef, CgArgs& p, void* const* ptrs, int64_t rows) {
    if (!d || !tab || !coef || !ptrs) return LGAE_E_BADARG;
    if (d->d1 < 1 || d->d2 < 1 || d->channels < 1 || d->n_out < 1 || d->n_out > LGAE_CG_MAX_OUT || d->n_terms < 1 || d->n_comp < 1)
        return LGAE_E_BADARG;
    p.C = d->channels; p.d1 = d->d1; p.d2 = d->d2; p.n_comp = d->n_comp; p.n_terms = d->n_terms; p.n_out = d->n_out;
    p.tab = tab; p.coef = coef; p.JS = 1;
    int comp = 0;
    for (int o = 0; o < d->n_out; ++o) {
        if (!ptrs[o] || d->out_comp0[o] != comp || d->out_d[o] < 1 || d->out_coffset[o] < 0 || d->out_coffset[o] + d->channels > d->out_ctotal[o])
            return LGAE_E_BADARG;
        p.out[o].ptr = (double*)ptrs[o];
        p.out[o].d = d->out_d[o]; p.out[o].comp0 = comp; p.out[o].ctot = d->out_ctotal[o]; p.out[o].coff = d->out_coffset[o];
        p.out[o].plane = rows * d->out_ctotal[o] * d->out_d[o];
        comp += d->out_d[o];
    }
    if (comp != d->n_comp) return LGAE_E_BADARG;
    return LGAE_OK;
}
// neighbour tile: as many particles as fit next to the fixed part in ~160 KB, and (adjoint) CG_ITEMS*CG_THREADS z1 items
static int cg_tile(const CgArgs& p, size_t fixed_bytes, bool bwd) {
    const size_t per_j = (size_t)(cg_row_stride(p.C * p.d1) + cg_row_stride(p.C * p.d2)) * sizeof(cplx);
    const size_t budget = 160 * 1024;
    if (fixed_bytes + per_j > budget) return 0;
    int64_t jt = (int64_t)((budget - fixed_bytes) / per_j);
    if (bwd) jt = std::min<int64_t>(jt, (CG_ITEMS * CG_THREADS) / (p.C * p.d1));
    return (int)std::min<int64_t>(jt, p.NJ);
}

}  // namespace lgae

using namespace lgae;

extern "C" {

int lgae_cg_product_forward(const LgaeCgPairDesc* d, const int32_t* tab, const double* coef, const double* z1, const double* z2, int64_t rows,
                            int32_t n_nbr, double* const* outs, void* stream) {
    CgArgs p;
    if (rows < 0 || n_nbr < 0) return LGAE_E_BADARG;
    if (int rc = cg_fill(d, tab, coef, p, (void* const*)outs, rows)) return rc;
    if (rows == 0) return LGAE_OK;
    if (!z1 || !z2) return LGAE_E_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    p.z1 = z1; p.z2 = z2; p.g1 = p.g2 = nullptr; p.acc1 = p.acc2 = 0;
    if (n_nbr == 0) {
        p.B = (int32_t)rows; p.N = 1; p.NJ = 0; p.JT = 0;
        if (rows > INT32_MAX) return LGAE_E_UNSUPPORTED;
        p.plane1 = rows * p.C * p.d1; p.plane2 = rows * p.C * p.d2;
        const size_t bytes = terms_doubles(p.n_terms, p.n_comp + 1) * sizeof(double);
        if (int rc = ensure_smem((const void*)cg_pt_fwd_kernel, bytes)) return rc;
        LaunchScope ls_("cg_product_fwd", st);
        launch_k(cg_pt_fwd_kernel, dim3(grid_for(rows * p.C * p.n_comp, CG_THREADS)), dim3(CG_THREADS), bytes, st, p);
        return check_launch("cg_product_fwd");
    }
    if (rows % n_nbr) return LGAE_E_BADARG;
    p.B = (int32_t)(rows / n_nbr); p.N = n_nbr; p.NJ = n_nbr;
    p.plane1 = rows * p.C * p.d1; p.plane2 = rows * n_nbr * p.C * p.d2;
    if (p.C * p.n_comp > CG_ITEMS * CG_THREADS) return LGAE_E_UNSUPPORTED;
    {
        // whole-jet variant when the node slab + at least one edge row block fit next to the term table
        const size_t fixed0 = terms_doubles(p.n_terms, p.n_comp + 1) * sizeof(double);
        const size_t z1b = (size_t)p.NJ * p.C * p.d1 * sizeof(cplx), rowb = (size_t)p.NJ * p.C * p.d2 * sizeof(cplx), budget = 100 * 1024;
        if (fixed0 + z1b + rowb <= budget) {
            int ib = std::max(1, CG_THREADS / (p.C * p.n_comp));
            ib = std::min<int>(ib, p.N);
            while (ib > 1 && fixed0 + z1b + ib * rowb > budget) --ib;
            p.JT = ib;
            const size_t kb = (size_t)ib * p.C * p.d1 * p.d2 * sizeof(cplx);
            const size_t bytes = fixed0 + z1b + ib * rowb;
            const dim3 grid(p.B, (p.N + ib - 1) / ib);
            LaunchScope ls_("cg_aggregate_fwd", st);
#define LGAE_KRON(D)                                                                                  \
    if (p.d2 == D) {                                                                                  \
        if (int rc = ensure_smem((const void*)cg_agg_fwd_kron_kernel<D>, bytes + kb)) return rc;      \
        launch_k(cg_agg_fwd_kron_kernel<D>, grid, dim3(CG_THREADS), bytes + kb, st, p);               \
        return check_launch("cg_aggregate_fwd");                                                      \
    }
            if (bytes + kb <= CG_SMEM_MAX) {   // the Kronecker form also holds IB * C * d1 * d2 of K
                LGAE_KRON(1) LGAE_KRON(3) LGAE_KRON(4) LGAE_KRON(9)
            }
#undef LGAE_KRON
            if (int rc = ensure_smem((const void*)cg_agg_fwd_block_kernel, bytes)) return rc;
            launch_k(cg_agg_fwd_block_kernel, grid, dim3(CG_THREADS), bytes, st, p);
            return check_launch("cg_aggregate_fwd");
        }
    }
    p.JS = 1;   // few output items per (jet, i): several lanes share an item and split its neighbour sum
    while (p.JS < 32 && 2 * p.JS * p.C * p.n_comp <= CG_THREADS && 2 * p.JS <= p.NJ) p.JS *= 2;
    const size_t fixed = terms_doubles(p.n_terms, p.n_comp + 1) * sizeof(double);
    p.JT = cg_tile(p, fixed, false);
    if (p.JT < 1) return LGAE_E_UNSUPPORTED;
    const size_t bytes = fixed + (size_t)p.JT * (cg_row_stride(p.C * p.d1) + cg_row_stride(p.C * p.d2)) * sizeof(cplx);
    if (int rc = ensure_smem((const void*)cg_agg_fwd_kernel, bytes)) return rc;
    int split = (2 * sm_count() + p.B - 1) / p.B;
    split = std::max(1, std::min(split, (int)p.N));
    LaunchScope ls_("cg_aggregate_fwd", st);
    launch_k(cg_agg_fwd_kernel, dim3(p.B, split), dim3(CG_THREADS), bytes, st, p);
    return check_launch("cg_aggregate_fwd");
}

int lgae_cg_product_backward(const LgaeCgPairDesc* d, const int32_t* tab, const double* coef, const double* z1, const double* z2, int64_t rows,
                             int32_t n_nbr, const double* const* g_outs, double* g_z1, double* g_z2, int32_t accumulate_z1,
                             int32_t accumulate_z2, void* stream) {
    CgArgs p;
    if (rows < 0 || n_nbr < 0) return LGAE_E_BADARG;
    if (int rc = cg_fill(d, tab, coef, p, (void* const*)g_outs, rows)) return rc;
    if (rows == 0 || (!g_z1 && !g_z2)) return LGAE_OK;
    if (!z1 || !z2) return LGAE_E_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    p.z1 = z1; p.z2 = z2; p.g1 = g_z1; p.g2 = g_z2; p.acc1 = accumulate_z1; p.acc2 = accumulate_z2;
    const size_t terms = (terms_doubles(p.n_terms, p.d1 + 1) + terms_doubles(p.n_terms, p.d2 + 1)) * sizeof(double);
    if (n_nbr == 0) {
        if (rows > INT32_MAX) return LGAE_E_UNSUPPORTED;
        p.B = (int32_t)rows; p.N = 1; p.NJ = 0; p.JT = 0;
        p.plane1 = rows * p.C * p.d1; p.plane2 = rows * p.C * p.d2;
        if (int rc = ensure_smem((const void*)cg_pt_bwd_kernel, terms)) return rc;
        LaunchScope ls_("cg_product_bwd", st);
        launch_k(cg_pt_bwd_kernel, dim3(grid_for(rows * p.C * (p.d1 + p.d2), CG_THREADS)), dim3(CG_THREADS), terms, st, p);
        return check_launch("cg_product_bwd");
    }
    if (rows % n_nbr) return LGAE_E_BADARG;
    p.B = (int32_t)(rows / n_nbr); p.N = n_nbr; p.NJ = n_nbr;
    p.plane1 = rows * p.C * p.d1; p.plane2 = rows * n_nbr * p.C * p.d2;
    if (p.C * p.d1 > CG_ITEMS * CG_THREADS) return LGAE_E_UNSUPPORTED;
    if (p.g2) {
        // the edge gradient as its own fully parallel launch when the jet's node slab fits in shared memory
        const int ib = std::min<int>(8, p.N);
        const size_t bytes = terms_doubles(p.n_terms, p.d2 + 1) * sizeof(double) + ((size_t)p.NJ * p.C * p.d1 + (size_t)ib * p.C * p.n_comp) * sizeof(cplx);
        if (bytes <= 100 * 1024) {
            CgArgs q = p;
            q.JT = ib; q.g1 = nullptr;
            {
                LaunchScope ls_("cg_aggregate_bwd_edge", st);
                const dim3 grid(q.B, (q.N + ib - 1) / ib);
                const size_t kbytes = terms_doubles(p.n_terms, p.d1 + 1) * sizeof(double) +
                                      ((size_t)p.NJ * p.C * p.d1 + (size_t)ib * p.C * p.n_comp + (size_t)ib * p.C * p.d1 * p.d2) * sizeof(cplx);
                // the Kronecker form also holds IB * C * d1 * d2 of gK: the generic kernel where that does not fit
                const bool kron_fits = kbytes <= CG_SMEM_MAX;
                bool done = false;
#define LGAE_KRON(D)                                                                                          \
    if (!done && kron_fits && p.d2 == D) {                                                                    \
        if (int rc = ensure_smem((const void*)cg_agg_bwd_edge_kron_kernel<D>, kbytes)) return rc;             \
        launch_k(cg_agg_bwd_edge_kron_kernel<D>, grid, dim3(CG_THREADS), kbytes, st, q);                      \
        done = true;                                                                                          \
    }
                LGAE_KRON(1) LGAE_KRON(3) LGAE_KRON(4) LGAE_KRON(9)
#undef LGAE_KRON
                if (!done) {
                    if (int rc = ensure_smem((const void*)cg_agg_bwd_edge_kernel, bytes)) return rc;
                    launch_k(cg_agg_bwd_edge_kernel, grid, dim3(CG_THREADS), bytes, st, q);
                }
                if (int rc = check_launch("cg_aggregate_bwd_edge")) return rc;
            }
            p.g2 = nullptr;
            if (!p.g1) return LGAE_OK;
        }
    }
    if (!p.g2 && p.g1 && p.NJ * p.C <= 2 * CG_THREADS) {
        // node gradient in Kronecker form, one CTA per jet, for the common (d1, d2)
        const size_t t1 = terms_doubles(p.n_terms, p.d1 + 1) * sizeof(double);
        const size_t rowb = (size_t)p.NJ * p.C * p.d2 * sizeof(cplx);
        const size_t per_ib = rowb + ((size_t)p.C * p.n_comp + (size_t)p.C * p.d1 * p.d2) * sizeof(cplx);
        int ib = std::min<int>(4, p.N);
        while (ib > 1 && t1 + ib * per_ib > 100 * 1024) --ib;
        const size_t nbytes = t1 + ib * per_ib;
        if (nbytes <= 100 * 1024) {
            CgArgs q = p;
            q.JT = ib;
            bool done = false;
            LaunchScope ls_("cg_aggregate_bwd_node", st);
#define LGAE_KRON(A, D)                                                                                           \
    if (!done && p.d1 == A && p.d2 == D) {                                                                        \
        if (int rc = ensure_smem((const void*)cg_agg_bwd_node_kron_kernel<A, D>, nbytes)) return rc;              \
        launch_k(cg_agg_bwd_node_kron_kernel<A, D>, dim3(q.B), dim3(CG_THREADS), nbytes, st, q);                  \
        done = true;                                                                                              \
    }
            LGAE_KRON(1, 1) LGAE_KRON(3, 1) LGAE_KRON(4, 1) LGAE_KRON(9, 1)
            LGAE_KRON(1, 4) LGAE_KRON(3, 4) LGAE_KRON(4, 4) LGAE_KRON(9, 4)
#undef LGAE_KRON
            if (done) return check_launch("cg_aggregate_bwd_node");
        }
    }
    const size_t fixed = terms + (size_t)p.C * p.n_comp * sizeof(cplx);
    p.JT = cg_tile(p, fixed, true);
    if (p.JT < 1) return LGAE_E_UNSUPPORTED;
    const size_t bytes = fixed + (size_t)p.JT * (cg_row_stride(p.C * p.d1) + cg_row_stride(p.C * p.d2)) * sizeof(cplx);
    if (int rc = ensure_smem((const void*)cg_agg_bwd_kernel, bytes)) return rc;
    LaunchScope ls_("cg_aggregate_bwd", st);
    launch_k(cg_agg_bwd_kernel, dim3(p.B, (p.NJ + p.JT - 1) / p.JT), dim3(CG_THREADS), bytes, st, p);
    return check_launch("cg_aggregate_bwd");
}

static int multi_fill(CgMultiArgs& p, const LgaeCgMultiDesc* d, const int32_t* tab, const double* coef, const double* const* node_parts,
                      const double* const* edge_parts, int64_t rows, int32_t n_nbr, double* const* outs);

int lgae_cg_aggregate_multi_backward(const LgaeCgMultiDesc* d, const int32_t* tab_b, const double* coef_b, const double* const* node_parts,
                                     const double* const* edge_parts, int64_t rows, int32_t n_nbr, const double* const* g_outs,
                                     double* const* g_node, double* const* g_edge, void* stream) {
    CgMultiArgs p;
    if (!g_node || !g_edge) return LGAE_E_BADARG;
    if (int rc = multi_fill(p, d, tab_b, coef_b, node_parts, edge_parts, rows, n_nbr, (double* const*)g_outs)) return rc;
    if (rows == 0) return LGAE_OK;
    p.tab_b = tab_b; p.coef_b = coef_b;
    bool want_node = false, want_edge = false;
    for (int i = 0; i < d->n_node; ++i) { p.gnode[i] = g_node[i]; want_node |= g_node[i] != nullptr; }
    for (int i = 0; i < d->n_edge; ++i) { p.gedge[i] = g_edge[i]; want_edge |= g_edge[i] != nullptr; }
    const int D1T = p.node_off[d->n_node], D2T = p.edge_off[d->n_edge], ncell = D1T * D2T;
    const size_t tabs = multi_bwd_tab_bytes(p.n_terms, p.n_comp, ncell);
    cudaStream_t st = (cudaStream_t)stream;
    if (want_node && !((D1T == 5 || D1T == 20) && D2T == 5 && p.NJ * p.C <= CG_THREADS)) return LGAE_E_UNSUPPORTED;
    if (want_edge && !(D2T == 1 || D2T == 4 || D2T == 5)) return LGAE_E_UNSUPPORTED;
    if (want_edge) {
        const size_t per_ib = ((size_t)p.C * p.n_comp + (size_t)p.C * ncell) * sizeof(cplx);
        int ib = std::min<int>(LGAE_AGG_EDGE_IB, p.N);
        while (ib > 1 && tabs + ib * per_ib > 100 * 1024) --ib;
        const size_t bytes = tabs + ib * per_ib;
        if (bytes > 160 * 1024) return LGAE_E_UNSUPPORTED;
        p.IB = ib;
        const dim3 grid(p.B, (p.N + ib - 1) / ib);
        LaunchScope ls_("cg_aggregate_multi_bwd_edge", st);
#define LGAE_MULTI(D)                                                                                      \
    if (D2T == D) {                                                                                        \
        if (int rc = ensure_smem((const void*)cg_agg_multi_bwd_edge_kernel<D>, bytes)) return rc;          \
        launch_k(cg_agg_multi_bwd_edge_kernel<D>, grid, dim3(CG_THREADS), bytes, st, p);                   \
    }
        LGAE_MULTI(1) LGAE_MULTI(4) LGAE_MULTI(5)
#undef LGAE_MULTI
        if (int rc = check_launch("cg_aggregate_multi_bwd_edge")) return rc;
    }
    if (want_node) {
        const size_t per_ib = ((size_t)p.NJ * p.C * D2T + (size_t)p.C * p.n_comp + (size_t)p.C * ncell) * sizeof(cplx);
        int ib = std::min<int>(2, p.N);
        while (ib > 1 && tabs + ib * per_ib > 100 * 1024) --ib;
        const size_t bytes = tabs + ib * per_ib;
        if (bytes > 160 * 1024) return LGAE_E_UNSUPPORTED;
        p.IB = ib;
        LaunchScope ls_("cg_aggregate_multi_bwd_node", st);
        if (D1T == 5) {
            if (int rc = ensure_smem((const void*)cg_agg_multi_bwd_node_kernel<5, 5>, bytes)) return rc;
            launch_k(cg_agg_multi_bwd_node_kernel<5, 5>, dim3(p.B), dim3(CG_THREADS), bytes, st, p);
        } else {
            if (int rc = ensure_smem((const void*)cg_agg_multi_bwd_node_kernel<20, 5>, bytes)) return rc;
            launch_k(cg_agg_multi_bwd_node_kernel<20, 5>, dim3(p.B), dim3(CG_THREADS), bytes, st, p);
        }
        if (int rc = check_launch("cg_aggregate_multi_bwd_node")) return rc;
    }
    return LGAE_OK;
}

static int multi_fill(CgMultiArgs& p, const LgaeCgMultiDesc* d, const int32_t* tab, const double* coef, const double* const* node_parts,
                      const double* const* edge_parts, int64_t rows, int32_t n_nbr, double* const* outs) {
    if (!d || !tab || !coef || !node_parts || !edge_parts || !outs || rows < 0 || n_nbr < 1) return LGAE_E_BADARG;
    if (d->n_node < 1 || d->n_node > LGAE_CG_MAX_PARTS || d->n_edge < 1 || d->n_edge > LGAE_CG_MAX_PARTS || d->n_out < 1 ||
        d->n_out > LGAE_CG_MAX_OUT || d->channels < 1 || d->n_comp < 1 || d->n_terms < 1)
        return LGAE_E_BADARG;
    if (rows % n_nbr) return LGAE_E_BADARG;
    memset(&p, 0, sizeof(p));
    p.B = (int32_t)(rows / n_nbr); p.N = n_nbr; p.NJ = n_nbr; p.C = d->channels; p.n_node = d->n_node; p.n_edge = d->n_edge;
    p.n_comp = d->n_comp; p.n_terms = d->n_terms; p.tab = tab; p.coef = coef;
    p.node_off[0] = p.edge_off[0] = 0;
    for (int i = 0; i < d->n_node; ++i) {
        if (!node_parts[i] || d->node_d[i] < 1) return LGAE_E_BADARG;
        p.node[i] = node_parts[i]; p.node_d[i] = d->node_d[i]; p.node_off[i + 1] = p.node_off[i] + d->node_d[i];
    }
    for (int i = 0; i < d->n_edge; ++i) {
        if (!edge_parts[i] || d->edge_d[i] < 1) return LGAE_E_BADARG;
        p.edge[i] = edge_parts[i]; p.edge_d[i] = d->edge_d[i]; p.edge_off[i + 1] = p.edge_off[i] + d->edge_d[i];
    }
    for (int i = 0; i < d->n_out; ++i) {
        if (!outs[i] || d->out_d[i] < 1 || d->out_ctotal[i] < d->channels) return LGAE_E_BADARG;
        p.out[i] = outs[i]; p.out_d[i] = d->out_d[i]; p.out_ctot[i] = d->out_ctotal[i];
    }
    return LGAE_OK;
}

int lgae_cg_aggregate_multi_forward(const LgaeCgMultiDesc* d, const int32_t* tab, const double* coef, const double* const* node_parts,
                                    const double* const* edge_parts, int64_t rows, int32_t n_nbr, double* const* outs, void* stream) {
    CgMultiArgs p;
    if (int rc = multi_fill(p, d, tab, coef, node_parts, edge_parts, rows, n_nbr, outs)) return rc;
    if (rows == 0) return LGAE_OK;
    const int D1T = p.node_off[d->n_node], D2T = p.edge_off[d->n_edge];
    const size_t fixed = (size_t)p.n_terms * sizeof(double) + ((size_t)2 * p.n_terms + (size_t)4 * p.n_comp + 2) * sizeof(int32_t) + 16;
    const size_t per_ib = ((size_t)p.NJ * p.C * D2T + (size_t)p.C * D1T * D2T) * sizeof(cplx);
    int ib = std::min<int>(LGAE_AGG_FWD_IB, p.N);
    while (ib > 1 && fixed + ib * per_ib > 100 * 1024) --ib;
    const size_t bytes = fixed + ib * per_ib;
    if (bytes > 160 * 1024) return LGAE_E_UNSUPPORTED;
    p.IB = ib;
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid(p.B, (p.N + ib - 1) / ib);
    LaunchScope ls_("cg_aggregate_multi_fwd", st);
#define LGAE_MULTI(D)                                                                                 \
    if (D2T == D) {                                                                                   \
        if (int rc = ensure_smem((const void*)cg_agg_multi_fwd_kernel<D>, bytes)) return rc;          \
        launch_k(cg_agg_multi_fwd_kernel<D>, grid, dim3(CG_THREADS), bytes, st, p);                   \
        return check_launch("cg_aggregate_multi_fwd");                                                \
    }
    LGAE_MULTI(1) LGAE_MULTI(4) LGAE_MULTI(5)
#undef LGAE_MULTI
    return LGAE_E_UNSUPPORTED;
}

int64_t lgae_mix_partials_doubles(int64_t rows, int32_t c_in, int32_t c_out) {
    if (rows < 0 || c_in < 1 || c_out < 1) return -1;
    const int64_t ctas = std::max<int64_t>(1, std::min<int64_t>(rows, 4 * (int64_t)sm_count()));
    return ctas * 2 * c_in * c_out;
}

int lgae_mix_forward(const double* w, const double* x, int64_t rows, int32_t c_in, int32_t c_out, int32_t d, double* out, void* stream) {
    if (rows < 0 || c_in < 1 || c_out < 1 || d < 1) return LGAE_E_BADARG;
    if (rows == 0) return LGAE_OK;
    if (!w || !x || !out) return LGAE_E_BADARG;
    MixArgs a = {};
    a.x = x; a.w = w; a.out = out; a.R = rows; a.cin = c_in; a.cout = c_out; a.d = d;
    cudaStream_t st = (cudaStream_t)stream;
    LaunchScope ls_("mix_fwd", st);
#define LGAE_MIXF(COV)                                                                                              \
    {                                                                                                               \
        const size_t bytes = (size_t)c_in * COV * sizeof(cplx);                                                     \
        if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;                                                          \
        if (int rc = ensure_smem((const void*)mix_fwd_kernel<COV>, bytes)) return rc;                               \
        launch_k(mix_fwd_kernel<COV>, dim3(grid_for(rows * d, MIX_THREADS)), dim3(MIX_THREADS), bytes, st, a);      \
    }
    if (c_out <= 4) LGAE_MIXF(4) else if (c_out <= 8) LGAE_MIXF(8) else
        for (a.co0 = 0; a.co0 < c_out; a.co0 += 16) LGAE_MIXF(16)
#undef LGAE_MIXF
    return check_launch("mix_fwd");
}

int lgae_mix_backward(const double* w, const double* x, const double* g_out, int64_t rows, int32_t c_in, int32_t c_out, int32_t d, double* g_x,
                      double* g_w, double* partials, void* stream) {
    if (rows < 0 || c_in < 1 || c_out < 1 || d < 1) return LGAE_E_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (rows == 0) {
        if (g_w && cudaMemsetAsync(g_w, 0, (size_t)2 * c_in * c_out * sizeof(double), st) != cudaSuccess) return check_launch("memset g_w");
        return LGAE_OK;
    }
    if (!w || !x || !g_out || (g_w && !partials)) return LGAE_E_BADARG;
    MixArgs a = {};
    a.x = x; a.w = w; a.g = g_out; a.gx = g_x; a.gw_part = partials; a.R = rows; a.cin = c_in; a.cout = c_out; a.d = d;
    if (g_x) {
        const size_t bytes = (size_t)c_in * c_out * sizeof(cplx);
        if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
        if (int rc = ensure_smem((const void*)mix_bwd_x_kernel, bytes)) return rc;
        LaunchScope ls_("mix_bwd_x", st);
        launch_k(mix_bwd_x_kernel, dim3(grid_for(rows * c_in * d, MIX_THREADS)), dim3(MIX_THREADS), bytes, st, a);
        if (int rc = check_launch("mix_bwd_x")) return rc;
    }
    if (g_w) {
        const int64_t ctas = std::max<int64_t>(1, std::min<int64_t>(rows, 4 * (int64_t)sm_count()));
        a.rows_per_cta = (int32_t)((rows + ctas - 1) / ctas);
        const int grid = (int)((rows + a.rows_per_cta - 1) / a.rows_per_cta);
        const size_t row_bytes = (size_t)(c_in + c_out) * d * sizeof(cplx);
        if (row_bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
        const int co_blk = c_out <= 4 ? 4 : 8;
        const int cb = std::min<int>(c_in, MIX_THREADS);
        // rows per stage: about 64 KB of staging, a multiple of the row lanes
        int rb = (int)std::max<size_t>(1, (64 * 1024) / row_bytes);
        const int nsub = std::max(1, std::min(MIX_THREADS / cb, rb));
        rb = std::max(nsub, rb / nsub * nsub);
        rb = std::min<int>(rb, std::max<int>(nsub, (a.rows_per_cta + nsub - 1) / nsub * nsub));
        const size_t red_bytes = (size_t)nsub * cb * co_blk * sizeof(cplx);
        const size_t bytes = std::max(row_bytes * rb, red_bytes);
        if (bytes > 200 * 1024) return LGAE_E_UNSUPPORTED;
        a.co0 = rb;
        a.nsub = nsub;
        {
            LaunchScope ls_("mix_bwd_w", st);
            if (co_blk == 4) {
                if (int rc = ensure_smem((const void*)mix_bwd_w_kernel<4>, bytes)) return rc;
                launch_k(mix_bwd_w_kernel<4>, dim3(grid), dim3(MIX_THREADS), bytes, st, a);
            } else {
                if (int rc = ensure_smem((const void*)mix_bwd_w_kernel<8>, bytes)) return rc;
                launch_k(mix_bwd_w_kernel<8>, dim3(grid), dim3(MIX_THREADS), bytes, st, a);
            }
            if (int rc = check_launch("mix_bwd_w")) return rc;
        }
        const int64_t n = (int64_t)2 * c_in * c_out;
        LaunchScope ls_("mix_bwd_w_sum", st);
        launch_k(colsum_kernel, dim3((unsigned)((n + 31) / 32)), dim3(32, COLSUM_Y), 0, st, (const double*)partials, grid, n, g_w);
        return check_launch("mix_bwd_w_sum");
    }
    return LGAE_OK;
}

}  // extern "C"
