// Shared device helpers for the LGAE sm_100a kernels: interleaved-complex arithmetic, the fp64 tensor-core
// instruction (DMMA m8n8k4), warp/block reductions and the host-side launch bookkeeping.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/lgae_b200.h"

namespace lgae {

typedef double2 cplx;  // x = re, y = im

#define LGAE_DEV __device__ __forceinline__

LGAE_DEV cplx cmake(double re, double im) { return make_double2(re, im); }
LGAE_DEV cplx czero() { return make_double2(0.0, 0.0); }
LGAE_DEV cplx cadd(cplx a, cplx b) { return make_double2(a.x + b.x, a.y + b.y); }
LGAE_DEV cplx csub(cplx a, cplx b) { return make_double2(a.x - b.x, a.y - b.y); }
LGAE_DEV cplx cneg(cplx a) { return make_double2(-a.x, -a.y); }
LGAE_DEV cplx cconj(cplx a) { return make_double2(a.x, -a.y); }
LGAE_DEV cplx cscale(cplx a, double s) { return make_double2(a.x * s, a.y * s); }
LGAE_DEV cplx cmul(cplx a, cplx b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
// conj(a) * b
LGAE_DEV cplx cmulc(cplx a, cplx b) { return make_double2(a.x * b.x + a.y * b.y, a.x * b.y - a.y * b.x); }
// acc += a * b
LGAE_DEV void cfma(cplx& acc, cplx a, cplx b) {
    acc.x = fma(a.x, b.x, acc.x);
    acc.x = fma(-a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y);
    acc.y = fma(a.y, b.x, acc.y);
}
// acc += conj(a) * b
LGAE_DEV void cfmac(cplx& acc, cplx a, cplx b) {
    acc.x = fma(a.x, b.x, acc.x);
    acc.x = fma(a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y);
    acc.y = fma(-a.y, b.x, acc.y);
}
// acc += a * s  (s real)
LGAE_DEV void cfmar(cplx& acc, cplx a, double s) {
    acc.x = fma(a.x, s, acc.x);
    acc.y = fma(a.y, s, acc.y);
}
// (1+i) * a   and   (1-i) * a
LGAE_DEV cplx cmul_1pi(cplx a) { return make_double2(a.x - a.y, a.x + a.y); }
LGAE_DEV cplx cmul_1mi(cplx a) { return make_double2(a.x + a.y, a.y - a.x); }

// Canonical-basis metric of the (1,1) irrep: eta(a,b) = a0 b0 + a1 b3 - a2 b2 + a3 b1 (complex bilinear,
// lgn/cg_lib/zonal_functions.py:396-438; equals the Minkowski product of the Cartesian components).
LGAE_DEV cplx ceta(const cplx* a, const cplx* b) {
    cplx r = cmul(a[0], b[0]);
    cfma(r, a[1], b[3]);
    cfma(r, cneg(a[2]), b[2]);
    cfma(r, a[3], b[1]);
    return r;
}
// ghat(a)_mu: eta(a,b) = sum_mu ghat(a)_mu b_mu
LGAE_DEV void cghat(const cplx* a, cplx* out) {
    out[0] = a[0];
    out[1] = a[3];
    out[2] = cneg(a[2]);
    out[3] = a[1];
}

#define LGAE_RSQRT2 0.70710678118654752440

// Real Cartesian (t,x,y,z) -> canonical complex components, with the reference's rounding
// (a matrix product with entries 1 and +-1/sqrt(2), lgn/cg_lib/zonal_functions.py:251-289).
LGAE_DEV void canon_from_real(const double* p, cplx* y) {
    const double a = __dmul_rn(LGAE_RSQRT2, p[1]);
    const double b = __dmul_rn(LGAE_RSQRT2, p[2]);
    y[0] = cmake(p[0], 0.0);
    y[1] = cmake(a, -b);
    y[2] = cmake(p[3], 0.0);
    y[3] = cmake(-a, -b);
}
// Complex Cartesian -> canonical (p_cplx_to_rep, zonal_functions.py:292-341)
LGAE_DEV void canon_from_cplx(const cplx* p, cplx* y) {
    y[0] = p[0];
    y[1] = cmake(LGAE_RSQRT2 * (p[1].x + p[2].y), LGAE_RSQRT2 * (p[1].y - p[2].x));    // (x - i y)/sqrt2
    y[2] = p[3];
    y[3] = cmake(-LGAE_RSQRT2 * (p[1].x - p[2].y), -LGAE_RSQRT2 * (p[1].y + p[2].x));  // -(x + i y)/sqrt2
}
// Adjoint of canon_from_cplx == rep_to_p (zonal_functions.py:344-381): canonical -> complex Cartesian
LGAE_DEV void cart_from_canon(const cplx* v, cplx* p) {
    p[0] = v[0];
    p[1] = cmake(LGAE_RSQRT2 * (v[1].x - v[3].x), LGAE_RSQRT2 * (v[1].y - v[3].y));
    // i * (v1 + v3) / sqrt2
    p[2] = cmake(-LGAE_RSQRT2 * (v[1].y + v[3].y), LGAE_RSQRT2 * (v[1].x + v[3].x));
    p[3] = v[2];
}

// Minkowski square of a real 4-vector with the reference's exact rounding sequence
// (zonal_functions.py:201-218: psq = p**2 ; 2*psq[0] - psq.sum(-1), torch sums the 4 terms left to right).
LGAE_DEV double minkowski_sq(double p0, double p1, double p2, double p3) {
    const double q0 = __dmul_rn(p0, p0), q1 = __dmul_rn(p1, p1), q2 = __dmul_rn(p2, p2), q3 = __dmul_rn(p3, p3);
    const double s = __dadd_rn(__dadd_rn(__dadd_rn(q0, q1), q2), q3);
    return __dsub_rn(__dmul_rn(2.0, q0), s);
}

// D(8x8) += A(8x4) * B(4x8), fp64 tensor-core MMA.  Fragment layout (g = lane>>2, q = lane&3):
//   a = A[g][q], b = B[q][g], c0/c1 = C[g][2q], C[g][2q+1].
LGAE_DEV void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// ---- TMA 1-D bulk copies global -> shared, completion signalled on an mbarrier -------------------------------------
// (cp.async.bulk: one elected thread issues the copy of a whole contiguous record -- a jet's node features --, every
// thread then waits on the barrier's phase parity; addresses and sizes must be multiples of 16 bytes.)
LGAE_DEV unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
LGAE_DEV void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
LGAE_DEV void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
LGAE_DEV void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// TMA bulk prefetch of a contiguous global range into L2 (no shared-memory destination, no completion to wait for).
LGAE_DEV void bulk_prefetch_l2(const void* src, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
LGAE_DEV void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LGAE_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LGAE_DONE;\n"
        "bra LGAE_WAIT;\n"
        "LGAE_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

LGAE_DEV double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sums of 32 per-lane values over the warp with 16+8+4+2+1 = 31 shuffles: on return lane l holds the total of value l.
LGAE_DEV double warp_sum32(const double (&v)[32]) {
    const int lane = threadIdx.x & 31;
    double a[16], b[8], c[4], d[2];
    {
        const bool up = lane & 16;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const double send = up ? v[j] : v[j + 16], keep = up ? v[j + 16] : v[j];
            a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
    }
    {
        const bool up = lane & 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const double send = up ? a[j] : a[j + 8], keep = up ? a[j + 8] : a[j];
            b[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool up = lane & 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double send = up ? b[j] : b[j + 4], keep = up ? b[j + 4] : b[j];
            c[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
    }
    {
        const bool up = lane & 2;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const double send = up ? c[j] : c[j + 2], keep = up ? c[j + 2] : c[j];
            d[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
        }
    }
    const bool up = lane & 1;
    const double send = up ? d[0] : d[1], keep = up ? d[1] : d[0];
    return keep + __shfl_xor_sync(0xffffffffu, send, 1);
}
// All-reduce of NV <= 32 per-lane values: v[t] becomes the warp total of value t in every lane (31 + NV shuffles).
template <int NV>
LGAE_DEV void warp_allsum_n(double (&v)[NV]) {
    double w[32];
#pragma unroll
    for (int t = 0; t < 32; ++t) w[t] = t < NV ? v[t] : 0.0;
    const double tot = warp_sum32(w);
#pragma unroll
    for (int t = 0; t < NV; ++t) v[t] = __shfl_sync(0xffffffffu, tot, t);
}

// Sum over the warp, result in every lane (the xor butterfly of warp_sum already has that property).
LGAE_DEV double warp_allsum(double v) { return warp_sum(v); }

// Block-wide sum; result valid in thread 0.  `scratch` must hold >= 32 doubles.
LGAE_DEV double block_sum(double v, double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    double r = 0.0;
    if (warp == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        r = lane < nw ? scratch[lane] : 0.0;
        r = warp_sum(r);
    }
    return r;
}

LGAE_DEV double leaky(double x, double slope) { return x > 0.0 ? x : x * slope; }

// Sums of 16 per-lane values over the 32 lanes of a warp with 8+4+2+1+1 = 16 shuffles instead of 5*16: a
// butterfly that halves the number of live values at every stage.  On return lane l holds the total of value
// number l >> 1 (each total is replicated in two neighbouring lanes).
LGAE_DEV double warp_sum16(const double (&v)[16]) {
    const int lane = threadIdx.x & 31;
    double a[8], b[4], c[2], d;
    {
        const bool up = lane & 16;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const double send = up ? v[j] : v[j + 8], keep = up ? v[j + 8] : v[j];
            a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
    }
    {
        const bool up = lane & 8;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double send = up ? a[j] : a[j + 4], keep = up ? a[j + 4] : a[j];
            b[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool up = lane & 4;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const double send = up ? b[j] : b[j + 2], keep = up ? b[j + 2] : b[j];
            c[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
    }
    {
        const bool up = lane & 2;
        const double send = up ? c[0] : c[1], keep = up ? c[1] : c[0];
        d = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    return d + __shfl_xor_sync(0xffffffffu, d, 1);
}

// ---- parameter-gradient partials ------------------------------------------------------------------------
// Every backward kernel writes one compact row of parameter-gradient partials per CTA into its own block of the
// scratch buffer `partials`; one reduce launch then sums the rows of every block into gtheta.  A segment maps a
// contiguous range of theta to a column range of a block.
#define LGAE_MAX_SEGS 64
struct Seg {
    int64_t theta_off;  // first parameter (offset in theta / gtheta)
    int64_t part_off;   // offset (doubles) of row 0, column 0 of this segment inside `partials`
    int64_t stride;     // row stride (doubles) of the block
    int32_t len;        // number of parameters
    int32_t rows;       // number of rows (CTAs of the producing kernel)
};
struct SegTable {
    int32_t n;
    int32_t pad;
    Seg s[LGAE_MAX_SEGS];
    int32_t chunk0[LGAE_MAX_SEGS + 1];   // filled by the reduce launcher: first 32-column chunk (= block index) of every segment
};
// Host-side allocator of blocks inside `partials`.
struct PartPlan {
    double* base = nullptr;
    int64_t used = 0;
    int64_t theta_base = 0;   // added to every segment's theta offset (two models sharing one gradient bucket)
    SegTable table;
    PartPlan() { table.n = 0; table.pad = 0; }
    // reserve rows x width doubles; returns the block's offset
    int64_t block(int rows, int64_t width) {
        const int64_t off = used;
        used += (int64_t)rows * width;
        return off;
    }
    // declare that columns [col, col+len) of the block at `off` hold the gradient of theta[theta_off ...]
    int seg(int64_t theta_off, int64_t off, int64_t stride, int64_t col, int64_t len, int rows) {
        if (len <= 0) return LGAE_OK;
        theta_off += theta_base;
        if (table.n > 0) {   // merge with the previous segment when both ranges continue it
            Seg& p = table.s[table.n - 1];
            if (p.rows == rows && p.stride == stride && p.theta_off + p.len == theta_off && p.part_off + p.len == off + col) {
                p.len += (int32_t)len;
                return LGAE_OK;
            }
        }
        if (table.n >= LGAE_MAX_SEGS) return LGAE_E_UNSUPPORTED;
        Seg& s = table.s[table.n++];
        s.theta_off = theta_off; s.part_off = off + col; s.stride = stride; s.len = (int32_t)len; s.rows = rows;
        return LGAE_OK;
    }
};

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------------
// Every kernel of the library is launched with the programmatic-stream-serialisation attribute and starts with
// pdl_launch(): the next kernel in the stream may then be scheduled while this one is still running, runs the part of its
// prologue that only touches step-constant data (weights in theta, index tables, barrier setup) and blocks in pdl_wait()
// until all earlier kernels have completed and flushed their writes.  Every read of a predecessor's output and every global
// write comes after pdl_wait().  The launch latency and the prologues of the ~45 kernels of a step overlap the previous
// kernel's tail; captured in a CUDA graph the edges become programmatic dependencies.
LGAE_DEV void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
LGAE_DEV void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- host side ------------------------------------------------------------------------------------
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
void count_launch(int n = 1);
// Scope around one kernel launch: counts it and, when per-kernel timing is enabled (lgae_timing_enable), brackets it with
// CUDA events on the launch stream so that bench.py can report measured per-kernel durations without a profiler.
struct LaunchScope {
    const char* name;
    cudaStream_t st;
    void* ev0;
    LaunchScope(const char* name_, cudaStream_t st_);
    ~LaunchScope();
};
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per kernel (and again only if a larger size is needed).
int ensure_smem(const void* kernel, size_t bytes);
int check_launch(const char* what);
int sm_count();

}  // namespace lgae
