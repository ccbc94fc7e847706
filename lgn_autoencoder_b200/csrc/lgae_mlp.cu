// CGMLP (lgn/models/lgn_levels.py:191-227): weight packing and the dispatch of the MLP kernels (lgae_mlp.cuh, and
// lgae_mlp_streamed.cuh for the layers those cannot hold) by activation and tiling; the resident LeakyReLU kernels are
// instantiated here.
#include <cstring>

#include "lgae_mlp_streamed.cuh"

namespace lgae {

// Stage W (out x in, row-major, from theta) into fragment order for  D[row][n] += A[row][k] W[n][k]:
//   Wp[((kt*2+e)*NO + nt)*32 + q*8 + g] = W[8nt+g][8kt+2q+e]
LGAE_DEV void stage_w_fwd(const double* w, int nout, int nink, int KT, int NO, double* Wp) {
    const int total = KT * 2 * NO * 32;
    for (int t = threadIdx.x; t < total; t += blockDim.x) {
        const int g = t & 7, q = (t >> 3) & 3, r = t >> 5, nt = r % NO, ke = r / NO, kt = ke >> 1, e = ke & 1;
        const int n = 8 * nt + g, k = 8 * kt + 2 * q + e;
        Wp[t] = (n < nout && k < nink) ? w[(int64_t)n * nink + k] : 0.0;
    }
}
// Transposed use  Gin[row][k] += Gout[row][n] W[n][k]:
//   Wq[((nt*2+e)*KI + kt)*32 + q*8 + g] = W[8nt+2q+e][8kt+g]
LGAE_DEV void stage_w_bwd(const double* w, int nout, int nink, int NO, int KI, double* Wq) {
    const int total = NO * 2 * KI * 32;
    for (int t = threadIdx.x; t < total; t += blockDim.x) {
        const int g = t & 7, q = (t >> 3) & 3, r = t >> 5, kt = r % KI, ne = r / KI, nt = ne >> 1, e = ne & 1;
        const int n = 8 * nt + 2 * q + e, k = 8 * kt + g;
        Wq[t] = (n < nout && k < nink) ? w[(int64_t)n * nink + k] : 0.0;
    }
}

// ------------------------------------------------------------------------------------------------------------
// Weight pre-packing: one launch per model forward writes every level's weights in both fragment orders, so the
// MLP kernels stage them with straight vector copies.  blockIdx = (layer, direction, level).
constexpr int PACK_SLOTS = 2 * LGAE_MAX_LEVELS;   // levels of up to two models (encoder + decoder) per launch
struct MlpPackArgs {
    const double* theta[PACK_SLOTS];
    double* out[PACK_SLOTS];           // where the level's packed weights go
    int n_lin[PACK_SLOTS];
    int nin[PACK_SLOTS], width[PACK_SLOTS];
    int64_t off_w[PACK_SLOTS][LGAE_MAX_LINEAR];
};
__global__ void __launch_bounds__(256) mlp_pack_kernel(const MlpPackArgs p) {
    // no early launch_dependents: the MLP kernels stage the packed weights in their prologues, before their own dependency
    // wait, so nothing later in the stream may start before this kernel has completed
    pdl_wait();   // (writes the packed weights that earlier kernels of a previous pass may still be reading)
    const int l = blockIdx.x, dir = blockIdx.y, lev = blockIdx.z;
    const int n_lin = p.n_lin[lev];
    if (l >= n_lin) return;
    const int nin = p.nin[lev], width = p.width[lev], NTW = (width + 7) / 8, NTI = (nin + 7) / 8, last = n_lin - 1;
    int off = 0, wtotal = 0;
    for (int i = 0; i <= last; ++i) {
        if (i < l) off += mlp_layer_frag(i, n_lin, NTW, NTI);
        wtotal += mlp_layer_frag(i, n_lin, NTW, NTI);
    }
    const int nout = l == last ? nin : width, nink = l == 0 ? nin : width;
    const double* w = p.theta[lev] + p.off_w[lev][l];
    double* dst = p.out[lev] + (dir ? wtotal : 0) + off;
    if (dir == 0)
        stage_w_fwd(w, nout, nink, l == 0 ? NTI : NTW, l == last ? NTI : NTW, dst);
    else
        stage_w_bwd(w, nout, nink, l == last ? NTI : NTW, l == 0 ? NTI : NTW, dst);
}

int mlp_bwd_grid() { return sm_count(); }

// Doubles of packed weights (both orders) of one level.
int64_t mlp_pack_doubles(const LgaeModelDesc* d, int level) {
    if (!d->has_mlp) return 0;
    return 2 * (int64_t)mlp_frag_total(d->mlp_hidden + 1, (d->mlp_width[level] + 7) / 8, (2 * d->channels[level + 1] + 7) / 8);
}
// Pack the MLP weights of every level: out + out_off[level] receives mlp_pack_doubles(d, level) doubles.
static int add_pack_slots(MlpPackArgs& p, int slot, const LgaeModelDesc* d, const double* theta, double* out, const int64_t* out_off) {
    if (!d->has_mlp) return slot;
    for (int l = 0; l < d->n_levels; ++l, ++slot) {
        p.theta[slot] = theta;
        p.out[slot] = out + out_off[l];
        p.n_lin[slot] = d->mlp_hidden + 1;
        p.nin[slot] = 2 * d->channels[l + 1];
        p.width[slot] = d->mlp_width[l];
        for (int i = 0; i < p.n_lin[slot]; ++i) p.off_w[slot][i] = d->off_mlp_w[l][i];
    }
    return slot;
}
// One launch packs the weights of all levels of one model -- or of two (d2 != NULL: the training step's encoder + decoder).
int run_mlp_pack(const LgaeModelDesc* d, const double* theta, double* out, const int64_t* out_off, cudaStream_t st,
                 const LgaeModelDesc* d2 = nullptr, const double* theta2 = nullptr, double* out2 = nullptr, const int64_t* out_off2 = nullptr) {
    MlpPackArgs p;
    memset(&p, 0, sizeof(p));
    int slots = add_pack_slots(p, 0, d, theta, out, out_off);
    if (d2) slots = add_pack_slots(p, slots, d2, theta2, out2, out_off2);
    if (slots == 0) return LGAE_OK;
    int max_lin = 0;
    for (int i = 0; i < slots; ++i) max_lin = p.n_lin[i] > max_lin ? p.n_lin[i] : max_lin;
    LaunchScope ls_("mlp_pack", st);
    launch_k(mlp_pack_kernel, dim3(max_lin, 2, slots), dim3(256), 0, st, p);
    return check_launch("mlp_pack");
}

// The other activations' kernels come from lgae_mlp_act_*.cu.
LGAE_MLP_INSTANCES(extern, LGAE_ACT_RELU)
LGAE_MLP_INSTANCES(extern, LGAE_ACT_ELU)
LGAE_MLP_INSTANCES(extern, LGAE_ACT_SIGMOID)
LGAE_MLP_INSTANCES(extern, LGAE_ACT_LOGSIGMOID)
LGAE_MLP_INSTANCES(extern, LGAE_ACT_TANH)
LGAE_MLP_INSTANCES(extern, LGAE_ACT_ATAN)
// The streamed kernels come from lgae_mlp_streamed_*.cu, one unit per activation.
LGAE_MLP_STREAMED_INSTANCES(extern, LGAE_ACT_LEAKYRELU)
LGAE_MLP_STREAMED_INSTANCES(extern, LGAE_ACT_RELU)
LGAE_MLP_STREAMED_INSTANCES(extern, LGAE_ACT_ELU)
LGAE_MLP_STREAMED_INSTANCES(extern, LGAE_ACT_SIGMOID)
LGAE_MLP_STREAMED_INSTANCES(extern, LGAE_ACT_LOGSIGMOID)
LGAE_MLP_STREAMED_INSTANCES(extern, LGAE_ACT_TANH)
LGAE_MLP_STREAMED_INSTANCES(extern, LGAE_ACT_ATAN)

// nti = ceil(2C'/8): 1 for C' <= 4 output channels, 2 for C' = 5..8.  The hidden width is mlp_width * 2C' >= nin, so with
// nti = 2 every ntw from 2 to 6 is reachable.  (LGAE_MLP_INSTANCES in lgae_mlp.cuh lists the same tilings.)
template <int ACT>
static int launch_mlp_shape(MlpArgs& a, int ntw, int nti, bool bwd, cudaStream_t st) {
#define LGAE_MLP_CASE(W, I) \
    if (ntw == W && nti == I) return launch_mlp<W, I, ACT>(a, bwd, st);
    LGAE_MLP_CASE(1, 1) LGAE_MLP_CASE(2, 1) LGAE_MLP_CASE(3, 1) LGAE_MLP_CASE(4, 1)
    LGAE_MLP_CASE(5, 1) LGAE_MLP_CASE(6, 1)
    LGAE_MLP_CASE(2, 2) LGAE_MLP_CASE(3, 2) LGAE_MLP_CASE(4, 2) LGAE_MLP_CASE(5, 2) LGAE_MLP_CASE(6, 2)
    LGAE_MLP_CASE(8, 2) LGAE_MLP_CASE(9, 2)
#undef LGAE_MLP_CASE
    return LGAE_E_UNSUPPORTED;
}

// The streamed kernels' range: hidden widths 49..96 (LGAE_MLP_STREAMED_INSTANCES lists the same tilings).
static bool mlp_streamed_tiling(int ntw, int nti) { return ntw >= 7 && ntw <= 12 && nti >= 1 && nti <= 2; }

// The tilings one of the two families takes: the resident instances cover nti <= ntw <= 6 and (8, 2), (9, 2), the streamed
// kernels 7 <= ntw <= 12.  (Whether a resident instance's shared memory holds all layers at the model's depth is decided at
// launch; the streamed kernels take the ones it does not in their range.)
bool mlp_tiling_supported(const LgaeModelDesc* d, int level) {
    const int ntw = (d->mlp_width[level] + 7) / 8, nti = (2 * d->channels[level + 1] + 7) / 8;
    return nti >= 1 && nti <= 2 && ntw >= nti && ntw <= 12;
}

// Resident kernels wherever they have an instance whose shared memory holds all layers; the streamed kernels exactly where
// they do not.  Both read the same packed weights and write the same activations and partial rows, so a level may run the
// resident forward and the streamed adjoint.
template <int ACT>
static int launch_mlp_any(MlpArgs& a, int ntw, int nti, bool bwd, cudaStream_t st) {
    const int rc = launch_mlp_shape<ACT>(a, ntw, nti, bwd, st);
    if (rc != LGAE_E_UNSUPPORTED || !mlp_streamed_tiling(ntw, nti)) return rc;
#define LGAE_MLP_STREAMED_CASE(W)                                      \
    if (ntw == W)                                                      \
        return nti == 1 ? launch_mlp_streamed<W, 1, ACT>(a, bwd, st) \
                        : launch_mlp_streamed<W, 2, ACT>(a, bwd, st);
    LGAE_MLP_STREAMED_CASE(7) LGAE_MLP_STREAMED_CASE(8) LGAE_MLP_STREAMED_CASE(9)
    LGAE_MLP_STREAMED_CASE(10) LGAE_MLP_STREAMED_CASE(11) LGAE_MLP_STREAMED_CASE(12)
#undef LGAE_MLP_STREAMED_CASE
    return LGAE_E_UNSUPPORTED;
}

int run_mlp(const LgaeModelDesc* d, int level, const double* theta, const double* wpack, const double* x, int64_t rows, double* acts,
            double* y, const double* g_y, double* g_x, PartPlan* plan, bool bwd, cudaStream_t st) {
    if (!d || level < 0 || level >= d->n_levels || !d->has_mlp) return LGAE_E_BADARG;
    MlpArgs a;
    memset(&a, 0, sizeof(a));
    a.theta = theta;
    a.wpack = wpack;
    a.n_lin = d->mlp_hidden + 1;
    if (!wpack) return LGAE_E_BADARG;
    if (a.n_lin < 2 || a.n_lin > LGAE_MAX_LINEAR) return LGAE_E_UNSUPPORTED;
    for (int i = 0; i < a.n_lin; ++i) { a.off_w[i] = d->off_mlp_w[level][i]; a.off_b[i] = d->off_mlp_b[level][i]; }
    a.nin = 2 * d->channels[level + 1];
    a.width = d->mlp_width[level];
    a.x = x; a.acts = acts; a.y = y; a.rows = rows; a.g_y = g_y; a.g_x = g_x;
    a.slope = 0.01;
    if (rows <= 0) return LGAE_OK;
    if (bwd) {
        if (!plan) return LGAE_E_BADARG;
        const int grid = mlp_bwd_grid();
        int64_t w = 0;
        for (int i = 0; i < a.n_lin; ++i) {
            const int nout = i == a.n_lin - 1 ? a.nin : a.width, nink = i == 0 ? a.nin : a.width;
            a.po_w[i] = w; w += (int64_t)nout * nink;
            a.po_b[i] = w; w += nout;
        }
        const int64_t off = plan->block(grid, w);
        a.part = plan->base + off;
        a.part_stride = w;
        for (int i = 0; i < a.n_lin; ++i) {
            const int nout = i == a.n_lin - 1 ? a.nin : a.width, nink = i == 0 ? a.nin : a.width;
            if (int rc = plan->seg(a.off_w[i], off, w, a.po_w[i], (int64_t)nout * nink, grid)) return rc;
            if (int rc = plan->seg(a.off_b[i], off, w, a.po_b[i], nout, grid)) return rc;
        }
    }
    const int ntw = (a.width + 7) / 8, nti = (a.nin + 7) / 8;
    switch (d->mlp_activation) {
        case LGAE_ACT_LEAKYRELU: return launch_mlp_any<LGAE_ACT_LEAKYRELU>(a, ntw, nti, bwd, st);
        case LGAE_ACT_RELU: return launch_mlp_any<LGAE_ACT_RELU>(a, ntw, nti, bwd, st);
        case LGAE_ACT_ELU: return launch_mlp_any<LGAE_ACT_ELU>(a, ntw, nti, bwd, st);
        case LGAE_ACT_SIGMOID: return launch_mlp_any<LGAE_ACT_SIGMOID>(a, ntw, nti, bwd, st);
        case LGAE_ACT_LOGSIGMOID: return launch_mlp_any<LGAE_ACT_LOGSIGMOID>(a, ntw, nti, bwd, st);
        case LGAE_ACT_TANH: return launch_mlp_any<LGAE_ACT_TANH>(a, ntw, nti, bwd, st);
        case LGAE_ACT_ATAN: return launch_mlp_any<LGAE_ACT_ATAN>(a, ntw, nti, bwd, st);
        default: return LGAE_E_UNSUPPORTED;
    }
}

// Width (doubles) of one row of partials of the MLP adjoint.
int64_t mlp_part_width(const LgaeModelDesc* d, int level) {
    const int n_lin = d->mlp_hidden + 1, nin = 2 * d->channels[level + 1], width = d->mlp_width[level];
    int64_t w = 0;
    for (int i = 0; i < n_lin; ++i) {
        const int nout = i == n_lin - 1 ? nin : width, nink = i == 0 ? nin : width;
        w += (int64_t)nout * nink + nout;
    }
    return w;
}

int mlp_padded_width(const LgaeModelDesc* d, int level) { return 8 * ((d->mlp_width[level] + 7) / 8); }

}  // namespace lgae
