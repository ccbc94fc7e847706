// extern "C" entry points of liblgae_b200.so (declared in include/lgae_b200.h): argument checks, workspace
// geometry, and the launch sequences of the whole-model forward / backward passes.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "lgae_common.cuh"

namespace lgae {

// ---- implemented in the other translation units -------------------------------------------------------------
int run_level_fwd(const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y, const uint8_t* node_mask, int batch,
                  const double* s_in, const double* v_in, double* sums, double* r_save, double* s_pre, double* v_out, cudaStream_t st);
int run_md3_level_fwd(const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y, const uint8_t* node_mask, int batch,
                      const double* s_in, const double* v_in, const double* h_in, double* nbr, double* s_pre, double* v_out, double* h_out,
                      cudaStream_t st);
int md3_level_check(const LgaeModelDesc* d);
int64_t md3_nbr_doubles(const LgaeModelDesc* d, int level, int64_t batch);
int run_level_bwd(const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y, const uint8_t* node_mask, int batch,
                  const double* s_in, const double* v_in, const double* sums, const double* r_save, double* g_r, const double* g_s_pre,
                  const double* g_v_out, double* g_s_in, double* g_v_in, double* g_y, PartPlan* plan, cudaStream_t st,
                  double* g_a = nullptr);
int pgrad_check(const LgaeModelDesc* d);
int run_pgrad_level(const LgaeModelDesc* d, int level, const double* theta, const double* p, const uint8_t* node_mask, int batch,
                    const double* s_in, const double* v_in, const double* gA, double* gp, cudaStream_t st);
int run_pgrad_input(const LgaeModelDesc* d, const double* theta, const double* p, int batch, const double* gS, const double* gV,
                    const double* gp, double scale, double* g_p4, cudaStream_t st);
int run_chamfer_target_grad(const double* recon, const double* target, int B, int N, int M, int mode, const double* g_loss,
                            double* g_target, cudaStream_t st);
int run_normalize_bwd(const double* p4, int B, int N, const double* g_out, const double* g_factor, double* g_p4, cudaStream_t st);
int run_radial_fwd_all(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int batch,
                       double* const* r, double* nrm, cudaStream_t st);
int run_radial_fwd(const LgaeModelDesc* d, int level, const double* theta, const double* p4, const uint8_t* node_mask, int batch,
                   double* r, double* nrm, cudaStream_t st);
int run_radial_bwd(const LgaeModelDesc* d, int level, const double* theta, const double* p4, const uint8_t* node_mask, int batch,
                   const double* g_r, const double* nrm, PartPlan* plan, cudaStream_t st);
int run_level_bwd_tiled(const LgaeModelDesc* d, int level, const double* theta, const double* p_or_y, const uint8_t* node_mask, int batch,
                        const double* s_in, const double* v_in, const double* sums, double* gA, double* g_r, const double* g_s_pre,
                        const double* g_v_out, double* g_s_in, double* g_v_in, double* g_y, PartPlan* plan, cudaStream_t st);
int level_bwd_tiled_check(const LgaeModelDesc* d);
int64_t level_tiled_part_doubles(const LgaeModelDesc* d, int level, int batch);
int glue_bwd_check(const LgaeModelDesc* d);
int train_step_glue_check(const LgaeModelDesc* de, const LgaeModelDesc* dd);
int64_t radial_nrm_stride(int n);
int radial_grid();
int radial_tiled_grid();
int64_t radial_part_width(const LgaeModelDesc* d, int level);
int level_bwd_grid(int batch);
int64_t level_part_width(const LgaeModelDesc* d, int level);
int run_mlp(const LgaeModelDesc* d, int level, const double* theta, const double* wpack, const double* x, int64_t rows, double* acts,
            double* y, const double* g_y, double* g_x, PartPlan* plan, bool bwd, cudaStream_t st);
int64_t mlp_pack_doubles(const LgaeModelDesc* d, int level);
int run_mlp_pack(const LgaeModelDesc* d, const double* theta, double* out, const int64_t* out_off, cudaStream_t st,
                 const LgaeModelDesc* d2 = nullptr, const double* theta2 = nullptr, double* out2 = nullptr, const int64_t* out_off2 = nullptr);
int mlp_padded_width(const LgaeModelDesc* d, int level);
int64_t mlp_part_width(const LgaeModelDesc* d, int level);
int mlp_bwd_grid();
bool mlp_tiling_supported(const LgaeModelDesc* d, int level);
int run_enc_input(const LgaeModelDesc* d, const double* theta, const double* p4, int B, double* mass, double* S, double* V, cudaStream_t st);
int run_enc_input_bwd(const LgaeModelDesc* d, const double* p4, const double* mass, int B, const double* gS, const double* gV, PartPlan* plan, cudaStream_t st);
int run_enc_latent(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V, double* lat00, double* lat11, int32_t* sel, cudaStream_t st, int parts = 3);
int run_enc_latent_bwd(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V, const int32_t* sel,
                       const double* g_lat00, const double* g_lat11, double* gS, double* gV, PartPlan* plan, cudaStream_t st);
int run_dec_input(const LgaeModelDesc* d, const double* theta, int B, const double* lat11, double* y, double* S, double* V, cudaStream_t st);
int run_dec_input_bwd(const LgaeModelDesc* d, const double* theta, int B, const double* lat11, double* y, const double* gS, const double* gV,
                      const double* gy, double* g_lat11, PartPlan* plan, cudaStream_t st);
int run_dec_output(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V, double* recon, double* gen00, cudaStream_t st);
int run_dec_output_bwd(const LgaeModelDesc* d, const double* theta, int B, const double* S, const double* V, const double* g_recon,
                       const double* g_gen00, double* gS, double* gV, PartPlan* plan, cudaStream_t st);
int run_latent_bridge_bwd(const LgaeModelDesc* dd, const double* theta_d, const LgaeModelDesc* de, const double* theta_e, int B,
                          const double* lat11, double* y, const double* gS_d, const double* gV_d, const double* gy, double* g_lat11,
                          const double* S, const double* V, const int32_t* sel, double* gS_e, double* gV_e, PartPlan* plan_d,
                          PartPlan* plan_e, cudaStream_t st);
int run_reduce_plan(PartPlan* plan, int64_t n_params, double* gtheta, const double* theta, double lambda, double* loss, cudaStream_t st);
int reduce_scratch_doubles();
int run_latent_bridge(const LgaeModelDesc* de, const double* theta_e, const LgaeModelDesc* dd, const double* theta_d, int B, const double* S,
                      const double* V, double* lat00, double* lat11, int32_t* sel, double* y, double* S0, double* V0, cudaStream_t st, int parts = 3);
int run_dec_tail(const LgaeModelDesc* d, const double* theta, int B, int M, const double* V, const double* target, double* recon,
                 double* g_recon, double* gV, double* jet_loss, double* loss, unsigned int* counter, int mode, PartPlan* plan, cudaStream_t st);
int run_grad_init2(const double* theta_a, int64_t na, const double* theta_b, int64_t nb, int64_t off_b, double* gtheta, double lambda,
                   double* psum, cudaStream_t st);
int run_reduce_segs(PartPlan* plan, int64_t n_params, double* gtheta, const double* psum, double lambda, double* loss, cudaStream_t st);
int run_reduce_plan2(PartPlan* plan, const double* theta_a, int64_t na, const double* theta_b, int64_t nb, int64_t off_b, double* gtheta,
                     double lambda, double* loss, cudaStream_t st);
int64_t glue_part_doubles(const LgaeModelDesc* d, int batch);
int run_chamfer(const double* recon, const double* target, int B, int N, int M, double* loss, double* jet_loss, const double* g_loss,
                double* g_recon, int mode, cudaStream_t st);
int run_normalize(const double* p4, int B, int N, double* out, double* factor, cudaStream_t st);
int run_norm_input(const LgaeModelDesc* d, const double* theta, const double* p4, int B, double* out, double* factor, double* mass, double* S,
                   double* V, cudaStream_t st);
int run_l1(const double* theta, int64_t n, double lambda, double* out, double* gtheta, cudaStream_t st);
int run_scale(const double* in, int64_t n, double s, double* out, cudaStream_t st);
int run_scores(const double* recon, const double* target, const double* factor, int B, int N, int mode, double* out, cudaStream_t st);

// ---- bookkeeping ------------------------------------------------------------------------------------------------
#define LGAE_MAX_DEVICES 64
static std::atomic<int64_t> g_launches{0};
static thread_local char g_cuda_error[512] = "";   // per calling thread: lgae_last_cuda_error() reports the caller's own failure

void count_launch(int n) { g_launches += n; }

// ---- optional per-kernel timing ---------------------------------------------------------------------------------
struct TimedLaunch { const char* name; cudaEvent_t a, b; };
static std::mutex g_timing_mu;
static bool g_timing_on = false;
static std::vector<TimedLaunch> g_timed;

LaunchScope::LaunchScope(const char* name_, cudaStream_t st_) : name(name_), st(st_), ev0(nullptr) {
    if (!g_timing_on) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) { cudaGetLastError(); return; }
    cudaEventRecord(e, st);
    ev0 = (void*)e;
}
LaunchScope::~LaunchScope() {
    g_launches += 1;
    if (!ev0) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) { cudaGetLastError(); cudaEventDestroy((cudaEvent_t)ev0); return; }
    cudaEventRecord(e, st);
    std::lock_guard<std::mutex> lock(g_timing_mu);
    g_timed.push_back({name, (cudaEvent_t)ev0, e});
}
int check_launch(const char* what) {
    const cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) return LGAE_OK;
    snprintf(g_cuda_error, sizeof(g_cuda_error), "%s: %s", what, cudaGetErrorString(e));
    return LGAE_E_CUDA;
}
// The opt-in applies to the current device's copy of the function: the cache is keyed by (device, kernel).
int ensure_smem(const void* kernel, size_t bytes) {
    static std::mutex mu;
    static std::unordered_map<const void*, size_t> seen[LGAE_MAX_DEVICES];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return check_launch("cudaGetDevice");
    const bool cached = dev >= 0 && dev < LGAE_MAX_DEVICES;
    std::lock_guard<std::mutex> lock(mu);
    if (cached) {
        auto it = seen[dev].find(kernel);
        if (it != seen[dev].end() && it->second >= bytes) return LGAE_OK;
    }
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return check_launch("cudaFuncSetAttribute");
    if (cached) seen[dev][kernel] = bytes;
    return LGAE_OK;
}
int sm_count() {
    static std::atomic<int> per_dev[LGAE_MAX_DEVICES];
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 148; }
    const bool cached = dev >= 0 && dev < LGAE_MAX_DEVICES;
    if (cached && (n = per_dev[dev].load()) > 0) return n;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return 148;
    }
    if (cached) per_dev[dev].store(n);
    return n;
}

// Auxiliary stream of the training step for its small, independent kernels (weight packing and gradient init at the start,
// the encoder-input adjoint next to the last radial adjoint): they become parallel branches of the step's graph instead of
// ~10 us links of its critical path.  One per device, created on first use; NULL if that fails (lgae_last_cuda_error says why),
// and the next call tries again.
struct AuxStream {
    cudaStream_t s = nullptr;
    cudaEvent_t fork[4] = {}, join[5] = {};
};
static AuxStream* aux_stream() {
    static std::unordered_map<int, AuxStream*> per_dev;
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { check_launch("cudaGetDevice"); return nullptr; }
    auto it = per_dev.find(dev);
    if (it != per_dev.end()) return it->second;
    AuxStream a;
    bool ok = cudaStreamCreateWithFlags(&a.s, cudaStreamNonBlocking) == cudaSuccess;
    for (cudaEvent_t& e : a.fork) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    for (cudaEvent_t& e : a.join) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        check_launch("auxiliary stream");
        for (cudaEvent_t e : a.fork) if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : a.join) if (e) cudaEventDestroy(e);
        if (a.s) cudaStreamDestroy(a.s);
        return nullptr;
    }
    return per_dev[dev] = new AuxStream(a);
}
static std::mutex g_aux_mu;   // serialises the training steps that share the auxiliary stream's events
#define LGAE_CUDA_TRY(expr, what)                                   \
    do {                                                            \
        if ((expr) != cudaSuccess) return check_launch(what);       \
    } while (0)

// ---- workspace layout -----------------------------------------------------------------------------------------------
struct Layout {
    int64_t S[LGAE_MAX_LEVELS + 1], V[LGAE_MAX_LEVELS + 1];
    int64_t sums[LGAE_MAX_LEVELS], spre[LGAE_MAX_LEVELS], acts[LGAE_MAX_LEVELS], rsave[LGAE_MAX_LEVELS], wpack[LGAE_MAX_LEVELS];
    int64_t y, mass, gS[2], gV[2], gSpre, gy, gr[LGAE_MAX_LEVELS], nrm, pscaled, total;
    int64_t H[LGAE_MAX_LEVELS + 1], nbr;   // maxdim 3 only: (2,0) | (0,2) | (2,2) parts of the nodes, neighbour sums of one level
};
static bool has_input_scale(const LgaeModelDesc* d) { return !d->is_decoder && d->input_scale != 0.0 && d->input_scale != 1.0; }
static int max_channels(const LgaeModelDesc* d) {
    int m = 1;
    for (int l = 0; l <= d->n_levels; ++l) m = d->channels[l] > m ? d->channels[l] : m;
    return m;
}
static bool is_md3(const LgaeModelDesc* d) { return d->maxdim == 3; }
// maxdim 3 (forward only): [y | mass | S, V, H per level | spre, acts, wpack per level | nbr | pscaled]; -1 for what it lacks
static Layout layout_md3(const LgaeModelDesc* d, int64_t B) {
    Layout L;
    memset(&L, 0xff, sizeof(L));
    const int64_t nodes = B * d->n_particles;
    int64_t o = 0;
    auto take = [&](int64_t n) { const int64_t r = o; o += (n + 3) & ~int64_t(3); return r; };   // 32-byte granules
    L.y = take(nodes * 8);
    L.mass = take(nodes);
    for (int l = 0; l <= d->n_levels; ++l) {
        L.S[l] = take(nodes * d->channels[l] * 2);
        L.V[l] = take(nodes * d->channels[l] * 8);
        L.H[l] = l > 0 ? take(nodes * d->channels[l] * 30) : -1;   // level 0 holds (0,0) and (1,1) only
    }
    int64_t nbr = 0;
    for (int l = 0; l < d->n_levels; ++l) {
        L.spre[l] = d->has_mlp ? take(nodes * d->channels[l + 1] * 2) : L.S[l + 1];
        L.acts[l] = d->has_mlp ? take((int64_t)d->mlp_hidden * nodes * mlp_padded_width(d, l)) : 0;
        L.wpack[l] = take(mlp_pack_doubles(d, l));
        const int64_t n = md3_nbr_doubles(d, l, B);
        nbr = n > nbr ? n : nbr;
    }
    L.nbr = take(nbr);
    L.pscaled = has_input_scale(d) ? take(nodes * 4) : -1;
    L.total = o;
    return L;
}
static Layout layout(const LgaeModelDesc* d, int64_t B) {
    if (is_md3(d)) return layout_md3(d, B);
    Layout L;
    const int64_t nodes = B * d->n_particles;
    int64_t o = 0;
    auto take = [&](int64_t n) { const int64_t r = o; o += (n + 3) & ~int64_t(3); return r; };   // 32-byte granules
    L.y = take(nodes * 8);
    L.mass = take(nodes);
    for (int l = 0; l <= d->n_levels; ++l) {
        L.S[l] = take(nodes * d->channels[l] * 2);
        L.V[l] = take(nodes * d->channels[l] * 8);
    }
    for (int l = 0; l < d->n_levels; ++l) {
        L.sums[l] = take(nodes * d->channels[l] * 20);
        L.spre[l] = d->has_mlp ? take(nodes * d->channels[l + 1] * 2) : L.S[l + 1];
        L.acts[l] = d->has_mlp ? take((int64_t)d->mlp_hidden * nodes * mlp_padded_width(d, l)) : 0;
        L.wpack[l] = take(mlp_pack_doubles(d, l));
        // encoder, N <= 32: the radial weights R_ij[c] of every level, kept for the adjoint
        L.rsave[l] = (!d->is_decoder && d->n_particles <= 32) ? take(nodes * d->channels[l] * 128) : -1;
    }
    const int cm = max_channels(d);
    for (int k = 0; k < 2; ++k) { L.gS[k] = take(nodes * cm * 2); L.gV[k] = take(nodes * cm * 8); }
    L.gSpre = take(nodes * cm * 2);
    L.gy = take(nodes * 8);
    // encoder, N <= 32: dL/dR of the ordered pairs, one buffer per level
    for (int l = 0; l < LGAE_MAX_LEVELS; ++l)
        L.gr[l] = (!d->is_decoder && d->n_particles <= 32 && l < d->n_levels) ? take(nodes * d->channels[l] * 128) : -1;
    // encoder, N <= 32: norms of the unordered pairs (NaN = masked), written by the radial forward
    L.nrm = (!d->is_decoder && d->n_particles <= 32) ? take(B * radial_nrm_stride(d->n_particles)) : -1;
    // encoder with an input scale: the scaled momenta every kernel of the model reads
    L.pscaled = has_input_scale(d) ? take(nodes * 4) : -1;
    L.total = o;
    for (int l = 0; l <= LGAE_MAX_LEVELS; ++l) L.H[l] = -1;
    L.nbr = -1;
    return L;
}

static int check_desc(const LgaeModelDesc* d) {
    if (!d) return LGAE_E_BADARG;
    if (d->n_levels < 1 || d->n_levels > LGAE_MAX_LEVELS || d->n_particles < 1 || d->n_params <= 0) return LGAE_E_BADARG;
    for (int l = 0; l <= d->n_levels; ++l)
        if (d->channels[l] < 1 || d->channels[l] > LGAE_MAX_CHANNELS) return LGAE_E_UNSUPPORTED;
    if (d->has_mlp && (d->mlp_hidden < 1 || d->mlp_hidden + 1 > LGAE_MAX_LINEAR)) return LGAE_E_UNSUPPORTED;
    if (d->has_mlp && (d->mlp_activation < 0 || d->mlp_activation >= LGAE_ACT_COUNT)) return LGAE_E_UNSUPPORTED;
    for (int l = 0; d->has_mlp && l < d->n_levels; ++l)
        if (!mlp_tiling_supported(d, l)) return LGAE_E_UNSUPPORTED;   // hidden width above 96: no MLP kernel takes it
    if (d->maxdim != 0 && d->maxdim != 2 && d->maxdim != 3) return LGAE_E_UNSUPPORTED;
    if (d->maxdim == 3 && md3_level_check(d) != LGAE_OK) return LGAE_E_UNSUPPORTED;
    return LGAE_OK;
}

// Scratch of the tiled adjoint (lgae_backward_tiled_scratch_doubles): [gA | g_r | partial rows + reduce scratch].
//   gA  (B,N,Cmax,10) complex: adjoints of the neighbour sums of the current level
//   g_r (B,nib,N,Cmax,32,4), encoder only: dL/dR of the current level's ordered pairs, the only O(N^2) piece
struct TiledScratch {
    int64_t gA, gr, part, total;
};
static TiledScratch tiled_scratch(const LgaeModelDesc* d, int64_t B) {
    TiledScratch T;
    const int64_t N = d->n_particles, cm = max_channels(d), nib = (N + 31) / 32;
    T.gA = 0;
    T.gr = T.gA + ((B * N * cm * 20 + 3) & ~int64_t(3));
    T.part = T.gr + (d->is_decoder ? 0 : B * nib * N * cm * 128);
    int64_t n = glue_part_doubles(d, (int)B) + reduce_scratch_doubles();
    for (int l = 0; l < d->n_levels; ++l) {
        n += level_tiled_part_doubles(d, l, (int)B);
        if (!d->is_decoder) n += (int64_t)radial_tiled_grid() * radial_part_width(d, l);
        if (d->has_mlp) n += (int64_t)mlp_bwd_grid() * mlp_part_width(d, l);
    }
    T.total = T.part + n;
    return T;
}
static int tiled_check(const LgaeModelDesc* d) {
    if (int rc = level_bwd_tiled_check(d)) return rc;
    return glue_bwd_check(d);
}
// The tiled adjoint's two large regions inside a caller's scratch; gA == nullptr selects the per-lane adjoint.
struct TiledBufs {
    double* gA = nullptr;
    double* gr = nullptr;   // encoder only
};

// Scratch of the encoder's input gradient (lgae_encoder_input_grad_scratch_doubles): [gp | gA]
//   gp (B,N,4): dL/dp of the levels, accumulated in level order
//   gA (B,N,Cmax,10) complex, N <= 32 only: the per-lane level adjoint's neighbour-sum adjoints of the current level (the tiled
//      adjoint keeps them in its own scratch)
struct InputGradScratch {
    int64_t gp, gA, total;
};
static InputGradScratch input_grad_scratch(const LgaeModelDesc* d, int64_t B) {
    InputGradScratch G;
    const int64_t nodes = B * d->n_particles;
    G.gp = 0;
    G.gA = (nodes * 4 + 3) & ~int64_t(3);
    G.total = G.gA + (d->n_particles <= 32 ? nodes * max_channels(d) * 20 : 0);
    return G;
}
// The input gradient requested from the encoder adjoint; g_p4 == nullptr: none (the adjoint's launches are unchanged).
struct InputGrad {
    double* g_p4 = nullptr;      // (B,N,4) out, with respect to the caller's unscaled p4
    double* scratch = nullptr;   // input_grad_scratch
};

// Scratch of the tiled training step (lgae_train_step_tiled_scratch_doubles):
//   [gA | g_r | decoder rows, encoder rows | reduce scratch (psum) | dec_tail counter]
// gA is sized for the larger model and used by the decoder adjoint, then by the encoder adjoint (same stream, in that order).
// The rows region holds both models' tiled partial rows (each with its own glue rows and reduce scratch, as in
// lgae_backward_tiled_scratch_doubles) and the dec_tail rows, like lgae_train_step_partials_doubles does for the per-lane step;
// the last reduce scratch takes the L1 partial sums of the gradient init, the last double the dec_tail completion counter.
struct StepScratch {
    int64_t gA, gr, part, total;
};
static StepScratch step_scratch(const LgaeModelDesc* enc, const LgaeModelDesc* dec, int64_t B) {
    const TiledScratch e = tiled_scratch(enc, B), d = tiled_scratch(dec, B);
    const int64_t ga_e = e.gr - e.gA, ga_d = d.gr - d.gA;
    StepScratch S;
    S.gA = 0;
    S.gr = ga_e > ga_d ? ga_e : ga_d;
    S.part = S.gr + (e.part - e.gr);
    S.total = S.part + (e.total - e.part) + (d.total - d.part) + B * 4 * dec->channels[dec->n_levels] + 1;
    return S;
}

// The momenta the encoder kernels read: p4 itself, or (input_scale != 1) the scaled copy kept in the workspace, written here
// when `write` (forward) and re-used by the adjoint.
static const double* scaled_input(const LgaeModelDesc* d, const double* p4, int64_t batch, double* ws, bool write, cudaStream_t st, int* rc) {
    *rc = LGAE_OK;
    if (!has_input_scale(d) || batch <= 0) return p4;
    double* out = ws + layout(d, batch).pscaled;
    if (write) *rc = run_scale(p4, batch * d->n_particles * 4, d->input_scale, out, st);
    return out;
}

#define LGAE_TRY(expr)            \
    do {                          \
        const int rc_ = (expr);   \
        if (rc_ != LGAE_OK) return rc_; \
    } while (0)

}  // namespace lgae

using namespace lgae;

extern "C" {

int lgae_version(void) { return 100; }

const char* lgae_error_string(int code) {
    switch (code) {
        case LGAE_OK: return "ok";
        case LGAE_E_BADARG: return "bad argument (null pointer, negative size or inconsistent descriptor)";
        case LGAE_E_UNSUPPORTED: return "configuration not supported by the fused sm_100a path";
        case LGAE_E_CUDA: return "CUDA error (see lgae_last_cuda_error)";
        case LGAE_E_NODEVICE: return "no CUDA device";
        default: return "unknown error";
    }
}
const char* lgae_last_cuda_error(void) { return g_cuda_error; }
int lgae_device_sm_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return LGAE_E_NODEVICE; }
    return sm_count();
}
int64_t lgae_launch_count(void) { return g_launches.load(); }

void lgae_timing_enable(int32_t on) {
    std::lock_guard<std::mutex> lock(g_timing_mu);
    g_timing_on = on != 0;
}
// Synchronises the device, then writes one line per kernel name "name count total_ms\n" into buf (NUL-terminated, at most
// cap bytes) and clears the records.  Returns the number of distinct names, or a negative error code.
int lgae_timing_report(char* buf, int32_t cap) {
    if (!buf || cap < 1) return LGAE_E_BADARG;
    if (cudaDeviceSynchronize() != cudaSuccess) return check_launch("timing sync");
    std::lock_guard<std::mutex> lock(g_timing_mu);
    std::vector<std::string> order;
    std::unordered_map<std::string, std::pair<int, double>> agg;
    for (auto& t : g_timed) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, t.a, t.b);
        cudaEventDestroy(t.a);
        cudaEventDestroy(t.b);
        auto it = agg.find(t.name);
        if (it == agg.end()) { order.push_back(t.name); agg[t.name] = {1, (double)ms}; }
        else { it->second.first += 1; it->second.second += ms; }
    }
    g_timed.clear();
    std::string out;
    for (auto& n : order) {
        char line[256];
        snprintf(line, sizeof(line), "%s %d %.6f\n", n.c_str(), agg[n].first, agg[n].second);
        out += line;
    }
    if ((int)out.size() + 1 > cap) return LGAE_E_BADARG;
    memcpy(buf, out.c_str(), out.size() + 1);
    return (int)order.size();
}

int64_t lgae_workspace_doubles(const LgaeModelDesc* d, int32_t batch) {
    if (check_desc(d) != LGAE_OK || batch < 0) return -1;
    return layout(d, batch).total;
}
int64_t lgae_workspace_offset(const LgaeModelDesc* d, int32_t batch, int32_t kind, int32_t level) {
    if (check_desc(d) != LGAE_OK || batch < 0 || level < 0 || level > d->n_levels) return -1;
    const Layout L = layout(d, batch);
    switch (kind) {
        case 0: return L.S[level];
        case 1: return L.V[level];
        case 2: return level < d->n_levels ? L.spre[level] : -1;
        case 3: return L.y;
        case 4: return level < d->n_levels ? L.sums[level] : -1;
        case 5: return L.mass;
        case 6: return level < d->n_levels ? L.acts[level] : -1;
        case 7: return level < d->n_levels ? L.rsave[level] : -1;
        case 8: return level < d->n_levels ? L.gr[level] : -1;
        case 9: return L.H[level];
        default: return -1;
    }
}
int64_t lgae_partials_doubles(const LgaeModelDesc* d, int32_t batch) {
    if (check_desc(d) != LGAE_OK || batch < 0) return -1;
    if (is_md3(d)) return LGAE_E_UNSUPPORTED;   // maxdim 3: forward only
    int64_t n = glue_part_doubles(d, batch) + reduce_scratch_doubles();
    for (int l = 0; l < d->n_levels; ++l) {
        n += (int64_t)level_bwd_grid(batch) * level_part_width(d, l);
        if (!d->is_decoder) n += (int64_t)radial_grid() * radial_part_width(d, l);
        if (d->has_mlp) n += (int64_t)mlp_bwd_grid() * mlp_part_width(d, l);
    }
    return n;
}
int64_t lgae_backward_tiled_scratch_doubles(const LgaeModelDesc* d, int32_t batch) {
    const int rc = check_desc(d);
    if (rc == LGAE_E_BADARG || batch < 0) return -1;
    if (rc != LGAE_OK || is_md3(d) || tiled_check(d) != LGAE_OK) return LGAE_E_UNSUPPORTED;
    return tiled_scratch(d, batch).total;
}
int64_t lgae_train_step_tiled_scratch_doubles(const LgaeModelDesc* enc, const LgaeModelDesc* dec, int32_t batch) {
    const int re = check_desc(enc), rd = check_desc(dec);
    if (re == LGAE_E_BADARG || rd == LGAE_E_BADARG || batch < 0 || enc->is_decoder || !dec->is_decoder) return -1;
    if (re != LGAE_OK || rd != LGAE_OK || is_md3(enc) || is_md3(dec) || tiled_check(enc) != LGAE_OK || tiled_check(dec) != LGAE_OK)
        return LGAE_E_UNSUPPORTED;
    if (const int rc = train_step_glue_check(enc, dec)) return rc == LGAE_E_BADARG ? -1 : LGAE_E_UNSUPPORTED;
    return step_scratch(enc, dec, batch).total;
}

}  // extern "C"

// Launch sequence of LGNEncoder.forward; `pack` = also pack the MLP weights (a caller that runs both models packs them once).
static int enc_forward_launch(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                              double* ws, double* lat00, double* lat11, int32_t* sel, bool pack, cudaStream_t st, bool with_latent = true,
                              bool with_input = true, cudaEvent_t pack_done = nullptr, bool skip_last_mlp = false) {
    const Layout L = layout(d, batch);
    const int64_t rows = (int64_t)batch * d->n_particles;
    if (pack) LGAE_TRY(run_mlp_pack(d, theta, ws, L.wpack, st));
    if (with_input) LGAE_TRY(run_enc_input(d, theta, p4, batch, ws + L.mass, ws + L.S[0], ws + L.V[0], st));
    // the radial weights of all levels in one launch ahead of the level chain (0.8442 -> 0.8413 ms per step against one launch
    // per level); level by level when the levels' MMA tilings differ
    bool merged = false;
    if (L.rsave[0] >= 0) {
        double* rs[LGAE_MAX_LEVELS];
        for (int l = 0; l < d->n_levels; ++l) rs[l] = ws + L.rsave[l];
        const int rc = run_radial_fwd_all(d, theta, p4, node_mask, batch, rs, ws + L.nrm, st);
        if (rc == LGAE_OK) merged = true;
        else if (rc != LGAE_E_UNSUPPORTED) return rc;
    }
    for (int l = 0; l < d->n_levels; ++l) {
        if (L.rsave[l] >= 0 && !merged)
            LGAE_TRY(run_radial_fwd(d, l, theta, p4, node_mask, batch, ws + L.rsave[l], ws + L.nrm, st));
        LGAE_TRY(run_level_fwd(d, l, theta, p4, node_mask, batch, ws + L.S[l], ws + L.V[l], ws + L.sums[l],
                               L.rsave[l] >= 0 ? ws + L.rsave[l] : nullptr, ws + L.spre[l], ws + L.V[l + 1], st));
        if (l == 0 && pack_done) LGAE_CUDA_TRY(cudaStreamWaitEvent(st, pack_done, 0), "pack wait");   // packed on another stream
        if (d->has_mlp && !(skip_last_mlp && l == d->n_levels - 1))
            LGAE_TRY(run_mlp(d, l, theta, ws + L.wpack[l], ws + L.spre[l], rows, ws + L.acts[l], ws + L.S[l + 1], nullptr, nullptr, nullptr, false, st));
    }
    if (!with_latent) return LGAE_OK;   // the caller runs the fused latent bridge
    return run_enc_latent(d, theta, batch, ws + L.S[d->n_levels], ws + L.V[d->n_levels], lat00, lat11, sel, st);
}

// Launch sequence of the encoder adjoint; appends its blocks / segments to `plan` (no reduce).
static int enc_backward_launch(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                               double* ws, const int32_t* sel, const double* g_lat00, const double* g_lat11, PartPlan& plan,
                               cudaStream_t st, bool with_latent = true, AuxStream* aux = nullptr, TiledBufs tiled = {},
                               InputGrad ig = {}) {
    if (batch > 0) {
        const Layout L = layout(d, batch);
        const int64_t rows = (int64_t)batch * d->n_particles;
        const int nl = d->n_levels;
        int cur = 0;
        double* gp = nullptr;   // input gradient: dL/dp of the levels
        double* ig_gA = nullptr;
        if (ig.g_p4) {
            const InputGradScratch G = input_grad_scratch(d, batch);
            gp = ig.scratch + G.gp;
            ig_gA = tiled.gA ? tiled.gA : ig.scratch + G.gA;
            if (cudaMemsetAsync(gp, 0, (size_t)rows * 4 * sizeof(double), st) != cudaSuccess) return check_launch("memset gp");
        }
        if (with_latent)   // otherwise the fused bridge adjoint already left dL/dS, dL/dV of the last level in gS[0], gV[0]
            LGAE_TRY(run_enc_latent_bwd(d, theta, batch, ws + L.S[nl], ws + L.V[nl], sel, g_lat00, g_lat11, ws + L.gS[cur], ws + L.gV[cur], &plan, st));
        // The scalar features of the last level only reach the latent scalars: without a gradient on those the
        // whole last-level MLP is dead in the backward pass (SURVEY.md section 8(a), "dead-in-training sub-paths").
        bool gs_zero = g_lat00 == nullptr;
        for (int l = nl - 1; l >= 0; --l) {
            const double* g_spre = nullptr;
            if (!gs_zero) {
                if (d->has_mlp) {
                    LGAE_TRY(run_mlp(d, l, theta, ws + L.wpack[l], ws + L.spre[l], rows, ws + L.acts[l], nullptr, ws + L.gS[cur], ws + L.gSpre, &plan, true, st));
                    g_spre = ws + L.gSpre;
                } else {
                    g_spre = ws + L.gS[cur];
                }
            }
            if (tiled.gA) {   // tiled adjoint: radial weights re-evaluated, dL/dR of every level in one scratch buffer
                LGAE_TRY(run_level_bwd_tiled(d, l, theta, p4, node_mask, batch, ws + L.S[l], ws + L.V[l], ws + L.sums[l], tiled.gA,
                                             tiled.gr, g_spre, ws + L.gV[cur], ws + L.gS[cur ^ 1], ws + L.gV[cur ^ 1], nullptr, &plan, st));
            } else {
                if (L.rsave[l] < 0 || L.gr[l] < 0) return LGAE_E_UNSUPPORTED;
                LGAE_TRY(run_level_bwd(d, l, theta, p4, node_mask, batch, ws + L.S[l], ws + L.V[l], ws + L.sums[l], ws + L.rsave[l],
                                       ws + L.gr[l], g_spre, ws + L.gV[cur], ws + L.gS[cur ^ 1], ws + L.gV[cur ^ 1], nullptr, &plan, st,
                                       ig_gA));
            }
            if (gp)   // before the next level's adjoint overwrites gA
                LGAE_TRY(run_pgrad_level(d, l, theta, p4, node_mask, batch, ws + L.S[l], ws + L.V[l], ig_gA, gp, st));
            if (aux && l == 0) {
                // the input-map adjoint (small) runs next to the last radial adjoint; both only feed the final reduce
                LGAE_CUDA_TRY(cudaEventRecord(aux->fork[1], st), "aux fork");
                LGAE_CUDA_TRY(cudaStreamWaitEvent(aux->s, aux->fork[1], 0), "aux fork wait");
                LGAE_TRY(run_enc_input_bwd(d, p4, ws + L.mass, batch, ws + L.gS[cur ^ 1], ws + L.gV[cur ^ 1], &plan, aux->s));
                LGAE_CUDA_TRY(cudaEventRecord(aux->join[2], aux->s), "aux join");
            }
            if (tiled.gA)
                LGAE_TRY(run_radial_bwd(d, l, theta, p4, node_mask, batch, tiled.gr, nullptr, &plan, st));
            else
                LGAE_TRY(run_radial_bwd(d, l, theta, p4, node_mask, batch, ws + L.gr[l], ws + L.nrm, &plan, st));
            cur ^= 1;
            gs_zero = false;
        }
        if (aux)
            LGAE_CUDA_TRY(cudaStreamWaitEvent(st, aux->join[2], 0), "aux join wait");
        else
            LGAE_TRY(run_enc_input_bwd(d, p4, ws + L.mass, batch, ws + L.gS[cur], ws + L.gV[cur], &plan, st));
        if (gp)
            LGAE_TRY(run_pgrad_input(d, theta, p4, batch, ws + L.gS[cur], ws + L.gV[cur], gp, has_input_scale(d) ? d->input_scale : 1.0,
                                     ig.g_p4, st));
    }
    return LGAE_OK;
}

// LGAE_KEEP_DEAD_MLP=1 also runs the decoder's last-level scalar MLP when no result of the entry point depends on its output.
static bool keep_dead_mlp() {
    static const bool keep = [] { const char* e = getenv("LGAE_KEEP_DEAD_MLP"); return e && e[0] == '1'; }();
    return keep;
}
static int dec_forward_launch(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch, double* ws, double* recon,
                              double* gen00, bool pack, cudaStream_t st, bool with_output = true, bool with_input = true,
                              bool scalars_unused = false) {
    const Layout L = layout(d, batch);
    const int64_t rows = (int64_t)batch * d->n_particles;
    if (pack) LGAE_TRY(run_mlp_pack(d, theta, ws, L.wpack, st));
    if (with_input) LGAE_TRY(run_dec_input(d, theta, batch, lat11, ws + L.y, ws + L.S[0], ws + L.V[0], st));
    for (int l = 0; l < d->n_levels; ++l) {
        LGAE_TRY(run_level_fwd(d, l, theta, ws + L.y, nullptr, batch, ws + L.S[l], ws + L.V[l], ws + L.sums[l], nullptr, ws + L.spre[l],
                               ws + L.V[l + 1], st));
        // scalars_unused: nothing reads the output scalars of the last level (the training step's loss only sees the 4-vectors,
        // lgn_decoder.py:305-345 + get_real; SURVEY.md section 8(a) "dead-in-training sub-paths"), so its MLP is not run
        if (d->has_mlp && !(scalars_unused && l == d->n_levels - 1))
            LGAE_TRY(run_mlp(d, l, theta, ws + L.wpack[l], ws + L.spre[l], rows, ws + L.acts[l], ws + L.S[l + 1], nullptr, nullptr, nullptr, false, st));
    }
    if (!with_output) return LGAE_OK;   // the caller runs the fused tail (reconstruction + loss + adjoint of the output map)
    return run_dec_output(d, theta, batch, ws + L.S[d->n_levels], ws + L.V[d->n_levels], recon, gen00, st);
}

static int dec_backward_launch(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch, double* ws,
                               const double* g_recon, const double* g_gen00, double* g_lat11, PartPlan& plan, cudaStream_t st,
                               bool with_output = true, bool with_input = true, double* tiled_gA = nullptr) {
    if (batch > 0) {
        const Layout L = layout(d, batch);
        const int64_t rows = (int64_t)batch * d->n_particles;
        const int nl = d->n_levels;
        if (cudaMemsetAsync(ws + L.gy, 0, (size_t)rows * 8 * sizeof(double), st) != cudaSuccess) return check_launch("memset gy");
        int cur = 0;
        if (with_output)   // otherwise the fused tail already left dL/dV of the last level in gV[0]
            LGAE_TRY(run_dec_output_bwd(d, theta, batch, ws + L.S[nl], ws + L.V[nl], g_recon, g_gen00, ws + L.gS[cur], ws + L.gV[cur], &plan, st));
        bool gs_zero = g_gen00 == nullptr;
        for (int l = nl - 1; l >= 0; --l) {
            const double* g_spre = nullptr;
            if (!gs_zero) {
                if (d->has_mlp) {
                    LGAE_TRY(run_mlp(d, l, theta, ws + L.wpack[l], ws + L.spre[l], rows, ws + L.acts[l], nullptr, ws + L.gS[cur], ws + L.gSpre, &plan, true, st));
                    g_spre = ws + L.gSpre;
                } else {
                    g_spre = ws + L.gS[cur];
                }
            }
            if (tiled_gA)
                LGAE_TRY(run_level_bwd_tiled(d, l, theta, ws + L.y, nullptr, batch, ws + L.S[l], ws + L.V[l], ws + L.sums[l], tiled_gA,
                                             nullptr, g_spre, ws + L.gV[cur], ws + L.gS[cur ^ 1], ws + L.gV[cur ^ 1], ws + L.gy, &plan, st));
            else
                LGAE_TRY(run_level_bwd(d, l, theta, ws + L.y, nullptr, batch, ws + L.S[l], ws + L.V[l], ws + L.sums[l], nullptr, nullptr, g_spre,
                                       ws + L.gV[cur], ws + L.gS[cur ^ 1], ws + L.gV[cur ^ 1], ws + L.gy, &plan, st));
            cur ^= 1;
            gs_zero = false;
        }
        if (with_input)   // otherwise the caller continues from gS/gV[n_levels & 1] and gy (fused bridge adjoint)
            LGAE_TRY(run_dec_input_bwd(d, theta, batch, lat11, ws + L.y, ws + L.gS[cur], ws + L.gV[cur], ws + L.gy, g_lat11, &plan, st));
    }
    return LGAE_OK;
}

// LGNEncoder.forward at maxdim 3: the same input map, scalar MLPs and latent glue as at maxdim 2 around the maxdim-3 level
// kernels (lgae_md3.cu); nothing is kept for an adjoint.
static int enc_forward_md3(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                           double* ws, double* lat00, double* lat11, int32_t* sel, cudaStream_t st) {
    const Layout L = layout(d, batch);
    const int64_t rows = (int64_t)batch * d->n_particles;
    LGAE_TRY(run_mlp_pack(d, theta, ws, L.wpack, st));
    LGAE_TRY(run_enc_input(d, theta, p4, batch, ws + L.mass, ws + L.S[0], ws + L.V[0], st));
    for (int l = 0; l < d->n_levels; ++l) {
        LGAE_TRY(run_md3_level_fwd(d, l, theta, p4, node_mask, batch, ws + L.S[l], ws + L.V[l], l > 0 ? ws + L.H[l] : nullptr, ws + L.nbr,
                                   ws + L.spre[l], ws + L.V[l + 1], ws + L.H[l + 1], st));
        if (d->has_mlp)
            LGAE_TRY(run_mlp(d, l, theta, ws + L.wpack[l], ws + L.spre[l], rows, ws + L.acts[l], ws + L.S[l + 1], nullptr, nullptr, nullptr, false, st));
    }
    return run_enc_latent(d, theta, batch, ws + L.S[d->n_levels], ws + L.V[d->n_levels], lat00, lat11, sel, st);
}

// LGNDecoder.forward at maxdim 3; scalars_unused: the last level's scalar MLP feeds only gen00 and is skipped, as at maxdim 2.
static int dec_forward_md3(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch, double* ws, double* recon,
                           double* gen00, cudaStream_t st, bool scalars_unused) {
    const Layout L = layout(d, batch);
    const int64_t rows = (int64_t)batch * d->n_particles;
    LGAE_TRY(run_mlp_pack(d, theta, ws, L.wpack, st));
    LGAE_TRY(run_dec_input(d, theta, batch, lat11, ws + L.y, ws + L.S[0], ws + L.V[0], st));
    for (int l = 0; l < d->n_levels; ++l) {
        LGAE_TRY(run_md3_level_fwd(d, l, theta, ws + L.y, nullptr, batch, ws + L.S[l], ws + L.V[l], l > 0 ? ws + L.H[l] : nullptr, ws + L.nbr,
                                   ws + L.spre[l], ws + L.V[l + 1], ws + L.H[l + 1], st));
        if (d->has_mlp && !(scalars_unused && l == d->n_levels - 1))
            LGAE_TRY(run_mlp(d, l, theta, ws + L.wpack[l], ws + L.spre[l], rows, ws + L.acts[l], ws + L.S[l + 1], nullptr, nullptr, nullptr, false, st));
    }
    return run_dec_output(d, theta, batch, ws + L.S[d->n_levels], ws + L.V[d->n_levels], recon, gen00, st);
}

extern "C" {

int lgae_encoder_forward(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                         double* ws, double* lat00, double* lat11, int32_t* sel, void* stream) {
    LGAE_TRY(check_desc(d));
    if (d->is_decoder || batch < 0) return LGAE_E_BADARG;
    if (batch == 0) return LGAE_OK;   // empty batch: nothing to launch (the tensors' pointers may be NULL)
    if (!theta || !p4 || !ws || !lat00 || !lat11) return LGAE_E_BADARG;
    int rc = LGAE_OK;
    const double* x = scaled_input(d, p4, batch, ws, true, (cudaStream_t)stream, &rc);
    if (rc) return rc;
    if (is_md3(d)) return enc_forward_md3(d, theta, x, node_mask, batch, ws, lat00, lat11, sel, (cudaStream_t)stream);
    return enc_forward_launch(d, theta, x, node_mask, batch, ws, lat00, lat11, sel, true, (cudaStream_t)stream);
}

}  // extern "C"

// lgae_encoder_backward(_p4) and lgae_encoder_backward_tiled(_p4); ig.g_p4 == nullptr: no input gradient.
static int encoder_backward_impl(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                                 double* ws, const int32_t* sel, const double* g_lat00, const double* g_lat11, double* gtheta,
                                 double* partials_or_scratch, double l1_lambda, double* loss_accumulate, bool tiled, InputGrad ig,
                                 void* stream) {
    LGAE_TRY(check_desc(d));
    if (is_md3(d)) return LGAE_E_UNSUPPORTED;   // maxdim 3: forward only
    if (d->is_decoder || !theta || !gtheta || !partials_or_scratch || batch < 0 || (batch > 0 && (!p4 || !ws))) return LGAE_E_BADARG;
    if (ig.g_p4 && batch > 0 && !ig.scratch) return LGAE_E_BADARG;
    // before anything is launched
    if (tiled) LGAE_TRY(tiled_check(d));
    else if (d->n_particles > 32) return LGAE_E_UNSUPPORTED;   // the per-lane adjoint holds one particle per lane
    if (ig.g_p4) LGAE_TRY(pgrad_check(d));
    PartPlan plan;
    TiledBufs bufs;
    if (tiled) {
        const TiledScratch T = tiled_scratch(d, batch);
        plan.base = partials_or_scratch + T.part;
        bufs = TiledBufs{partials_or_scratch + T.gA, partials_or_scratch + T.gr};
    } else {
        plan.base = partials_or_scratch;
    }
    int rc = LGAE_OK;
    p4 = scaled_input(d, p4, batch, ws, false, (cudaStream_t)stream, &rc);   // the forward left the scaled momenta in the workspace
    LGAE_TRY(enc_backward_launch(d, theta, p4, node_mask, batch, ws, sel, g_lat00, g_lat11, plan, (cudaStream_t)stream, true, nullptr,
                                 bufs, ig));
    return run_reduce_plan(&plan, d->n_params, gtheta, theta, l1_lambda, loss_accumulate, (cudaStream_t)stream);
}

extern "C" {

int lgae_encoder_backward(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                          double* ws, const int32_t* sel, const double* g_lat00, const double* g_lat11, double* gtheta,
                          double* partials, double l1_lambda, double* loss_accumulate, void* stream) {
    return encoder_backward_impl(d, theta, p4, node_mask, batch, ws, sel, g_lat00, g_lat11, gtheta, partials, l1_lambda, loss_accumulate,
                                 false, InputGrad{}, stream);
}

int lgae_encoder_backward_p4(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                             double* ws, const int32_t* sel, const double* g_lat00, const double* g_lat11, double* gtheta,
                             double* partials, double l1_lambda, double* loss_accumulate, double* g_p4, double* gp_scratch, void* stream) {
    return encoder_backward_impl(d, theta, p4, node_mask, batch, ws, sel, g_lat00, g_lat11, gtheta, partials, l1_lambda, loss_accumulate,
                                 false, InputGrad{g_p4, gp_scratch}, stream);
}

int64_t lgae_encoder_input_grad_scratch_doubles(const LgaeModelDesc* d, int32_t batch) {
    const int rc = check_desc(d);
    if (rc == LGAE_E_BADARG || batch < 0 || d->is_decoder) return -1;
    if (rc != LGAE_OK || is_md3(d) || pgrad_check(d) != LGAE_OK) return LGAE_E_UNSUPPORTED;
    if (d->n_particles > 32 && tiled_check(d) != LGAE_OK) return LGAE_E_UNSUPPORTED;   // the tiled adjoint runs these jets
    return input_grad_scratch(d, batch).total;
}

int lgae_decoder_forward(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch, double* ws, double* recon,
                         double* gen00, void* stream) {
    LGAE_TRY(check_desc(d));
    if (!d->is_decoder || batch < 0) return LGAE_E_BADARG;
    if (batch == 0) return LGAE_OK;
    if (!theta || !lat11 || !ws || !recon) return LGAE_E_BADARG;
    // gen00 == NULL: the caller does not want the output scalars, and the adjoint never reads the last level's saved
    // activations when there is no gradient on them, so the last level's scalar MLP is not evaluated
    if (is_md3(d)) return dec_forward_md3(d, theta, lat11, batch, ws, recon, gen00, (cudaStream_t)stream, !gen00 && !keep_dead_mlp());
    return dec_forward_launch(d, theta, lat11, batch, ws, recon, gen00, true, (cudaStream_t)stream, true, true, !gen00 && !keep_dead_mlp());
}

int lgae_decoder_backward(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch, double* ws,
                          const double* g_recon, const double* g_gen00, double* g_lat11, double* gtheta, double* partials,
                          double l1_lambda, double* loss_accumulate, void* stream) {
    LGAE_TRY(check_desc(d));
    if (is_md3(d)) return LGAE_E_UNSUPPORTED;   // maxdim 3: forward only
    if (!d->is_decoder || !theta || !gtheta || !partials || batch < 0 || (batch > 0 && (!lat11 || !ws || !g_recon || !g_lat11)))
        return LGAE_E_BADARG;
    if (d->n_particles > 32) return LGAE_E_UNSUPPORTED;   // before anything is launched: the adjoint holds one particle per lane
    PartPlan plan;
    plan.base = partials;
    LGAE_TRY(dec_backward_launch(d, theta, lat11, batch, ws, g_recon, g_gen00, g_lat11, plan, (cudaStream_t)stream));
    return run_reduce_plan(&plan, d->n_params, gtheta, theta, l1_lambda, loss_accumulate, (cudaStream_t)stream);
}

int lgae_encoder_backward_tiled(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                                double* ws, const int32_t* sel, const double* g_lat00, const double* g_lat11, double* gtheta,
                                double* scratch, double l1_lambda, double* loss_accumulate, void* stream) {
    return encoder_backward_impl(d, theta, p4, node_mask, batch, ws, sel, g_lat00, g_lat11, gtheta, scratch, l1_lambda, loss_accumulate,
                                 true, InputGrad{}, stream);
}

int lgae_encoder_backward_tiled_p4(const LgaeModelDesc* d, const double* theta, const double* p4, const uint8_t* node_mask, int32_t batch,
                                   double* ws, const int32_t* sel, const double* g_lat00, const double* g_lat11, double* gtheta,
                                   double* scratch, double l1_lambda, double* loss_accumulate, double* g_p4, double* gp_scratch,
                                   void* stream) {
    return encoder_backward_impl(d, theta, p4, node_mask, batch, ws, sel, g_lat00, g_lat11, gtheta, scratch, l1_lambda, loss_accumulate,
                                 true, InputGrad{g_p4, gp_scratch}, stream);
}

int lgae_decoder_backward_tiled(const LgaeModelDesc* d, const double* theta, const double* lat11, int32_t batch, double* ws,
                                const double* g_recon, const double* g_gen00, double* g_lat11, double* gtheta, double* scratch,
                                double l1_lambda, double* loss_accumulate, void* stream) {
    LGAE_TRY(check_desc(d));
    if (is_md3(d)) return LGAE_E_UNSUPPORTED;   // maxdim 3: forward only
    if (!d->is_decoder || !theta || !gtheta || !scratch || batch < 0 || (batch > 0 && (!lat11 || !ws || !g_recon || !g_lat11)))
        return LGAE_E_BADARG;
    LGAE_TRY(tiled_check(d));
    const TiledScratch T = tiled_scratch(d, batch);
    PartPlan plan;
    plan.base = scratch + T.part;
    LGAE_TRY(dec_backward_launch(d, theta, lat11, batch, ws, g_recon, g_gen00, g_lat11, plan, (cudaStream_t)stream, true, true, scratch + T.gA));
    return run_reduce_plan(&plan, d->n_params, gtheta, theta, l1_lambda, loss_accumulate, (cudaStream_t)stream);
}

void* lgae_aux_stream(void) {
    AuxStream* aux = aux_stream();
    return aux ? (void*)aux->s : nullptr;
}

int64_t lgae_train_step_partials_doubles(const LgaeModelDesc* enc, const LgaeModelDesc* dec, int32_t batch) {
    if (check_desc(enc) == LGAE_OK && check_desc(dec) == LGAE_OK && batch >= 0 && (is_md3(enc) || is_md3(dec))) return LGAE_E_UNSUPPORTED;
    const int64_t a = lgae_partials_doubles(enc, batch), b = lgae_partials_doubles(dec, batch);
    if (a < 0 || b < 0) return -1;
    // + the fused decoder tail's rows (one per jet) and one trailing double whose first 4 bytes are its completion counter
    return a + b + (int64_t)batch * 4 * dec->channels[dec->n_levels] + 1;
}

}  // extern "C"

// Plan of the encoder's partial rows handed from phase 1 to phase 2 of a split step (same thread, back to back).
static thread_local PartPlan tl_plan_e;
static thread_local bool tl_phase1 = false;

// Body of lgae_train_step / lgae_train_step_host.  phase: 0 = the whole step; 1 = everything up to the point where the
// decoder's gradient bucket is final (its reduce is enqueued on the auxiliary stream, lgae_aux_stream()); 2 = the rest (encoder
// adjoint + encoder reduce).  Between phases 1 and 2 the caller may enqueue work on the auxiliary stream -- the data-parallel
// all-reduce of the decoder bucket -- which then overlaps the encoder adjoint; phase 2 joins the auxiliary stream back.  host_p4 / host_mask / host_loss (pinned host memory, may be NULL): the jets
// are copied to p4_in (and the mask to node_mask) at the start and the loss back at the end, on the same stream -- after the
// auxiliary branch has been forked, so that weight packing and gradient init overlap the host-to-device copy.
// tiled: the adjoints are the tiled ones (any N) and `buf` is the scratch of lgae_train_step_tiled_scratch_doubles; otherwise
// the per-lane ones (N <= 32) and `buf` is the partials buffer of lgae_train_step_partials_doubles.
static int train_step_impl(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc, const double* theta_dec,
                           double* p4_in, uint8_t* node_mask, int32_t batch, int32_t normalize, double* p4, double* norm_factor,
                           double* ws_enc, double* ws_dec, double* lat00, double* lat11, int32_t* sel, double* recon, double* g_recon,
                           double* g_lat11, double* jet_loss, double* loss, double* gtheta, int64_t gtheta_dec_offset, double* buf,
                           double l1_lambda, int32_t get_real, const double* host_p4, const uint8_t* host_mask, double* host_loss, int32_t phase,
                           bool tiled, void* stream) {
    LGAE_TRY(check_desc(enc));
    LGAE_TRY(check_desc(dec));
    if (is_md3(enc) || is_md3(dec)) return LGAE_E_UNSUPPORTED;   // maxdim 3: forward only
    if (enc->is_decoder || !dec->is_decoder || batch < 1 || gtheta_dec_offset < enc->n_params) return LGAE_E_BADARG;
    if (get_real < LGAE_GET_REAL_REAL || get_real > LGAE_GET_REAL_NORM || phase < 0 || phase > 2) return LGAE_E_BADARG;
    if (!theta_enc || !theta_dec || !p4_in || !p4 || !ws_enc || !ws_dec || !lat00 || !lat11 || !sel || !recon || !g_recon || !g_lat11 ||
        !jet_loss || !loss || !gtheta || !buf)
        return LGAE_E_BADARG;
    if (!tiled && enc->n_particles > 32) return LGAE_E_UNSUPPORTED;   // the per-lane adjoint holds one particle per lane
    // size of `buf`; for the tiled step also the refusal of a configuration before anything is launched
    const int64_t n_buf = tiled ? lgae_train_step_tiled_scratch_doubles(enc, dec, batch) : lgae_train_step_partials_doubles(enc, dec, batch);
    if (n_buf < 0) return (int)n_buf;
    const StepScratch SS = tiled ? step_scratch(enc, dec, batch) : StepScratch{};
    double* partials = tiled ? buf + SS.part : buf;   // the two plans' rows
    cudaStream_t st = (cudaStream_t)stream;
    const double* x = normalize ? p4 : p4_in;
    const bool scaled = has_input_scale(enc);
    AuxStream* aux = aux_stream();
    if (!aux) return LGAE_E_CUDA;
    if (phase == 2 && !tl_phase1) return LGAE_E_BADARG;
    std::lock_guard<std::mutex> aux_lock(g_aux_mu);
    // L1 partial sums of the gradient init: the second reduce-scratch region at the end of `buf` (the first one, behind the
    // plan's blocks, is unused by this entry point)
    double* psum = buf + n_buf - 1 - reduce_scratch_doubles();
    const int64_t n_all = enc->n_params + dec->n_params;
    PartPlan plan_d, plan_e;
    int rc_scale = LGAE_OK;
    const double* xe = x;
    if (phase != 2) {
    // forward: one launch packs the MLP weights of both models
    {
        const Layout Le = layout(enc, batch), Ld = layout(dec, batch);
        // weight packing and gradient init only need theta: a parallel branch next to normalise + radial functions
        LGAE_CUDA_TRY(cudaEventRecord(aux->fork[0], st), "aux fork");
        LGAE_CUDA_TRY(cudaStreamWaitEvent(aux->s, aux->fork[0], 0), "aux fork wait");
        LGAE_TRY(run_mlp_pack(enc, theta_enc, ws_enc, Le.wpack, aux->s, dec, theta_dec, ws_dec, Ld.wpack));
        LGAE_CUDA_TRY(cudaEventRecord(aux->join[0], aux->s), "aux join");
        LGAE_TRY(run_grad_init2(theta_enc, enc->n_params, theta_dec, dec->n_params, gtheta_dec_offset, gtheta, l1_lambda, psum, aux->s));
        LGAE_CUDA_TRY(cudaEventRecord(aux->join[1], aux->s), "aux join");
        if (host_p4)
            LGAE_CUDA_TRY(cudaMemcpyAsync(p4_in, host_p4, (size_t)batch * enc->n_particles * 4 * sizeof(double), cudaMemcpyHostToDevice, st), "H2D jets");
        if (host_mask && node_mask)
            LGAE_CUDA_TRY(cudaMemcpyAsync(node_mask, host_mask, (size_t)batch * enc->n_particles, cudaMemcpyHostToDevice, st), "H2D mask");
        if (normalize && !scaled)   // normalisation + encoder input map, one CTA per jet
            LGAE_TRY(run_norm_input(enc, theta_enc, p4_in, batch, p4, norm_factor, ws_enc + Le.mass, ws_enc + Le.S[0], ws_enc + Le.V[0], st));
        else if (normalize)
            LGAE_TRY(run_normalize(p4_in, batch, enc->n_particles, p4, norm_factor, st));
    }
    // x: the (normalised) jets = the loss target; xe: what the encoder reads (x times the encoder's input scale)
    xe = scaled_input(enc, x, batch, ws_enc, true, st, &rc_scale);
    LGAE_TRY(rc_scale);
    // The scalar MLP of the encoder's last level only feeds the latent scalars, an output of the step that neither the decoder nor
    // the loss reads: it runs, with the scalar half of the latent map, as a branch on the auxiliary stream (0.8507 -> 0.8360 ms
    // per step against running it in line; the split step runs it in line)
    const bool defer = phase == 0 && enc->has_mlp;
    LGAE_TRY(enc_forward_launch(enc, theta_enc, xe, node_mask, batch, ws_enc, lat00, lat11, sel, false, st, false, !normalize || scaled,
                                aux->join[0], defer));
    {
        // fused encoder latent map + decoder input map
        const Layout Le = layout(enc, batch), Ld = layout(dec, batch);
        const int nl = enc->n_levels;
        if (defer) {
            LGAE_CUDA_TRY(cudaEventRecord(aux->fork[3], st), "aux fork");
            LGAE_CUDA_TRY(cudaStreamWaitEvent(aux->s, aux->fork[3], 0), "aux fork wait");
            LGAE_TRY(run_mlp(enc, nl - 1, theta_enc, ws_enc + Le.wpack[nl - 1], ws_enc + Le.spre[nl - 1], (int64_t)batch * enc->n_particles,
                             ws_enc + Le.acts[nl - 1], ws_enc + Le.S[nl], nullptr, nullptr, nullptr, false, aux->s));
            LGAE_TRY(run_enc_latent(enc, theta_enc, batch, ws_enc + Le.S[nl], ws_enc + Le.V[nl], lat00, lat11, sel, aux->s, 1));
            LGAE_CUDA_TRY(cudaEventRecord(aux->join[4], aux->s), "aux join");
        }
        LGAE_TRY(run_latent_bridge(enc, theta_enc, dec, theta_dec, batch, ws_enc + Le.S[nl], ws_enc + Le.V[nl], lat00,
                                   lat11, sel, ws_dec + Ld.y, ws_dec + Ld.S[0], ws_dec + Ld.V[0], st, defer ? 2 : 3));
    }
    LGAE_TRY(dec_forward_launch(dec, theta_dec, lat11, batch, ws_dec, recon, nullptr, false, st, false, false, !keep_dead_mlp()));
    // one plan per model over the same partials buffer (the encoder's continues where the decoder's ends): the decoder's rows are
    // reduced on the auxiliary stream while the encoder adjoint runs, the encoder's at the end
    plan_d.base = plan_e.base = partials;
    plan_d.theta_base = gtheta_dec_offset;
    {
        // fused decoder tail: reconstruction, chamfer (+ batch sum), loss gradient, adjoint of the output map
        const Layout Ld = layout(dec, batch);
        unsigned int* counter = reinterpret_cast<unsigned int*>(buf + n_buf - 1);
        LGAE_TRY(run_dec_tail(dec, theta_dec, batch, enc->n_particles, ws_dec + Ld.V[dec->n_levels], x, recon, g_recon, ws_dec + Ld.gV[0],
                              jet_loss, loss, counter, get_real, &plan_d, st));
    }
    LGAE_TRY(dec_backward_launch(dec, theta_dec, lat11, batch, ws_dec, g_recon, nullptr, g_lat11, plan_d, st, false, false,
                                 tiled ? buf + SS.gA : nullptr));
    {
        // fused adjoint of the bridge: decoder input map, then encoder latent map, latent gradient handed over on chip
        const Layout Le = layout(enc, batch), Ld = layout(dec, batch);
        const int cur = dec->n_levels & 1;
        if (defer) LGAE_CUDA_TRY(cudaStreamWaitEvent(st, aux->join[4], 0), "aux join wait");   // S of the last level, latent scalars, sel
        LGAE_TRY(run_latent_bridge_bwd(dec, theta_dec, enc, theta_enc, batch, lat11, ws_dec + Ld.y, ws_dec + Ld.gS[cur], ws_dec + Ld.gV[cur],
                                       ws_dec + Ld.gy, g_lat11, ws_enc + Le.S[enc->n_levels], ws_enc + Le.V[enc->n_levels], sel,
                                       ws_enc + Le.gS[0], ws_enc + Le.gV[0], &plan_d, &plan_e, st));
    }
    {
        // the decoder's gradient is complete: reduce it now, next to the encoder adjoint (the gradient init ran on this stream)
        LGAE_CUDA_TRY(cudaEventRecord(aux->fork[2], st), "aux fork");
        LGAE_CUDA_TRY(cudaStreamWaitEvent(aux->s, aux->fork[2], 0), "aux fork wait");
        // ... and the loss is final once the L1 term joins the chamfer sum (dec_tail): add it here and send it to the host now,
        // so that the device-to-host copy overlaps the encoder adjoint instead of trailing the step
        LGAE_TRY(run_reduce_segs(&plan_d, n_all, gtheta, psum, l1_lambda, loss, aux->s));
        if (host_loss) LGAE_CUDA_TRY(cudaMemcpyAsync(host_loss, loss, sizeof(double), cudaMemcpyDeviceToHost, aux->s), "D2H loss");
    }
    if (phase == 1) {
        tl_plan_e = plan_e;
        tl_phase1 = true;
        return LGAE_OK;
    }
    } else {
        plan_e = tl_plan_e;
        tl_phase1 = false;
        xe = scaled_input(enc, x, batch, ws_enc, false, st, &rc_scale);
    }
    // (split step: whatever the caller enqueued on the auxiliary stream between the phases is joined here too)
    LGAE_CUDA_TRY(cudaEventRecord(aux->join[3], aux->s), "aux join");
    LGAE_TRY(enc_backward_launch(enc, theta_enc, xe, node_mask, batch, ws_enc, sel, nullptr, g_lat11, plan_e, st, false, aux,
                                 tiled ? TiledBufs{buf + SS.gA, buf + SS.gr} : TiledBufs{}));
    LGAE_CUDA_TRY(cudaStreamWaitEvent(st, aux->join[1], 0), "aux join wait");
    LGAE_CUDA_TRY(cudaStreamWaitEvent(st, aux->join[3], 0), "aux join wait");
    return run_reduce_segs(&plan_e, n_all, gtheta, psum, 0.0, nullptr, st);
}

extern "C" {

int lgae_train_step(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc, const double* theta_dec,
                    const double* p4_in, const uint8_t* node_mask, int32_t batch, int32_t normalize, double* p4, double* norm_factor,
                    double* ws_enc, double* ws_dec, double* lat00, double* lat11, int32_t* sel, double* recon, double* g_recon,
                    double* g_lat11, double* jet_loss, double* loss, double* gtheta, int64_t gtheta_dec_offset, double* partials,
                    double l1_lambda, int32_t get_real, int32_t phase, void* stream) {
    return train_step_impl(enc, dec, theta_enc, theta_dec, const_cast<double*>(p4_in), const_cast<uint8_t*>(node_mask), batch, normalize, p4,
                           norm_factor, ws_enc, ws_dec, lat00, lat11, sel, recon, g_recon, g_lat11, jet_loss, loss, gtheta, gtheta_dec_offset,
                           partials, l1_lambda, get_real, nullptr, nullptr, nullptr, phase, false, stream);
}

int lgae_train_step_host(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc, const double* theta_dec,
                         const double* host_p4, const uint8_t* host_mask, double* host_loss, double* p4_in, uint8_t* node_mask,
                         int32_t batch, int32_t normalize, double* p4, double* norm_factor, double* ws_enc, double* ws_dec, double* lat00,
                         double* lat11, int32_t* sel, double* recon, double* g_recon, double* g_lat11, double* jet_loss, double* loss,
                         double* gtheta, int64_t gtheta_dec_offset, double* partials, double l1_lambda, int32_t get_real, int32_t phase,
                         void* stream) {
    if (!host_p4 || !host_loss) return LGAE_E_BADARG;
    return train_step_impl(enc, dec, theta_enc, theta_dec, p4_in, node_mask, batch, normalize, p4, norm_factor, ws_enc, ws_dec, lat00, lat11, sel,
                           recon, g_recon, g_lat11, jet_loss, loss, gtheta, gtheta_dec_offset, partials, l1_lambda, get_real, host_p4, host_mask,
                           host_loss, phase, false, stream);
}

int lgae_train_step_tiled(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc, const double* theta_dec,
                          const double* p4_in, const uint8_t* node_mask, int32_t batch, int32_t normalize, double* p4, double* norm_factor,
                          double* ws_enc, double* ws_dec, double* lat00, double* lat11, int32_t* sel, double* recon, double* g_recon,
                          double* g_lat11, double* jet_loss, double* loss, double* gtheta, int64_t gtheta_dec_offset, double* scratch,
                          double l1_lambda, int32_t get_real, int32_t phase, void* stream) {
    return train_step_impl(enc, dec, theta_enc, theta_dec, const_cast<double*>(p4_in), const_cast<uint8_t*>(node_mask), batch, normalize, p4,
                           norm_factor, ws_enc, ws_dec, lat00, lat11, sel, recon, g_recon, g_lat11, jet_loss, loss, gtheta, gtheta_dec_offset,
                           scratch, l1_lambda, get_real, nullptr, nullptr, nullptr, phase, true, stream);
}

int lgae_train_step_tiled_host(const LgaeModelDesc* enc, const LgaeModelDesc* dec, const double* theta_enc, const double* theta_dec,
                               const double* host_p4, const uint8_t* host_mask, double* host_loss, double* p4_in, uint8_t* node_mask,
                               int32_t batch, int32_t normalize, double* p4, double* norm_factor, double* ws_enc, double* ws_dec,
                               double* lat00, double* lat11, int32_t* sel, double* recon, double* g_recon, double* g_lat11, double* jet_loss,
                               double* loss, double* gtheta, int64_t gtheta_dec_offset, double* scratch, double l1_lambda, int32_t get_real,
                               int32_t phase, void* stream) {
    if (!host_p4 || !host_loss) return LGAE_E_BADARG;
    return train_step_impl(enc, dec, theta_enc, theta_dec, p4_in, node_mask, batch, normalize, p4, norm_factor, ws_enc, ws_dec, lat00, lat11, sel,
                           recon, g_recon, g_lat11, jet_loss, loss, gtheta, gtheta_dec_offset, scratch, l1_lambda, get_real, host_p4, host_mask,
                           host_loss, phase, true, stream);
}

int lgae_chamfer(const double* recon, const double* target, int32_t batch, int32_t n, int32_t m, int32_t get_real, double* loss,
                 double* jet_loss, const double* g_loss, double* g_recon, void* stream) {
    if (batch < 0 || n < 1 || m < 1 || (batch > 0 && (!recon || !target || !jet_loss))) return LGAE_E_BADARG;
    if (get_real < LGAE_GET_REAL_REAL || get_real > LGAE_GET_REAL_NORM) return LGAE_E_BADARG;
    if (batch == 0) {
        if (loss && cudaMemsetAsync(loss, 0, sizeof(double), (cudaStream_t)stream) != cudaSuccess) return check_launch("memset loss");
        return LGAE_OK;
    }
    return run_chamfer(recon, target, batch, n, m, loss, jet_loss, g_loss, g_recon, get_real, (cudaStream_t)stream);
}

int lgae_anomaly_scores(const double* recon, const double* target, const double* factor, int32_t batch, int32_t n, int32_t get_real,
                        double* scores, void* stream) {
    if (batch < 0 || n < 1 || (batch > 0 && (!recon || !target || !scores))) return LGAE_E_BADARG;
    if (get_real < LGAE_GET_REAL_REAL || get_real > LGAE_GET_REAL_NORM) return LGAE_E_BADARG;
    if (batch == 0) return LGAE_OK;
    return run_scores(recon, target, factor, batch, n, get_real, scores, (cudaStream_t)stream);
}

int lgae_normalize_p4(const double* p4, int32_t batch, int32_t n, double* out, double* factor, void* stream) {
    if (batch < 0 || n < 1 || (batch > 0 && (!p4 || !out))) return LGAE_E_BADARG;
    if (batch == 0) return LGAE_OK;
    return run_normalize(p4, batch, n, out, factor, (cudaStream_t)stream);
}

int lgae_normalize_p4_backward(const double* p4, int32_t batch, int32_t n, const double* g_out, const double* g_factor, double* g_p4,
                               void* stream) {
    if (batch < 0 || n < 1 || (batch > 0 && (!p4 || !g_p4))) return LGAE_E_BADARG;
    if (batch == 0) return LGAE_OK;
    return run_normalize_bwd(p4, batch, n, g_out, g_factor, g_p4, (cudaStream_t)stream);
}

int lgae_chamfer_target_grad(const double* recon, const double* target, int32_t batch, int32_t n, int32_t m, int32_t get_real,
                             const double* g_loss, double* g_target, void* stream) {
    if (batch < 0 || n < 1 || m < 1 || (batch > 0 && (!recon || !target || !g_target))) return LGAE_E_BADARG;
    if (get_real < LGAE_GET_REAL_REAL || get_real > LGAE_GET_REAL_NORM) return LGAE_E_BADARG;
    if (batch == 0) return LGAE_OK;
    return run_chamfer_target_grad(recon, target, batch, n, m, get_real, g_loss, g_target, (cudaStream_t)stream);
}

int lgae_l1(const double* theta, int64_t n, double lambda, double* out_accumulate, double* gtheta_accumulate, void* stream) {
    if (!theta || n < 0) return LGAE_E_BADARG;
    if (n == 0) return LGAE_OK;
    return run_l1(theta, n, lambda, out_accumulate, gtheta_accumulate, (cudaStream_t)stream);
}

int lgae_level_forward(const LgaeModelDesc* d, int32_t level, const double* theta, const double* p_or_y, const uint8_t* node_mask,
                       int32_t batch, const double* s_in, const double* v_in, double* sums, double* r_save, double* s_pre, double* v_out,
                       void* stream) {
    LGAE_TRY(check_desc(d));
    if (is_md3(d)) return LGAE_E_UNSUPPORTED;   // the stage-level entry points are the maxdim-2 level
    if (!theta || !p_or_y || !s_in || !v_in || !sums || !s_pre || !v_out || batch < 0 || level < 0 || level >= d->n_levels) return LGAE_E_BADARG;
    if (!d->is_decoder && r_save && d->n_particles > 32) return LGAE_E_UNSUPPORTED;   // the saved radial weights are a 32-particle layout
    if (!d->is_decoder && d->n_particles <= 32 && r_save)
        LGAE_TRY(run_radial_fwd(d, level, theta, p_or_y, node_mask, batch, r_save, nullptr, (cudaStream_t)stream));
    return run_level_fwd(d, level, theta, p_or_y, node_mask, batch, s_in, v_in, sums, r_save, s_pre, v_out, (cudaStream_t)stream);
}
int lgae_level_backward(const LgaeModelDesc* d, int32_t level, const double* theta, const double* p_or_y, const uint8_t* node_mask,
                        int32_t batch, const double* s_in, const double* v_in, const double* sums, const double* r_save,
                        double* g_r_scratch, const double* g_s_pre, const double* g_v_out, double* g_s_in, double* g_v_in,
                        double* g_y_accumulate, double* gtheta, double* partials, void* stream) {
    LGAE_TRY(check_desc(d));
    if (is_md3(d)) return LGAE_E_UNSUPPORTED;   // the stage-level entry points are the maxdim-2 level
    if (!theta || !p_or_y || !s_in || !v_in || !sums || !g_v_out || !g_s_in || !g_v_in || !gtheta || !partials || batch < 0 || level < 0 ||
        level >= d->n_levels)
        return LGAE_E_BADARG;
    if (d->is_decoder && !g_y_accumulate) return LGAE_E_BADARG;
    if (!d->is_decoder && (!r_save || !g_r_scratch)) return LGAE_E_BADARG;
    PartPlan plan;
    plan.base = partials;
    LGAE_TRY(run_level_bwd(d, level, theta, p_or_y, node_mask, batch, s_in, v_in, sums, r_save, g_r_scratch, g_s_pre, g_v_out, g_s_in,
                           g_v_in, g_y_accumulate, &plan, (cudaStream_t)stream));
    if (!d->is_decoder) {
        // the pair norms live behind the dL/dR scratch: g_r_scratch holds B*N*C*128 + B*nrm_stride doubles
        double* nrm = g_r_scratch + (int64_t)batch * d->n_particles * d->channels[level] * 128;
        double* r_tmp = const_cast<double*>(r_save);
        LGAE_TRY(run_radial_fwd(d, level, theta, p_or_y, node_mask, batch, r_tmp, nrm, (cudaStream_t)stream));   // refreshes R, writes the norms
        LGAE_TRY(run_radial_bwd(d, level, theta, p_or_y, node_mask, batch, g_r_scratch, nrm, &plan, (cudaStream_t)stream));
    }
    return run_reduce_plan(&plan, d->n_params, gtheta, nullptr, 0.0, nullptr, (cudaStream_t)stream);
}
int64_t lgae_mlp_pack_doubles(const LgaeModelDesc* d, int32_t level) {
    if (check_desc(d) != LGAE_OK || level < 0 || level >= d->n_levels) return -1;
    return mlp_pack_doubles(d, level);
}
static int pack_one_level(const LgaeModelDesc* d, int level, const double* theta, double* wpack, cudaStream_t st) {
    // pack every level's weights contiguously starting at `wpack` would need more room than one level: pack only `level`
    LgaeModelDesc one = *d;
    one.n_levels = 1;
    one.channels[0] = d->channels[level]; one.channels[1] = d->channels[level + 1];
    one.mlp_width[0] = d->mlp_width[level];
    for (int i = 0; i < LGAE_MAX_LINEAR; ++i) { one.off_mlp_w[0][i] = d->off_mlp_w[level][i]; one.off_mlp_b[0][i] = d->off_mlp_b[level][i]; }
    const int64_t off0 = 0;
    return run_mlp_pack(&one, theta, wpack, &off0, st);
}
int lgae_mlp_forward(const LgaeModelDesc* d, int32_t level, const double* theta, const double* x, int64_t rows, double* wpack,
                     double* acts, double* y, void* stream) {
    LGAE_TRY(check_desc(d));
    if (!theta || !x || !wpack || !acts || !y || rows < 0 || level < 0 || level >= d->n_levels) return LGAE_E_BADARG;
    LGAE_TRY(pack_one_level(d, level, theta, wpack, (cudaStream_t)stream));
    return run_mlp(d, level, theta, wpack, x, rows, acts, y, nullptr, nullptr, nullptr, false, (cudaStream_t)stream);
}
int lgae_mlp_backward(const LgaeModelDesc* d, int32_t level, const double* theta, const double* x, int64_t rows, const double* wpack,
                      const double* acts, const double* g_y, double* g_x, double* gtheta, double* partials, void* stream) {
    LGAE_TRY(check_desc(d));
    if (!theta || !x || !wpack || !acts || !g_y || !gtheta || !partials || rows < 0 || level < 0 || level >= d->n_levels) return LGAE_E_BADARG;
    PartPlan plan;
    plan.base = partials;
    LGAE_TRY(run_mlp(d, level, theta, wpack, x, rows, const_cast<double*>(acts), nullptr, g_y, g_x, &plan, true, (cudaStream_t)stream));
    return run_reduce_plan(&plan, d->n_params, gtheta, nullptr, 0.0, nullptr, (cudaStream_t)stream);
}

}  // extern "C"
