// extern "C" entry points declared in include/gf_b200.h: argument validation, workspace carving,
// kernel sequencing.  No torch types, no allocation, no synchronisation (except gf_splat_read_flags).
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include <cstdlib>

#include "common.cuh"
#include "gf_b200_debug.h"

namespace gf {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what) {
    set_error("CUDA error %d (%s) in %s", static_cast<int>(e), cudaGetErrorString(e), what);
    return GF_ERR_CUDA;
}

// defined in the kernel translation units
int plan_forward_workspace(const gf_splat_desc &d, void *base, SplatWorkspace *ws);
int launch_prep(const gf_splat_desc &d, const gf_splat_inputs &in, const SplatWorkspace &ws, uint32_t initial_flags,
                cudaStream_t stream, bool raw_records = false);
int launch_render(const gf_splat_desc &d, const gf_splat_inputs &in, const gf_splat_outputs &out,
                  const SplatWorkspace &ws, bool tile_path, int num_sms, cudaStream_t stream);
size_t backward_workspace_bytes(const gf_splat_desc &d);
int launch_backward(const gf_splat_desc &d, const gf_splat_inputs &in, const gf_splat_grads &gr, void *workspace,
                    int num_sms, cudaStream_t stream);
int render_ctas_per_sample(const gf_splat_desc &d);
extern thread_local cudaEvent_t g_ev_before, g_ev_after;
extern const int kSupportedClasses[];
extern const int kNumSupportedClasses;

struct DafParams;
int launch_daf_forward(const gf_daf_desc &d, const float *feat, const int32_t *shape, const int32_t *start,
                       const float *loc, const float *weights, float *out, int num_sms, cudaStream_t stream);
int launch_daf_format(const gf_daf_format_desc &d, float *const *maps, float *table, bool inverse, cudaStream_t stream);
int launch_daf_backward(const gf_daf_desc &d, const float *feat, const int32_t *shape, const int32_t *start,
                        const float *loc, const float *weights, const float *grad_out, float *grad_feat,
                        float *grad_loc, float *grad_weights, int num_sms, cudaStream_t stream);

bool daf_fused_supported(const gf_daf_desc &d, int K);
int launch_daf_fused_forward(const gf_daf_desc &d, int K, const float *feat, const int32_t *shape, const int32_t *start,
                             const float *loc, const float *logits, const uint8_t *pmask, const uint8_t *wmask,
                             float *out, float *stats, int num_sms, cudaStream_t stream);
int launch_daf_fused_backward(const gf_daf_desc &d, int K, const float *feat, const int32_t *shape, const int32_t *start,
                              const float *loc, const float *logits, const uint8_t *pmask, const uint8_t *wmask,
                              const float *stats, const float *out, const float *grad_out, float *grad_feat,
                              float *grad_loc, float *grad_logits, int num_sms, cudaStream_t stream);

int occ_loss_check(const gf_occ_loss_desc *d);
size_t occ_loss_workspace_bytes(const gf_occ_loss_desc &d);
int occ_loss_forward(const gf_occ_loss_desc &d, const float *pred, const uint8_t *labels, const uint8_t *mask,
                     const float *weights, float *loss3, float *grad, uint32_t *status, void *ws, cudaStream_t stream);

thread_local cudaEvent_t g_ev_before = nullptr, g_ev_after = nullptr;

bool pdl_enabled() {
    static const bool on = [] {
        const char *e = getenv("GF_B200_PDL");
        return !(e && e[0] == '0');
    }();
    return on;
}

static int num_sms_of_current_device(int *out) {
    static int cached[64];
    int dev = 0;
    GF_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) dev = 0;
    if (cached[dev] == 0) {
        int n = 0;
        GF_CUDA_TRY(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
        cached[dev] = n > 0 ? n : 1;
    }
    *out = cached[dev];
    return GF_OK;
}

static int check_desc(const gf_splat_desc *d) {
    GF_REQUIRE(d != nullptr, GF_ERR_INVALID_ARG, "splat: desc is NULL");
    GF_REQUIRE(d->G >= 0 && d->N >= 0, GF_ERR_INVALID_ARG, "splat: negative G or N");
    GF_REQUIRE(d->H > 0 && d->W > 0 && d->D > 0, GF_ERR_INVALID_ARG, "splat: grid dims must be positive");
    GF_REQUIRE(d->H <= 65535 && d->W <= 65535 && d->D <= 65535, GF_ERR_UNSUPPORTED,
               "splat: grid dims above 65535 are not supported (boxes are packed to 16 bits per bound)");
    GF_REQUIRE(static_cast<long long>(d->H) * d->W * d->D < (1ll << 31), GF_ERR_UNSUPPORTED,
               "splat: more than 2^31 voxels");
    GF_REQUIRE(d->variant == GF_SPLAT_BASE || d->variant == GF_SPLAT_PROB, GF_ERR_INVALID_ARG,
               "splat: unknown variant %d", d->variant);
    GF_REQUIRE(d->radii_axes == 1 || d->radii_axes == 3, GF_ERR_INVALID_ARG, "splat: radii_axes must be 1 or 3");
    GF_REQUIRE(d->cov_stride == 6 || d->cov_stride == 9, GF_ERR_INVALID_ARG, "splat: cov_stride must be 6 or 9");
    GF_REQUIRE(d->batch >= 0 && d->batch <= 65535, GF_ERR_INVALID_ARG, "splat: batch=%d outside [0, 65535]", d->batch);
    GF_REQUIRE(static_cast<long long>(batch_of(*d)) * d->N * d->C < (1ll << 40), GF_ERR_UNSUPPORTED,
               "splat: batch x N x C too large");
    bool ok = false;
    for (int i = 0; i < kNumSupportedClasses; ++i) ok = ok || kSupportedClasses[i] == d->C;
    GF_REQUIRE(ok, GF_ERR_UNSUPPORTED, "splat: class count C=%d is not compiled in", d->C);
    return GF_OK;
}

static int check_inputs(const gf_splat_desc *d, const gf_splat_inputs *in) {
    GF_REQUIRE(in != nullptr, GF_ERR_INVALID_ARG, "splat: inputs struct is NULL");
    if (d->N > 0) GF_REQUIRE(in->pts != nullptr, GF_ERR_INVALID_ARG, "splat: pts is NULL");
    if (d->G > 0) {
        GF_REQUIRE(in->means && in->opacities && in->semantics, GF_ERR_INVALID_ARG,
                   "splat: means / opacities / semantics must not be NULL");
        GF_REQUIRE(in->cov || (in->scales && in->rotations), GF_ERR_INVALID_ARG,
                   "splat: need cov, or scales + rotations to build the inverse covariance from");
        GF_REQUIRE(in->radii || in->scales, GF_ERR_INVALID_ARG, "splat: need radii or scales");
        if (!in->means_int || !in->radii || !in->points_int)
            GF_REQUIRE(d->grid_size > 0.f, GF_ERR_INVALID_ARG, "splat: grid_size must be > 0 for fused host prep");
    }
    return GF_OK;
}

}  // namespace gf

using namespace gf;

extern "C" {

int gf_abi_version(void) { return GF_ABI_VERSION; }

const char *gf_last_error(void) { return g_err; }

int gf_debug_set_render_events(void *before, void *after) {
    g_ev_before = static_cast<cudaEvent_t>(before);
    g_ev_after = static_cast<cudaEvent_t>(after);
    return GF_OK;
}

int gf_splat_supported_classes(int32_t *out, int cap) {
    int n = 0;
    for (; n < kNumSupportedClasses && n < cap; ++n) out[n] = kSupportedClasses[n];
    return n;
}

size_t gf_splat_forward_workspace_bytes(const gf_splat_desc *desc) {
    if (check_desc(desc) != GF_OK) return 0;
    SplatWorkspace ws;
    plan_forward_workspace(*desc, nullptr, &ws);
    return ws.bytes;
}

int gf_splat_ce_partials(const gf_splat_desc *desc) {
    if (check_desc(desc) != GF_OK) return 0;
    if (static_cast<long long>(desc->N) != static_cast<long long>(desc->H) * desc->W * desc->D) return 0;
    return render_ctas_per_sample(*desc) * batch_of(*desc);
}

size_t gf_splat_backward_workspace_bytes(const gf_splat_desc *desc) {
    if (check_desc(desc) != GF_OK) return 0;
    return backward_workspace_bytes(*desc);
}

int gf_splat_forward(const gf_splat_desc *desc, const gf_splat_inputs *in, const gf_splat_outputs *out,
                     void *workspace, size_t workspace_bytes, gf_stream_t stream_) {
    int rc = check_desc(desc);
    if (rc != GF_OK) return rc;
    rc = check_inputs(desc, in);
    if (rc != GF_OK) return rc;
    GF_REQUIRE(out != nullptr && (desc->N == 0 || out->logits || out->logits_cn || out->argmax || out->ce_partials),
               GF_ERR_INVALID_ARG, "splat: no output requested (logits, logits_cn, argmax and ce_partials are all NULL)");
    const bool tile_path = static_cast<long long>(desc->N) == static_cast<long long>(desc->H) * desc->W * desc->D;
    if (out->ce_partials)
        GF_REQUIRE(out->labels != nullptr && tile_path, GF_ERR_INVALID_ARG,
                   "splat: ce_partials needs labels and one point per voxel (N == H*W*D)");
    if (desc->variant == GF_SPLAT_PROB && desc->N > 0)
        GF_REQUIRE(out->bin_logits && out->density && out->probability, GF_ERR_INVALID_ARG,
                   "splat(prob): bin_logits / density / probability must not be NULL");
    SplatWorkspace ws;
    plan_forward_workspace(*desc, workspace, &ws);
    GF_REQUIRE(workspace != nullptr && workspace_bytes >= ws.bytes, GF_ERR_WORKSPACE,
               "splat: workspace too small (%zu < %zu bytes)", workspace_bytes, ws.bytes);
    GF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, GF_ERR_WORKSPACE,
               "splat: workspace must be 256-byte aligned");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int num_sms = 1;
    rc = num_sms_of_current_device(&num_sms);
    if (rc != GF_OK) return rc;
    // The tile path needs exactly one point per voxel in x-major order; it verifies that on the
    // device and hands over to the generic kernel otherwise.  N != H*W*D can only be generic.
    // (The preparation kernels run for N == 0 too: they initialise the status word gf_splat_read_flags reports.)
    rc = launch_prep(*desc, *in, ws, tile_path ? 0u : GF_FLAG_GENERIC_PATH, stream);
    if (rc != GF_OK) return rc;
    if (desc->N == 0) return GF_OK;
    return launch_render(*desc, *in, *out, ws, tile_path, num_sms, stream);
}

int gf_splat_backward(const gf_splat_desc *desc, const gf_splat_inputs *in, const gf_splat_grads *gr,
                      void *workspace, size_t workspace_bytes, gf_stream_t stream_) {
    int rc = check_desc(desc);
    if (rc != GF_OK) return rc;
    rc = check_inputs(desc, in);
    if (rc != GF_OK) return rc;
    GF_REQUIRE(gr != nullptr, GF_ERR_INVALID_ARG, "splat backward: grads struct is NULL");
    if (desc->G == 0) return GF_OK;
    GF_REQUIRE(gr->means_grad && gr->opacity_grad && gr->semantics_grad, GF_ERR_INVALID_ARG,
               "splat backward: output gradient pointers must not be NULL");
    if (in->cov)
        GF_REQUIRE(gr->cov_grad != nullptr, GF_ERR_INVALID_ARG, "splat backward: cov_grad is NULL");
    else
        GF_REQUIRE(gr->scales_grad && gr->rotations_grad, GF_ERR_INVALID_ARG,
                   "splat backward: scales_grad / rotations_grad must not be NULL when the inverse covariance is "
                   "built from scales + rotations");
    if (desc->N > 0) {
        GF_REQUIRE(gr->logits_grad != nullptr, GF_ERR_INVALID_ARG, "splat backward: logits_grad is NULL");
        if (desc->variant == GF_SPLAT_PROB)
            GF_REQUIRE(gr->bin_logits_grad && gr->density_grad && gr->logits && gr->bin_logits && gr->probability,
                       GF_ERR_INVALID_ARG, "splat(prob) backward: upstream grads and saved outputs must not be NULL");
    }
    const size_t need = backward_workspace_bytes(*desc);
    GF_REQUIRE(workspace != nullptr && workspace_bytes >= need, GF_ERR_WORKSPACE,
               "splat backward: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    GF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, GF_ERR_WORKSPACE,
               "splat backward: workspace must be 256-byte aligned");
    int num_sms = 1;
    rc = num_sms_of_current_device(&num_sms);
    if (rc != GF_OK) return rc;
    return launch_backward(*desc, *in, *gr, workspace, num_sms, static_cast<cudaStream_t>(stream_));
}

int gf_splat_read_flags(const void *workspace, gf_stream_t stream_, uint32_t *host_flags) {
    GF_REQUIRE(workspace != nullptr && host_flags != nullptr, GF_ERR_INVALID_ARG, "read_flags: NULL argument");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    GF_CUDA_TRY(cudaMemcpyAsync(host_flags, workspace, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    GF_CUDA_TRY(cudaStreamSynchronize(stream));
    return GF_OK;
}

static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static int check_daf(const gf_daf_desc *d) {
    GF_REQUIRE(d != nullptr, GF_ERR_INVALID_ARG, "daf: desc is NULL");
    GF_REQUIRE(d->batch >= 0 && d->num_pts >= 0 && d->num_cams > 0 && d->num_feat > 0 && d->num_embeds > 0 &&
                   d->num_scale > 0 && d->num_groups > 0,
               GF_ERR_INVALID_ARG, "daf: non-positive dimension");
    GF_REQUIRE(d->num_embeds % d->num_groups == 0, GF_ERR_INVALID_ARG, "daf: num_embeds %% num_groups != 0");
    GF_REQUIRE(d->num_scale <= 8, GF_ERR_UNSUPPORTED, "daf: more than 8 pyramid levels");
    return GF_OK;
}

int gf_daf_forward(const gf_daf_desc *desc, const float *feat, const int32_t *shape, const int32_t *start,
                   const float *loc, const float *weights, float *output, gf_stream_t stream_) {
    int rc = check_daf(desc);
    if (rc != GF_OK) return rc;
    if (static_cast<long long>(desc->batch) * desc->num_pts == 0) return GF_OK;
    GF_REQUIRE(feat && shape && start && loc && weights && output, GF_ERR_INVALID_ARG, "daf forward: NULL pointer");
    GF_REQUIRE(aligned16(feat) && aligned16(output), GF_ERR_INVALID_ARG,
               "daf forward: mc_ms_feat and output must be 16-byte aligned (the kernels use 16-byte vector accesses)");
    int num_sms = 1;
    rc = num_sms_of_current_device(&num_sms);
    if (rc != GF_OK) return rc;
    return launch_daf_forward(*desc, feat, shape, start, loc, weights, output, num_sms,
                              static_cast<cudaStream_t>(stream_));
}

int gf_daf_backward(const gf_daf_desc *desc, const float *feat, const int32_t *shape, const int32_t *start,
                    const float *loc, const float *weights, const float *grad_output, float *grad_feat,
                    float *grad_loc, float *grad_weights, gf_stream_t stream_) {
    int rc = check_daf(desc);
    if (rc != GF_OK) return rc;
    if (static_cast<long long>(desc->batch) * desc->num_pts == 0) return GF_OK;
    GF_REQUIRE(feat && shape && start && loc && weights && grad_output && grad_feat && grad_loc && grad_weights,
               GF_ERR_INVALID_ARG, "daf backward: NULL pointer");
    GF_REQUIRE(aligned16(feat) && aligned16(grad_output) && aligned16(grad_feat), GF_ERR_INVALID_ARG,
               "daf backward: mc_ms_feat, grad_output and grad_mc_ms_feat must be 16-byte aligned");
    int num_sms = 1;
    rc = num_sms_of_current_device(&num_sms);
    if (rc != GF_OK) return rc;
    return launch_daf_backward(*desc, feat, shape, start, loc, weights, grad_output, grad_feat, grad_loc,
                               grad_weights, num_sms, static_cast<cudaStream_t>(stream_));
}

static int check_daf_fused(const gf_daf_fused_desc *fd) {
    GF_REQUIRE(fd != nullptr, GF_ERR_INVALID_ARG, "daf fused: desc is NULL");
    int rc = check_daf(&fd->d);
    if (rc != GF_OK) return rc;
    GF_REQUIRE(fd->pts_per_anchor >= 1, GF_ERR_INVALID_ARG, "daf fused: pts_per_anchor < 1");
    GF_REQUIRE(fd->d.num_pts % fd->pts_per_anchor == 0, GF_ERR_INVALID_ARG,
               "daf fused: num_pts=%d is not a multiple of pts_per_anchor=%d", fd->d.num_pts, fd->pts_per_anchor);
    GF_REQUIRE(daf_fused_supported(fd->d, fd->pts_per_anchor), GF_ERR_UNSUPPORTED,
               "daf fused: shape not supported by the fused kernel (C=%d, groups=%d, cams*levels=%d); use gf_daf_forward",
               fd->d.num_embeds, fd->d.num_groups, fd->d.num_cams * fd->d.num_scale);
    return GF_OK;
}

int gf_daf_fused_supported(const gf_daf_fused_desc *fd) {
    if (fd == nullptr || check_daf(&fd->d) != GF_OK || fd->pts_per_anchor < 1) return 0;
    return daf_fused_supported(fd->d, fd->pts_per_anchor) ? 1 : 0;
}

int gf_daf_fused_forward(const gf_daf_fused_desc *fd, const float *feat, const int32_t *shape, const int32_t *start,
                         const float *loc, const float *logits, const uint8_t *point_mask, const uint8_t *weight_mask,
                         float *output, float *stats, gf_stream_t stream_) {
    int rc = check_daf_fused(fd);
    if (rc != GF_OK) return rc;
    if (static_cast<long long>(fd->d.batch) * fd->d.num_pts == 0) return GF_OK;
    GF_REQUIRE(feat && shape && start && loc && logits && output && stats, GF_ERR_INVALID_ARG,
               "daf fused forward: NULL pointer");
    GF_REQUIRE(aligned16(feat) && aligned16(output), GF_ERR_INVALID_ARG,
               "daf fused forward: mc_ms_feat and output must be 16-byte aligned");
    int num_sms = 1;
    rc = num_sms_of_current_device(&num_sms);
    if (rc != GF_OK) return rc;
    return launch_daf_fused_forward(fd->d, fd->pts_per_anchor, feat, shape, start, loc, logits, point_mask, weight_mask,
                                    output, stats, num_sms, static_cast<cudaStream_t>(stream_));
}

int gf_daf_fused_backward(const gf_daf_fused_desc *fd, const float *feat, const int32_t *shape, const int32_t *start,
                          const float *loc, const float *logits, const uint8_t *point_mask, const uint8_t *weight_mask,
                          const float *stats, const float *output, const float *grad_output, float *grad_feat,
                          float *grad_loc, float *grad_logits, gf_stream_t stream_) {
    int rc = check_daf_fused(fd);
    if (rc != GF_OK) return rc;
    if (static_cast<long long>(fd->d.batch) * fd->d.num_pts == 0) return GF_OK;
    GF_REQUIRE(feat && shape && start && loc && logits && stats && output && grad_output && grad_feat && grad_loc &&
                   grad_logits,
               GF_ERR_INVALID_ARG, "daf fused backward: NULL pointer");
    GF_REQUIRE(aligned16(feat) && aligned16(output) && aligned16(grad_output) && aligned16(grad_feat), GF_ERR_INVALID_ARG,
               "daf fused backward: mc_ms_feat, output, grad_output and grad_mc_ms_feat must be 16-byte aligned");
    int num_sms = 1;
    rc = num_sms_of_current_device(&num_sms);
    if (rc != GF_OK) return rc;
    return launch_daf_fused_backward(fd->d, fd->pts_per_anchor, feat, shape, start, loc, logits, point_mask, weight_mask,
                                     stats, output, grad_output, grad_feat, grad_loc, grad_logits, num_sms,
                                     static_cast<cudaStream_t>(stream_));
}

int gf_daf_format(const gf_daf_format_desc *desc, float *const *maps, float *table, int inverse, gf_stream_t stream_) {
    GF_REQUIRE(desc && maps && table, GF_ERR_INVALID_ARG, "daf format: NULL argument");
    GF_REQUIRE(desc->num_scale >= 1 && desc->num_scale <= GF_DAF_MAX_LEVELS, GF_ERR_UNSUPPORTED,
               "daf format: num_scale=%d outside [1,%d]", desc->num_scale, GF_DAF_MAX_LEVELS);
    GF_REQUIRE(desc->batch_cams >= 0 && desc->num_embeds >= 0, GF_ERR_INVALID_ARG, "daf format: negative size");
    long long rows = 0;
    for (int l = 0; l < desc->num_scale; ++l) {
        GF_REQUIRE(desc->hw[l] >= 0, GF_ERR_INVALID_ARG, "daf format: negative level size");
        GF_REQUIRE(maps[l] || desc->hw[l] == 0, GF_ERR_INVALID_ARG, "daf format: NULL map pointer");
        rows += desc->hw[l];
    }
    GF_REQUIRE(rows < (1ll << 31), GF_ERR_UNSUPPORTED, "daf format: too many rows");
    GF_REQUIRE(aligned16(table), GF_ERR_INVALID_ARG, "daf format: table must be 16-byte aligned");
    for (int l = 0; l < desc->num_scale; ++l)
        GF_REQUIRE(aligned16(maps[l]), GF_ERR_INVALID_ARG, "daf format: map %d must be 16-byte aligned", l);
    return gf::launch_daf_format(*desc, maps, table, inverse != 0, static_cast<cudaStream_t>(stream_));
}

size_t gf_occ_loss_workspace_bytes(const gf_occ_loss_desc *desc) {
    if (occ_loss_check(desc) != GF_OK) return 0;
    return occ_loss_workspace_bytes(*desc);
}

int gf_occ_loss_forward(const gf_occ_loss_desc *desc, const float *pred, const uint8_t *labels, const uint8_t *mask,
                        const float *class_weights, float *loss3, float *grad_pred, uint32_t *status, void *workspace,
                        size_t workspace_bytes, gf_stream_t stream_) {
    int rc = occ_loss_check(desc);
    if (rc != GF_OK) return rc;
    GF_REQUIRE(loss3 != nullptr, GF_ERR_INVALID_ARG, "occ_loss: loss3 is NULL");
    if (static_cast<long long>(desc->B) * desc->N > 0)
        GF_REQUIRE(pred && labels, GF_ERR_INVALID_ARG, "occ_loss: pred / labels is NULL");
    const size_t need = occ_loss_workspace_bytes(*desc);
    GF_REQUIRE(workspace != nullptr && workspace_bytes >= need, GF_ERR_WORKSPACE,
               "occ_loss: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    GF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, GF_ERR_WORKSPACE,
               "occ_loss: workspace must be 256-byte aligned");
    return occ_loss_forward(*desc, pred, labels, mask, class_weights, loss3, grad_pred, status, workspace,
                            static_cast<cudaStream_t>(stream_));
}

}  // extern "C"
