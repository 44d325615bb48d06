/*
 * include/gut_b200.h -- C ABI of the B200-native 3DGUT renderer (lib: 3dgrut_b200/libgut_b200.so).
 *
 * Drop-in boundary.  The reference's FFI for this path is pybind11 + ATen, not extern "C"
 * (threedgut_tracer/bindings.cpp:103-109): class SplatRaster{trace, trace_bwd, collect_times}.
 * This header is the raw-pointer core a maintainer binds instead (see INTEGRATION.md): every entry
 * point takes plain device/host pointers, sizes and a cudaStream_t passed as void*; no torch types.
 *
 *   gutb200_create / destroy      <- SplatRaster::SplatRaster / ~SplatRaster   (threedgut_tracer/src/splatRaster.cpp:163-182)
 *   gutb200_forward               <- SplatRaster::trace                         (src/splatRaster.cpp:184-262) -> GUTRenderer::renderForward (src/gutRenderer.cu:241-421)
 *   gutb200_backward              <- SplatRaster::traceBwd                      (src/splatRaster.cpp:264-350) -> GUTRenderer::renderBackward (src/gutRenderer.cu:423-519)
 *   gutb200_collect_times         <- SplatRaster::collectTimes                  (src/splatRaster.cpp:352-382)
 *   gutb200_forward_host/_backward_host : same calls with HOST buffers (copies inside), used for the e2e metric.
 *   gutb200_backward_compact / gutb200_sph_grad_from_views / gutb200_camera_position : view-parallel training (no reference twin).
 *   gutb200_debug_copy            : test-only read-back of the binning artefacts (tile counts, sort keys, ranges).
 *
 * Data layouts (all fp32 unless noted; identical to the reference tensors):
 *   particles [N,12] = pos3, density, quat(w,x,y,z), scale3, pad     (threedgut_tracer/tracer.py:176-178)
 *   sph       [N,48] = 16 SH coefficients x rgb                       (gaussianParticles.cuh:208-221)
 *   rays_o/d  [H,W,3] sensor space                                    (tracer.py:317-330)
 *   out_rgba  [H,W,4], out_dist [H,W], out_hits [H,W], visibility [N] (src/splatRaster.cpp:212-216)
 *   d_particles [N,12], d_sph [N,48]                                  (src/splatRaster.cpp:291-293)
 * Errors: every call returns 0 on success, non-zero on failure; gutb200_last_error() gives the message
 * (the reference logs and drops its Status codes, src/splatRaster.cpp:242,254; we surface them).
 */
#ifndef GUT_B200_H
#define GUT_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* OpenCV pinhole + global shutter (CameraModelParameters, include/3dgut/sensors/cameraModels.h:22-72).
 * Poses are world->sensor [t.xyz, q.xyzw] at shutter open / close (include/3dgut/sensors/sensors.h:33-42). */
typedef struct gutb200_camera {
    int32_t width, height;
    float principal[2];
    float focal[2];
    float radial[6];
    float tangential[2];
    float thin_prism[4];
    float pose_start[7];
    float pose_end[7];
    int32_t model;      /* TSensorModel::ModelType (sensors/cameraModels.h:59-72): 0 = OpenCV pinhole (radial[6], tangential, thin prism),
                         * 1 = OpenCV fisheye (radial[0..3] = k1..k4, max_angle; bindings.cpp:68-84), 2 = f-theta (fields below). */
    float max_angle;    /* OpenCVFisheyeProjectionParameters::maxAngle (cameraModels.h:30-35) / FThetaProjectionParameters::maxAngle */
    /* model 2 = f-theta (FThetaProjectionParameters, cameraModels.h:37-47; bindings.cpp:86-101); principal point = principal[] */
    int32_t ftheta_reference_poly;  /* 0 PIXELDIST_TO_ANGLE, 1 ANGLE_TO_PIXELDIST */
    float ftheta_bw[6];             /* pixeldist_to_angle_poly (backward) */
    float ftheta_fw[6];             /* angle_to_pixeldist_poly (forward)  */
    float ftheta_cde[3];            /* linear_cde */
    int32_t rolling_shutter;        /* 0 global shutter; 1..4 = CameraModelParameters::ShutterType + 1 (cameraModels.h:49-57): rolling
                                     * top-to-bottom, left-to-right, bottom-to-top, right-to-left.  Affects the projection only
                                     * (projectPointWithShutter, cameraProjections.cuh:218-257); rays use the mid-exposure pose like the
                                     * reference (gutRenderer.cu:266-267,406). */
} gutb200_camera;

/* Render configuration == the reference's compile-time -D constants (threedgut_tracer/setup_3dgut.py:64-95). */
typedef struct gutb200_config {
    int32_t kernel_degree;    /* GAUSSIAN_PARTICLE_KERNEL_DEGREE: 2 (3DGUT default) or 4          */
    float min_kernel_density; /* GAUSSIAN_PARTICLE_MIN_KERNEL_DENSITY                              */
    float min_alpha;          /* GAUSSIAN_PARTICLE_MIN_ALPHA                                       */
    float max_alpha;          /* GAUSSIAN_PARTICLE_MAX_ALPHA                                       */
    float min_transmittance;  /* GAUSSIAN_MIN_TRANSMITTANCE_THRESHOLD                               */
    float ut_alpha, ut_beta, ut_kappa, ut_delta;
    float ut_margin;          /* GAUSSIAN_UT_IN_IMAGE_MARGIN_FACTOR                                */
    int32_t rect_bounding, tight_opacity_bounding, tile_culling;
    int32_t global_z_order;
    int32_t enable_timings;   /* render.enable_kernel_timings (src/splatRaster.cpp:168-169); 2 = also per-stage events */
    int32_t n_rolling_shutter_iterations; /* GAUSSIAN_N_ROLLING_SHUTTER_ITERATIONS (configs/render/3dgut.yaml:18): 5 */
    int32_t k_buffer_size;    /* GAUSSIAN_K_BUFFER_SIZE (render.splat.k_buffer_size): 0 = unsorted (default), 1..16 = sorted 3DGUT */
    int32_t subtile_culling;  /* ours (no reference twin), bit mask, default 7: bit 1 = exact-conservative sub-tile screens in render,
                               * bit 2 = renderBackward walks only the list entries some pixel of a sub-block accepted in the forward
                               * ("hit words"); bits 4..5 = sub-block of that walk: 0 quarter-warp (4x2 pixels), 1 half-warp (4x4),
                               * 2 whole warp (8x4); bit 0 unused.  Forward results are bit-identical with bit 1 on or off. */
} gutb200_config;

typedef struct gutb200_ctx gutb200_ctx;

void gutb200_default_config(gutb200_config* cfg);
int gutb200_create(const gutb200_config* cfg, int device, gutb200_ctx** out);
void gutb200_destroy(gutb200_ctx* ctx);
const char* gutb200_last_error(const gutb200_ctx* ctx);
const char* gutb200_version(void);

int gutb200_forward(gutb200_ctx* ctx, void* stream, const gutb200_camera* cam, int64_t n, const float* particles,
                    const float* sph, int32_t sph_degree, const float* rays_o, const float* rays_d, float* out_rgba,
                    float* out_dist, float* out_hits, float* visibility);

int gutb200_backward(gutb200_ctx* ctx, void* stream, const gutb200_camera* cam, int64_t n, const float* particles,
                     const float* sph, int32_t sph_degree, const float* rays_o, const float* rays_d,
                     const float* out_rgba, const float* d_rgba, const float* out_dist, const float* d_dist,
                     float* d_particles, float* d_sph);

/* Host-buffer variants: pinned or pageable host pointers; H2D/D2H copies happen inside on the context's stream. */
/* View-parallel training (ours, no reference twin -- the reference is single-GPU): the [N,48] SH gradient row of a view is the outer
 * product basis16(direction particle <- sensor) x g, g = masked dL/d(radiance) of the particle in that view.  gutb200_backward_compact
 * emits g ([N,4], .w = 0) instead of the row; ranks all-gather the g's and all-reduce d_particles (16 + 48 instead of 240 bytes per
 * particle on the wire), then gutb200_sph_grad_from_views rebuilds sum_v basis(direction_v) x g_v on every rank in view order.
 * view_positions_host: [views,3] sensor positions from gutb200_camera_position (host pointers); d_radiance_all: [views,N,4] device. */
int gutb200_backward_compact(gutb200_ctx* ctx, void* stream, const gutb200_camera* cam, int64_t n, const float* particles,
                             const float* sph, int32_t sph_degree, const float* rays_o, const float* rays_d, const float* out_rgba,
                             const float* d_rgba, const float* out_dist, const float* d_dist, float* d_particles, float* d_radiance);
int gutb200_sph_grad_from_views(gutb200_ctx* ctx, void* stream, int64_t n, const float* particles, int32_t sph_degree, int32_t views,
                                const float* view_positions_host, const float* d_radiance_all, float* d_sph);
int gutb200_camera_position(const gutb200_camera* cam, float* pos3);

/* Optimizer step (SURVEY.md 8f row 2).  No context: plain launches on `stream` of the current device; 0 on success.
 * gutb200_selective_adam_update replaces selective_adam_update of the reference's optimizer plugin
 * (threedgrut/optimizers/optimizers.cu:49-108, optimizers.cpp): param/grad/exp_avg/exp_avg_sq [n,m] fp32, visibility [n] bytes
 * (bool), Adam without bias correction on the visible rows.  visibility == NULL updates every row.
 * gutb200_gaussian_adam_step (ours) updates the six raw parameter tensors of the SH model in ONE launch from the renderer's
 * gradients: params6 / exp_avg6 / exp_avg_sq6 = {positions [n,3], density [n,1], rotation [n,4], scale [n,3], features_albedo [n,3],
 * features_specular [n,45]} (device pointers in a host array), lr6 their learning rates, d_particles [n,12] and d_sph [n,48] the
 * gradients w.r.t. the ACTIVATED values as gutb200_backward writes them; the activation chain rule (sigmoid / exp / normalize,
 * threedgrut/model/model.py:102-118) is applied inside.  selective = 0: torch.optim.Adam with bias correction at `step` (>= 1,
 * model.py:807-810); selective = 1: the plugin's rule on rows with visibility != 0 (visibility = the renderer's [n] float output). */
int gutb200_selective_adam_update(void* stream, float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                                  const uint8_t* visibility, float lr, float b1, float b2, float eps, int64_t n, int64_t m);
int gutb200_gaussian_adam_step(void* stream, int64_t n, float* const* params6, float* const* exp_avg6, float* const* exp_avg_sq6,
                               const float* lr6, float b1, float b2, float eps, int64_t step, int32_t selective, const float* d_particles,
                               const float* d_sph, const float* visibility);
/* gutb200_gaussian_adam_step plus the opacity and scale regularisers of the reference's loss (threedgrut/trainer.py:722-739):
 *   loss += lambda_opacity * mean|sigmoid(density)|  +  lambda_scale * mean|exp(scale)|      (means over [n,1] and [n,3])
 * Their gradients are added to the density / scale gradients inside the launch, once per call: called after the view-parallel
 * exchange, every replica adds the same term.  Selective mode masks rows exactly as gutb200_gaussian_adam_step does (invisible rows get
 * no update, as the reference's SelectiveAdam drops their regulariser gradient too).  reg_loss2: NULL, or a device float[2] that is
 * zeroed on `stream` and receives (mean sigmoid(density), mean exp(scale)) of the parameters BEFORE the update; the summation order,
 * and so the last bits of these two values, may vary between runs, the parameters never do. */
int gutb200_gaussian_adam_step_reg(void* stream, int64_t n, float* const* params6, float* const* exp_avg6, float* const* exp_avg_sq6,
                                   const float* lr6, float b1, float b2, float eps, int64_t step, int32_t selective, const float* d_particles,
                                   const float* d_sph, const float* visibility, float lambda_opacity, float lambda_scale, float* reg_loss2);

/* Image loss of the training step and its gradient (SURVEY.md 8f row 3): loss = lambda_l1 mean|x - y| + lambda_ssim (1 - SSIM(x, y))
 * (threedgrut/trainer.py:698-739, model/losses.py:20-33 -> fused_ssim(..., padding="valid"), third-party fused-ssim @ 1272e21).
 * pred_rgba [H,W,4] (the renderer's output, channels 0..2 are used), target_rgb [H,W,3], d_rgba [H,W,4] = d loss / d pred with a zero
 * alpha gradient (directly the d_rgba of gutb200_backward), sums2 [2] device floats = (sum |x - y|, sum of the SSIM map over the valid
 * region): l1 = sums2[0] / (3 H W), ssim = sums2[1] / (3 (H-10) (W-10)).  scratch: gutb200_image_loss_scratch_bytes(H, W) device bytes. */
size_t gutb200_image_loss_scratch_bytes(int32_t height, int32_t width);
int gutb200_image_loss(void* stream, int32_t height, int32_t width, const float* pred_rgba, const float* target_rgb, float lambda_l1,
                       float lambda_ssim, void* scratch, float* d_rgba, float* sums2);

int gutb200_forward_host(gutb200_ctx* ctx, const gutb200_camera* cam, int64_t n, const float* particles,
                         const float* sph, int32_t sph_degree, const float* rays_o, const float* rays_d,
                         float* out_rgba, float* out_dist, float* out_hits, float* visibility);
int gutb200_backward_host(gutb200_ctx* ctx, const gutb200_camera* cam, int64_t n, const float* particles,
                          const float* sph, int32_t sph_degree, const float* rays_o, const float* rays_d,
                          const float* out_rgba, const float* d_rgba, const float* out_dist, const float* d_dist,
                          float* d_particles, float* d_sph);

/* Statistics of the last forward: N, I (= particle/tile intersections), V (= particles with tiles_count>0), T tiles. */
int gutb200_last_stats(gutb200_ctx* ctx, int64_t* n, int64_t* num_intersections, int64_t* num_visible, int64_t* num_tiles);

/* Test-only read-back (synchronises).  `what`: */
enum {
    GUTB200_DBG_TILES_COUNT = 0,   /* u32 [N]   */
    GUTB200_DBG_SORTED_KEYS = 1,   /* u64 [I]   */
    GUTB200_DBG_SORTED_VALUES = 2, /* u32 [I]   */
    GUTB200_DBG_TILE_RANGES = 3,   /* u32 [T,2] */
    GUTB200_DBG_DEPTH = 4,         /* f32 [N]   */
    GUTB200_DBG_RGB = 5,           /* f32 [N,3] (unclamped precomputed radiance) */
    GUTB200_DBG_PROJ = 6           /* f32 [N,8] = centre2, extent2, conic3, opacity */
};
int gutb200_debug_copy(gutb200_ctx* ctx, int what, void* host_dst, size_t bytes);

/* Mean device time (ms) of the forward / backward calls since the last collect (needs enable_timings). */
int gutb200_collect_times(gutb200_ctx* ctx, float* forward_ms, float* backward_ms);

/* Change the timing level of a live context: 0 off, 1 forward/backward events, 2 also per-stage events. */
int gutb200_set_timings(gutb200_ctx* ctx, int level);

/* Mean device time (ms) per stage since the last collect (needs enable_timings >= 2); order:
 * project, scan, expand, sort, tile_ranges, render, render_backward, project_backward. */
int gutb200_collect_stage_times(gutb200_ctx* ctx, float* mean_ms /*[8]*/);

/* Measurement helpers (debug, synchronise; never on the render path).
 * work counters of the last forward (unsorted path): counters16 = { tests_ref: (pixel, entry) pairs the reference's per-pixel loop
 * evaluates, tests_exec: lane-level exact tests our forward ran after sub-tile screening, hits: accepted pairs (the adjoint's work),
 * fwd_iters / hit_iters: warp iterations of the forward / of the backward, screens: lane-level sub-tile screens, bwd_lanes: live lanes
 * summed over those, iters16 / iters8: backward iterations when half- / quarter-warps walk their own entries in lockstep, sub16_hits /
 * sub8_hits: (half- / quarter-warp, entry) pairs with a hit = gradient rows flushed, 0... }.  particles / rays_* are the device pointers
 * the forward was called with. */
int gutb200_debug_work_counters(gutb200_ctx* ctx, const float* particles, const float* rays_o, const float* rays_d, uint64_t* counters16);
/* FP32 FMA throughput of the device in TFLOP/s (micro-benchmark, best of `repeats` launches): the roofline_fp32 denominator. */
int gutb200_debug_fma_peak(gutb200_ctx* ctx, int repeats, float* tflops);

/* Number of kernels this library launched since the context was created (bench.py's gpu_launches). */
int64_t gutb200_launch_count(const gutb200_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif
