/*
 * fluid.h — C ABI of libfluid_b200: the drop-in boundary for the simulation path of
 * PavelDoGreat/WebGL-Fluid-Simulation (script.js step()/splat()/config).
 *
 * The reference has no FFI: its "interface" is a set of global JS functions and a global
 * `config` object inside one classic <script> (index.html:222).  Every entry point below cites
 * the reference construct (script.js = "S") it replaces; INTEGRATION.md shows the N-API / ctypes
 * binding a maintainer would add on the reference side.
 *
 * Conventions (all from the reference):
 *   - fields are row-major, x fastest, ROW 0 = BOTTOM (GL texture convention, S:452, S:1531);
 *   - velocity is float2 interleaved (RG texture, S:994-997), dye is float4 interleaved
 *     (RGBA texture, S:989-992), pressure/divergence/curl are float (R texture, S:999-1001);
 *   - uv of cell (i,j) = ((i+.5)/W, (j+.5)/H) (S:452); sampling is CLAMP_TO_EDGE (S:1051-1052);
 *   - velocity is measured in sim-texels per second (S:777 with texelSize = 1/W).
 *   - storage is fp32 (BASELINE.json asks fp32; the reference stores fp16, S:138-147).
 *
 * Error convention: every int-returning call returns FLUID_OK (0) or a negative fluid_status;
 * fluid_last_error() returns the message.  There is NO CPU fallback anywhere in this library:
 * without a CUDA device fluid_create() fails with FLUID_ERR_NO_DEVICE.
 *
 * Threading: a handle is single-threaded like the JS it replaces.  step/splat/pass calls enqueue
 * work on the handle's CUDA stream and return; fluid_read()/fluid_sync() block.
 */
#ifndef FLUID_B200_H
#define FLUID_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FLUID_ABI_VERSION 2

typedef struct fluid fluid_t; /* opaque; owns device buffers, streams, events, graphs, NCCL comm */

typedef enum fluid_status {
    FLUID_OK = 0,
    FLUID_ERR_INVALID = -1,      /* bad argument / bad field id / size mismatch            */
    FLUID_ERR_NO_DEVICE = -2,    /* no CUDA device or device is not sm_100                 */
    FLUID_ERR_CUDA = -3,         /* a CUDA runtime/driver call failed                      */
    FLUID_ERR_NCCL = -4,         /* NCCL could not be loaded or a NCCL call failed         */
    FLUID_ERR_HALO = -5,         /* multi-GPU: an advection back-trace left the ghost zone */
    FLUID_ERR_NOMEM = -6
} fluid_status;

/* Field ids.  S:950-954: `dye, velocity, divergence, curl, pressure` globals. */
typedef enum fluid_field {
    FLUID_FIELD_VELOCITY = 0,   /* velocity.read   float2  sim_w x sim_h */
    FLUID_FIELD_DYE = 1,        /* dye.read        float4  dye_w x dye_h */
    FLUID_FIELD_PRESSURE = 2,   /* pressure.read   float   sim_w x sim_h */
    FLUID_FIELD_DIVERGENCE = 3, /* divergence      float   sim_w x sim_h */
    FLUID_FIELD_CURL = 4        /* curl            float   sim_w x sim_h */
} fluid_field;

/* Scalar parameter keys = the simulation keys of the reference `config` object (S:59-69, S:73).
 * The reference reads config live on every call; the host mirror pushes changed keys with
 * fluid_set_param() before step()/splat(). */
typedef enum fluid_param {
    FLUID_DENSITY_DISSIPATION = 0,  /* S:63 default 1     */
    FLUID_VELOCITY_DISSIPATION = 1, /* S:64 default 0.2   */
    FLUID_PRESSURE = 2,             /* S:65 default 0.8   */
    FLUID_PRESSURE_ITERATIONS = 3,  /* S:66 default 20    */
    FLUID_CURL = 4,                 /* S:67 default 30    */
    FLUID_SPLAT_RADIUS = 5,         /* S:68 default 0.25  */
    FLUID_ASPECT = 6,               /* canvas.width/canvas.height, S:1444, S:1457-1462 */
    FLUID_JACOBI_BLOCK = 7,         /* build-only tunable: max temporal-block depth, 1 = naive */
    FLUID_BACKGROUND = 8            /* what fluid_render* draws the display over (render(), S:1296-1317):
                                       0 = drawColor(BACK_COLOR); 1 = drawCheckerboard — config.TRANSPARENT on
                                       the screen (S:1325-1329, checkerboardShader S:531-547, aspect = ASPECT);
                                       2 = nothing, blending off — TRANSPARENT into a capture target          */
} fluid_param;

/* Creation flags */
#define FLUID_FLAG_UNFUSED   0x1u /* run curl / vorticity / divergence as 3 separate passes      */
#define FLUID_FLAG_NO_GRAPH  0x2u /* launch step() pass by pass instead of as one CUDA graph     */
#define FLUID_FLAG_NAIVE_JACOBI 0x4u /* one Jacobi sweep per launch (the literal S:1262 loop)    */
#define FLUID_FLAG_HALF_STORAGE 0x10u /* store every field as fp16 like the reference's textures (S:138-147,
                                         S:986-1006): fp32 arithmetic, round-to-nearest-even on every pass
                                         write, one launch per reference blit; single GPU; the ABI still
                                         speaks fp32 (fluid_read widens, fluid_write narrows).
                                         fluid_render_postfx then uses fp16 post-FX FBOs as well     */
#define FLUID_FLAG_TILED_PASSES 0x8u /* generation-1 kernels (one thread per fragment / smem tile) for
                                        curl-vorticity-divergence and gradientSubtract instead of the
                                        row-streaming ones (comparison + fallback path)              */

typedef struct fluid_config {
    int32_t sim_w, sim_h;           /* getResolution(SIM_RESOLUTION)  S:983, S:1612-1624 */
    int32_t dye_w, dye_h;           /* getResolution(DYE_RESOLUTION)  S:984              */
    float density_dissipation;      /* S:63 */
    float velocity_dissipation;     /* S:64 */
    float pressure;                 /* S:65 */
    int32_t pressure_iterations;    /* S:66 */
    float curl;                     /* S:67 */
    float splat_radius;             /* S:68 */
    float aspect;                   /* canvas.width / canvas.height; <=0 means sim_w/sim_h */
    int32_t device;                 /* CUDA ordinal; -1 = current device */
    uint32_t flags;                 /* FLUID_FLAG_* */
    int32_t jacobi_block;           /* 0 = library default */
} fluid_config;

/* Per-pass device timing of the last fluid_step() (milliseconds, CUDA events on the handle's
 * stream).  Only recorded when FLUID_FLAG_NO_GRAPH is set. */
typedef struct fluid_timing {
    float curl_vort_div_ms, jacobi_ms, gradient_ms, advect_velocity_ms, advect_dye_ms, total_ms;
    int32_t jacobi_launches;        /* kernels launched for the pressure loop */
    int32_t total_launches;         /* kernels launched by the step */
} fluid_timing;

/* ---- lifetime -------------------------------------------------------------------------------- */

/* Fills *cfg with the reference defaults (S:59-69): SIM 128, DYE 1024, dissipation 1 / 0.2,
 * PRESSURE 0.8, 20 iterations, CURL 30, SPLAT_RADIUS 0.25, aspect 1. */
void fluid_config_default(fluid_config* cfg);

/* getResolution(resolution) of S:1612-1624 for a canvas_w x canvas_h drawing buffer. */
void fluid_get_resolution(int resolution, int canvas_w, int canvas_h, int* out_w, int* out_h);

/* initFramebuffers() of S:982-1010 on first call (dye == null branch): allocates velocity, dye,
 * pressure (double-buffered) and divergence, curl; all zero, dye alpha = 1 (clearColor S:136
 * + gl.clear in createFBO S:1059). */
int fluid_create(const fluid_config* cfg, fluid_t** out);

/* Same, for rank `rank` of `world` row-slab ranks (one process per GPU).  `nccl_uid` is the
 * 128-byte ncclUniqueId obtained on rank 0 from fluid_nccl_unique_id() and broadcast by the
 * caller (torch.distributed in this repo).  The rank owns sim rows [rank*H/world,(rank+1)*H/world)
 * and the matching dye rows; fluid_read()/fluid_write() address the OWNED rows only. */
int fluid_create_slab(const fluid_config* cfg, int rank, int world, const void* nccl_uid,
                      size_t uid_bytes, fluid_t** out);
int fluid_nccl_unique_id(void* out_uid, size_t uid_bytes); /* uid_bytes must be >= 128 */

/* Optional peer-memory halo path for slab handles on one NVLink/NVSwitch box (no reference
 * counterpart).  Every rank exports a 256-byte blob (a CUDA IPC handle of its field arena + layout),
 * the launcher all-gathers them, and each rank connects to rank-1 / rank+1 (NULL at the ends).
 * Afterwards halo rows are stored straight into the neighbours' ghost rows by one kernel that
 * also carries the free/ready handshake (system-scope release/acquire flag words, bounded spins);
 * without it the NCCL send/recv path is used. */
int fluid_p2p_export(fluid_t* h, void* blob, size_t blob_bytes);   /* blob_bytes >= 256 */
int fluid_p2p_connect(fluid_t* h, const void* blob_below, const void* blob_above);
int fluid_p2p_disable(fluid_t* h);   /* back to NCCL; call on every rank if any rank failed to connect */

void fluid_destroy(fluid_t* h);

/* initFramebuffers() on a live simulation (S:982-1010 else-branches + resizeDoubleFBO S:1116-1126):
 * velocity and dye are bilinearly resampled to the new size (copyShader through a LINEAR sampler),
 * pressure / divergence / curl are re-created zeroed.
 * On a slab handle the call is collective (same sizes on every rank): ghost rows of the old velocity and
 * dye are refreshed, the rank's new rows are resampled into a new arena, and the peer-memory mappings
 * are dropped (export / connect again, or stay on NCCL).  FLUID_ERR_HALO: the factor needs more ghost
 * rows than the slab keeps. */
int fluid_resize(fluid_t* h, int sim_w, int sim_h, int dye_w, int dye_h);

/* ---- the hot path ---------------------------------------------------------------------------- */

/* step(dt) of S:1231-1294: curl -> vorticity -> divergence -> clear(pressure) ->
 * PRESSURE_ITERATIONS x Jacobi -> gradientSubtract -> advect velocity -> advect dye. */
int fluid_step(fluid_t* h, float dt);

/* splat(x, y, dx, dy, color) of S:1441-1455: velocity += exp(-|p|^2/radius)*(dx,dy), then
 * dye.rgb += exp(..)*(r,g,b), dye.a = 1; radius = correctRadius(SPLAT_RADIUS/100) (S:1457-1462). */
int fluid_splat(fluid_t* h, float x, float y, float dx, float dy, float r, float g, float b);

/* config.<KEY> = value (S:59-69).  PRESSURE_ITERATIONS / JACOBI_BLOCK are rounded to int. */
int fluid_set_param(fluid_t* h, int key, float value);
int fluid_get_param(fluid_t* h, int key, float* value);
/* Same as fluid_set_param, at the precision the JS `config` values have.  SPLAT_RADIUS and ASPECT
 * enter DOUBLE arithmetic on the host (correctRadius(config.SPLAT_RADIUS / 100.0), S:1447 +
 * S:1457-1462) before the one narrowing of gl.uniform1f; host mirrors should use this entry point. */
int fluid_set_param_f64(fluid_t* h, int key, double value);

/* ---- individual passes (the reference's one-blit-per-program granularity; used by the parity
 *      tests and by callers that drive the loop themselves).  Each reads the `.read` buffers and
 *      performs the same swap() the reference does after its blit. ------------------------------ */
int fluid_pass_curl(fluid_t* h);                       /* S:1234-1237, curlShader S:814-833        */
int fluid_pass_vorticity(fluid_t* h, float dt);        /* S:1239-1246, vorticityShader S:835-866   */
int fluid_pass_divergence(fluid_t* h);                 /* S:1248-1251, divergenceShader S:786-812  */
int fluid_pass_clear_pressure(fluid_t* h);             /* S:1253-1257, clearShader S:508-519       */
int fluid_pass_jacobi(fluid_t* h, int iters);          /* S:1259-1266, pressureShader S:868-890    */
int fluid_pass_pressure_solve(fluid_t* h);             /* clear + PRESSURE_ITERATIONS Jacobi, fused */
int fluid_pass_gradient_subtract(fluid_t* h);          /* S:1268-1273, gradientSubtractShader S:892-913 */
int fluid_pass_advect_velocity(fluid_t* h, float dt);  /* S:1275-1285, advectionShader S:746-784   */
int fluid_pass_advect_dye(fluid_t* h, float dt);       /* S:1287-1293                              */
int fluid_pass_curl_vorticity_divergence(fluid_t* h, float dt); /* the three above in one kernel  */

/* ---- data in / out ---------------------------------------------------------------------------- */

/* Element count (floats) of the rows of `field` this handle owns: w*h*channels. */
size_t fluid_field_elems(fluid_t* h, int field);
int fluid_field_dims(fluid_t* h, int field, int* w, int* h_rows, int* channels, int* row0);

/* framebufferToTexture() of S:301-307 (gl.readPixels FLOAT) generalised to every field: copies
 * the `.read` buffer to host memory (blocks until the stream has drained). */
int fluid_read(fluid_t* h, int field, float* host, size_t n_floats);
/* Test / checkpoint hook with no reference counterpart: overwrites the `.read` buffer. */
int fluid_write(fluid_t* h, int field, const float* host, size_t n_floats);

/* End-to-end form of the pressure solve for callers that keep fields in HOST memory: uploads
 * divergence and pressure, runs clear + `iters` Jacobi sweeps, downloads pressure.  All three
 * copies are inside the call (this is what bench.py's `e2e` times).  On a single-GPU handle the grid
 * is cut into row bands that are solved and downloaded while later bands still upload (same bits as
 * the one-piece solve; FLUID_E2E_BANDS=1 disables it); pass pinned buffers (fluid_host_alloc) for the
 * copies to overlap.  The divergence and pressure fields of the handle hold the uploaded divergence
 * and the result afterwards. */
int fluid_pressure_solve_host(fluid_t* h, const float* div_host, float* pressure_host_inout,
                              int iters);

/* The consumer on the far side of the path ("next" row of SURVEY §8f, partially built):
 * render(target) of S:1296-1317 with config.BLOOM = config.SUNRAYS = false and TRANSPARENT = false —
 * drawColor(BACK_COLOR) (S:1319-1323) then drawDisplay (S:1331-1348, displayShaderSource S:549-612,
 * SHADING keyword when `shading` != 0) blended ONE / ONE_MINUS_SRC_ALPHA.  Writes width*height RGBA
 * floats (row 0 = bottom, not yet quantised to 8 bits) to host memory.  back_* are BACK_COLOR / 255. */
int fluid_render(fluid_t* h, int width, int height, int shading, float back_r, float back_g,
                 float back_b, float* host_rgba, size_t n_floats);
/* On a slab handle fluid_render draws (and returns) only the band of target rows [*y0, *y1) that
 * corresponds to the dye rows the rank owns — width * (*y1 - *y0) RGBA texels — after refreshing
 * the few dye ghost rows the display / shading taps reach; on a single GPU the band is the whole
 * target.  Ranks concatenate their bands in rank order. */
int fluid_render_band(fluid_t* h, int height, int* y0, int* y1);

/* The same with the reference's desktop defaults SHADING = BLOOM = SUNRAYS = true (S:70-84):
 * applyBloom (S:1350-1394), applySunrays + blur (S:1396-1419), then the display shader with all three
 * keywords.  fx = the BLOOM_* / SUNRAYS_* keys of `config`; dither_rgb = the dw x dh RGB dithering
 * texture (LDR_LLL1_0.png / 255, first image row first, S:1128-1158).  host_bloom (bloom FBO,
 * getResolution(BLOOM_RESOLUTION) x RGBA) and host_sunrays (getResolution(SUNRAYS_RESOLUTION) x R)
 * may be NULL.  The sunrays mask is drawn into dye.write, like the reference (S:1300); dye.read is
 * untouched.  On a FLUID_FLAG_HALF_STORAGE handle the bloom FBO, the bloom pyramid, both sunrays
 * FBOs and the mask are fp16, as the reference creates them (S:1012-1043): every blit rounds its
 * output to fp16 (RN-even), and host_bloom / host_sunrays come back widened to fp32 (exactly).  The
 * dithering texture and host_rgba are fp32 in both modes.  Not available on slab handles. */
typedef struct fluid_postfx {
    int32_t bloom_iterations;    /* S:77 default 8    */
    int32_t bloom_resolution;    /* S:78 default 256  */
    double bloom_intensity;      /* S:79 default 0.8  (double: knee / curve are derived in double like the JS) */
    double bloom_threshold;      /* S:80 default 0.6  */
    double bloom_soft_knee;      /* S:81 default 0.7  */
    int32_t sunrays_resolution;  /* S:83 default 196  */
    double sunrays_weight;       /* S:84 default 1.0  */
} fluid_postfx;
int fluid_render_postfx(fluid_t* h, int width, int height, const fluid_postfx* fx, const float* dither_rgb,
                        int dw, int dh, float back_r, float back_g, float back_b, float* host_rgba,
                        size_t n_floats, float* host_bloom, float* host_sunrays);

int fluid_sync(fluid_t* h);
int fluid_timing_last(fluid_t* h, fluid_timing* out);

/* Page-locked host memory for the buffers a binding hands to fluid_read / fluid_write /
 * fluid_pressure_solve_host / fluid_render (DMA without a staging copy).  The N-API shim wraps these in
 * external ArrayBuffers (readPixels' destination, S:301-307), so it needs no CUDA headers itself. */
void* fluid_host_alloc(size_t bytes);
void fluid_host_free(void* p);

/* Device time (ms) between two fluid_mark() calls on the handle's stream; slot is 0 or 1.
 * bench.py uses it because torch.cuda.Event cannot see this library's stream. */
int fluid_mark(fluid_t* h, int slot);
int fluid_elapsed_ms(fluid_t* h, float* ms);

/* Number of CUDA kernels this handle has launched since creation (graph replays count their
 * kernel nodes). */
uint64_t fluid_launch_count(fluid_t* h);

/* Counters since creation (no reference counterpart; bench.py and the tests read them). */
typedef enum fluid_stat_key {
    FLUID_STAT_LAUNCHES = 0,         /* == fluid_launch_count                                        */
    FLUID_STAT_JACOBI_LAUNCHES = 1,  /* Jacobi kernels only (graph replays count their kernel nodes)  */
    FLUID_STAT_HALO_LAUNCHES = 2,    /* halo_push / halo_wait kernels of the peer-memory transport    */
    FLUID_STAT_HALO_EXCHANGES = 3,   /* halo exchanges issued (either transport)                      */
    FLUID_STAT_GRAPH_CAPTURES = 4,   /* step() graphs captured + instantiated                         */
    FLUID_STAT_GRAPH_LAUNCHES = 5,   /* step() graphs replayed                                        */
    FLUID_STAT_HALO_TRANSPORT_P2P = 6 /* 1 when the peer-memory halo path is active                    */
} fluid_stat_key;
uint64_t fluid_stat(fluid_t* h, int key);

/* Raw device pointer of a field's `.read` buffer (for zero-copy interop, e.g. torch.as_tensor
 * through __cuda_array_interface__); valid until the next call that swaps that field. */
void* fluid_device_ptr(fluid_t* h, int field);

const char* fluid_last_error(fluid_t* h); /* h may be NULL: last error of a failed create */
int fluid_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* FLUID_B200_H */
