/* skyrim_b200 — C-ABI of the B200-native step operators behind the Skyrim rollout path.
 *
 * The reference has no FFI of its own: its seam is the Python earth2mip ``TimeLoop``
 * protocol consumed at
 *   /root/reference/skyrim/core/models/utils.py:34-40   (for k,(time,output,_) in model(time,x))
 *   /root/reference/skyrim/core/models/pangu.py:45-46   (pangu.load(registry.get_model(...)))
 *   /root/reference/skyrim/core/models/fourcastnet_v2.py:36-37
 * Each entry point below replaces what one of those call sites reaches inside the
 * ONNXRuntime / earth2mip back-ends.  Plain pointers and sizes only; no Python or torch
 * types cross this boundary.  Device pointers are raw CUDA device addresses (the Python
 * host passes ``tensor.data_ptr()``), ``stream`` is a ``cudaStream_t`` cast to void*.
 *
 * Conventions: every function returns 0 on success, <0 on error (never exits);
 * sky_last_error() returns a thread-local message.  A handle is bound to one device and is
 * not thread-safe; distinct handles on distinct devices may be driven concurrently.
 * The caller owns state / workspace buffers; the engine owns its device weights.
 */
#ifndef SKYRIM_B200_H
#define SKYRIM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SKY_ABI_VERSION 1

enum { SKY_MODEL_PANGU6 = 1, SKY_MODEL_SFNO73 = 2, SKY_MODEL_GRAPHCAST = 3, SKY_MODEL_AFNO26 = 4 };
enum { SKY_OK = 0, SKY_ERR_ARG = -1, SKY_ERR_CUDA = -2, SKY_ERR_STATE = -3, SKY_ERR_NOMEM = -4 };

/* Pangu-Weather 6-h operator shape (patch (2,4,4) and window (2,6,12) are fixed).
 * Replaces the shape information baked into pangu_weather_6.onnx (pangu.py:46). */
typedef struct {
  int32_t nlat, nlon;      /* 721, 1440 */
  int32_t n_levels;        /* 13 */
  int32_t dim;             /* 192 */
  int32_t depths[4];       /* 2,6,6,2 */
  int32_t heads[4];        /* 6,12,12,6 */
  float ln_eps;            /* 1e-5 */
  float mask_value;        /* -100 */
} sky_pangu_config_t;

/* SFNO (FourCastNet-v2-small) operator shape; replaces the hyper-parameters read from the
 * fcnv2_sm checkpoint (fourcastnet_v2.py:37). */
typedef struct {
  int32_t nlat, nlon;      /* 721, 1440 */
  int32_t n_channels;      /* 73 */
  int32_t embed;           /* 384 */
  int32_t layers;          /* 8 */
  int32_t scale_factor;    /* 3 */
  int32_t mlp_ratio;       /* 2 */
  float eps;               /* instance-norm epsilon */
} sky_sfno_config_t;

/* GraphCast (operational 0.25 deg / 13 levels) operator shape; replaces what
 * graphcast.load_time_loop_operational reads from the checkpoint and builds as mesh tables
 * (/root/reference/skyrim/core/models/graphcast.py:51-54).  The graph itself (edge lists, edge / node features)
 * travels in the weight arena as entries named "graph.*" (skyrim_b200/icomesh.py); the counts below size them. */
typedef struct {
  int32_t nlat, nlon;      /* 721, 1440 */
  int32_t n_mesh;          /* 40962 multimesh nodes (icosahedron refined 6 times) */
  int32_t n_mesh_edges;    /* 327660 directed multimesh edges, sorted by receiver */
  int32_t n_g2m_edges;     /* grid2mesh edges, sorted by receiver (mesh node) */
  int32_t latent;          /* 512 */
  int32_t layers;          /* 16 processor layers */
  int32_t n_state;         /* 83 channels per time slice: 82 prognostic + toa radiation (graphcast.py:17-41) */
  int32_t n_prog;          /* 82 */
  int32_t n_static;        /* 2: geopotential at the surface, land-sea mask */
  int32_t dt_hours;        /* 6 */
  float ln_eps;            /* 1e-5 */
} sky_graphcast_config_t;
/* Arena entries of a GraphCast model (all fp32; index tables hold exact integers < 2^24):
 *   norm.mean, norm.std, norm.diff_std (n_state each), static.fields (n_static, nlat, nlon)
 *   <mlp>.w1 (512, fan_in), .b1 (512), .w2 (fan_out, 512), .b2 (fan_out), .ln.g / .ln.b (fan_out; not for dec.out) for <mlp> in
 *     enc.grid_embed (184), enc.mesh_embed (3), enc.g2m_edge_embed (4), enc.g2m_edge (1536), enc.g2m_mesh (1024), enc.g2m_grid (512),
 *     proc.edge_embed (4), proc<i>.edge (1536), proc<i>.node (1024) for i < layers, dec.m2g_edge_embed (4), dec.m2g_edge (1536),
 *     dec.m2g_grid (1024), dec.out (512 -> n_state)          [first-layer input order: edge | sender | receiver, node | aggregate]
 *   graph.mesh.senders / .receivers (n_mesh_edges, sorted by receiver), graph.mesh.ptr (n_mesh + 1), graph.mesh.edge_feat (n_mesh_edges, 4),
 *   graph.mesh.node_feat (n_mesh, 3), graph.g2m.senders / .receivers / .ptr / .edge_feat (same, grid -> mesh),
 *   graph.m2g.senders (3 * nlat * nlon, k-major: edge k of grid point g at k * n_grid + g), graph.m2g.edge_feat (3 * n_grid, 4),
 *   graph.grid.coslat (nlat), graph.grid.sinlon / .coslon (nlon)
 * (skyrim_b200/weights.py::graphcast_param_shapes, skyrim_b200/icomesh.py::graph_arena_entries build exactly this set). */

/* FourCastNet v1 (AFNONet) operator shape; replaces the hyper-parameters earth2mip's networks.fcn package reads
 * (/root/reference/skyrim/core/models/fourcastnet.py:build_model). */
typedef struct {
  int32_t nlat, nlon;      /* 720, 1440 (no south-pole row) */
  int32_t n_channels;      /* 26 */
  int32_t patch;           /* 8 */
  int32_t embed;           /* 768 */
  int32_t depth;           /* 12 */
  int32_t num_blocks;      /* 8 spectral blocks of embed / num_blocks = 96 */
  int32_t mlp_ratio;       /* 4 */
  float sparsity;          /* softshrink lambda, 0.01 */
  float hard_thresholding_fraction;  /* 1.0 */
  float ln_eps;            /* 1e-6 */
} sky_afno_config_t;
/* Arena entries of a FourCastNet model (all fp32, upstream names):
 *   norm.mean, norm.std (n_channels), patch_embed.proj.weight (embed, n_channels, 8, 8), patch_embed.proj.bias (embed),
 *   pos_embed (1, (nlat / 8) * (nlon / 8), embed), head.weight (n_channels * 64, embed) [columns (p1, p2, c)], and per block i
 *   blocks.<i>.norm1.weight / .bias, blocks.<i>.norm2.weight / .bias (embed), blocks.<i>.filter.w1 / .w2 (2, num_blocks, 96, 96)
 *   [re / im, block, in, out], blocks.<i>.filter.b1 / .b2 (2, num_blocks, 96), blocks.<i>.mlp.fc1.weight (mlp_ratio * embed,
 *   embed), .fc1.bias, blocks.<i>.mlp.fc2.weight (embed, mlp_ratio * embed), .fc2.bias
 * (skyrim_b200/weights.py::fcn_param_shapes builds exactly this set). */

/* one named fp32 tensor inside a flat weight arena */
typedef struct {
  char name[96];
  uint64_t offset;         /* in floats from the arena start */
  uint64_t count;          /* number of floats */
} sky_param_desc_t;

typedef struct sky_model sky_model_t;

/* Everything but these entry points is built with hidden visibility: the product and the development build of the
 * library can then live in one process without their template statics / inline functions being merged by the
 * dynamic linker (round 2: a shared `configured` flag made the second library skip its shared-memory opt-in). */
#if defined(__GNUC__)
#define SKY_API __attribute__((visibility("default")))
#else
#define SKY_API
#endif

SKY_API int sky_abi_version(void);
SKY_API const char* sky_last_error(void);

/* model_kind: SKY_MODEL_*; cfg points at the matching sky_*_config_t. */
SKY_API int sky_model_create(sky_model_t** out, int model_kind, const void* cfg, size_t cfg_bytes, int device);

/* Load (copy + repack for the tensor cores) the fp32 weight arena.  `arena` is a host
 * pointer (arena_on_device = 0) or a device pointer on the model's device (= 1, e.g. the
 * buffer that received the one-time NCCL broadcast).  The caller keeps ownership.
 * Replaces ONNX initialiser loading / torch.load in the reference back-ends. */
SKY_API int sky_model_load_weights(sky_model_t* m, const float* arena, uint64_t n_floats,
                           const sky_param_desc_t* manifest, int32_t n_params, int32_t arena_on_device,
                           void* stream);

/* scratch bytes one step needs for `batch` members */
SKY_API size_t sky_model_workspace_bytes(const sky_model_t* m, int32_t batch);

/* One 6-h step for `batch` independent members: x_in, x_out are device fp32
 * (batch, C, nlat, nlon), may not alias.  Asynchronous and stream-ordered; no host sync.
 * Replaces one `next()` of the TimeLoop generator (utils.py:34). */
SKY_API int sky_model_step(sky_model_t* m, const float* x_in, float* x_out, int32_t batch, void* workspace,
                   size_t workspace_bytes, void* stream);

/* Valid time (unix seconds, UTC) of the LAST time slice of the state the next sky_model_step starts from.  Operators
 * with time-dependent forcings (GraphCast: toa radiation, year / day progress) keep this clock on the device and advance
 * it by one step per sky_model_step, so a rollout sets it once; the others ignore it.
 * Replaces the `time` argument of `stepper.initialize(x, time)` (graphcast.py:110). */
SKY_API int sky_model_set_clock(sky_model_t* m, double unix_seconds, void* stream);

/* Top-of-atmosphere incident solar radiation of the hour ending at `unix_seconds` [J m^-2] on the (nlat, nlon) grid
 * (lat 90 -> -90, lon 0 -> 360): the forcing channel the reference calls "tp06" (graphcast.py:16,40).  `out` is device
 * fp32 (nlat * nlon).  Used to fill that channel of an initial condition. */
SKY_API int sky_toa_radiation(float* out, int32_t nlat, int32_t nlon, double unix_seconds, void* stream);

/* Intermediate tensor taps for kernel-level parity tests: after a step, copy the named
 * internal buffer ("embed"/"tokens1"/"tokens2"...) of the LAST step into dst (device fp32). */
SKY_API int sky_model_debug_copy(sky_model_t* m, const char* what, float* dst, uint64_t max_floats, void* workspace,
                         int32_t batch, void* stream);

/* Switches of a handle (never read from the environment).  "fp32_stream" = 1 (Pangu) keeps the token stream as fp32 rows beside
 * its fp16 operand image instead of the default image-only stream: 1.1 ms per step slower, one rounding per residual add less
 * (DESIGN.md section 3).  Test taps: "stop_after" = n makes step() return after
 * stage n (0 embed, 1 layer0, 2 down, 3 layer1, 4 layer2, 5 up, 6 layer3; 99 = run the whole step) so that
 * sky_model_debug_copy can read the intermediate token buffers. */
SKY_API int sky_model_debug_set(sky_model_t* m, const char* key, int64_t value);

/* x[m, c, :, :] += amp * sigma[c] * N(0,1), Philox4x32-10 keyed by (seed, member0 + m):
 * perturbed-IC ensemble members (new functionality; the reference's only perturbation
 * helper is the single-point edit at models/utils.py:70-92). */
SKY_API int sky_perturb_ic(float* x, const float* sigma_c, float amp, uint64_t seed, int32_t member0,
                   int32_t members, int32_t channels, int64_t plane, void* stream);

/* Per-kernel-family device timing (CUDA events recorded on the launching stream around the
 * launches whose family bit is set in tag_mask).  profile_end synchronises on the recorded
 * events and returns the summed milliseconds and launch counts per family.  Used by bench.py
 * for the live roofline figure; off by default (no events are recorded). */
SKY_API int sky_model_profile_begin(sky_model_t* m, uint64_t tag_mask);
SKY_API int sky_model_profile_end(sky_model_t* m, double* ms_per_tag, uint64_t* launches_per_tag, int32_t n_tags);
SKY_API int sky_profile_tag_count(void);
SKY_API const char* sky_profile_tag_name(int32_t tag);

/* how many kernels this library has launched since load (bench.py's gpu_launches) */
SKY_API uint64_t sky_launch_count(void);

SKY_API int sky_model_destroy(sky_model_t* m);

#ifdef __cplusplus
}
#endif
#endif /* SKYRIM_B200_H */
