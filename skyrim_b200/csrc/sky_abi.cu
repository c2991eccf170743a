// C-ABI entry points (include/skyrim_b200.h) + engine base plumbing + IC perturbation.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "engine.h"
#include "sky_common.cuh"

namespace sky {

std::atomic<uint64_t> g_launches{0};
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}

void Engine::drop_graphs() {
  for (auto& g : graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  graphs.clear();
}

int Engine::step_cached(const float* x_in, float* x_out, int batch, void* ws, size_t ws_bytes, cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (!use_graphs || prof_mask != 0 || stop_after != 99 || range_guard || cudaStreamIsCapturing(st, &cs) != cudaSuccess ||
      cs != cudaStreamCaptureStatusNone)
    return step(x_in, x_out, batch, ws, ws_bytes, st);
  GraphEntry* e = nullptr;
  for (auto& g : graphs)
    if (g.x_in == x_in && g.x_out == x_out && g.ws == ws && g.batch == batch) { e = &g; break; }
  if (e && e->exec) {
    SKY_CUDA_OK(cudaGraphLaunch(e->exec, st));
    count_launch((int)e->launches);
    return 0;
  }
  if (!e) {   // first sight of this tuple: run eagerly (opt-ins and lazy set-up happen here), remember it
    if (graphs.size() >= 8) { if (graphs.front().exec) cudaGraphExecDestroy(graphs.front().exec); graphs.erase(graphs.begin()); }
    graphs.push_back(GraphEntry{x_in, x_out, ws, batch, nullptr, 0, 1});
    return step(x_in, x_out, batch, ws, ws_bytes, st);
  }
  // second call: capture the launch sequence, instantiate, launch
  const uint64_t l0 = g_launches.load();
  if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return step(x_in, x_out, batch, ws, ws_bytes, st); }
  const int rc = step(x_in, x_out, batch, ws, ws_bytes, st);
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(st, &graph);
  if (rc || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    use_graphs = false;                       // never retry; fall back to plain launches
    return rc ? rc : step(x_in, x_out, batch, ws, ws_bytes, st);
  }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess || !exec) { cudaGetLastError(); use_graphs = false; return step(x_in, x_out, batch, ws, ws_bytes, st); }
  e->exec = exec;
  e->launches = g_launches.load() - l0;       // kernels recorded by the capture (they did not run yet)
  SKY_CUDA_OK(cudaGraphLaunch(exec, st));
  return 0;
}

Engine::~Engine() {
  drop_graphs();
  if (arena) cudaFree(arena);
  for (void* p : kept) cudaFree(p);
  for (auto e : prof_pool) cudaEventDestroy(e);
  for (auto& r : prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
}


// max |h| over an fp16 buffer -> *slot (atomic max on the bits of a non-negative float; NaN counts as +inf)
__global__ void __launch_bounds__(256) k_absmax_half(const uint4* __restrict__ p, size_t n16, float* __restrict__ slot) {
  float m = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 v = p[i];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __half2 h = *reinterpret_cast<const __half2*>(&w[j]);
      const float2 f = __half22float2(h);
      const float a = fabsf(f.x), b = fabsf(f.y);
      m = fmaxf(m, (a == a) ? a : __int_as_float(0x7f800000));
      m = fmaxf(m, (b == b) ? b : __int_as_float(0x7f800000));
    }
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, d));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(slot), __float_as_int(m));
}
int Engine::range_scan(int slot, const void* img, size_t bytes, cudaStream_t st) {
  if (!range_guard || !range_dev || !img || bytes < 16) return 0;
  const size_t n16 = bytes / 16;
  const unsigned grid = (unsigned)std::min<size_t>((n16 + 255) / 256, 148 * 8);
  k_absmax_half<<<grid, 256, 0, st>>>(reinterpret_cast<const uint4*>(img), n16, range_dev + slot);
  SKY_CUDA_OK(cudaGetLastError());
  return 0;
}

const char* ktag_name(int t) {
  static const char* n[KT_COUNT] = {"embed", "qkv", "attn", "proj", "fc1", "fc2", "mlp", "down", "up", "recover", "copy",
                                    "sfno_enc", "sfno_sht", "sfno_spec", "sfno_isht", "sfno_mlp", "sfno_dec", "sfno_misc",
                                    "gc_feat", "gc_hidden", "gc_ln", "gc_table", "gc_agg", "gc_out", "gc_misc",
                                    "fcn_embed", "fcn_ln", "fcn_spec", "fcn_mlp", "fcn_head"};
  return t >= 0 && t < KT_COUNT ? n[t] : "?";
}

cudaEvent_t Engine::prof_event() {
  if (!prof_pool.empty()) { cudaEvent_t e = prof_pool.back(); prof_pool.pop_back(); return e; }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

int Engine::prof_collect(double* ms, uint64_t* counts, int n) {
  for (int i = 0; i < n; ++i) { ms[i] = 0; counts[i] = 0; }
  for (auto& r : prof_recs) {
    SKY_CUDA_OK(cudaEventSynchronize(r.b));
    float t = 0;
    SKY_CUDA_OK(cudaEventElapsedTime(&t, r.a, r.b));
    if (r.tag < n) { ms[r.tag] += t; counts[r.tag] += 1; }
    prof_pool.push_back(r.a); prof_pool.push_back(r.b);
  }
  prof_recs.clear();
  return 0;
}

int Engine::load_arena(const float* src, uint64_t n_floats, const sky_param_desc_t* manifest, int n_params,
                       int on_device, cudaStream_t st) {
  drop_graphs();
  if (arena) { cudaFree(arena); arena = nullptr; }
  for (void* p : kept) cudaFree(p);
  kept.clear();
  loaded = false;
  SKY_CUDA_OK(cudaMalloc(&arena, n_floats * sizeof(float)));
  arena_floats = n_floats;
  SKY_CUDA_OK(cudaMemcpyAsync(arena, src, n_floats * sizeof(float),
                              on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  params.clear();
  for (int i = 0; i < n_params; ++i) {
    const sky_param_desc_t& d = manifest[i];
    if (d.offset + d.count > n_floats) { set_error("param %s exceeds the arena", d.name); return SKY_ERR_ARG; }
    if (d.offset % 4) { set_error("param %s is not 16-byte aligned in the arena", d.name); return SKY_ERR_ARG; }
    char nm[97];
    memcpy(nm, d.name, 96); nm[96] = 0;
    params[nm] = ParamView{arena + d.offset, d.count};
  }
  int rc = prepare(st);
  // the repacked operand images and the kept vectors are all the step needs: drop the fp32 arena
  // (0.26 GB for Pangu, ~4 GB for SFNO that used to stay resident next to the packed copies)
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(arena);
  arena = nullptr;
  params.clear();
  if (rc) return rc;
  SKY_CUDA_OK(e);
  loaded = true;
  return 0;
}

const float* Engine::keep(const char* name, uint64_t expect, cudaStream_t st) {
  const float* src = param(name, expect);
  if (!src) return nullptr;
  void* p = nullptr;
  if (cudaMalloc(&p, expect * sizeof(float)) != cudaSuccess) { set_error("cudaMalloc(%llu) failed", (unsigned long long)(expect * 4)); return nullptr; }
  kept.push_back(p);
  if (cudaMemcpyAsync(p, src, expect * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess) { set_error("copy of '%s' failed", name); return nullptr; }
  return static_cast<const float*>(p);
}

int Engine::debug_set(const char* key, long long value) {
  if (!strcmp(key, "stop_after")) { stop_after = (int)value; return 0; }
  if (!strcmp(key, "use_graphs")) { use_graphs = value != 0; return 0; }
  if (!strcmp(key, "range_guard")) {
    range_guard = value != 0;
    if (range_guard && !range_dev) {
      if (cudaMalloc(&range_dev, 8 * sizeof(float)) != cudaSuccess) { set_error("cudaMalloc failed"); return SKY_ERR_NOMEM; }
      kept.push_back(range_dev);
    }
    if (range_dev) SKY_CUDA_OK(cudaMemset(range_dev, 0, 8 * sizeof(float)));
    return 0;
  }
  set_error("unknown debug key '%s'", key);
  return SKY_ERR_ARG;
}

const float* Engine::param(const char* name, uint64_t expect) {
  auto it = params.find(name);
  if (it == params.end()) { set_error("missing parameter '%s'", name); return nullptr; }
  if (it->second.count != expect) {
    set_error("parameter '%s' has %llu floats, expected %llu", name, (unsigned long long)it->second.count,
              (unsigned long long)expect);
    return nullptr;
  }
  return it->second.dev;
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10 Gaussian perturbation (K11)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
  uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
  uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
  c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
}
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
// each thread perturbs 4 consecutive floats of one (member, channel) plane
__global__ void k_perturb_ic(float* __restrict__ x, const float* __restrict__ sigma, float amp, uint64_t seed,
                             int member0, int channels, long long plane, long long n_quads_per_plane,
                             long long total_quads) {
  long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= total_quads) return;
  long long pc = q / n_quads_per_plane, qi = q % n_quads_per_plane;  // pc = member*channels + c
  int c = (int)(pc % channels);
  int member = member0 + (int)(pc / channels);
  uint32_t ctr[4] = {(uint32_t)qi, (uint32_t)(qi >> 32), (uint32_t)c, (uint32_t)member};
  philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
  // Box-Muller on two pairs
  const float s = amp * sigma[c];
  float u0 = ((float)ctr[0] + 0.5f) * 2.3283064365386963e-10f, u1 = ((float)ctr[1] + 0.5f) * 2.3283064365386963e-10f;
  float u2 = ((float)ctr[2] + 0.5f) * 2.3283064365386963e-10f, u3 = ((float)ctr[3] + 0.5f) * 2.3283064365386963e-10f;
  float r0 = sqrtf(-2.f * __logf(u0)), r1 = sqrtf(-2.f * __logf(u2));
  float z[4];
  __sincosf(6.283185307179586f * u1, &z[1], &z[0]);
  __sincosf(6.283185307179586f * u3, &z[3], &z[2]);
  z[0] *= r0; z[1] *= r0; z[2] *= r1; z[3] *= r1;
  long long base = pc * plane + qi * 4;
#pragma unroll
  for (int e = 0; e < 4; ++e)
    if (qi * 4 + e < plane) x[base + e] += s * z[e];
}

}  // namespace sky

using namespace sky;

struct sky_model {
  Engine* eng;
};

extern "C" {

int sky_abi_version(void) { return SKY_ABI_VERSION; }
const char* sky_last_error(void) { return g_err; }
uint64_t sky_launch_count(void) { return g_launches.load(); }

int sky_model_create(sky_model_t** out, int kind, const void* cfg, size_t cfg_bytes, int device) {
  if (!out || !cfg) { set_error("null argument"); return SKY_ERR_ARG; }
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_error("no CUDA device visible: the skyrim_b200 engine has no CPU fallback");
    return SKY_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) { set_error("device %d out of range (%d visible)", device, ndev); return SKY_ERR_ARG; }
  DeviceGuard guard(device);
  cudaDeviceProp prop;
  SKY_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major, prop.minor);
    return SKY_ERR_CUDA;
  }
  Engine* e = nullptr;
  if (kind == SKY_MODEL_PANGU6) {
    if (cfg_bytes != sizeof(sky_pangu_config_t)) { set_error("bad config size"); return SKY_ERR_ARG; }
    e = make_pangu_engine(*static_cast<const sky_pangu_config_t*>(cfg), device);
  } else if (kind == SKY_MODEL_SFNO73) {
    if (cfg_bytes != sizeof(sky_sfno_config_t)) { set_error("bad config size"); return SKY_ERR_ARG; }
    e = make_sfno_engine(*static_cast<const sky_sfno_config_t*>(cfg), device);
  } else if (kind == SKY_MODEL_GRAPHCAST) {
    if (cfg_bytes != sizeof(sky_graphcast_config_t)) { set_error("bad config size"); return SKY_ERR_ARG; }
    e = make_graphcast_engine(*static_cast<const sky_graphcast_config_t*>(cfg), device);
  } else if (kind == SKY_MODEL_AFNO26) {
    if (cfg_bytes != sizeof(sky_afno_config_t)) { set_error("bad config size"); return SKY_ERR_ARG; }
    e = make_fcn_engine(*static_cast<const sky_afno_config_t*>(cfg), device);
  } else {
    set_error("unknown model kind %d", kind);
    return SKY_ERR_ARG;
  }
  if (!e) return SKY_ERR_ARG;
  e->num_sms = prop.multiProcessorCount;
  *out = new sky_model{e};
  return SKY_OK;
}

int sky_model_load_weights(sky_model_t* m, const float* arena, uint64_t n_floats, const sky_param_desc_t* manifest,
                           int32_t n_params, int32_t on_device, void* stream) {
  if (!m || !arena || !manifest) { set_error("null argument"); return SKY_ERR_ARG; }
  DeviceGuard guard(m->eng->device);
  return m->eng->load_arena(arena, n_floats, manifest, n_params, on_device, (cudaStream_t)stream);
}

size_t sky_model_workspace_bytes(const sky_model_t* m, int32_t batch) {
  return m && batch > 0 ? m->eng->workspace_bytes(batch) : 0;
}

int sky_model_step(sky_model_t* m, const float* x_in, float* x_out, int32_t batch, void* ws, size_t ws_bytes,
                   void* stream) {
  if (!m || !x_in || !x_out || !ws || batch <= 0) { set_error("bad argument"); return SKY_ERR_ARG; }
  if (x_in == x_out) { set_error("x_in and x_out may not alias"); return SKY_ERR_ARG; }
  DeviceGuard guard(m->eng->device);
  return m->eng->step_cached(x_in, x_out, batch, ws, ws_bytes, (cudaStream_t)stream);
}

int sky_model_set_clock(sky_model_t* m, double unix_seconds, void* stream) {
  if (!m) { set_error("null model"); return SKY_ERR_ARG; }
  DeviceGuard guard(m->eng->device);
  // captured steps stay valid: the clock lives in device memory, nothing in a graph depends on the host value
  return m->eng->set_clock(unix_seconds, (cudaStream_t)stream);
}

int sky_toa_radiation(float* out, int32_t nlat, int32_t nlon, double unix_seconds, void* stream) {
  if (!out || nlat < 2 || nlon < 1) { set_error("bad argument"); return SKY_ERR_ARG; }
  cudaPointerAttributes attr;
  SKY_CUDA_OK(cudaPointerGetAttributes(&attr, out));
  if (attr.type != cudaMemoryTypeDevice) { set_error("out must be device memory"); return SKY_ERR_ARG; }
  DeviceGuard guard(attr.device);
  return toa_radiation_launch(out, nlat, nlon, unix_seconds, (cudaStream_t)stream);
}

int sky_model_debug_copy(sky_model_t* m, const char* what, float* dst, uint64_t max_floats, void* ws, int32_t batch,
                         void* stream) {
  if (!m || !what || !dst || !ws) { set_error("bad argument"); return SKY_ERR_ARG; }
  DeviceGuard guard(m->eng->device);
  return m->eng->debug_copy(what, dst, max_floats, ws, batch, (cudaStream_t)stream);
}

int sky_model_debug_set(sky_model_t* m, const char* key, int64_t value) {
  if (!m || !key) { set_error("bad argument"); return SKY_ERR_ARG; }
  return m->eng->debug_set(key, (long long)value);
}

int sky_perturb_ic(float* x, const float* sigma_c, float amp, uint64_t seed, int32_t member0, int32_t members,
                   int32_t channels, int64_t plane, void* stream) {
  if (!x || !sigma_c || members <= 0 || channels <= 0 || plane <= 0) { set_error("bad argument"); return SKY_ERR_ARG; }
  cudaPointerAttributes attr;
  SKY_CUDA_OK(cudaPointerGetAttributes(&attr, x));
  if (attr.type != cudaMemoryTypeDevice) { set_error("x must be device memory"); return SKY_ERR_ARG; }
  DeviceGuard guard(attr.device);   // launch on the device that owns the state, whatever the caller's current device is
  long long qpp = (plane + 3) / 4;
  long long total = qpp * channels * members;
  k_perturb_ic<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, sigma_c, amp, seed, member0,
                                                                                  channels, plane, qpp, total);
  count_launch();
  SKY_CUDA_OK(cudaGetLastError());
  return SKY_OK;
}

int sky_model_profile_begin(sky_model_t* m, uint64_t tag_mask) {
  if (!m) { set_error("null model"); return SKY_ERR_ARG; }
  DeviceGuard guard(m->eng->device);
  double ms[KT_COUNT]; uint64_t c[KT_COUNT];
  m->eng->prof_collect(ms, c, KT_COUNT);
  m->eng->prof_mask = tag_mask;
  return SKY_OK;
}
int sky_model_profile_end(sky_model_t* m, double* ms_per_tag, uint64_t* launches_per_tag, int32_t n_tags) {
  if (!m || !ms_per_tag || !launches_per_tag) { set_error("null argument"); return SKY_ERR_ARG; }
  DeviceGuard guard(m->eng->device);
  m->eng->prof_mask = 0;
  return m->eng->prof_collect(ms_per_tag, launches_per_tag, n_tags);
}
int sky_profile_tag_count(void) { return KT_COUNT; }
const char* sky_profile_tag_name(int32_t tag) { return ktag_name(tag); }

int sky_model_destroy(sky_model_t* m) {
  if (!m) return SKY_OK;
  DeviceGuard guard(m->eng->device);
  delete m->eng;
  delete m;
  return SKY_OK;
}

}  // extern "C"
