// Host-side engine interface shared by the per-model translation units and the C-ABI.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <atomic>
#include <map>
#include <string>
#include <vector>

#include "../../include/skyrim_b200.h"

namespace sky {

extern std::atomic<uint64_t> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }
void set_error(const char* fmt, ...);

// kernel families, used for per-kernel CUDA-event timing (bench.py roofline) and launch counting
enum KTag { KT_EMBED = 0, KT_QKV, KT_ATTN, KT_PROJ, KT_FC1, KT_FC2, KT_MLP, KT_DOWN, KT_UP, KT_RECOVER, KT_COPY,
            KT_SFNO_ENC, KT_SFNO_SHT, KT_SFNO_SPEC, KT_SFNO_ISHT, KT_SFNO_MLP, KT_SFNO_DEC, KT_SFNO_MISC,
            KT_GC_FEAT, KT_GC_HIDDEN, KT_GC_LN, KT_GC_TABLE, KT_GC_AGG, KT_GC_OUT, KT_GC_MISC,
            KT_FCN_EMBED, KT_FCN_LN, KT_FCN_SPEC, KT_FCN_MLP, KT_FCN_HEAD, KT_COUNT };
const char* ktag_name(int tag);

struct ParamView {
  const float* dev;  // device pointer inside the resident fp32 arena
  uint64_t count;
};

// Base class of a step operator bound to one device.
struct Engine {
  int device = 0;
  int num_sms = 148;
  float* arena = nullptr;  // fp32 copy of the weight arena: alive during load_arena() only (freed after repacking)
  uint64_t arena_floats = 0;
  std::map<std::string, ParamView> params;
  std::vector<void*> kept;  // small persistent fp32 tensors (biases, norm vectors, masks): copies that outlive the arena
  bool loaded = false;
  int stop_after = 99;      // debug tap (sky_model_debug_set "stop_after"): return from step() after stage n
  // fp16-range guard (sky_model_debug_set "range_guard" 1): the step scans the fp16 operand images it produced and keeps
  // max |value| per class in range_dev[8] (read back with debug_copy "range").  The tensor cores take fp16 operands (5
  // exponent bits): with real checkpoints the caller runs the first step of a rollout guarded and refuses anything > 3e4.
  // Slots: 0 token images (LN outputs), 1 q/k/v, 2 attention output, 3 down / up-sampled images (Pangu);
  //        4 pixel images, 5 hidden images, 6 spectral images (SFNO).  FourCastNet scans its LN2 rows (0) and its MLP
  //        hidden rows (5); its spectral filter runs in fp32 and has no fp16 image.
  int range_guard = 0;
  float* range_dev = nullptr;
  int range_scan(int slot, const void* img, size_t bytes, cudaStream_t st);   // no-op unless range_guard

  // optional per-kernel timing: events are recorded around launches whose tag is in prof_mask
  uint64_t prof_mask = 0;
  struct ProfRec { cudaEvent_t a, b; int tag; };
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> prof_pool;
  cudaEvent_t prof_event();
  void prof_begin(int tag, cudaStream_t st) {
    if (prof_mask >> tag & 1) { ProfRec r{prof_event(), prof_event(), tag}; cudaEventRecord(r.a, st); prof_recs.push_back(r); }
  }
  void prof_end(int tag, cudaStream_t st) {
    if (prof_mask >> tag & 1) cudaEventRecord(prof_recs.back().b, st);
  }
  int prof_collect(double* ms, uint64_t* counts, int n);  // synchronises; resets the records

  // CUDA-graph replay of the step's launch sequence (one graph per (x_in, x_out, workspace, batch) tuple; a rollout
  // alternates between two or three such tuples).  The first call with a tuple runs eagerly (shared-memory opt-ins,
  // lazy allocations), the second is captured, later ones are replayed: one graph launch instead of ~85 (Pangu) / ~170
  // (SFNO) kernel launches.  Bypassed while per-kernel profiling or a debug tap is active, or when the caller's stream is
  // itself being captured.
  struct GraphEntry { const float* x_in; float* x_out; void* ws; int batch; cudaGraphExec_t exec; uint64_t launches; int seen; };
  std::vector<GraphEntry> graphs;
  bool use_graphs = true;
  int step_cached(const float* x_in, float* x_out, int batch, void* ws, size_t ws_bytes, cudaStream_t st);
  void drop_graphs();

  virtual ~Engine();
  int load_arena(const float* src, uint64_t n_floats, const sky_param_desc_t* manifest, int n_params,
                 int on_device, cudaStream_t st);
  const float* param(const char* name, uint64_t expect_count);  // nullptr + error if missing / wrong size; valid during prepare() only
  const float* keep(const char* name, uint64_t expect_count, cudaStream_t st);  // persistent device copy of a parameter

  virtual int prepare(cudaStream_t st) = 0;  // repack weights after load_arena
  virtual size_t workspace_bytes(int batch) const = 0;
  virtual int step(const float* x_in, float* x_out, int batch, void* ws, size_t ws_bytes, cudaStream_t st) = 0;
  virtual int debug_copy(const char* what, float* dst, uint64_t max_floats, void* ws, int batch,
                         cudaStream_t st) = 0;
  virtual int debug_set(const char* key, long long value);
  // valid time (unix seconds) of the state the next step starts from; only operators with time-dependent forcings use it
  virtual int set_clock(double /*unix_seconds*/, cudaStream_t) { return 0; }
};

Engine* make_pangu_engine(const sky_pangu_config_t& cfg, int device);
Engine* make_sfno_engine(const sky_sfno_config_t& cfg, int device);
Engine* make_graphcast_engine(const sky_graphcast_config_t& cfg, int device);
Engine* make_fcn_engine(const sky_afno_config_t& cfg, int device);
int toa_radiation_launch(float* out, int nlat, int nlon, double unix_seconds, cudaStream_t st);

}  // namespace sky
