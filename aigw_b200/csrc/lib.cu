// aigw_b200 C-ABI implementation: context, arenas, device- and host-buffer entry points.
// The host path is a 3-slot pipeline: H2D(chunk c+1) ‖ kernel(chunk c) ‖ D2H(chunk c-1) on three
// CUDA streams; everything computed is computed by the kernels in this directory — there is no
// CPU fallback anywhere in this library.
#include <cstdio>
#include <sched.h>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "chat_kernel.cuh"
#include "lib_internal.h"
#include "sse_kernel.cuh"
#include "bedrock_stream_kernel.cuh"
#include "mutate_kernel.cuh"
#include "sha256_kernel.cuh"
#include "cel_kernel.cuh"
#include "stream_kernel.cuh"
#include "bpe_kernel.cuh"
#include "emb_kernel.cuh"

#include <mutex>

using namespace aigw;

struct aigw_cost_program { aigw::CelProgramHost h; };

// a failed call is reported once: its code is also taken off the thread's "last error", so that the launch check of a later call does not find it
#define CK(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) { ctx->err = std::string(#x) + ": " + cudaGetErrorString(_e); (void)cudaGetLastError(); return (int)_e; } } while (0)

static constexpr int kSlots = 3;
static bool plain_json_text(const char* s) { for (; *s; s++) { unsigned char c = (unsigned char)*s; if (c < 0x20 || c > 0x7e || c == '"' || c == '\\') return false; } return true; }

struct ChunkSlot {
  uint8_t* d_in = nullptr; size_t in_cap = 0;
  uint64_t* d_off = nullptr; uint32_t* d_len = nullptr; size_t doc_cap = 0;
  uint32_t* d_map = nullptr; size_t map_cap = 0;   // size-class bucketing: documents of the chunk grouped by class
  uint8_t* d_out = nullptr; size_t out_cap = 0;
  aigw_doc_result* d_res = nullptr;
  cudaEvent_t ev_h2d, ev_k1, ev_done;
};

struct aigw_bpe { uint2* d_table = nullptr; uint16_t* d_b2i = nullptr; uint32_t slots = 0; };

struct aigw_ctx {
  int device = 0, sm_count = 0;
  cudaStream_t s_compute = nullptr, s_h2d = nullptr, s_d2h = nullptr;
  std::string err;
  // counters for the device API (ring so independent launches do not share a counter)
  unsigned int* d_counters = nullptr; int counter_next = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  ChunkSlot slot[kSlots];
  // host-API output (pinned)
  uint8_t* h_out = nullptr; size_t h_out_cap = 0;
  aigw_doc_result* h_res = nullptr; size_t h_res_cap = 0;
  long small_max = -1;   // aigw_chat_set_small_batch; -1: 512
  // BPE count (host form): device staging
  uint8_t* d_bpe_text = nullptr; size_t bpe_text_cap = 0; uint64_t* d_bpe_off = nullptr; size_t bpe_off_cap = 0; uint32_t* d_bpe_len = nullptr; size_t bpe_len_cap = 0; uint32_t* d_bpe_cnt = nullptr; size_t bpe_cnt_cap = 0;
  // large embeddings requests (aigw_embeddings_count_*): token workspace, text table, counts, host-form staging
  uint32_t* d_emb_tok = nullptr; size_t emb_tok_cap = 0; uint64_t* d_emb_toff = nullptr; size_t emb_toff_cap = 0; uint32_t* d_emb_tlen = nullptr; size_t emb_tlen_cap = 0;
  uint32_t* d_emb_cnt = nullptr; size_t emb_cnt_cap = 0; uint8_t* d_emb_body = nullptr; size_t emb_body_cap = 0; uint64_t* d_emb_off = nullptr; size_t emb_off_cap = 0;
  uint32_t* d_emb_len = nullptr; size_t emb_len_cap = 0; aigw_emb_count_result* d_emb_res = nullptr; size_t emb_res_cap = 0;
  uint8_t* h_small = nullptr; size_t h_small_cap = 0;   // small-batch path: tables + bodies, read by the kernel in place (mapped pinned)
  // chat workspace (intermediates of one sub-batch) + per-stage timing events
  uint8_t* d_work = nullptr; size_t work_cap = 0;
  unsigned long long* d_used_arr = nullptr; unsigned long long* h_used_arr = nullptr; size_t used_cap = 0;  // per-chunk bump counters
  cudaEvent_t stage_ev[64]; float stage_ms[3] = {0, 0, 0}; int last_launches = 0;
  bool profile_stages = false;   // aigw_chat_set_profile: next device calls time the stages
  // sse host-API device buffers
  uint8_t* d_sse_bytes = nullptr; size_t sse_bytes_cap = 0;
  uint64_t* d_sse_coff = nullptr; size_t sse_coff_cap = 0;
  uint32_t* d_sse_first = nullptr; size_t sse_first_cap = 0;
  aigw_sse_result* d_sse_res = nullptr; size_t sse_res_cap = 0;
  // bedrock stream workspace (records + counts) and host-API buffers
  uint8_t* d_bs_work = nullptr; size_t bs_work_cap = 0;
  uint64_t* d_bs_off[2] = {nullptr, nullptr}; size_t bs_off_cap[2] = {0, 0};
  aigw_stream_result* h_sres = nullptr; size_t h_sres_cap = 0;
  aigw_mut_result* h_mres = nullptr; size_t h_mres_cap = 0;
  std::vector<uint32_t> h_map;   // size-class bucketing scratch (host)
  // ---- stateful response streams (aigw_stream_*): device-resident slots + per-call staging
  struct StreamPool {
    std::mutex mu;
    StreamSlot* d_slots = nullptr; uint32_t cap = 0;
    std::vector<uint32_t> free_list, carry, gen, stamp; std::vector<uint8_t> open; uint32_t call_no = 0;
    uint8_t* h_in = nullptr; size_t h_in_cap = 0; uint8_t* d_in = nullptr; size_t d_in_cap = 0;
    StreamStep* h_steps = nullptr; size_t h_steps_cap = 0; StreamStep* d_steps = nullptr; size_t d_steps_cap = 0;
    aigw_chunk_result* d_res = nullptr; size_t d_res_cap = 0; aigw_chunk_result* h_res = nullptr; size_t h_res_cap = 0;
    uint8_t* d_out = nullptr; size_t d_out_cap = 0; uint8_t* d_packed = nullptr; size_t d_packed_cap = 0; uint8_t* h_packed = nullptr; size_t h_packed_cap = 0;
    unsigned long long* d_used = nullptr; unsigned long long* h_used = nullptr;
    uint8_t* d_tmpl = nullptr; uint32_t* d_ids = nullptr; size_t d_ids_cap = 0; uint32_t* h_ids = nullptr; size_t h_ids_cap = 0;
  } sp;
};

// response bodies expand (escaped tool arguments, configuration text): plan them in a roomier size class
static uint32_t resp_class_len(uint32_t max_len) { uint64_t m = (uint64_t)max_len * 4; if (m < 5120) m = 5120; if (m > 65536) m = max_len > 65536u ? max_len : 65536u; return (uint32_t)m; }

static void fill_params(ChatParams& P, const aigw_backend_cfg* cfg) {
  P.schema = cfg ? cfg->schema : AIGW_SCHEMA_OPENAI;
  P.cost_configured = cfg ? cfg->cost_configured : 0;
  P.force_mutation = cfg ? cfg->force_body_mutation : 0;
  P.override_len = 0; P.prefix_len = 0; P.version_len = 0; memset(P.api_version, 0, sizeof P.api_version);
  if (cfg && cfg->api_version) { size_t n = strlen(cfg->api_version); if (n > sizeof P.api_version) n = sizeof P.api_version; memcpy(P.api_version, cfg->api_version, n); P.version_len = (uint16_t)n; }
  memset(P.override_model, 0, sizeof P.override_model); memset(P.openai_path, 0, sizeof P.openai_path);
  if (cfg && cfg->model_name_override) {
    size_t n = strlen(cfg->model_name_override); if (n > sizeof P.override_model) n = sizeof P.override_model;
    memcpy(P.override_model, cfg->model_name_override, n); P.override_len = (uint16_t)n;
  }
  // path.Join("/", prefix, "chat/completions") (openai_openai.go:30)
  std::string pfx = (cfg && cfg->openai_prefix) ? cfg->openai_prefix : "v1";
  while (!pfx.empty() && pfx.front() == '/') pfx.erase(0, 1);
  while (!pfx.empty() && pfx.back() == '/') pfx.pop_back();
  std::string path = "/" + (pfx.empty() ? std::string() : pfx + "/") + ((cfg && (cfg->schema & AIGW_SCHEMA_EMBEDDINGS)) ? "embeddings" : "chat/completions");
  if (path.size() > sizeof P.openai_path) path.resize(sizeof P.openai_path);
  memcpy(P.openai_path, path.data(), path.size()); P.prefix_len = (uint16_t)path.size();
  P.created = 0; P.rid_len = 0; memset(P.response_id, 0, sizeof P.response_id);
  if (cfg && (cfg->schema & 48) == AIGW_SCHEMA_RESP_AWS_BEDROCK) {   // response direction (any backend)
    P.created = cfg->created;
    if (cfg->response_id) { size_t n = strlen(cfg->response_id); if (n > sizeof P.response_id) n = sizeof P.response_id; memcpy(P.response_id, cfg->response_id, n); P.rid_len = (uint16_t)n; }
  }
}

static int ensure(aigw_ctx* ctx, void** p, size_t* cap, size_t want, bool host) {
  if (*cap >= want) return 0;
  if (*p) { if (host) cudaFreeHost(*p); else cudaFree(*p); *p = nullptr; *cap = 0; }
  size_t sz = want + want / 8 + 4096;
  cudaError_t e = host ? cudaHostAlloc(p, sz, cudaHostAllocMapped) : cudaMalloc(p, sz);
  if (e != cudaSuccess) { ctx->err = std::string(host ? "cudaHostAlloc" : "cudaMalloc") + ": " + cudaGetErrorString(e); return (int)e; }
  *cap = sz;
  return 0;
}
#define ENSURE(p, cap, want, host) do { int _r = ensure(ctx, (void**)&(p), &(cap), (want), (host)); if (_r) return _r; } while (0)

namespace aigw {
int ctx_device(const aigw_ctx* ctx) { return ctx->device; }
bool chat_small_fits(const aigw_backend_cfg* cfg, uint32_t len) {
  const bool resp = cfg && (cfg->schema & 48) == AIGW_SCHEMA_RESP_AWS_BEDROCK;
  return len > 0 && (resp ? resp_class_len(len) : len) <= kSmallMaxLen;
}
cudaError_t chat_small_launch(const aigw_backend_cfg* cfg, const uint8_t* in, const uint64_t* offsets, const uint32_t* lens, const uint64_t* out_slot, uint32_t n, uint8_t* out,
                              aigw_doc_result* results, cudaStream_t st) {
  ChatParams P; fill_params(P, cfg);
  P.bodies = in; P.offsets = offsets; P.lens = lens; P.n = n;
  P.out = out; P.out_capacity = 0; P.results = results; P.out_used = nullptr; P.next_doc = nullptr; P.out_bias = 0; P.doc_map = nullptr;
  return launch_chat_small(P, 0, n, out_slot, st);
}
}  // namespace aigw

// host loops over the calls of one window (byte staging, result hand-back) run on a few threads when the window is large
template <class F>
static void host_parallel_for(uint32_t n, F&& f) {
  constexpr unsigned hw = 2;   // measured: more staging threads slow the DMA that follows (17.3 / 20.0 / 19.5 / 15.9 M chunks/s at 1 / 2 / 4 / 8)
  if (n < 16384) { f(0u, n); return; }
  std::vector<std::thread> th;
  const uint32_t per = (n + hw - 1) / hw;
  for (unsigned t = 1; t < hw; t++) { const uint32_t b = t * per, e = b + per < n ? b + per : n; if (b < e) th.emplace_back([&f, b, e] { f(b, e); }); }
  f(0u, per < n ? per : n);
  for (auto& x : th) x.join();
}

extern "C" {

const char* aigw_version(void) { return "aigw_b200 0.1 (sm_100a)"; }

int aigw_init(int device, aigw_ctx** out) {
  *out = nullptr;
  aigw_ctx* ctx = new aigw_ctx();
  ctx->device = device;
  cudaError_t e = cudaSetDevice(device);
  // a failed runtime call leaves its code as the thread's "last error": clear it, or the next launch check of ANOTHER context on this
  // thread (cudaGetLastError after a kernel launch) reports it as its own (found by tests/test_multi_context_gpu.py)
  if (e != cudaSuccess) { fprintf(stderr, "aigw_init: cudaSetDevice(%d): %s\n", device, cudaGetErrorString(e)); (void)cudaGetLastError(); delete ctx; return (int)e; }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { (void)cudaGetLastError(); delete ctx; return (int)e; }
  ctx->sm_count = prop.multiProcessorCount;
  if (prop.major < 10) { fprintf(stderr, "aigw_init: device %d is sm_%d%d; this library is built for sm_100a only\n", device, prop.major, prop.minor); delete ctx; return (int)cudaErrorNoKernelImageForDevice; }
  // every allocation is checked on its own: a half-built context is destroyed, never returned
  auto fail = [&](const char* what, cudaError_t err) { fprintf(stderr, "aigw_init: %s: %s\n", what, cudaGetErrorString(err)); aigw_destroy(ctx); return (int)err; };
#define INIT_CK(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) return fail(#x, _e); } while (0)
  INIT_CK(cudaStreamCreateWithFlags(&ctx->s_compute, cudaStreamNonBlocking));
  INIT_CK(cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking));
  INIT_CK(cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking));
  INIT_CK(cudaMalloc(&ctx->d_counters, 256 * sizeof(unsigned int)));
  INIT_CK(cudaEventCreate(&ctx->ev0)); INIT_CK(cudaEventCreate(&ctx->ev1));
  for (auto& e2 : ctx->stage_ev) INIT_CK(cudaEventCreate(&e2));
  for (auto& s : ctx->slot) {
    INIT_CK(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming)); INIT_CK(cudaEventCreate(&s.ev_k1)); INIT_CK(cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
  }
#undef INIT_CK
  *out = ctx;
  return 0;
}

void aigw_destroy(aigw_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto& s : ctx->slot) {
    cudaFree(s.d_in); cudaFree(s.d_off); cudaFree(s.d_len); cudaFree(s.d_map); cudaFree(s.d_out); cudaFree(s.d_res);
    cudaEventDestroy(s.ev_h2d); cudaEventDestroy(s.ev_k1); cudaEventDestroy(s.ev_done);
  }
  cudaFreeHost(ctx->h_out); cudaFreeHost(ctx->h_res); cudaFreeHost(ctx->h_small); cudaFree(ctx->d_bpe_text); cudaFree(ctx->d_bpe_off); cudaFree(ctx->d_bpe_len); cudaFree(ctx->d_bpe_cnt); cudaFree(ctx->d_emb_tok); cudaFree(ctx->d_emb_toff); cudaFree(ctx->d_emb_tlen); cudaFree(ctx->d_emb_cnt); cudaFree(ctx->d_emb_body); cudaFree(ctx->d_emb_off); cudaFree(ctx->d_emb_len); cudaFree(ctx->d_emb_res); cudaFree(ctx->d_counters); cudaFree(ctx->d_work); cudaFree(ctx->d_used_arr); cudaFreeHost(ctx->h_used_arr);
  for (auto& e2 : ctx->stage_ev) cudaEventDestroy(e2);
  cudaFree(ctx->d_sse_bytes); cudaFree(ctx->d_sse_coff); cudaFree(ctx->d_sse_first); cudaFree(ctx->d_sse_res); cudaFree(ctx->d_bs_work); cudaFree(ctx->d_bs_off[0]); cudaFree(ctx->d_bs_off[1]); cudaFreeHost(ctx->h_sres); cudaFreeHost(ctx->h_mres);
  cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
  cudaStreamDestroy(ctx->s_compute); cudaStreamDestroy(ctx->s_h2d); cudaStreamDestroy(ctx->s_d2h);
  {
    auto& sp = ctx->sp;
    cudaFree(sp.d_slots); cudaFreeHost(sp.h_in); cudaFree(sp.d_in); cudaFreeHost(sp.h_steps); cudaFree(sp.d_steps); cudaFree(sp.d_res); cudaFreeHost(sp.h_res);
    cudaFree(sp.d_out); cudaFree(sp.d_packed); cudaFreeHost(sp.h_packed); cudaFree(sp.d_used); cudaFreeHost(sp.h_used); cudaFree(sp.d_tmpl); cudaFree(sp.d_ids); cudaFreeHost(sp.h_ids);
  }
  delete ctx;
}

// Bind the calling thread (and the threads it starts later) to the CPUs of the NUMA node the GPU hangs off, so that pinned
// arenas allocated afterwards are node-local (first touch) and the copy engines do not cross the socket interconnect
// (VERDICT r1: 8 ranks on one host lost 4x end to end with unbound ranks).  Returns the node, or -1 when it cannot be determined.
int aigw_bind_numa(int device) {
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) return -1;
  for (char* c = bus; *c; c++) if (*c >= 'A' && *c <= 'F') *c = (char)(*c - 'A' + 'a');
  char path[128]; snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
  FILE* f = fopen(path, "r"); if (!f) return -1;
  int node = -1; if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f);
  if (node < 0) return -1;
  snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
  f = fopen(path, "r"); if (!f) return -1;
  char list[4096] = {0}; if (!fgets(list, sizeof list, f)) { fclose(f); return -1; } fclose(f);
  cpu_set_t want; CPU_ZERO(&want);
  for (char* p = list; *p;) {
    char* end; long a = strtol(p, &end, 10); if (end == p) break; long b = a;
    if (*end == '-') { p = end + 1; b = strtol(p, &end, 10); }
    for (long c = a; c <= b && c < CPU_SETSIZE; c++) CPU_SET((int)c, &want);
    p = *end == ',' ? end + 1 : end; if (*end != ',' ) break;
  }
  cpu_set_t cur; CPU_ZERO(&cur);
  if (sched_getaffinity(0, sizeof cur, &cur) == 0) { cpu_set_t both; CPU_AND(&both, &cur, &want); if (CPU_COUNT(&both) > 0) want = both; }
  if (CPU_COUNT(&want) == 0 || sched_setaffinity(0, sizeof want, &want) != 0) return -1;
  return node;
}

const char* aigw_last_error(aigw_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }
int aigw_device_sm_count(aigw_ctx* ctx) { return ctx->sm_count; }

void* aigw_host_alloc(aigw_ctx* ctx, size_t bytes) { void* p = nullptr; cudaSetDevice(ctx->device); if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { ctx->err = "cudaHostAlloc failed"; return nullptr; } return p; }
void aigw_host_free(aigw_ctx*, void* p) { cudaFreeHost(p); }
void* aigw_device_alloc(aigw_ctx* ctx, size_t bytes) { void* p = nullptr; cudaSetDevice(ctx->device); if (cudaMalloc(&p, bytes) != cudaSuccess) { ctx->err = "cudaMalloc failed"; return nullptr; } return p; }
void aigw_device_free(aigw_ctx* ctx, void* p) { cudaSetDevice(ctx->device); cudaFree(p); }
int aigw_memcpy_h2d(aigw_ctx* ctx, void* dst, const void* src, size_t bytes) { CK(cudaSetDevice(ctx->device)); CK(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); return 0; }
int aigw_memcpy_d2h(aigw_ctx* ctx, void* dst, const void* src, size_t bytes) { CK(cudaSetDevice(ctx->device)); CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost)); return 0; }
int aigw_memset_d(aigw_ctx* ctx, void* dst, int v, size_t bytes) { CK(cudaSetDevice(ctx->device)); CK(cudaMemset(dst, v, bytes)); return 0; }
int aigw_sync(aigw_ctx* ctx) { CK(cudaSetDevice(ctx->device)); CK(cudaDeviceSynchronize()); return 0; }

static int chat_translate_device_impl(aigw_ctx* ctx, const aigw_backend_cfg* cfg, const uint8_t* d_bodies, const uint64_t* d_offsets,
                                      const uint32_t* d_lens, const uint32_t* d_doc_map, uint32_t first, uint32_t n, uint32_t max_len, uint8_t* d_out, uint64_t out_capacity,
                                      aigw_doc_result* d_results, uint64_t* d_out_used, void* stream, float* kernel_ms) {
  if (n == 0) { if (kernel_ms) *kernel_ms = 0; return 0; }
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  ChatParams P;
  fill_params(P, cfg);
  P.bodies = d_bodies; P.offsets = d_offsets; P.lens = d_lens; P.n = n; P.out = d_out; P.out_capacity = out_capacity;
  P.results = d_results; P.out_used = (unsigned long long*)d_out_used;
  P.next_doc = nullptr; P.out_bias = 0; P.doc_map = d_doc_map;
  uint32_t ml = max_len ? max_len : 65536u;
  if (cfg && (cfg->schema & 48) == AIGW_SCHEMA_RESP_AWS_BEDROCK) ml = resp_class_len(ml);
  const bool stages = ctx->profile_stages && kernel_ms;
  {  // workspace: one sub-batch of intermediates
    size_t need = chat_work_bytes_for(ml, n);
    const size_t cap = (size_t)3 << 30, floor1 = chat_work_bytes(ml, 1024);
    if (need > cap) need = cap > floor1 ? cap : floor1;
    ENSURE(ctx->d_work, ctx->work_cap, need, false);
  }
  if (kernel_ms) CK(cudaEventRecord(ctx->ev0, st));
  CK(launch_chat_translate(P, ml, ctx->device, ctx->sm_count, st, ctx->d_work, ctx->work_cap, &ctx->last_launches, stages ? ctx->stage_ev : nullptr, 64, first));
  if (kernel_ms) {
    CK(cudaEventRecord(ctx->ev1, st)); CK(cudaEventSynchronize(ctx->ev1)); CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1));
    if (stages) {
      ctx->stage_ms[0] = ctx->stage_ms[1] = ctx->stage_ms[2] = 0;
      const int nsb = ctx->last_launches / 4;
      for (int sb = 0; sb < nsb && 4 * sb + 3 < 64; sb++) for (int k = 0; k < 3; k++) { float ms = 0; cudaEventElapsedTime(&ms, ctx->stage_ev[4 * sb + k], ctx->stage_ev[4 * sb + k + 1]); ctx->stage_ms[k] += ms; }
    }
  }
  return 0;
}

int aigw_chat_translate_device(aigw_ctx* ctx, const aigw_backend_cfg* cfg, const uint8_t* d_bodies, const uint64_t* d_offsets,
                               const uint32_t* d_lens, uint32_t n, uint32_t max_len, uint8_t* d_out, uint64_t out_capacity,
                               aigw_doc_result* d_results, uint64_t* d_out_used, void* stream, float* kernel_ms) {
  return chat_translate_device_impl(ctx, cfg, d_bodies, d_offsets, d_lens, nullptr, 0, n, max_len, d_out, out_capacity, d_results, d_out_used, stream, kernel_ms);
}
int aigw_chat_translate_device_mapped(aigw_ctx* ctx, const aigw_backend_cfg* cfg, const uint8_t* d_bodies, const uint64_t* d_offsets, const uint32_t* d_lens,
                                      const uint32_t* d_doc_map, uint32_t first, uint32_t count, uint32_t max_len, uint8_t* d_out, uint64_t out_capacity,
                                      aigw_doc_result* d_results, uint64_t* d_out_used, void* stream, float* kernel_ms) {
  return chat_translate_device_impl(ctx, cfg, d_bodies, d_offsets, d_lens, d_doc_map, first, count, max_len, d_out, out_capacity, d_results, d_out_used, stream, kernel_ms);
}

int aigw_chat_set_profile(aigw_ctx* ctx, int on) { ctx->profile_stages = on != 0; return 0; }

/* per-stage CUDA-event times (index, walk, emit) of the last profiled call and the launch count of the last device call */
int aigw_chat_last_profile(aigw_ctx* ctx, float stage_ms[3], int* launches) {
  for (int k = 0; k < 3; k++) stage_ms[k] = ctx->stage_ms[k];
  if (launches) *launches = ctx->last_launches;
  return 0;
}

// Small batches (a single request, or what a batching window collects): one fused kernel, no workspace, no device copies.
// Every body owns a fixed output slot of 3 x its length + 1 KiB (the embeddings -> Vertex instances translation expands short
// inputs up to 5x; a record that does not fit is DECLINED with AIGW_R_ARENA_FULL, never truncated).
// The bodies are packed into a mapped pinned buffer the kernel reads in place, the records and results are stored straight
// into the pinned output arenas, and the call is launch + kernel + one synchronisation.
static int chat_small_host(aigw_ctx* ctx, const aigw_backend_cfg* cfg, const uint8_t* bodies, const uint64_t* offsets, const uint32_t* lens, uint32_t n, aigw_batch_out* out) {
  uint64_t in_bytes = 0, out_bytes = 0;
  for (uint32_t i = 0; i < n; i++) { in_bytes += (((uint64_t)lens[i] + 15u) & ~15ull) + 16; out_bytes += ((uint64_t)lens[i] * 3 + 1024 + 15) & ~15ull; }
  const size_t tab = (((size_t)n + 1) * 16 + (size_t)n * 4 + 63) & ~(size_t)63;
  ENSURE(ctx->h_small, ctx->h_small_cap, tab + in_bytes + 64, true);
  ENSURE(ctx->h_out, ctx->h_out_cap, out_bytes + 64, true);
  ENSURE(ctx->h_res, ctx->h_res_cap, (size_t)n * sizeof(aigw_doc_result), true);
  uint64_t* h_off = (uint64_t*)ctx->h_small; uint64_t* h_slot = h_off + n + 1; uint32_t* h_len = (uint32_t*)(h_slot + n + 1);
  uint8_t* h_in = ctx->h_small + tab;
  uint64_t o = 0, so = 0;
  for (uint32_t i = 0; i < n; i++) {
    h_off[i] = o; h_slot[i] = so; h_len[i] = lens[i];
    memcpy(h_in + o, bodies + offsets[i], lens[i]);
    o += (((uint64_t)lens[i] + 15u) & ~15ull) + 16; so += ((uint64_t)lens[i] * 3 + 1024 + 15) & ~15ull;
  }
  h_off[n] = o; h_slot[n] = so;
  uint8_t* d_small = nullptr; uint8_t* d_out = nullptr; aigw_doc_result* d_res = nullptr;
  CK(cudaHostGetDevicePointer((void**)&d_small, ctx->h_small, 0)); CK(cudaHostGetDevicePointer((void**)&d_out, ctx->h_out, 0)); CK(cudaHostGetDevicePointer((void**)&d_res, ctx->h_res, 0));
  ChatParams P; fill_params(P, cfg);
  P.bodies = d_small + tab; P.offsets = (const uint64_t*)d_small; P.lens = (const uint32_t*)(d_small + ((size_t)n + 1) * 16); P.n = n;
  P.out = d_out; P.out_capacity = so; P.results = d_res; P.out_used = nullptr; P.next_doc = nullptr; P.out_bias = 0; P.doc_map = nullptr;
  CK(cudaEventRecord(ctx->ev0, ctx->s_compute));
  CK(launch_chat_small(P, 0, n, (const uint64_t*)d_small + n + 1, ctx->s_compute));
  CK(cudaEventRecord(ctx->ev1, ctx->s_compute));
  CK(cudaEventSynchronize(ctx->ev1));
  float kms = 0; cudaEventElapsedTime(&kms, ctx->ev0, ctx->ev1);
  uint64_t produced = 0;
  for (uint32_t i = 0; i < n; i++) if (ctx->h_res[i].status == AIGW_OK) produced += ((uint64_t)ctx->h_res[i].path_len + ctx->h_res[i].body_len + 15u) & ~15ull;
  out->results = ctx->h_res; out->out = ctx->h_out; out->out_used = so; out->h2d_bytes = in_bytes + tab; out->d2h_bytes = produced + (uint64_t)n * sizeof(aigw_doc_result);
  out->gpu_launches = 1; out->kernel_ms = kms;
  return 0;
}

void aigw_chat_set_small_batch(aigw_ctx* ctx, int max_docs) { if (ctx) ctx->small_max = max_docs; }

int aigw_chat_translate_host(aigw_ctx* ctx, const aigw_backend_cfg* cfg, const uint8_t* bodies, const uint64_t* offsets,
                             const uint32_t* lens, uint32_t n, aigw_batch_out* out) {
  // Three-stage pipeline over 256 MiB chunks, both PCIe directions busy at once:
  //   copy engine A   H2D of chunk c+1                               (s_h2d)
  //   SMs             index / sort / walk / emit of chunk c → device (s_compute)
  //   copy engine B   D2H of chunk c-1: exactly the bytes the emit stage produced + the chunk's result table (s_d2h)
  // The host runs one chunk behind the GPU (it waits for chunk c-1's byte count while chunk c's kernels are queued).
  memset(out, 0, sizeof *out);
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  if ((long)n <= (ctx->small_max >= 0 ? ctx->small_max : 512)) {   // 0 disables the fused small-batch path
    const bool resp = cfg && (cfg->schema & 48) == AIGW_SCHEMA_RESP_AWS_BEDROCK;
    uint32_t ml = 0; for (uint32_t i = 0; i < n; i++) if (lens[i] > ml) ml = lens[i];
    if ((resp ? resp_class_len(ml) : ml) <= kSmallMaxLen) return chat_small_host(ctx, cfg, bodies, offsets, lens, n, out);
  }
  constexpr uint64_t kChunkBytes = 256ull << 20;   // pipeline granularity (fill / drain cost vs per-chunk launches)
  std::vector<uint32_t> cb;  // chunk begin doc index
  cb.push_back(0);
  uint32_t max_len = 0;
  {
    uint64_t start = offsets[0];
    for (uint32_t i = 0; i < n; i++) {
      const uint64_t end = offsets[i] + (((uint64_t)lens[i] + 15u) & ~15ull);
      if (end - start > kChunkBytes && i > cb.back()) { cb.push_back(i); start = offsets[i]; }
      if (lens[i] > max_len) max_len = lens[i];
    }
    cb.push_back(n);
  }
  const int nch = (int)cb.size() - 1;
  uint64_t max_in = 0, max_out = 0; uint32_t max_docs = 0;
  std::vector<uint64_t> in_bytes(nch), out_cap(nch), out_base(nch);
  uint64_t total_out_cap = 0;
  for (int c = 0; c < nch; c++) {
    const uint32_t b = cb[c], e = cb[c + 1];
    const uint64_t ib = offsets[e - 1] + (((uint64_t)lens[e - 1] + 15u) & ~15ull) - offsets[b] + 16;
    in_bytes[c] = ib; if (ib > max_in) max_in = ib; if (e - b > max_docs) max_docs = e - b;
    out_cap[c] = ((ib + ib / 4 + (uint64_t)(e - b) * 528 + 255) & ~255ull);
    if (out_cap[c] > max_out) max_out = out_cap[c];
    out_base[c] = total_out_cap; total_out_cap += out_cap[c];
  }
  const int nslots = nch < kSlots ? nch : kSlots;
  for (int s = 0; s < nslots; s++) {
    ChunkSlot& S = ctx->slot[s];
    ENSURE(S.d_in, S.in_cap, max_in + 64, false);
    ENSURE(S.d_out, S.out_cap, max_out + 64, false);
    if (S.doc_cap < max_docs) {
      cudaFree(S.d_off); cudaFree(S.d_len); cudaFree(S.d_res); S.doc_cap = 0;
      const size_t dc = max_docs + max_docs / 8 + 16;
      CK(cudaMalloc(&S.d_off, dc * 8)); CK(cudaMalloc(&S.d_len, dc * 4)); CK(cudaMalloc(&S.d_res, dc * sizeof(aigw_doc_result)));
      S.doc_cap = dc;
    }
  }
  const bool resp_dir = cfg && (cfg->schema & 48) == AIGW_SCHEMA_RESP_AWS_BEDROCK;
  if (resp_dir) max_len = resp_class_len(max_len);
  // size classes (the kernels' shared-memory footprints, chat_kernel.cu launch_chat_translate)
  static const uint32_t kClsMax[6] = {2048, 5120, 9216, 17408, 33792, 65536};
  auto cls_of = [&](uint32_t len) { const uint32_t l = resp_dir ? resp_class_len(len) : len; int k = 0; while (k < 5 && l > kClsMax[k]) k++; return k; };
  {
    size_t need = chat_work_bytes_for(max_len, max_docs);
    const size_t cap = (size_t)3 << 30;   // the launcher walks a class in sub-batches that fit the workspace
    const size_t floor1 = chat_work_bytes(max_len, 1024);
    if (need > cap) need = cap > floor1 ? cap : floor1;
    ENSURE(ctx->d_work, ctx->work_cap, need, false);
  }
  ENSURE(ctx->h_out, ctx->h_out_cap, total_out_cap, true);
  ENSURE(ctx->h_res, ctx->h_res_cap, (size_t)n * sizeof(aigw_doc_result), true);
  if ((size_t)nch > ctx->used_cap) {
    cudaFree(ctx->d_used_arr); cudaFreeHost(ctx->h_used_arr); ctx->used_cap = 0;
    const size_t cap = (size_t)nch + 64;
    CK(cudaMalloc(&ctx->d_used_arr, cap * 8)); CK(cudaHostAlloc(&ctx->h_used_arr, cap * 8, cudaHostAllocDefault));
    ctx->used_cap = cap;
  }

  ChatParams P0; fill_params(P0, cfg);
  uint64_t h2d = 0, d2h = (uint64_t)n * sizeof(aigw_doc_result) + (uint64_t)nch * 8;
  CK(cudaMemsetAsync(ctx->d_used_arr, 0, (size_t)nch * 8, ctx->s_compute));
  CK(cudaEventRecord(ctx->ev0, ctx->s_compute));
  auto drain = [&](int k) -> int {   // chunk k's kernels are done: move exactly what they produced
    ChunkSlot& S = ctx->slot[k % nslots];
    CK(cudaEventSynchronize(S.ev_k1));
    const uint64_t used = ctx->h_used_arr[k] < out_cap[k] ? ctx->h_used_arr[k] : out_cap[k];
    d2h += used;
    const uint32_t b = cb[k], nd = cb[k + 1] - b;
    if (used) CK(cudaMemcpyAsync(ctx->h_out + out_base[k], S.d_out, used, cudaMemcpyDeviceToHost, ctx->s_d2h));
    CK(cudaMemcpyAsync(ctx->h_res + b, S.d_res, (size_t)nd * sizeof(aigw_doc_result), cudaMemcpyDeviceToHost, ctx->s_d2h));
    CK(cudaEventRecord(S.ev_done, ctx->s_d2h));
    return 0;
  };
  for (int c = 0; c < nch; c++) {
    ChunkSlot& S = ctx->slot[c % nslots];
    const uint32_t b = cb[c], e = cb[c + 1], nd = e - b;
    if (c >= nslots) {
      CK(cudaStreamWaitEvent(ctx->s_h2d, S.ev_k1, 0));                       // the slot's input has been consumed
      CK(cudaStreamWaitEvent(ctx->s_compute, S.ev_done, 0));                 // the slot's output has left the device
    }
    CK(cudaMemcpyAsync(S.d_in, bodies + offsets[b], in_bytes[c] - 16, cudaMemcpyHostToDevice, ctx->s_h2d));
    CK(cudaMemcpyAsync(S.d_off, offsets + b, (size_t)nd * 8, cudaMemcpyHostToDevice, ctx->s_h2d));
    CK(cudaMemcpyAsync(S.d_len, lens + b, (size_t)nd * 4, cudaMemcpyHostToDevice, ctx->s_h2d));
    // size-class bucketing: a chunk whose documents span several classes is launched class by class over a document map,
    // so that a few large bodies do not force the small ones into the large class's shared-memory footprint
    uint32_t cls_cnt[6] = {0, 0, 0, 0, 0, 0};
    for (uint32_t i = b; i < e; i++) cls_cnt[cls_of(lens[i])]++;
    int n_cls = 0, top_cls = 0; for (int k = 0; k < 6; k++) if (cls_cnt[k]) { n_cls++; top_cls = k; }
    uint32_t cls_start[7] = {0, 0, 0, 0, 0, 0, 0};
    if (n_cls > 1) {
      for (int k = 0; k < 6; k++) cls_start[k + 1] = cls_start[k] + cls_cnt[k];
      ctx->h_map.resize(nd);
      uint32_t cur[6]; for (int k = 0; k < 6; k++) cur[k] = cls_start[k];
      for (uint32_t i = b; i < e; i++) ctx->h_map[cur[cls_of(lens[i])]++] = i;
      ENSURE(S.d_map, S.map_cap, (size_t)nd * 4, false);
      CK(cudaMemcpyAsync(S.d_map, ctx->h_map.data(), (size_t)nd * 4, cudaMemcpyHostToDevice, ctx->s_h2d));   // pageable source: staged before the call returns
      h2d += (uint64_t)nd * 4;
    }
    CK(cudaEventRecord(S.ev_h2d, ctx->s_h2d));
    h2d += in_bytes[c] - 16 + (uint64_t)nd * 12;
    CK(cudaStreamWaitEvent(ctx->s_compute, S.ev_h2d, 0));
    ChatParams P = P0;
    P.bodies = S.d_in - offsets[b];  // absolute offsets index straight into the chunk
    P.offsets = S.d_off - b; P.lens = S.d_len - b; P.n = nd;
    P.out = S.d_out; P.out_capacity = out_cap[c];
    P.results = S.d_res - b; P.out_used = ctx->d_used_arr + c; P.next_doc = nullptr; P.out_bias = out_base[c]; P.doc_map = nullptr;
    // documents keep their global index: kernels address offsets/lens/results with doc0 + i (or doc_map[i])
    if (n_cls <= 1) {
      int nl = 0;
      CK(launch_chat_translate_range(P, b, nd, kClsMax[top_cls], ctx->device, ctx->sm_count, ctx->s_compute, ctx->d_work, ctx->work_cap, &nl));
      out->gpu_launches += nl;
    } else {
      P.doc_map = S.d_map;
      for (int k = 0; k < 6; k++) {
        if (!cls_cnt[k]) continue;
        int nl = 0;
        CK(launch_chat_translate_range(P, cls_start[k], cls_cnt[k], kClsMax[k], ctx->device, ctx->sm_count, ctx->s_compute, ctx->d_work, ctx->work_cap, &nl));
        out->gpu_launches += nl;
      }
    }
    CK(cudaMemcpyAsync(ctx->h_used_arr + c, ctx->d_used_arr + c, 8, cudaMemcpyDeviceToHost, ctx->s_compute));
    CK(cudaEventRecord(S.ev_k1, ctx->s_compute));
    if (c >= 1) { const int rc = drain(c - 1); if (rc) return rc; }
  }
  CK(cudaEventRecord(ctx->ev1, ctx->s_compute));
  { const int rc = drain(nch - 1); if (rc) return rc; }
  CK(cudaStreamSynchronize(ctx->s_d2h));
  CK(cudaStreamSynchronize(ctx->s_compute));
  float ms_total = 0; cudaEventElapsedTime(&ms_total, ctx->ev0, ctx->ev1);
  out->results = ctx->h_res; out->out = ctx->h_out; out->out_used = total_out_cap; out->h2d_bytes = h2d; out->d2h_bytes = d2h; out->kernel_ms = ms_total;
  return 0;
}

// ------------------------------------------------------------------ K4: BPE token count
int aigw_bpe_load(aigw_ctx* ctx, const uint16_t* byte_to_id, const uint32_t* merges, uint32_t n_merges, aigw_bpe** out) {
  if (!ctx || !byte_to_id || (!merges && n_merges) || !out || n_merges >= 65535u) return -2;
  for (uint32_t r = 0; r < n_merges * 3; r++) if (merges[r] >= 65536u) return -2;
  CK(cudaSetDevice(ctx->device));
  uint32_t slots = 1024; while (slots < n_merges * 2u) slots <<= 1;
  if (bpe_smem_bytes(slots) > 220u * 1024u) { ctx->err = "aigw_bpe_load: merge table does not fit shared memory"; return -2; }
  std::vector<uint2> tab(slots, make_uint2(0xffffffffu, 0xffffffffu));
  for (uint32_t r = 0; r < n_merges; r++) {
    const uint32_t key = (merges[3 * r] << 16) | merges[3 * r + 1];
    uint32_t h = key * 0x9E3779B1u; h ^= h >> 15;
    uint32_t s = h & (slots - 1);
    bool dup = false;
    while (tab[s].x != 0xffffffffu) { if (tab[s].x == key) { dup = true; break; } s = (s + 1) & (slots - 1); }
    if (dup) continue;   // the first rank of a pair wins (a well-formed merge list has no duplicates)
    tab[s] = make_uint2(key, (r << 16) | merges[3 * r + 2]);
  }
  aigw_bpe* b = new aigw_bpe();
  b->slots = slots;
  if (cudaMalloc(&b->d_table, (size_t)slots * 8) != cudaSuccess || cudaMalloc(&b->d_b2i, 512) != cudaSuccess) { cudaFree(b->d_table); delete b; return (int)cudaErrorMemoryAllocation; }
  CK(cudaMemcpy(b->d_table, tab.data(), (size_t)slots * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(b->d_b2i, byte_to_id, 512, cudaMemcpyHostToDevice));
  *out = b;
  return 0;
}
void aigw_bpe_free(aigw_ctx* ctx, aigw_bpe* b) { if (!b) return; if (ctx) cudaSetDevice(ctx->device); cudaFree(b->d_table); cudaFree(b->d_b2i); delete b; }

int aigw_bpe_count_device(aigw_ctx* ctx, const aigw_bpe* bpe, const uint8_t* d_text, const uint64_t* d_offsets, const uint32_t* d_lens, uint32_t n, uint32_t* d_counts,
                          void* stream, float* kernel_ms) {
  if (!ctx || !bpe) return -2;
  if (n == 0) { if (kernel_ms) *kernel_ms = 0; return 0; }
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  BpeParams P; P.text = d_text; P.offsets = d_offsets; P.lens = d_lens; P.n = n; P.counts = d_counts; P.table = bpe->d_table; P.slots = bpe->slots; P.byte_to_id = bpe->d_b2i;
  P.next = ctx->d_counters + (ctx->counter_next++ & 255);
  CK(cudaMemsetAsync(P.next, 0, sizeof(unsigned int), st));
  if (kernel_ms) CK(cudaEventRecord(ctx->ev0, st));
  CK(launch_bpe_count(P, ctx->sm_count, st));
  if (kernel_ms) { CK(cudaEventRecord(ctx->ev1, st)); CK(cudaEventSynchronize(ctx->ev1)); CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1)); }
  return 0;
}

int aigw_bpe_count_host(aigw_ctx* ctx, const aigw_bpe* bpe, const uint8_t* text, const uint64_t* offsets, const uint32_t* lens, uint32_t n, uint32_t* counts,
                        uint64_t* h2d_bytes, uint64_t* d2h_bytes, float* kernel_ms) {
  if (!ctx || !bpe) return -2;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  uint64_t nbytes = 0; for (uint32_t i = 0; i < n; i++) { const uint64_t e = offsets[i] + lens[i]; if (e > nbytes) nbytes = e; }
  ENSURE(ctx->d_bpe_text, ctx->bpe_text_cap, nbytes + 64, false);
  ENSURE(ctx->d_bpe_off, ctx->bpe_off_cap, (size_t)n * 8, false);
  ENSURE(ctx->d_bpe_len, ctx->bpe_len_cap, (size_t)n * 4, false);
  ENSURE(ctx->d_bpe_cnt, ctx->bpe_cnt_cap, (size_t)n * 4, false);
  cudaStream_t st = ctx->s_compute;
  CK(cudaMemcpyAsync(ctx->d_bpe_text, text, nbytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->d_bpe_off, offsets, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->d_bpe_len, lens, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  float ms = 0;
  if (int rc = aigw_bpe_count_device(ctx, bpe, ctx->d_bpe_text, ctx->d_bpe_off, ctx->d_bpe_len, n, ctx->d_bpe_cnt, st, &ms)) return rc;
  CK(cudaMemcpyAsync(counts, ctx->d_bpe_cnt, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (kernel_ms) *kernel_ms = ms;
  if (h2d_bytes) *h2d_bytes = nbytes + (uint64_t)n * 12;
  if (d2h_bytes) *d2h_bytes = (uint64_t)n * 4;
  return 0;
}

// ------------------------------------------------------------------ large /v1/embeddings requests: ParseBody + BPE count (BASELINE config 3)
int aigw_embeddings_count_device(aigw_ctx* ctx, const aigw_bpe* bpe, const uint8_t* d_bodies, const uint64_t* d_offsets, const uint32_t* d_lens, uint32_t n, uint32_t max_len,
                                 uint64_t total_bytes, aigw_emb_count_result* d_results, void* stream, float* kernel_ms) {
  if (!ctx || !bpe) return -2;
  if (kernel_ms) kernel_ms[0] = kernel_ms[1] = kernel_ms[2] = kernel_ms[3] = 0;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  // every input costs at least three request bytes (two quotes and a comma); one row per four bytes covers inputs of two characters and up,
  // a request that would overflow the table is declined (AIGW_R_ARENA_FULL)
  const uint64_t text_cap64 = total_bytes / 4 + 1024;
  if (text_cap64 >= (1ull << 32)) { ctx->err = "aigw_embeddings_count: more than 16 GiB in one call; split it into waves"; return -2; }
  const uint32_t text_cap = (uint32_t)text_cap64;
  const uint32_t tok_cap = max_len / 2 + 64;
  const int grid = emb_scan_grid(ctx->sm_count);
  ENSURE(ctx->d_emb_tok, ctx->emb_tok_cap, (size_t)grid * tok_cap * 4, false);
  ENSURE(ctx->d_emb_toff, ctx->emb_toff_cap, (size_t)text_cap * 8, false);
  ENSURE(ctx->d_emb_tlen, ctx->emb_tlen_cap, (size_t)text_cap * 4, false);
  ENSURE(ctx->d_emb_cnt, ctx->emb_cnt_cap, (size_t)text_cap * 4, false);
  unsigned int* c0 = ctx->d_counters + (ctx->counter_next++ & 255);
  unsigned int* c1 = ctx->d_counters + (ctx->counter_next++ & 255);
  unsigned int* c2 = ctx->d_counters + (ctx->counter_next++ & 255);
  CK(cudaMemsetAsync(c0, 0, sizeof(unsigned int), st)); CK(cudaMemsetAsync(c1, 0, sizeof(unsigned int), st)); CK(cudaMemsetAsync(c2, 0, sizeof(unsigned int), st));
  EmbScanParams E; E.bodies = d_bodies; E.offsets = d_offsets; E.lens = d_lens; E.n = n; E.results = d_results; E.tok_ws = ctx->d_emb_tok; E.tok_cap = tok_cap;
  E.text_off = ctx->d_emb_toff; E.text_len = ctx->d_emb_tlen; E.text_cap = text_cap; E.next = c0; E.text_used = c1;
  cudaEvent_t* ev = ctx->stage_ev;
  if (kernel_ms) CK(cudaEventRecord(ev[0], st));
  CK(launch_emb_scan(E, ctx->sm_count, st));
  if (kernel_ms) CK(cudaEventRecord(ev[1], st));
  // the number of texts is only known on the device: read the row count back (4 bytes; the count kernel's grid is sized by it)
  unsigned int n_texts = 0;
  CK(cudaMemcpyAsync(&n_texts, c1, sizeof n_texts, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (n_texts > text_cap) n_texts = text_cap;   // requests past the capacity were declined; rows below it are all valid
  if (kernel_ms) CK(cudaEventRecord(ev[2], st));
  if (n_texts) {
    BpeParams P; P.text = d_bodies; P.offsets = ctx->d_emb_toff; P.lens = ctx->d_emb_tlen; P.n = n_texts; P.counts = ctx->d_emb_cnt; P.table = bpe->d_table; P.slots = bpe->slots; P.byte_to_id = bpe->d_b2i; P.next = c2;
    CK(launch_bpe_count(P, ctx->sm_count, st));
  }
  if (kernel_ms) CK(cudaEventRecord(ev[3], st));
  CK(launch_emb_sum(d_results, n, ctx->d_emb_cnt, st));
  if (kernel_ms) {
    CK(cudaEventRecord(ev[4], st)); CK(cudaEventSynchronize(ev[4]));
    CK(cudaEventElapsedTime(&kernel_ms[0], ev[0], ev[1])); CK(cudaEventElapsedTime(&kernel_ms[1], ev[2], ev[3])); CK(cudaEventElapsedTime(&kernel_ms[2], ev[3], ev[4])); CK(cudaEventElapsedTime(&kernel_ms[3], ev[0], ev[4]));
  }
  return 0;
}

int aigw_embeddings_count_host(aigw_ctx* ctx, const aigw_bpe* bpe, const uint8_t* bodies, const uint64_t* offsets, const uint32_t* lens, uint32_t n,
                               aigw_emb_count_result* results, uint64_t* h2d_bytes, uint64_t* d2h_bytes, float* kernel_ms) {
  if (!ctx || !bpe) return -2;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  uint64_t nbytes = 0; uint32_t max_len = 0;
  for (uint32_t i = 0; i < n; i++) { const uint64_t e = offsets[i] + lens[i]; if (e > nbytes) nbytes = e; if (lens[i] > max_len) max_len = lens[i]; if (offsets[i] & 15u) { ctx->err = "aigw_embeddings_count_host: request starts must be 16-byte aligned"; return -2; } }
  ENSURE(ctx->d_emb_body, ctx->emb_body_cap, nbytes + 64, false);
  ENSURE(ctx->d_emb_off, ctx->emb_off_cap, (size_t)n * 8, false);
  ENSURE(ctx->d_emb_len, ctx->emb_len_cap, (size_t)n * 4, false);
  ENSURE(ctx->d_emb_res, ctx->emb_res_cap, (size_t)n * sizeof(aigw_emb_count_result), false);
  cudaStream_t st = ctx->s_compute;
  CK(cudaMemcpyAsync(ctx->d_emb_body, bodies, nbytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->d_emb_off, offsets, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->d_emb_len, lens, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  if (int rc = aigw_embeddings_count_device(ctx, bpe, ctx->d_emb_body, ctx->d_emb_off, ctx->d_emb_len, n, max_len, nbytes, ctx->d_emb_res, st, kernel_ms)) return rc;
  CK(cudaMemcpyAsync(results, ctx->d_emb_res, (size_t)n * sizeof(aigw_emb_count_result), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (h2d_bytes) *h2d_bytes = nbytes + (uint64_t)n * 12;
  if (d2h_bytes) *d2h_bytes = (uint64_t)n * sizeof(aigw_emb_count_result) + 4;
  return 0;
}

// ------------------------------------------------------------------ SSE
int aigw_sse_usage_device(aigw_ctx* ctx, const uint8_t* d_bytes, const uint64_t* d_chunk_off, const uint32_t* d_chunk_first,
                          uint32_t n_streams, aigw_sse_result* d_results, void* stream, float* kernel_ms) {
  if (n_streams == 0) { if (kernel_ms) *kernel_ms = 0; return 0; }
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  SseParams P; P.bytes = d_bytes; P.chunk_off = d_chunk_off; P.chunk_first = d_chunk_first; P.n_streams = n_streams; P.results = d_results;
  P.next = ctx->d_counters + (ctx->counter_next++ & 255);
  CK(cudaMemsetAsync(P.next, 0, sizeof(unsigned int), st));
  if (kernel_ms) CK(cudaEventRecord(ctx->ev0, st));
  CK(launch_sse_usage(P, ctx->sm_count, st));
  if (kernel_ms) { CK(cudaEventRecord(ctx->ev1, st)); CK(cudaEventSynchronize(ctx->ev1)); CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1)); }
  return 0;
}

int aigw_sse_usage_host(aigw_ctx* ctx, const uint8_t* bytes, const uint64_t* chunk_off, const uint32_t* chunk_first,
                        uint32_t n_streams, uint32_t n_chunks, aigw_sse_result* results, uint64_t* h2d_bytes, uint64_t* d2h_bytes, float* kernel_ms) {
  if (n_streams == 0) return 0;
  cudaSetDevice(ctx->device);
  const uint64_t nbytes = chunk_off[n_chunks];
  ENSURE(ctx->d_sse_bytes, ctx->sse_bytes_cap, nbytes + 64, false);
  ENSURE(ctx->d_sse_coff, ctx->sse_coff_cap, ((size_t)n_chunks + 1) * 8, false);
  ENSURE(ctx->d_sse_first, ctx->sse_first_cap, ((size_t)n_streams + 1) * 4, false);
  ENSURE(ctx->d_sse_res, ctx->sse_res_cap, (size_t)n_streams * sizeof(aigw_sse_result), false);
  cudaStream_t st = ctx->s_compute;
  CK(cudaMemcpyAsync(ctx->d_sse_bytes, bytes, nbytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->d_sse_coff, chunk_off, ((size_t)n_chunks + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->d_sse_first, chunk_first, ((size_t)n_streams + 1) * 4, cudaMemcpyHostToDevice, st));
  SseParams P; P.bytes = ctx->d_sse_bytes; P.chunk_off = ctx->d_sse_coff; P.chunk_first = ctx->d_sse_first; P.n_streams = n_streams; P.results = ctx->d_sse_res;
  P.next = ctx->d_counters + (ctx->counter_next++ & 255);
  CK(cudaMemsetAsync(P.next, 0, sizeof(unsigned int), st));
  CK(cudaEventRecord(ctx->ev0, st));
  CK(launch_sse_usage(P, ctx->sm_count, st));
  CK(cudaEventRecord(ctx->ev1, st));
  CK(cudaMemcpyAsync(results, ctx->d_sse_res, (size_t)n_streams * sizeof(aigw_sse_result), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (kernel_ms) CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1));
  if (h2d_bytes) *h2d_bytes = nbytes + ((uint64_t)n_chunks + 1) * 8 + ((uint64_t)n_streams + 1) * 4;
  if (d2h_bytes) *d2h_bytes = (uint64_t)n_streams * sizeof(aigw_sse_result);
  return 0;
}

// ------------------------------------------------------------------ stateful per-chunk response streams
static int stream_pool_grow(aigw_ctx* ctx, uint32_t want) {
  auto& sp = ctx->sp;
  if (want <= sp.cap) return 0;
  uint32_t ncap = sp.cap ? sp.cap : 1024u;
  while (ncap < want) ncap *= 2;
  if (ncap > (1u << 22)) { ctx->err = "too many open streams"; return -3; }
  StreamSlot* nd = nullptr;
  CK(cudaMalloc(&nd, (size_t)ncap * sizeof(StreamSlot)));
  if (sp.d_slots) { CK(cudaMemcpyAsync(nd, sp.d_slots, (size_t)sp.cap * sizeof(StreamSlot), cudaMemcpyDeviceToDevice, ctx->s_compute)); CK(cudaStreamSynchronize(ctx->s_compute)); cudaFree(sp.d_slots); }
  sp.d_slots = nd;
  sp.carry.resize(ncap, 0); sp.gen.resize(ncap, 0); sp.stamp.resize(ncap, 0); sp.open.resize(ncap, 0);
  for (uint32_t i = ncap; i-- > sp.cap;) sp.free_list.push_back(i);
  sp.cap = ncap;
  return 0;
}
static bool stream_handle_ok(aigw_ctx* ctx, uint64_t h, uint32_t& slot) {
  auto& sp = ctx->sp;
  const uint32_t lo = (uint32_t)h; if (lo == 0 || lo > sp.cap) return false;
  slot = lo - 1;
  return sp.open[slot] && sp.gen[slot] == (uint32_t)(h >> 32);
}

int aigw_stream_open_batch(aigw_ctx* ctx, const aigw_stream_cfg* cfg, uint32_t n, uint64_t* handles) {
  if (!cfg || (n && !handles)) return -2;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  auto& sp = ctx->sp;
  std::lock_guard<std::mutex> lk(sp.mu);
  const char* model = cfg->request_model ? cfg->request_model : ""; const char* id = cfg->response_id ? cfg->response_id : "";
  if (cfg->kind < AIGW_STREAM_OPENAI || cfg->kind > AIGW_STREAM_MESSAGES_AWS_ANTHROPIC || strlen(model) > 160 || strlen(id) > 160 || !plain_json_text(model) || !plain_json_text(id)) {
    ctx->err = "stream cfg: unknown kind, or request_model / response_id need JSON escaping or exceed 160 bytes"; return -2;
  }
  if (sp.free_list.size() < n) { const int rc = stream_pool_grow(ctx, sp.cap + (uint32_t)(n - sp.free_list.size())); if (rc) return rc; }
  std::vector<uint8_t> tmpl(kStreamHdrBytes, 0);
  StreamSlot* t = (StreamSlot*)tmpl.data();   // header part only
  t->kind = (uint32_t)cfg->kind; t->beg = t->end = 0; t->flags = 0; t->tool_index = cfg->kind == AIGW_STREAM_GCP_ANTHROPIC ? -1 : 0; t->active_index = -1;
  t->created = cfg->created; t->model_len = (uint32_t)strlen(model); memcpy(t->model, model, t->model_len);
  if (cfg->kind == AIGW_STREAM_AWS_BEDROCK) { t->id_len = (uint32_t)strlen(id); memcpy(t->id, id, t->id_len); t->flags |= SF_HAVE_CREATED; }
  if (!sp.d_tmpl) CK(cudaMalloc(&sp.d_tmpl, kStreamHdrBytes));
  ENSURE(sp.d_ids, sp.d_ids_cap, (size_t)n * 4, false);
  ENSURE(sp.h_ids, sp.h_ids_cap, (size_t)n * 4, true);
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t slot = sp.free_list.back(); sp.free_list.pop_back();
    sp.open[slot] = 1; sp.gen[slot]++; sp.carry[slot] = 0;
    sp.h_ids[i] = slot; handles[i] = ((uint64_t)sp.gen[slot] << 32) | (uint64_t)(slot + 1);
  }
  cudaStream_t st = ctx->s_compute;
  CK(cudaMemcpyAsync(sp.d_tmpl, tmpl.data(), kStreamHdrBytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(sp.d_ids, sp.h_ids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  CK(launch_stream_init(sp.d_slots, sp.d_ids, n, sp.d_tmpl, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}
int aigw_stream_open(aigw_ctx* ctx, const aigw_stream_cfg* cfg, uint64_t* handle) { return aigw_stream_open_batch(ctx, cfg, 1, handle); }

int aigw_stream_close_batch(aigw_ctx* ctx, const uint64_t* handles, uint32_t n) {
  auto& sp = ctx->sp;
  std::lock_guard<std::mutex> lk(sp.mu);
  int rc = 0;
  for (uint32_t i = 0; i < n; i++) { uint32_t slot; if (!stream_handle_ok(ctx, handles[i], slot)) { rc = -2; continue; } sp.open[slot] = 0; sp.free_list.push_back(slot); }
  return rc;
}
int aigw_stream_close(aigw_ctx* ctx, uint64_t handle) { return aigw_stream_close_batch(ctx, &handle, 1); }

// One window of ResponseBody calls.  get(i) = {handle, bytes, len, eos} of call i.  zc_base != nullptr: every call's bytes lie in one
// mapped pinned buffer starting at zc_base (device view zc_dev): the kernels read them in place, nothing is staged or copied.
extern "C++" {
struct StreamCallIn { uint64_t handle; const uint8_t* bytes; uint32_t len; uint32_t eos; };
template <class GET>
static int stream_chunks_core(aigw_ctx* ctx, uint32_t n, GET&& get, aigw_chunk_result* results, const uint8_t** arena, const uint8_t* zc_base, const uint8_t* zc_dev) {
  auto& sp = ctx->sp;
  if (arena) *arena = nullptr;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  ENSURE(sp.h_steps, sp.h_steps_cap, (size_t)n * sizeof(StreamStep), true);
  sp.call_no++;
  uint64_t in_bytes = 0, out_bytes = 0;
  for (uint32_t i = 0; i < n; i++) {
    const StreamCallIn c = get(i);
    uint32_t slot;
    if (!stream_handle_ok(ctx, c.handle, slot) || (c.len && !c.bytes)) { ctx->err = "aigw_stream_chunks: bad handle"; return -2; }
    if (sp.stamp[slot] == sp.call_no) { ctx->err = "aigw_stream_chunks: a stream appears twice in one call"; return -2; }
    sp.stamp[slot] = sp.call_no;
    StreamStep& s = sp.h_steps[i];
    s.slot = slot; s.len = c.len; s.eos = c.eos ? 1u : 0u;
    if (zc_base) s.in_off = (uint64_t)(c.bytes - zc_base);
    else { s.in_off = in_bytes; in_bytes += ((uint64_t)c.len + 15u) & ~15ull; }
    // output bound: every unit of input (≥ 20 bytes) yields at most one chunk of ≤ 96 + id + model + its own text
    const uint64_t oc = 16ull * ((uint64_t)sp.carry[slot] + c.len) + 1024u;
    s.out_cap = (uint32_t)(oc > 0x7fffffffull ? 0x7fffffffull : oc);
    s.out_off = out_bytes; out_bytes += ((uint64_t)s.out_cap + 15u) & ~15ull;
  }
  if (!zc_base) { ENSURE(sp.h_in, sp.h_in_cap, in_bytes + 16, true); ENSURE(sp.d_in, sp.d_in_cap, in_bytes + 16, false); }
  ENSURE(sp.d_steps, sp.d_steps_cap, (size_t)n * sizeof(StreamStep), false);
  ENSURE(sp.d_res, sp.d_res_cap, (size_t)n * sizeof(aigw_chunk_result), false);
  ENSURE(sp.h_res, sp.h_res_cap, (size_t)n * sizeof(aigw_chunk_result), true);
  ENSURE(sp.d_out, sp.d_out_cap, out_bytes + 16, false);
  ENSURE(sp.d_packed, sp.d_packed_cap, out_bytes + 16, false);
  if (!sp.d_used) { CK(cudaMalloc(&sp.d_used, 8)); CK(cudaHostAlloc(&sp.h_used, 8, cudaHostAllocDefault)); }
  if (!zc_base) host_parallel_for(n, [&](uint32_t b, uint32_t e) { for (uint32_t i = b; i < e; i++) { const StreamCallIn c = get(i); if (c.len) memcpy(sp.h_in + sp.h_steps[i].in_off, c.bytes, c.len); } });   // no caller pointer is retained
  cudaStream_t st = ctx->s_compute;
  if (!zc_base) CK(cudaMemcpyAsync(sp.d_in, sp.h_in, in_bytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(sp.d_steps, sp.h_steps, (size_t)n * sizeof(StreamStep), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(sp.d_used, 0, 8, st));
  StreamParams P; P.slots = sp.d_slots; P.in = zc_base ? zc_dev : sp.d_in; P.out = sp.d_out; P.packed = sp.d_packed; P.packed_used = sp.d_used; P.packed_cap = sp.d_packed_cap; P.steps = sp.d_steps; P.results = sp.d_res; P.n = n;
  CK(launch_stream_steps(P, st));
  // results: straight into the caller's array when it is pinned (one DMA), else through the pinned staging array
  cudaPointerAttributes ra; const bool res_pinned = cudaPointerGetAttributes(&ra, results) == cudaSuccess && ra.type == cudaMemoryTypeHost;
  if (!res_pinned) cudaGetLastError();
  aigw_chunk_result* hres = res_pinned ? results : sp.h_res;
  CK(cudaMemcpyAsync(hres, sp.d_res, (size_t)n * sizeof(aigw_chunk_result), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(sp.h_used, sp.d_used, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const uint64_t used = *sp.h_used < sp.d_packed_cap ? *sp.h_used : sp.d_packed_cap;
  if (used) {
    ENSURE(sp.h_packed, sp.h_packed_cap, used + 16, true);
    CK(cudaMemcpyAsync(sp.h_packed, sp.d_packed, used, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  if (res_pinned) { for (uint32_t i = 0; i < n; i++) sp.carry[sp.h_steps[i].slot] = results[i].carry_len; }
  else host_parallel_for(n, [&](uint32_t b, uint32_t e) { for (uint32_t i = b; i < e; i++) { results[i] = sp.h_res[i]; sp.carry[sp.h_steps[i].slot] = sp.h_res[i].carry_len; } });   // a stream appears once per call: the carry writes are disjoint
  if (arena) *arena = sp.h_packed;
  return 0;
}
}  // extern "C++"
int aigw_stream_chunks(aigw_ctx* ctx, const aigw_chunk_in* in, uint32_t n, aigw_chunk_result* results, const uint8_t** arena) {
  std::lock_guard<std::mutex> lk(ctx->sp.mu);
  return stream_chunks_core(ctx, n, [&](uint32_t i) { return StreamCallIn{in[i].handle, in[i].bytes, in[i].len, in[i].eos}; }, results, arena, nullptr, nullptr);
}
/* structure-of-arrays form: chunk i of the call = base[off[i] .. off[i]+len[i]) for stream handles[i] (batch drivers, bench config 4).
 * When `base` is mapped pinned memory (aigw_host_alloc) the kernels read the chunks in place: no staging copy, no H2D of the bytes. */
int aigw_stream_chunks_soa(aigw_ctx* ctx, const uint64_t* handles, const uint8_t* base, const uint64_t* off, const uint32_t* len, const uint8_t* eos, uint32_t n,
                           aigw_chunk_result* results, const uint8_t** arena) {
  std::lock_guard<std::mutex> lk(ctx->sp.mu);
  const uint8_t* zc_dev = nullptr;
  {
    cudaPointerAttributes at;
    if (base && cudaPointerGetAttributes(&at, base) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) zc_dev = (const uint8_t*)at.devicePointer;
    else cudaGetLastError();
  }
  return stream_chunks_core(ctx, n, [&](uint32_t i) { return StreamCallIn{handles[i], base + off[i], len[i], eos ? (uint32_t)eos[i] : 0u}; }, results, arena, zc_dev ? base : nullptr, zc_dev);
}
int aigw_stream_chunk(aigw_ctx* ctx, uint64_t handle, const uint8_t* bytes, uint32_t len, int eos, uint8_t* out, uint32_t out_cap, aigw_chunk_result* res) {
  std::lock_guard<std::mutex> lk(ctx->sp.mu);
  aigw_chunk_in in; in.handle = handle; in.bytes = bytes; in.len = len; in.eos = eos ? 1u : 0u;
  const uint8_t* arena = nullptr;
  const int rc = stream_chunks_core(ctx, 1, [&](uint32_t) { return StreamCallIn{in.handle, in.bytes, in.len, in.eos}; }, res, &arena, nullptr, nullptr);
  if (rc) return rc;
  const uint32_t tot = res->out_len + res->model_len;
  if (tot > out_cap) return -4;
  if (tot) memcpy(out, arena + res->out_off, tot);
  res->out_off = 0;
  return 0;
}

// ------------------------------------------------------------------ S2: Bedrock eventstream → OpenAI SSE
static int fill_stream_params(aigw_ctx* ctx, BedrockStreamParams& P, const aigw_bedrock_stream_cfg* cfg) {
  memset(P.id, 0, sizeof P.id); memset(P.model, 0, sizeof P.model); P.id_len = P.model_len = 0; P.created = cfg ? cfg->created : 0;
  const char* id = cfg && cfg->response_id ? cfg->response_id : ""; const char* model = cfg && cfg->request_model ? cfg->request_model : "";
  if (strlen(id) > sizeof P.id || strlen(model) > sizeof P.model || !plain_json_text(id) || !plain_json_text(model)) { ctx->err = "response_id/request_model need JSON escaping or exceed 128 bytes"; return -2; }
  P.id_len = (uint32_t)strlen(id); memcpy(P.id, id, P.id_len); P.model_len = (uint32_t)strlen(model); memcpy(P.model, model, P.model_len);
  return 0;
}
int aigw_bedrock_stream_device(aigw_ctx* ctx, const aigw_bedrock_stream_cfg* cfg, const uint8_t* d_bytes, const uint64_t* d_stream_off, uint32_t n_streams,
                               uint64_t total_bytes, uint8_t* d_out, uint64_t out_capacity, aigw_stream_result* d_results, uint64_t* d_out_used,
                               void* stream, float* kernel_ms) {
  if (kernel_ms) *kernel_ms = 0;
  if (n_streams == 0) return 0;
  cudaSetDevice(ctx->device);
  BedrockStreamParams P;
  if (int rc = fill_stream_params(ctx, P, cfg)) return rc;
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  ENSURE(ctx->d_bs_work, ctx->bs_work_cap, bedrock_work_bytes(total_bytes, n_streams), false);
  P.bytes = d_bytes; P.stream_off = d_stream_off; P.off_base = 0; P.out_bias = 0; P.n_streams = n_streams; P.out = d_out; P.out_capacity = out_capacity; P.results = d_results;
  P.out_used = (unsigned long long*)d_out_used;
  bedrock_work_layout(P, ctx->d_bs_work, n_streams);
  ctx->counter_next = (ctx->counter_next + 1) & ~1;   // two adjacent counters
  P.next = ctx->d_counters + (ctx->counter_next & 255); ctx->counter_next += 2;
  CK(cudaMemsetAsync(d_out_used, 0, sizeof(uint64_t), st));
  if (kernel_ms) CK(cudaEventRecord(ctx->ev0, st));
  CK(launch_bedrock_stream(P, ctx->sm_count, st));
  if (kernel_ms) { CK(cudaEventRecord(ctx->ev1, st)); CK(cudaEventSynchronize(ctx->ev1)); CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1)); }
  return 0;
}
int aigw_bedrock_stream_host(aigw_ctx* ctx, const aigw_bedrock_stream_cfg* cfg, const uint8_t* bytes, const uint64_t* stream_off, uint32_t n_streams,
                             uint64_t out_capacity_hint, aigw_stream_batch_out* out) {
  memset(out, 0, sizeof *out);
  if (n_streams == 0) return 0;
  cudaSetDevice(ctx->device);
  BedrockStreamParams P0;
  if (int rc = fill_stream_params(ctx, P0, cfg)) return rc;
  // sub-batches of ~64 MiB of stream bytes
  constexpr uint64_t kChunk = 64ull << 20;
  std::vector<uint32_t> cb; cb.push_back(0);
  { uint64_t start = stream_off[0]; for (uint32_t i = 1; i < n_streams; i++) if (stream_off[i + 1] - start > kChunk) { cb.push_back(i); start = stream_off[i]; } cb.push_back(n_streams); }
  const int nch = (int)cb.size() - 1;
  const uint64_t total_in = stream_off[n_streams] - stream_off[0];
  const double ratio = out_capacity_hint ? (double)out_capacity_hint / (double)(total_in + 1) : 2.0;
  std::vector<uint64_t> out_cap(nch), out_base(nch);
  uint64_t max_in = 0, total_cap = 0; uint32_t max_n = 0;
  for (int c = 0; c < nch; c++) {
    const uint64_t ib = stream_off[cb[c + 1]] - stream_off[cb[c]]; const uint32_t nd = cb[c + 1] - cb[c];
    if (ib > max_in) max_in = ib; if (nd > max_n) max_n = nd;
    out_cap[c] = ((uint64_t)((double)ib * ratio) + (uint64_t)nd * 64 + 4096 + 255) & ~255ull;
    out_base[c] = total_cap; total_cap += out_cap[c];
  }
  const int nslots = nch < 2 ? 1 : 2;
  for (int k = 0; k < nslots; k++) {
    ENSURE(ctx->slot[k].d_in, ctx->slot[k].in_cap, max_in + 64, false);
    ENSURE(ctx->d_bs_off[k], ctx->bs_off_cap[k], ((size_t)max_n + 1) * 8, false);
  }
  ENSURE(ctx->d_bs_work, ctx->bs_work_cap, bedrock_work_bytes(max_in, max_n), false);
  ENSURE(ctx->h_out, ctx->h_out_cap, total_cap, true);
  ENSURE(ctx->h_sres, ctx->h_sres_cap, (size_t)n_streams * sizeof(aigw_stream_result), true);
  if ((size_t)nch > ctx->used_cap) {
    cudaFree(ctx->d_used_arr); cudaFreeHost(ctx->h_used_arr); ctx->used_cap = 0;
    const size_t cap = (size_t)nch + 64;
    CK(cudaMalloc(&ctx->d_used_arr, cap * 8)); CK(cudaHostAlloc(&ctx->h_used_arr, cap * 8, cudaHostAllocDefault));
    ctx->used_cap = cap;
  }
  uint8_t* dev_out = nullptr; aigw_stream_result* dev_res = nullptr;
  CK(cudaHostGetDevicePointer((void**)&dev_out, ctx->h_out, 0));
  CK(cudaHostGetDevicePointer((void**)&dev_res, ctx->h_sres, 0));
  uint64_t h2d = 0;
  CK(cudaMemsetAsync(ctx->d_used_arr, 0, (size_t)nch * 8, ctx->s_compute));
  CK(cudaEventRecord(ctx->ev0, ctx->s_compute));
  for (int c = 0; c < nch; c++) {
    ChunkSlot& S = ctx->slot[c % nslots];
    uint64_t* d_off = ctx->d_bs_off[c % nslots];
    const uint32_t b = cb[c], e = cb[c + 1], nd = e - b;
    const uint64_t ib = stream_off[e] - stream_off[b];
    if (c >= nslots) CK(cudaStreamWaitEvent(ctx->s_h2d, S.ev_k1, 0));
    CK(cudaMemcpyAsync(S.d_in, bytes + stream_off[b], ib, cudaMemcpyHostToDevice, ctx->s_h2d));
    CK(cudaMemcpyAsync(d_off, stream_off + b, ((size_t)nd + 1) * 8, cudaMemcpyHostToDevice, ctx->s_h2d));
    CK(cudaEventRecord(S.ev_h2d, ctx->s_h2d));
    h2d += ib + ((uint64_t)nd + 1) * 8;
    CK(cudaStreamWaitEvent(ctx->s_compute, S.ev_h2d, 0));
    BedrockStreamParams P = P0;
    P.bytes = S.d_in - stream_off[b]; P.stream_off = d_off; P.off_base = stream_off[b]; P.n_streams = nd;
    P.out = dev_out + out_base[c]; P.out_capacity = out_cap[c]; P.out_bias = out_base[c];
    P.results = dev_res + b; P.out_used = ctx->d_used_arr + c;
    bedrock_work_layout(P, ctx->d_bs_work, nd);
    ctx->counter_next = (ctx->counter_next + 1) & ~1;
    P.next = ctx->d_counters + (ctx->counter_next & 255); ctx->counter_next += 2;
    CK(launch_bedrock_stream(P, ctx->sm_count, ctx->s_compute));
    CK(cudaEventRecord(S.ev_k1, ctx->s_compute));
    out->gpu_launches += 2;
  }
  CK(cudaEventRecord(ctx->ev1, ctx->s_compute));
  CK(cudaMemcpyAsync(ctx->h_used_arr, ctx->d_used_arr, (size_t)nch * 8, cudaMemcpyDeviceToHost, ctx->s_compute));
  CK(cudaStreamSynchronize(ctx->s_compute));
  uint64_t d2h = (uint64_t)n_streams * sizeof(aigw_stream_result) + (uint64_t)nch * 8;
  for (int c = 0; c < nch; c++) d2h += ctx->h_used_arr[c] < out_cap[c] ? ctx->h_used_arr[c] : out_cap[c];
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  out->results = ctx->h_sres; out->out = ctx->h_out; out->out_used = total_cap; out->h2d_bytes = h2d; out->d2h_bytes = d2h; out->kernel_ms = ms;
  return 0;
}

// ------------------------------------------------------------------ B1: body mutation
static bool mut_path_ok(const char* p) {
  bool digits = true;
  for (const char* q = p; *q; q++) {
    const unsigned char c = (unsigned char)*q;
    if (c == '.' || c == '*' || c == '?' || c == '#' || c == '|' || c == ':' || c == '\\' || c == '@' || c < 0x21 || c > 0x7e || c == '"') return false;
    if (c < '0' || c > '9') digits = false;
  }
  return !digits && strcmp(p, "-1") != 0;
}
// isJSONValue (internal/bodymutator/body_mutator.go:33-75)
static bool mut_is_json_value(const std::string& value) {
  size_t b = 0, e = value.size();
  auto sp = [](unsigned char c) { return c == ' ' || c == '\t' || c == '\n' || c == '\v' || c == '\f' || c == '\r' || c == 0x85 || c == 0xA0; };
  while (b < e && sp((unsigned char)value[b])) b++;
  while (e > b && sp((unsigned char)value[e - 1])) e--;
  const std::string v = value.substr(b, e - b);
  if (!v.empty() && v.front() == '"' && v.back() == '"') return true;
  if (v == "0" || v == "true" || v == "false" || v == "null") return true;
  if (!v.empty()) {
    const char f = v[0];
    if ((f >= '0' && f <= '9') || f == '-' || f == '+') {
      bool num = true;
      for (char c : v) if ((c < '0' || c > '9') && c != '.' && c != '-' && c != '+' && c != 'e' && c != 'E') { num = false; break; }
      if (num) return true;
    }
  }
  if (!v.empty() && v.front() == '{' && v.back() == '}') return true;
  if (!v.empty() && v.front() == '[' && v.back() == ']') return true;
  return false;
}
// fold the configured remove / set lists into per-key actions (see mutate_kernel.cuh)
static int fill_mutate_params(aigw_ctx* ctx, MutateParams& P, const aigw_body_mutation* m) {
  memset(P.keys, 0, sizeof P.keys); memset(P.text, 0, sizeof P.text); P.n_keys = 0;
  P.text[kMutTextCap - 4] = ',';
  struct K { std::string name, raw; bool remove = false, set = false; };
  std::vector<K> keys;
  auto find = [&](const char* name) -> K* { for (auto& k : keys) if (k.name == name) return &k; return nullptr; };
  for (uint32_t i = 0; m && i < m->n_set; i++) {
    const char* path = m->set[i].path; const char* val = m->set[i].value ? m->set[i].value : "";
    if (!path || !*path) continue;
    if (!mut_path_ok(path)) { ctx->err = std::string("body mutation path is not a plain top-level key: ") + path; return -2; }
    std::string raw;
    if (mut_is_json_value(val)) raw = val;
    else {   // sjson.SetBytes of a Go string: plain quoting when nothing needs escaping
      for (const char* q = val; *q; q++) { const unsigned char c = (unsigned char)*q; if (c < ' ' || c > 0x7f || c == '"' || c == '\\') { ctx->err = std::string("body mutation value needs JSON escaping: ") + path; return -2; } }
      raw = std::string("\"") + val + "\"";
    }
    K* k = find(path);
    if (!k) { keys.push_back(K{}); k = &keys.back(); k->name = path; }
    k->set = true; k->raw = raw;
  }
  for (uint32_t i = 0; m && i < m->n_remove; i++) {
    const char* path = m->remove[i];
    if (!path || !*path) continue;
    if (!mut_path_ok(path)) { ctx->err = std::string("body mutation path is not a plain top-level key: ") + path; return -2; }
    K* k = find(path);
    if (!k) { keys.push_back(K{}); k = &keys.back(); k->name = path; }
    k->remove = true;
  }
  if (keys.size() > (size_t)kMutMaxKeys) { ctx->err = "more than 16 distinct body mutation keys"; return -2; }
  size_t o = 0;
  for (size_t i = 0; i < keys.size(); i++) {
    const K& k = keys[i]; MutateKey& mk = P.keys[i];
    const std::string memb = "\"" + k.name + "\":" + k.raw;
    if (o + k.name.size() + memb.size() + 8 > (size_t)kMutTextCap - 8) { ctx->err = "body mutation text exceeds 3 KiB"; return -2; }
    mk.name_off = (uint16_t)o; mk.name_len = (uint16_t)k.name.size(); memcpy(P.text + o, k.name.data(), k.name.size()); o += (k.name.size() + 3) & ~(size_t)3;
    mk.memb_off = (uint16_t)o; mk.memb_len = (uint16_t)memb.size(); memcpy(P.text + o, memb.data(), memb.size());
    mk.val_off = (uint16_t)(o + k.name.size() + 3); mk.val_len = (uint16_t)k.raw.size();
    o += (memb.size() + 3) & ~(size_t)3;
    mk.remove = k.remove; mk.set = k.set;
  }
  P.n_keys = (uint32_t)keys.size();
  return 0;
}
int aigw_body_mutate_device(aigw_ctx* ctx, const aigw_body_mutation* m, const uint8_t* d_bodies, const uint64_t* d_offsets, const uint32_t* d_lens, uint32_t n,
                            uint32_t max_len, uint8_t* d_out, uint64_t out_capacity, aigw_mut_result* d_results, uint64_t* d_out_used, void* stream, float* kernel_ms) {
  if (kernel_ms) *kernel_ms = 0;
  if (n == 0) return 0;
  cudaSetDevice(ctx->device);
  MutateParams P;
  if (int rc = fill_mutate_params(ctx, P, m)) return rc;
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  P.bodies = d_bodies; P.offsets = d_offsets; P.lens = d_lens; P.n = n; P.out = d_out; P.out_capacity = out_capacity; P.out_bias = 0; P.results = d_results;
  P.out_used = (unsigned long long*)d_out_used;
  P.next = ctx->d_counters + (ctx->counter_next++ & 255);
  CK(cudaMemsetAsync(P.next, 0, sizeof(unsigned int), st));
  CK(cudaMemsetAsync(d_out_used, 0, sizeof(uint64_t), st));
  if (kernel_ms) CK(cudaEventRecord(ctx->ev0, st));
  CK(launch_body_mutate(P, max_len ? max_len : 65536u, ctx->sm_count, st));
  if (kernel_ms) { CK(cudaEventRecord(ctx->ev1, st)); CK(cudaEventSynchronize(ctx->ev1)); CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1)); }
  return 0;
}
int aigw_body_mutate_host(aigw_ctx* ctx, const aigw_body_mutation* m, const uint8_t* bodies, const uint64_t* offsets, const uint32_t* lens, uint32_t n,
                          aigw_mut_batch_out* out) {
  // Same pipeline as aigw_chat_translate_host: 256 MiB chunks, the H2D copy of chunk c+1 overlaps the kernel of chunk c, the
  // kernel stores records and results straight into mapped pinned host memory, one synchronisation at the end.
  memset(out, 0, sizeof *out);
  if (n == 0) return 0;
  cudaSetDevice(ctx->device);
  MutateParams P0;
  if (int rc = fill_mutate_params(ctx, P0, m)) return rc;
  uint64_t extra = 0;
  for (uint32_t k = 0; k < P0.n_keys; k++) extra += P0.keys[k].memb_len + 2;
  const uint64_t kChunkBytes = 256ull << 20;
  std::vector<uint32_t> cb; cb.push_back(0);
  uint32_t max_len = 0;
  {
    uint64_t start = offsets[0];
    for (uint32_t i = 0; i < n; i++) {
      const uint64_t end = offsets[i] + lens[i];
      if (end - start > kChunkBytes && i > cb.back()) { cb.push_back(i); start = offsets[i]; }
      if (lens[i] > max_len) max_len = lens[i];
    }
    cb.push_back(n);
  }
  const int nch = (int)cb.size() - 1;
  std::vector<uint64_t> in_bytes(nch), out_cap(nch), out_base(nch);
  uint64_t max_in = 0, total_cap = 0; uint32_t max_docs = 0;
  for (int c = 0; c < nch; c++) {
    const uint32_t b = cb[c], e = cb[c + 1];
    const uint64_t ib = offsets[e - 1] + lens[e - 1] - offsets[b];
    in_bytes[c] = ib; if (ib > max_in) max_in = ib; if (e - b > max_docs) max_docs = e - b;
    out_cap[c] = (ib + (uint64_t)(e - b) * (extra + 32) + 4096 + 255) & ~255ull;
    out_base[c] = total_cap; total_cap += out_cap[c];
  }
  const int nslots = nch < 2 ? 1 : 2;
  for (int k = 0; k < nslots; k++) {
    ChunkSlot& S = ctx->slot[k];
    ENSURE(S.d_in, S.in_cap, max_in + 64, false);
    if (S.doc_cap < max_docs) { cudaFree(S.d_off); cudaFree(S.d_len); S.doc_cap = 0; const size_t dc = (size_t)max_docs + max_docs / 8 + 16; CK(cudaMalloc(&S.d_off, dc * 8)); CK(cudaMalloc(&S.d_len, dc * 4)); S.doc_cap = dc; }
  }
  ENSURE(ctx->h_out, ctx->h_out_cap, total_cap, true);
  ENSURE(ctx->h_mres, ctx->h_mres_cap, (size_t)n * sizeof(aigw_mut_result), true);
  if ((size_t)nch > ctx->used_cap) {
    cudaFree(ctx->d_used_arr); cudaFreeHost(ctx->h_used_arr); ctx->used_cap = 0;
    const size_t cap = (size_t)nch + 64;
    CK(cudaMalloc(&ctx->d_used_arr, cap * 8)); CK(cudaHostAlloc(&ctx->h_used_arr, cap * 8, cudaHostAllocDefault));
    ctx->used_cap = cap;
  }
  uint8_t* dev_out = nullptr; aigw_mut_result* dev_res = nullptr;
  CK(cudaHostGetDevicePointer((void**)&dev_out, ctx->h_out, 0));
  CK(cudaHostGetDevicePointer((void**)&dev_res, ctx->h_mres, 0));
  uint64_t h2d = 0;
  CK(cudaMemsetAsync(ctx->d_used_arr, 0, (size_t)nch * 8, ctx->s_compute));
  CK(cudaEventRecord(ctx->ev0, ctx->s_compute));
  for (int c = 0; c < nch; c++) {
    ChunkSlot& S = ctx->slot[c % nslots];
    const uint32_t b = cb[c], e = cb[c + 1], nd = e - b;
    if (c >= nslots) CK(cudaStreamWaitEvent(ctx->s_h2d, S.ev_k1, 0));
    CK(cudaMemcpyAsync(S.d_in, bodies + offsets[b], in_bytes[c], cudaMemcpyHostToDevice, ctx->s_h2d));
    CK(cudaMemcpyAsync(S.d_off, offsets + b, (size_t)nd * 8, cudaMemcpyHostToDevice, ctx->s_h2d));
    CK(cudaMemcpyAsync(S.d_len, lens + b, (size_t)nd * 4, cudaMemcpyHostToDevice, ctx->s_h2d));
    CK(cudaEventRecord(S.ev_h2d, ctx->s_h2d));
    h2d += in_bytes[c] + (uint64_t)nd * 12;
    CK(cudaStreamWaitEvent(ctx->s_compute, S.ev_h2d, 0));
    MutateParams P = P0;
    P.bodies = S.d_in - offsets[b]; P.offsets = S.d_off; P.lens = S.d_len; P.n = nd;
    P.out = dev_out + out_base[c]; P.out_capacity = out_cap[c]; P.out_bias = out_base[c]; P.results = dev_res + b;
    P.out_used = ctx->d_used_arr + c;
    P.next = ctx->d_counters + (ctx->counter_next++ & 255);
    CK(cudaMemsetAsync(P.next, 0, sizeof(unsigned int), ctx->s_compute));
    CK(launch_body_mutate(P, max_len, ctx->sm_count, ctx->s_compute));
    CK(cudaEventRecord(S.ev_k1, ctx->s_compute));
    out->gpu_launches += 1;
  }
  CK(cudaEventRecord(ctx->ev1, ctx->s_compute));
  CK(cudaMemcpyAsync(ctx->h_used_arr, ctx->d_used_arr, (size_t)nch * 8, cudaMemcpyDeviceToHost, ctx->s_compute));
  CK(cudaStreamSynchronize(ctx->s_compute));
  uint64_t d2h = (uint64_t)n * sizeof(aigw_mut_result) + (uint64_t)nch * 8;
  for (int c = 0; c < nch; c++) d2h += ctx->h_used_arr[c] < out_cap[c] ? ctx->h_used_arr[c] : out_cap[c];
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  out->results = ctx->h_mres; out->out = ctx->h_out; out->out_used = total_cap; out->h2d_bytes = h2d; out->d2h_bytes = d2h; out->kernel_ms = ms;
  return 0;
}

// ------------------------------------------------------------------ SigV4 payload hash
static int sha_common(aigw_ctx* ctx, const uint8_t* d_bytes, const uint64_t* d_off, const uint32_t* d_len, const aigw_doc_result* d_res, uint32_t n, uint8_t* d_dig, void* stream, float* kernel_ms) {
  if (kernel_ms) *kernel_ms = 0;
  if (n == 0) return 0;
  cudaSetDevice(ctx->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  if (kernel_ms) CK(cudaEventRecord(ctx->ev0, st));
  CK(launch_sha256(d_bytes, d_off, d_len, d_res, n, d_dig, st));
  if (kernel_ms) { CK(cudaEventRecord(ctx->ev1, st)); CK(cudaEventSynchronize(ctx->ev1)); CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1)); }
  return 0;
}
int aigw_sha256_device(aigw_ctx* ctx, const uint8_t* d_bytes, const uint64_t* d_off, const uint32_t* d_len, uint32_t n, uint8_t* d_digests, void* stream, float* kernel_ms) {
  return sha_common(ctx, d_bytes, d_off, d_len, nullptr, n, d_digests, stream, kernel_ms);
}
int aigw_chat_body_sha256_device(aigw_ctx* ctx, const uint8_t* d_out, const aigw_doc_result* d_results, uint32_t n, uint8_t* d_digests, void* stream, float* kernel_ms) {
  return sha_common(ctx, d_out, nullptr, nullptr, d_results, n, d_digests, stream, kernel_ms);
}
int aigw_sha256_host(aigw_ctx* ctx, const uint8_t* bytes, const uint64_t* off, const uint32_t* len, uint32_t n, uint8_t* digests) {
  if (n == 0) return 0;
  cudaSetDevice(ctx->device);
  uint64_t lo = ~0ull, hi = 0;
  for (uint32_t i = 0; i < n; i++) { if (off[i] < lo) lo = off[i]; if (off[i] + len[i] > hi) hi = off[i] + len[i]; }
  const uint64_t nbytes = hi - lo;
  ChunkSlot& S = ctx->slot[0];
  ENSURE(S.d_in, S.in_cap, nbytes + 64, false);
  if (S.doc_cap < n) { cudaFree(S.d_off); cudaFree(S.d_len); S.doc_cap = 0; const size_t dc = (size_t)n + n / 8 + 16; CK(cudaMalloc(&S.d_off, dc * 8)); CK(cudaMalloc(&S.d_len, dc * 4)); S.doc_cap = dc; }
  ENSURE(ctx->d_sse_res, ctx->sse_res_cap, (size_t)n * 32, false);
  cudaStream_t st = ctx->s_compute;
  CK(cudaMemcpyAsync(S.d_in, bytes + lo, nbytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(S.d_off, off, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(S.d_len, len, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  CK(launch_sha256(S.d_in - lo, S.d_off, S.d_len, nullptr, n, (uint8_t*)ctx->d_sse_res, st));
  CK(cudaMemcpyAsync(digests, ctx->d_sse_res, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

// ------------------------------------------------------------------ CEL cost expressions
int aigw_cost_compile(aigw_ctx* ctx, const char* expr, aigw_cost_program** out) {
  *out = nullptr;
  cudaSetDevice(ctx->device);
  aigw_cost_program* p = new aigw_cost_program();
  std::string err;
  const int rc = cel_compile(expr ? expr : "", p->h, err);
  if (rc) { ctx->err = std::string(rc == 1 ? "CEL expression outside the compiled subset: " : "CEL expression rejected: ") + err; delete p; return rc == 1 ? -2 : -3; }
  std::vector<CelInstr> padded(p->h.code); padded.resize(kCelMaxInstr, CelInstr{});
  if (cudaMalloc(&p->h.d_code, sizeof(CelInstr) * kCelMaxInstr) != cudaSuccess || cudaMalloc(&p->h.d_strings, p->h.strings.size() + 16) != cudaSuccess) { ctx->err = "cudaMalloc"; delete p; return (int)cudaErrorMemoryAllocation; }
  CK(cudaMemcpy(p->h.d_code, padded.data(), sizeof(CelInstr) * kCelMaxInstr, cudaMemcpyHostToDevice));
  if (!p->h.strings.empty()) CK(cudaMemcpy(p->h.d_strings, p->h.strings.data(), p->h.strings.size(), cudaMemcpyHostToDevice));
  *out = p;
  return 0;
}
void aigw_cost_program_free(aigw_ctx* ctx, aigw_cost_program* p) { if (!p) return; cudaSetDevice(ctx->device); cudaFree(p->h.d_code); cudaFree(p->h.d_strings); delete p; }

static int cel_fill(aigw_ctx* ctx, CelLaunch& L, aigw_cost_program* const* progs, uint32_t n_progs, const char* model, const char* backend, const char* route) {
  if (n_progs > (uint32_t)kCelMaxProgs) { ctx->err = "more than 8 CEL programs per call"; return -2; }
  memset(&L.cs, 0, sizeof L.cs);
  auto put = [&](char* dst, uint32_t& len, const char* src) -> bool { const size_t l = src ? strlen(src) : 0; if (l >= (size_t)kCelStrCap) return false; if (l) memcpy(dst, src, l); len = (uint32_t)l; return true; };
  if (!put(L.cs.model, L.cs.model_len, model) || !put(L.cs.backend, L.cs.backend_len, backend) || !put(L.cs.route, L.cs.route_len, route)) { ctx->err = "model / backend / route_name longer than 255 bytes"; return -2; }
  L.n_progs = n_progs;
  for (uint32_t p = 0; p < n_progs; p++) {
    const CelProgramHost& h = progs[p]->h;
    L.code[p] = h.d_code; L.strings[p] = h.d_strings; L.result_is_int[p] = h.result_is_int;
    uint32_t bits = 0;
    for (size_t k = 0; k < h.sites.size(); k++) {   // string comparisons that do not involve the per-record model
      const CelHostSite& st = h.sites[k];
      auto str = [&](uint8_t kind, uint32_t off, uint32_t len) { return kind == 0 ? h.strings.substr(off, len) : kind == 1 ? std::string(L.cs.backend, L.cs.backend_len) : std::string(L.cs.route, L.cs.route_len); };
      if ((str(st.lk, st.loff, st.llen) == str(st.rk, st.roff, st.rlen)) != st.negate) bits |= 1u << k;
    }
    L.host_bits[p] = bits;
  }
  return 0;
}
int aigw_usage_costs_cel_device(aigw_ctx* ctx, const aigw_sse_result* d_results, uint32_t n, aigw_cost_program* const* progs, uint32_t n_progs,
                                const uint8_t* d_model_bytes, const uint32_t* d_model_off, const uint32_t* d_model_len, const char* model, const char* backend,
                                const char* route_name, uint64_t* d_costs, uint8_t* d_errs, void* stream) {
  if (n == 0 || n_progs == 0) return 0;
  cudaSetDevice(ctx->device);
  CelLaunch L;
  if (int rc = cel_fill(ctx, L, progs, n_progs, model, backend, route_name)) return rc;
  L.results = d_results; L.n = n; L.model_bytes = d_model_bytes; L.model_off = d_model_off; L.model_len = d_model_len;
  L.costs = (unsigned long long*)d_costs; L.errs = d_errs;
  CK(launch_cel(L, stream ? (cudaStream_t)stream : ctx->s_compute));
  return 0;
}
int aigw_usage_costs_cel_host(aigw_ctx* ctx, const aigw_sse_result* results, uint32_t n, aigw_cost_program* const* progs, uint32_t n_progs,
                              const uint8_t* model_bytes, uint64_t model_bytes_len, const uint32_t* model_off, const uint32_t* model_len, const char* model,
                              const char* backend, const char* route_name, uint64_t* costs, uint8_t* errs) {
  if (n == 0 || n_progs == 0) return 0;
  cudaSetDevice(ctx->device);
  const size_t nres = (size_t)n * sizeof(aigw_sse_result), nout = (size_t)n * n_progs;
  ENSURE(ctx->d_sse_res, ctx->sse_res_cap, nres, false);
  ENSURE(ctx->d_sse_coff, ctx->sse_coff_cap, nout * 9 + 64, false);
  ENSURE(ctx->d_sse_bytes, ctx->sse_bytes_cap, model_bytes_len + (size_t)n * 8 + 64, false);
  cudaStream_t st = ctx->s_compute;
  CK(cudaMemcpyAsync(ctx->d_sse_res, results, nres, cudaMemcpyHostToDevice, st));
  uint32_t* d_off = nullptr; uint32_t* d_len = nullptr;
  if (model_off && model_len) {
    d_off = (uint32_t*)ctx->d_sse_bytes; d_len = d_off + n;
    uint8_t* d_mb = (uint8_t*)(d_len + n);
    CK(cudaMemcpyAsync(d_off, model_off, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_len, model_len, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_mb, model_bytes, model_bytes_len, cudaMemcpyHostToDevice, st));
    if (int rc = aigw_usage_costs_cel_device(ctx, ctx->d_sse_res, n, progs, n_progs, d_mb, d_off, d_len, model, backend, route_name, (uint64_t*)ctx->d_sse_coff, (uint8_t*)ctx->d_sse_coff + nout * 8, st)) return rc;
  } else if (int rc = aigw_usage_costs_cel_device(ctx, ctx->d_sse_res, n, progs, n_progs, nullptr, nullptr, nullptr, model, backend, route_name, (uint64_t*)ctx->d_sse_coff, (uint8_t*)ctx->d_sse_coff + nout * 8, st)) return rc;
  CK(cudaMemcpyAsync(costs, ctx->d_sse_coff, nout * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(errs, (uint8_t*)ctx->d_sse_coff + nout * 8, nout, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

// ------------------------------------------------------------------ R1 + C2
static int response_usage_device_impl(aigw_ctx* ctx, const uint8_t* d_bodies, const uint64_t* d_offsets, const uint32_t* d_lens, uint32_t n,
                                      aigw_sse_result* d_results, void* stream, float* kernel_ms, int embeddings) {
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  if (kernel_ms) CK(cudaEventRecord(ctx->ev0, st));
  CK(launch_response_usage(d_bodies, d_offsets, d_lens, n, d_results, st, embeddings));
  if (kernel_ms) { CK(cudaEventRecord(ctx->ev1, st)); CK(cudaEventSynchronize(ctx->ev1)); CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1)); }
  return 0;
}

int aigw_response_usage_device(aigw_ctx* ctx, const uint8_t* d_bodies, const uint64_t* d_offsets, const uint32_t* d_lens, uint32_t n,
                               aigw_sse_result* d_results, void* stream, float* kernel_ms) {
  return response_usage_device_impl(ctx, d_bodies, d_offsets, d_lens, n, d_results, stream, kernel_ms, 0);
}
int aigw_embeddings_response_usage_device(aigw_ctx* ctx, const uint8_t* d_bodies, const uint64_t* d_offsets, const uint32_t* d_lens, uint32_t n,
                                          aigw_sse_result* d_results, void* stream, float* kernel_ms) {
  return response_usage_device_impl(ctx, d_bodies, d_offsets, d_lens, n, d_results, stream, kernel_ms, 1);
}
int aigw_completions_response_usage_device(aigw_ctx* ctx, const uint8_t* d_bodies, const uint64_t* d_offsets, const uint32_t* d_lens, uint32_t n,
                                           aigw_sse_result* d_results, void* stream, float* kernel_ms) {
  return response_usage_device_impl(ctx, d_bodies, d_offsets, d_lens, n, d_results, stream, kernel_ms, 2);
}

static int response_usage_host_impl(aigw_ctx* ctx, const uint8_t* bodies, const uint64_t* offsets, const uint32_t* lens, uint32_t n, aigw_sse_result* results,
                                    const int32_t* cost_types, uint32_t n_costs, uint64_t* costs, int embeddings) {
  if (n == 0) return 0;
  cudaSetDevice(ctx->device);
  const uint64_t nbytes = offsets[n - 1] + lens[n - 1] - offsets[0];
  ENSURE(ctx->d_sse_bytes, ctx->sse_bytes_cap, nbytes + 64, false);
  ENSURE(ctx->d_sse_coff, ctx->sse_coff_cap, ((size_t)n + 1) * 8 + (size_t)n_costs * 8 * n + 64, false);
  ENSURE(ctx->d_sse_first, ctx->sse_first_cap, ((size_t)n + 1) * 4 + (size_t)n_costs * 4 + 64, false);
  ENSURE(ctx->d_sse_res, ctx->sse_res_cap, (size_t)n * sizeof(aigw_sse_result), false);
  cudaStream_t st = ctx->s_compute;
  CK(cudaMemcpyAsync(ctx->d_sse_bytes, bodies + offsets[0], nbytes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->d_sse_coff, offsets, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->d_sse_first, lens, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  CK(launch_response_usage(ctx->d_sse_bytes - offsets[0], ctx->d_sse_coff, ctx->d_sse_first, n, ctx->d_sse_res, st, embeddings));
  CK(cudaMemcpyAsync(results, ctx->d_sse_res, (size_t)n * sizeof(aigw_sse_result), cudaMemcpyDeviceToHost, st));
  if (n_costs && costs) {
    int32_t* d_types = (int32_t*)(ctx->d_sse_first + n + 1);
    unsigned long long* d_costs = (unsigned long long*)(ctx->d_sse_coff + n + 1);
    CK(cudaMemcpyAsync(d_types, cost_types, (size_t)n_costs * 4, cudaMemcpyHostToDevice, st));
    CK(launch_usage_costs(ctx->d_sse_res, n, d_types, n_costs, d_costs, st));
    CK(cudaMemcpyAsync(costs, d_costs, (size_t)n * n_costs * 8, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  return 0;
}
int aigw_response_usage_host(aigw_ctx* ctx, const uint8_t* bodies, const uint64_t* offsets, const uint32_t* lens, uint32_t n, aigw_sse_result* results,
                             const int32_t* cost_types, uint32_t n_costs, uint64_t* costs) {
  return response_usage_host_impl(ctx, bodies, offsets, lens, n, results, cost_types, n_costs, costs, 0);
}
int aigw_embeddings_response_usage_host(aigw_ctx* ctx, const uint8_t* bodies, const uint64_t* offsets, const uint32_t* lens, uint32_t n, aigw_sse_result* results,
                                        const int32_t* cost_types, uint32_t n_costs, uint64_t* costs) {
  return response_usage_host_impl(ctx, bodies, offsets, lens, n, results, cost_types, n_costs, costs, 1);
}
int aigw_completions_response_usage_host(aigw_ctx* ctx, const uint8_t* bodies, const uint64_t* offsets, const uint32_t* lens, uint32_t n, aigw_sse_result* results,
                                         const int32_t* cost_types, uint32_t n_costs, uint64_t* costs) {
  return response_usage_host_impl(ctx, bodies, offsets, lens, n, results, cost_types, n_costs, costs, 2);
}

int aigw_usage_costs_device(aigw_ctx* ctx, const aigw_sse_result* d_results, uint32_t n, const int32_t* d_cost_types, uint32_t n_costs, uint64_t* d_costs, void* stream) {
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->s_compute;
  CK(launch_usage_costs(d_results, n, d_cost_types, n_costs, (unsigned long long*)d_costs, st));
  return 0;
}

}  // extern "C"
