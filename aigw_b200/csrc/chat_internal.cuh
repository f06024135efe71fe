// See chat_kernel.cuh for the design.  sm_100a only.
//
// v2 layout of the work (driven by profiles/r01_chat_v1.md: 72 % of v1's time was single-lane
// sequential code at ~22 cycles per instruction):
//   * tokens carry their byte (tty) and a precomputed key / value id (tkid) that 32 lanes compute in
//     parallel, so the schema walk compares one byte instead of strings;
//   * the copy-op under construction lives in registers; shared memory is touched once per finished op;
//   * the output record is assembled as 16-byte chunks (one chunk per lane, funnel-shifted unaligned
//     reads from shared memory) and stored straight to the arena — no shared-memory image of the
//     output, which lifts residency from 12 to 17+ warps per SM.
#pragma once
#include "chat_kernel.cuh"

namespace aigw {

static __device__ __constant__ LitTable c_lits = make_lit_table();
static_assert(make_lit_table().off[L_COUNT] + 24 <= sizeof(LitTable::bytes), "literal table overflow (keep slack for unaligned reads)");

#define FULL 0xffffffffu
#ifndef AIGW_WALK_BLOCKS
#define AIGW_WALK_BLOCKS 4
#endif

// ------------------------------------------------------------------ small device helpers
__device__ __forceinline__ uint32_t nib_from_ff(uint32_t m) {  // m: 0xFF per selected byte → 4-bit mask
  return ((m & 0x08040201u) * 0x01010101u) >> 24;
}
__device__ __forceinline__ bool is_ws(uint32_t c) { return c == ' ' || c == '\n' || c == '\r' || c == '\t'; }
__device__ __forceinline__ bool is_op(uint32_t c) { return c == '{' || c == '}' || c == '[' || c == ']' || c == ':' || c == ','; }
__device__ __forceinline__ bool is_digit(uint32_t c) { return c - '0' < 10u; }

// ------------------------------------------------------------------ key / value ids
enum Kid : uint8_t {
  K_NONE = 0,
  K_model, K_messages, K_max_tokens, K_max_completion_tokens, K_modalities, K_temperature, K_top_p, K_tools, K_tool_choice, K_thinking, K_top_logprobs,
  K_stop, K_stream, K_stream_options, K_service_tier, K_seed, K_safetySettings, K_frequency_penalty, K_logit_bias, K_logprobs, K_n, K_presence_penalty,
  K_parallel_tool_calls, K_prediction, K_response_format, K_reasoning_effort, K_verbosity, K_user, K_audio, K_web_search_options, K_generationConfig,
  K_guided_choice, K_guided_regex, K_guided_json, K_TOP_END,
  K_role = K_TOP_END, K_content, K_name, K_tool_calls, K_tool_call_id, K_refusal, K_type, K_text, K_cache_control, K_ttl, K_signature, K_redactedContent,
  K_id, K_function, K_arguments, K_description, K_strict, K_parameters, K_google_search, K_budget_tokens, K_includeThoughts, K_include_usage,
  K_input, K_encoding_format, K_dimensions, K_auto_truncate, K_task_type, K_title,   // /v1/embeddings
  K_COUNT
};
static_assert(K_TOP_END <= 63, "top-level seen mask is 64 bits");
static_assert(K_COUNT <= 64, "ids are 6 bits in the token word");
enum Vid : uint8_t {
  V_NONE = 0, V_user, V_assistant, V_system, V_developer, V_tool, V_text, V_refusal, V_thinking, V_redacted_thinking, V_ephemeral,
  V_enabled, V_disabled, V_adaptive, V_auto, V_required, V_image_url, V_input_audio, V_file,
  V_tool_use, V_tool_result, V_custom, V_any, V_none   // /v1/messages content blocks, tools, tool_choice
};

// Perfect-enough hash tables (FNV-1a, open addressing, verified by a byte compare) built at compile time and copied to
// shared memory by the index kernel: every lane runs the same few instructions whatever the string is.
#define AIGW_KEYS(X) \
  X("n", K_n) X("id", K_id) X("ttl", K_ttl) X("role", K_role) X("name", K_name) X("type", K_type) X("text", K_text) X("stop", K_stop) X("seed", K_seed) X("user", K_user) \
  X("model", K_model) X("tools", K_tools) X("top_p", K_top_p) X("audio", K_audio) X("stream", K_stream) X("strict", K_strict) X("content", K_content) X("refusal", K_refusal) \
  X("messages", K_messages) X("thinking", K_thinking) X("logprobs", K_logprobs) X("function", K_function) X("verbosity", K_verbosity) X("signature", K_signature) \
  X("arguments", K_arguments) X("max_tokens", K_max_tokens) X("modalities", K_modalities) X("tool_calls", K_tool_calls) X("logit_bias", K_logit_bias) X("prediction", K_prediction) \
  X("parameters", K_parameters) X("temperature", K_temperature) X("tool_choice", K_tool_choice) X("description", K_description) X("guided_json", K_guided_json) \
  X("service_tier", K_service_tier) X("top_logprobs", K_top_logprobs) X("tool_call_id", K_tool_call_id) X("guided_regex", K_guided_regex) X("cache_control", K_cache_control) \
  X("guided_choice", K_guided_choice) X("budget_tokens", K_budget_tokens) X("google_search", K_google_search) X("include_usage", K_include_usage) X("stream_options", K_stream_options) \
  X("safetySettings", K_safetySettings) X("response_format", K_response_format) X("redactedContent", K_redactedContent) X("includeThoughts", K_includeThoughts) \
  X("presence_penalty", K_presence_penalty) X("reasoning_effort", K_reasoning_effort) X("generationConfig", K_generationConfig) X("frequency_penalty", K_frequency_penalty) \
  X("web_search_options", K_web_search_options) X("parallel_tool_calls", K_parallel_tool_calls) X("max_completion_tokens", K_max_completion_tokens) \
  X("input", K_input) X("encoding_format", K_encoding_format) X("dimensions", K_dimensions) X("auto_truncate", K_auto_truncate) X("task_type", K_task_type) X("title", K_title)
#define AIGW_VALS(X) \
  X("user", V_user) X("tool", V_tool) X("text", V_text) X("auto", V_auto) X("system", V_system) X("refusal", V_refusal) X("enabled", V_enabled) X("thinking", V_thinking) \
  X("disabled", V_disabled) X("adaptive", V_adaptive) X("required", V_required) X("assistant", V_assistant) X("developer", V_developer) X("ephemeral", V_ephemeral) \
  X("redacted_thinking", V_redacted_thinking) X("image_url", V_image_url) X("input_audio", V_input_audio) X("file", V_file)
// the value strings a /v1/messages request can carry (own table: the chat table above is full enough for its 32 slots)
#define AIGW_MVALS(X) \
  X("user", V_user) X("assistant", V_assistant) X("text", V_text) X("ephemeral", V_ephemeral) X("auto", V_auto) X("tool", V_tool) \
  X("tool_use", V_tool_use) X("tool_result", V_tool_result) X("custom", V_custom) X("any", V_any) X("none", V_none)

// Response direction ((P.schema & 48) == AIGW_SCHEMA_RESP_AWS_BEDROCK): the index kernel loads this key table instead; ids share
// the 6-bit field of the token word.  awsbedrock.ConverseResponse, internal/apischema/awsbedrock/awsbedrock.go:178-182,264-279,330-432.
enum RKid : uint8_t {
  RK_NONE = 0, RK_output, RK_message, RK_content, RK_role, RK_text, RK_toolUse, RK_toolUseId, RK_name, RK_input, RK_reasoningContent, RK_reasoningText,
  RK_signature, RK_redactedContent, RK_stopReason, RK_usage, RK_inputTokens, RK_outputTokens, RK_totalTokens, RK_cacheReadInputTokens, RK_cacheWriteInputTokens,
  RK_serviceTier, RK_type, RK_metrics, RK_latencyMs, RK_document, RK_image, RK_toolResult, RK_cachePoint,
  // anthropic.Message (buffered GCP / AWS Anthropic responses)
  RK_id, RK_model, RK_stop_reason, RK_thinking, RK_data, RK_input_tokens, RK_output_tokens, RK_cache_read_input_tokens, RK_cache_creation_input_tokens, RK_stop_sequence,
  // error bodies (Translator.ResponseError)
  RK_error, RK_status, RK_details, RK_code, RK_request_id, RK_COUNT
};
#define AIGW_RKEYS(X) \
  X("output", RK_output) X("message", RK_message) X("content", RK_content) X("role", RK_role) X("text", RK_text) X("toolUse", RK_toolUse) X("toolUseId", RK_toolUseId) \
  X("name", RK_name) X("input", RK_input) X("reasoningContent", RK_reasoningContent) X("reasoningText", RK_reasoningText) X("signature", RK_signature) \
  X("redactedContent", RK_redactedContent) X("stopReason", RK_stopReason) X("usage", RK_usage) X("inputTokens", RK_inputTokens) X("outputTokens", RK_outputTokens) \
  X("totalTokens", RK_totalTokens) X("cacheReadInputTokens", RK_cacheReadInputTokens) X("cacheWriteInputTokens", RK_cacheWriteInputTokens) X("serviceTier", RK_serviceTier) \
  X("type", RK_type) X("metrics", RK_metrics) X("latencyMs", RK_latencyMs) X("document", RK_document) X("image", RK_image) X("toolResult", RK_toolResult) X("cachePoint", RK_cachePoint) \
  X("id", RK_id) X("model", RK_model) X("stop_reason", RK_stop_reason) X("thinking", RK_thinking) X("data", RK_data) X("input_tokens", RK_input_tokens) X("output_tokens", RK_output_tokens) \
  X("cache_read_input_tokens", RK_cache_read_input_tokens) X("cache_creation_input_tokens", RK_cache_creation_input_tokens) X("stop_sequence", RK_stop_sequence) \
  X("error", RK_error) X("status", RK_status) X("details", RK_details) X("code", RK_code) X("request_id", RK_request_id)

// /v1/messages requests (P.schema & AIGW_SCHEMA_MESSAGES): the members of anthropic.MessagesRequest the restated subset knows
// (internal/apischema/anthropic/anthropic.go:26-140); every other key has id 0 and declines the body.  Values use AIGW_VALS.
enum MKid : uint8_t {
  MK_NONE = 0, MK_model, MK_max_tokens, MK_messages, MK_stream, MK_system, MK_temperature, MK_top_p, MK_top_k, MK_stop_sequences, MK_metadata,
  MK_tools, MK_tool_choice,   // top-level members only the full re-maps (OpenAI / Bedrock targets, plan_messages_full) take
  MK_user_id, MK_role, MK_content, MK_type, MK_text, MK_cache_control, MK_anthropic_version,
  MK_id, MK_name, MK_input, MK_tool_use_id, MK_is_error, MK_description, MK_input_schema, MK_properties, MK_required, MK_disable_parallel_tool_use, MK_COUNT
};
static_assert(MK_COUNT <= 64, "ids are 6 bits in the token word");
#define AIGW_MKEYS(X) \
  X("model", MK_model) X("max_tokens", MK_max_tokens) X("messages", MK_messages) X("stream", MK_stream) X("system", MK_system) X("temperature", MK_temperature) X("top_p", MK_top_p) \
  X("top_k", MK_top_k) X("stop_sequences", MK_stop_sequences) X("metadata", MK_metadata) X("user_id", MK_user_id) X("role", MK_role) X("content", MK_content) X("type", MK_type) \
  X("text", MK_text) X("cache_control", MK_cache_control) X("anthropic_version", MK_anthropic_version) X("tools", MK_tools) X("tool_choice", MK_tool_choice) X("id", MK_id) \
  X("name", MK_name) X("input", MK_input) X("tool_use_id", MK_tool_use_id) X("is_error", MK_is_error) X("description", MK_description) X("input_schema", MK_input_schema) \
  X("properties", MK_properties) X("required", MK_required) X("disable_parallel_tool_use", MK_disable_parallel_tool_use)

static constexpr int kKeySlots = 128, kValSlots = 32, kMaxIdLen = 28, kIdWords = 7;
// slot = { seven little-endian words of the string zero-padded to 28 bytes, len | id << 8 }
struct IdSlot { uint32_t w[kIdWords]; uint32_t meta; };
struct alignas(16) IdTables { IdSlot key[kKeySlots]; IdSlot val[kValSlots]; };
__host__ __device__ constexpr uint32_t id_hash(const uint32_t* v, uint32_t n) {
  uint32_t h = v[0] * 0x9E3779B1u ^ v[1] * 0x85EBCA77u ^ v[2] * 0xC2B2AE3Du ^ v[3] * 0x27D4EB2Fu ^ v[4] * 0x165667B1u ^ v[5] * 0x2545F491u ^ v[6] * 0x7FEB352Du;
  h ^= h >> 15; h += n * 0x9E3779B1u; h ^= h >> 13;
  return h;
}
constexpr void id_insert(IdSlot* tab, int slots, const char* lit, int idv) {
  uint32_t v[kIdWords] = {0, 0, 0, 0, 0, 0, 0};
  int n = 0; while (lit[n]) { v[n >> 2] |= (uint32_t)(uint8_t)lit[n] << ((n & 3) * 8); n++; }
  int sl = id_hash(v, (uint32_t)n) & (slots - 1);
  while (tab[sl].meta) sl = (sl + 1) & (slots - 1);
  for (int k = 0; k < kIdWords; k++) tab[sl].w[k] = v[k];
  tab[sl].meta = (uint32_t)n | ((uint32_t)idv << 8);
}
constexpr IdTables make_id_tables() {
  IdTables t{};
#define X(lit, idv) id_insert(t.key, kKeySlots, lit, idv);
  AIGW_KEYS(X)
#undef X
#define X(lit, idv) id_insert(t.val, kValSlots, lit, idv);
  AIGW_VALS(X)
#undef X
  return t;
}
// the device lookup probes at most 6 slots: every inserted string must sit within 6 of its home slot
constexpr int id_max_probe(const IdSlot* tab, int slots) {
  int worst = 0;
  for (int sl = 0; sl < slots; sl++) {
    if (!tab[sl].meta) continue;
    const int home = (int)(id_hash(tab[sl].w, tab[sl].meta & 0xffu) & (uint32_t)(slots - 1));
    const int dist = (sl - home + slots) & (slots - 1);
    if (dist > worst) worst = dist;
  }
  return worst + 1;
}
static_assert(id_max_probe(make_id_tables().key, kKeySlots) <= 6 && id_max_probe(make_id_tables().val, kValSlots) <= 6, "id hash table needs more than 6 probes");
static __device__ __constant__ IdTables c_ids = make_id_tables();
constexpr IdTables make_resp_id_tables() {
  IdTables t{};
#define X(lit, idv) id_insert(t.key, kKeySlots, lit, idv);
  AIGW_RKEYS(X)
#undef X
  return t;
}
static_assert(id_max_probe(make_resp_id_tables().key, kKeySlots) <= 6, "response id hash table needs more than 6 probes");
static __device__ __constant__ IdTables c_ids_resp = make_resp_id_tables();
constexpr IdTables make_msg_id_tables() {
  IdTables t{};
#define X(lit, idv) id_insert(t.key, kKeySlots, lit, idv);
  AIGW_MKEYS(X)
#undef X
#define X(lit, idv) id_insert(t.val, kValSlots, lit, idv);
  AIGW_MVALS(X)
#undef X
  return t;
}
static_assert(id_max_probe(make_msg_id_tables().key, kKeySlots) <= 6 && id_max_probe(make_msg_id_tables().val, kValSlots) <= 6, "messages id hash table needs more than 6 probes");
static __device__ __constant__ IdTables c_ids_msg = make_msg_id_tables();

// id of a short string (1 ≤ n ≤ kMaxIdLen) held in shared memory, against the key or the value table (also in shared
// memory).  Straight-line code: seven aligned word loads, funnel shifts, length mask, multiplicative hash, ≤ 4 probes.
__device__ __forceinline__ uint32_t lookup_id(const IdTables* T, const uint8_t* p, uint32_t n, bool key) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  const uint32_t sh = (a & 3u) * 8u;
  const uint32_t* wp = (const uint32_t*)(p - (a & 3u));
  uint32_t x[kIdWords + 1];
#pragma unroll
  for (int k = 0; k < kIdWords + 1; k++) x[k] = wp[k];
  uint32_t v[kIdWords];
#pragma unroll
  for (int k = 0; k < kIdWords; k++) {
    const uint32_t rem = n > 4u * k ? n - 4u * k : 0u;
    const uint32_t m = rem >= 4u ? 0xffffffffu : ((1u << (8u * rem)) - 1u);
    v[k] = __funnelshift_r(x[k], x[k + 1], sh) & m;
  }
  const uint32_t h = id_hash(v, n);
  const IdSlot* tab = key ? T->key : T->val;
  const uint32_t mask = key ? (kKeySlots - 1) : (kValSlots - 1);
  uint32_t sl = h & mask;
#pragma unroll 1
  for (int probe = 0; probe < 6; probe++) {
    const IdSlot e = tab[sl];
    if (e.meta == 0) return 0;
    if ((e.meta & 0xffu) == n && e.w[0] == v[0] && e.w[1] == v[1] && e.w[2] == v[2] && e.w[3] == v[3] && e.w[4] == v[4] && e.w[5] == v[5] && e.w[6] == v[6]) return e.meta >> 8;
    sl = (sl + 1) & mask;
  }
  return 0;
}


__device__ __forceinline__ int hex_val(uint32_t c) { if (c - '0' < 10u) return (int)(c - '0'); c |= 0x20u; if (c - 'a' < 6u) return (int)(c - 'a') + 10; return -1; }

// id of a string that contains escapes: the lookup runs on the DECODED bytes (a key spelled "mod\u0065l" is the model member for
// the reference's decoder).  Decoded strings longer than kMaxIdLen, malformed escapes and escapes that decode to non-ASCII
// (no table entry has any) give 0.
static __device__ uint32_t lookup_id_escaped(const IdTables* T, const uint8_t* p, uint32_t n, bool key) {
  uint32_t v[kIdWords];
#pragma unroll
  for (int k = 0; k < kIdWords; k++) v[k] = 0;
  uint32_t m = 0;
  for (uint32_t i = 0; i < n; i++) {
    uint32_t c = p[i];
    if (c == '\\') {
      if (++i >= n) return 0;
      const uint32_t e = p[i];
      if (e == 'n') c = '\n'; else if (e == 't') c = '\t'; else if (e == 'r') c = '\r'; else if (e == 'b') c = 8; else if (e == 'f') c = 12; else if (e == '"' || e == '\\' || e == '/') c = e;
      else if (e == 'u') { if (i + 4 >= n) return 0; int h = 0; for (int k = 1; k <= 4; k++) { const int x = hex_val(p[i + k]); if (x < 0) return 0; h = h * 16 + x; } if (h >= 0x80) return 0; c = (uint32_t)h; i += 4; }
      else return 0;
    }
    if (m >= (uint32_t)kMaxIdLen) return 0;
    v[m >> 2] |= c << ((m & 3u) * 8u);
    m++;
  }
  if (m == 0) return 0;
  const uint32_t h = id_hash(v, m);
  const IdSlot* tab = key ? T->key : T->val;
  const uint32_t mask = key ? (kKeySlots - 1) : (kValSlots - 1);
  uint32_t sl = h & mask;
  for (int probe = 0; probe < 6; probe++) {
    const IdSlot e = tab[sl];
    if (e.meta == 0) return 0;
    bool same = (e.meta & 0xffu) == m;
    for (int k = 0; k < kIdWords; k++) same = same && e.w[k] == v[k];
    if (same) return e.meta >> 8;
    sl = (sl + 1) & mask;
  }
  return 0;
}

// ------------------------------------------------------------------ workspace shared by the three stages
struct PlanOut { uint32_t nops, olen, path_len, model_off; uint16_t model_len; uint8_t flags, reason; };  // 20 bytes
static constexpr int kBins = 1024;
static constexpr int kWorkHdr = 16 + 2 * kBins * 4;   // [index counter][emit counter][walk counter][pad][bins][cursor]: zeroed by one memset per sub-batch

// per-document slot sizes of a size class (runtime copy of Cls<MAXD>, so that the walk kernel is compiled once)
struct WorkLayout { uint32_t kTok, kOps, kScr; };
template <int MAXD>
__host__ __device__ constexpr WorkLayout layout_of() { return WorkLayout{(uint32_t)Cls<MAXD>::kTok, (uint32_t)Cls<MAXD>::kOps, (uint32_t)Cls<MAXD>::kScr}; }
__host__ __device__ constexpr size_t work_per_doc(const WorkLayout& l) { return (size_t)l.kTok * 6 + (size_t)(l.kOps + kSysCap) * 4 + l.kScr + 32; }

struct WorkPtrs { unsigned int* c_index; unsigned int* c_emit; unsigned int* c_walk; uint32_t* tw; uint16_t* jmp; uint32_t* ops; uint8_t* scr; uint32_t* ntok; PlanOut* plan; uint32_t* perm; uint32_t* bins; uint32_t* cursor; };

__host__ __device__ inline WorkPtrs carve(uint8_t* base, size_t ndocs, const WorkLayout& l) {
  WorkPtrs w; uint8_t* p = base;
  w.c_index = (unsigned int*)p; w.c_emit = (unsigned int*)(p + 4); w.c_walk = (unsigned int*)(p + 8); p += 16;
  w.bins = (uint32_t*)p; p += kBins * 4;
  w.cursor = (uint32_t*)p; p += kBins * 4;
  w.tw = (uint32_t*)p; p += (size_t)l.kTok * 4 * ndocs;
  w.ops = (uint32_t*)p; p += (size_t)(l.kOps + kSysCap) * 4 * ndocs;
  w.ntok = (uint32_t*)p; p += 4 * ndocs;
  w.perm = (uint32_t*)p; p += 4 * ndocs;
  w.plan = (PlanOut*)p; p += 20 * ndocs;
  w.jmp = (uint16_t*)p; p += (size_t)l.kTok * 2 * ndocs;
  w.scr = p;
  return w;
}

// K2 (chat_walk.cu): validate + schema walk, one thread per document of the sub-batch
cudaError_t launch_chat_walk(const ChatParams& P, uint32_t doc0, uint32_t ndocs, uint8_t* work, const WorkLayout& layout, cudaStream_t st);

}  // namespace aigw
