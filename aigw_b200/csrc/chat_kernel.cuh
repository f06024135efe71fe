// aigw_b200 — /v1/chat/completions parse + translate kernel for sm_100a.
//
// One warp per request body ("document"), persistent CTAs pulling documents from a global
// counter.  Per document:
//   stage 1  load      16-byte coalesced global loads → per-warp shared-memory copy of the body
//   stage 2  index     lane-local byte classification (32 B per lane per round), escape/quote
//                      carry resolution with ballots, in-string prefix-xor, structural token list
//   stage 3  validate  JSON grammar over the token list, bracket matching (jump table)
//   stage 4  plan      schema walk (OpenAI ChatCompletionRequest → target layout) producing a
//                      list of copy ops (input span | literal | scratch span)
//   stage 5  emit      warp-cooperative gather of the ops into a shared-memory image of the
//                      output record, bump-allocate space in the output arena, 16-byte stores
//
// Behavioural source of truth for stage 4: internal/translator/openai_awsbedrock.go:91-585 and
// internal/apischema/awsbedrock/awsbedrock.go:41-70,126-200,310-367,536-604 (field order, omit
// rules); internal/translator/openai_openai.go:55-84 and internal/endpointspec/endpointspec.go:107-123
// for the OpenAI passthrough edits.  Anything outside the fast path is DECLINED (the caller runs
// the stock path); the kernel never guesses.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/aigw_b200.h"

namespace aigw {

// ------------------------------------------------------------------ literal table
#define AIGW_LITERALS(X)                                                                       \
  X(L_LBRACE, "{")                                                                             \
  X(L_RBRACE, "}")                                                                             \
  X(L_LBRACK, "[")                                                                             \
  X(L_RBRACK, "]")                                                                             \
  X(L_COMMA, ",")                                                                              \
  X(L_COLON, ":")                                                                              \
  X(L_ZERO, "0")                                                                               \
  X(L_NULL, "null")                                                                            \
  X(L_TRUE, "true")                                                                            \
  X(L_EMPTY_STR, "\"\"")                                                                       \
  X(L_ADDL_EN_PRE, "\"additionalModelRequestFields\":{\"thinking\":{\"budget_tokens\":")       \
  X(L_ADDL_EN_POST, ",\"type\":\"enabled\"}},")                                                \
  X(L_ADDL_DIS, "\"additionalModelRequestFields\":{\"thinking\":{\"type\":\"disabled\"}},")    \
  X(L_INF_OPEN, "\"inferenceConfig\":{")                                                       \
  X(L_MAXTOK, "\"maxTokens\":")                                                                \
  X(L_STOPSEQ, "\"stopSequences\":[")                                                          \
  X(L_TEMP, "\"temperature\":")                                                                \
  X(L_TOPP, "\"topP\":")                                                                       \
  X(L_INF_CLOSE_MSGS, "},\"messages\":[")                                                      \
  X(L_MSG_TEXT_OPEN, "{\"content\":[{\"text\":")                                               \
  X(L_MSG_CONTENT_OPEN, "{\"content\":[")                                                      \
  X(L_TEXT_OPEN, "{\"text\":")                                                                 \
  X(L_USER_CLOSE1, "}],\"role\":\"user\"}")                                                    \
  X(L_ASST_CLOSE1, "}],\"role\":\"assistant\"}")                                               \
  X(L_USER_CLOSE, "],\"role\":\"user\"}")                                                      \
  X(L_ASST_CLOSE, "],\"role\":\"assistant\"}")                                                 \
  X(L_CACHEPOINT, "{\"cachePoint\":{\"type\":\"default\"}}")                                   \
  X(L_TOOLRESULT_OPEN, "{\"toolResult\":{\"content\":[")                                       \
  X(L_TOOLRESULT_MID, "],\"status\":null,\"toolUseId\":")                                      \
  X(L_TOOLRESULT_CLOSE, "}}")                                                                  \
  X(L_TOOLUSE_OPEN, "{\"toolUse\":{\"name\":")                                                 \
  X(L_TOOLUSE_INPUT, ",\"input\":")                                                            \
  X(L_TOOLUSE_ID, ",\"toolUseId\":")                                                           \
  X(L_REASON_OPEN, "{\"reasoningContent\":{\"reasoningText\":{\"text\":")                      \
  X(L_REASON_SIG, ",\"signature\":")                                                           \
  X(L_REASON_CLOSE, "}}}")                                                                     \
  X(L_SYSTEM_OPEN, ",\"system\":[")                                                            \
  X(L_SERVICE_TIER, ",\"serviceTier\":{\"type\":")                                             \
  X(L_TOOLCFG_OPEN, ",\"toolConfig\":{")                                                       \
  X(L_TOOLCHOICE_AUTO, "\"toolChoice\":{\"auto\":{}},")                                        \
  X(L_TOOLCHOICE_ANY, "\"toolChoice\":{\"any\":{}},")                                          \
  X(L_TOOLCHOICE_TOOL, "\"toolChoice\":{\"tool\":{\"name\":")                                  \
  X(L_TOOLCHOICE_TOOL_END, "}},")                                                              \
  X(L_TOOLS_OPEN, "\"tools\":[")                                                               \
  X(L_TOOLSPEC_OPEN, "{\"toolSpec\":{")                                                        \
  X(L_DESC, "\"description\":")                                                                \
  X(L_INPUTSCHEMA, "\"inputSchema\":{\"json\":")                                               \
  X(L_NAME, "},\"name\":")                                                                     \
  X(L_TOOL_CACHE, ",\"cachePoint\":{\"type\":\"default\"}")                                    \
  X(L_TOOLS_CLOSE, "]}")                                                                       \
  X(L_PATH_MODEL, "/model/")                                                                   \
  X(L_PATH_CONVERSE, "/converse")                                                              \
  X(L_PATH_STREAM, "-stream")                                                                  \
  X(L_STREAMOPT_APPEND, "\"stream_options\":{\"include_usage\":true}")                         \
  X(L_INCLUDE_USAGE_MEMBER, "\"include_usage\":true")                                          \
  X(L_INCLUDE_USAGE_OBJ, "{\"include_usage\":true}")                                           \
  X(L_MODEL_MEMBER, "\"model\":")                                                              \
  X(L_QUOTE, "\"")                                                                         \
  X(L_AZURE_PREFIX, "/openai/deployments/")                                                    \
  X(L_AZURE_SUFFIX, "/chat/completions?api-version=")                                         \
  X(L_AN_OPEN, "{\"max_tokens\":")                                                              \
  X(L_AN_MSGS, ",\"messages\":[")                                                               \
  X(L_AN_TEXT_CLOSE, ",\"type\":\"text\"}")                                                     \
  X(L_AN_TEXT_CACHE_CLOSE, ",\"cache_control\":{\"type\":\"ephemeral\"},\"type\":\"text\"}")      \
  X(L_AN_TOOLUSE_OPEN, "{\"id\":")                                                              \
  X(L_AN_NAME, ",\"name\":")                                                                    \
  X(L_AN_TOOLUSE_CLOSE, ",\"type\":\"tool_use\"}")                                              \
  X(L_AN_TR_OPEN, "{\"tool_use_id\":")                                                          \
  X(L_AN_TR_ERR_F, ",\"is_error\":false,\"content\":[")                                         \
  X(L_AN_TR_ERR_T, ",\"is_error\":true,\"content\":[")                                          \
  X(L_AN_TR_CLOSE, "],\"type\":\"tool_result\"}")                                               \
  X(L_AN_TOPP, ",\"top_p\":")                                                                  \
  X(L_AN_STOPSEQ, ",\"stop_sequences\":[")                                                     \
  X(L_AN_STREAM, ",\"stream\":true")                                                            \
  X(L_AN_VERSION, ",\"anthropic_version\":\"")                                                   \
  X(L_AN_END, "\"}")                                                                            \
  X(L_AN_GCP_PATH, "publishers/anthropic/models/")                                             \
  X(L_AN_RAWPREDICT, ":rawPredict")                                                            \
  X(L_AN_STREAMRAWPREDICT, ":streamRawPredict")                                                \
  X(L_AN_INVOKE, "/invoke")                                                                    \
  X(L_AN_INVOKE_STREAM, "/invoke-with-response-stream")                                        \
  X(L_AN_VER_GCP, "vertex-2023-10-16")                                                         \
  X(L_AN_VER_AWS, "bedrock-2023-05-31")                                                        \
  X(L_R_ID_OPEN, "\"id\":\"")                                                                   \
  X(L_R_QUOTE_COMMA, "\",")                                                                      \
  X(L_R_QUOTE, "\"")                                                                             \
  X(L_R_CHOICES, "\"choices\":[{\"finish_reason\":\"")                                           \
  X(L_R_MSG, "\",\"index\":0,\"message\":{")                                                     \
  X(L_R_CONTENT, "\"content\":")                                                                \
  X(L_R_ROLE, "\"role\":")                                                                      \
  X(L_R_TOOLCALLS, "\"tool_calls\":[")                                                          \
  X(L_R_TC_ID, "{\"id\":")                                                                      \
  X(L_R_TC_ARGS, ",\"function\":{\"arguments\":\"")                                              \
  X(L_R_TC_NAME, "\",\"name\":")                                                                 \
  X(L_R_TC_END, "},\"type\":\"function\"}")                                                     \
  X(L_R_REASON, "\"reasoning_content\":{\"reasoningContent\":{")                                \
  X(L_R_RTEXT, "\"reasoningText\":{\"text\":")                                                  \
  X(L_R_RSIG, ",\"signature\":")                                                                \
  X(L_R_RBRACE2, "}}")                                                                          \
  X(L_R_CREATED, "}}],\"created\":")                                                            \
  X(L_R_MODEL, ",\"model\":\"")                                                                  \
  X(L_R_TIER, ",\"service_tier\":")                                                             \
  X(L_R_OBJECT, ",\"object\":\"chat.completion\"")                                              \
  X(L_R_USAGE, ",\"usage\":{")                                                                  \
  X(L_R_PROMPT, "\"prompt_tokens\":")                                                           \
  X(L_R_COMPLETION, "\"completion_tokens\":")                                                   \
  X(L_R_TOTAL, "\"total_tokens\":")                                                             \
  X(L_R_PTD, "\"prompt_tokens_details\":{")                                                     \
  X(L_R_CACHED, "\"cached_tokens\":")                                                           \
  X(L_R_CC, "\"cache_creation_input_tokens\":")                                                 \
  X(L_R_FR_STOP, "stop")                                                                        \
  X(L_R_FR_LENGTH, "length")                                                                    \
  X(L_R_FR_FILTER, "content_filter")                                                            \
  X(L_R_FR_TOOLS, "tool_calls")                                                                \
  X(L_R_Q_ASSISTANT, "\"assistant\"")                                                          \
  X(L_R_Q_USER, "\"user\"")                                                                    \
  X(L_R_MODEL_KEY, ",\"model\":")                                                              \
  X(L_R_ID_KEY, "\"id\":")                                                                     \
  X(L_EM_OPEN, "{\"instances\":")                                                               \
  X(L_EM_CONTENT, "{\"content\":")                                                              \
  X(L_EM_TASK, ",\"task_type\":")                                                               \
  X(L_EM_TITLE, ",\"title\":")                                                                  \
  X(L_EM_PARAMS, ",\"parameters\":{")                                                           \
  X(L_EM_AUTOTRUNC, "\"auto_truncate\":true")                                                   \
  X(L_EM_DIMS, "\"outputDimensionality\":")                                                     \
  X(L_EM_END, "}}")                                                                             \
  X(L_EM_GOOGLE_PATH, "publishers/google/models/")                                              \
  X(L_EM_PREDICT, ":predict")                                                                   \
  X(L_EM_AZ_PATH1, "/openai/deployments/")                                                      \
  X(L_EM_AZ_PATH2, "/embeddings?api-version=")                                                 \
  X(L_EM_NEXT, "},{\"content\":")                                                               \
  X(L_GEM_GENERATE, ":generateContent")                                                        \
  X(L_GEM_STREAM, ":streamGenerateContent?alt=sse")                                            \
  X(L_GEM_CONTENTS, "{\"contents\":")                                                          \
  X(L_GEM_PARTS_OPEN, "{\"parts\":[")                                                          \
  X(L_GEM_MODEL_EMPTY, "{\"role\":\"model\"}")                                                 \
  X(L_GEM_MODEL_CLOSE, "],\"role\":\"model\"}")                                                \
  X(L_GEM_TOOLS, ",\"tools\":")                                                                \
  X(L_GEM_DECLS_OPEN, "[{\"functionDeclarations\":[")                                          \
  X(L_GEM_DECLS_CLOSE, "]}]")                                                                  \
  X(L_GEM_NAME, "\"name\":")                                                                   \
  X(L_GEM_PARAMS, "\"parameters\":")                                                           \
  X(L_GEM_PARAMS_JS, "\"parametersJsonSchema\":")                                              \
  X(L_GEM_GENCFG, ",\"generation_config\":{")                                                  \
  X(L_GEM_CANDIDATES, "\"candidateCount\":")                                                   \
  X(L_GEM_FREQ, "\"frequencyPenalty\":")                                                       \
  X(L_GEM_LOGPROBS, "\"logprobs\":")                                                           \
  X(L_GEM_MAXOUT, "\"maxOutputTokens\":")                                                      \
  X(L_GEM_PRES, "\"presencePenalty\":")                                                        \
  X(L_GEM_RESP_LOGPROBS, "\"responseLogprobs\":true")                                          \
  X(L_GEM_SEED, "\"seed\":")                                                                   \
  X(L_GEM_SYS_OPEN, ",\"system_instruction\":{\"parts\":[")                                    \
  X(L_GEM_SYS_CLOSE, "]}")                                                                     \
  X(L_EM_LAST, "}]")                                                                            \
  X(L_TITAN_OPEN, "{\"inputText\":")                                                          \
  X(L_TITAN_DIMS, ",\"dimensions\":")                                                         \
  X(L_MSG_PATH, "/v1/messages")                                                                \
  X(L_MSG_VERSION_MEMBER, "\"anthropic_version\":")                                            \
  X(L_ERR_OPEN, "{\"type\":\"error\",\"error\":{\"type\":")                                   \
  X(L_ERR_CODE, ",\"code\":\"")                                                               \
  X(L_ERR_MESSAGE, "\",\"message\":")                                                         \
  X(L_ERR_CLOSE_AFTER_CODE, "\"}}")                                                            \
  X(L_ERR_CLOSE, "}}")                                                                         \
  X(L_ERR_T_AWS, "\"AWSBedrockBackendError\"")                                                \
  X(L_ERR_T_GCP, "\"GCPBackendError\"")                                                       \
  X(L_ERR_T_VERTEX, "\"GCPVertexAIBackendError\"")                                            \
  X(L_MX_OPEN, "{\"messages\":")                                                               \
  X(L_MX_CONTENT_Q, "{\"content\":\"")                                                         \
  X(L_MX_SYS_CLOSE, "\",\"role\":\"system\"}")                                                 \
  X(L_MX_USER_CLOSE_Q, "\",\"role\":\"user\"}")                                                \
  X(L_MX_TOOL_MID, "\",\"role\":\"tool\",\"tool_call_id\":")                                  \
  X(L_MX_ASST_OPEN, "{\"role\":\"assistant\",\"content\":")                                   \
  X(L_MX_MAXCT, ",\"max_completion_tokens\":")                                                 \
  X(L_MX_TOPP, ",\"top_p\":")                                                                  \
  X(L_MX_TOOLS, ",\"tools\":[")                                                                \
  X(L_MX_TOOL_OPEN, "{\"type\":\"function\",\"function\":{\"name\":")                          \
  X(L_MX_SCHEMA_TYPE, "{\"type\":")                                                            \
  X(L_MX_PROPS, ",\"properties\":")                                                            \
  X(L_MX_REQUIRED, ",\"required\":[")                                                          \
  X(L_MX_TC_AUTO, ",\"tool_choice\":\"auto\"")                                                 \
  X(L_MX_TC_NONE, ",\"tool_choice\":\"none\"")                                                 \
  X(L_MX_TC_REQUIRED, ",\"tool_choice\":\"required\"")                                         \
  X(L_MX_TC_NAMED, ",\"tool_choice\":{\"type\":\"function\",\"function\":{\"name\":")         \
  X(L_MX_STOP, ",\"stop\":[")                                                                  \
  X(L_MX_TOPK, "\"additionalModelRequestFields\":{\"top_k\":")                                 \
  X(L_MX_TR_NULL, "{\"toolResult\":{\"content\":null")                                         \
  X(L_MX_TR_STATUS_ERR, ",\"status\":\"error\",\"toolUseId\":")                             \
  X(L_AM_HEAD, "\",\"type\":\"message\",\"role\":\"assistant\",\"content\":[")                 \
  X(L_AM_TEXT, "{\"type\":\"text\",\"text\":")                                                 \
  X(L_AM_TOOLUSE, "{\"type\":\"tool_use\",\"id\":")                                            \
  X(L_AM_THINKING, "{\"type\":\"thinking\",\"thinking\":")                                     \
  X(L_AM_STOP, ",\"stop_reason\":")                                                            \
  X(L_AM_END_TURN, "\"end_turn\"")                                                             \
  X(L_AM_CACHE_READ, ",\"cache_read_input_tokens\":")                                          \
  X(L_AM_INPUT, ",\"input_tokens\":")                                                          \
  X(L_AM_OUTPUT, ",\"output_tokens\":")

enum LitId : int {
#define X(name, text) name,
  AIGW_LITERALS(X)
#undef X
      L_COUNT
};

struct alignas(16) LitTable {
  uint16_t off[L_COUNT + 1];
  alignas(16) char bytes[3328];   // copied to shared memory with 32-bit loads
};
constexpr LitTable make_lit_table() {
  LitTable t{};
  int o = 0, k = 0;
#define X(name, text)                                   \
  t.off[k++] = (uint16_t)o;                             \
  for (int i = 0; text[i]; i++) t.bytes[o++] = text[i];
  AIGW_LITERALS(X)
#undef X
  t.off[k] = (uint16_t)o;
  return t;
}

// ------------------------------------------------------------------ kernel parameters
struct ChatParams {
  const uint8_t* bodies;
  const uint64_t* offsets;
  const uint32_t* lens;
  uint32_t n;
  uint8_t* out;
  uint64_t out_capacity;
  aigw_doc_result* results;
  unsigned long long* out_used;  // bump allocator
  unsigned int* next_doc;        // work counter
  uint64_t out_bias;             // added to every out_off (host pipeline: chunk base in the host arena)
  const uint32_t* doc_map;       // optional: unit i of the launch is document doc_map[first + i] (size-class bucketing)
  int schema;
  int cost_configured;
  int force_mutation;
  uint16_t override_len;  // model_name_override (≤ 128 bytes, in cfgbuf)
  uint16_t prefix_len;    // normalised OpenAI path "/…/chat/completions"
  uint16_t version_len;   // VersionedAPISchema.Version (Azure api-version)
  char api_version[64];
  char override_model[128];
  char openai_path[128];
  long long created;      // response schemas: ChatCompletionResponse.created
  uint16_t rid_len;       // response schemas: response id (x-amzn-requestid)
  char response_id[128];
};

// size classes: MAXD bytes of input per document.  Per-warp shared memory:
//   in[kIn] | tpos u16[kTok] | jmp u16[kTok] | tty u8[kTok] | tkid u8[kTok] | ops u32[kOps+kSys] | pre u32[kOps] | scr[kScr]
static constexpr int kSysCap = 192;   // system-message ops parked until the messages array is closed (a re-spelled escape run costs two ops)
template <int MAXD>
struct Cls {
  static constexpr int kIn = MAXD + 16;                  // multiple of 16; slack for unaligned word reads
  static constexpr int kTok = (MAXD / 8 < 512 ? 512 : (MAXD / 8 + 63) / 64 * 64); // ≈ one token per 8 input bytes, else the body is declined
  static constexpr int kOps = 160 + MAXD / 32;
  static constexpr int kScr = 256 + MAXD / 8;
  static constexpr int kWarpBytes = kIn + kTok * 6 + (kOps + kSysCap) * 4 + kOps * 4 + kScr;
};

// Workspace: chat_work_bytes(max_len, docs_per_sub_batch) bytes hold one sub-batch of intermediates; the launcher walks P.n
// documents in sub-batches of at most 256 Ki documents (4 launches each), one after the other on the caller's stream, each
// reusing the whole workspace.  chat_work_bytes_for(max_len, n) is the size that holds the largest sub-batch a call of n
// documents needs.  `stage_events` (profiling) receives four events per sub-batch at the stage boundaries (before index,
// after index, after sort + walk, after emit) for the first stage_event_cap / 4 sub-batches.
// Per-device kernel attributes are configured on first use of each (device, size class).
static constexpr int kMaxDevices = 16;
static constexpr uint32_t kSmallMaxLen = 5120;   // the fused small-batch kernel's size class
// fused index + walk + emit, one CTA per document; out_slot[i] .. out_slot[i+1] is document i's output slot in P.out; no workspace
cudaError_t launch_chat_small(const ChatParams& P, uint32_t doc0, uint32_t ndocs, const uint64_t* out_slot, cudaStream_t st);
size_t chat_work_bytes(uint32_t max_len, size_t ndocs);
size_t chat_work_bytes_for(uint32_t max_len, size_t n);
cudaError_t launch_chat_translate(const ChatParams& P, uint32_t max_len, int device, int sm_count, cudaStream_t st, uint8_t* work, size_t work_cap, int* launches,
                                  cudaEvent_t* stage_events, int stage_event_cap, uint32_t first = 0);
// documents [first, first+count): offsets / lens / results are indexed with the global document number
cudaError_t launch_chat_translate_range(const ChatParams& P, uint32_t first, uint32_t count, uint32_t max_len, int device, int sm_count, cudaStream_t st, uint8_t* work,
                                        size_t work_cap, int* launches);

}  // namespace aigw
