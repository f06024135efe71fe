// K2 launcher: picks the walk kernel of the schema's group (chat_walk_g*.cu, one translation unit per group).
#include "chat_internal.cuh"

namespace aigw {

#define AIGW_WALK_DECL(g) cudaError_t launch_chat_walk_g##g(const ChatParams&, uint32_t, uint32_t, uint8_t*, const WorkLayout&, cudaStream_t, int);
AIGW_WALK_DECL(0) AIGW_WALK_DECL(1) AIGW_WALK_DECL(2) AIGW_WALK_DECL(3) AIGW_WALK_DECL(4) AIGW_WALK_DECL(5) AIGW_WALK_DECL(6) AIGW_WALK_DECL(7) AIGW_WALK_DECL(8) AIGW_WALK_DECL(9)
#undef AIGW_WALK_DECL
#define AIGW_SMALL_DECL(g) cudaError_t launch_chat_small_g##g(const ChatParams&, uint32_t, uint32_t, const uint64_t*, cudaStream_t);
AIGW_SMALL_DECL(0) AIGW_SMALL_DECL(1) AIGW_SMALL_DECL(2) AIGW_SMALL_DECL(3) AIGW_SMALL_DECL(4) AIGW_SMALL_DECL(5) AIGW_SMALL_DECL(6) AIGW_SMALL_DECL(7) AIGW_SMALL_DECL(8) AIGW_SMALL_DECL(9)
#undef AIGW_SMALL_DECL

cudaError_t launch_chat_walk(const ChatParams& P, uint32_t doc0, uint32_t ndocs, uint8_t* work, const WorkLayout& layout, cudaStream_t st) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  { static int sm_cache[kMaxDevices] = {0}; if (dev >= 0 && dev < kMaxDevices) { if (!sm_cache[dev]) cudaDeviceGetAttribute(&sm_cache[dev], cudaDevAttrMultiProcessorCount, dev); sms = sm_cache[dev] ? sm_cache[dev] : 148; } }
  sms *= AIGW_WALK_BLOCKS;
  const uint32_t s = P.schema;
  if (s & (uint32_t)AIGW_SCHEMA_MESSAGES)   // the full re-maps (OpenAI / Bedrock targets) have their own kernel
    return ((s & 15u) == (uint32_t)AIGW_SCHEMA_OPENAI || (s & 15u) == (uint32_t)AIGW_SCHEMA_AWS_BEDROCK) ? launch_chat_walk_g9(P, doc0, ndocs, work, layout, st, sms) : launch_chat_walk_g7(P, doc0, ndocs, work, layout, st, sms);
  if ((s & 56u) == (uint32_t)AIGW_SCHEMA_RESP_ERROR) return launch_chat_walk_g8(P, doc0, ndocs, work, layout, st, sms);
  if ((s & 48u) == (uint32_t)AIGW_SCHEMA_RESP_AWS_BEDROCK)
    return ((s & 15u) == (uint32_t)AIGW_SCHEMA_GCP_ANTHROPIC || (s & 15u) == (uint32_t)AIGW_SCHEMA_ANTHROPIC) ? launch_chat_walk_g5(P, doc0, ndocs, work, layout, st, sms) : launch_chat_walk_g4(P, doc0, ndocs, work, layout, st, sms);
  if (s & (uint32_t)AIGW_SCHEMA_EMBEDDINGS) return launch_chat_walk_g6(P, doc0, ndocs, work, layout, st, sms);
  switch (s) {
    case AIGW_SCHEMA_AWS_BEDROCK: return launch_chat_walk_g0(P, doc0, ndocs, work, layout, st, sms);
    case AIGW_SCHEMA_GCP_ANTHROPIC: case AIGW_SCHEMA_AWS_ANTHROPIC: return launch_chat_walk_g2(P, doc0, ndocs, work, layout, st, sms);
    case AIGW_SCHEMA_GCP_VERTEX: return launch_chat_walk_g3(P, doc0, ndocs, work, layout, st, sms);
    default: return launch_chat_walk_g1(P, doc0, ndocs, work, layout, st, sms);   // OpenAI / Azure; a schema without a planner declines every document with AIGW_R_SCHEMA
  }
}

// fused small-batch kernel (one CTA per document, bodies of at most 5120 bytes): chat_walk_impl.cuh
cudaError_t launch_chat_small(const ChatParams& P, uint32_t doc0, uint32_t ndocs, const uint64_t* out_slot, cudaStream_t st) {
  const uint32_t s = P.schema;
  if (s & (uint32_t)AIGW_SCHEMA_MESSAGES)
    return ((s & 15u) == (uint32_t)AIGW_SCHEMA_OPENAI || (s & 15u) == (uint32_t)AIGW_SCHEMA_AWS_BEDROCK) ? launch_chat_small_g9(P, doc0, ndocs, out_slot, st) : launch_chat_small_g7(P, doc0, ndocs, out_slot, st);
  if ((s & 56u) == (uint32_t)AIGW_SCHEMA_RESP_ERROR) return launch_chat_small_g8(P, doc0, ndocs, out_slot, st);
  if ((s & 48u) == (uint32_t)AIGW_SCHEMA_RESP_AWS_BEDROCK)
    return ((s & 15u) == (uint32_t)AIGW_SCHEMA_GCP_ANTHROPIC || (s & 15u) == (uint32_t)AIGW_SCHEMA_ANTHROPIC) ? launch_chat_small_g5(P, doc0, ndocs, out_slot, st) : launch_chat_small_g4(P, doc0, ndocs, out_slot, st);
  if (s & (uint32_t)AIGW_SCHEMA_EMBEDDINGS) return launch_chat_small_g6(P, doc0, ndocs, out_slot, st);
  switch (s) {
    case AIGW_SCHEMA_AWS_BEDROCK: return launch_chat_small_g0(P, doc0, ndocs, out_slot, st);
    case AIGW_SCHEMA_GCP_ANTHROPIC: case AIGW_SCHEMA_AWS_ANTHROPIC: return launch_chat_small_g2(P, doc0, ndocs, out_slot, st);
    case AIGW_SCHEMA_GCP_VERTEX: return launch_chat_small_g3(P, doc0, ndocs, out_slot, st);
    default: return launch_chat_small_g1(P, doc0, ndocs, out_slot, st);
  }
}

}  // namespace aigw
