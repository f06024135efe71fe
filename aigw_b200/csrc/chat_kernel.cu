// Index (K1), sort (Ks) and emit (K3) stages of the chat translate pass + the launcher.  See chat_kernel.cuh for the design;
// the schema walk (K2) is in chat_walk.cu.  sm_100a only.
//
//   * tokens carry their byte (tty) and a precomputed key / value id (tkid) that 32 lanes compute in
//     parallel, so the schema walk compares one byte instead of strings;
//   * request bodies are staged into shared memory by 1-D bulk asynchronous copies (bulk.cuh);
//   * the output record is assembled as 16-byte chunks (one chunk per lane, funnel-shifted unaligned
//     reads from shared memory) and stored straight to the arena — no shared-memory image of the output.
#include "chat_internal.cuh"

#include <mutex>

#include "bulk.cuh"
#include "chat_stage.cuh"

namespace aigw {


// ------------------------------------------------------------------ the kernels
// Launch sequence per sub-batch of documents, intermediates in a reusable global workspace:
//   K1 index   (warp per document)    stage 1+2+2.5 → token words, token count, histogram of token counts
//   Ks sort    (tiny)                 counting sort of the documents by token count → permutation
//   K2 walk    (thread per document)  stage 3+4 → jump table, copy ops, scratch, plan header
//   K3 emit    (warp per document)    stage 5 → output record + result
// K2 is where SIMT pays: 32 bodies with the same token count (≈ the same shape) share every instruction fetch.
// Sub-batches run one after the other on the caller's stream, each in the whole workspace.
// ---- K1: structural index, one warp per document
template <int MAXD, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) chat_index_kernel(const __grid_constant__ ChatParams P, uint32_t doc0, uint32_t ndocs, uint8_t* work) {
  using C = Cls<MAXD>;
  extern __shared__ __align__(128) uint8_t smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // CTA-shared tables: key/value id hash tables
  IdTables* s_ids = (IdTables*)smem;
  uint64_t* s_bar = (uint64_t*)(smem + sizeof(IdTables));
  {
    const uint32_t* src = (const uint32_t*)((P.schema & AIGW_SCHEMA_MESSAGES) ? &c_ids_msg : (P.schema & 48) == AIGW_SCHEMA_RESP_AWS_BEDROCK ? &c_ids_resp : &c_ids);
    for (uint32_t i = threadIdx.x; i < sizeof(IdTables) / 4; i += blockDim.x) ((uint32_t*)s_ids)[i] = src[i];
  }
  if (threadIdx.x == 0) { for (int w = 0; w < WARPS; w++) mbar_init(&s_bar[w], 1); mbar_fence_init(); }
  __syncthreads();
  constexpr int kHdr = (int)((sizeof(IdTables) + 8 * WARPS + 15) & ~(size_t)15);
  constexpr int kNcBytes = ((MAXD / 1024 + 1) * 4 + 15) & ~15;   // one word per round: lanes (32-byte blocks) that hold a valid escape the encoder rewrites
  constexpr int kWarpBytes = C::kIn + C::kTok * 6 + kNcBytes;
  uint8_t* wb = smem + kHdr + (size_t)warp * kWarpBytes;
  uint8_t* s_in = wb;
  uint32_t* s_tw = (uint32_t*)(wb + C::kIn);
  uint16_t* s_bs = (uint16_t*)(s_tw + C::kTok);   // running backslash count in front of each token; later overlaid by the lookup list
  uint32_t* s_nc = (uint32_t*)(wb + C::kIn + C::kTok * 6);
  uint64_t* bar = &s_bar[warp];
  const WorkPtrs wp = carve(work, ndocs, layout_of<MAXD>());
  uint32_t phase = 0;

  // work fetch, one document ahead: the atomic and the location loads of document k+1 complete under the scan of document k
  uint32_t li = 0;
  if (lane == 0) li = atomicAdd(wp.c_index, 1u);
  li = __shfl_sync(FULL, li, 0);
  uint32_t doc = 0, len = 0; const uint8_t* g = nullptr;
  if (li < ndocs) { doc = P.doc_map ? P.doc_map[doc0 + li] : doc0 + li; len = P.lens[doc]; g = P.bodies + P.offsets[doc]; }
  while (li < ndocs) {
    uint32_t li_next = 0;
    if (lane == 0) li_next = atomicAdd(wp.c_index, 1u);
    li_next = __shfl_sync(FULL, li_next, 0);
    uint32_t ndoc = 0, nlen = 0; const uint8_t* ng = nullptr;
    if (li_next < ndocs) { ndoc = P.doc_map ? P.doc_map[doc0 + li_next] : doc0 + li_next; nlen = P.lens[ndoc]; ng = P.bodies + P.offsets[ndoc]; }
#define AIGW_NEXT_DOC() do { li = li_next; doc = ndoc; len = nlen; g = ng; } while (0)
    if (len > (uint32_t)MAXD || len == 0) {
      if (lane == 0) { wp.ntok[li] = 0x80000000u | (len ? AIGW_R_TOO_LARGE : AIGW_R_E400_SYNTAX); atomicAdd(&wp.bins[0], 1u); }
      AIGW_NEXT_DOC();
      continue;
    }
    // ---- stage 1: one bulk asynchronous copy stages the body (no load / store issue slots)
    // (a caller that broke the 16-byte alignment contract gets an ordinary cooperative copy instead of a fault)
    if ((reinterpret_cast<uintptr_t>(g) & 15u) == 0) {
      if (lane == 0) { const uint32_t nbytes = (len + 15u) & ~15u; mbar_expect_tx(bar, nbytes); bulk_g2s(s_in, g, nbytes, bar); }
      mbar_wait(bar, phase); phase ^= 1u;
    } else {
      for (uint32_t i = lane; i < len; i += 32) s_in[i] = g[i];
      __syncwarp();
    }
    // the next document starts its way from DRAM to L2 now (its location was loaded before this one's copy was issued)
    if (lane == 0 && nlen && nlen <= (uint32_t)MAXD && (reinterpret_cast<uintptr_t>(ng) & 15u) == 0) bulk_prefetch_l2(ng, (nlen + 15u) & ~15u);
    // ---- stages 2 + 2.5: structural index (chat_stage.cuh)
    const uint32_t ntw = index_doc<MAXD>(s_in, len, lane, s_tw, s_bs, s_nc, s_ids);
    if (ntw & 0x80000000u) { if (lane == 0) { wp.ntok[li] = ntw; atomicAdd(&wp.bins[0], 1u); } AIGW_NEXT_DOC(); continue; }
    const uint32_t ntok = ntw & 0x3fffffffu;
    // ---- write the token words out, coalesced; histogram of token counts for the shape sort
    {
      uint32_t* gt = wp.tw + (size_t)li * C::kTok;
      for (uint32_t i = lane; i < ntok; i += 32) gt[i] = s_tw[i];
      if (lane == 0) { wp.ntok[li] = ntw; atomicAdd(&wp.bins[bin_of(ntok)], 1u); }
    }
    __syncwarp();
    AIGW_NEXT_DOC();
  }
#undef AIGW_NEXT_DOC
}

// ---- Ks: counting sort by token count (documents with the same count almost always have the same shape).  Every block
// scans the (tiny) histogram itself; positions inside a bin come from a global cursor.
__global__ void __launch_bounds__(1024) chat_sort_kernel(const uint32_t* ntok, const uint32_t* bins, uint32_t* cursor, uint32_t* perm, uint32_t ndocs) {
  __shared__ uint32_t s[kBins];
  const int t = threadIdx.x;
  const uint32_t v = bins[t];
  s[t] = v;
  __syncthreads();
  for (int off = 1; off < kBins; off <<= 1) { const uint32_t x = t >= off ? s[t - off] : 0u; __syncthreads(); s[t] += x; __syncthreads(); }
  const uint32_t excl = s[t] - v;
  __syncthreads();
  s[t] = excl;
  __syncthreads();
  for (uint32_t li = blockIdx.x * blockDim.x + t; li < ndocs; li += gridDim.x * blockDim.x) {
    const uint32_t b = bin_of(ntok[li]);
    perm[s[b] + atomicAdd(&cursor[b], 1u)] = li;
  }
}

// ---- K3: emit, one warp per document.
// The body is staged by one bulk asynchronous copy while the warp loads the ops and scans their lengths.  Output is built
// as 16-byte chunks, one chunk per lane: the op a chunk starts in comes from a scatter (last op starting at or before each
// chunk) + running max scan instead of a search; chunks inside one op are a single funnel-shifted shared-memory read; the
// chunks that straddle op boundaries are collected and assembled afterwards with every lane busy.
template <int MAXD, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) chat_emit_kernel(const __grid_constant__ ChatParams P, uint32_t doc0, uint32_t ndocs, uint8_t* work) {
  using C = Cls<MAXD>;
  using E = EmitSmem<MAXD>;
  extern __shared__ __align__(128) uint8_t smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* s_lits = smem;
  uint64_t* s_bar = (uint64_t*)(smem + sizeof(c_lits.bytes));
  for (uint32_t i = threadIdx.x; i < sizeof(c_lits.bytes) / 4; i += blockDim.x) ((uint32_t*)s_lits)[i] = ((const uint32_t*)c_lits.bytes)[i];
  if (threadIdx.x == 0) { for (int w = 0; w < WARPS; w++) mbar_init(&s_bar[w], 1); mbar_fence_init(); }
  __syncthreads();
  constexpr int kHdr = (int)((sizeof(c_lits.bytes) + 8 * WARPS + 15) & ~(size_t)15);
  uint8_t* wb = smem + kHdr + (size_t)warp * E::kWarpBytes;
  uint8_t* s_in = wb;
  uint32_t* s_pre = (uint32_t*)(wb + C::kIn);
  uint32_t* s_ops = s_pre + C::kOps + 4;
  uint8_t* s_scr = (uint8_t*)(s_ops + C::kOps);
  uint16_t* s_first = (uint16_t*)(s_scr + E::kScrB);
  uint32_t* s_bl = (uint32_t*)(s_first + kEmitTile);
  uint64_t* bar = &s_bar[warp];
  const WorkPtrs wp = carve(work, ndocs, layout_of<MAXD>());
  uint32_t phase = 0;

  // work fetch, one document ahead: plan header, location and the first 32 ops of document k+1 are loaded under the emit of
  // document k (each of these loads used to stall the warp for a DRAM round trip at the top of the loop)
  struct Meta { uint32_t doc, len; const uint8_t* g; PlanOut po; uint32_t op0; };
  auto load_meta = [&](uint32_t l) {
    Meta m;
    m.doc = P.doc_map ? P.doc_map[doc0 + l] : doc0 + l;
    m.len = P.lens[m.doc]; m.g = P.bodies + P.offsets[m.doc];
    m.po = wp.plan[l];
    m.op0 = (wp.ops + (size_t)l * (C::kOps + kSysCap))[lane];
    return m;
  };
  uint32_t li = 0;
  if (lane == 0) li = atomicAdd(wp.c_emit, 1u);
  li = __shfl_sync(FULL, li, 0);
  Meta cur{};
  if (li < ndocs) cur = load_meta(li);
  while (li < ndocs) {
    uint32_t li_next = 0;
    if (lane == 0) li_next = atomicAdd(wp.c_emit, 1u);
    li_next = __shfl_sync(FULL, li_next, 0);
    Meta nxt{};
    if (li_next < ndocs) nxt = load_meta(li_next);
    const uint32_t doc = cur.doc, len = cur.len;
    const PlanOut po = cur.po;
    const uint32_t op_first = cur.op0;
    const uint8_t* g = cur.g;
    aigw_doc_result res = blank_result(len);
    if (po.reason) {
      res.reason = po.reason;
      res.status = po.reason >= 48 ? AIGW_INTERNAL : po.reason >= 40 ? AIGW_INVALID_422 : po.reason >= 32 ? AIGW_MALFORMED_400 : AIGW_DECLINED;
      if (lane == 0) P.results[doc] = res;
      li = li_next; cur = nxt;
      continue;
    }
    const uint32_t nops = po.nops, olen = po.olen;
    const bool bulk = (reinterpret_cast<uintptr_t>(g) & 15u) == 0;
    if (bulk) { if (lane == 0) { const uint32_t nbytes = (len + 15u) & ~15u; mbar_expect_tx(bar, nbytes); bulk_g2s(s_in, g, nbytes, bar); } }
    else for (uint32_t i = lane; i < len; i += 32) s_in[i] = g[i];
    // while the body is in flight: ops (+ exclusive prefix of their lengths) and the scratch bytes they reference
    const uint32_t scr_hi = emit_prefix<MAXD>(wp.ops + (size_t)li * (C::kOps + kSysCap), op_first, nops, olen, s_ops, s_pre, lane);
    { const uint8_t* gs = wp.scr + (size_t)li * C::kScr; for (uint32_t i = lane; i < ((scr_hi + 3u) >> 2); i += 32) ((uint32_t*)s_scr)[i] = ((const uint32_t*)gs)[i]; }
    const uint32_t rec = (olen + 15u) & ~15u;
    const uint32_t nchunks = rec >> 4;
    unsigned long long obase = 0;
    if (lane == 0) obase = atomicAdd(P.out_used, (unsigned long long)rec);
    obase = __shfl_sync(FULL, obase, 0);
    __syncwarp();
    if (bulk) { mbar_wait(bar, phase); phase ^= 1u; }
    if (obase + rec > P.out_capacity || nchunks > 0xffffu) {
      res.reason = nchunks > 0xffffu ? AIGW_R_OUT_SPACE : AIGW_R_ARENA_FULL;
      if (lane == 0) P.results[doc] = res;
      __syncwarp();
      li = li_next; cur = nxt;
      continue;
    }
    if (lane == 0 && li_next < ndocs && !nxt.po.reason && (reinterpret_cast<uintptr_t>(nxt.g) & 15u) == 0) bulk_prefetch_l2(nxt.g, (nxt.len + 15u) & ~15u);
    uint4* o4 = (uint4*)(P.out + obase);
    emit_doc<MAXD>(s_in, s_lits, s_scr, s_pre, s_ops, s_first, s_bl, nops, nchunks, o4, lane);
    if (lane == 0) {
      res.out_off = obase + P.out_bias; res.body_len = olen - po.path_len; res.path_len = (uint16_t)po.path_len; res.status = AIGW_OK; res.reason = 0;
      res.model_off = po.model_off; res.model_len = po.model_len; res.body_kind = (po.flags & 0x80u) ? AIGW_BODY_UNCHANGED : AIGW_BODY_BYTES; res.flags = po.flags & 0x7fu;
      P.results[doc] = res;
    }
    __syncwarp();
    li = li_next; cur = nxt;
  }
}

// ------------------------------------------------------------------ host-side launcher
template <int MAXD>
size_t work_bytes_cls(size_t ndocs) { return work_per_doc(layout_of<MAXD>()) * ndocs + kWorkHdr + 256; }

struct ClsConfig { bool ready = false; int bps1 = 1, bps3 = 1; };

// the most documents one sub-batch takes (fewer when the workspace cannot hold that many)
static constexpr size_t kSubBatchDocs = 262144;

template <int MAXD, int WARPS>
static cudaError_t launch_cls(const ChatParams& P, uint32_t first, int device, int sm_count, cudaStream_t st, uint8_t* work, size_t work_cap, cudaEvent_t* ev, int ev_cap,
                              int* launches) {
  using C = Cls<MAXD>;
  constexpr size_t hdr1 = (sizeof(IdTables) + 8 * WARPS + 15) & ~(size_t)15, hdr3 = (sizeof(LitTable::bytes) + 8 * WARPS + 15) & ~(size_t)15;
  const size_t smem1 = hdr1 + (size_t)(C::kIn + C::kTok * 6 + (((MAXD / 1024 + 1) * 4 + 15) & ~15)) * WARPS;
  const size_t smem3 = hdr3 + (size_t)EmitSmem<MAXD>::kWarpBytes * WARPS;
  static ClsConfig cfgs[kMaxDevices];
  static std::mutex mu;
  if (device < 0 || device >= kMaxDevices) return cudaErrorInvalidDevice;
  ClsConfig& cc = cfgs[device];
  {
    std::lock_guard<std::mutex> lk(mu);
    if (!cc.ready) {
      cudaError_t e = cudaFuncSetAttribute(chat_index_kernel<MAXD, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1);
      if (e != cudaSuccess) return e;
      e = cudaFuncSetAttribute(chat_emit_kernel<MAXD, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3);
      if (e != cudaSuccess) return e;
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cc.bps1, chat_index_kernel<MAXD, WARPS>, WARPS * 32, smem1);
      if (e != cudaSuccess) return e;
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cc.bps3, chat_emit_kernel<MAXD, WARPS>, WARPS * 32, smem3);
      if (e != cudaSuccess) return e;
      if (cc.bps1 < 1) cc.bps1 = 1;
      if (cc.bps3 < 1) cc.bps3 = 1;
      cc.ready = true;
    }
  }
  size_t sub = ((work_cap & ~(size_t)255) - kWorkHdr - 256) / work_per_doc(layout_of<MAXD>());
  if (sub > kSubBatchDocs) sub = kSubBatchDocs;
  if (sub == 0) return cudaErrorMemoryAllocation;
  cudaError_t e;
  int nl = 0, sb = 0;
  for (uint32_t rel = 0; rel < P.n; rel += (uint32_t)sub, sb++) {
    const uint32_t doc0 = first + rel;
    const uint32_t nd = (uint32_t)(P.n - rel < sub ? P.n - rel : sub);
    const WorkPtrs wp = carve(work, nd, layout_of<MAXD>());
    if ((e = cudaMemsetAsync(work, 0, kWorkHdr, st)) != cudaSuccess) return e;
    long long want = ((long long)nd + WARPS - 1) / WARPS;
    long long g1 = (long long)sm_count * cc.bps1; if (want < g1) g1 = want;
    long long g3 = (long long)sm_count * cc.bps3; if (want < g3) g3 = want;
    const bool timed = ev && 4 * sb + 3 < ev_cap;
    if (timed) cudaEventRecord(ev[4 * sb + 0], st);
    chat_index_kernel<MAXD, WARPS><<<(unsigned)g1, WARPS * 32, smem1, st>>>(P, doc0, nd, work);
    if (timed) cudaEventRecord(ev[4 * sb + 1], st);
    { const unsigned gs = (nd + 8191) / 8192; chat_sort_kernel<<<gs < 32 ? gs : 32, kBins, 0, st>>>(wp.ntok, wp.bins, wp.cursor, wp.perm, nd); }
    if ((e = launch_chat_walk(P, doc0, nd, work, layout_of<MAXD>(), st)) != cudaSuccess) return e;
    if (timed) cudaEventRecord(ev[4 * sb + 2], st);
    chat_emit_kernel<MAXD, WARPS><<<(unsigned)g3, WARPS * 32, smem3, st>>>(P, doc0, nd, work);
    if (timed) cudaEventRecord(ev[4 * sb + 3], st);
    nl += 4;
  }
  if (launches) *launches = nl;
  return cudaGetLastError();
}

size_t chat_work_bytes(uint32_t max_len, size_t ndocs) {
  if (max_len <= 2048) return work_bytes_cls<2048>(ndocs);
  if (max_len <= 5120) return work_bytes_cls<5120>(ndocs);
  if (max_len <= 9216) return work_bytes_cls<9216>(ndocs);
  if (max_len <= 17408) return work_bytes_cls<17408>(ndocs);
  if (max_len <= 33792) return work_bytes_cls<33792>(ndocs);
  return work_bytes_cls<65536>(ndocs);
}
// workspace that lets a call of n documents run in one sub-batch, or in sub-batches of the largest size
size_t chat_work_bytes_for(uint32_t max_len, size_t n) { return chat_work_bytes(max_len, n < kSubBatchDocs ? n : kSubBatchDocs) + 512; }

cudaError_t launch_chat_translate_range(const ChatParams& P, uint32_t first, uint32_t count, uint32_t max_len, int device, int sm_count, cudaStream_t st, uint8_t* work, size_t work_cap,
                                        int* launches) {
  ChatParams Q = P; Q.n = count;
  return launch_chat_translate(Q, max_len, device, sm_count, st, work, work_cap, launches, nullptr, 0, first);
}

cudaError_t launch_chat_translate(const ChatParams& P, uint32_t max_len, int device, int sm_count, cudaStream_t st, uint8_t* work, size_t work_cap, int* launches,
                                  cudaEvent_t* ev, int ev_cap, uint32_t first) {
  if (max_len <= 2048) return launch_cls<2048, 4>(P, first, device, sm_count, st, work, work_cap, ev, ev_cap, launches);
  if (max_len <= 5120) return launch_cls<5120, 4>(P, first, device, sm_count, st, work, work_cap, ev, ev_cap, launches);
  if (max_len <= 9216) return launch_cls<9216, 2>(P, first, device, sm_count, st, work, work_cap, ev, ev_cap, launches);
  if (max_len <= 17408) return launch_cls<17408, 2>(P, first, device, sm_count, st, work, work_cap, ev, ev_cap, launches);
  if (max_len <= 33792) return launch_cls<33792, 1>(P, first, device, sm_count, st, work, work_cap, ev, ev_cap, launches);
  return launch_cls<65536, 1>(P, first, device, sm_count, st, work, work_cap, ev, ev_cap, launches);
}

}  // namespace aigw
