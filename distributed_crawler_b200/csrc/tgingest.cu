// tgingest.cu — host side of libtgingest: the C ABI of include/tgingest.h on top of the sm_100a
// kernels in kernels.cuh.  One context = one GPU.  Three staging slots, each with its own stream
// and worker thread, so H2D of one batch, kernels of another and D2H of a third overlap.
// There is no CPU fallback: without a CUDA device tgi_create fails with TGI_E_NODEVICE.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types only: the library itself is loaded with dlopen at tgi_comm_init

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "kernels.cuh"
#include "tg_page.cuh"
#include "yt_page.cuh"

using namespace tgi;

namespace {

constexpr size_t PAD = 64;  // zero bytes behind every device blob (kernels over-read <= 16 bytes)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }  // error paths of the one-shot entry points must not leak device memory
  cudaError_t ensure(size_t bytes) {
    bytes += PAD;
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    size_t want = bytes + bytes / 8;
    cudaError_t e = cudaMalloc(&p, want);
    cap = e == cudaSuccess ? want : 0;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return (T*)p; }
};
struct HostBuf {  // pinned
  void* p = nullptr;
  size_t cap = 0;
  unsigned flags = cudaHostAllocDefault;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap && p) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    size_t want = bytes + bytes / 8 + 64;
    cudaError_t e = cudaHostAlloc(&p, want, flags);
    cap = e == cudaSuccess ? want : 0;
    return e;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return (T*)p; }
};

enum JobKind { JOB_NONE = 0, JOB_TG, JOB_TG_RESIDENT, JOB_TG_UPLOAD, JOB_YT, JOB_YT_RESIDENT, JOB_YT_UPLOAD, JOB_GM, JOB_QUIT };

struct InsertScratch {
  DevBuf arena, cnt, lstate, recnew, newoff, btable, tiles, sc;
};

// the NCCL entry points the merge uses, resolved at run time
struct NcclApi {
  void* h = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

struct Slot {
  int idx = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr, ev_mid = nullptr, ev_p0 = nullptr, ev_p1 = nullptr, ev_e0 = nullptr, ev_e1 = nullptr, ev_f1 = nullptr, ev_fr0 = nullptr, ev_fr1 = nullptr;
  // device inputs
  DevBuf d_recs, d_strs, d_ent_off, d_ents, d_react_off, d_reacts, d_comment_off, d_comments, d_aux,
      d_chans, d_chan_strs;
  // device intermediates / outputs
  DevBuf d_chan_derived, d_chan_len, d_chan_off, d_chan_blob, d_status, d_linelen, d_line_off,
      d_link_start, d_link_count, d_xlen, d_xpos, d_lists, d_arena, d_lstate, d_rec_new, d_new_off, d_link_off, d_links_out,
      d_link_off32, d_btable, d_tiles, d_scalars, d_jsonl, d_url_start, d_url_count, d_urls, d_ent_range;
  // pinned host outputs
  HostBuf h_status, h_line_off, h_jsonl, h_link_off, h_links, h_scalars;
  // page-sized Telegram batches (tg_page.cuh): the input arrays in ONE block / copy, the result arrays in one block / copy
  DevBuf d_page_in, d_page_out;
  HostBuf h_page_in, h_page_out;
  uint32_t page_bpr = 3072;              // running estimate of result bytes per record (sizes the speculative read)
  const uint8_t* dev_jsonl = nullptr;    // where the last batch's JSONL lives on the device (tgi_result_read_jsonl)
  // resident batch descriptor
  JobKind batch = JOB_NONE;  // the kind of the last uploaded batch: JOB_TG, JOB_YT or JOB_GM
  TgBatchDev tg{};
  YtBatchDev yt{};
  GmBatchDev gm{};
  uint64_t yt_desc_bytes = 0;
  uint64_t n_ents = 0, n_reacts = 0, n_comments = 0, in_bytes = 0, chan_strs_len = 0;
  bool resident = false;
  uint64_t dev_jsonl_len = 0;
  // what tgi_pending_edges needs from the slot's last batch
  uint64_t last_n = 0, last_new = 0;
  bool last_frontier = false;
  // job hand-off
  std::mutex mu;
  std::condition_variable cv;
  JobKind job = JOB_NONE;
  bool busy = false, done = false, claimed = false;
  const tgi_tg_batch* in_tg = nullptr;
  const tgi_yt_batch* in_yt = nullptr;
  const tgi_gm_batch* in_gm = nullptr;
  uint32_t run_flags = 0;
  uint64_t ticket = 0;
  bool has_ticket = false;
  int rc = 0;
  tgi_result res{};
  std::thread worker;
};

}  // namespace

struct tgi_ctx {
  tgi_config cfg{};
  std::string label;
  int device = 0;
  int sms = 148;
  std::string err;
  std::mutex err_mu;
  Slot slots[TGI_SLOTS];
  HostBuf h_zero;  // PAD pinned zero bytes (h2d)
  // config blob on device
  DevBuf d_cfg;
  CfgDev cfgdev{};
  std::mutex cfg_mu;
  // frontier: the local set (every key this GPU has seen)
  DevBuf d_pool, d_table, d_fcount, d_err;
  FrontierDev fr{};
  std::mutex fr_mu;
  cudaEvent_t fr_event = nullptr;
  bool fr_event_valid = false;
  // frontier turns: batches with TGI_RUN_FRONTIER take a ticket when they are submitted and enter their frontier phase in
  // ticket order, so NEW flags / n_new / the export order are those of one thread processing the batches in submission order
  std::mutex tk_mu;
  std::condition_variable tk_cv;
  uint64_t tk_next = 0, tk_serving = 0;
  InsertScratch ins;  // scratch of tgi_frontier_insert* / the merge (under fr_mu)
  // frontier -> validator hand-off: resident exclusion sets (tgi_set_add)
  DevBuf x_pool[2], x_table[2], x_count[2], x_payload;
  ExclusionDev excl{};
  // multi-GPU merge: communicator + this rank's partition of the global set
  NcclApi* nccl = nullptr;
  ncclComm_t comm = nullptr;
  int rank = 0, nranks = 1;
  DevBuf o_pool, o_table, o_count, o_payload;
  FrontierDev owned{};
  uint64_t merged_upto = 0, merge_round = 0;
  DevBuf m_cnt, m_all, m_cursor, m_send_keys, m_send_pay, m_recv_keys, m_recv_pay, m_gsize;
  HostBuf m_host;
  cudaEvent_t m_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  tgi_merge_stats mstats{};
  // pinned input staging blocks handed to the packer
  std::mutex stg_mu;
  std::map<void*, size_t> stg_live;
  std::multimap<size_t, void*> stg_free;
  // stats
  std::mutex st_mu;
  tgi_stats stats{};
  // slot allocation for the blocking entry points
  std::mutex alloc_mu;
  std::condition_variable alloc_cv;
};

namespace {

std::string g_create_err;

void set_err(tgi_ctx* c, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) {
    std::lock_guard<std::mutex> g(c->err_mu);
    c->err = buf;
  } else {
    g_create_err = buf;
  }
}

// TGI_TRACE_SLOTS=1: host time (ms since the first stamp) at the synchronisation points of a bulk batch, one line each,
// to stderr — the only timeline tool this image has (no nsys): which slot's copies / kernels overlap with which
void trace_slot(const Slot& s, const char* what) {
  static const bool on = getenv("TGI_TRACE_SLOTS") != nullptr;
  if (!on) return;
  static const auto t0 = std::chrono::steady_clock::now();
  const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  fprintf(stderr, "slot %d %9.3f ms  %s\n", s.idx, ms, what);
}

#define CK(call)                                                                        \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess) {                                                            \
      set_err(c, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return _e == cudaErrorMemoryAllocation ? TGI_E_NOMEM : TGI_E_CUDA;                \
    }                                                                                   \
  } while (0)

// ---- host-side rendering of the injected clock (same rules as render_time on the device) --------
int host_render_time(char* dst, int64_t sec, int32_t nsec, int32_t tz) {
  int64_t t = sec + tz;
  int64_t days = t / 86400, rem = t % 86400;
  if (rem < 0) { rem += 86400; days -= 1; }
  int64_t z = days + 719468;
  int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  int64_t doe = z - era * 146097;
  int64_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  int64_t y = yoe + era * 400;
  int64_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  int64_t mp = (5 * doy + 2) / 153;
  int64_t d = doy - (153 * mp + 2) / 5 + 1;
  int64_t m = mp < 10 ? mp + 3 : mp - 9;
  if (m <= 2) y += 1;
  if (y < 0 || y > 9999) return 0;
  int o = snprintf(dst, 40, "\"%04d-%02d-%02dT%02d:%02d:%02d", (int)y, (int)m, (int)d, (int)(rem / 3600),
                   (int)(rem % 3600 / 60), (int)(rem % 60));
  if (nsec) {
    char f[16];
    snprintf(f, sizeof f, "%09d", nsec);
    int k = 9;
    while (k > 0 && f[k - 1] == '0') k--;
    dst[o++] = '.';
    memcpy(dst + o, f, k);
    o += k;
  }
  if (tz == 0) dst[o++] = 'Z';
  else {
    int a = tz < 0 ? -tz : tz;
    o += snprintf(dst + o, 8, "%c%02d:%02d", tz < 0 ? '-' : '+', a / 3600, a % 3600 / 60);
  }
  dst[o++] = '"';
  return o;
}

// Builds the per-context constant blob (escaped label + clock strings) and uploads it.  The label
// is JSON-escaped ON THE DEVICE by the same Emitter code that escapes everything else.
__global__ void cfg_label_size_kernel(const uint8_t* s, uint32_t n, uint32_t* out) {
  uint32_t e = warp_esc_len(s, n);
  if (lane_id() == 0) *out = e;
}
__global__ void cfg_label_emit_kernel(const uint8_t* s, uint32_t n, uint8_t* out) { esc_to_global(out, s, n); }

int build_cfg_blob(tgi_ctx* c) {
  const tgi_config& cfg = c->cfg;
  char t_tg[48], t_yt[48], t_cap[48];
  int n_tg = host_render_time(t_tg, cfg.created_at_sec, 0, 0);
  int n_yt = host_render_time(t_yt, cfg.created_at_sec, cfg.created_at_nsec, cfg.tz_offset_sec);
  int n_cap = host_render_time(t_cap, cfg.capture_sec, cfg.capture_nsec, cfg.tz_offset_sec);
  cudaStream_t s = c->slots[0].stream;
  uint32_t n = (uint32_t)c->label.size();
  DevBuf raw, len;
  CK(raw.ensure(n));
  CK(len.ensure(4));
  CK(cudaMemsetAsync(raw.p, 0, n + PAD, s));
  if (n) CK(cudaMemcpyAsync(raw.p, c->label.data(), n, cudaMemcpyHostToDevice, s));
  cfg_label_size_kernel<<<1, 32, 0, s>>>(raw.as<uint8_t>(), n, len.as<uint32_t>());
  uint32_t esc = 0;
  CK(cudaMemcpyAsync(&esc, len.p, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  auto pad16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const size_t o_tg = pad16(esc), o_yt = o_tg + pad16(n_tg), o_cap = o_yt + pad16(n_yt);
  size_t total = o_cap + pad16(n_cap);
  CK(c->d_cfg.ensure(total + 16));
  CK(cudaMemsetAsync(c->d_cfg.p, 0, total + 16 + PAD, s));
  cfg_label_emit_kernel<<<1, 32, 0, s>>>(raw.as<uint8_t>(), n, c->d_cfg.as<uint8_t>());
  uint8_t* b = c->d_cfg.as<uint8_t>();
  if (n_tg) CK(cudaMemcpyAsync(b + o_tg, t_tg, n_tg, cudaMemcpyHostToDevice, s));
  if (n_yt) CK(cudaMemcpyAsync(b + o_yt, t_yt, n_yt, cudaMemcpyHostToDevice, s));
  if (n_cap) CK(cudaMemcpyAsync(b + o_cap, t_cap, n_cap, cudaMemcpyHostToDevice, s));
  CK(cudaStreamSynchronize(s));
  raw.release();
  len.release();
  CfgDev d{};
  d.blob = b;
  d.off[0] = 0;
  d.off[1] = (uint32_t)o_tg;
  d.off[2] = (uint32_t)o_yt;
  d.off[3] = (uint32_t)o_cap;
  d.label_len = esc;
  d.created_tg_len = (uint32_t)n_tg;
  d.created_yt_len = (uint32_t)n_yt;
  d.capture_len = (uint32_t)n_cap;
  d.flags = cfg.flags | ((n_tg == 0 || n_cap == 0) ? CFGDEV_CLOCK_INVALID : 0);
  d.tz = cfg.tz_offset_sec;
  d.min_post_date = cfg.min_post_date;
  c->cfgdev = d;
  return TGI_OK;
}

uint64_t next_pow2(uint64_t v) {
  uint64_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

// exclusive scan u32[n] -> u64[n+1]; total also lands in *d_total
int launch_scan(tgi_ctx* c, Slot& s, const uint32_t* in, uint64_t n, uint64_t* out, uint64_t* d_total, uint32_t& launches) {
  if (n <= (uint64_t)SCAN_SMALL_MAX) {  // page-sized batch: one launch instead of three
    scan_small_kernel<<<1, SCAN_SMALL_THREADS, 0, s.stream>>>(in, n, out, d_total);
    launches += 1;
    CK(cudaGetLastError());
    return TGI_OK;
  }
  uint64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  if (ntiles == 0) ntiles = 1;
  CK(s.d_tiles.ensure(ntiles * 8));
  scan_tile_sums_kernel<<<(unsigned)ntiles, SCAN_THREADS, 0, s.stream>>>(in, n, s.d_tiles.as<uint64_t>());
  scan_tiles_kernel<<<1, 1024, 0, s.stream>>>(s.d_tiles.as<uint64_t>(), ntiles, d_total);
  scan_apply_kernel<<<(unsigned)ntiles, SCAN_THREADS, 0, s.stream>>>(in, n, s.d_tiles.as<uint64_t>(), d_total, out);
  launches += 3;
  CK(cudaGetLastError());
  return TGI_OK;
}

int h2d(tgi_ctx* c, Slot& s, DevBuf& d, const void* src, size_t bytes) {
  cudaStream_t st = s.stream;
  CK(d.ensure(bytes));
  if (bytes) CK(cudaMemcpyAsync(d.p, src, bytes, cudaMemcpyHostToDevice, st));
  // the pad behind the array: a COPY of zeros, not a memset — a memset is a kernel and would queue behind whatever the
  // other slots' (persistent, SM-filling) kernels are doing, which chains every one of the eleven uploads to them
  CK(cudaMemcpyAsync((uint8_t*)d.p + bytes, c->h_zero.p, PAD, cudaMemcpyHostToDevice, st));
  s.in_bytes += bytes;
  return TGI_OK;
}

// Small read-backs (the scalars block between the size and the emit pass, the validation flag) do NOT go through the copy
// engine: a device->host cudaMemcpyAsync queues behind the other slots' bulk result copies (1.1 GB each at 500 K messages)
// and the slot's host thread then waits ~45 ms for 96 bytes — measured with TGI_TRACE_SLOTS, profiles/README.md.  A
// one-warp kernel stores them into mapped pinned memory instead; the host sees them after the stream synchronises.
__global__ void publish_kernel(const uint64_t* src, uint64_t* dst_mapped, int n) {
  if ((int)threadIdx.x < n) dst_mapped[threadIdx.x] = src[threadIdx.x];
  __threadfence_system();
}
int publish(tgi_ctx* c, const void* d_src, HostBuf& h, int n_words, cudaStream_t st) {
  void* dp = nullptr;
  CK(cudaHostGetDevicePointer(&dp, h.p, 0));
  publish_kernel<<<1, 32, 0, st>>>((const uint64_t*)d_src, (uint64_t*)dp, n_words);
  CK(cudaGetLastError());
  return TGI_OK;
}

constexpr uint64_t HOST_VALIDATE_MAX = 1u << 16;  // batches up to this many elements are range-checked on the host

// the checks of tg_validate_kernel, on the host (small batches: no extra launch / sync in a page-sized call)
int host_validate_tg(const TgBatchDev& b, const TgBounds& lim) {
  int e = 0;
  for (uint64_t i = 0; i < b.n; i++) e |= tg_check_record(b, lim, i);
  if (e) return e;  // the entity count itself comes from ent_off: do not follow it if the offsets are broken
  for (uint64_t i = 0; i < lim.n_ents; i++) e |= tg_check_entity(b, lim, i);
  for (uint64_t i = 0; i < lim.n_reacts; i++) e |= tg_check_reaction(b, lim, i);
  for (uint64_t i = 0; i < lim.n_comments; i++) e |= tg_check_comment(b, lim, i);
  for (uint32_t i = 0; i < b.n_chans; i++) e |= tg_check_channel(b, lim, i);
  return e;
}

int validate_tg(tgi_ctx* c, const tgi_tg_batch* in) {
  if (!in) { set_err(c, "null batch"); return TGI_E_ARG; }
  if (in->n && (!in->recs || !in->ent_off || !in->react_off || !in->comment_off || !in->chans)) {
    set_err(c, "telegram batch: recs/ent_off/react_off/comment_off/chans must be non-null");
    return TGI_E_ARG;
  }
  if (in->n >= (1ull << 32)) { set_err(c, "telegram batch: too many records (the work lists hold 32-bit record indices)"); return TGI_E_ARG; }
  if (!(c->cfg.flags & TGI_CFG_SKIP_MEDIA)) {
    set_err(c, "TGI_CFG_SKIP_MEDIA is required: media download is an RPC outside this path");
    return TGI_E_ARG;
  }
  const uint64_t n_ents = in->n ? in->ent_off[in->n] : 0;
  if ((n_ents && !in->ents) || (in->n_reacts && !in->reacts) || (in->n_comments && !in->comments) ||
      (in->strs_len && !in->strs) || (in->aux_len && !in->aux) || (in->chan_strs_len && !in->chan_strs)) {
    set_err(c, "telegram batch: a non-empty array has a null pointer");
    return TGI_E_ARG;
  }
  return TGI_OK;
}

// CTAs per SM in the grids of the grid-stride kernels.  Records differ in cost (text length, entities, comments), so a
// grid of exactly the resident CTAs leaves SMs idle behind the slowest stride; many more CTAs than fit let the hardware
// scheduler balance: 8 per SM 41.2 ms per config-2 step, 24: 38.9, 48: 37.7, 96-192: 37.1 (TGI_GRID_MULT, tools/variants_bench.sh)
unsigned grid_mult() {
  static const unsigned v = [] {
    const char* e = getenv("TGI_GRID_MULT");
    return e && atoi(e) > 0 ? (unsigned)atoi(e) : 128u;
  }();
  return v;
}

// ---- page-sized batches: one block in, one launch, one block out (tg_page.cuh, yt_page.cuh) -------------------------
constexpr uint64_t PAGE_MAX_RECS = 8192;          // the in-kernel scans are single-CTA
constexpr uint64_t PAGE_MAX_IN_BYTES = 4u << 20;
// Which batches take the page kernels.  At upload, page_sized(packed size) selects the one-block upload; at run time,
// page_run (the sizes of the resident batch and the run flags) selects the page kernel.
bool page_sized(uint64_t n, uint32_t n_chans, uint64_t in_bytes) {
  if (getenv("TGI_NO_PAGE")) return false;  // A/B switch (read per call): the ordinary pipeline for every size
  return n && n <= PAGE_MAX_RECS && n_chans <= PAGE_MAX_RECS && in_bytes <= PAGE_MAX_IN_BYTES;
}
bool page_run(const Slot& s, uint64_t n, uint32_t n_chans, uint32_t flags) {
  if (!page_sized(n, n_chans, s.in_bytes)) return false;
  if (flags & TGI_RUN_NO_D2H) return false;  // a device-resident result keeps the ordinary buffers
  return (flags & (TGI_RUN_JSONL | TGI_RUN_LINKS | TGI_RUN_FRONTIER)) != 0;
}

// One input array of a batch: the slot buffer it goes to when sent on its own, where it comes from, its size.
struct InArray {
  DevBuf* buf;
  const void* src;
  size_t bytes;
};
size_t packed_bytes(const InArray& a) { return (a.bytes + PAD + 15) & ~(size_t)15; }  // PAD zero bytes behind, as h2d() leaves them
size_t packed_size(const InArray* a, int k) {
  size_t t = 0;
  for (int i = 0; i < k; i++) t += packed_bytes(a[i]);
  return t;
}
// Sends a batch's input arrays and stores their device addresses in dev[].  packed: all of them in one pinned block and
// ONE copy (for a page, eleven copies and eleven pads are a third of what a 100-message call costs; the pack is a host
// memcpy of tens of KB).  Otherwise one copy per array into its slot buffer.
int upload_arrays(tgi_ctx* c, Slot& s, const InArray* a, int k, bool packed, const uint8_t** dev) {
  s.in_bytes = 0;
  if (!packed) {
    for (int i = 0; i < k; i++) {
      const int rc = h2d(c, s, *a[i].buf, a[i].src, a[i].bytes);
      if (rc) return rc;
      dev[i] = a[i].buf->as<uint8_t>();
    }
    return TGI_OK;
  }
  const size_t total = packed_size(a, k);
  CK(s.h_page_in.ensure(total));
  CK(s.d_page_in.ensure(total));
  uint8_t* h = s.h_page_in.as<uint8_t>();
  size_t o = 0;
  for (int i = 0; i < k; i++) {
    if (a[i].bytes) memcpy(h + o, a[i].src, a[i].bytes);
    memset(h + o + a[i].bytes, 0, packed_bytes(a[i]) - a[i].bytes);
    dev[i] = s.d_page_in.as<uint8_t>() + o;
    s.in_bytes += a[i].bytes;
    o += packed_bytes(a[i]);
  }
  CK(cudaMemcpyAsync(s.d_page_in.p, h, total, cudaMemcpyHostToDevice, s.stream));
  return TGI_OK;
}

int upload_tg(tgi_ctx* c, Slot& s, const tgi_tg_batch* in) {
  int rc = validate_tg(c, in);
  if (rc) return rc;
  const uint64_t n = in->n, n_ents = n ? in->ent_off[n] : 0;
  const TgBounds lim{in->strs_len, n_ents, in->n_reacts, in->n_comments, in->aux_len, in->chan_strs_len};
  const bool host_checked = n + n_ents + in->n_reacts + in->n_comments + in->n_chans <= HOST_VALIDATE_MAX;
  if (host_checked) {
    const TgBatchDev hb{n, in->recs, in->strs, in->ent_off, in->ents, in->react_off, in->reacts, in->comment_off, in->comments,
                        in->aux, in->n_chans, in->chans, in->chan_strs};
    const int e = host_validate_tg(hb, lim);
    if (e) { set_err(c, "telegram batch: offsets outside their arrays (mask 0x%x)", e); return TGI_E_ARG; }
  }
  trace_slot(s, "upload: enqueue");
  const InArray arr[11] = {{&s.d_recs, in->recs, n * sizeof(tgi_tg_rec)},
                           {&s.d_strs, in->strs, in->strs_len},
                           {&s.d_ent_off, in->ent_off, (n + 1) * 4},
                           {&s.d_ents, in->ents, n_ents * sizeof(tgi_entity)},
                           {&s.d_react_off, in->react_off, (n + 1) * 4},
                           {&s.d_reacts, in->reacts, in->n_reacts * sizeof(tgi_reaction)},
                           {&s.d_comment_off, in->comment_off, (n + 1) * 4},
                           {&s.d_comments, in->comments, in->n_comments * sizeof(tgi_comment)},
                           {&s.d_aux, in->aux, in->aux_len},
                           {&s.d_chans, in->chans, in->n_chans * sizeof(tgi_tg_chan)},
                           {&s.d_chan_strs, in->chan_strs, in->chan_strs_len}};
  const uint8_t* d[11];
  // a packed page has no device check, so only a batch the host has range-checked is packed
  rc = upload_arrays(c, s, arr, 11, host_checked && page_sized(n, in->n_chans, packed_size(arr, 11)), d);
  if (rc) return rc;
  TgBatchDev& b = s.tg;
  b.n = n;
  b.recs = (const tgi_tg_rec*)d[0];
  b.strs = d[1];
  b.ent_off = (const uint32_t*)d[2];
  b.ents = (const tgi_entity*)d[3];
  b.react_off = (const uint32_t*)d[4];
  b.reacts = (const tgi_reaction*)d[5];
  b.comment_off = (const uint32_t*)d[6];
  b.comments = (const tgi_comment*)d[7];
  b.aux = d[8];
  b.n_chans = in->n_chans;
  b.chans = (const tgi_tg_chan*)d[9];
  b.chan_strs = d[10];
  s.n_ents = n_ents;
  s.n_reacts = in->n_reacts;
  s.n_comments = in->n_comments;
  s.chan_strs_len = in->chan_strs_len;
  s.batch = JOB_TG;
  if (!host_checked) {  // big batch: range-check on the device
    CK(s.d_scalars.ensure(SC_COUNT * 8));
    int* bad = (int*)s.d_scalars.p;
    CK(cudaMemsetAsync(bad, 0, 4, s.stream));
    const uint64_t count = std::max<uint64_t>({n, n_ents, in->n_reacts, in->n_comments, (uint64_t)in->n_chans});
    tg_validate_kernel<<<(unsigned)((count + 255) / 256), 256, 0, s.stream>>>(b, lim, count, bad);
    CK(s.h_scalars.ensure(SC_COUNT * 8));
    rc = publish(c, bad, s.h_scalars, 1, s.stream);
    if (rc) return rc;
    CK(cudaStreamSynchronize(s.stream));
    const int hbad = *s.h_scalars.as<int>();
    trace_slot(s, "upload: landed + validated");
    if (hbad) {
      s.resident = false;
      set_err(c, "telegram batch: offsets outside their arrays (mask 0x%x)", hbad);
      return TGI_E_ARG;
    }
  }
  s.resident = true;
  return TGI_OK;
}

// ---- frontier turns ---------------------------------------------------------------------------------------------------
void take_ticket(tgi_ctx* c, Slot& s, JobKind kind, uint32_t flags) {
  const bool runs = kind == JOB_TG || kind == JOB_TG_RESIDENT || kind == JOB_YT || kind == JOB_YT_RESIDENT;
  if (!runs || !(flags & TGI_RUN_FRONTIER)) return;
  std::lock_guard<std::mutex> g(c->tk_mu);
  s.ticket = c->tk_next++;
  s.has_ticket = true;
}
void turn_begin(tgi_ctx* c, Slot& s) {
  if (!s.has_ticket) return;
  std::unique_lock<std::mutex> lk(c->tk_mu);
  c->tk_cv.wait(lk, [&] { return c->tk_serving == s.ticket; });
}
void turn_end(tgi_ctx* c, Slot& s) {
  if (!s.has_ticket) return;
  {
    std::lock_guard<std::mutex> g(c->tk_mu);
    c->tk_serving++;
    s.has_ticket = false;
  }
  c->tk_cv.notify_all();
}
// a job that ended without a frontier phase (error, empty batch) still has to let the next ticket through
void turn_pass(tgi_ctx* c, Slot& s) {
  if (!s.has_ticket) return;
  turn_begin(c, s);
  turn_end(c, s);
}

// Scratch of a batch's frontier phases: the batch hash table (a power of two >= 2 x table_rows entries), one link state
// per arena row, the new-key count and offset of every record.
int frontier_scratch(tgi_ctx* c, Slot& s, uint64_t n, uint64_t table_rows, uint64_t arena_cap, FrontierBatch& fb) {
  const uint64_t bslots = next_pow2(std::max<uint64_t>(2 * table_rows, 1024));
  CK(s.d_btable.ensure(bslots * 8));
  CK(s.d_lstate.ensure((size_t)arena_cap * 4));
  CK(s.d_rec_new.ensure(n * 4));
  CK(s.d_new_off.ensure((n + 1) * 8));
  fb.btable = s.d_btable.as<uint64_t>();
  fb.bmask = bslots - 1;
  fb.lstate = s.d_lstate.as<uint32_t>();
  fb.rec_new = s.d_rec_new.as<uint32_t>();
  return TGI_OK;
}

// ---- the result: shared by the bulk and the page paths of every batch kind -----------------------------------------------
// the error bits every path reports the same way once the batch is done
int device_errors(tgi_ctx* c, int dev_err) {
  if (dev_err & ERR_FRONTIER_FULL) { set_err(c, "frontier capacity %llu exceeded", (unsigned long long)c->fr.cap); return TGI_E_CAPACITY; }
  if (dev_err & ERR_LINE_MISMATCH) { set_err(c, "internal: sized and emitted line lengths disagree"); return TGI_E_STATE; }
  return TGI_OK;
}
int check_out_bytes(tgi_ctx* c, uint64_t line_total) {
  if (c->cfg.max_out_bytes && line_total > c->cfg.max_out_bytes) {
    set_err(c, "JSONL output %llu bytes exceeds max_out_bytes", (unsigned long long)line_total);
    return TGI_E_CAPACITY;
  }
  return TGI_OK;
}
// The fields of a batch's tgi_result that do not depend on the path (out is zeroed by the caller), from the scalars block
// `hsc` on the host; what tgi_pending_edges needs from the slot's last batch; the context's stats.
void fill_result(tgi_ctx* c, Slot& s, uint64_t n, uint32_t flags, const uint64_t* hsc, uint64_t line_total, uint64_t n_links,
                 uint32_t launches, tgi_result* out) {
  const bool want_json = flags & TGI_RUN_JSONL, want_fr = flags & TGI_RUN_FRONTIER;
  out->n = n;
  float ms = 0;
  cudaEventElapsedTime(&ms, s.ev_k0, s.ev_k1);
  out->kernel_ms = ms;
  out->gpu_launches = launches;
  out->slot = s.idx;
  if (n && want_json) {
    out->var_bytes = hsc[SC_LONG];
    out->main_bytes_out = hsc[SC_LANE_OUT];
    out->main_bytes_in = hsc[SC_LANE_IN];
  }
  out->jsonl_len = want_json ? line_total : 0;
  out->n_links = n_links;
  out->n_new = want_fr ? hsc[SC_NEW] : 0;
  out->frontier_size = want_fr ? hsc[SC_FSIZE] : 0;
  s.last_n = n;
  s.last_new = out->n_new;
  s.last_frontier = want_fr && n;
  std::lock_guard<std::mutex> g(c->st_mu);
  c->stats.records += n;
  c->stats.bytes_in += s.in_bytes;
  c->stats.bytes_out += out->jsonl_len;
  c->stats.links += n_links;
  c->stats.launches += launches;
  c->stats.kernel_ms_total += ms;
  if (want_fr) c->stats.frontier_size = out->frontier_size;
}

// shared tail of the Telegram, YouTube and generic pipelines: frontier phases, link compaction, D2H, result
int finish_batch(tgi_ctx* c, Slot& s, uint64_t n, uint32_t flags, uint64_t line_total, uint32_t arena_used,
                 uint64_t arena_cap, uint32_t launches, tgi_result* out) {
  cudaStream_t st = s.stream;
  const bool want_json = flags & TGI_RUN_JSONL, want_links = flags & TGI_RUN_LINKS, want_fr = flags & TGI_RUN_FRONTIER;
  uint64_t* dsc = s.d_scalars.as<uint64_t>();
  uint64_t* hsc = s.h_scalars.as<uint64_t>();
  s.dev_jsonl_len = want_json ? line_total : 0;
  s.dev_jsonl = s.d_jsonl.as<uint8_t>();

  if (want_fr && n) {
    // frontier phases of different slots are serialised in submission order (tickets)
    turn_begin(c, s);
    std::unique_lock<std::mutex> fg(c->fr_mu);
    if (c->fr_event_valid) CK(cudaStreamWaitEvent(st, c->fr_event, 0));
    FrontierBatch fb;
    int rc = frontier_scratch(c, s, n, arena_used, arena_cap, fb);
    if (rc) return rc;
    CK(cudaEventRecord(s.ev_fr0, st));
    CK(cudaMemsetAsync(fb.btable, 0, (fb.bmask + 1) * 8, st));
    unsigned g = (unsigned)((n + 255) / 256);
    frontier_probe_kernel<<<g, 256, 0, st>>>(n, s.d_link_start.as<uint32_t>(), s.d_link_count.as<uint32_t>(),
                                             s.d_arena.as<tgi_link>(), flags, c->fr, fb, c->excl);
    frontier_count_kernel<<<g, 256, 0, st>>>(n, s.d_link_start.as<uint32_t>(), s.d_link_count.as<uint32_t>(), fb);
    launches += 2;
    rc = launch_scan(c, s, fb.rec_new, n, s.d_new_off.as<uint64_t>(), dsc + SC_NEW, launches);
    if (rc) return rc;
    int* derr = (int*)(dsc + SC_CURSOR) + 1;
    frontier_append_kernel<<<g, 256, 0, st>>>(n, s.d_link_start.as<uint32_t>(), s.d_link_count.as<uint32_t>(),
                                              s.d_arena.as<tgi_link>(), c->fr, fb, s.d_new_off.as<uint64_t>(), derr);
    frontier_commit_kernel<<<1, 1, 0, st>>>(c->fr, s.d_new_off.as<uint64_t>(), n, dsc + SC_NEW, derr);
    launches += 2;
    CK(cudaGetLastError());
    CK(cudaEventRecord(s.ev_fr1, st));
    CK(cudaEventRecord(c->fr_event, st));
    c->fr_event_valid = true;
    fg.unlock();
    turn_end(c, s);
  }
  if (want_links) {
    CK(s.d_link_off.ensure((n + 1) * 8));
    CK(s.d_link_off32.ensure((n + 1) * 4));
    int rc = launch_scan(c, s, s.d_link_count.as<uint32_t>(), n, s.d_link_off.as<uint64_t>(), dsc + SC_LINK_TOTAL, launches);
    if (rc) return rc;
    CK(s.d_links_out.ensure((size_t)arena_used * sizeof(tgi_link) + 64));
    unsigned g = (unsigned)((n + 1 + 255) / 256);
    links_compact_kernel<<<g, 256, 0, st>>>(n, s.d_link_start.as<uint32_t>(), s.d_link_count.as<uint32_t>(),
                                            s.d_link_off.as<uint64_t>(), s.d_arena.as<tgi_link>(),
                                            s.d_links_out.as<tgi_link>(), s.d_link_off32.as<uint32_t>());
    launches++;
    CK(cudaGetLastError());
  }
  CK(cudaEventRecord(s.ev_k1, st));
  CK(cudaMemcpyAsync(hsc, dsc, SC_COUNT * 8, cudaMemcpyDeviceToHost, st));

  memset(out, 0, sizeof *out);
  out->n = n;
  const bool d2h = !(flags & TGI_RUN_NO_D2H);
  if (d2h) {
    CK(s.h_status.ensure(n + 1));
    CK(cudaMemcpyAsync(s.h_status.p, s.d_status.p, n, cudaMemcpyDeviceToHost, st));
    if (want_json) {
      CK(s.h_line_off.ensure((n + 1) * 8));
      CK(s.h_jsonl.ensure(line_total + 1));
      CK(cudaMemcpyAsync(s.h_line_off.p, s.d_line_off.p, (n + 1) * 8, cudaMemcpyDeviceToHost, st));
      if (line_total) CK(cudaMemcpyAsync(s.h_jsonl.p, s.d_jsonl.p, line_total, cudaMemcpyDeviceToHost, st));
    }
    if (want_links) {
      // the exact link count is one more host round trip away (behind the other slots' bulk copies on the copy engine);
      // the arena's fill is an upper bound the host already has: copy that many rows, the tail past n_links is unused
      CK(s.h_link_off.ensure((n + 1) * 4));
      CK(s.h_links.ensure((size_t)arena_used * sizeof(tgi_link) + 64));
      CK(cudaMemcpyAsync(s.h_link_off.p, s.d_link_off32.p, (n + 1) * 4, cudaMemcpyDeviceToHost, st));
      if (arena_used) CK(cudaMemcpyAsync(s.h_links.p, s.d_links_out.p, (size_t)arena_used * sizeof(tgi_link), cudaMemcpyDeviceToHost, st));
    }
  }
  trace_slot(s, "emit + frontier + result copy: enqueued");
  CK(cudaStreamSynchronize(st));
  trace_slot(s, "result landed");
  const int rc = device_errors(c, ((int*)(hsc + SC_CURSOR))[1]);
  if (rc) return rc;
  const uint64_t n_links_total = want_links ? hsc[SC_LINK_TOTAL] : 0;
  if (n_links_total > arena_used) { set_err(c, "internal: more links than arena rows"); return TGI_E_STATE; }
  fill_result(c, s, n, flags, hsc, line_total, n_links_total, launches, out);
  if (n) cudaEventElapsedTime(&out->parse_ms, s.ev_p0, s.ev_p1);
  if (n && want_json) {
    cudaEventElapsedTime(&out->emit_ms, s.ev_e0, s.ev_e1);
    cudaEventElapsedTime(&out->emit_main_ms, s.ev_e0, s.ev_f1);
  }
  if (want_fr && n) cudaEventElapsedTime(&out->frontier_ms, s.ev_fr0, s.ev_fr1);
  if (d2h) {
    out->status = s.h_status.as<uint8_t>();
    if (want_json) {
      out->jsonl = s.h_jsonl.as<uint8_t>();
      out->line_off = s.h_line_off.as<uint64_t>();
    }
    if (want_links) {
      out->link_off = s.h_link_off.as<uint32_t>();
      out->links = s.h_links.as<tgi_link>();
    }
  }
  return TGI_OK;
}

// One cooperative launch and one result copy for a page-sized batch.  PAGE_FALLBACK: the batch did not fit the
// estimate-sized result block or the link arena (nothing was committed): the caller goes on with the ordinary pipeline.
constexpr int PAGE_FALLBACK = -1000;
// ---- shared by the Telegram and the YouTube page paths ------------------------------------------------------------------
struct PageOut {  // the result block: scalars | status | line_off | link_off | links, JSONL
  uint64_t o_status, o_line_off, o_link_off, o_var, var_cap;
};
int page_out_prepare(tgi_ctx* c, Slot& s, uint64_t n, PageOut& L) {
  auto up = [](uint64_t v, uint64_t a) { return (v + a - 1) / a * a; };
  L.o_status = 256;
  L.o_line_off = L.o_status + up(n + 1, 16);
  L.o_link_off = L.o_line_off + (n + 1) * 8;
  L.o_var = up(L.o_link_off + (n + 1) * 4, 256);
  L.var_cap = up(6 * s.in_bytes + 3072 * n + 65536, 256);
  if (const char* v = getenv("TGI_PAGE_VAR_CAP")) L.var_cap = up(strtoull(v, nullptr, 10), 256);  // tests: force the fallback
  CK(s.d_page_out.ensure(L.o_var + L.var_cap));
  CK(s.h_page_out.ensure(L.o_var + L.var_cap));
  return TGI_OK;
}
// launch (in the batch's frontier turn), ONE read of the result block, the result.  PAGE_FALLBACK: nothing was committed.
int page_launch_and_read(tgi_ctx* c, Slot& s, uint32_t flags, uint64_t n, const void* kernel, void** kargs, int occ, const PageOut& L,
                         FrontierDev* fr_arg, ExclusionDev* excl_arg, const char* name, tgi_result* out) {
  cudaStream_t st = s.stream;
  const bool want_json = flags & TGI_RUN_JSONL, want_links = flags & TGI_RUN_LINKS, want_fr = flags & TGI_RUN_FRONTIER;
  auto up = [](uint64_t v, uint64_t a) { return (v + a - 1) / a * a; };
  const uint64_t o_status = L.o_status, o_line_off = L.o_line_off, o_link_off = L.o_link_off, o_var = L.o_var, var_cap = L.var_cap;
  uint8_t* d = s.d_page_out.as<uint8_t>();
  uint8_t* h = s.h_page_out.as<uint8_t>();
  const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)c->sms * occ, std::max<uint64_t>(1, (n + WARPS_PER_CTA - 1) / WARPS_PER_CTA));
  {
    // the launch holds frontier phases: serialised with the other slots' in submission order, like finish_batch
    std::unique_lock<std::mutex> fg(c->fr_mu, std::defer_lock);
    if (want_fr) {
      turn_begin(c, s);
      fg.lock();
      if (c->fr_event_valid) CK(cudaStreamWaitEvent(st, c->fr_event, 0));
      *fr_arg = c->fr;
      *excl_arg = c->excl;
    }
    CK(cudaEventRecord(s.ev_k0, st));
    if (cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(CTA_THREADS), kargs, 0, st) != cudaSuccess) {
      cudaGetLastError();  // e.g. the device is shared and cannot hold the grid: the bulk pipeline needs no co-residency
      return PAGE_FALLBACK;
    }
    CK(cudaEventRecord(s.ev_k1, st));
    if (want_fr) {
      CK(cudaEventRecord(c->fr_event, st));
      c->fr_event_valid = true;
    }
  }
  // ONE read of the result block, sized by what the previous pages needed; a second one only for the rest of a bigger page
  const uint64_t spec = std::min<uint64_t>(var_cap, up((uint64_t)s.page_bpr * n * 5 / 4 + 4096, 256));
  CK(cudaMemcpyAsync(h, d, o_var + spec, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const uint64_t* hsc = (const uint64_t*)h;
  const int dev_err = ((const int*)(hsc + SC_CURSOR))[1];
  if (dev_err & (ERR_ARENA_OVERFLOW | ERR_TOO_MANY_LINKS | ERR_PAGE_OVERFLOW)) return PAGE_FALLBACK;  // keeps its turn
  turn_end(c, s);
  int rc = device_errors(c, dev_err);
  if (rc) return rc;
  const uint64_t line_total = want_json ? hsc[SC_LINE_TOTAL] : 0, n_links_total = want_links ? hsc[SC_LINK_TOTAL] : 0;
  const uint64_t links_bytes = want_links ? up(n_links_total * sizeof(tgi_link), 256) : 0;
  if (want_json) {
    rc = check_out_bytes(c, line_total);
    if (rc) return rc;
  }
  const uint64_t need = links_bytes + line_total;
  if (need > spec) {
    CK(cudaMemcpyAsync(h + o_var + spec, d + o_var + spec, need - spec, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  if (getenv("TGI_PAGE_TRACE")) {
    const uint64_t* t = hsc + PAGE_TRACE_AT;
    fprintf(stderr, "%s n=%llu grid=%u phases us:", name, (unsigned long long)n, grid);
    for (int k = 0; k < PAGE_PHASES; k++) fprintf(stderr, " P%d %.1f", k, (double)(t[k + 1] - t[k]) * 1e-3);
    fprintf(stderr, "  total %.1f |", (double)(t[PAGE_PHASES] - t[0]) * 1e-3);
    static const char* const what[3] = {"parse", "size", "emit"};
    for (int k = 0; k < 3; k++)  // SM cycles (1.965 GHz)
      fprintf(stderr, " slowest %s: rec %u %.1f us", what[k], (unsigned)t[PAGE_PHASES + 1 + k], (double)(t[PAGE_PHASES + 1 + k] >> 32) / 1965.0);
    fprintf(stderr, "\n");
  }
  s.page_bpr = (uint32_t)std::min<uint64_t>(1u << 20, (3ull * s.page_bpr + need / n + 1) / 4 + (need > spec ? need / n / 4 : 0));

  memset(out, 0, sizeof *out);
  fill_result(c, s, n, flags, hsc, line_total, n_links_total, 1, out);
  out->status = h + o_status;
  if (want_json) {
    out->jsonl = h + o_var + links_bytes;
    out->line_off = (const uint64_t*)(h + o_line_off);
  }
  if (want_links) {
    out->link_off = (const uint32_t*)(h + o_link_off);
    out->links = (const tgi_link*)(h + o_var);
  }
  s.dev_jsonl_len = line_total;
  s.dev_jsonl = d + o_var + links_bytes;
  return TGI_OK;
}


int run_tg_page(tgi_ctx* c, Slot& s, const CfgDev& cfg, uint32_t flags, tgi_result* out) {
  TgBatchDev& b = s.tg;
  const uint64_t n = b.n;
  static const int occ = [] {
    int o = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, tg_page_kernel, CTA_THREADS, 0) != cudaSuccess) return 0;
    return o;
  }();
  if (occ <= 0) { cudaGetLastError(); return PAGE_FALLBACK; }
  PageArgs pa{};
  pa.cfg = cfg;
  pa.run_flags = flags;
  const uint64_t arena_cap = s.n_ents + 2 * n + 1024;
  const uint64_t blob_cap = 8 * s.chan_strs_len + 1024ull * b.n_chans + 1024;
  // scratch (the buffers of the ordinary pipeline, so that tgi_pending_edges finds the same arrays afterwards)
  CK(s.d_linelen.ensure(n * 4));
  CK(s.d_link_start.ensure(n * 4));
  CK(s.d_link_count.ensure(n * 4));
  CK(s.d_xlen.ensure(n * 32));
  CK(s.d_xpos.ensure(n * 32));
  CK(s.d_lists.ensure(3 * n * 4));
  CK(s.d_arena.ensure(arena_cap * sizeof(tgi_link)));
  CK(s.d_ent_range.ensure((size_t)s.n_ents * sizeof(int2)));
  CK(s.d_link_off.ensure((n + 1) * 8));
  CK(s.d_chan_derived.ensure((size_t)b.n_chans * sizeof(ChanDerived)));
  CK(s.d_chan_len.ensure((size_t)b.n_chans * 4));
  CK(s.d_chan_off.ensure(((size_t)b.n_chans + 1) * 8));
  CK(s.d_chan_blob.ensure(blob_cap));
  if (flags & TGI_RUN_FRONTIER) {
    const int rc = frontier_scratch(c, s, n, arena_cap, arena_cap, pa.fb);
    if (rc) return rc;
  }
  PageOut L;
  {
    const int rc = page_out_prepare(c, s, n, L);
    if (rc) return rc;
  }
  const uint64_t o_status = L.o_status, o_line_off = L.o_line_off, o_link_off = L.o_link_off, o_var = L.o_var, var_cap = L.var_cap;
  uint8_t* d = s.d_page_out.as<uint8_t>();
  uint64_t* dsc = (uint64_t*)d;

  b.chan_derived = s.d_chan_derived.as<ChanDerived>();
  b.chan_blob = s.d_chan_blob.as<uint8_t>();
  pa.b = b;
  ParseOut& po = pa.po;
  po.status = d + o_status;
  po.linelen = s.d_linelen.as<uint32_t>();
  po.link_start = s.d_link_start.as<uint32_t>();
  po.link_count = s.d_link_count.as<uint32_t>();
  po.xlen = s.d_xlen.as<uint32_t>();
  po.var_total = (unsigned long long*)(dsc + SC_LONG);
  po.arena = s.d_arena.as<tgi_link>();
  po.arena_cap = (uint32_t)arena_cap;
  po.cursor = (uint32_t*)(dsc + SC_CURSOR);
  po.err = (int*)(dsc + SC_CURSOR) + 1;
  po.ent_range = s.d_ent_range.as<int2>();
  EmitIn& ei = pa.ei;
  ei.status = po.status;
  ei.line_off = (const uint64_t*)(d + o_line_off);
  ei.link_start = po.link_start;
  ei.link_count = po.link_count;
  ei.xlen = po.xlen;
  ei.xpos = s.d_xpos.as<uint32_t>();
  ei.arena = po.arena;
  ei.out = nullptr;
  ei.err = po.err;
  ei.lane_text_max = LANE_TEXT_MAX;
  ei.counters = (unsigned long long*)(dsc + SC_LANE_OUT);
  for (int k = 0; k < 3; k++) ei.list[k] = s.d_lists.as<uint32_t>() + (size_t)k * n;
  ei.list_count = (uint32_t*)(dsc + SC_LISTS);
  pa.chan_derived = s.d_chan_derived.as<ChanDerived>();
  pa.chan_len = s.d_chan_len.as<uint32_t>();
  pa.chan_off = s.d_chan_off.as<uint64_t>();
  pa.chan_blob = s.d_chan_blob.as<uint8_t>();
  pa.chan_blob_cap = blob_cap;
  pa.scalars = dsc;
  pa.line_off = (uint64_t*)(d + o_line_off);
  pa.link_off = s.d_link_off.as<uint64_t>();
  pa.link_off32 = (uint32_t*)(d + o_link_off);
  pa.var = d + o_var;
  pa.var_cap = var_cap;
  pa.max_out = c->cfg.max_out_bytes;
  pa.fr = c->fr;
  pa.excl = c->excl;
  pa.bslots = pa.fb.bmask + 1;
  pa.new_off = s.d_new_off.as<uint64_t>();

  void* kargs[] = {&pa};
  return page_launch_and_read(c, s, flags, n, (const void*)tg_page_kernel, kargs, occ, L, &pa.fr, &pa.excl, "tg_page", out);
}

int run_tg(tgi_ctx* c, Slot& s, const CfgDev& cfg, uint32_t flags, tgi_result* out) {
  TgBatchDev& b = s.tg;
  uint64_t n = b.n;
  cudaStream_t st = s.stream;
  uint32_t launches = 0;
  const bool want_json = flags & TGI_RUN_JSONL;
  if (page_run(s, n, b.n_chans, flags)) {
    const int rc = run_tg_page(c, s, cfg, flags, out);
    if (rc != PAGE_FALLBACK) return rc;
  }
  CK(s.d_scalars.ensure(SC_COUNT * 8));
  CK(s.h_scalars.ensure(SC_COUNT * 8));
  uint64_t* dsc = s.d_scalars.as<uint64_t>();
  uint64_t* hsc = s.h_scalars.as<uint64_t>();
  CK(s.d_status.ensure(n));
  CK(s.d_linelen.ensure(n * 4));
  CK(s.d_line_off.ensure((n + 1) * 8));
  CK(s.d_link_start.ensure(n * 4));
  CK(s.d_link_count.ensure(n * 4));
  CK(s.d_xlen.ensure(n * 32));
  uint64_t arena_cap = s.n_ents + n / 2 + 1024;
  if (s.d_arena.cap / sizeof(tgi_link) > arena_cap + 8) arena_cap = (s.d_arena.cap - PAD) / sizeof(tgi_link);

  CK(cudaEventRecord(s.ev_k0, st));
  int dev_err = 0;
  for (int attempt = 0; attempt < 3; attempt++) {
    CK(s.d_arena.ensure(arena_cap * sizeof(tgi_link)));
    CK(cudaMemsetAsync(dsc, 0, SC_COUNT * 8, st));
    if (want_json) {
      CK(s.d_chan_derived.ensure((size_t)b.n_chans * sizeof(ChanDerived)));
      CK(s.d_chan_len.ensure((size_t)b.n_chans * 4));
      CK(s.d_chan_off.ensure(((size_t)b.n_chans + 1) * 8));
      b.chan_derived = s.d_chan_derived.as<ChanDerived>();
      unsigned g = (b.n_chans + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
      if (g) {
        tg_chan_size_kernel<<<g, CTA_THREADS, 0, st>>>(b, s.d_chan_derived.as<ChanDerived>(), s.d_chan_len.as<uint32_t>());
        launches++;
      }
      int rc = launch_scan(c, s, s.d_chan_len.as<uint32_t>(), b.n_chans, s.d_chan_off.as<uint64_t>(), dsc + SC_CHAN_TOTAL, launches);
      if (rc) return rc;
    }
    ParseOut po;
    po.status = s.d_status.as<uint8_t>();
    po.linelen = s.d_linelen.as<uint32_t>();
    po.link_start = s.d_link_start.as<uint32_t>();
    po.link_count = s.d_link_count.as<uint32_t>();
    po.xlen = s.d_xlen.as<uint32_t>();
    po.var_total = (unsigned long long*)(dsc + SC_LONG);
    po.arena = s.d_arena.as<tgi_link>();
    po.arena_cap = (uint32_t)arena_cap;
    po.cursor = (uint32_t*)(dsc + SC_CURSOR);
    po.err = (int*)(dsc + SC_CURSOR) + 1;
    CK(s.d_ent_range.ensure((size_t)s.n_ents * sizeof(int2)));
    po.ent_range = s.d_ent_range.as<int2>();
    if (n) {
      uint64_t want = (n + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
      unsigned g = (unsigned)std::min<uint64_t>(want, (uint64_t)c->sms * grid_mult());
      CK(cudaEventRecord(s.ev_p0, st));
      const uint64_t groups = (n + 31) / 32;
      unsigned ge = (unsigned)std::min<uint64_t>((groups + WARPS_PER_CTA - 1) / WARPS_PER_CTA, (uint64_t)c->sms * grid_mult());
      if (s.n_ents) {  // records with entities first: status + links (two kernels by instruction footprint)
        tg_ent_map_kernel<<<ge, CTA_THREADS, 0, st>>>(b, po);
        tg_parse_ent_kernel<<<ge, CTA_THREADS, 0, st>>>(b, cfg, flags, po);
        launches += 2;
      }
      tg_parse_kernel<<<g, CTA_THREADS, 0, st>>>(b, cfg, flags, po);  // records without entities
      launches++;
      if (want_json) {
        tg_size_lane_kernel<<<ge, CTA_THREADS, 0, st>>>(b, cfg, po);
        launches++;
      }
      CK(cudaEventRecord(s.ev_p1, st));
    }
    if (want_json) {
      int rc = launch_scan(c, s, s.d_linelen.as<uint32_t>(), n, s.d_line_off.as<uint64_t>(), dsc + SC_LINE_TOTAL, launches);
      if (rc) return rc;
    }
    CK(cudaGetLastError());
    {
      const int rc = publish(c, dsc, s.h_scalars, SC_COUNT, st);
      if (rc) return rc;
      launches++;
    }
    trace_slot(s, "parse + size: enqueued");
    CK(cudaStreamSynchronize(st));
    trace_slot(s, "parse + size: done");
    dev_err = ((int*)(hsc + SC_CURSOR))[1];
    uint32_t cursor = ((uint32_t*)(hsc + SC_CURSOR))[0];
    if (dev_err & ERR_ARENA_OVERFLOW) {
      arena_cap = (uint64_t)cursor + 1024;  // exact demand is known now: rerun the parse
      continue;
    }
    break;
  }
  if (dev_err & ERR_ARENA_OVERFLOW) { set_err(c, "link arena overflow persisted"); return TGI_E_CAPACITY; }
  if (dev_err & ERR_TOO_MANY_LINKS) { set_err(c, "a record has 2^20 or more link candidates"); return TGI_E_ARG; }
  uint64_t chan_total = hsc[SC_CHAN_TOTAL], line_total = hsc[SC_LINE_TOTAL];
  uint32_t arena_used = ((uint32_t*)(hsc + SC_CURSOR))[0];

  if (want_json) {
    const int rc = check_out_bytes(c, line_total);
    if (rc) return rc;
    CK(s.d_chan_blob.ensure(chan_total));
    CK(s.d_jsonl.ensure(line_total));
    if (chan_total) CK(cudaMemsetAsync(s.d_chan_blob.p, 0, chan_total, st));  // segment padding must read as zero
    b.chan_blob = s.d_chan_blob.as<uint8_t>();
    unsigned g = (b.n_chans + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    if (g) {
      tg_chan_emit_kernel<<<g, CTA_THREADS, 0, st>>>(b, s.d_chan_derived.as<ChanDerived>(), s.d_chan_off.as<uint64_t>(), s.d_chan_blob.as<uint8_t>());
      launches++;
    }
    if (n) {
      EmitIn ei;
      ei.status = s.d_status.as<uint8_t>();
      ei.line_off = s.d_line_off.as<uint64_t>();
      ei.link_start = s.d_link_start.as<uint32_t>();
      ei.link_count = s.d_link_count.as<uint32_t>();
      ei.xlen = s.d_xlen.as<uint32_t>();
      ei.arena = s.d_arena.as<tgi_link>();
      ei.out = s.d_jsonl.as<uint8_t>();
      ei.err = (int*)(dsc + SC_CURSOR) + 1;
      ei.counters = (unsigned long long*)(dsc + SC_LANE_OUT);
      static const bool attr_set = [] {
        return cudaFuncSetAttribute(tg_emit_lane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(LaneShared)) == cudaSuccess;
      }();
      if (!attr_set) { set_err(c, "cannot reserve %zu bytes of shared memory for the lane emitter", sizeof(LaneShared)); return TGI_E_CUDA; }
      const uint64_t groups = (n + 31) / 32;
      const uint64_t ctas = (groups + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
      CK(cudaEventRecord(s.ev_e0, st));
      CK(s.d_xpos.ensure(n * 32));
      ei.xpos = s.d_xpos.as<uint32_t>();
      CK(s.d_lists.ensure(3 * n * 4));  // work lists of the clean-up kernels (record indices; n < 2^32 checked at upload)
      for (int k = 0; k < 3; k++) ei.list[k] = s.d_lists.as<uint32_t>() + (size_t)k * n;
      ei.list_count = (uint32_t*)(dsc + SC_LISTS);
      ei.lane_text_max = LANE_TEXT_MAX;
      // one LANE per record (tg_lane.cuh): 3 resident CTAs per SM by shared memory, persistent over the record groups
      static const unsigned lane_mult = [] { const char* e = getenv("TGI_LANE_MULT"); return e && atoi(e) > 0 ? (unsigned)atoi(e) : 24u; }();  // 3 resident: 13.06 ms, 24: 12.58
      unsigned gl = (unsigned)std::min<uint64_t>(ctas, (uint64_t)c->sms * lane_mult);
      tg_emit_lane_kernel<<<gl, CTA_THREADS, sizeof(LaneShared), st>>>(b, cfg, ei);
      CK(cudaEventRecord(s.ev_f1, st));
      unsigned gg = (unsigned)std::min<uint64_t>(ctas, (uint64_t)c->sms * grid_mult());
      tg_emit_esc_kernel<ESC_SPARSE><<<gg, CTA_THREADS, 0, st>>>(b, ei);  // descriptions with a few line breaks
      tg_emit_esc_kernel<ESC_DENSE><<<gg, CTA_THREADS, 0, st>>>(b, ei);   // the other strings that need escaping or are long
      tg_emit_maps_kernel<<<gg, CTA_THREADS, 0, st>>>(b, ei);  // comment lists, non-trivial maps, long outlink lists
      launches += 4;
      CK(cudaEventRecord(s.ev_e1, st));
    }
    CK(cudaGetLastError());
  }
  return finish_batch(c, s, n, flags, line_total, arena_used, arena_cap, launches, out);
}

int upload_yt(tgi_ctx* c, Slot& s, const tgi_yt_batch* in) {
  if (!in) { set_err(c, "null batch"); return TGI_E_ARG; }
  if (in->n && (!in->recs || !in->chans)) { set_err(c, "youtube batch: recs/chans must be non-null"); return TGI_E_ARG; }
  if (in->n >= (1ull << 40)) { set_err(c, "youtube batch: too many records"); return TGI_E_ARG; }
  {  // every offset the kernels will follow stays inside its array (O(n) on the host: 80-byte records, no side arrays)
    int e = 0;
    for (uint64_t i = 0; i < in->n; i++) {
      const tgi_yt_rec& r = in->recs[i];
      uint64_t end = r.str_off + (uint64_t)r.id_len + r.title_len + r.desc_len + r.duration_len + r.lang_len;
      for (int k = 0; k < 5; k++) end += r.thumb_len[k] == TGI_YT_THUMB_ABSENT ? 0u : r.thumb_len[k];
      if (end > in->strs_len || end < r.str_off) e |= 1;
      if (r.chan_idx >= in->n_chans) e |= 2;
    }
    for (uint32_t i = 0; i < in->n_chans; i++) {
      const tgi_yt_chan& ch = in->chans[i];
      if ((uint64_t)ch.str_off + ch.id_len + ch.title_len + ch.desc_len + ch.thumb_len + ch.country_len > in->chan_strs_len) e |= 512;
    }
    if (e) { set_err(c, "youtube batch: offsets outside their arrays (mask 0x%x)", e); return TGI_E_ARG; }
  }
  const InArray arr[4] = {{&s.d_recs, in->recs, in->n * sizeof(tgi_yt_rec)},
                          {&s.d_strs, in->strs, in->strs_len},
                          {&s.d_chans, in->chans, in->n_chans * sizeof(tgi_yt_chan)},
                          {&s.d_chan_strs, in->chan_strs, in->chan_strs_len}};
  const uint8_t* d[4];
  const int rc = upload_arrays(c, s, arr, 4, page_sized(in->n, in->n_chans, packed_size(arr, 4)), d);
  if (rc) return rc;
  YtBatchDev& b = s.yt;
  b.n = in->n;
  b.recs = (const tgi_yt_rec*)d[0];
  b.strs = d[1];
  b.n_chans = in->n_chans;
  b.chans = (const tgi_yt_chan*)d[2];
  b.chan_strs = d[3];
  s.yt_desc_bytes = in->strs_len;
  s.batch = JOB_YT;
  s.resident = true;
  s.tg.n = 0;  // the slot no longer holds a Telegram batch: a Telegram resident run finds an empty one
  return TGI_OK;
}

// a page of the Data API (50 videos) in one cooperative launch (yt_page.cuh); PAGE_FALLBACK as in run_tg_page
int run_yt_page(tgi_ctx* c, Slot& s, const CfgDev& cfg, uint32_t flags, tgi_result* out) {
  YtBatchDev& b = s.yt;
  const uint64_t n = b.n;
  static const int occ = [] {
    int o = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, yt_page_kernel, CTA_THREADS, 0) != cudaSuccess) return 0;
    return o;
  }();
  if (occ <= 0) { cudaGetLastError(); return PAGE_FALLBACK; }
  YtPageArgs pa{};
  pa.cfg = cfg;
  pa.run_flags = flags;
  pa.b = b;
  // every URL needs "http://x" (8 bytes), every channel link "youtube.com/" (12 bytes): upper bounds, as in run_yt
  const uint64_t urls_cap = s.yt_desc_bytes / 4 + 1024, arena_cap = s.yt_desc_bytes / 12 + 1024;
  CK(s.d_linelen.ensure(n * 4));
  CK(s.d_link_start.ensure(n * 4));
  CK(s.d_link_count.ensure(n * 4));
  CK(s.d_url_start.ensure(n * 4));
  CK(s.d_url_count.ensure(n * 4));
  CK(s.d_urls.ensure(urls_cap * sizeof(YtUrl)));
  CK(s.d_arena.ensure(arena_cap * sizeof(tgi_link)));
  CK(s.d_xlen.ensure(n * 12));
  CK(s.d_link_off.ensure((n + 1) * 8));
  if (flags & TGI_RUN_FRONTIER) {
    const int rc = frontier_scratch(c, s, n, arena_cap, arena_cap, pa.fb);
    if (rc) return rc;
  }
  PageOut L;
  {
    const int rc = page_out_prepare(c, s, n, L);
    if (rc) return rc;
  }
  uint8_t* d = s.d_page_out.as<uint8_t>();
  uint64_t* dsc = (uint64_t*)d;
  YtOut& yo = pa.yo;
  yo.status = d + L.o_status;
  yo.linelen = s.d_linelen.as<uint32_t>();
  yo.esc_len = s.d_xlen.as<uint32_t>();
  yo.url_start = s.d_url_start.as<uint32_t>();
  yo.url_count = s.d_url_count.as<uint32_t>();
  yo.urls = s.d_urls.as<YtUrl>();
  yo.urls_cap = (uint32_t)urls_cap;
  yo.url_cursor = (uint32_t*)(dsc + SC_URL_CURSOR);
  yo.link_start = s.d_link_start.as<uint32_t>();
  yo.link_count = s.d_link_count.as<uint32_t>();
  yo.arena = s.d_arena.as<tgi_link>();
  yo.arena_cap = (uint32_t)arena_cap;
  yo.cursor = (uint32_t*)(dsc + SC_CURSOR);
  yo.err = (int*)(dsc + SC_CURSOR) + 1;
  pa.scalars = dsc;
  pa.line_off = (uint64_t*)(d + L.o_line_off);
  pa.link_off = s.d_link_off.as<uint64_t>();
  pa.link_off32 = (uint32_t*)(d + L.o_link_off);
  pa.var = d + L.o_var;
  pa.var_cap = L.var_cap;
  pa.max_out = c->cfg.max_out_bytes;
  pa.fr = c->fr;
  pa.excl = c->excl;
  pa.bslots = pa.fb.bmask + 1;
  pa.new_off = s.d_new_off.as<uint64_t>();
  void* kargs[] = {&pa};
  return page_launch_and_read(c, s, flags, n, (const void*)yt_page_kernel, kargs, occ, L, &pa.fr, &pa.excl, "yt_page", out);
}

int run_yt(tgi_ctx* c, Slot& s, const CfgDev& cfg, uint32_t flags, tgi_result* out) {
  YtBatchDev& b = s.yt;
  uint64_t n = b.n;
  cudaStream_t st = s.stream;
  uint32_t launches = 0;
  const bool want_json = flags & TGI_RUN_JSONL;
  if (page_run(s, n, b.n_chans, flags)) {
    const int rc = run_yt_page(c, s, cfg, flags, out);
    if (rc != PAGE_FALLBACK) return rc;
  }
  CK(s.d_scalars.ensure(SC_COUNT * 8));
  CK(s.h_scalars.ensure(SC_COUNT * 8));
  uint64_t* dsc = s.d_scalars.as<uint64_t>();
  uint64_t* hsc = s.h_scalars.as<uint64_t>();
  CK(s.d_status.ensure(n));
  CK(s.d_linelen.ensure(n * 4));
  CK(s.d_line_off.ensure((n + 1) * 8));
  CK(s.d_link_start.ensure(n * 4));
  CK(s.d_link_count.ensure(n * 4));
  CK(s.d_url_start.ensure(n * 4));
  CK(s.d_url_count.ensure(n * 4));
  // every URL needs "http://x" (8 bytes), every channel link "youtube.com/" (12 bytes)
  uint64_t urls_cap = s.yt_desc_bytes / 4 + 1024, arena_cap = s.yt_desc_bytes / 12 + 1024;
  CK(s.d_urls.ensure(urls_cap * sizeof(YtUrl)));
  CK(s.d_arena.ensure(arena_cap * sizeof(tgi_link)));
  CK(cudaEventRecord(s.ev_k0, st));
  CK(cudaMemsetAsync(dsc, 0, SC_COUNT * 8, st));
  YtOut yo;
  yo.status = s.d_status.as<uint8_t>();
  yo.linelen = s.d_linelen.as<uint32_t>();
  CK(s.d_xlen.ensure(n * 12));
  yo.esc_len = s.d_xlen.as<uint32_t>();
  yo.url_start = s.d_url_start.as<uint32_t>();
  yo.url_count = s.d_url_count.as<uint32_t>();
  yo.urls = s.d_urls.as<YtUrl>();
  yo.urls_cap = (uint32_t)std::min<uint64_t>(urls_cap, 0xFFFFFFFFu);
  yo.url_cursor = (uint32_t*)(dsc + SC_URL_CURSOR);
  yo.link_start = s.d_link_start.as<uint32_t>();
  yo.link_count = s.d_link_count.as<uint32_t>();
  yo.arena = s.d_arena.as<tgi_link>();
  yo.arena_cap = (uint32_t)std::min<uint64_t>(arena_cap, 0xFFFFFFFFu);
  yo.cursor = (uint32_t*)(dsc + SC_CURSOR);
  yo.err = (int*)(dsc + SC_CURSOR) + 1;
  unsigned g = (unsigned)std::min<uint64_t>((n + WARPS_PER_CTA - 1) / WARPS_PER_CTA, (uint64_t)c->sms * grid_mult());
  // the lane kernels: one warp per 32 records
  unsigned gl = (unsigned)std::min<uint64_t>(((n + 31) / 32 + WARPS_PER_CTA - 1) / WARPS_PER_CTA, (uint64_t)c->sms * grid_mult());
  if (n) {
    CK(cudaEventRecord(s.ev_p0, st));
    yt_parse_kernel<<<g, CTA_THREADS, 0, st>>>(b, cfg, flags, yo);
    launches++;
    if (want_json) {
      yt_size_lane_kernel<<<gl, CTA_THREADS, 0, st>>>(b, cfg, yo);
      launches++;
    }
    CK(cudaEventRecord(s.ev_p1, st));
  }
  if (want_json) {
    int rc = launch_scan(c, s, s.d_linelen.as<uint32_t>(), n, s.d_line_off.as<uint64_t>(), dsc + SC_LINE_TOTAL, launches);
    if (rc) return rc;
  }
  CK(cudaGetLastError());
  {
    const int rc = publish(c, dsc, s.h_scalars, SC_COUNT, st);
    if (rc) return rc;
    launches++;
  }
  CK(cudaStreamSynchronize(st));
  int dev_err = ((int*)(hsc + SC_CURSOR))[1];
  if (dev_err & ERR_ARENA_OVERFLOW) { set_err(c, "youtube url/link arena overflow (cannot happen: capacities are upper bounds)"); return TGI_E_CAPACITY; }
  if (dev_err & ERR_TOO_MANY_LINKS) { set_err(c, "a record has 2^20 or more channel-link candidates"); return TGI_E_ARG; }
  uint64_t line_total = hsc[SC_LINE_TOTAL];
  uint32_t arena_used = ((uint32_t*)(hsc + SC_CURSOR))[0];
  if (want_json) {
    const int rc = check_out_bytes(c, line_total);
    if (rc) return rc;
    CK(s.d_jsonl.ensure(line_total));
    if (n) {
      CK(cudaEventRecord(s.ev_e0, st));
      // the lane writer takes the clean records, the warp writer the ones with a string that needs escaping
      yt_emit_lane_kernel<<<gl, CTA_THREADS, 0, st>>>(b, cfg, yo, s.d_line_off.as<uint64_t>(), s.d_jsonl.as<uint8_t>(), yo.err);
      yt_emit_kernel<<<gl, CTA_THREADS, 0, st>>>(b, cfg, yo, s.d_line_off.as<uint64_t>(), s.d_jsonl.as<uint8_t>(), yo.err);
      CK(cudaEventRecord(s.ev_f1, st));
      CK(cudaEventRecord(s.ev_e1, st));
      launches += 2;
    }
    CK(cudaGetLastError());
  }
  return finish_batch(c, s, n, flags, line_total, arena_used, arena_cap, launches, out);
}

// generic client.Message batch (a12): upload, size, scan, emit; no links
int run_gm(tgi_ctx* c, Slot& s, const CfgDev& cfg, const tgi_gm_batch* in, uint32_t flags, tgi_result* out) {
  if (!in) { set_err(c, "null batch"); return TGI_E_ARG; }
  if (in->n && !in->recs) { set_err(c, "generic batch: recs must be non-null"); return TGI_E_ARG; }
  if (in->n >= (1ull << 40)) { set_err(c, "generic batch: too many records"); return TGI_E_ARG; }
  {
    int e = 0;
    for (uint64_t i = 0; i < in->n; i++) {
      const tgi_gm_rec& r = in->recs[i];
      const uint64_t end = r.str_off + (uint64_t)r.id_len + r.channel_len + r.text_len + r.sender_len;
      if (end > in->strs_len || end < r.str_off) e |= 1;
      if (in->react_off && (in->react_off[i] > in->react_off[i + 1] || in->react_off[i + 1] > in->n_reacts)) e |= 8;
    }
    for (uint64_t i = 0; i < in->n_reacts; i++)
      if ((uint64_t)in->reacts[i].key_off + in->reacts[i].key_len > in->aux_len) e |= 64;
    if (e) { set_err(c, "generic batch: offsets outside their arrays (mask 0x%x)", e); return TGI_E_ARG; }
  }
  const uint64_t n = in->n;
  cudaStream_t st = s.stream;
  s.resident = false;
  const InArray arr[5] = {{&s.d_recs, in->recs, n * sizeof(tgi_gm_rec)},
                          {&s.d_strs, in->strs, in->strs_len},
                          {&s.d_react_off, in->react_off, in->react_off ? (n + 1) * 4 : 0},
                          {&s.d_reacts, in->reacts, in->n_reacts * sizeof(tgi_gm_reaction)},
                          {&s.d_aux, in->aux, in->aux_len}};
  const uint8_t* d[5];
  int rc = upload_arrays(c, s, arr, 5, false, d);
  if (rc) return rc;
  GmBatchDev& b = s.gm;
  b.n = n;
  b.recs = (const tgi_gm_rec*)d[0];
  b.strs = d[1];
  b.react_off = in->react_off ? (const uint32_t*)d[2] : nullptr;
  b.reacts = (const tgi_gm_reaction*)d[3];
  b.aux = d[4];
  s.batch = JOB_GM;
  uint32_t launches = 0;
  const bool want_json = flags & TGI_RUN_JSONL;
  CK(s.d_scalars.ensure(SC_COUNT * 8));
  CK(s.h_scalars.ensure(SC_COUNT * 8));
  uint64_t* dsc = s.d_scalars.as<uint64_t>();
  uint64_t* hsc = s.h_scalars.as<uint64_t>();
  CK(s.d_status.ensure(n));
  CK(s.d_linelen.ensure(n * 4));
  CK(s.d_line_off.ensure((n + 1) * 8));
  CK(s.d_link_start.ensure(n * 4));
  CK(s.d_link_count.ensure(n * 4));
  CK(s.d_arena.ensure(1024 * sizeof(tgi_link)));
  CK(cudaEventRecord(s.ev_k0, st));
  CK(cudaMemsetAsync(dsc, 0, SC_COUNT * 8, st));
  if (n) {
    CK(cudaMemsetAsync(s.d_link_start.p, 0, n * 4, st));
    CK(cudaMemsetAsync(s.d_link_count.p, 0, n * 4, st));
  }
  int* derr = (int*)(dsc + SC_CURSOR) + 1;
  unsigned g = (unsigned)std::min<uint64_t>((n + WARPS_PER_CTA - 1) / WARPS_PER_CTA, (uint64_t)c->sms * grid_mult());
  CK(cudaEventRecord(s.ev_p0, st));
  if (n) {  // the status does not depend on TGI_RUN_JSONL: the size pass always runs
    gm_size_kernel<<<g, CTA_THREADS, 0, st>>>(b, cfg, s.d_status.as<uint8_t>(), s.d_linelen.as<uint32_t>());
    launches++;
  }
  CK(cudaEventRecord(s.ev_p1, st));
  uint64_t line_total = 0;
  if (want_json) {
    rc = launch_scan(c, s, s.d_linelen.as<uint32_t>(), n, s.d_line_off.as<uint64_t>(), dsc + SC_LINE_TOTAL, launches);
    if (rc) return rc;
    rc = publish(c, dsc, s.h_scalars, SC_COUNT, st);
    if (rc) return rc;
    launches++;
    CK(cudaStreamSynchronize(st));
    line_total = hsc[SC_LINE_TOTAL];
    rc = check_out_bytes(c, line_total);
    if (rc) return rc;
    CK(s.d_jsonl.ensure(line_total));
    CK(cudaEventRecord(s.ev_e0, st));
    if (n) {
      gm_emit_kernel<<<g, CTA_THREADS, 0, st>>>(b, cfg, s.d_status.as<uint8_t>(), s.d_line_off.as<uint64_t>(), s.d_jsonl.as<uint8_t>(), derr);
      launches++;
    }
    CK(cudaEventRecord(s.ev_f1, st));
    CK(cudaEventRecord(s.ev_e1, st));
    CK(cudaGetLastError());
  }
  return finish_batch(c, s, n, flags & ~(uint32_t)TGI_RUN_FRONTIER, line_total, 0, 1024, launches, out);
}

// One job on the slot, with the inputs and flags the slot holds: upload (JOB_TG, JOB_YT, the *_UPLOAD kinds), run
// (JOB_TG, JOB_YT, the *_RESIDENT kinds, JOB_GM), then the job's frontier turn if the run did not take it.
int run_job(tgi_ctx* c, Slot& s, JobKind kind) {
  CfgDev cfg;
  {
    std::lock_guard<std::mutex> g(c->cfg_mu);
    cfg = c->cfgdev;
  }
  int rc = TGI_OK;
  if (kind == JOB_TG || kind == JOB_TG_UPLOAD) rc = upload_tg(c, s, s.in_tg);
  if (kind == JOB_YT || kind == JOB_YT_UPLOAD) rc = upload_yt(c, s, s.in_yt);
  if (rc == TGI_OK && (kind == JOB_TG_UPLOAD || kind == JOB_YT_UPLOAD)) {
    const cudaError_t e = cudaStreamSynchronize(s.stream);
    if (e != cudaSuccess) { set_err(c, "upload sync: %s", cudaGetErrorString(e)); rc = TGI_E_CUDA; }
  }
  if (rc == TGI_OK && (kind == JOB_TG || kind == JOB_TG_RESIDENT)) rc = run_tg(c, s, cfg, s.run_flags, &s.res);
  if (rc == TGI_OK && (kind == JOB_YT || kind == JOB_YT_RESIDENT)) rc = run_yt(c, s, cfg, s.run_flags, &s.res);
  if (kind == JOB_GM) rc = run_gm(c, s, cfg, s.in_gm, s.run_flags, &s.res);
  turn_pass(c, s);
  return rc;
}

void worker_main(tgi_ctx* c, Slot* s) {
  cudaSetDevice(c->device);
  for (;;) {
    JobKind job;
    {
      std::unique_lock<std::mutex> lk(s->mu);
      s->cv.wait(lk, [&] { return s->job != JOB_NONE; });
      job = s->job;
    }
    if (job == JOB_QUIT) return;
    const int rc = run_job(c, *s, job);
    {
      std::lock_guard<std::mutex> lk(s->mu);
      s->rc = rc;
      s->job = JOB_NONE;
      s->done = true;
    }
    s->cv.notify_all();
  }
}

int post_job(tgi_ctx* c, int slot, JobKind kind, const tgi_tg_batch* in, uint32_t flags, const tgi_yt_batch* in_yt = nullptr,
             const tgi_gm_batch* in_gm = nullptr) {
  if (!c) return TGI_E_ARG;
  if (slot < 0 || slot >= TGI_SLOTS) { set_err(c, "bad slot %d", slot); return TGI_E_ARG; }
  Slot& s = c->slots[slot];
  std::lock_guard<std::mutex> lk(s.mu);
  if (s.busy) { set_err(c, "slot %d is busy (wait/release it first)", slot); return TGI_E_STATE; }
  if ((kind == JOB_TG_RESIDENT || kind == JOB_YT_RESIDENT) && !s.resident) { set_err(c, "slot %d holds no resident batch", slot); return TGI_E_STATE; }
  s.busy = true;
  s.done = false;
  s.in_tg = in;
  s.in_yt = in_yt;
  s.in_gm = in_gm;
  s.run_flags = flags;
  take_ticket(c, s, kind, flags);
  s.job = kind;
  s.cv.notify_all();
  return TGI_OK;
}

int wait_job(tgi_ctx* c, int slot, tgi_result* out) {
  if (!c || slot < 0 || slot >= TGI_SLOTS) return TGI_E_ARG;
  Slot& s = c->slots[slot];
  std::unique_lock<std::mutex> lk(s.mu);
  if (!s.busy) { set_err(c, "slot %d has no submitted job", slot); return TGI_E_STATE; }
  s.cv.wait(lk, [&] { return s.done; });
  if (out) *out = s.res;
  int rc = s.rc;
  if (rc != TGI_OK) s.busy = false;  // nothing to release after a failed job (blocking callers still call
                                     // tgi_result_release, which also clears `claimed` and wakes the waiters)
  return rc;
}

// Blocking entry points run the job on the CALLER's thread (the slot is claimed exclusively): two condition-variable
// hand-offs per call are most of what a page-sized batch costs besides the launches themselves.
int run_inline(tgi_ctx* c, int slot, JobKind kind, const tgi_tg_batch* in_tg, const tgi_yt_batch* in_yt, const tgi_gm_batch* in_gm,
               uint32_t flags, tgi_result* out) {
  Slot& s = c->slots[slot];
  {
    std::lock_guard<std::mutex> lk(s.mu);
    if (s.busy) { set_err(c, "slot %d is busy", slot); return TGI_E_STATE; }
    s.busy = true;
    s.done = false;
    s.in_tg = in_tg;
    s.in_yt = in_yt;
    s.in_gm = in_gm;
    s.run_flags = flags;
  }
  take_ticket(c, s, kind, flags);
  cudaSetDevice(c->device);
  const int rc = run_job(c, s, kind);
  {
    std::lock_guard<std::mutex> lk(s.mu);
    s.rc = rc;
    s.done = true;
    if (rc != TGI_OK) s.busy = false;
  }
  if (rc == TGI_OK && out) *out = s.res;
  return rc;
}

int claim_slot(tgi_ctx* c) {
  std::unique_lock<std::mutex> lk(c->alloc_mu);
  for (;;) {
    for (int i = 0; i < TGI_SLOTS; i++) {
      Slot& s = c->slots[i];
      std::lock_guard<std::mutex> g(s.mu);
      if (!s.busy && !s.claimed) { s.claimed = true; return i; }
    }
    c->alloc_cv.wait(lk);
  }
}

}  // namespace

extern "C" {

int tgi_create(const tgi_config* cfg, tgi_ctx** out) {
  tgi_ctx* c = nullptr;
  if (!cfg || !out) { set_err(nullptr, "null argument"); return TGI_E_ARG; }
  if (cfg->abi_version != TGI_ABI_VERSION) { set_err(nullptr, "ABI version mismatch: library %d, caller %u", TGI_ABI_VERSION, cfg->abi_version); return TGI_E_ARG; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_err(nullptr, "no CUDA device visible: libtgingest has no CPU fallback");
    return TGI_E_NODEVICE;
  }
  if (cfg->device < 0 || cfg->device >= ndev) { set_err(nullptr, "device %d out of range (%d visible)", cfg->device, ndev); return TGI_E_ARG; }
  tgi_ctx* ctx = new tgi_ctx();
  ctx->cfg = *cfg;
  ctx->label.assign(cfg->crawl_label ? cfg->crawl_label : "", cfg->crawl_label ? cfg->crawl_label_len : 0);
  ctx->cfg.crawl_label = nullptr;
  ctx->device = cfg->device;
  c = ctx;
  auto fail = [&](int rc) {
    g_create_err = ctx->err;
    tgi_destroy(ctx);
    return rc;
  };
  if (cudaSetDevice(ctx->device) != cudaSuccess) { set_err(c, "cudaSetDevice failed"); return fail(TGI_E_CUDA); }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, ctx->device) == cudaSuccess) ctx->sms = prop.multiProcessorCount;
  if (ctx->h_zero.ensure(PAD) != cudaSuccess) { set_err(c, "pinned allocation failed"); return fail(TGI_E_CUDA); }
  memset(ctx->h_zero.p, 0, PAD);
  for (int i = 0; i < TGI_SLOTS; i++) {
    Slot& s = ctx->slots[i];
    s.idx = i;
    s.h_scalars.flags = cudaHostAllocMapped;  // publish() stores into it from the device
    if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&s.ev_k0) != cudaSuccess || cudaEventCreate(&s.ev_k1) != cudaSuccess ||
        cudaEventCreate(&s.ev_p0) != cudaSuccess || cudaEventCreate(&s.ev_p1) != cudaSuccess ||
        cudaEventCreate(&s.ev_e0) != cudaSuccess || cudaEventCreate(&s.ev_e1) != cudaSuccess || cudaEventCreate(&s.ev_f1) != cudaSuccess ||
        cudaEventCreate(&s.ev_fr0) != cudaSuccess || cudaEventCreate(&s.ev_fr1) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.ev_mid, cudaEventDisableTiming) != cudaSuccess) {
      set_err(c, "stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
      return fail(TGI_E_CUDA);
    }
  }
  if (cudaEventCreateWithFlags(&ctx->fr_event, cudaEventDisableTiming) != cudaSuccess) { set_err(c, "event creation failed"); return fail(TGI_E_CUDA); }
  // frontier
  uint64_t fcap = cfg->frontier_capacity ? cfg->frontier_capacity : (1ull << 22);
  uint64_t tslots = next_pow2(2 * fcap);
  if (ctx->d_pool.ensure(fcap * 32) != cudaSuccess || ctx->d_table.ensure(tslots * 8) != cudaSuccess ||
      ctx->d_fcount.ensure(16) != cudaSuccess) {
    set_err(c, "frontier allocation failed (%llu keys)", (unsigned long long)fcap);
    return fail(TGI_E_NOMEM);
  }
  cudaMemsetAsync(ctx->d_table.p, 0, tslots * 8, ctx->slots[0].stream);
  cudaMemsetAsync(ctx->d_fcount.p, 0, 16, ctx->slots[0].stream);
  cudaStreamSynchronize(ctx->slots[0].stream);
  ctx->fr.pool = ctx->d_pool.as<uint8_t>();
  ctx->fr.cap = fcap;
  ctx->fr.table = ctx->d_table.as<uint64_t>();
  ctx->fr.tmask = tslots - 1;
  ctx->fr.count = ctx->d_fcount.as<uint64_t>();
  ctx->fr.payload = nullptr;
  int rc = build_cfg_blob(ctx);
  if (rc) return fail(rc);
  for (int i = 0; i < TGI_SLOTS; i++) ctx->slots[i].worker = std::thread(worker_main, ctx, &ctx->slots[i]);
  *out = ctx;
  return TGI_OK;
}

void tgi_destroy(tgi_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  tgi_comm_destroy(c);  // while the stream its collectives ran on still exists
  for (int i = 0; i < TGI_SLOTS; i++) {
    Slot& s = c->slots[i];
    if (s.worker.joinable()) {
      {
        std::unique_lock<std::mutex> lk(s.mu);
        s.cv.wait(lk, [&] { return s.job == JOB_NONE; });
        s.job = JOB_QUIT;
      }
      s.cv.notify_all();
      s.worker.join();
    }
    if (s.stream) cudaStreamSynchronize(s.stream);
    DevBuf* db[] = {&s.d_recs, &s.d_strs, &s.d_ent_off, &s.d_ents, &s.d_react_off, &s.d_reacts, &s.d_comment_off,
                    &s.d_comments, &s.d_aux, &s.d_chans, &s.d_chan_strs, &s.d_chan_derived, &s.d_chan_len,
                    &s.d_chan_off, &s.d_chan_blob, &s.d_status, &s.d_linelen, &s.d_line_off, &s.d_link_start,
                    &s.d_link_count, &s.d_xlen, &s.d_xpos, &s.d_lists, &s.d_arena, &s.d_lstate, &s.d_rec_new, &s.d_new_off, &s.d_link_off,
                    &s.d_links_out, &s.d_link_off32, &s.d_btable, &s.d_tiles, &s.d_scalars, &s.d_jsonl,
                    &s.d_url_start, &s.d_url_count, &s.d_urls, &s.d_ent_range, &s.d_page_in, &s.d_page_out};
    for (DevBuf* d : db) d->release();
    HostBuf* hb[] = {&s.h_status, &s.h_line_off, &s.h_jsonl, &s.h_link_off, &s.h_links, &s.h_scalars, &s.h_page_in, &s.h_page_out};
    for (HostBuf* h : hb) h->release();
    if (s.ev_k0) cudaEventDestroy(s.ev_k0);
    if (s.ev_k1) cudaEventDestroy(s.ev_k1);
    if (s.ev_mid) cudaEventDestroy(s.ev_mid);
    for (cudaEvent_t e : {s.ev_p0, s.ev_p1, s.ev_e0, s.ev_e1, s.ev_f1, s.ev_fr0, s.ev_fr1}) if (e) cudaEventDestroy(e);
    if (s.stream) cudaStreamDestroy(s.stream);
  }
  for (auto& f : c->stg_free) cudaFreeHost(f.second);
  for (auto& f : c->stg_live) cudaFreeHost(f.first);
  c->stg_free.clear();
  c->stg_live.clear();
  c->h_zero.release();
  c->m_host.release();
  for (int k = 0; k < 2; k++) { c->x_pool[k].release(); c->x_table[k].release(); c->x_count[k].release(); }
  c->x_payload.release();
  c->d_cfg.release();
  c->d_pool.release();
  c->d_table.release();
  c->d_fcount.release();
  c->d_err.release();
  if (c->fr_event) cudaEventDestroy(c->fr_event);
  delete c;
}

const char* tgi_last_error(tgi_ctx* c) {
  if (!c) return g_create_err.c_str();
  std::lock_guard<std::mutex> g(c->err_mu);
  return c->err.c_str();
}

void tgi_get_stats(tgi_ctx* c, tgi_stats* out) {
  if (!c || !out) return;
  std::lock_guard<std::mutex> g(c->st_mu);
  *out = c->stats;
}

int tgi_set_clock(tgi_ctx* c, int64_t created_at_sec, int32_t created_at_nsec, int64_t capture_sec, int32_t capture_nsec) {
  if (!c) return TGI_E_ARG;
  cudaSetDevice(c->device);
  for (int i = 0; i < TGI_SLOTS; i++) {
    std::lock_guard<std::mutex> lk(c->slots[i].mu);
    if (c->slots[i].busy && !c->slots[i].done) { set_err(c, "tgi_set_clock while slot %d is in flight", i); return TGI_E_STATE; }
  }
  std::lock_guard<std::mutex> g(c->cfg_mu);
  c->cfg.created_at_sec = created_at_sec;
  c->cfg.created_at_nsec = created_at_nsec;
  c->cfg.capture_sec = capture_sec;
  c->cfg.capture_nsec = capture_nsec;
  return build_cfg_blob(c);
}

int tgi_telegram_submit(tgi_ctx* c, int slot, const tgi_tg_batch* in, uint32_t run_flags) {
  return post_job(c, slot, JOB_TG, in, run_flags);
}
int tgi_telegram_wait(tgi_ctx* c, int slot, tgi_result* out) { return wait_job(c, slot, out); }

void tgi_result_release(tgi_ctx* c, int slot) {
  if (!c || slot < 0 || slot >= TGI_SLOTS) return;
  Slot& s = c->slots[slot];
  {
    // alloc_mu is held across the state change: a claim_slot() that has scanned the slots and not yet started to
    // wait would otherwise miss this notification
    std::lock_guard<std::mutex> ag(c->alloc_mu);
    std::lock_guard<std::mutex> lk(s.mu);
    s.busy = false;
    s.claimed = false;
  }
  c->alloc_cv.notify_all();
}

int tgi_telegram_batch(tgi_ctx* c, const tgi_tg_batch* in, uint32_t run_flags, tgi_result* out) {
  if (!c) return TGI_E_ARG;
  int slot = claim_slot(c);
  int rc = run_inline(c, slot, JOB_TG, in, nullptr, nullptr, run_flags, out);
  if (rc != TGI_OK) {
    tgi_result_release(c, slot);
    return rc;
  }
  return TGI_OK;  // result stays valid until tgi_result_release(ctx, out->slot)
}

int tgi_telegram_upload(tgi_ctx* c, int slot, const tgi_tg_batch* in) {
  int rc = post_job(c, slot, JOB_TG_UPLOAD, in, 0);
  if (rc) return rc;
  rc = wait_job(c, slot, nullptr);
  tgi_result_release(c, slot);
  return rc;
}
int tgi_telegram_run_resident(tgi_ctx* c, int slot, uint32_t run_flags, tgi_result* out) {
  int rc = post_job(c, slot, JOB_TG_RESIDENT, nullptr, run_flags);
  if (rc) return rc;
  rc = wait_job(c, slot, out);
  if (rc != TGI_OK) tgi_result_release(c, slot);
  return rc;
}

int tgi_result_read_jsonl(tgi_ctx* c, int slot, uint64_t off, uint64_t len, uint8_t* dst) {
  if (!c || slot < 0 || slot >= TGI_SLOTS || !dst) return TGI_E_ARG;
  cudaSetDevice(c->device);
  Slot& s = c->slots[slot];
  if (off + len > s.dev_jsonl_len) { set_err(c, "read_jsonl out of range"); return TGI_E_ARG; }
  CK(cudaMemcpy(dst, s.dev_jsonl + off, len, cudaMemcpyDeviceToHost));
  return TGI_OK;
}

int tgi_youtube_submit(tgi_ctx* c, int slot, const tgi_yt_batch* in, uint32_t run_flags) {
  return post_job(c, slot, JOB_YT, nullptr, run_flags, in);
}
int tgi_youtube_wait(tgi_ctx* c, int slot, tgi_result* out) { return wait_job(c, slot, out); }
int tgi_youtube_batch(tgi_ctx* c, const tgi_yt_batch* in, uint32_t run_flags, tgi_result* out) {
  if (!c) return TGI_E_ARG;
  int slot = claim_slot(c);
  int rc = run_inline(c, slot, JOB_YT, nullptr, in, nullptr, run_flags, out);
  if (rc != TGI_OK) tgi_result_release(c, slot);
  return rc;
}
int tgi_key_join(tgi_ctx* c, const int64_t* a_keys, uint64_t na, const int64_t* b_keys, uint64_t nb, int64_t* b_index) {
  if (!c || (na && !a_keys) || (nb && (!b_keys || !b_index))) return TGI_E_ARG;
  if (na >= 0xFFFFFFFFull) { set_err(c, "key join: list A has too many elements"); return TGI_E_ARG; }
  cudaSetDevice(c->device);
  if (!nb) return TGI_OK;
  const uint64_t slots = next_pow2(std::max<uint64_t>(2 * na, 1024));
  DevBuf da, db, dt, dout;
  CK(da.ensure(na * 16 + 16));
  CK(db.ensure(nb * 16));
  CK(dt.ensure(slots * 4));
  CK(dout.ensure(nb * 8));
  CK(cudaMemset(dt.p, 0, slots * 4));
  if (na) CK(cudaMemcpy(da.p, a_keys, na * 16, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(db.p, b_keys, nb * 16, cudaMemcpyHostToDevice));
  if (na) join_build_kernel<<<(unsigned)((na + 255) / 256), 256>>>((const longlong2*)da.p, na, dt.as<uint32_t>(), slots - 1);
  join_probe_kernel<<<(unsigned)((nb + 255) / 256), 256>>>((const longlong2*)da.p, dt.as<uint32_t>(), slots - 1, (const longlong2*)db.p, nb,
                                                       (long long*)dout.p);
  CK(cudaGetLastError());
  CK(cudaMemcpy(b_index, dout.p, nb * 8, cudaMemcpyDeviceToHost));
  da.release();
  db.release();
  dt.release();
  dout.release();
  return TGI_OK;
}

int tgi_plan_chunks(const uint64_t* line_off, uint64_t n, uint64_t trigger, uint64_t hard_cap, uint64_t* groups,
                    uint64_t max_groups, uint64_t* n_groups, uint8_t* dropped) {
  if (!line_off || !groups || !n_groups) return TGI_E_ARG;
  uint64_t g = 0, size = 0, files = 0, begin = 0;
  auto flush = [&](uint64_t end) -> bool {  // chunk/main.go:298-311; end = one past the last line of the group
    if (!files) return true;
    if (g >= max_groups) return false;
    groups[2 * g] = begin;
    groups[2 * g + 1] = end;
    g++;
    size = 0;
    files = 0;
    return true;
  };
  for (uint64_t i = 0; i < n; i++) {
    const uint64_t len = line_off[i + 1] - line_off[i];
    if (dropped) dropped[i] = 0;
    if (len == 0) continue;  // no line for this record: no file
    if (len > hard_cap) {    // :316-322
      if (dropped) dropped[i] = 1;
      continue;
    }
    if (size > 0 && size + len > hard_cap) {  // :324-327
      if (!flush(i)) return TGI_E_CAPACITY;
    }
    if (!files) begin = i;
    files++;
    size += len;
    if (size >= trigger) {  // :334-337
      if (!flush(i + 1)) return TGI_E_CAPACITY;
    }
  }
  if (!flush(n)) return TGI_E_CAPACITY;  // :339-343
  *n_groups = g;
  return TGI_OK;
}

int tgi_plan_channel_appends(const uint64_t* line_off, const void* chan_idx, uint32_t chan_stride, uint64_t n, tgi_append_run* runs,
                             uint64_t max_runs, uint64_t* n_runs) {
  if (!line_off || !n_runs || (n && !chan_idx) || (max_runs && !runs)) return TGI_E_ARG;
  uint64_t g = 0;
  bool open = false;
  tgi_append_run cur{};
  for (uint64_t i = 0; i < n; i++) {
    if (line_off[i + 1] == line_off[i]) continue;  // no post was stored for this record
    const uint32_t ch = *(const uint32_t*)((const uint8_t*)chan_idx + (size_t)i * chan_stride);
    if (open && ch == cur.chan_idx) {  // lines without a post in between are empty ranges: the bytes stay contiguous
      cur.end = i + 1;
      cur.byte_end = line_off[i + 1];
      cur.n_lines++;
      continue;
    }
    if (open) {
      if (g >= max_runs) return TGI_E_CAPACITY;
      runs[g++] = cur;
    }
    cur.chan_idx = ch;
    cur.n_lines = 1;
    cur.first = i;
    cur.end = i + 1;
    cur.byte_begin = line_off[i];
    cur.byte_end = line_off[i + 1];
    open = true;
  }
  if (open) {
    if (g >= max_runs) return TGI_E_CAPACITY;
    runs[g++] = cur;
  }
  *n_runs = g;
  return TGI_OK;
}

int tgi_generic_batch(tgi_ctx* c, const tgi_gm_batch* in, uint32_t run_flags, tgi_result* out) {
  if (!c) return TGI_E_ARG;
  int slot = claim_slot(c);
  int rc = run_inline(c, slot, JOB_GM, nullptr, nullptr, in, run_flags, out);
  if (rc != TGI_OK) tgi_result_release(c, slot);
  return rc;
}
int tgi_youtube_upload(tgi_ctx* c, int slot, const tgi_yt_batch* in) {
  int rc = post_job(c, slot, JOB_YT_UPLOAD, nullptr, 0, in);
  if (rc) return rc;
  rc = wait_job(c, slot, nullptr);
  tgi_result_release(c, slot);
  return rc;
}
int tgi_youtube_run_resident(tgi_ctx* c, int slot, uint32_t run_flags, tgi_result* out) {
  int rc = post_job(c, slot, JOB_YT_RESIDENT, nullptr, run_flags);
  if (rc) return rc;
  rc = wait_job(c, slot, out);
  if (rc != TGI_OK) tgi_result_release(c, slot);
  return rc;
}

// ---- frontier host API ------------------------------------------------------------------------------
// Inserts n device-resident 32-byte keys into set `f` (the local set, or this rank's partition of the global set).
// Runs on slot 0's stream under the frontier lock (taken by the caller); the scratch lives in the context.
static int frontier_insert_locked(tgi_ctx* c, FrontierDev& f, const void* d_keys, const uint64_t* d_payload, uint64_t n, void* d_is_new) {
  Slot& s = c->slots[0];
  cudaStream_t st = s.stream;
  InsertScratch& z = c->ins;
  if (c->fr_event_valid) CK(cudaStreamWaitEvent(st, c->fr_event, 0));
  CK(z.arena.ensure(n * sizeof(tgi_link)));
  CK(z.cnt.ensure(n * 4));
  CK(z.lstate.ensure(n * 4));
  CK(z.recnew.ensure(n * 4));
  CK(z.newoff.ensure((n + 1) * 8));
  CK(z.sc.ensure(64));
  uint64_t bslots = next_pow2(std::max<uint64_t>(2 * n, 1024));
  CK(z.btable.ensure(bslots * 8));
  CK(cudaMemsetAsync(z.btable.p, 0, bslots * 8, st));
  CK(cudaMemsetAsync(z.sc.p, 0, 64, st));
  unsigned g = (unsigned)((n + 255) / 256);
  if (!g) g = 1;
  keys_to_links_kernel<<<g, 256, 0, st>>>((const uint8_t*)d_keys, n, z.arena.as<tgi_link>(), z.cnt.as<uint32_t>());
  FrontierBatch fb;
  fb.btable = z.btable.as<uint64_t>();
  fb.bmask = bslots - 1;
  fb.lstate = z.lstate.as<uint32_t>();
  fb.rec_new = z.recnew.as<uint32_t>();
  frontier_probe_kernel<<<g, 256, 0, st>>>(n, nullptr, z.cnt.as<uint32_t>(), z.arena.as<tgi_link>(), 0, f, fb, ExclusionDev{});
  frontier_count_kernel<<<g, 256, 0, st>>>(n, nullptr, z.cnt.as<uint32_t>(), fb);
  {
    uint64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (!ntiles) ntiles = 1;
    CK(z.tiles.ensure(ntiles * 8));
    scan_tile_sums_kernel<<<(unsigned)ntiles, SCAN_THREADS, 0, st>>>(fb.rec_new, n, z.tiles.as<uint64_t>());
    scan_tiles_kernel<<<1, 1024, 0, st>>>(z.tiles.as<uint64_t>(), ntiles, z.sc.as<uint64_t>());
    scan_apply_kernel<<<(unsigned)ntiles, SCAN_THREADS, 0, st>>>(fb.rec_new, n, z.tiles.as<uint64_t>(), z.sc.as<uint64_t>(), z.newoff.as<uint64_t>());
  }
  int* derr = (int*)(z.sc.as<uint64_t>() + 4);
  frontier_append_kernel<<<g, 256, 0, st>>>(n, nullptr, z.cnt.as<uint32_t>(), z.arena.as<tgi_link>(), f, fb, z.newoff.as<uint64_t>(), derr, d_payload);
  frontier_commit_kernel<<<1, 1, 0, st>>>(f, z.newoff.as<uint64_t>(), n, z.sc.as<uint64_t>() + 1, derr);
  if (d_is_new) links_new_flags_kernel<<<g, 256, 0, st>>>(z.arena.as<tgi_link>(), n, (uint8_t*)d_is_new);
  CK(cudaGetLastError());
  CK(cudaEventRecord(c->fr_event, st));
  c->fr_event_valid = true;
  return TGI_OK;
}
static int frontier_insert_check(tgi_ctx* c, const FrontierDev& f) {  // after a stream synchronize
  int herr = 0;
  CK(cudaMemcpy(&herr, (int*)(c->ins.sc.as<uint64_t>() + 4), 4, cudaMemcpyDeviceToHost));
  if (herr & ERR_FRONTIER_FULL) { set_err(c, "frontier capacity %llu exceeded", (unsigned long long)f.cap); return TGI_E_CAPACITY; }
  return TGI_OK;
}
static int frontier_insert_impl(tgi_ctx* c, const void* d_keys, uint64_t n, void* d_is_new) {
  std::unique_lock<std::mutex> fg(c->fr_mu);
  int rc = frontier_insert_locked(c, c->fr, d_keys, nullptr, n, d_is_new);
  if (rc) return rc;
  CK(cudaStreamSynchronize(c->slots[0].stream));
  return frontier_insert_check(c, c->fr);
}

int tgi_frontier_insert(tgi_ctx* c, const uint8_t* keys32, uint64_t n, uint8_t* is_new) {
  if (!c || (n && !keys32)) return TGI_E_ARG;
  if (n >= (1ull << 32)) { set_err(c, "too many keys in one call"); return TGI_E_ARG; }
  cudaSetDevice(c->device);
  if (!n) return TGI_OK;
  cudaStream_t st = c->slots[0].stream;
  DevBuf dk, dn;
  CK(dk.ensure(n * 32));
  CK(dn.ensure(n));
  CK(cudaMemcpyAsync(dk.p, keys32, n * 32, cudaMemcpyHostToDevice, st));
  int rc = frontier_insert_impl(c, dk.p, n, dn.p);
  if (rc == TGI_OK && is_new) {
    CK(cudaMemcpyAsync(is_new, dn.p, n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  return rc;
}
int tgi_frontier_insert_dev(tgi_ctx* c, const void* d_keys32, uint64_t n, void* d_is_new) {
  if (!c || (n && !d_keys32)) return TGI_E_ARG;
  cudaSetDevice(c->device);
  if (!n) return TGI_OK;
  return frontier_insert_impl(c, d_keys32, n, d_is_new);
}
int tgi_frontier_sync(tgi_ctx* c) {
  if (!c) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  if (c->fr_event_valid) CK(cudaEventSynchronize(c->fr_event));
  return TGI_OK;
}
// all copies / memsets of the frontier go through slot 0's stream (the library's streams are non-blocking: work on
// the legacy default stream would not be ordered with them) and are synchronised before returning
static int frontier_read_count(tgi_ctx* c, const FrontierDev& f, uint64_t* n) {
  cudaStream_t st = c->slots[0].stream;
  if (c->fr_event_valid) CK(cudaStreamWaitEvent(st, c->fr_event, 0));
  CK(cudaMemcpyAsync(n, f.count, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return TGI_OK;
}
int tgi_frontier_size(tgi_ctx* c, uint64_t* n) {
  if (!c || !n) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  return frontier_read_count(c, c->fr, n);
}
int tgi_frontier_export(tgi_ctx* c, uint8_t* keys32, uint64_t cap, uint64_t* n) {
  if (!c || !n) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  uint64_t sz = 0;
  int rc = frontier_read_count(c, c->fr, &sz);
  if (rc) return rc;
  uint64_t m = sz < cap ? sz : cap;
  if (m && keys32) {
    CK(cudaMemcpyAsync(keys32, c->fr.pool, m * 32, cudaMemcpyDeviceToHost, c->slots[0].stream));
    CK(cudaStreamSynchronize(c->slots[0].stream));
  }
  *n = sz;
  return TGI_OK;
}
int tgi_frontier_export_dev(tgi_ctx* c, void* d_keys32, uint64_t cap, uint64_t first, uint64_t* n) {
  if (!c || !n) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  uint64_t sz = 0;
  int rc = frontier_read_count(c, c->fr, &sz);
  if (rc) return rc;
  uint64_t avail = first < sz ? sz - first : 0;
  uint64_t m = avail < cap ? avail : cap;
  if (m && d_keys32) {
    CK(cudaMemcpyAsync(d_keys32, c->fr.pool + 32 * first, m * 32, cudaMemcpyDeviceToDevice, c->slots[0].stream));
    CK(cudaStreamSynchronize(c->slots[0].stream));  // the caller's stream may read the keys as soon as this returns
  }
  *n = m;
  return TGI_OK;
}
static int frontier_clear_set(tgi_ctx* c, FrontierDev& f) {
  cudaStream_t st = c->slots[0].stream;
  CK(cudaMemsetAsync(f.table, 0, (f.tmask + 1) * 8, st));
  CK(cudaMemsetAsync(f.count, 0, 8, st));
  return TGI_OK;
}
int tgi_frontier_clear(tgi_ctx* c) {
  if (!c) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  cudaStream_t st = c->slots[0].stream;
  if (c->fr_event_valid) CK(cudaStreamWaitEvent(st, c->fr_event, 0));
  int rc = frontier_clear_set(c, c->fr);
  if (rc == TGI_OK && c->owned.table) rc = frontier_clear_set(c, c->owned);
  if (rc) return rc;
  c->merged_upto = 0;
  CK(cudaEventRecord(c->fr_event, st));
  c->fr_event_valid = true;
  CK(cudaStreamSynchronize(st));
  return TGI_OK;
}

// ---- frontier -> validator hand-off (SURVEY 8f rank 3) ------------------------------------------------------------
static FrontierDev* excl_set(tgi_ctx* c, int which) {
  return which == TGI_SET_INVALID ? &c->excl.invalid : which == TGI_SET_DISCOVERED ? &c->excl.discovered : nullptr;
}
int tgi_set_add(tgi_ctx* c, int which, const uint8_t* keys32, const int64_t* stamp_sec, uint64_t n) {
  if (!c || (n && !keys32)) return TGI_E_ARG;
  FrontierDev* f = excl_set(c, which);
  if (!f) { set_err(c, "tgi_set_add: unknown set %d", which); return TGI_E_ARG; }
  if (n >= (1ull << 32)) { set_err(c, "too many keys in one call"); return TGI_E_ARG; }
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  cudaStream_t st = c->slots[0].stream;
  const int k = which == TGI_SET_INVALID ? 0 : 1;
  if (!f->table) {  // first use: same capacity as the dedup set
    const uint64_t fcap = c->fr.cap, tslots = c->fr.tmask + 1;
    CK(c->x_pool[k].ensure(fcap * 32));
    CK(c->x_table[k].ensure(tslots * 8));
    CK(c->x_count[k].ensure(16));
    if (k == 0) CK(c->x_payload.ensure(fcap * 8));
    CK(cudaMemsetAsync(c->x_table[k].p, 0, tslots * 8, st));
    CK(cudaMemsetAsync(c->x_count[k].p, 0, 16, st));
    f->pool = c->x_pool[k].as<uint8_t>();
    f->cap = fcap;
    f->table = c->x_table[k].as<uint64_t>();
    f->tmask = tslots - 1;
    f->count = c->x_count[k].as<uint64_t>();
    f->payload = k == 0 ? c->x_payload.as<uint64_t>() : nullptr;
  }
  if (!n) return TGI_OK;
  DevBuf dk, dp;
  CK(dk.ensure(n * 32));
  CK(cudaMemcpyAsync(dk.p, keys32, n * 32, cudaMemcpyHostToDevice, st));
  const uint64_t* pay = nullptr;
  if (k == 0 && stamp_sec) {
    CK(dp.ensure(n * 8));
    CK(cudaMemcpyAsync(dp.p, stamp_sec, n * 8, cudaMemcpyHostToDevice, st));
    pay = dp.as<uint64_t>();
  }
  int rc = frontier_insert_locked(c, *f, dk.p, pay, n, nullptr);
  if (rc) return rc;
  CK(cudaStreamSynchronize(st));
  return frontier_insert_check(c, *f);
}
int tgi_set_clear(tgi_ctx* c, int which) {
  if (!c) return TGI_E_ARG;
  FrontierDev* f = excl_set(c, which);
  if (!f) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  if (!f->table) return TGI_OK;
  cudaStream_t st = c->slots[0].stream;
  if (c->fr_event_valid) CK(cudaStreamWaitEvent(st, c->fr_event, 0));
  int rc = frontier_clear_set(c, *f);
  if (rc) return rc;
  CK(cudaStreamSynchronize(st));
  return TGI_OK;
}
int tgi_set_size(tgi_ctx* c, int which, uint64_t* n) {
  if (!c || !n) return TGI_E_ARG;
  FrontierDev* f = excl_set(c, which);
  if (!f) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  *n = 0;
  if (!f->table) return TGI_OK;
  return frontier_read_count(c, *f, n);
}
int tgi_set_now(tgi_ctx* c, int64_t now_sec) {
  if (!c) return TGI_E_ARG;
  std::lock_guard<std::mutex> g(c->fr_mu);
  c->excl.now_sec = now_sec;
  return TGI_OK;
}
int tgi_pending_edges(tgi_ctx* c, int slot, int64_t now_sec, tgi_edge* rows, uint64_t cap, uint64_t* n) {
  if (!c || !n || slot < 0 || slot >= TGI_SLOTS || (cap && !rows)) return TGI_E_ARG;
  cudaSetDevice(c->device);
  Slot& s = c->slots[slot];
  if (!s.last_frontier) { *n = 0; if (s.last_n == 0) return TGI_OK; set_err(c, "tgi_pending_edges: the slot's last batch ran without TGI_RUN_FRONTIER"); return TGI_E_STATE; }
  *n = s.last_new;
  const uint64_t m = s.last_new < cap ? s.last_new : cap;
  if (!m) return TGI_OK;
  std::lock_guard<std::mutex> g(c->fr_mu);
  cudaStream_t st = s.stream;
  if (c->fr_event_valid) CK(cudaStreamWaitEvent(st, c->fr_event, 0));
  DevBuf drows;
  CK(drows.ensure(m * sizeof(tgi_edge)));
  ExclusionDev x = c->excl;
  x.now_sec = now_sec;
  // the resident batch descriptor, not the upload buffers: a page-sized batch lives in the slot's one-block upload
  const bool yt = s.batch == JOB_YT;
  const uint32_t* chan = yt ? &s.yt.recs->chan_idx : &s.tg.recs->chan_idx;
  const uint32_t stride = yt ? (uint32_t)sizeof(tgi_yt_rec) : (uint32_t)sizeof(tgi_tg_rec);
  edges_emit_kernel<<<(unsigned)((s.last_n + 255) / 256), 256, 0, st>>>(s.last_n, s.d_link_start.as<uint32_t>(), s.d_link_count.as<uint32_t>(),
                                                                    s.d_arena.as<tgi_link>(), chan, stride, s.d_new_off.as<uint64_t>(), x,
                                                                    drows.as<tgi_edge>(), m);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(rows, drows.p, m * sizeof(tgi_edge), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return TGI_OK;
}

// ---- pinned input staging ---------------------------------------------------------------------------------
int tgi_acquire_staging(tgi_ctx* c, uint64_t bytes, void** out) {
  if (!c || !out) return TGI_E_ARG;
  cudaSetDevice(c->device);
  if (bytes == 0) bytes = 1;
  std::lock_guard<std::mutex> g(c->stg_mu);
  auto it = c->stg_free.lower_bound(bytes);
  if (it != c->stg_free.end() && it->first <= bytes + bytes / 2 + 4096) {  // recycle a block that is not much larger
    *out = it->second;
    c->stg_live[it->second] = it->first;
    c->stg_free.erase(it);
    return TGI_OK;
  }
  const size_t want = (bytes + 4095 + 64) & ~(size_t)4095;
  void* p = nullptr;
  cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    set_err(c, "cudaHostAlloc(%zu) failed: %s", want, cudaGetErrorString(e));
    return TGI_E_NOMEM;
  }
  c->stg_live[p] = want;
  *out = p;
  return TGI_OK;
}
int tgi_release_staging(tgi_ctx* c, void* block) {
  if (!c || !block) return TGI_E_ARG;
  std::lock_guard<std::mutex> g(c->stg_mu);
  auto it = c->stg_live.find(block);
  if (it == c->stg_live.end()) { set_err(c, "tgi_release_staging: not a live staging block"); return TGI_E_ARG; }
  size_t held = 0;
  for (auto& f : c->stg_free) held += f.first;
  if (held + it->second > (4ull << 30)) cudaFreeHost(block);  // keep at most 4 GiB of idle pinned memory around
  else c->stg_free.emplace(it->second, block);
  c->stg_live.erase(it);
  return TGI_OK;
}

// ---- multi-GPU merge (SURVEY 8e option A) ---------------------------------------------------------------------
#define NK(call)                                                                                  \
  do {                                                                                            \
    ncclResult_t _r = (call);                                                                     \
    if (_r != ncclSuccess) {                                                                      \
      set_err(c, "%s failed: %s", #call, c->nccl && c->nccl->GetErrorString ? c->nccl->GetErrorString(_r) : "?"); \
      return TGI_E_CUDA;                                                                          \
    }                                                                                             \
  } while (0)

static NcclApi* load_nccl(std::string& why) {
  static std::mutex mu;
  static NcclApi api;
  std::lock_guard<std::mutex> g(mu);
  if (api.h) return &api;
  void* h = nullptr;
  for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
    h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) { why = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "?"); return nullptr; }
#define SYM(field, name)                                        \
  api.field = (decltype(api.field))dlsym(h, name);              \
  if (!api.field) { why = std::string("libnccl lacks ") + name; return nullptr; }
  SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(CommDestroy, "ncclCommDestroy")
  SYM(AllGather, "ncclAllGather") SYM(AllReduce, "ncclAllReduce") SYM(Broadcast, "ncclBroadcast") SYM(Send, "ncclSend")
  SYM(Recv, "ncclRecv") SYM(GroupStart, "ncclGroupStart") SYM(GroupEnd, "ncclGroupEnd") SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
  api.h = h;
  return &api;
}

int tgi_comm_unique_id(uint8_t id[TGI_COMM_ID_BYTES]) {
  if (!id) return TGI_E_ARG;
  std::string why;
  NcclApi* a = load_nccl(why);
  if (!a) { set_err(nullptr, "%s", why.c_str()); return TGI_E_STATE; }
  ncclUniqueId u;
  static_assert(sizeof(u) == TGI_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
  if (a->GetUniqueId(&u) != ncclSuccess) { set_err(nullptr, "ncclGetUniqueId failed"); return TGI_E_CUDA; }
  memcpy(id, &u, sizeof u);
  return TGI_OK;
}

int tgi_comm_init(tgi_ctx* c, const uint8_t id[TGI_COMM_ID_BYTES], int rank, int nranks) {
  if (!c || !id || nranks < 1 || nranks > 64 || rank < 0 || rank >= nranks) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  if (c->comm) { set_err(c, "communicator already initialised"); return TGI_E_STATE; }
  std::string why;
  c->nccl = load_nccl(why);
  if (!c->nccl) { set_err(c, "%s", why.c_str()); return TGI_E_STATE; }
  ncclUniqueId u;
  memcpy(&u, id, sizeof u);
  NK(c->nccl->CommInitRank(&c->comm, nranks, u, rank));
  c->rank = rank;
  c->nranks = nranks;
  // this rank's partition of the global set: sized like the local set (a skewed hash cannot overflow it before the
  // local sets do)
  const uint64_t fcap = c->fr.cap, tslots = c->fr.tmask + 1;
  CK(c->o_pool.ensure(fcap * 32));
  CK(c->o_table.ensure(tslots * 8));
  CK(c->o_count.ensure(16));
  CK(c->o_payload.ensure(fcap * 8));
  cudaStream_t st = c->slots[0].stream;
  CK(cudaMemsetAsync(c->o_table.p, 0, tslots * 8, st));
  CK(cudaMemsetAsync(c->o_count.p, 0, 16, st));
  c->owned.pool = c->o_pool.as<uint8_t>();
  c->owned.cap = fcap;
  c->owned.table = c->o_table.as<uint64_t>();
  c->owned.tmask = tslots - 1;
  c->owned.count = c->o_count.as<uint64_t>();
  c->owned.payload = c->o_payload.as<uint64_t>();
  CK(c->m_cnt.ensure(64 * 8));
  CK(c->m_all.ensure(64 * 64 * 8));
  CK(c->m_cursor.ensure(64 * 8));
  CK(c->m_gsize.ensure(16));
  CK(c->m_host.ensure(64 * 64 * 8 + 64));
  for (auto& e : c->m_ev) CK(cudaEventCreate(&e));
  CK(cudaStreamSynchronize(st));
  c->merged_upto = 0;
  c->merge_round = 0;
  return TGI_OK;
}

int tgi_comm_destroy(tgi_ctx* c) {
  if (!c) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  if (c->comm) {
    cudaStreamSynchronize(c->slots[0].stream);
    c->nccl->CommDestroy(c->comm);
    c->comm = nullptr;
  }
  for (auto& e : c->m_ev) if (e) { cudaEventDestroy(e); e = nullptr; }
  c->owned = FrontierDev{};
  return TGI_OK;
}

int tgi_frontier_merge(tgi_ctx* c, uint64_t* global_size, uint64_t* owned) {
  if (!c) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  if (!c->comm) { set_err(c, "tgi_frontier_merge needs tgi_comm_init first"); return TGI_E_STATE; }
  NcclApi& N = *c->nccl;
  const int G = c->nranks, me = c->rank;
  cudaStream_t st = c->slots[0].stream;
  uint64_t* hb = c->m_host.as<uint64_t>();
  uint64_t sz = 0;
  int rc = frontier_read_count(c, c->fr, &sz);
  if (rc) return rc;
  const uint64_t first = c->merged_upto, m = sz > first ? sz - first : 0;
  // 1. how many of my new keys go to each owner; every rank learns every count
  CK(cudaEventRecord(c->m_ev[0], st));
  CK(cudaMemsetAsync(c->m_cnt.p, 0, 64 * 8, st));
  if (m) merge_count_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(c->fr.pool, first, m, (uint32_t)G, c->m_cnt.as<unsigned long long>());
  CK(cudaGetLastError());
  NK(N.AllGather(c->m_cnt.p, c->m_all.p, (size_t)G, ncclUint64, c->comm, st));
  CK(cudaMemcpyAsync(hb, c->m_all.p, (size_t)G * G * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  std::vector<uint64_t> send_off(G + 1, 0), recv_off(G + 1, 0);
  for (int p = 0; p < G; p++) {
    send_off[p + 1] = send_off[p] + hb[(size_t)me * G + p];
    recv_off[p + 1] = recv_off[p] + hb[(size_t)p * G + me];
  }
  const uint64_t R = recv_off[G];
  if (send_off[G] != m) { set_err(c, "merge: bucket counts do not add up"); return TGI_E_STATE; }
  // 2. bucket my new keys by owner
  CK(c->m_send_keys.ensure(m * 32));
  CK(c->m_send_pay.ensure(m * 8));
  CK(c->m_recv_keys.ensure(R * 32));
  CK(c->m_recv_pay.ensure(R * 8));
  uint64_t* hcur = hb + (size_t)G * G;
  for (int p = 0; p < G; p++) hcur[p] = send_off[p];
  CK(cudaMemcpyAsync(c->m_cursor.p, hcur, (size_t)G * 8, cudaMemcpyHostToDevice, st));
  const uint64_t pay_base = (c->merge_round << 52) | ((uint64_t)me << 44);
  if (m) merge_scatter_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(c->fr.pool, first, m, (uint32_t)G, c->m_cursor.as<unsigned long long>(),
                                                                      c->m_send_keys.as<uint8_t>(), c->m_send_pay.as<uint64_t>(), pay_base);
  CK(cudaGetLastError());
  CK(cudaEventRecord(c->m_ev[1], st));
  // 3. exchange: grouped send / recv, the receive buffer laid out by source rank
  NK(N.GroupStart());
  for (int p = 0; p < G; p++) {
    const uint64_t sc = send_off[p + 1] - send_off[p], rc2 = recv_off[p + 1] - recv_off[p];
    if (p == me) continue;
    if (sc) {
      NK(N.Send(c->m_send_keys.as<uint8_t>() + 32 * send_off[p], sc * 32, ncclUint8, p, c->comm, st));
      NK(N.Send(c->m_send_pay.as<uint64_t>() + send_off[p], sc, ncclUint64, p, c->comm, st));
    }
    if (rc2) {
      NK(N.Recv(c->m_recv_keys.as<uint8_t>() + 32 * recv_off[p], rc2 * 32, ncclUint8, p, c->comm, st));
      NK(N.Recv(c->m_recv_pay.as<uint64_t>() + recv_off[p], rc2, ncclUint64, p, c->comm, st));
    }
  }
  NK(N.GroupEnd());
  {
    const uint64_t sc = send_off[me + 1] - send_off[me];
    if (sc) {
      CK(cudaMemcpyAsync(c->m_recv_keys.as<uint8_t>() + 32 * recv_off[me], c->m_send_keys.as<uint8_t>() + 32 * send_off[me], sc * 32, cudaMemcpyDeviceToDevice, st));
      CK(cudaMemcpyAsync(c->m_recv_pay.as<uint64_t>() + recv_off[me], c->m_send_pay.as<uint64_t>() + send_off[me], sc * 8, cudaMemcpyDeviceToDevice, st));
    }
  }
  CK(cudaEventRecord(c->m_ev[2], st));
  // 4. the owner inserts what it received (source-rank-major: the lowest rank's copy of a key wins)
  if (R) {
    rc = frontier_insert_locked(c, c->owned, c->m_recv_keys.p, c->m_recv_pay.as<uint64_t>(), R, nullptr);
    if (rc) return rc;
  }
  // 5. global size = sum of the partitions
  NK(N.AllReduce(c->owned.count, c->m_gsize.p, 1, ncclUint64, ncclSum, c->comm, st));
  CK(cudaEventRecord(c->m_ev[3], st));
  CK(cudaMemcpyAsync(hb, c->m_gsize.p, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(hb + 1, c->owned.count, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (R) {
    rc = frontier_insert_check(c, c->owned);
    if (rc) return rc;
  }
  if (global_size) *global_size = hb[0];
  if (owned) *owned = hb[1];
  float t0 = 0, t1 = 0, t2 = 0;
  cudaEventElapsedTime(&t0, c->m_ev[0], c->m_ev[1]);
  cudaEventElapsedTime(&t1, c->m_ev[1], c->m_ev[2]);
  cudaEventElapsedTime(&t2, c->m_ev[2], c->m_ev[3]);
  c->mstats.merges++;
  c->mstats.keys_sent += m - (send_off[me + 1] - send_off[me]);
  c->mstats.keys_received += R - (recv_off[me + 1] - recv_off[me]);
  c->mstats.keys_owned = hb[1];
  c->mstats.bytes_sent += (m - (send_off[me + 1] - send_off[me])) * 40;
  c->mstats.bucket_ms += t0;
  c->mstats.exchange_ms += t1;
  c->mstats.insert_ms += t2;
  c->mstats.last_bucket_ms = t0;
  c->mstats.last_exchange_ms = t1;
  c->mstats.last_insert_ms = t2;
  c->merged_upto = sz;
  c->merge_round++;
  return TGI_OK;
}

int tgi_merge_get_stats(tgi_ctx* c, tgi_merge_stats* out) {
  if (!c || !out) return TGI_E_ARG;
  std::lock_guard<std::mutex> g(c->fr_mu);
  *out = c->mstats;
  return TGI_OK;
}

int tgi_frontier_global_export(tgi_ctx* c, uint8_t* keys32, uint64_t cap, uint64_t* n) {
  if (!c || !n) return TGI_E_ARG;
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->fr_mu);
  if (!c->comm) { set_err(c, "tgi_frontier_global_export needs tgi_comm_init first"); return TGI_E_STATE; }
  NcclApi& N = *c->nccl;
  const int G = c->nranks;
  cudaStream_t st = c->slots[0].stream;
  uint64_t* hb = c->m_host.as<uint64_t>();
  if (c->fr_event_valid) CK(cudaStreamWaitEvent(st, c->fr_event, 0));
  NK(N.AllGather(c->owned.count, c->m_all.p, 1, ncclUint64, c->comm, st));
  CK(cudaMemcpyAsync(hb, c->m_all.p, (size_t)G * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  std::vector<uint64_t> off(G + 1, 0);
  for (int p = 0; p < G; p++) off[p + 1] = off[p] + hb[p];
  const uint64_t T = off[G];
  DevBuf dk, dp;
  CK(dk.ensure(T * 32));
  CK(dp.ensure(T * 8));
  for (int p = 0; p < G; p++) {
    const uint64_t cnt = off[p + 1] - off[p];
    if (!cnt) continue;
    NK(N.Broadcast(c->owned.pool, dk.as<uint8_t>() + 32 * off[p], cnt * 32, ncclUint8, p, c->comm, st));
    NK(N.Broadcast(c->owned.payload, dp.as<uint64_t>() + off[p], cnt, ncclUint64, p, c->comm, st));
  }
  std::vector<uint8_t> hk(T * 32);
  std::vector<uint64_t> hp(T);
  if (T) {
    CK(cudaMemcpyAsync(hk.data(), dk.p, T * 32, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(hp.data(), dp.p, T * 8, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  std::vector<uint64_t> idx(T);
  for (uint64_t i = 0; i < T; i++) idx[i] = i;
  std::sort(idx.begin(), idx.end(), [&](uint64_t a, uint64_t b) { return hp[a] < hp[b]; });
  const uint64_t m = T < cap ? T : cap;
  if (keys32)
    for (uint64_t i = 0; i < m; i++) memcpy(keys32 + 32 * i, hk.data() + 32 * idx[i], 32);
  *n = T;
  return TGI_OK;
}

int tgi_filter_usernames(tgi_ctx* c, const uint8_t* names, const uint32_t* off, uint64_t n, uint8_t* reason) {
  if (!c || !off || !reason) return TGI_E_ARG;
  cudaSetDevice(c->device);
  if (!n) return TGI_OK;
  DevBuf dn, doff, dr;
  uint32_t total = off[n];
  CK(dn.ensure(total));
  CK(doff.ensure((n + 1) * 4));
  CK(dr.ensure(n));
  CK(cudaMemset(dn.p, 0, total + PAD));
  if (total) CK(cudaMemcpy(dn.p, names, total, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(doff.p, off, (n + 1) * 4, cudaMemcpyHostToDevice));
  unsigned g = (unsigned)((n * 32 + 255) / 256);
  filter_usernames_kernel<<<g, 256>>>(dn.as<uint8_t>(), doff.as<uint32_t>(), n, dr.as<uint8_t>());
  CK(cudaGetLastError());
  CK(cudaMemcpy(reason, dr.p, n, cudaMemcpyDeviceToHost));
  dn.release();
  doff.release();
  dr.release();
  return TGI_OK;
}

}  // extern "C"
