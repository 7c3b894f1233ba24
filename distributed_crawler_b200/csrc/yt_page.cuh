// yt_page.cuh — a page-sized YouTube batch in ONE cooperative launch (the reference asks the Data API for 50 videos per
// page, crawler/youtube/youtube_crawler.go:353-427).  Same construction as tg_page.cuh: the bulk pipeline's passes as phases
// of one grid, one WARP per record (yt_size_record / yt_emit_record: the warp sizer and the warp writer of the YouTube
// walk), grid-wide frontier phases, the result arrays contiguous for one copy out.
//
//   P0  zero the scalars / the batch hash table
//   P1  per record: unique URLs, channel-id links, status            (yt_parse_body)
//   P2  per record: line length.  Frontier probe
//   P3  line / link offsets (two single-CTA scans).  Frontier count
//   P4  offsets of the new keys, then the capacity check (nothing committed yet)
//   P5  per record: the line.  Frontier append
//   P6  link compaction into the result block, frontier commit
#pragma once
#include "tg_page.cuh"

namespace tgi {

struct YtPageArgs {
  YtBatchDev b;
  CfgDev cfg;
  uint32_t run_flags;
  YtOut yo;
  uint64_t* scalars;
  uint64_t* line_off;    // [n+1] result block
  uint64_t* link_off;    // [n+1] scratch
  uint32_t* link_off32;  // [n+1] result block
  uint8_t* var;          // result block: links, then the JSONL at the next 256-byte boundary
  uint64_t var_cap;
  uint64_t max_out;      // as PageArgs.max_out
  FrontierDev fr;
  FrontierBatch fb;
  ExclusionDev excl;
  uint64_t bslots;
  uint64_t* new_off;
};

__global__ void __launch_bounds__(CTA_THREADS, 2) yt_page_kernel(const __grid_constant__ YtPageArgs a) {
  __shared__ YtScratch scs[WARPS_PER_CTA];
  cg::grid_group grid = cg::this_grid();
  const uint64_t n = a.b.n;
  const bool want_json = a.run_flags & TGI_RUN_JSONL, want_links = a.run_flags & TGI_RUN_LINKS, want_fr = a.run_flags & TGI_RUN_FRONTIER;
  const unsigned last = gridDim.x - 1;
  const int wid = threadIdx.x >> 5;
  const uint64_t w0 = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  const uint64_t t0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (uint64_t)gridDim.x * blockDim.x;
  int phase = 0;
  auto stamp = [&] {  // phase clock, as in tg_page_kernel
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      a.scalars[PAGE_TRACE_AT + phase] = t;
    }
    phase++;
  };
  stamp();

  // P0
  if (blockIdx.x == 0 && threadIdx.x < SC_COUNT) a.scalars[threadIdx.x] = 0;
  if (blockIdx.x == 0 && threadIdx.x < 3) a.scalars[PAGE_TRACE_AT + PAGE_PHASES + 1 + threadIdx.x] = 0;
  if (want_fr) grid_zero16(a.fb.btable, a.bslots * 8);
  grid.sync();
  stamp();

  // P1
  yt_parse_body(a.b, a.cfg, a.run_flags, a.yo);
  grid.sync();
  stamp();
  if (*(volatile int*)a.yo.err & (ERR_ARENA_OVERFLOW | ERR_TOO_MANY_LINKS)) return;  // the host reruns the bulk pipeline

  // P2
  if (want_json)
    for (uint64_t r = w0; r < n; r += nwarps)
      if (a.yo.status[r] == TGI_ST_EMITTED) yt_size_record(a.b, a.cfg, a.yo, r, &scs[wid]);
  if (want_fr) frontier_probe_body(n, a.yo.link_start, a.yo.link_count, a.yo.arena, a.run_flags, a.fr, a.fb, a.excl, t0, nt);
  grid.sync();
  stamp();

  // P3
  if (want_json && blockIdx.x == 0) cta_scan_u32(a.yo.linelen, n, a.line_off, a.scalars + SC_LINE_TOTAL);
  if (want_links && blockIdx.x == 1 % gridDim.x) cta_scan_u32(a.yo.link_count, n, a.link_off, a.scalars + SC_LINK_TOTAL);
  if (want_fr) frontier_count_body(n, a.yo.link_start, a.yo.link_count, a.fb, t0, nt);
  grid.sync();
  stamp();

  // P4
  if (want_fr) {
    if (blockIdx.x == last) cta_scan_u32(a.fb.rec_new, n, a.new_off, a.scalars + SC_NEW);
    grid.sync();
  }
  stamp();
  const uint64_t links_bytes = want_links ? (a.scalars[SC_LINK_TOTAL] * sizeof(tgi_link) + 255) & ~255ull : 0;
  const uint64_t line_total = want_json ? a.scalars[SC_LINE_TOTAL] : 0;
  if (links_bytes + line_total > a.var_cap || (a.max_out && line_total > a.max_out)) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(a.yo.err, ERR_PAGE_OVERFLOW);
    return;
  }

  // P5
  if (want_json) {
    uint8_t* out = a.var + links_bytes;
    for (uint64_t r = w0; r < n; r += nwarps)
      if (a.yo.status[r] == TGI_ST_EMITTED) yt_emit_record(a.b, a.cfg, a.yo, a.line_off, out, a.yo.err, r, &scs[wid]);
  }
  if (want_fr) {
    frontier_append_body(n, a.yo.link_start, a.yo.link_count, a.yo.arena, a.fr, a.fb, a.new_off, a.yo.err, nullptr, t0, nt);
    grid.sync();  // the NEW flags of the links
  }
  stamp();

  // P6
  if (want_links) links_compact_body(n, a.yo.link_start, a.yo.link_count, a.link_off, a.yo.arena, (tgi_link*)a.var, a.link_off32);
  if (want_fr && blockIdx.x == last && threadIdx.x == 0) frontier_commit_body(a.fr, a.new_off, n, a.scalars + SC_NEW, a.yo.err);
  stamp();
}

}  // namespace tgi
