// tg_page.cuh — a page-sized Telegram batch in ONE cooperative launch.
//
// The reference hands ParseMessage one page at a time (crawl/runner.go:1110: 100 messages).  At that size the seven-pass
// pipeline of run_tg is all latency: 19 launches, 22 copies / memsets and three host synchronisations.  The page kernel
// runs the whole batch as phases of one grid, separated by grid-wide barriers instead of kernel boundaries:
//
//   P0  zero the scalars / the batch hash table / the channel blob, channel sizes
//   P1  per record: entity byte ranges, status + links.  One CTA: channel offsets
//   P2  per record: line length.  Channel blob.  Frontier probe
//   P3  two CTAs: line offsets, link offsets.  Frontier count
//   P4  one CTA: offsets of the new keys              (capacity check before anything is committed)
//   P5  per record: the line (fixed part, escaped strings, maps).  Frontier append
//   P6  link compaction into the result block, frontier commit
//
// "Per record" is one WARP per record (emit_tg_fixed / emit_tg_escapes / size_tg_record of tg_walk.cuh), not the
// lane-per-record kernels of the bulk pipeline: those are built for throughput (32 records in lockstep through ~10 K
// dependent instructions per lane: 70 us for the first line to appear, however small the batch — measured, profiles/
// README.md); the warp walkers finish a record in a few microseconds, which is what a page waits for.
//
// No host round trip in between: the output goes to a block sized by the host's estimate, and a batch that does not fit
// (or overflows the link arena) sets ERR_PAGE_OVERFLOW / ERR_ARENA_OVERFLOW BEFORE the frontier is touched; the host then runs the ordinary pipeline
// on the same resident input.  The result arrays (scalars | status | line_off | link_off | links | JSONL) are contiguous
// in device memory, so the host reads them with one copy.
#pragma once
#include <cooperative_groups.h>
#include "kernels.cuh"

namespace tgi {
namespace cg = cooperative_groups;

constexpr int PAGE_PHASES = 7;  // scalars[PAGE_TRACE_AT .. + 8): start, after each barrier, end

struct PageArgs {
  TgBatchDev b;
  CfgDev cfg;
  uint32_t run_flags;
  ParseOut po;
  EmitIn ei;               // ei.out is set by the kernel (behind the compacted links)
  // channel job
  ChanDerived* chan_derived;
  uint32_t* chan_len;
  uint64_t* chan_off;
  uint8_t* chan_blob;
  uint64_t chan_blob_cap;
  // offsets and the result block
  uint64_t* scalars;       // SC_* (first bytes of the result block)
  uint64_t* line_off;      // [n+1] result block
  uint64_t* link_off;      // [n+1] scratch
  uint32_t* link_off32;    // [n+1] result block
  uint8_t* var;            // result block: links (36 bytes each), then the JSONL at the next 256-byte boundary
  uint64_t var_cap;
  uint64_t max_out;        // tgi_config.max_out_bytes (0 = no limit): a page over it falls back BEFORE the frontier is touched
  // frontier
  FrontierDev fr;
  FrontierBatch fb;
  ExclusionDev excl;
  uint64_t bslots;
  uint64_t* new_off;       // [n+1]
};

// exclusive scan u32[n] -> u64[n+1] by ONE CTA of CTA_THREADS threads (all of them call it)
DEVI void cta_scan_u32(const uint32_t* in, uint64_t n, uint64_t* out, uint64_t* total) {
  constexpr int ITEMS = 8;
  __shared__ uint64_t sm[WARPS_PER_CTA];
  const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint64_t carry = 0;
  for (uint64_t base = 0; base < n; base += (uint64_t)CTA_THREADS * ITEMS) {
    const uint64_t i0 = base + (uint64_t)threadIdx.x * ITEMS;
    uint32_t v[ITEMS];
    uint64_t s = 0;
#pragma unroll
    for (int k = 0; k < ITEMS; k++) {
      v[k] = i0 + k < n ? in[i0 + k] : 0u;
      s += v[k];
    }
    uint64_t x = s;
    for (int d = 1; d < 32; d <<= 1) {
      const uint64_t t = __shfl_up_sync(FULL, x, d);
      if (l >= d) x += t;
    }
    if (l == 31) sm[w] = x;
    __syncthreads();
    uint64_t woff = 0, chunk = 0;
#pragma unroll
    for (int k = 0; k < WARPS_PER_CTA; k++) {
      if (k < w) woff += sm[k];
      chunk += sm[k];
    }
    uint64_t excl = carry + woff + x - s;
#pragma unroll
    for (int k = 0; k < ITEMS; k++) {
      if (i0 + k < n) out[i0 + k] = excl;
      excl += v[k];
    }
    carry += chunk;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[n] = carry;
    *total = carry;
  }
}

DEVI void grid_zero16(void* p, uint64_t bytes) {  // p 16-byte aligned, bytes rounded up to 16 by the caller's allocation
  uint4* q = (uint4*)p;
  const uint64_t n16 = (bytes + 15) / 16;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x) q[i] = make_uint4(0, 0, 0, 0);
}

__global__ void __launch_bounds__(CTA_THREADS, 2) tg_page_kernel(const __grid_constant__ PageArgs a) {
  __shared__ WarpScratch wss[WARPS_PER_CTA];
  __shared__ MapScratch mss[WARPS_PER_CTA];
  __shared__ CtaShared cs;
  cg::grid_group grid = cg::this_grid();
  const uint64_t n = a.b.n;
  const bool want_json = a.run_flags & TGI_RUN_JSONL, want_links = a.run_flags & TGI_RUN_LINKS, want_fr = a.run_flags & TGI_RUN_FRONTIER;
  const unsigned last = gridDim.x - 1;
  const int wid = threadIdx.x >> 5, l = lane_id();
  const uint64_t w0 = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  // phase clock: block 0 stamps %globaltimer (ns) behind the scalars after every barrier (TGI_PAGE_TRACE prints the deltas)
  int phase = 0;
  auto stamp = [&] {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      a.scalars[PAGE_TRACE_AT + phase] = t;
    }
    phase++;
  };
  stamp();
  // slowest record of the per-record phases: (cycles << 32 | record), atomicMax'd behind the phase clock
  auto slowest = [&](int k, long long t_begin, uint64_t r) {
    if (l == 0) atomicMax((unsigned long long*)&a.scalars[PAGE_TRACE_AT + PAGE_PHASES + 1 + k],
                          ((unsigned long long)(clock64() - t_begin) << 32) | (unsigned long long)(r & 0xffffffffu));
  };
  if (blockIdx.x == 0 && threadIdx.x < 3) a.scalars[PAGE_TRACE_AT + PAGE_PHASES + 1 + threadIdx.x] = 0;

  // P0
  if (blockIdx.x == 0 && threadIdx.x < SC_COUNT) a.scalars[threadIdx.x] = 0;
  if (want_fr) grid_zero16(a.fb.btable, a.bslots * 8);
  if (want_json) {
    grid_zero16(a.chan_blob, a.chan_blob_cap);  // segment padding must read as zero
    tg_chan_size_body(a.b, a.chan_derived, a.chan_len);
    for (int i = threadIdx.x; i < kTgNEnt; i += blockDim.x) cs.ents[i] = kTgPieces[i];
    for (int i = threadIdx.x; i < kTgNWords; i += blockDim.x) {
      cs.tmpl[i] = ((const uint32_t*)kTgTemplate)[i];
      cs.wmeta[i] = kTgWordMeta[i];
    }
  }
  grid.sync();
  stamp();

  // P1: one warp per record
  for (uint64_t r = w0; r < n; r += nwarps) {
    const long long tb = clock64();
    const TgRecView v = load_rec_view(a.b, r);
    if (v.e1 != v.e0) {
      warp_map_entities(v, a.b.ents, a.po.ent_range);
      __syncwarp();  // lane 0's ranges, read back by every lane
      parse_one_record<true>(a.b, a.cfg, a.po, r, v);
    } else {
      parse_one_record<false>(a.b, a.cfg, a.po, r, v);
    }
    slowest(0, tb, r);
  }
  if (want_json && blockIdx.x == last) {
    cta_scan_u32(a.chan_len, a.b.n_chans, a.chan_off, a.scalars + SC_CHAN_TOTAL);
    __syncthreads();
    for (uint32_t c = threadIdx.x; c < a.b.n_chans; c += blockDim.x) a.chan_derived[c].off = a.chan_off[c];
  }
  grid.sync();
  stamp();
  if (*(volatile int*)a.po.err & (ERR_ARENA_OVERFLOW | ERR_TOO_MANY_LINKS)) return;  // the host reruns the ordinary pipeline
  if (want_json && a.scalars[SC_CHAN_TOTAL] > a.chan_blob_cap) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(a.po.err, ERR_PAGE_OVERFLOW);
    return;
  }

  // P2
  if (want_json) {
    uint64_t var_sum = 0;
    for (uint64_t r = w0; r < n; r += nwarps) {
      if (a.po.status[r] != TGI_ST_EMITTED) continue;
      const long long tb = clock64();
      TgWalkArgs wa;
      wa.b = &a.b;
      wa.cfg = &a.cfg;
      wa.r = r;
      wa.v = load_rec_view(a.b, r);
      wa.links = a.po.arena + a.po.link_start[r];
      wa.n_links = a.po.link_count[r];
      uint32_t xl[8];
      const uint32_t llen = size_tg_record(wa, xl);
      uint32_t mine = 0;
#pragma unroll
      for (int j = 0; j < 8; j++)
        if (l == j) mine = xl[j];
      if (l < 8) a.po.xlen[r * 8 + l] = mine;
      if (llen) var_sum += warp_sum(l < XL_COUNT ? mine : 0u);
      if (l == 0) {
        if (llen == 0) a.po.status[r] = TGI_ST_NOLINE;
        a.po.linelen[r] = llen;
      }
      slowest(1, tb, r);
    }
    if (l == 0 && var_sum) atomicAdd(a.po.var_total, (unsigned long long)var_sum);
    tg_chan_emit_body(a.b, a.chan_derived, a.chan_off, a.chan_blob, false);
  }
  const uint64_t t0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (uint64_t)gridDim.x * blockDim.x;
  if (want_fr) frontier_probe_body(n, a.po.link_start, a.po.link_count, a.po.arena, a.run_flags, a.fr, a.fb, a.excl, t0, nt);
  grid.sync();
  stamp();

  // P3
  if (want_json && blockIdx.x == 0) cta_scan_u32(a.po.linelen, n, a.line_off, a.scalars + SC_LINE_TOTAL);
  if (want_links && blockIdx.x == 1 % gridDim.x) cta_scan_u32(a.po.link_count, n, a.link_off, a.scalars + SC_LINK_TOTAL);
  if (want_fr) frontier_count_body(n, a.po.link_start, a.po.link_count, a.fb, t0, nt);
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
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(a.po.err, ERR_PAGE_OVERFLOW);
    return;
  }

  // P5
  if (want_json) {
    uint8_t* out = a.var + links_bytes;
    for (uint64_t r = w0; r < n; r += nwarps) {
      if (a.po.status[r] != TGI_ST_EMITTED) continue;
      const long long tb = clock64();
      TgWalkArgs wa;
      wa.b = &a.b;
      wa.cfg = &a.cfg;
      wa.r = r;
      wa.v = load_rec_view(a.b, r);
      wa.links = nullptr;
      wa.n_links = 0;
      const uint64_t lo = a.line_off[r];
      uint8_t* line = out + lo;
      const uint32_t* xlen_g = a.po.xlen + r * 8;
      uint32_t* xp = a.ei.xpos + r * 8;
      emit_tg_fixed(line, &wss[wid], &cs, wa, (uint32_t)(a.line_off[r + 1] - lo), xlen_g, xp, a.po.err);
      __syncwarp();  // the offsets of the variable pieces (xpos), written by their owning lanes
      emit_tg_escapes<ESC_ALL>(line, wa, xlen_g, xp, 0xffffffffu);  // every string: no lane emitter ran
      const uint32_t c0 = a.b.comment_off[r], c1 = a.b.comment_off[r + 1];
      if (a.b.recs[r].flags & TGI_RF_COMMENTS_NIL) gcopy_g(line + xp[XL_COMMENTS], (const uint8_t*)kNullLit, 4);
      else if (c1 == c0) gput2(line + xp[XL_COMMENTS], '[', ']');
      else emit_tg_comments(line + xp[XL_COMMENTS], &mss[wid], a.b, c0, c1);
      emit_reaction_map(line + xp[XL_REACTIONS], &mss[wid], a.b.reacts, a.b.react_off[r], a.b.react_off[r + 1], a.b.aux);
      const uint32_t nl = a.po.link_count[r];
      if (nl) emit_tg_outlinks(line + xp[XL_OUTLINKS], a.po.arena + a.po.link_start[r], nl);
      __syncwarp();
      slowest(2, tb, r);
    }
  }
  if (want_fr) {
    frontier_append_body(n, a.po.link_start, a.po.link_count, a.po.arena, a.fr, a.fb, a.new_off, a.po.err, nullptr, t0, nt);
    grid.sync();  // the NEW flags of the links
  }
  stamp();

  // P6
  if (want_links) links_compact_body(n, a.po.link_start, a.po.link_count, a.link_off, a.po.arena, (tgi_link*)a.var, a.link_off32);
  if (want_fr && blockIdx.x == last && threadIdx.x == 0) frontier_commit_body(a.fr, a.new_off, n, a.scalars + SC_NEW, a.po.err);
  stamp();  // block 0's own end of P6
}

}  // namespace tgi
