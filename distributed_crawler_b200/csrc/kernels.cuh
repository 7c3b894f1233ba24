// kernels.cuh — __global__ kernels of the ingest engine (sm_100a).  See DESIGN.md §4 for the data layout and the
// roofline bookkeeping.  All of it is integer/byte work:
//   tg_chan_size / tg_chan_emit            per-channel constant strings (once per batch, tiny)
//   tg_parse / tg_ent_map / tg_parse_ent   status + link extraction, one warp per record (split by code footprint)
//   tg_size_lane                           JSONL line length, one LANE per record (+ the warp for the message text)
//   scan_*                                 exclusive scan u32 -> u64 offsets
//   tg_emit_lane                           the line, one LANE per record (tg_lane.cuh)
//   tg_emit_esc / tg_emit_maps             what the lane emitter leaves: strings that need escaping, comment lists ...
//   frontier_*                             exact open-addressed hash set over 32-byte keys
//   yt_* / gm_*                            YouTube (config 4) and generic-message (a12) lines
//   join_*                                 message-status join (SURVEY 8f)
#pragma once
#include "tg_walk.cuh"
#include "tg_lane.cuh"
#include "yt_walk.cuh"
#include "gm_walk.cuh"
#include "yt_lane.cuh"

namespace tgi {

constexpr int WARPS_PER_CTA = 8;
constexpr int CTA_THREADS = WARPS_PER_CTA * 32;
// Resident CTAs per SM the compiler budgets registers for.  Swept on the config-2 step (tools/variants.sh, profiles/README.md):
// 4 (64 registers) 41.2 ms, 5: 38.6, 6: 38.0, 7 (32 registers): 37.7, 8: 38.2 — the spills barely grow (most of the "spill"
// is local arrays), the extra warps per scheduler are worth more.
#ifndef LB_PARSE
#define LB_PARSE 7
#endif
#ifndef LB_SIZE
#define LB_SIZE 7
#endif
#ifndef LB_ESC
#define LB_ESC 7
#endif
#ifndef LB_MAPS
#define LB_MAPS 7
#endif
#ifndef LB_YT
#define LB_YT 6  // 3: 22.8 ms per 2 M config-4 records, 4: 20.4, 5: 19.2, 6: 18.7, 8: 18.6 (tools/variants_yt.sh)
#endif

// ---- batch validation: every offset the kernels will follow stays inside its array ------------------------------
// A malformed batch that crossed the C ABI must come back as TGI_E_ARG, not as an illegal address (or as foreign
// bytes in the JSONL).  One rule per element, shared by the host (small batches, host pointers in the TgBatchDev) and
// tg_validate_kernel (big ones); the result is a mask of the broken checks.
struct TgBounds {
  uint64_t strs_len, n_ents, n_reacts, n_comments, aux_len, chan_strs_len;
};
#define HDI __host__ __device__ __forceinline__
HDI int tg_check_record(const TgBatchDev& b, const TgBounds& lim, uint64_t i) {
  const tgi_tg_rec rc = b.recs[i];
  const uint64_t end = rc.str_off + (uint64_t)rc.text_len + rc.alt_len + rc.media_len + rc.handle_len;
  int e = 0;
  if (end > lim.strs_len || end < rc.str_off) e |= 1;
  if (rc.chan_idx >= b.n_chans || rc.content_type >= TGI_CT__COUNT) e |= 2;
  if (b.ent_off[i] > b.ent_off[i + 1] || b.ent_off[i + 1] > lim.n_ents) e |= 4;
  if (b.react_off[i] > b.react_off[i + 1] || b.react_off[i + 1] > lim.n_reacts) e |= 8;
  if (b.comment_off[i] > b.comment_off[i + 1] || b.comment_off[i + 1] > lim.n_comments) e |= 16;
  return e;
}
HDI int tg_check_entity(const TgBatchDev& b, const TgBounds& lim, uint64_t i) {
  const tgi_entity en = b.ents[i];
  return en.type == TGI_ENT_TEXT_URL && (uint64_t)en.url_off + en.url_len > lim.aux_len ? 32 : 0;
}
HDI int tg_check_reaction(const TgBatchDev& b, const TgBounds& lim, uint64_t i) {
  const tgi_reaction rc = b.reacts[i];
  return (uint64_t)rc.emoji_off + rc.emoji_len > lim.aux_len ? 64 : 0;
}
HDI int tg_check_comment(const TgBatchDev& b, const TgBounds& lim, uint64_t i) {
  const tgi_comment cm = b.comments[i];
  int e = 0;
  if ((uint64_t)cm.text_off + cm.text_len > lim.aux_len || (uint64_t)cm.handle_off + cm.handle_len > lim.aux_len) e |= 128;
  if ((cm.flags & 1) && (uint64_t)cm.react_start + cm.react_count > lim.n_reacts) e |= 256;
  return e;
}
HDI int tg_check_channel(const TgBatchDev& b, const TgBounds& lim, uint64_t i) {
  const tgi_tg_chan ch = b.chans[i];
  return (uint64_t)ch.str_off + ch.title_len + ch.name_len + ch.user_len > lim.chan_strs_len ? 512 : 0;
}
// one thread per index of the longest array
__global__ void tg_validate_kernel(TgBatchDev b, TgBounds lim, uint64_t count, int* bad) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  int e = 0;
  if (i < b.n) e |= tg_check_record(b, lim, i);
  if (i < lim.n_ents) e |= tg_check_entity(b, lim, i);
  if (i < lim.n_reacts) e |= tg_check_reaction(b, lim, i);
  if (i < lim.n_comments) e |= tg_check_comment(b, lim, i);
  if (i < b.n_chans) e |= tg_check_channel(b, lim, i);
  if (e) atomicOr(bad, e);
}

// ---- channel job -----------------------------------------------------------------------------------
// Every kernel of the Telegram pipeline is a *_body (grid-stride over blockIdx / gridDim) plus a one-line __global__
// wrapper: the page kernel (tg_page.cuh) runs the same bodies as phases of ONE cooperative launch.
DEVI void tg_chan_size_body(const TgBatchDev& b, ChanDerived* cd, uint32_t* len) {
  const int wid = threadIdx.x >> 5;
  for (uint32_t c = blockIdx.x * WARPS_PER_CTA + wid; c < b.n_chans; c += gridDim.x * WARPS_PER_CTA) {
    ChanDerived d = size_tg_chan(b, c);
    if (lane_id() == 0) {
      cd[c] = d;
      len[c] = pad16(d.user_len) + pad16(d.name_len) + pad16(d.title_len) + pad16(d.cdata_len);
    }
  }
}
__global__ void __launch_bounds__(CTA_THREADS) tg_chan_size_kernel(TgBatchDev b, ChanDerived* cd, uint32_t* len) { tg_chan_size_body(b, cd, len); }

DEVI void tg_chan_emit_body(const TgBatchDev& b, ChanDerived* cd, const uint64_t* off, uint8_t* blob, bool write_off = true) {
  __shared__ WarpScratch wss[WARPS_PER_CTA];
  const int wid = threadIdx.x >> 5;
  for (uint32_t c = blockIdx.x * WARPS_PER_CTA + wid; c < b.n_chans; c += gridDim.x * WARPS_PER_CTA) {
    if (write_off && lane_id() == 0) cd[c].off = off[c];
    emit_tg_chan(blob + off[c], &wss[wid], b, c);
    __syncwarp();
  }
}
__global__ void __launch_bounds__(CTA_THREADS) tg_chan_emit_kernel(TgBatchDev b, ChanDerived* cd, const uint64_t* off, uint8_t* blob) {
  tg_chan_emit_body(b, cd, off, blob);
}

// ---- parse: status + links + line length ---------------------------------------------------------
struct ParseOut {
  uint8_t* status;       // [n]
  uint32_t* linelen;     // [n]
  uint32_t* link_start;  // [n] arena index of the record's first link
  uint32_t* link_count;  // [n]
  uint32_t* xlen;        // [n][8] emitted lengths of the variable pieces (XL_*)
  unsigned long long* var_total;  // sum of the variable pieces' lengths (statistics)
  tgi_link* arena;
  uint32_t arena_cap;
  uint32_t* cursor;      // arena allocation cursor (keeps counting past arena_cap)
  int2* ent_range;       // [n_ents] byte range of every mention / url entity (tg_ent_map_kernel)
  int* err;
};

DEVI TgRecView load_rec_view(const TgBatchDev& b, uint64_t r) {
  TgRecView v;
  const tgi_tg_rec* rec = &b.recs[r];
  v.rec = rec;
  v.text = b.strs + rec->str_off;
  v.text_len = rec->text_len;
  v.alt = v.text + v.text_len;
  v.alt_len = rec->alt_len;
  v.media = v.alt + v.alt_len;
  v.media_len = rec->media_len;
  v.handle = v.media + v.media_len;
  v.handle_len = rec->handle_len;
  v.ct = rec->content_type;
  v.flags = rec->flags;
  v.e0 = b.ent_off[r];
  v.e1 = b.ent_off[r + 1];
  return v;
}

// One record.  ENTITIES == false: the record has no entities, so the whole UTF-16 offset machinery
// (warp_utf16_to_bytes, the exact UTF-8 path) is compiled out.
template <bool ENTITIES>
DEVI void parse_one_record(const TgBatchDev& b, const CfgDev& cfg, const ParseOut& o, uint64_t r, TgRecView v) {
  const int l = lane_id();
  uint32_t status = TGI_ST_EMITTED, nlinks = 0, lstart = 0;
  if ((cfg.flags & TGI_CFG_HAS_MIN_POST_DATE) && (int64_t)v.rec->date < cfg.min_post_date) {
    status = TGI_ST_SKIPPED;  // tdutils.go:419-421
  } else if (v.flags & TGI_RF_PANIC) {
    status = TGI_ST_FAILED;
  } else {
    if (!ENTITIES) v.e1 = v.e0;
    uint32_t ub = warp_link_upper_bound(v, b.ents);
    if (ub >= (1u << 20)) {  // seq packing of the frontier needs ordinal < 2^20 (SEQ_ORD_BITS)
      if (l == 0) atomicOr(o.err, ERR_TOO_MANY_LINKS);
      ub = 0;
    }
    if (ub) {
      if (l == 0) lstart = atomicAdd(o.cursor, ub);
      lstart = __shfl_sync(FULL, lstart, 0);
      if (lstart + ub > o.arena_cap || lstart + ub < lstart) {
        if (l == 0) atomicOr(o.err, ERR_ARENA_OVERFLOW);
      } else {
        const tgi_tg_chan* ch = &b.chans[v.rec->chan_idx];
        LinkSink ls;
        ls.out = o.arena + lstart;
        ls.cap = ub;
        ls.count = 0;
        ls.name_bytes = 0;
        ls.self = b.chan_strs + ch->str_off + ch->title_len;
        ls.self_len = ch->name_len;
        bool ok = warp_extract_links(v, b.ents, b.aux, o.ent_range, ls);
        nlinks = ls.count;
        if (!ok) {
          status = TGI_ST_FAILED;
          nlinks = 0;
        }
      }
    }
  }
  if (l == 0) {
    o.status[r] = (uint8_t)status;
    o.linelen[r] = 0;
    o.link_start[r] = lstart;
    o.link_count[r] = nlinks;
  }
}

// The parse step is split by instruction footprint (the B200 instruction caches are 6 KB L0 / 32 KB L1.5):
// tg_parse_kernel = status + links of the records WITHOUT entities (three quarters of the corpus; small code),
// tg_ent_map_kernel = UTF-16 entity offsets -> byte ranges, tg_parse_ent_kernel = links of the records with
// entities (lanes pick them out of groups of 32), tg_size_lane_kernel = line lengths.  Fusing them was measured twice:
// one parse kernel (2 560 SASS instructions) showed 3.5 stall_no_instruction cycles per issue in round 1; the round-2
// attempt to fold parse + size into ONE pass over the text (8.7 G instead of 9.2 G warp instructions per 10 M
// messages) ran at 18.6 no_instruction stall cycles per issue and took 27.2 ms instead of 14.3 (profiles/README.md).
DEVI void tg_parse_body(const TgBatchDev& b, const CfgDev& cfg, uint32_t run_flags, const ParseOut& o) {
  int wid = threadIdx.x >> 5;
  uint64_t nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t r = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; r < b.n; r += nwarps) {
    // The chain header -> string offset -> text is two DRAM round trips per record and this kernel has little else to
    // do (long_scoreboard 9 cycles per issue): read the NEXT record's header now, touch its text at the bottom of
    // the loop, when that load has long completed.
    const uint64_t rn = r + nwarps;
    unsigned long long nx_off = 0;
    uint32_t nx_len = 0;
    if (rn < b.n) {
      asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(nx_off) : "l"(&b.recs[rn].str_off));
      asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(nx_len) : "l"(&b.recs[rn].text_len));
    }
    if (b.ent_off[r + 1] == b.ent_off[r])  // the others: tg_parse_ent_kernel
      parse_one_record<false>(b, cfg, o, r, load_rec_view(b, r));
    if (rn < b.n) {
      const uint32_t off = (uint32_t)lane_id() * 128u;
      if (off < nx_len + 127u && off < 2048u) asm volatile("prefetch.global.L1 [%0];" ::"l"(b.strs + nx_off + off));
    }
  }
}
__global__ void __launch_bounds__(CTA_THREADS, LB_PARSE) tg_parse_kernel(TgBatchDev b, CfgDev cfg, uint32_t run_flags, ParseOut o) { tg_parse_body(b, cfg, run_flags, o); }
DEVI void tg_ent_map_body(const TgBatchDev& b, const ParseOut& o) {
  const int wid = threadIdx.x >> 5, l = lane_id();
  const uint64_t ngroups = (b.n + 31) / 32, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t g = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; g < ngroups; g += nwarps) {
    const uint64_t rl = g * 32 + l;
    uint32_t todo = __ballot_sync(FULL, rl < b.n && b.ent_off[rl + 1] != b.ent_off[rl]);
    while (todo) {
      const uint64_t r = g * 32 + (uint32_t)(__ffs(todo) - 1);
      todo &= todo - 1;
      warp_map_entities(load_rec_view(b, r), b.ents, o.ent_range);
    }
  }
}
__global__ void __launch_bounds__(CTA_THREADS, LB_PARSE) tg_ent_map_kernel(TgBatchDev b, ParseOut o) { tg_ent_map_body(b, o); }
DEVI void tg_parse_ent_body(const TgBatchDev& b, const CfgDev& cfg, uint32_t run_flags, const ParseOut& o) {
  const int wid = threadIdx.x >> 5, l = lane_id();
  const uint64_t ngroups = (b.n + 31) / 32, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t g = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; g < ngroups; g += nwarps) {
    const uint64_t rl = g * 32 + l;
    uint32_t todo = __ballot_sync(FULL, rl < b.n && b.ent_off[rl + 1] != b.ent_off[rl]);
    while (todo) {
      const uint64_t r = g * 32 + (uint32_t)(__ffs(todo) - 1);
      todo &= todo - 1;
      parse_one_record<true>(b, cfg, o, r, load_rec_view(b, r));
    }
  }
}
__global__ void __launch_bounds__(CTA_THREADS, LB_PARSE) tg_parse_ent_kernel(TgBatchDev b, CfgDev cfg, uint32_t run_flags, ParseOut o) {
  tg_parse_ent_body(b, cfg, run_flags, o);
}

// The same sizes, 32 records per warp: every lane sizes the small pieces of its own record (numbers,
// handle / media strings, comments, reactions, outlinks); only the message text, the one long string,
// is measured by the whole warp, record after record; the rare complicated pieces (a comment list, a
// reactions map that is not "simple") go through the warp-wide routines as well.
DEVI void tg_size_lane_body(const TgBatchDev& b, const CfgDev& cfg, const ParseOut& o) {
  const int wid = threadIdx.x >> 5, l = lane_id();
  const uint64_t ngroups = (b.n + 31) / 32, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  uint64_t var_sum = 0;
  for (uint64_t g = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; g < ngroups; g += nwarps) {
    uint64_t r = g * 32 + l;
    bool active = r < b.n;
    if (!active) r = b.n - 1;
    active = active && o.status[r] == TGI_ST_EMITTED;
    if (!__any_sync(FULL, active)) continue;
    TgWalkArgs a;
    a.b = &b;
    a.cfg = &cfg;
    a.r = r;
    a.v = load_rec_view(b, r);
    a.links = o.arena + o.link_start[r];
    a.n_links = active ? o.link_count[r] : 0u;
    const tgi_tg_rec* rec = a.v.rec;
    const ChanDerived cd = b.chan_derived[rec->chan_idx];
    const TgDerived d = tg_derive(a, cd);
    uint32_t xl[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t tot = 0;
    bool warp_comments = false, warp_map = false;
    const uint32_t r0 = b.react_off[r], nr = b.react_off[r + 1] - r0;
    if (active && !(cfg.flags & CFGDEV_CLOCK_INVALID)) {
      uint32_t L[8] = {ndigits_i64(rec->id / 1048576), ndigits_i64(rec->chat_id), ndigits_i64(rec->view_count),
                       ndigits_i64(rec->share_count), ndigits_i64(d.ncomments), cfg.tz == 0 ? 22u : 27u, 0, 0};
      uint32_t chan[4] = {cd.user_len, cd.name_len, cd.title_len, cd.cdata_len};
      uint32_t cf[4] = {cfg.label_len, cfg.created_tg_len, cfg.created_yt_len, cfg.capture_len};
      tot = tg_size_fixed(L, chan, cf, d.has_user, d.album);
      tot += a.v.ct == TGI_CT_OTHER ? 0u : (uint32_t)kPostTypeLen[a.v.ct];
      if (a.v.ct == TGI_CT_OTHER) xl[XL_ALT] = thread_esc_len(a.v.alt, a.v.alt_len);
      if (d.has_media) xl[XL_MEDIA] = thread_esc_len(a.v.media, a.v.media_len);
      xl[XL_HANDLE] = thread_esc_len(a.v.handle, a.v.handle_len);
      if (d.comments_nil) xl[XL_COMMENTS] = 4;
      else if (d.c1 == d.c0) xl[XL_COMMENTS] = 2;
      else warp_comments = true;
      if (nr == 0) {
        xl[XL_REACTIONS] = 2;
        xl[XL_FLAGS] = XLF_SIMPLE_MAP;
      } else if (nr <= LANE_MAP_MAX) {  // size_reaction_map, one lane: "key":n , ... ; simple = short clean keys
        uint32_t sz = 2u, live = 0;
        bool simple = true;
        for (uint32_t j = 0; j < nr; j++) {
          const tgi_reaction rc = b.reacts[r0 + j];
          const uint8_t* kp = b.aux + rc.emoji_off;
          const uint32_t el = thread_esc_len(kp, rc.emoji_len);
          simple = simple && el == rc.emoji_len && rc.emoji_len >= 1 && rc.emoji_len <= 8;
          bool last = true;  // a later entry with the same key overwrites this one (Go map assignment)
          for (uint32_t i = j + 1; i < nr; i++) {
            const tgi_reaction ri = b.reacts[r0 + i];
            if (key_cmp(b.aux + ri.emoji_off, ri.emoji_len, kp, rc.emoji_len) == 0) last = false;
          }
          if (last) {
            sz += 3u + el + ndigits_i64(rc.count);
            live++;
          }
        }
        if (simple) {
          xl[XL_REACTIONS] = sz + (live - 1u);
          xl[XL_FLAGS] = XLF_SIMPLE_MAP;
        } else {
          warp_map = true;
        }
      } else {
        warp_map = true;
      }
      if (a.n_links) {
        uint32_t s = a.n_links - 1u;
        for (uint32_t k = 0; k < a.n_links; k++) s += a.links[k].len + 2u;
        xl[XL_OUTLINKS] = s;
      }
    }
    // the message text (or the other description sources), one record at a time, all lanes
    const bool sized = active && !(cfg.flags & CFGDEV_CLOCK_INVALID);
    uint32_t todo = __ballot_sync(FULL, sized && d.desc_len != 0);
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint8_t* p = (const uint8_t*)__shfl_sync(FULL, (unsigned long long)(uintptr_t)d.desc, src);
      const uint32_t n = __shfl_sync(FULL, d.desc_len, src);
      bool ex = false;
      const uint32_t e = warp_esc_len(p, n, &ex);
      if (l == src) {
        xl[XL_DESC] = e;
        if (ex) xl[XL_FLAGS] |= XLF_DESC_EXACT;
      }
    }
    todo = __ballot_sync(FULL, warp_comments);
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t e = size_tg_comments(b, __shfl_sync(FULL, d.c0, src), __shfl_sync(FULL, d.c1, src));
      if (l == src) xl[XL_COMMENTS] = e;
    }
    todo = __ballot_sync(FULL, warp_map);
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t q0 = __shfl_sync(FULL, r0, src), qn = __shfl_sync(FULL, nr, src);
      uint32_t simple = 0;
      const uint32_t e = size_reaction_map(b.reacts, q0, q0 + qn, b.aux, &simple);
      if (l == src) {
        xl[XL_REACTIONS] = e;
        xl[XL_FLAGS] = (xl[XL_FLAGS] & ~XLF_SIMPLE_MAP) | (simple ? XLF_SIMPLE_MAP : 0u);
      }
    }
    if (active) {
      uint32_t var = 0;
#pragma unroll
      for (int j = 0; j < XL_COUNT; j++) var += xl[j];
      const uint32_t llen = sized ? tot + var : 0u;
      *(uint4*)(o.xlen + r * 8) = make_uint4(xl[0], xl[1], xl[2], xl[3]);
      *(uint4*)(o.xlen + r * 8 + 4) = make_uint4(xl[4], xl[5], xl[6], xl[7]);
      if (llen == 0) o.status[r] = TGI_ST_NOLINE;
      o.linelen[r] = llen;
      if (llen) var_sum += var;
    }
  }
  for (int dd = 16; dd; dd >>= 1) var_sum += __shfl_down_sync(FULL, var_sum, dd);
  if (l == 0 && var_sum) atomicAdd(o.var_total, (unsigned long long)var_sum);
}
__global__ void __launch_bounds__(CTA_THREADS, LB_SIZE) tg_size_lane_kernel(TgBatchDev b, CfgDev cfg, ParseOut o) { tg_size_lane_body(b, cfg, o); }

// ---- emit --------------------------------------------------------------------------------------------------------
struct EmitIn {
  const uint8_t* status;
  const uint64_t* line_off;
  const uint32_t* link_start;
  const uint32_t* link_count;
  const uint32_t* xlen;  // [n][8] lengths of the variable pieces + flags
  uint32_t* xpos;        // [n][8] offsets of the variable pieces inside the line (written by the lane emitter)
  const tgi_link* arena;
  uint8_t* out;
  int* err;
  uint32_t lane_text_max;        // see emit_tg_escapes
  unsigned long long* counters;  // [0] JSONL bytes written by the main emit kernel, [1] source bytes it read from HBM
  // work lists written by the lane emitter: the records whose line it did not finish, by what is left
  uint32_t* list[3];             // WL_SPARSE, WL_DENSE, WL_MAPS: record indices
  uint32_t* list_count;          // [3]
};
enum { WL_SPARSE = 0, WL_DENSE = 1, WL_MAPS = 2 };
// warp-aggregated append of the lanes with `need` to a work list
DEVI void wl_append(uint32_t* list, uint32_t* count, bool need, uint32_t value) {
  const uint32_t m = __ballot_sync(FULL, need);
  if (!m) return;
  uint32_t base = 0;
  if (lane_id() == 0) base = atomicAdd(count, (uint32_t)__popc(m));
  base = __shfl_sync(FULL, base, 0);
  if (need) list[base + __popc(m & ((1u << lane_id()) - 1u))] = value;
}

// the same job, one LANE per record (tg_lane.cuh): 32 records per warp task
DEVI void tg_emit_lane_body(const TgBatchDev& b, const CfgDev& cfg, const EmitIn& in, LaneShared& sh) {
  static_assert(LANE_WARPS == WARPS_PER_CTA, "one field row block per warp");
  lane_shared_fill(sh);
  __syncthreads();
  const int wid = threadIdx.x >> 5, l = lane_id();
  const uint64_t ngroups = (b.n + 31) / 32, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  LaneStream s;
  ls_init(s, smem_addr(sh.stage[wid][l]));
  uint64_t bytes_out = 0, bytes_in = 0;
  for (uint64_t g = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; g < ngroups; g += nwarps) {
    uint64_t r = g * 32 + l;
    bool active = r < b.n;
    if (!active) r = b.n - 1;
    active = active && in.status[r] == TGI_ST_EMITTED;
    if (!__any_sync(FULL, active)) continue;
    uint32_t left = 0;
    emit_tg_lane(sh, sh.rows[wid][l], s, b, cfg, r, active, in.out, in.line_off, in.xlen + r * 8, in.xpos + r * 8,
                 in.arena + in.link_start[r], active ? in.link_count[r] : 0u, in.err, bytes_out, bytes_in, left);
    // hand the unfinished lines to the clean-up kernels as lists (they used to re-derive this from every record)
    bool sparse = false;
    if (active && (left & 1u)) {
      const tgi_tg_rec* rec = &b.recs[r];
      const uint32_t ct = rec->content_type;
      const bool text_desc = ct == TGI_CT_TEXT || ct == TGI_CT_VIDEO || ct == TGI_CT_PHOTO || ct == TGI_CT_ANIMATION;
      const uint32_t dlen = text_desc ? ((rec->flags & TGI_RF_HAS_TEXT) ? rec->text_len : 0u) : rec->alt_len;
      sparse = esc_desc_is_sparse(in.xlen[r * 8 + XL_DESC], dlen, in.xlen[r * 8 + XL_FLAGS]);
    }
    wl_append(in.list[WL_SPARSE], in.list_count + WL_SPARSE, active && sparse, (uint32_t)r);
    wl_append(in.list[WL_DENSE], in.list_count + WL_DENSE, active && (((left & 1u) && !sparse) || (left & 0xEu)), (uint32_t)r);
    wl_append(in.list[WL_MAPS], in.list_count + WL_MAPS, active && (left & 16u), (uint32_t)r);
  }
  for (int dd = 16; dd; dd >>= 1) {
    bytes_out += __shfl_down_sync(FULL, bytes_out, dd);
    bytes_in += __shfl_down_sync(FULL, bytes_in, dd);
  }
  if (l == 0) {
    atomicAdd(in.counters, (unsigned long long)bytes_out);
    atomicAdd(in.counters + 1, (unsigned long long)bytes_in);
  }
}
#ifndef LB_LANE
#define LB_LANE 3
#endif
__global__ void __launch_bounds__(CTA_THREADS, LB_LANE) tg_emit_lane_kernel(TgBatchDev b, CfgDev cfg, EmitIn in) {
  extern __shared__ __align__(128) uint8_t lane_smem[];
  tg_emit_lane_body(b, cfg, in, *(LaneShared*)lane_smem);
}

// The esc and maps kernels take what the lane emitter left, from its work lists: one warp per listed record.
// Two instantiations of the escape kernel by instruction footprint: ESC_SPARSE writes the descriptions whose only specials
// are a few line breaks (segment copies), ESC_DENSE the rest (per-byte placement, exact UTF-8 path, long clean strings,
// the other three strings).
template <int MODE>
DEVI void tg_emit_esc_body(const TgBatchDev& b, const EmitIn& in) {
  const int wid = threadIdx.x >> 5;
  const uint32_t* list = in.list[MODE == ESC_SPARSE ? WL_SPARSE : WL_DENSE];
  const uint32_t cnt = in.list_count[MODE == ESC_SPARSE ? WL_SPARSE : WL_DENSE];
  const uint32_t nwarps = gridDim.x * WARPS_PER_CTA;
  for (uint32_t i = blockIdx.x * WARPS_PER_CTA + wid; i < cnt; i += nwarps) {
    const uint64_t rr = list[i];
    TgWalkArgs a;
    a.b = &b;
    a.cfg = nullptr;
    a.r = rr;
    a.v = load_rec_view(b, rr);
    emit_tg_escapes<MODE>(in.out + in.line_off[rr], a, in.xlen + rr * 8, in.xpos + rr * 8, in.lane_text_max);
  }
}
template <int MODE>
__global__ void __launch_bounds__(CTA_THREADS, LB_ESC) tg_emit_esc_kernel(TgBatchDev b, EmitIn in) { tg_emit_esc_body<MODE>(b, in); }

DEVI void tg_emit_maps_body(const TgBatchDev& b, const EmitIn& in) {
  __shared__ MapScratch mss[WARPS_PER_CTA];
  const int wid = threadIdx.x >> 5;
  const uint32_t cnt = in.list_count[WL_MAPS], nwarps = gridDim.x * WARPS_PER_CTA;
  for (uint32_t i = blockIdx.x * WARPS_PER_CTA + wid; i < cnt; i += nwarps) {
    const uint64_t r = in.list[WL_MAPS][i];
    uint8_t* line = in.out + in.line_off[r];
    const uint32_t* xp = in.xpos + r * 8;
    // the lane emitter wrote the simple cases itself (tg_lane.cuh): nil / empty comment lists, simple maps, short outlink lists
    const bool comments_nil = (b.recs[r].flags & TGI_RF_COMMENTS_NIL) != 0;
    const uint32_t c0 = b.comment_off[r], c1 = b.comment_off[r + 1];
    if (!comments_nil && c1 != c0) emit_tg_comments(line + xp[XL_COMMENTS], &mss[wid], b, c0, c1);
    const uint32_t r0 = b.react_off[r], r1 = b.react_off[r + 1];
    if (r1 != r0 && !(in.xlen[r * 8 + XL_FLAGS] & XLF_SIMPLE_MAP)) emit_reaction_map(line + xp[XL_REACTIONS], &mss[wid], b.reacts, r0, r1, b.aux);
    const uint32_t nl = in.link_count[r];
    if (nl > LANE_LINKS_MAX) emit_tg_outlinks(line + xp[XL_OUTLINKS], in.arena + in.link_start[r], nl);
    __syncwarp();
  }
}
__global__ void __launch_bounds__(CTA_THREADS, LB_MAPS) tg_emit_maps_kernel(TgBatchDev b, EmitIn in) { tg_emit_maps_body(b, in); }

// ---- YouTube (config 4) ------------------------------------------------------------------------------
struct YtOut {
  uint8_t* status;
  uint32_t* linelen;
  uint32_t* url_start;   // [n] first unique URL of the record in `urls`
  uint32_t* url_count;
  YtUrl* urls;
  uint32_t urls_cap;
  uint32_t* url_cursor;
  uint32_t* esc_len;     // [n][3] escaped length of the description / title, clean flag (size pass -> emit pass)
  uint32_t* link_start;  // [n] channel-id links (frontier candidates)
  uint32_t* link_count;
  tgi_link* arena;
  uint32_t arena_cap;
  uint32_t* cursor;
  int* err;
};

// unique outlink URLs (extractURLs) and snowball channel ids (extractChannelIDsFromText)
DEVI void yt_parse_body(const YtBatchDev& b, const CfgDev& cfg, uint32_t run_flags, const YtOut& o) {
  int wid = threadIdx.x >> 5, l = lane_id();
  uint64_t nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t r = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; r < b.n; r += nwarps) {
    const tgi_yt_rec v = b.recs[r];
    const uint8_t* desc = b.strs + v.str_off + v.id_len + v.title_len;
    uint32_t us = 0, uc = 0, ls = 0, lc = 0;
    uint32_t ub = yt_count_http(desc, v.desc_len);
    if (ub) {
      if (l == 0) us = atomicAdd(o.url_cursor, ub);
      us = __shfl_sync(FULL, us, 0);
      if (us + ub > o.urls_cap || us + ub < us) {
        if (l == 0) atomicOr(o.err, ERR_ARENA_OVERFLOW);
      } else {
        uc = yt_extract_urls(desc, v.desc_len, o.urls + us, ub);
      }
    }
    if (run_flags & (TGI_RUN_LINKS | TGI_RUN_FRONTIER)) {
      uint32_t lb = yt_count_ytcom(desc, v.desc_len);
      if (lb >= (1u << 20)) {
        if (l == 0) atomicOr(o.err, ERR_TOO_MANY_LINKS);
        lb = 0;
      }
      if (lb) {
        if (l == 0) ls = atomicAdd(o.cursor, lb);
        ls = __shfl_sync(FULL, ls, 0);
        if (ls + lb > o.arena_cap || ls + lb < ls) {
          if (l == 0) atomicOr(o.err, ERR_ARENA_OVERFLOW);
        } else {
          lc = yt_channel_ids(desc, v.desc_len, o.arena + ls, lb);
        }
      }
    }
    if (l == 0) {
      // json.Marshal fails (no line, record still "fetched") when a time.Time is outside year
      // [0,9999]; decided here so that the status does not depend on TGI_RUN_JSONL
      uint8_t tmp[40];
      bool ok = !(cfg.flags & CFGDEV_CLOCK_INVALID) && cfg.created_yt_len != 0 &&
                render_time(tmp, v.published_sec, v.published_nsec, 0) != 0;
      if (ok) {
        const tgi_yt_chan& ch = b.chans[v.chan_idx];
        if (ch.cached) ok = render_time(tmp, ch.published_sec, ch.published_nsec, 0) != 0;
      }
      o.status[r] = ok ? TGI_ST_EMITTED : TGI_ST_NOLINE;
      o.linelen[r] = 0;
      o.url_start[r] = us;
      o.url_count[r] = uc;
      o.link_start[r] = ls;
      o.link_count[r] = lc;
    }
  }
}
__global__ void __launch_bounds__(CTA_THREADS, LB_YT) yt_parse_kernel(YtBatchDev b, CfgDev cfg, uint32_t run_flags, YtOut o) { yt_parse_body(b, cfg, run_flags, o); }

// one record by one warp (yt_page_kernel)
DEVI void yt_size_record(const YtBatchDev& b, const CfgDev& cfg, const YtOut& o, uint64_t r, YtScratch* sc) {
  const int l = lane_id();
  {
    YtArgs a;
    a.b = &b;
    a.cfg = &cfg;
    a.r = r;
    a.urls = o.urls + o.url_start[r];
    a.n_urls = o.url_count[r];
    YtSizer z;
    z.sc = sc;
    {
      const tgi_yt_rec* rec = &b.recs[r];
      const uint8_t* title = b.strs + rec->str_off + rec->id_len;
      z.el[1] = warp_esc_len(title, rec->title_len);
      z.el[0] = warp_esc_len(title + rec->title_len, rec->desc_len);
    }
    bool ok = walk_yt_record(z, a);
    if (l == 0) {
      o.esc_len[3 * r] = z.el[0];
      o.esc_len[3 * r + 1] = z.el[1];
      o.esc_len[3 * r + 2] = z.dirty ? 0u : 1u;  // clean: the lane writer takes the record
      o.linelen[r] = ok ? (uint32_t)z.total : 0u;
      if (!ok) o.status[r] = TGI_ST_NOLINE;
    }
  }
}
// length pass, one lane per record (yt_lane.cuh); the description and the title are measured by the warp
__global__ void __launch_bounds__(CTA_THREADS, LB_YT) yt_size_lane_kernel(YtBatchDev b, CfgDev cfg, YtOut o) {
  const int wid = threadIdx.x >> 5, l = lane_id();
  const uint64_t ngroups = (b.n + 31) / 32, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t g = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; g < ngroups; g += nwarps) {
    uint64_t r = g * 32 + l;
    bool active = r < b.n;
    if (!active) r = b.n - 1;
    active = active && o.status[r] == TGI_ST_EMITTED;
    const tgi_yt_rec* rec = &b.recs[r];
    const uint8_t* title = b.strs + rec->str_off + rec->id_len;
    const uint32_t tn = rec->title_len, dn = rec->desc_len;
    uint32_t el0 = 0, el1 = 0;
    bool exact = false;  // the description / title holds invalid UTF-8 or U+2028/9: only the exact (warp) escaper may write it
    uint32_t todo = __ballot_sync(FULL, active);
    while (todo) {  // the two long strings of every record, all lanes
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint8_t* t = (const uint8_t*)__shfl_sync(FULL, (unsigned long long)(uintptr_t)title, src);
      const uint32_t a = __shfl_sync(FULL, tn, src), d = __shfl_sync(FULL, dn, src);
      bool x1 = false, x0 = false;
      const uint32_t e1 = warp_esc_len(t, a, &x1), e0 = warp_esc_len(t + a, d, &x0);
      if (l == src) {
        el0 = e0;
        el1 = e1;
        exact = x0 || x1;
      }
    }
    if (!active) continue;
    YtArgs a;
    a.b = &b;
    a.cfg = &cfg;
    a.r = r;
    a.urls = o.urls + o.url_start[r];
    a.n_urls = o.url_count[r];
    YtLaneSizer z;
    z.el[0] = el0;
    z.el[1] = el1;
    const bool ok = walk_yt_record(z, a);
    o.esc_len[3 * r] = el0;
    o.esc_len[3 * r + 1] = el1;
    // 1: clean, 2: the lane writer escapes the description / title itself, 0: left to the warp writer
    o.esc_len[3 * r + 2] = !z.dirty ? 1u : (!z.small_dirty && !exact) ? 2u : 0u;
    o.linelen[r] = ok ? (uint32_t)z.total : 0u;
    if (!ok) o.status[r] = TGI_ST_NOLINE;
  }
}

// warp writer: the records the lane writer does not take (a string needs escaping); lanes pick them out of
// groups of 32.  yt_page_kernel writes every record with yt_emit_record.
DEVI void yt_emit_record(const YtBatchDev& b, const CfgDev& cfg, const YtOut& o, const uint64_t* line_off, uint8_t* out, int* err,
                         uint64_t r, YtScratch* sc) {
  YtArgs a;
  a.b = &b;
  a.cfg = &cfg;
  a.r = r;
  a.urls = o.urls + o.url_start[r];
  a.n_urls = o.url_count[r];
  YtWriter w;
  w.sc = sc;
  w.el[0] = o.esc_len[3 * r];
  w.el[1] = o.esc_len[3 * r + 1];
  w.p = out + line_off[r];
  walk_yt_record(w, a);
  if (lane_id() == 0 && (uint64_t)(w.p - out) != line_off[r + 1]) atomicOr(err, ERR_LINE_MISMATCH);
  __syncwarp();
}
__global__ void __launch_bounds__(CTA_THREADS, LB_YT) yt_emit_kernel(YtBatchDev b, CfgDev cfg, YtOut o, const uint64_t* line_off, uint8_t* out, int* err) {
  __shared__ YtScratch scs[WARPS_PER_CTA];
  int wid = threadIdx.x >> 5, l = lane_id();
  const uint64_t ngroups = (b.n + 31) / 32, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t g = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; g < ngroups; g += nwarps) {
    const uint64_t rl = g * 32 + l;
    uint32_t todo = __ballot_sync(FULL, rl < b.n && o.status[rl] == TGI_ST_EMITTED && !o.esc_len[3 * rl + 2]);
    while (todo) {
      const uint64_t r = g * 32 + (uint32_t)(__ffs(todo) - 1);
      todo &= todo - 1;
      yt_emit_record(b, cfg, o, line_off, out, err, r, &scs[wid]);
    }
  }
}

// lane writer (yt_lane.cuh): one lane per clean record
__global__ void __launch_bounds__(CTA_THREADS, LB_YT) yt_emit_lane_kernel(YtBatchDev b, CfgDev cfg, YtOut o, const uint64_t* line_off, uint8_t* out, int* err) {
  const int wid = threadIdx.x >> 5, l = lane_id();
  const uint64_t ngroups = (b.n + 31) / 32, nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t g = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; g < ngroups; g += nwarps) {
    const uint64_t r = g * 32 + l;
    const bool active = r < b.n && o.status[r] == TGI_ST_EMITTED && o.esc_len[3 * r + 2];
    YtLaneWriter w;
    if (active) {
      w.el[0] = o.esc_len[3 * r];
      w.el[1] = o.esc_len[3 * r + 1];
      YtArgs a;
      a.b = &b;
      a.cfg = &cfg;
      a.r = r;
      a.urls = o.urls + o.url_start[r];
      a.n_urls = o.url_count[r];
      w.begin((uint64_t)(uintptr_t)out + line_off[r]);
      walk_yt_record(w, a);
      w.end();
      if (w.s.pos != (uint64_t)(uintptr_t)out + line_off[r + 1]) atomicOr(err, ERR_LINE_MISMATCH);
    }
    __syncwarp();
    w.flush_pending(active);
  }
}

// ---- message-status join (SURVEY 8f rank 2): first index in A of every key of B ---------------------------------
DEVI uint64_t join_hash(long long chat, long long msg) {  // splitmix64 finaliser over both words
  uint64_t x = (uint64_t)chat * 0x9E3779B97F4A7C15ull ^ (uint64_t)msg;
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// table[slot] = 1 + smallest index of an A element with that slot's key, 0 = empty
__global__ void join_build_kernel(const longlong2* a, uint64_t na, uint32_t* table, uint64_t mask) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= na) return;
  const longlong2 k = a[i];
  for (uint64_t s = join_hash(k.x, k.y) & mask;; s = (s + 1) & mask) {
    uint32_t cur = atomicCAS(&table[s], 0u, (uint32_t)i + 1u);
    if (cur == 0) return;  // claimed
    const longlong2 o = a[cur - 1];  // the occupant's key never changes (only its index may get smaller)
    if (o.x == k.x && o.y == k.y) {
      atomicMin(&table[s], (uint32_t)i + 1u);
      return;
    }
  }
}
__global__ void join_probe_kernel(const longlong2* a, const uint32_t* table, uint64_t mask, const longlong2* b, uint64_t nb, long long* out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nb) return;
  const longlong2 k = b[i];
  long long res = -1;
  for (uint64_t s = join_hash(k.x, k.y) & mask;; s = (s + 1) & mask) {
    const uint32_t cur = table[s];
    if (cur == 0) break;
    const longlong2 o = a[cur - 1];
    if (o.x == k.x && o.y == k.y) {
      res = (long long)cur - 1;
      break;
    }
  }
  out[i] = res;
}

// ---- generic client.Message -> sparse Post (a12) ---------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS, 4) gm_size_kernel(GmBatchDev b, CfgDev cfg, uint8_t* status, uint32_t* linelen) {
  __shared__ YtScratch scs[WARPS_PER_CTA];
  int wid = threadIdx.x >> 5, l = lane_id();
  uint64_t nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t r = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; r < b.n; r += nwarps) {
    YtSizer z;
    z.sc = &scs[wid];
    bool ok = walk_gm_record(z, b, cfg, r);
    if (l == 0) {
      status[r] = ok ? TGI_ST_EMITTED : TGI_ST_NOLINE;
      linelen[r] = ok ? (uint32_t)z.total : 0u;
    }
  }
}
__global__ void __launch_bounds__(CTA_THREADS, 4) gm_emit_kernel(GmBatchDev b, CfgDev cfg, const uint8_t* status, const uint64_t* line_off,
                                                                 uint8_t* out, int* err) {
  __shared__ YtScratch scs[WARPS_PER_CTA];
  int wid = threadIdx.x >> 5, l = lane_id();
  uint64_t nwarps = (uint64_t)gridDim.x * WARPS_PER_CTA;
  for (uint64_t r = (uint64_t)blockIdx.x * WARPS_PER_CTA + wid; r < b.n; r += nwarps) {
    if (status[r] != TGI_ST_EMITTED) continue;
    YtWriter w;
    w.sc = &scs[wid];
    w.p = out + line_off[r];
    walk_gm_record(w, b, cfg, r);
    if (l == 0 && (uint64_t)(w.p - out) != line_off[r + 1]) atomicOr(err, ERR_LINE_MISMATCH);
  }
}

// ---- exclusive scan u32 -> u64 (out has n+1 entries) ----------------------------------------------
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 8, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ uint64_t block_reduce_u64(uint64_t v, uint64_t* sm) {
  for (int d = 16; d; d >>= 1) v += __shfl_down_sync(FULL, v, d);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  uint64_t t = 0;
  if (threadIdx.x < 32) {
    t = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0;
    for (int d = 16; d; d >>= 1) t += __shfl_down_sync(FULL, t, d);
  }
  return t;  // valid in thread 0
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_tile_sums_kernel(const uint32_t* in, uint64_t n, uint64_t* tile_sums) {
  __shared__ uint64_t sm[32];
  uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE;
  uint64_t s = 0;
  for (int k = 0; k < SCAN_ITEMS; k++) {
    uint64_t i = base + (uint64_t)k * SCAN_THREADS + threadIdx.x;
    if (i < n) s += in[i];
  }
  uint64_t t = block_reduce_u64(s, sm);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = t;
}

// single block: exclusive scan of tile sums in place; total -> out_total
__global__ void __launch_bounds__(1024) scan_tiles_kernel(uint64_t* tile_sums, uint64_t ntiles, uint64_t* out_total) {
  __shared__ uint64_t sm[32];
  __shared__ uint64_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (uint64_t base = 0; base < ntiles; base += 1024) {
    uint64_t i = base + threadIdx.x;
    uint64_t v = i < ntiles ? tile_sums[i] : 0;
    uint64_t x = v;
    int l = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int d = 1; d < 32; d <<= 1) {
      uint64_t t = __shfl_up_sync(FULL, x, d);
      if (l >= d) x += t;
    }
    if (l == 31) sm[w] = x;
    __syncthreads();
    if (w == 0) {
      uint64_t y = sm[l];
      for (int d = 1; d < 32; d <<= 1) {
        uint64_t t = __shfl_up_sync(FULL, y, d);
        if (l >= d) y += t;
      }
      sm[l] = y;
    }
    __syncthreads();
    uint64_t carry = carry_s;
    uint64_t incl = x + (w ? sm[w - 1] : 0);
    if (i < ntiles) tile_sums[i] = carry + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = carry + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) *out_total = carry_s;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const uint32_t* in, uint64_t n, const uint64_t* tile_base,
                                                               const uint64_t* total, uint64_t* out) {
  __shared__ uint64_t sm[32];
  // blocked arrangement: thread t owns items [t*ITEMS, (t+1)*ITEMS) of the tile
  uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS];
  uint64_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) {
    v[k] = base + k < n ? in[base + k] : 0;
    s += v[k];
  }
  uint64_t x = s;
  int l = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int d = 1; d < 32; d <<= 1) {
    uint64_t t = __shfl_up_sync(FULL, x, d);
    if (l >= d) x += t;
  }
  if (l == 31) sm[w] = x;
  __syncthreads();
  if (w == 0) {
    uint64_t y = l < (SCAN_THREADS >> 5) ? sm[l] : 0;
    for (int d = 1; d < 32; d <<= 1) {
      uint64_t t = __shfl_up_sync(FULL, y, d);
      if (l >= d) y += t;
    }
    sm[l] = y;
  }
  __syncthreads();
  uint64_t excl = tile_base[blockIdx.x] + (w ? sm[w - 1] : 0) + x - s;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) {
    if (base + k < n) out[base + k] = excl;
    excl += v[k];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = *total;
}

// the whole scan in ONE launch for page-sized batches (n <= SCAN_SMALL_MAX): one CTA, SCAN_SMALL_ITEMS per thread
constexpr int SCAN_SMALL_THREADS = 1024, SCAN_SMALL_ITEMS = 8, SCAN_SMALL_MAX = SCAN_SMALL_THREADS * SCAN_SMALL_ITEMS;
__global__ void __launch_bounds__(SCAN_SMALL_THREADS) scan_small_kernel(const uint32_t* in, uint64_t n, uint64_t* out, uint64_t* out_total) {
  __shared__ uint64_t sm[32];
  const uint64_t base = (uint64_t)threadIdx.x * SCAN_SMALL_ITEMS;
  uint32_t v[SCAN_SMALL_ITEMS];
  uint64_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_SMALL_ITEMS; k++) {
    v[k] = base + k < n ? in[base + k] : 0;
    s += v[k];
  }
  uint64_t x = s;
  const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int d = 1; d < 32; d <<= 1) {
    const uint64_t t = __shfl_up_sync(FULL, x, d);
    if (l >= d) x += t;
  }
  if (l == 31) sm[w] = x;
  __syncthreads();
  if (w == 0) {
    uint64_t y = sm[l];
    for (int d = 1; d < 32; d <<= 1) {
      const uint64_t t = __shfl_up_sync(FULL, y, d);
      if (l >= d) y += t;
    }
    sm[l] = y;
  }
  __syncthreads();
  uint64_t excl = (w ? sm[w - 1] : 0) + x - s;
#pragma unroll
  for (int k = 0; k < SCAN_SMALL_ITEMS; k++) {
    if (base + k < n) out[base + k] = excl;
    excl += v[k];
  }
  if (threadIdx.x == SCAN_SMALL_THREADS - 1) {
    out[n] = sm[31];
    *out_total = sm[31];
  }
}

// ---- frontier: exact hash set of 32-byte keys ------------------------------------------------------
struct FrontierDev {
  uint8_t* pool;     // [cap][32] distinct keys in first-occurrence order
  uint64_t cap;
  uint64_t* table;   // persistent table: 0 = empty, else (pool_idx+1) | fp << 40
  uint64_t tmask;
  uint64_t* count;   // device scalar: number of keys in the pool
  uint64_t* payload; // optional [cap]: 64-bit payload of every key (the owned partition of the multi-GPU merge)
};
struct FrontierBatch {
  uint64_t* btable;  // per-batch table: 0 = empty, else ((rec << SEQ_ORD_BITS) | ordinal) + 1 (atomicMin'd)
  uint64_t bmask;
  uint32_t* lstate;  // per arena slot: LS_* or batch-table slot index
  uint32_t* rec_new; // [n] new keys first seen in this record
};
// sequence number of a link inside a batch: (record << 20) | ordinal.  Records < 2^40 (checked by the host), so a
// record may carry up to 2^20 link candidates (> 10 MB of text: beyond anything TDLib delivers; the host checks)
constexpr int SEQ_ORD_BITS = 20;
#define LS_INELIGIBLE 0xFFFFFFFFu
#define LS_KNOWN 0xFFFFFFFEu

struct Key32 {
  uint32_t w[8];
};
DEVI Key32 load_key(const uint8_t* p) {  // 4-byte aligned
  Key32 k;
  const uint32_t* q = (const uint32_t*)p;
#pragma unroll
  for (int i = 0; i < 8; i++) k.w[i] = q[i];
  return k;
}
DEVI bool key_eq(const Key32& a, const Key32& b) {
  uint32_t d = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) d |= a.w[i] ^ b.w[i];
  return d == 0;
}
DEVI uint64_t key_hash(const Key32& k) {
  uint64_t h = 0x9E3779B97F4A7C15ull;
#pragma unroll
  for (int i = 0; i < 8; i += 2) {
    uint64_t x = (uint64_t)k.w[i] | ((uint64_t)k.w[i + 1] << 32);
    h = (h ^ x) * 0xFF51AFD7ED558CCDull;
    h ^= h >> 32;
  }
  h *= 0xC4CEB9FE1A85EC53ull;
  return h ^ (h >> 29);
}

// pool index of `key` in set f, or -1
DEVI int64_t set_lookup(const FrontierDev& f, const Key32& key, uint64_t h) {
  if (!f.table) return -1;
  const uint64_t fp = (h >> 40) | 1ull;
  for (uint64_t s = h & f.tmask;; s = (s + 1) & f.tmask) {
    const uint64_t e = f.table[s];
    if (e == 0) return -1;
    if ((e >> 40) == fp) {
      const uint64_t pi = (e & 0xFFFFFFFFFFull) - 1;
      if (key_eq(key, load_key(f.pool + 32 * pi))) return (int64_t)pi;
    }
  }
}
// the resident exclusion sets of the frontier -> validator hand-off (tgi_set_add): invalid channels expire after
// TGI_INVALID_TTL_SEC (state/daprstate.go:3556-3564: time.Since(t) < invalidChannelTTL), stamp 0 = never
struct ExclusionDev {
  FrontierDev invalid, discovered;
  long long now_sec;
};
DEVI bool set_invalid_hit(const ExclusionDev& x, const Key32& key, uint64_t h, long long now_sec) {
  const int64_t pi = set_lookup(x.invalid, key, h);
  if (pi < 0) return false;
  const long long t = (long long)x.invalid.payload[pi];
  return t == 0 || now_sec - t < (long long)TGI_INVALID_TTL_SEC;
}

DEVI bool link_eligible(const tgi_link& lk, uint32_t run_flags) {
  if ((run_flags & TGI_RUN_SKIP_SELF) && (lk.flags & TGI_LF_SELF)) return false;    // runner.go:1231
  if ((run_flags & TGI_RUN_FILTER) && !(lk.flags & TGI_LF_FILTER_OK)) return false; // runner.go:1261
  return true;
}

// phase 1: probe the persistent set; unseen keys race into the batch table, min sequence wins
DEVI void frontier_probe_body(uint64_t n, const uint32_t* link_start, const uint32_t* link_count, tgi_link* arena,
                              uint32_t run_flags, const FrontierDev& f, const FrontierBatch& fb, const ExclusionDev& x,
                              uint64_t t0, uint64_t nt) {  // thread t0 of nt: the whole grid, or one CTA (page kernel)
 for (uint64_t r = t0; r < n; r += nt) {
  uint32_t cnt = link_count[r];
  if (!cnt) continue;
  uint32_t ls = link_start ? link_start[r] : (uint32_t)r;
  for (uint32_t k = 0; k < cnt; k++) {
    uint32_t idx = ls + k;
    tgi_link& lk = arena[idx];
    if ((run_flags & TGI_RUN_SKIP_SELF) && (lk.flags & TGI_LF_SELF)) {  // runner.go:1231
      fb.lstate[idx] = LS_INELIGIBLE;
      continue;
    }
    Key32 key = load_key(lk.name);
    uint64_t h = key_hash(key);
    if ((run_flags & TGI_RUN_SKIP_INVALID) && set_invalid_hit(x, key, h, x.now_sec)) {  // runner.go:1247 (before the filter)
      lk.flags |= TGI_LF_INVALID;
      fb.lstate[idx] = LS_INELIGIBLE;
      continue;
    }
    if ((run_flags & TGI_RUN_FILTER) && !(lk.flags & TGI_LF_FILTER_OK)) {  // runner.go:1261
      fb.lstate[idx] = LS_INELIGIBLE;
      continue;
    }
    uint64_t fp = (h >> 40) | 1ull;  // 24-bit fingerprint, never 0
    bool known = false;
    for (uint64_t s = h & f.tmask;; s = (s + 1) & f.tmask) {
      uint64_t e = f.table[s];
      if (e == 0) break;
      if ((e >> 40) == fp) {
        uint64_t pi = (e & 0xFFFFFFFFFFull) - 1;
        if (key_eq(key, load_key(f.pool + 32 * pi))) {
          known = true;
          break;
        }
      }
    }
    if (known) {
      fb.lstate[idx] = LS_KNOWN;
      continue;
    }
    uint64_t v = (((uint64_t)r << SEQ_ORD_BITS) | k) + 1;
    for (uint64_t s = (h >> 7) & fb.bmask;; s = (s + 1) & fb.bmask) {
      uint64_t cur = fb.btable[s];
      if (cur == 0) {
        cur = atomicCAS((unsigned long long*)&fb.btable[s], 0ull, (unsigned long long)v);
        if (cur == 0) {
          fb.lstate[idx] = (uint32_t)s;
          break;
        }
      }
      uint64_t r2 = (cur - 1) >> SEQ_ORD_BITS, k2 = (cur - 1) & ((1u << SEQ_ORD_BITS) - 1u);
      uint32_t ls2 = link_start ? link_start[r2] : (uint32_t)r2;
      if (key_eq(key, load_key(arena[ls2 + k2].name))) {
        atomicMin((unsigned long long*)&fb.btable[s], (unsigned long long)v);
        fb.lstate[idx] = (uint32_t)s;
        break;
      }
    }
  }
 }
}
__global__ void frontier_probe_kernel(uint64_t n, const uint32_t* link_start, const uint32_t* link_count,
                                      tgi_link* arena, uint32_t run_flags, FrontierDev f, FrontierBatch fb, ExclusionDev x) {
  frontier_probe_body(n, link_start, link_count, arena, run_flags, f, fb, x, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, (uint64_t)gridDim.x * blockDim.x);
}

// phase 2: per record, how many of its links are the global first occurrence of a new key
DEVI void frontier_count_body(uint64_t n, const uint32_t* link_start, const uint32_t* link_count, const FrontierBatch& fb,
                              uint64_t t0, uint64_t nt) {
  for (uint64_t r = t0; r < n; r += nt) {
    uint32_t cnt = link_count[r], c = 0;
    uint32_t ls = link_start ? link_start[r] : (uint32_t)r;
    for (uint32_t k = 0; k < cnt; k++) {
      uint32_t st = fb.lstate[ls + k];
      if (st >= LS_KNOWN) continue;
      if (fb.btable[st] == (((uint64_t)r << SEQ_ORD_BITS) | k) + 1) c++;
    }
    fb.rec_new[r] = c;
  }
}
__global__ void frontier_count_kernel(uint64_t n, const uint32_t* link_start, const uint32_t* link_count,
                                      FrontierBatch fb) {
  frontier_count_body(n, link_start, link_count, fb, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, (uint64_t)gridDim.x * blockDim.x);
}

// phase 3: append the new keys to the pool in (record, ordinal) order and publish them
DEVI void frontier_append_body(uint64_t n, const uint32_t* link_start, const uint32_t* link_count, tgi_link* arena,
                               const FrontierDev& f, const FrontierBatch& fb, const uint64_t* new_off, int* err,
                               const uint64_t* payload_in, uint64_t t0, uint64_t nt) {
 for (uint64_t r = t0; r < n; r += nt) {
  if (!fb.rec_new[r]) continue;
  uint64_t base = *f.count, total = new_off[n];
  if (base + total > f.cap) {
    atomicOr(err, ERR_FRONTIER_FULL);
    return;
  }
  uint32_t cnt = link_count[r];
  uint32_t ls = link_start ? link_start[r] : (uint32_t)r;
  uint64_t pi = base + new_off[r];
  for (uint32_t k = 0; k < cnt; k++) {
    uint32_t st = fb.lstate[ls + k];
    if (st >= LS_KNOWN) continue;
    if (fb.btable[st] != (((uint64_t)r << SEQ_ORD_BITS) | k) + 1) continue;
    tgi_link& lk = arena[ls + k];
    Key32 key = load_key(lk.name);
    uint32_t* dst = (uint32_t*)(f.pool + 32 * pi);
#pragma unroll
    for (int i = 0; i < 8; i++) dst[i] = key.w[i];
    if (f.payload) f.payload[pi] = payload_in ? payload_in[r] : 0ull;  // keys mode: one key per "record"
    uint64_t h = key_hash(key);
    uint64_t e = (pi + 1) | (((h >> 40) | 1ull) << 40);
    for (uint64_t s = h & f.tmask;; s = (s + 1) & f.tmask) {
      if (f.table[s] == 0 && atomicCAS((unsigned long long*)&f.table[s], 0ull, (unsigned long long)e) == 0) break;
    }
    lk.flags |= TGI_LF_NEW;
    pi++;
  }
 }
}
__global__ void frontier_append_kernel(uint64_t n, const uint32_t* link_start, const uint32_t* link_count,
                                       tgi_link* arena, FrontierDev f, FrontierBatch fb,
                                       const uint64_t* new_off, int* err, const uint64_t* payload_in = nullptr) {
  frontier_append_body(n, link_start, link_count, arena, f, fb, new_off, err, payload_in, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, (uint64_t)gridDim.x * blockDim.x);
}
DEVI void frontier_commit_body(const FrontierDev& f, const uint64_t* new_off, uint64_t n, uint64_t* out_new, int* err) {
  uint64_t total = new_off[n];
  if (*f.count + total <= f.cap) {
    *f.count += total;
    *out_new = total;
  } else {
    *out_new = 0;
    atomicOr(err, ERR_FRONTIER_FULL);
  }
  out_new[1] = *f.count;
}
__global__ void frontier_commit_kernel(FrontierDev f, const uint64_t* new_off, uint64_t n, uint64_t* out_new, int* err) {
  frontier_commit_body(f, new_off, n, out_new, err);
}

// ---- multi-GPU merge (SURVEY 8e option A): bucket the new local keys by owner rank ----------------------------------
DEVI uint32_t key_owner(const Key32& k, uint32_t nranks) { return (uint32_t)((key_hash(k) >> 17) % nranks); }
__global__ void merge_count_kernel(const uint8_t* pool, uint64_t first, uint64_t m, uint32_t nranks, unsigned long long* cnt) {
  __shared__ unsigned int sc[64];
  if (threadIdx.x < 64) sc[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) atomicAdd(&sc[key_owner(load_key(pool + 32 * (first + i)), nranks)], 1u);
  __syncthreads();
  if (threadIdx.x < nranks && sc[threadIdx.x]) atomicAdd(&cnt[threadIdx.x], (unsigned long long)sc[threadIdx.x]);
}
// cursor[p] starts at the offset of bucket p in the send buffers; the order inside a bucket is irrelevant (the keys
// of one rank are distinct and every key carries its sequence number)
__global__ void merge_scatter_kernel(const uint8_t* pool, uint64_t first, uint64_t m, uint32_t nranks, unsigned long long* cursor,
                                     uint8_t* send_keys, uint64_t* send_pay, uint64_t pay_base) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const Key32 k = load_key(pool + 32 * (first + i));
  const unsigned long long pos = atomicAdd(&cursor[key_owner(k, nranks)], 1ull);
  uint32_t* dst = (uint32_t*)(send_keys + 32 * pos);
#pragma unroll
  for (int j = 0; j < 8; j++) dst[j] = k.w[j];
  send_pay[pos] = pay_base | (first + i);
}

// ---- frontier -> validator hand-off (SURVEY 8f rank 3): the new edges of a batch as packed pending_edges rows --------
// rec_new / new_off are what the frontier phase of the batch left behind: row index = new_off[r] + ordinal among the
// record's NEW links, i.e. (record, first-insertion) order — the order of the reference's INSERTs.
__global__ void edges_emit_kernel(uint64_t n, const uint32_t* link_start, const uint32_t* link_count, const tgi_link* arena,
                                  const uint32_t* chan_idx_of, uint32_t chan_stride, const uint64_t* new_off, ExclusionDev x,
                                  tgi_edge* rows, uint64_t cap) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint32_t cnt = link_count[r];
  if (!cnt) return;
  uint64_t row = new_off[r];
  const tgi_link* lk = arena + link_start[r];
  for (uint32_t k = 0; k < cnt; k++) {
    if (!(lk[k].flags & TGI_LF_NEW)) continue;
    if (row < cap) {
      const Key32 key = load_key(lk[k].name);
      const uint64_t h = key_hash(key);
      tgi_edge e;
      uint32_t* d = (uint32_t*)e.destination;
#pragma unroll
      for (int i = 0; i < 8; i++) d[i] = key.w[i];
      e.record = r;
      e.chan_idx = chan_idx_of ? *(const uint32_t*)((const uint8_t*)chan_idx_of + (size_t)r * chan_stride) : 0u;
      e.dest_len = lk[k].len;
      e.source_type = lk[k].src;
      e.status = set_invalid_hit(x, key, h, x.now_sec) ? TGI_EDGE_INVALID_CACHED           // validator.go:205-212
                 : set_lookup(x.discovered, key, h) >= 0 ? TGI_EDGE_DUPLICATE : TGI_EDGE_PENDING;  // :214-226
      e.reserved = 0;
      rows[row] = e;
    }
    row++;
  }
}

// keys32 -> pseudo arena (one link per "record") for tgi_frontier_insert
__global__ void keys_to_links_kernel(const uint8_t* keys, uint64_t n, tgi_link* arena, uint32_t* link_count) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  tgi_link lk;
  int len = 0;
  for (int k = 0; k < 32; k++) {
    lk.name[k] = keys[32 * i + k];
    if (lk.name[k]) len = k + 1;
  }
  lk.len = (uint8_t)len;
  lk.src = 0;
  lk.flags = 0;
  lk.filter_reason = 0;
  arena[i] = lk;
  link_count[i] = 1;
}
__global__ void links_new_flags_kernel(const tgi_link* arena, uint64_t n, uint8_t* is_new) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) is_new[i] = (arena[i].flags & TGI_LF_NEW) ? 1 : 0;
}

// ---- compaction of the per-record links for the host result -----------------------------------------
DEVI void links_compact_body(uint64_t n, const uint32_t* link_start, const uint32_t* link_count, const uint64_t* link_off,
                             const tgi_link* arena, tgi_link* out, uint32_t* link_off32) {
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= n; r += (uint64_t)gridDim.x * blockDim.x) {
    link_off32[r] = (uint32_t)link_off[r];
    if (r == n) break;
    uint32_t cnt = link_count[r];
    const uint32_t* src = (const uint32_t*)(arena + link_start[r]);
    uint32_t* dst = (uint32_t*)(out + link_off[r]);
    for (uint32_t k = 0; k < cnt * 9; k++) dst[k] = src[k];
  }
}
__global__ void links_compact_kernel(uint64_t n, const uint32_t* link_start, const uint32_t* link_count,
                                     const uint64_t* link_off, const tgi_link* arena, tgi_link* out,
                                     uint32_t* link_off32) {
  links_compact_body(n, link_start, link_count, link_off, arena, out, link_off32);
}

// FilterUsername over a list of names (tgi_filter_usernames): one warp per name
__global__ void filter_usernames_kernel(const uint8_t* names, const uint32_t* off, uint64_t n, uint8_t* reason) {
  uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  int l = lane_id();
  uint32_t a = off[i], len = off[i + 1] - a;
  uint32_t c = ((uint32_t)l < len) ? ldb(names + a + l) : 0u;
  uint32_t res = warp_filter_username(c, len);
  if (res == TGI_FU_INVALID_CHAR || res == TGI_FU_VALID || res == TGI_FU_BOT_SUFFIX) {
    // names longer than a warp cannot reach here (len > 32 -> too_long)
  }
  if (l == 0) reason[i] = (uint8_t)res;
}

}  // namespace tgi
