// tg_lane.cuh — lane-per-record emission of the fixed part of the Telegram Post line.
//
// One warp takes 32 consecutive records and every lane streams ITS OWN line: the scalar work
// (number / time rendering, piece lengths, offsets) that kept 31 lanes idle in the warp-per-record
// walker now runs 32 records wide, and the bytes leave the SM as 16-byte aligned vector stores.
// The line is the same generated piece program as everywhere else (tools/gen_pieces.py); control
// flow is uniform across the warp (same piece sequence for every record), only lengths, sources
// and the output phase differ per lane.
//
// A lane's output is a byte stream at an arbitrary address: LaneStream keeps the bytes of the
// current 16-byte block in four registers.  Full blocks are staged in the lane's own shared-memory
// row; the warp drains all 32 rows together with coalesced 16-byte stores (ls_drain_warp).  Blocks
// shared with somebody else (the neighbouring
// line, or a variable piece written by the esc / maps kernels) are stored byte-exact (store_bytes),
// so the kernels never overwrite each other's bytes.
//
// Reference semantics: telegramhelper/tdutils.go:633-717 (field map) + encoding/json of model.Post
// (model/data.go:9-75); see tg_walk.cuh.
#pragma once
#include "tg_walk.cuh"

namespace tgi {

#ifndef LANE_STAGE
#define LANE_STAGE 128
#endif
constexpr uint32_t LANE_STAGE_BYTES = LANE_STAGE;             // staged per lane between two drains (128 or 64)
constexpr uint32_t LANE_STAGE_ROW = LANE_STAGE_BYTES + 16;    // +16 spreads the lanes' rows over the banks

struct LaneStream {
  uint64_t pos;             // absolute address of the next output byte
  uint32_t c0, c1, c2, c3;  // bytes [head, pos & 15) of the current block, zero elsewhere
  uint32_t head;            // first byte of the current block that belongs to this stream
  uint64_t seg;             // global address of the first block staged in the row
  uint32_t row_s;           // shared-space address of the lane's staging row
  uint32_t fill;            // bytes staged in the row (consecutive blocks starting at seg)
};

DEVI void ls_stage(LaneStream& s, uint64_t blk) {
  if (s.fill == 0) s.seg = blk;
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(s.row_s + s.fill), "r"(s.c0), "r"(s.c1), "r"(s.c2), "r"(s.c3) : "memory");
  s.fill += 16;
}

// Warp-collective: write every lane's staged blocks to HBM.  Eight lanes take one row (8 x 16 B), so
// one LDS.128 / STG.128 pair moves four rows and the global stores are coalesced per row (the per-lane
// alternatives, measured: ST.128 straight from the lanes = 32 lines per instruction, 1.2 TB/s in
// tools/tma_bench.cu; per-lane TMA bulk stores reach 4.8-6.1 TB/s there but cost ~10 issue slots
// each, because UBLKCP is a uniform-datapath instruction and the compiler serialises the lanes).
DEVI void ls_drain_warp(LaneStream& s) {
  if (!__any_sync(FULL, s.fill != 0)) return;
  __syncwarp();
  constexpr int LPR = LANE_STAGE_BYTES / 16, RPP = 32 / LPR;  // lanes per row, rows per pass
  const int l = lane_id(), sub = l / LPR, t16 = (l % LPR) * 16;
  const uint32_t warp_rows = s.row_s - (uint32_t)l * LANE_STAGE_ROW;
#pragma unroll 2
  for (int j = 0; j < 32; j += RPP) {
    const int rj = j + sub;
    const uint32_t f = __shfl_sync(FULL, s.fill, rj);
    const uint64_t sg = __shfl_sync(FULL, s.seg, rj);
    if ((uint32_t)t16 < f) {
      uint4 w;
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "r"(warp_rows + (uint32_t)rj * LANE_STAGE_ROW + (uint32_t)t16) : "memory");
      *(uint4*)(uintptr_t)(sg + (uint32_t)t16) = w;
    }
  }
  __syncwarp();
  s.fill = 0;
}
DEVI void ls_maybe_drain(LaneStream& s) {
  if (__any_sync(FULL, s.fill >= LANE_STAGE_BYTES)) ls_drain_warp(s);
}

// bytes [lo, hi) of the 16-byte block at blk (16-byte aligned)
__device__ __noinline__ void store_bytes(uint64_t blk, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t lo,
                                         uint32_t hi) {
  const uint32_t w[4] = {c0, c1, c2, c3};
#pragma unroll
  for (uint32_t i = 0; i < 4; i++) {
    const uint32_t a = 4u * i;
    if (lo <= a && a + 4u <= hi) {
      *(uint32_t*)(uintptr_t)(blk + a) = w[i];
    } else {
#pragma unroll
      for (uint32_t k = 0; k < 4; k++)
        if (lo <= a + k && a + k < hi) *(uint8_t*)(uintptr_t)(blk + a + k) = (uint8_t)(w[i] >> (8u * k));
    }
  }
}

DEVI void ls_init(LaneStream& s, uint32_t row_s) {  // once per kernel
  s.row_s = row_s;
  s.fill = 0;
  s.seg = 0;
}
DEVI void ls_begin(LaneStream& s, uint64_t addr) {
  s.pos = addr;
  s.head = (uint32_t)addr & 15u;
  s.c0 = s.c1 = s.c2 = s.c3 = 0;
}

// append n (1..16) bytes held little-endian in w (zero beyond n)
DEVI void ls_append(LaneStream& s, uint4 w, uint32_t n) {
  const uint32_t ph = (uint32_t)s.pos & 15u, sh = (ph & 3u) * 8u;
  // shift left by ph bytes into an 8-word window: first the byte part ...
  const uint32_t v0 = w.x << sh, v1 = __funnelshift_l(w.x, w.y, sh), v2 = __funnelshift_l(w.y, w.z, sh),
                 v3 = __funnelshift_l(w.z, w.w, sh), v4 = __funnelshift_l(w.w, 0u, sh);
  // ... then the word part (two select levels)
  const bool b0 = (ph & 4u) != 0, b1 = (ph & 8u) != 0;
  const uint32_t z0 = b0 ? 0u : v0, z1 = b0 ? v0 : v1, z2 = b0 ? v1 : v2, z3 = b0 ? v2 : v3, z4 = b0 ? v3 : v4,
                 z5 = b0 ? v4 : 0u;
  s.c0 |= b1 ? 0u : z0;
  s.c1 |= b1 ? 0u : z1;
  s.c2 |= b1 ? z0 : z2;
  s.c3 |= b1 ? z1 : z3;
  if (ph + n >= 16u) {
    const uint64_t blk = s.pos & ~15ull;
    if (s.head == 0) {
      ls_stage(s, blk);
    } else {
      store_bytes(blk, s.c0, s.c1, s.c2, s.c3, s.head, 16u);
      s.head = 0;
    }
    s.c0 = b1 ? z2 : z4;
    s.c1 = b1 ? z3 : z5;
    s.c2 = b1 ? z4 : 0u;
    s.c3 = b1 ? z5 : 0u;
  }
  s.pos += n;
}

// w >> (8 * sb) over 128 bits, sb in 0..15 (per lane)
DEVI uint4 shr128_bytes(uint4 w, uint32_t sb) {
  const uint32_t sh = (sb & 3u) * 8u;
  const uint32_t v0 = __funnelshift_r(w.x, w.y, sh), v1 = __funnelshift_r(w.y, w.z, sh), v2 = __funnelshift_r(w.z, w.w, sh),
                 v3 = w.w >> sh;
  const bool b0 = (sb & 4u) != 0, b1 = (sb & 8u) != 0;
  const uint32_t a0 = b0 ? v1 : v0, a1 = b0 ? v2 : v1, a2 = b0 ? v3 : v2, a3 = b0 ? 0u : v3;
  return make_uint4(b1 ? a2 : a0, b1 ? a3 : a1, b1 ? 0u : a2, b1 ? 0u : a3);
}
// keep the low k bytes (k in 0..16)
DEVI uint4 mask128(uint4 w, uint32_t k) {
  auto m = [&](uint32_t lo) -> uint32_t {  // mask of word starting at byte lo
    return k >= lo + 4u ? 0xffffffffu : (k <= lo ? 0u : (1u << ((k - lo) * 8u)) - 1u);
  };
  return make_uint4(w.x & m(0), w.y & m(4), w.z & m(8), w.w & m(12));
}

// write out what the current block holds (before a gap / at the end of the line); the staged blocks
// stay in the row until the next warp-collective drain
DEVI void ls_flush(LaneStream& s) {
  const uint32_t ph = (uint32_t)s.pos & 15u;
  if (ph > s.head) store_bytes(s.pos & ~15ull, s.c0, s.c1, s.c2, s.c3, s.head, ph);
  s.c0 = s.c1 = s.c2 = s.c3 = 0;
  s.head = ph;
}

// leave g bytes to another writer.  Warp-collective: the staged blocks of a lane must be consecutive,
// so a gap in any lane drains the rows first.
DEVI void ls_skip(LaneStream& s, uint32_t g) {
  if (__any_sync(FULL, g != 0)) ls_drain_warp(s);
  if (g) {
    ls_flush(s);
    s.pos += g;
    s.head = (uint32_t)s.pos & 15u;
  }
}

// ---- the kernel's shared state ------------------------------------------------------------------------
constexpr int LANE_ROW_WORDS = 36;  // per lane: 8 blocks of rendered fields + 8 length bytes; 36 = 4 * odd
                                    // keeps the lanes' LDS.128 on distinct banks
constexpr int LANE_WARPS = 8;
constexpr uint32_t LANE_LINKS_MAX = 4;   // more outlinks than this are left to the maps kernel
#ifndef LANE_TEXT
#define LANE_TEXT 512
#endif
constexpr uint32_t LANE_TEXT_MAX = LANE_TEXT;  // longer (or escaped) strings are left to the warp-per-record esc kernel
struct LaneShared {
  uint4 tmpl[kTgLaneTemplateLen / 16];
  uint4 ptype[TGI_CT__COUNT * 2];  // MessageContentType() strings, 32 bytes each, zero padded
  uint32_t pieces[64];
  uint32_t rows[LANE_WARPS][32][LANE_ROW_WORDS];
  uint4 stage[LANE_WARPS][32][LANE_STAGE_ROW / 16];
};

DEVI void lane_shared_fill(LaneShared& sh) {
  for (int i = threadIdx.x; i < kTgLaneTemplateLen / 16; i += blockDim.x) sh.tmpl[i] = ((const uint4*)kTgLaneTemplate)[i];
  for (int i = threadIdx.x; i < kTgLaneNPieces; i += blockDim.x) sh.pieces[i] = kTgLanePieces[i];
  uint32_t* pt = (uint32_t*)sh.ptype;
  for (int i = threadIdx.x; i < TGI_CT__COUNT * 8; i += blockDim.x) {
    const int ct = i >> 3, w = i & 7;
    pt[i] = w < 7 ? ((const uint32_t*)kPostType[ct])[w] : 0u;
  }
}

// One lane, one record.  `active` lanes emit; the others only keep the warp's control flow company.
DEVI void emit_tg_lane(LaneShared& sh, uint32_t* row, LaneStream& s, const TgBatchDev& b, const CfgDev& cfg, uint64_t r, bool active,
                       uint8_t* out, const uint64_t* line_off, const uint32_t* xlen_g, uint32_t* xpos_g, const tgi_link* links,
                       uint32_t nl, int* err, uint64_t& bytes_out, uint64_t& bytes_in, uint32_t& left) {
  uint32_t gaps = 0, copied = 0;  // statistics: bytes left to the other emit kernels / bytes copied from HBM sources
  left = 0;  // what this lane leaves to the other emit kernels: bit arg (XL_DESC..XL_ALT) = that string, bit 4 = a map / list
  TgWalkArgs a;
  a.b = &b;
  a.cfg = &cfg;
  a.r = r;
  a.links = nullptr;
  a.n_links = 0;
  {  // the record header, as load_rec_view (kernels.cuh)
    const tgi_tg_rec* rec = &b.recs[r];
    a.v.rec = rec;
    a.v.text = b.strs + rec->str_off;
    a.v.text_len = rec->text_len;
    a.v.alt = a.v.text + a.v.text_len;
    a.v.alt_len = rec->alt_len;
    a.v.media = a.v.alt + a.v.alt_len;
    a.v.media_len = rec->media_len;
    a.v.handle = a.v.media + a.v.media_len;
    a.v.handle_len = rec->handle_len;
    a.v.ct = rec->content_type;
    a.v.flags = rec->flags;
    a.v.e0 = a.v.e1 = 0;
  }
  const tgi_tg_rec* rec = a.v.rec;
  const ChanDerived cd = b.chan_derived[rec->chan_idx];
  const TgDerived d = tg_derive(a, cd);
  const uint32_t condmask = active ? tg_condmask(a, d) : 0u;
  const uint32_t ct = a.v.ct;

  // rendered fields: block 0 msgno, 1-2 chat id, 3 views, 4 shares, 5 comments, 6-7 time; lengths at byte 128+
  uint8_t* rb = (uint8_t*)row;
#pragma unroll
  for (int k = 0; k < 8; k++) ((uint4*)row)[k] = make_uint4(0, 0, 0, 0);
#pragma unroll 1
  for (int f = 0; f < 5; f++) {
    const int64_t v = f == 0 ? rec->id / 1048576  // tdutils.go:1008
                             : f == 1 ? rec->chat_id
                                      : f == 2 ? (int64_t)rec->view_count : f == 3 ? (int64_t)rec->share_count : d.ncomments;
    const uint32_t fo = f ? 16u + (f >= 2 ? 16u * f : 0u) : 0u;
    rb[128 + f] = (uint8_t)render_i64(rb + fo, v);
  }
  rb[128 + F_TIME] = (uint8_t)render_time(rb + 96, rec->date, 0, cfg.tz);  // tdutils.go:417

  const uint64_t line_start = (uint64_t)(uintptr_t)out + line_off[r];
  const uint32_t total = (uint32_t)(line_off[r + 1] - line_off[r]);
  ls_begin(s, active ? line_start : 0ull);

  // One state machine over (piece, sub-step) with a single copy loop behind it: every piece -- literal,
  // rendered field, channel / context string, message string, map entry, outlink -- is described as
  // "skip g bytes, then copy n bytes from src" (src: any address space, any alignment), so the shift
  // network of ls_append exists once in the kernel (instruction-cache footprint, see profiles/README.md).
  // Map entries and outlinks are composed in the lane's field row first: every rendered field has been
  // used by the time the comments / reactions / outlinks pieces come (they follow all K_FIELD pieces).
  uint32_t p = 0, t = 0;
  uint32_t multi_n = 0, multi_max = 0;  // entries of the current multi-step piece: this lane's / the warp's maximum
  uint32_t map_nr = 0;                  // reactions: entries in the lane's table (>= multi_n when keys repeat)
  uint64_t prev = 0;                    // reactions: compare key of the entry emitted last
  while (p < (uint32_t)kTgLaneNPieces) {
    const uint32_t en = sh.pieces[p];
    const uint32_t kind = en & 15u, arg = (en >> 4) & 15u;
    const bool on = ((condmask >> ((en >> 8) & 15u)) & 1u) != 0;
    const uint8_t* src = nullptr;
    uint32_t n = 0, g = 0;
    bool more = false, padded = true;  // padded: the source is zero beyond n up to the next 16-byte boundary
    if (kind == K_LIT) {
      src = (const uint8_t*)(sh.tmpl + ((en >> 12) & 0x7FFu));
      n = on ? en >> 23 : 0u;
    } else if (kind == K_FIELD) {
      src = rb + (arg ? 16u + (arg >= 2 ? 16u * arg : 0u) : 0u);
      n = on ? rb[128 + arg] : 0u;
    } else if (kind == K_POSTTYPE) {
      src = (const uint8_t*)(sh.ptype + 2u * ct);
      n = on ? kPostTypeLen[ct] : 0u;
    } else if (kind == K_CHAN) {
      const uint32_t o = arg == 0 ? 0u : arg == 1 ? pad16(cd.user_len) : arg == 2 ? pad16(cd.user_len) + pad16(cd.name_len)
                                                             : pad16(cd.user_len) + pad16(cd.name_len) + pad16(cd.title_len);
      src = b.chan_blob + cd.off + o;
      n = !on ? 0u : arg == 0 ? cd.user_len : arg == 1 ? cd.name_len : arg == 2 ? cd.title_len : cd.cdata_len;
      copied += n;
    } else if (kind == K_CFG) {
      src = cfg.blob + (arg == 0 ? cfg.off[0] : arg == 1 ? cfg.off[1] : arg == 2 ? cfg.off[2] : cfg.off[3]);
      n = !on ? 0u : arg == 0 ? cfg.label_len : arg == 1 ? cfg.created_tg_len : arg == 2 ? cfg.created_yt_len : cfg.capture_len;
      copied += n;
    } else if (kind == K_ESC) {  // a string of the record: copied here if it needs no escaping and is short
      const uint8_t* sp = arg == XL_DESC ? d.desc : arg == XL_MEDIA ? a.v.media : arg == XL_HANDLE ? a.v.handle : a.v.alt;
      const uint32_t sn = arg == XL_DESC ? d.desc_len : arg == XL_MEDIA ? a.v.media_len : arg == XL_HANDLE ? a.v.handle_len : a.v.alt_len;
      uint32_t xl = 0;
      if (active) {
        xpos_g[arg] = (uint32_t)(s.pos - line_start);
        if (on) xl = xlen_g[arg];
      }
      const bool mine = on && xl == sn && sn <= LANE_TEXT_MAX;  // same rule in emit_tg_escapes
      g = mine ? 0u : xl;                                       // else the esc kernel writes it
      if (g) left |= 1u << arg;
      if (mine) {
        src = sp;
        n = sn;
        copied += sn;
      }
      padded = false;
    } else if (kind == K_COMMENTS) {  // nil -> null, empty -> []; a real list is left to the maps kernel
      const bool mine = on && (d.comments_nil || d.c1 == d.c0);
      if (active) {
        xpos_g[XL_COMMENTS] = (uint32_t)(s.pos - line_start);
        if (on && !mine) g = xlen_g[XL_COMMENTS];
      }
      if (mine) {
        *(uint4*)(rb + 96) = make_uint4(d.comments_nil ? 0x6c6c756eu : 0x5d5bu, 0, 0, 0);
        src = rb + 96;
        n = d.comments_nil ? 4u : 2u;
      }
    } else if (kind == K_REACTIONS) {  // map[string]int, keys in byte order (see size_reaction_map for "simple")
      uint4* ent = (uint4*)row;        // entry table: key (8 bytes), count, key length
      uint8_t* sc = rb + 96;           // 32 bytes to compose one entry in
      if (t == 0) {
        const uint32_t r0 = b.react_off[r], nr = b.react_off[r + 1] - r0;
        bool mine = false;
        if (active) {
          xpos_g[XL_REACTIONS] = (uint32_t)(s.pos - line_start);
          mine = on && (nr == 0 || (xlen_g[XL_FLAGS] & XLF_SIMPLE_MAP));
          if (on && !mine) g = xlen_g[XL_REACTIONS];
        }
        const uint32_t nn = mine ? nr : 0u;  // <= LANE_MAP_MAX
        map_nr = nn;
        const uint32_t nmax = __reduce_max_sync(FULL, nn);
        for (uint32_t j = 0; j < nmax; j++) {
          if (j < nn) {
            const tgi_reaction rc = b.reacts[r0 + j];
            const uint8_t* kp = b.aux + rc.emoji_off;
            const uint32_t kl = rc.emoji_len;
            uint32_t k0 = ld_u32_unaligned(kp), k1 = kl > 4 ? ld_u32_unaligned(kp + 4) : 0u;
            if (kl < 4) k0 &= (1u << (8u * kl)) - 1u;
            if (kl > 4 && kl < 8) k1 &= (1u << (8u * (kl - 4u))) - 1u;
            ent[j] = make_uint4(k0, k1, (uint32_t)rc.count, kl);
          }
        }
        // entries to emit = distinct keys (a later entry of the same key overwrites the earlier one)
        uint32_t live = 0;
        for (uint32_t j = 0; j < nmax; j++) {
          if (j < nn) {
            const uint4 e = ent[j];
            bool last = true;
            for (uint32_t i = j + 1; i < nn; i++) {
              const uint4 f = ent[i];
              if (f.x == e.x && f.y == e.y && f.w == e.w) last = false;
            }
            live += last ? 1u : 0u;
          }
        }
        multi_n = live;
        multi_max = __reduce_max_sync(FULL, multi_n);
        if (mine) {
          *(uint4*)sc = make_uint4(multi_n ? 0x7bu : 0x7d7bu, 0, 0, 0);  // { or {}
          src = sc;
          n = multi_n ? 1u : 2u;
        }
        prev = 0;  // keys are non-empty and contain no NUL: every compare key is > 0
      } else if (t <= multi_n) {  // entry t-1 in key order:  "key":count, or "key":count}
        uint4 be = make_uint4(0, 0, 0, 0);
        uint64_t best = ~0ull;
        for (uint32_t j = 0; j < LANE_MAP_MAX; j++) {
          if (j < map_nr) {
            const uint4 e = ent[j];
            const uint64_t ck = ((uint64_t)__byte_perm(e.x, 0, 0x0123) << 32) | __byte_perm(e.y, 0, 0x0123);
            if (ck > prev && ck <= best) {  // <=: the last entry of a key wins
              best = ck;
              be = e;
            }
          }
        }
        prev = best;
        const uint32_t kl = be.w;
        *(uint4*)sc = make_uint4(0x22u | (be.x << 8), (be.x >> 24) | (be.y << 8), be.y >> 24, 0);
        *(uint4*)(sc + 16) = make_uint4(0, 0, 0, 0);
        sc[1 + kl] = '"';
        sc[2 + kl] = ':';
        const uint32_t dl = (uint32_t)render_i64(sc + 3 + kl, (int64_t)(int32_t)be.z);
        sc[3 + kl + dl] = t == multi_n ? '}' : ',';
        src = sc;
        n = 4u + kl + dl;
      }
      more = t < multi_max;
      padded = false;
    } else {  // K_OUTLINKS: "name","name" (the names are [a-z0-9_], tg_links.cuh)
      if (t == 0) {
        const bool mine = on && nl <= LANE_LINKS_MAX;
        if (active) {
          xpos_g[XL_OUTLINKS] = (uint32_t)(s.pos - line_start);
          if (on && !mine) g = xlen_g[XL_OUTLINKS];
        }
        multi_n = mine ? nl : 0u;
        multi_max = __reduce_max_sync(FULL, multi_n);
      }
      if (t < multi_n) {  // compose  ,"name"  (without the comma for the first) in the field row
        const uint32_t* lw = (const uint32_t*)(links + t);
        const uint32_t len = links[t].len, lead = t ? 2u : 1u;
        uint8_t* sc = rb;
        sc[0] = t ? ',' : '"';
        sc[1] = '"';
#pragma unroll 1
        for (uint32_t k = 0; k < len; k += 4) {  // the name field is zero padded to 32 bytes
          const uint32_t w = __ldg(lw + (k >> 2));
          sc[lead + k] = (uint8_t)w;
          sc[lead + k + 1] = (uint8_t)(w >> 8);
          sc[lead + k + 2] = (uint8_t)(w >> 16);
          sc[lead + k + 3] = (uint8_t)(w >> 24);
        }
        sc[lead + len] = '"';
        src = sc;
        n = lead + len + 1u;
      }
      more = t + 1 < multi_max;
      padded = false;
    }
    if (g && kind != K_ESC) left |= 16u;  // a comment list, a map or an outlink list for the maps kernel
    ls_skip(s, g);
    gaps += g;
    {  // the copy loop: one aligned 16-byte block of the source per step, bytes [0, n) of src
      const uint32_t s0 = (uint32_t)(uintptr_t)src & 15u;
      const uint4* A = (const uint4*)(src - s0);
      const uint32_t steps = __reduce_max_sync(FULL, n ? (s0 + n + 15u) >> 4 : 0u);
      uint32_t rem = n, first = s0;
      for (uint32_t i = 0; i < steps; i++, A++) {
        if (rem) {
          uint4 w = *A;
          if (first) w = shr128_bytes(w, first);
          const uint32_t k = min(rem, 16u - first);
          if (k < 16u && !padded) w = mask128(w, k);
          ls_append(s, w, k);
          rem -= k;
          first = 0;
        }
        ls_maybe_drain(s);
      }
    }
    if (more) {
      t++;
    } else {
      p++;
      t = 0;
    }
  }
  ls_flush(s);
  ls_drain_warp(s);
  if (active) {
    if ((uint32_t)(s.pos - line_start) != total) atomicOr(err, ERR_LINE_MISMATCH);
    bytes_out += total - gaps;
    bytes_in += copied;
  }
}

}  // namespace tgi
