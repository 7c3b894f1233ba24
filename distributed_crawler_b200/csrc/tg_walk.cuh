// tg_walk.cuh — the Telegram Post line: closed-form length (parse kernel) and table-driven emission
// (emit kernel), both derived from the same generated piece table (tools/gen_pieces.py).
//
// Replaces telegramhelper/tdutils.go:380-732 ParseMessage (field map :633-717) followed by
// json.Marshal(post)+'\n' (state/storageproviders.go:276-282, state/daprstate.go:1118-1120) for
// model.Post (model/data.go:9-75).  Key order = struct declaration order; see SURVEY Appendix A.6
// for the encoding/json rules restated in dev_common.cuh.
#pragma once
#include <cstddef>

#include "dev_common.cuh"
#include "tg_links.cuh"

namespace tgi {

// per-channel strings pre-rendered once per batch by the channel job
// the four segments start 16-byte aligned and are zero padded (the lane emitter fetches them in
// 16-byte blocks): segment k starts at off + sum_{j<k} pad16(len_j)
DEVI uint32_t pad16(uint32_t x) { return (x + 15u) & ~15u; }
struct ChanDerived {
  uint64_t off;        // into chan_blob: esc_user | esc_name | "esc_title" | cdata
  uint32_t user_len;   // JSON-escaped ActiveUsernames[0] (0 = no public link)
  uint32_t name_len;   // JSON-escaped channelName
  uint32_t title_len;  // "esc(chat.Title)" with quotes
  uint32_t cdata_len;  // ,"channel_name":...,"published_at":"0001-01-01T00:00:00Z"}
};

struct TgBatchDev {
  uint64_t n;
  const tgi_tg_rec* recs;
  const uint8_t* strs;
  const uint32_t* ent_off;
  const tgi_entity* ents;
  const uint32_t* react_off;
  const tgi_reaction* reacts;
  const uint32_t* comment_off;
  const tgi_comment* comments;
  const uint8_t* aux;
  uint32_t n_chans;
  const tgi_tg_chan* chans;
  const uint8_t* chan_strs;
  const ChanDerived* chan_derived;
  const uint8_t* chan_blob;
};

struct CfgDev {             // per-context constants in a small device blob
  const uint8_t* blob;      // label_esc | created_tg | created_yt | capture: 16-byte aligned, zero padded
  uint32_t off[4];          // segment offsets into blob
  uint32_t label_len;       // JSON-escaped crawl_label (no quotes)
  uint32_t created_tg_len;  // quoted RFC3339 of created_at.UTC().Truncate(s)
  uint32_t created_yt_len;  // quoted RFC3339Nano of created_at in the local zone
  uint32_t capture_len;     // quoted RFC3339Nano of capture_time
  uint32_t flags;           // TGI_CFG_*; bit 31: injected clock not representable (Marshal error)
  int32_t tz;
  int64_t min_post_date;
};
#define CFGDEV_CLOCK_INVALID 0x80000000u

__device__ const char kPostType[TGI_CT__COUNT][28] = {
    "unknown",          "messageText",          "messageVideo",           "messagePhoto",
    "messageAnimation", "messageAnimatedEmoji", "messagePoll",            "messageGiveaway",
    "messagePaidMedia", "messageSticker",       "messageGiveawayWinners", "messageGiveawayCompleted",
    "messageVideoNote", "messageDocument",      "messageAudio",           "messageVoiceNote",
    ""};
__device__ const uint8_t kPostTypeLen[TGI_CT__COUNT] = {7, 11, 12, 12, 16, 20, 11, 15, 16, 14, 22, 24, 16, 15, 12, 16, 0};

// per-warp shared scratch of the emitting kernels
struct WarpScratch {
  uint8_t field[8][40];    // rendered numeric / time fields (F_*)
  uint32_t flen[8];        // their lengths
  uint64_t src_ptr[8];     // global sources: chan segments 0..3, cfg segments 4..7
  uint32_t src_len[8];
  uint32_t xlen[8];        // emitted lengths of the variable pieces (XL_*), computed by the size kernel
  uint32_t vshift[64];     // per piece: output offset - template offset (literal pieces), or VSHIFT_SKIP
};
struct MapScratch {        // maps kernel: per-lane rendered map entries  "key":count
  uint8_t rslot[32][64];
  uint8_t num[2][16];
};

enum { K_LIT, K_FIELD, K_CHAN, K_CFG, K_ESC, K_POSTTYPE, K_COMMENTS, K_REACTIONS, K_OUTLINKS };
enum { C_NONE, C_USER, C_ALBUM, C_CT_OTHER, C_NOT_CT_OTHER, C_HAS_MEDIA };
enum { F_MSGNO, F_CHAT, F_VIEW, F_SHARE, F_NCOMM, F_TIME, F_POSTTYPE };
enum { XL_DESC, XL_MEDIA, XL_HANDLE, XL_ALT, XL_COMMENTS, XL_REACTIONS, XL_OUTLINKS, XL_COUNT, XL_FLAGS = 7 };
#define XLF_SIMPLE_MAP 1u  // xlen[XL_FLAGS]: the reactions map is lane-renderable (size_reaction_map)
#define XLF_DESC_EXACT 2u  // the description holds invalid UTF-8 or U+2028/9: only the exact escaper may write it
constexpr uint32_t K_NOP = 15;
#include "tg_pieces.inc"

// block-shared copies of the template and the lane-parallel entry table (filled once per CTA)
#define VSHIFT_SKIP 0x80000000u
struct CtaShared {
  uint32_t ents[kTgNEnt];
  uint32_t tmpl[kTgNWords];
  uint16_t wmeta[kTgNWords];
};

// ---- map[string]int (reactions) ------------------------------------------------------------------
// encoding/json sorts map keys bytewise; later duplicates of a key overwrite earlier ones (Go map
// assignment, tdutils.go:598).  Up to 32 entries per map (checked in the parse kernel).
DEVI int key_cmp(const uint8_t* a, uint32_t la, const uint8_t* b, uint32_t lb) {
  uint32_t m = la < lb ? la : lb;
  for (uint32_t i = 0; i < m; i++) {
    uint32_t x = ldb(a + i), y = ldb(b + i);
    if (x != y) return x < y ? -1 : 1;
  }
  return la < lb ? -1 : (la > lb ? 1 : 0);
}

struct MapLane {  // one map entry per lane
  const uint8_t* kp;
  uint32_t kl;
  int32_t cnt;
  bool live;       // last occurrence of its key
  uint32_t rank;   // position among the live keys in bytewise order
  uint32_t nlive;
};
DEVI MapLane warp_map_prepare(const tgi_reaction* reacts, uint32_t r0, uint32_t r1, const uint8_t* aux, bool want_rank) {
  int l = lane_id();
  uint32_t n = r1 - r0;
  if (n > 32) n = 32;
  MapLane m;
  m.kp = nullptr;
  m.kl = 0;
  m.cnt = 0;
  if ((uint32_t)l < n) {
    tgi_reaction rc = reacts[r0 + l];
    m.kp = aux + rc.emoji_off;
    m.kl = rc.emoji_len;
    m.cnt = rc.count;
  }
  m.live = (uint32_t)l < n;
  for (uint32_t j = 1; j < n; j++) {
    const uint8_t* pj = (const uint8_t*)__shfl_sync(FULL, (unsigned long long)m.kp, j);
    uint32_t lj = __shfl_sync(FULL, m.kl, j);
    if ((uint32_t)l < j && m.live && key_cmp(m.kp, m.kl, pj, lj) == 0) m.live = false;
  }
  uint32_t livemask = __ballot_sync(FULL, m.live);
  m.nlive = __popc(livemask);
  m.rank = 0;
  if (want_rank) {
    for (uint32_t j = 0; j < n; j++) {
      if (!((livemask >> j) & 1u)) continue;
      const uint8_t* pj = (const uint8_t*)__shfl_sync(FULL, (unsigned long long)m.kp, j);
      uint32_t lj = __shfl_sync(FULL, m.kl, j);
      if (m.live && (uint32_t)l != j && key_cmp(pj, lj, m.kp, m.kl) < 0) m.rank++;
    }
  }
  return m;
}

// ---- maps with more than 32 entries (no format limit: the reference builds map[string]int from however many
// reactions TDLib delivers) ----------------------------------------------------------------------------------------
// Entries are visited 32 at a time; every entry looks at all the others (quadratic, warp-parallel, keys read through
// L1): live = no later entry has the same key; rank = live entries with a smaller key.  Rare by construction.
struct BigMapEntry {
  bool live;
  uint32_t rank, before;  // before = bytes of the live entries that sort in front of this one (with their commas)
  uint32_t len;           // "key":count
};
DEVI BigMapEntry big_map_entry(const tgi_reaction* reacts, uint32_t r0, uint32_t r1, const uint8_t* aux, uint32_t i, bool want_order) {
  BigMapEntry m;
  const tgi_reaction me = reacts[i];
  const uint8_t* kp = aux + me.emoji_off;
  m.live = true;
  for (uint32_t j = i + 1; j < r1 && m.live; j++) {
    const tgi_reaction o = reacts[j];
    if (o.emoji_len == me.emoji_len && key_cmp(aux + o.emoji_off, o.emoji_len, kp, me.emoji_len) == 0) m.live = false;
  }
  m.len = m.live ? 3u + thread_esc_len(kp, me.emoji_len) + ndigits_i64(me.count) : 0u;
  m.rank = 0;
  m.before = 0;
  if (want_order && m.live) {
    for (uint32_t j = r0; j < r1; j++) {
      if (j == i) continue;
      const tgi_reaction o = reacts[j];
      const uint8_t* op = aux + o.emoji_off;
      if (key_cmp(op, o.emoji_len, kp, me.emoji_len) >= 0) continue;
      bool olive = true;  // only the last occurrence of a smaller key counts
      for (uint32_t q = j + 1; q < r1 && olive; q++) {
        const tgi_reaction o2 = reacts[q];
        if (o2.emoji_len == o.emoji_len && key_cmp(aux + o2.emoji_off, o2.emoji_len, op, o.emoji_len) == 0) olive = false;
      }
      if (olive) {
        m.rank++;
        m.before += 4u + thread_esc_len(op, o.emoji_len) + ndigits_i64(o.count);
      }
    }
  }
  return m;
}
__device__ __noinline__ uint32_t size_reaction_map_big(const tgi_reaction* reacts, uint32_t r0, uint32_t r1, const uint8_t* aux) {
  uint32_t bytes = 0, nlive = 0;
  for (uint32_t i = r0 + lane_id(); i < r1; i += 32) {
    const BigMapEntry m = big_map_entry(reacts, r0, r1, aux, i, false);
    bytes += m.len;
    nlive += m.live ? 1u : 0u;
  }
  bytes = warp_sum(bytes);
  nlive = warp_sum(nlive);
  return 2u + bytes + (nlive - 1u);
}
template <class D>
__device__ __noinline__ uint32_t emit_reaction_map_big_to(D dst, const tgi_reaction* reacts, uint32_t r0, uint32_t r1, const uint8_t* aux) {
  uint32_t bytes = 0, nlive = 0;
  if (lane_id() == 0) dst.st(0, '{');
  for (uint32_t i = r0 + lane_id(); i < r1; i += 32) {
    const BigMapEntry m = big_map_entry(reacts, r0, r1, aux, i, true);
    if (!m.live) continue;
    bytes += m.len;
    nlive++;
    const tgi_reaction me = reacts[i];
    const uint8_t* kp = aux + me.emoji_off;
    uint32_t o = 1u + m.before;  // behind the brace and the smaller entries (each followed by a comma)
    dst.st(o++, '"');
    for (uint32_t q = 0; q < me.emoji_len;) {  // thread_esc without a staging buffer: one rune at a time
      const uint32_t bq = ldb(kp + q);
      if (bq < 0x80) {
        const uint32_t el = ascii_esc_len(bq);
        put_escaped(dst, o, bq, el);
        o += el;
        q++;
        continue;
      }
      const int need = utf8_valid_lead(kp, q, me.emoji_len);
      if (need == 0) {
        put_u(dst, o, 'f', 'f', 'f', 'd');
        o += 6;
        q++;
      } else if (need == 3 && bq == 0xE2 && ldb(kp + q + 1) == 0x80 && (ldb(kp + q + 2) | 1u) == 0xA9) {
        put_u(dst, o, '2', '0', '2', ldb(kp + q + 2) == 0xA8 ? '8' : '9');
        o += 6;
        q += 3;
      } else {
        for (int k = 0; k < need; k++) dst.st(o + k, ldb(kp + q + k));
        o += (uint32_t)need;
        q += (uint32_t)need;
      }
    }
    dst.st(o++, '"');
    dst.st(o++, ':');
    uint8_t num[12];
    const int nd = render_i64(num, me.count);
    for (int k = 0; k < nd; k++) dst.st(o + k, num[k]);
    o += (uint32_t)nd;
    dst.st(o, ',');  // the last entry's comma is overwritten by the closing brace below
  }
  bytes = warp_sum(bytes);
  nlive = warp_sum(nlive);
  const uint32_t total = 2u + bytes + (nlive - 1u);
  __syncwarp();
  if (lane_id() == 0) dst.st(total - 1u, '}');
  return total;
}

// *simple (optional): the map can be rendered by one lane (tg_lane.cuh): at most LANE_MAP_MAX entries,
// keys of 1..8 bytes that need no escaping, no duplicate keys
constexpr uint32_t LANE_MAP_MAX = 6;
__device__ __noinline__ uint32_t size_reaction_map(const tgi_reaction* reacts, uint32_t r0, uint32_t r1, const uint8_t* aux,
                                                   uint32_t* simple = nullptr) {
  if (r1 == r0) {
    if (simple) *simple = 1;
    return 2;
  }
  if (r1 - r0 > 32) {
    if (simple) *simple = 0;
    return size_reaction_map_big(reacts, r0, r1, aux);
  }
  MapLane m = warp_map_prepare(reacts, r0, r1, aux, false);
  const uint32_t el = m.live ? thread_esc_len(m.kp, m.kl) : 0u;
  uint32_t mine = m.live ? 3u + el + ndigits_i64(m.cnt) : 0u;  // "key":n
  if (simple) {
    const uint32_t n = r1 - r0;
    const bool ok = (uint32_t)lane_id() >= n || (m.live && el == m.kl && m.kl >= 1 && m.kl <= 8);
    *simple = (n <= LANE_MAP_MAX && __all_sync(FULL, ok)) ? 1u : 0u;
  }
  return 2u + warp_sum(mine) + (m.nlive - 1);
}

// writes the map at dst, returns its length.  Every live lane renders its own  "key":count  into a
// shared slot; the warp then concatenates the slots in key order.  D = byte sink (DstG / DstS).
template <class D>
__device__ __noinline__ uint32_t emit_reaction_map_to(D dst, MapScratch* ms, const tgi_reaction* reacts, uint32_t r0,
                                                      uint32_t r1, const uint8_t* aux) {
  if (r1 == r0) {
    put2(dst, '{', '}');
    return 2;
  }
  if (r1 - r0 > 32) return emit_reaction_map_big_to(dst, reacts, r0, r1, aux);
  int l = lane_id();
  MapLane m = warp_map_prepare(reacts, r0, r1, aux, true);
  uint32_t slot = smem_addr(ms->rslot[l]);
  uint32_t sl = 0;
  __syncwarp();
  if (m.live) {
    sts8(slot, '"');
    uint32_t k = thread_esc(m.kp, m.kl, slot + 1, 64 - 1 - 2 - 11);
    if (k != ~0u) {
      sts8(slot + 1 + k, '"');
      sts8(slot + 2 + k, ':');
      sl = 3 + k + (uint32_t)render_i64(ms->rslot[l] + 3 + k, m.cnt);
    } else {
      sl = ~0u;
    }
  }
  __syncwarp();
  uint32_t o = 0;
  put1(dst, '{');
  o++;
  for (uint32_t r = 0; r < m.nlive; r++) {
    uint32_t who = __ballot_sync(FULL, m.live && m.rank == r);
    int src = __ffs(who) - 1;
    uint32_t len = __shfl_sync(FULL, sl, src);
    if (r) {
      put1(dst.at(o), ',');
      o++;
    }
    if (len != ~0u) {
      copy_s(dst.at(o), smem_addr(ms->rslot[src]), len);
      o += len;
    } else {  // key too long for a slot: escape it cooperatively
      const uint8_t* pj = (const uint8_t*)__shfl_sync(FULL, (unsigned long long)m.kp, src);
      uint32_t lj = __shfl_sync(FULL, m.kl, src);
      int32_t cj = __shfl_sync(FULL, m.cnt, src);
      put1(dst.at(o), '"');
      o++;
      o += esc_to(dst.at(o), pj, lj);
      put2(dst.at(o), '"', ':');
      o += 2;
      uint32_t dl = 0;
      __syncwarp();
      if (l == 0) dl = (uint32_t)render_i64(ms->num[0], cj);
      __syncwarp();
      dl = __shfl_sync(FULL, dl, 0);
      copy_s(dst.at(o), smem_addr(ms->num[0]), dl);
      o += dl;
      __syncwarp();
    }
  }
  put1(dst.at(o), '}');
  return o + 1;
}
DEVI uint32_t emit_reaction_map(uint8_t* dst, MapScratch* ms, const tgi_reaction* reacts, uint32_t r0, uint32_t r1, const uint8_t* aux) {
  return emit_reaction_map_to(DstG{dst}, ms, reacts, r0, r1, aux);
}

// ---- []model.Comment --------------------------------------------------------------------------------
__device__ const char kCm0[] = "{\"text\":\"";
__device__ const char kCm1[] = "\",\"reactions\":";
__device__ const char kCm2[] = ",\"view_count\":";
__device__ const char kCm3[] = ",\"reply_count\":";
__device__ const char kCm4[] = ",\"handle\":\"";
__device__ const char kCm5[] = "\"}";
__device__ const char kNullLit[] = "null";
constexpr uint32_t kCmFixed = sizeof(kCm0) + sizeof(kCm1) + sizeof(kCm2) + sizeof(kCm3) + sizeof(kCm4) + sizeof(kCm5) - 6;

__device__ __noinline__ uint32_t size_tg_comments(const TgBatchDev& b, uint32_t c0, uint32_t c1) {
  uint32_t tot = 2 + (c1 > c0 ? c1 - c0 - 1 : 0);  // [ ] and commas
  for (uint32_t k = c0; k < c1; k++) {
    tgi_comment cm = b.comments[k];
    tot += kCmFixed + warp_esc_len(b.aux + cm.text_off, cm.text_len) + warp_esc_len(b.aux + cm.handle_off, cm.handle_len) +
           ndigits_i64(cm.view_count) + ndigits_i64(cm.reply_count) +
           ((cm.flags & 1) ? size_reaction_map(b.reacts, cm.react_start, cm.react_start + cm.react_count, b.aux) : 4u);
  }
  return tot;
}

template <class D>
__device__ __noinline__ uint32_t emit_tg_comments_to(D dst, MapScratch* ms, const TgBatchDev& b, uint32_t c0, uint32_t c1) {
  int l = lane_id();
  uint32_t o = 0;
  put1(dst, '[');
  o++;
#define CM_LIT(x)                                           \
  do {                                                      \
    copy_g(dst.at(o), (const uint8_t*)(x), sizeof(x) - 1);  \
    o += sizeof(x) - 1;                                     \
  } while (0)
  for (uint32_t k = c0; k < c1; k++) {
    tgi_comment cm = b.comments[k];
    uint32_t dl = 0;
    __syncwarp();
    if (l < 2) dl = (uint32_t)render_i64(ms->num[l], l == 0 ? cm.view_count : cm.reply_count);
    __syncwarp();
    uint32_t d0 = __shfl_sync(FULL, dl, 0), d1 = __shfl_sync(FULL, dl, 1);
    if (k > c0) {
      put1(dst.at(o), ',');
      o++;
    }
    CM_LIT(kCm0);
    o += esc_to(dst.at(o), b.aux + cm.text_off, cm.text_len);
    CM_LIT(kCm1);
    // the two counts must leave the scratch before a long-key map entry reuses it
    const uint32_t n0 = l < 12 ? ms->num[0][l] : 0u, n1 = l < 12 ? ms->num[1][l] : 0u;
    __syncwarp();
    if (cm.flags & 1) o += emit_reaction_map_to(dst.at(o), ms, b.reacts, cm.react_start, cm.react_start + cm.react_count, b.aux);
    else CM_LIT(kNullLit);
    CM_LIT(kCm2);
    if ((uint32_t)l < d0) dst.st(o + l, n0);
    o += d0;
    CM_LIT(kCm3);
    if ((uint32_t)l < d1) dst.st(o + l, n1);
    o += d1;
    CM_LIT(kCm4);
    o += esc_to(dst.at(o), b.aux + cm.handle_off, cm.handle_len);
    CM_LIT(kCm5);
    __syncwarp();
  }
#undef CM_LIT
  put1(dst.at(o), ']');
  return o + 1;
}
DEVI uint32_t emit_tg_comments(uint8_t* dst, MapScratch* ms, const TgBatchDev& b, uint32_t c0, uint32_t c1) {
  return emit_tg_comments_to(DstG{dst}, ms, b, c0, c1);
}

template <class D>
DEVI uint32_t emit_tg_outlinks_to(D dst, const tgi_link* links, uint32_t n) {
  uint32_t o = 0;
  for (uint32_t k = 0; k < n; k++) {
    uint32_t len = links[k].len;
    if (k) {
      put2(dst.at(o), ',', '"');
      o += 2;
    } else {
      put1(dst.at(o), '"');
      o += 1;
    }
    copy_g(dst.at(o), links[k].name, len);  // [a-z0-9_] only: no escaping needed
    o += len;
    put1(dst.at(o), '"');
    o += 1;
  }
  return o;
}
DEVI uint32_t emit_tg_outlinks(uint8_t* dst, const tgi_link* links, uint32_t n) { return emit_tg_outlinks_to(DstG{dst}, links, n); }
DEVI uint32_t size_tg_outlinks(const tgi_link* links, uint32_t n) {
  if (!n) return 0;
  uint32_t s = 0;
  for (uint32_t k = lane_id(); k < n; k += 32) s += links[k].len + 2u;
  return warp_sum(s) + (n - 1);
}

// ---- record ---------------------------------------------------------------------------------------
struct TgWalkArgs {
  const TgBatchDev* b;
  const CfgDev* cfg;
  uint64_t r;
  TgRecView v;
  const tgi_link* links;  // this record's outlinks (arena)
  uint32_t n_links;
};

struct TgDerived {  // what both passes need to know about a record
  const uint8_t* desc;
  uint32_t desc_len;
  bool has_media, has_user, album, comments_nil;
  uint32_t c0, c1;
  int64_t ncomments;
};
DEVI TgDerived tg_derive(const TgWalkArgs& a, const ChanDerived& cd) {
  TgDerived d;
  const TgBatchDev& b = *a.b;
  d.c0 = b.comment_off[a.r];
  d.c1 = b.comment_off[a.r + 1];
  d.comments_nil = (a.v.flags & TGI_RF_COMMENTS_NIL) != 0;
  d.ncomments = d.comments_nil ? 0 : (int64_t)(d.c1 - d.c0);
  // description / media by content type (tdutils.go:443-587)
  d.desc = nullptr;
  d.desc_len = 0;
  uint32_t ct = a.v.ct;
  if (ct == TGI_CT_TEXT || ct == TGI_CT_VIDEO || ct == TGI_CT_PHOTO || ct == TGI_CT_ANIMATION) {
    if (a.v.flags & TGI_RF_HAS_TEXT) { d.desc = a.v.text; d.desc_len = a.v.text_len; }
  } else if (ct == TGI_CT_ANIMATED_EMOJI || ct == TGI_CT_POLL || ct == TGI_CT_GIVEAWAY ||
             ct == TGI_CT_PAID_MEDIA || ct == TGI_CT_DOCUMENT) {
    d.desc = a.v.alt; d.desc_len = a.v.alt_len;
  }
  d.has_media = ct == TGI_CT_VIDEO || ct == TGI_CT_VIDEO_NOTE || ct == TGI_CT_DOCUMENT;
  d.has_user = cd.user_len != 0;
  d.album = d.has_user && a.v.rec->media_album_id != 0;
  return d;
}

// line length in bytes; 0 if a time field is not representable (Marshal error -> TGI_ST_NOLINE).
// The formula's coefficients come from the generated piece table, so it cannot drift from emit.
DEVI uint32_t size_tg_record(const TgWalkArgs& a, uint32_t* xl) {
  const TgBatchDev& b = *a.b;
  const CfgDev& cfg = *a.cfg;
  const tgi_tg_rec* rec = a.v.rec;
  const ChanDerived cd = b.chan_derived[rec->chan_idx];
  TgDerived d = tg_derive(a, cd);
  if (cfg.flags & CFGDEV_CLOCK_INVALID) return 0;
  // int32 dates are always inside year [0,9999]: RFC3339 with quotes, 'Z' or a +hh:mm offset
  uint32_t L[8] = {ndigits_i64(rec->id / 1048576), ndigits_i64(rec->chat_id), ndigits_i64(rec->view_count),
                   ndigits_i64(rec->share_count), ndigits_i64(d.ncomments), cfg.tz == 0 ? 22u : 27u, 0, 0};
  uint32_t chan[4] = {cd.user_len, cd.name_len, cd.title_len, cd.cdata_len};
  uint32_t cf[4] = {cfg.label_len, cfg.created_tg_len, cfg.created_yt_len, cfg.capture_len};
  uint32_t tot = tg_size_fixed(L, chan, cf, d.has_user, d.album);
  bool desc_exact = false;
  xl[XL_DESC] = warp_esc_len(d.desc, d.desc_len, &desc_exact);
  xl[XL_ALT] = a.v.ct == TGI_CT_OTHER ? warp_esc_len(a.v.alt, a.v.alt_len) : 0u;
  xl[XL_MEDIA] = d.has_media ? warp_esc_len(a.v.media, a.v.media_len) : 0u;
  xl[XL_HANDLE] = warp_esc_len(a.v.handle, a.v.handle_len);
  xl[XL_COMMENTS] = d.comments_nil ? 4u : size_tg_comments(b, d.c0, d.c1);
  uint32_t simple_map = 0;
  xl[XL_REACTIONS] = size_reaction_map(b.reacts, b.react_off[a.r], b.react_off[a.r + 1], b.aux, &simple_map);
  xl[XL_FLAGS] = (simple_map ? XLF_SIMPLE_MAP : 0u) | (desc_exact ? XLF_DESC_EXACT : 0u);
  xl[XL_OUTLINKS] = size_tg_outlinks(a.links, a.n_links);
  tot += a.v.ct == TGI_CT_OTHER ? 0u : (uint32_t)kPostTypeLen[a.v.ct];
  for (int j = 0; j < XL_COUNT; j++) tot += xl[j];
  return tot;
}

// per-record prologue: lanes render the numeric / time fields and fill the source tables
DEVI void emit_tg_prologue(WarpScratch* ws, const TgWalkArgs& a, const ChanDerived& cd, const TgDerived& d,
                           const uint32_t* xlen_g) {
  const TgBatchDev& b = *a.b;
  const CfgDev& cfg = *a.cfg;
  const tgi_tg_rec* rec = a.v.rec;
  int l = lane_id();
  __syncwarp();
  if (l < 5) {
    int64_t v = l == 0 ? rec->id / 1048576                                     // tdutils.go:1008
                       : l == 1 ? rec->chat_id
                                : l == 2 ? (int64_t)rec->view_count
                                         : l == 3 ? (int64_t)rec->share_count : d.ncomments;
    ws->flen[l] = (uint32_t)render_i64(ws->field[l], v);
  } else if (l == 5) {
    ws->flen[5] = (uint32_t)render_time(ws->field[5], rec->date, 0, cfg.tz);  // :417
  } else if (l == 6) {  // MessageContentType() string (28-byte rows, 4-byte aligned)
    const uint32_t* src = (const uint32_t*)kPostType[a.v.ct];
    uint32_t* dst = (uint32_t*)ws->field[F_POSTTYPE];
#pragma unroll
    for (int w = 0; w < 7; w++) dst[w] = src[w];
    ws->flen[F_POSTTYPE] = kPostTypeLen[a.v.ct];
  } else if (l >= 8 && l < 12) {
    int k = l - 8;
    uint32_t o = k == 0 ? 0u : k == 1 ? pad16(cd.user_len) : k == 2 ? pad16(cd.user_len) + pad16(cd.name_len)
                                                            : pad16(cd.user_len) + pad16(cd.name_len) + pad16(cd.title_len);
    ws->src_ptr[k] = (uint64_t)(uintptr_t)(b.chan_blob + cd.off + o);
    ws->src_len[k] = k == 0 ? cd.user_len : k == 1 ? cd.name_len : k == 2 ? cd.title_len : cd.cdata_len;
  } else if (l >= 12 && l < 16) {
    int k = l - 12;
    ws->src_ptr[4 + k] = (uint64_t)(uintptr_t)(cfg.blob + cfg.off[k]);
    ws->src_len[4 + k] = k == 0 ? cfg.label_len : k == 1 ? cfg.created_tg_len : k == 2 ? cfg.created_yt_len : cfg.capture_len;
  } else if (l >= 16 && l < 16 + XL_COUNT) {
    ws->xlen[l - 16] = xlen_g[l - 16];
  }
  __syncwarp();
}

DEVI uint32_t tg_condmask(const TgWalkArgs& a, const TgDerived& d) {
  return 1u | (d.has_user ? 1u << C_USER : 0) | (d.album ? 1u << C_ALBUM : 0) |
         (a.v.ct == TGI_CT_OTHER ? 1u << C_CT_OTHER : 1u << C_NOT_CT_OTHER) | (d.has_media ? 1u << C_HAS_MEDIA : 0);
}

// ---- emit, kernel 1 of 3: the fixed part of the line -----------------------------------------------
// Lane i owns pieces kTgEPL*i ..; an exclusive scan over the lanes' length sums gives each piece its
// offset in the line.  Literal pieces only publish their shift (output offset - template offset);
// the template is then copied word by word (340 words = 11 steps) with the shift of the owning
// piece.  Rendered fields are copied by their owning lane, per-channel / per-context strings
// cooperatively.  The offsets of the variable pieces are saved for kernels 2 and 3.
DEVI void emit_tg_fixed(uint8_t* line, WarpScratch* ws, const CtaShared* cs, const TgWalkArgs& a, uint32_t total,
                        const uint32_t* xlen_g, uint32_t* xpos_g, int* err) {
  const TgBatchDev& b = *a.b;
  const ChanDerived cd = b.chan_derived[a.v.rec->chan_idx];
  const TgDerived d = tg_derive(a, cd);
  emit_tg_prologue(ws, a, cd, d, xlen_g);
  const uint32_t ws_s = smem_addr(ws), ents_s = smem_addr(cs->ents), tmpl_s = smem_addr(cs->tmpl);
  const uint32_t vs_s = ws_s + (uint32_t)offsetof(WarpScratch, vshift);
  const uint32_t condmask = tg_condmask(a, d);
  const int l = lane_id();
  uint32_t ent[kTgEPL], len[kTgEPL], off[kTgEPL];
  uint32_t sum = 0;
#pragma unroll
  for (int k = 0; k < kTgEPL; k++) {
    uint32_t en = lds32(ents_s + 4u * (uint32_t)(kTgEPL * l + k));
    uint32_t kind = en & 15u, arg = (en >> 4) & 15u;
    uint32_t ln = 0;
    if ((condmask >> ((en >> 8) & 15u)) & 1u) {
      if (kind == K_LIT) ln = en >> 23;
      else if (kind == K_FIELD) ln = lds32(ws_s + (uint32_t)offsetof(WarpScratch, flen) + 4u * arg);
      else if (kind == K_POSTTYPE) ln = lds32(ws_s + (uint32_t)offsetof(WarpScratch, flen) + 4u * F_POSTTYPE);
      else if (kind == K_CHAN) ln = lds32(ws_s + (uint32_t)offsetof(WarpScratch, src_len) + 4u * arg);
      else if (kind == K_CFG) ln = lds32(ws_s + (uint32_t)offsetof(WarpScratch, src_len) + 4u * (4u + arg));
      else if (kind == K_ESC) ln = lds32(ws_s + (uint32_t)offsetof(WarpScratch, xlen) + 4u * arg);
      else if (kind == K_COMMENTS) ln = lds32(ws_s + (uint32_t)offsetof(WarpScratch, xlen) + 4u * XL_COMMENTS);
      else if (kind == K_REACTIONS) ln = lds32(ws_s + (uint32_t)offsetof(WarpScratch, xlen) + 4u * XL_REACTIONS);
      else if (kind == K_OUTLINKS) ln = lds32(ws_s + (uint32_t)offsetof(WarpScratch, xlen) + 4u * XL_OUTLINKS);
    }
    ent[k] = en;
    len[k] = ln;
    sum += ln;
  }
  uint32_t incl = warp_incl_scan(sum);
  uint32_t run = incl - sum;
#pragma unroll
  for (int k = 0; k < kTgEPL; k++) {
    off[k] = run;
    run += len[k];
  }
  if (__shfl_sync(FULL, incl, 31) != total) {  // the host reports it
    if (l == 0) atomicOr(err, ERR_LINE_MISMATCH);
    return;
  }
#pragma unroll
  for (int k = 0; k < kTgEPL; k++) {
    uint32_t kind = ent[k] & 15u, arg = (ent[k] >> 4) & 15u;
    if (kind == K_LIT) {
      sts32(vs_s + 4u * (uint32_t)(kTgEPL * l + k), len[k] ? off[k] - ((ent[k] >> 12) & 0x7FFu) : VSHIFT_SKIP);
    } else if (kind == K_FIELD || kind == K_POSTTYPE) {
      if (len[k]) {
        uint32_t src = ws_s + (uint32_t)offsetof(WarpScratch, field) + 40u * (kind == K_FIELD ? arg : F_POSTTYPE);
        uint8_t* dst = line + off[k];
        uint32_t n = len[k];
        for (uint32_t w = 0; w < n; w += 4) {
          uint32_t v = lds32(src + w);
          dst[w] = (uint8_t)v;
          if (w + 1 < n) dst[w + 1] = (uint8_t)(v >> 8);
          if (w + 2 < n) dst[w + 2] = (uint8_t)(v >> 16);
          if (w + 3 < n) dst[w + 3] = (uint8_t)(v >> 24);
        }
      }
    } else if (kind == K_ESC) {
      xpos_g[arg] = off[k];
    } else if (kind == K_COMMENTS || kind == K_REACTIONS || kind == K_OUTLINKS) {
      xpos_g[kind == K_COMMENTS ? XL_COMMENTS : kind == K_REACTIONS ? XL_REACTIONS : XL_OUTLINKS] = off[k];
    }
  }
  __syncwarp();
  {  // the template, word by word
    const uint32_t wm_s = smem_addr(cs->wmeta);
#pragma unroll 2
    for (uint32_t j = l; j < (uint32_t)kTgNWords; j += 32) {
      uint32_t m = lds16(wm_s + 2u * j);
      uint32_t sh = lds32(vs_s + 4u * (m >> 3));
      if (sh != VSHIFT_SKIP) {
        uint32_t v = lds32(tmpl_s + 4u * j);
        uint8_t* dst = line + (uint32_t)(4u * j + sh);  // sh may be "negative" mod 2^32: add in 32 bits
        uint32_t nv = m & 7u;
        dst[0] = (uint8_t)v;
        if (nv > 1) dst[1] = (uint8_t)(v >> 8);
        if (nv > 2) dst[2] = (uint8_t)(v >> 16);
        if (nv > 3) dst[3] = (uint8_t)(v >> 24);
      }
    }
  }
  for (int bi = 0; bi < kTgNCopy; bi++) {  // per-channel / per-context strings
    const uint32_t idx = kTgCopy[bi];
    const uint32_t owner = idx / kTgEPL, kk = idx % kTgEPL;
    uint32_t o_sel = off[0], l_sel = len[0];
#pragma unroll
    for (int k = 1; k < kTgEPL; k++)
      if (kk == (uint32_t)k) { o_sel = off[k]; l_sel = len[k]; }
    const uint32_t ln = __shfl_sync(FULL, l_sel, owner);
    if (ln == 0) continue;
    const uint32_t o = __shfl_sync(FULL, o_sel, owner);
    const uint32_t en = kTgPieces[idx];
    uint32_t si = ((en & 15u) == K_CFG ? 4u : 0u) + ((en >> 4) & 15u);
    gcopy_g(line + o, (const uint8_t*)(uintptr_t)ws->src_ptr[si], ln);
  }
}

// ---- emit, kernel 2 of 3: the escaped strings --------------------------------------------------------
// lane_text_max: strings that need no escaping and are at most this long were already copied by the
// lane emitter (tg_lane.cuh, same rule); 0xffffffff = none were.
// MODE splits the work between two kernels by instruction footprint: ESC_ALL = every string; ESC_SPARSE = only a
// description with few special bytes (esc_sparse_to_global); ESC_DENSE = everything else.
enum { ESC_ALL = 0, ESC_DENSE = 1, ESC_SPARSE = 2 };
constexpr uint32_t ESC_SPARSE_EXTRA = 24;  // at most this many added bytes (a line break adds 1, a control character 5)
DEVI bool esc_desc_is_sparse(uint32_t xl, uint32_t n, uint32_t flags) { return xl > n && xl - n <= ESC_SPARSE_EXTRA && !(flags & XLF_DESC_EXACT); }
template <int MODE>
DEVI void emit_tg_escapes(uint8_t* line, const TgWalkArgs& a, const uint32_t* xlen_g, const uint32_t* xpos_g, uint32_t lane_text_max) {
  // description / media by content type (tdutils.go:443-587), as in tg_derive
  const uint32_t ct = a.v.ct;
  const uint8_t* desc = nullptr;
  uint32_t desc_len = 0;
  if (ct == TGI_CT_TEXT || ct == TGI_CT_VIDEO || ct == TGI_CT_PHOTO || ct == TGI_CT_ANIMATION) {
    if (a.v.flags & TGI_RF_HAS_TEXT) { desc = a.v.text; desc_len = a.v.text_len; }
  } else if (ct == TGI_CT_ANIMATED_EMOJI || ct == TGI_CT_POLL || ct == TGI_CT_GIVEAWAY ||
             ct == TGI_CT_PAID_MEDIA || ct == TGI_CT_DOCUMENT) {
    desc = a.v.alt; desc_len = a.v.alt_len;
  }
  uint32_t myl = 0, myp = 0;
  if (lane_id() < 4) {
    myl = xlen_g[lane_id()];
    myp = xpos_g[lane_id()];
  }
#pragma unroll
  for (int j = 0; j < (MODE == ESC_SPARSE ? 1 : 4); j++) {  // XL_DESC, XL_MEDIA, XL_HANDLE, XL_ALT
    uint32_t ln = __shfl_sync(FULL, myl, j);
    if (ln == 0) continue;
    uint32_t o = __shfl_sync(FULL, myp, j);
    const uint8_t* p = j == 0 ? desc : j == 1 ? a.v.media : j == 2 ? a.v.handle : a.v.alt;
    uint32_t n = j == 0 ? desc_len : j == 1 ? a.v.media_len : j == 2 ? a.v.handle_len : a.v.alt_len;
    if (MODE != ESC_ALL && j == 0) {
      const bool sparse = esc_desc_is_sparse(ln, n, xlen_g[XL_FLAGS]);
      if (MODE == ESC_SPARSE) {
        if (sparse) esc_sparse_to_global(line + o, p, n);
        continue;
      }
      if (sparse) continue;  // ESC_DENSE: the other kernel writes it
    }
    if (ln == n) {  // nothing to escape
      if (n <= lane_text_max && lane_text_max != 0xffffffffu) continue;
      if (n >= 64) {
        warp_copy_vec(line + o, p, n);
        continue;
      }
    }
    if (j == 0 && !(xlen_g[XL_FLAGS] & XLF_DESC_EXACT)) esc_ascii_to_global(line + o, p, n);
    else esc_to_global(line + o, p, n);
  }
}

// ---- channel job: the per-channel constant strings, rendered once per batch ----------------------
// blob layout per channel: esc(username) | esc(channelName) | "esc(title)" | channel_data tail
__device__ const char kCd0[] = ",\"channel_name\":\"";
__device__ const char kCd1[] = "\",\"channel_description\":\"\",\"channel_profile_image\":\"\",\"channel_engagement_data\":{\"follower_count\":";
__device__ const char kCd2[] = ",\"following_count\":0,\"like_count\":0,\"post_count\":";
__device__ const char kCd3[] = ",\"views_count\":";
__device__ const char kCd4[] = ",\"comment_count\":0,\"share_count\":0},\"channel_url_external\":\"https://t.me/c/";
__device__ const char kCd5[] = "\",\"channel_url\":\"https://t.me/c/";
__device__ const char kCd6[] = "\",\"country_code\":\"\",\"published_at\":\"0001-01-01T00:00:00Z\"}";
constexpr uint32_t kCdFixed = sizeof(kCd0) + sizeof(kCd1) + sizeof(kCd2) + sizeof(kCd3) + sizeof(kCd4) + sizeof(kCd5) + sizeof(kCd6) - 7;

DEVI ChanDerived size_tg_chan(const TgBatchDev& b, uint32_t c) {
  const tgi_tg_chan ch = b.chans[c];
  const uint8_t* cs = b.chan_strs + ch.str_off;
  uint32_t et = warp_esc_len(cs, ch.title_len), en = warp_esc_len(cs + ch.title_len, ch.name_len),
           eu = warp_esc_len(cs + ch.title_len + ch.name_len, ch.user_len);
  ChanDerived d;
  d.off = 0;
  d.user_len = eu;
  d.name_len = en;
  d.title_len = et + 2;
  d.cdata_len = kCdFixed + et + 2 * en + ndigits_i64(ch.member_count) + ndigits_i64(ch.post_count) + ndigits_i64(ch.view_count);
  return d;
}

DEVI void emit_tg_chan(uint8_t* dst, WarpScratch* ws, const TgBatchDev& b, uint32_t c) {
  const tgi_tg_chan ch = b.chans[c];
  const uint8_t* cs = b.chan_strs + ch.str_off;
  const uint8_t *title = cs, *name = cs + ch.title_len, *user = name + ch.name_len;
  int l = lane_id();
  __syncwarp();
  if (l < 3) ws->flen[l] = (uint32_t)render_i64(ws->field[l], l == 0 ? ch.member_count : l == 1 ? ch.post_count : ch.view_count);
  __syncwarp();
  uint32_t L0 = ws->flen[0], L1 = ws->flen[1], L2 = ws->flen[2];
  uint32_t o = 0;
#define CH_LIT(x)                                    \
  do {                                               \
    gcopy_g(dst + o, (const uint8_t*)(x), sizeof(x) - 1); \
    o += sizeof(x) - 1;                              \
  } while (0)
  o += esc_to_global(dst + o, user, ch.user_len);
  o = pad16(o);
  o += esc_to_global(dst + o, name, ch.name_len);
  o = pad16(o);
  gput1(dst + o, '"');
  o++;
  o += esc_to_global(dst + o, title, ch.title_len);
  gput1(dst + o, '"');
  o++;
  o = pad16(o);
  CH_LIT(kCd0);
  o += esc_to_global(dst + o, title, ch.title_len);
  CH_LIT(kCd1);
  gcopy_s(dst + o, smem_addr(ws->field[0]), L0);
  o += L0;
  CH_LIT(kCd2);
  gcopy_s(dst + o, smem_addr(ws->field[1]), L1);
  o += L1;
  CH_LIT(kCd3);
  gcopy_s(dst + o, smem_addr(ws->field[2]), L2);
  o += L2;
  CH_LIT(kCd4);
  o += esc_to_global(dst + o, name, ch.name_len);
  CH_LIT(kCd5);
  o += esc_to_global(dst + o, name, ch.name_len);
  CH_LIT(kCd6);
#undef CH_LIT
  __syncwarp();
}

}  // namespace tgi
