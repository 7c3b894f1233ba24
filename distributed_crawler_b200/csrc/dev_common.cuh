// dev_common.cuh — warp-level building blocks shared by the ingest kernels (sm_100a).
//
// Everything here is integer/byte work on HBM-resident packed batches (include/tgingest.h).
// Convention: functions named warp_* are warp-collective (all 32 lanes call them with
// warp-uniform arguments unless stated otherwise).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tgingest.h"

#define FULL 0xffffffffu
#define DEVI __device__ __forceinline__

namespace tgi {

// Error bits the kernels atomicOr into a batch's error word, and the layout of the batch's scalars block (u64 words,
// zeroed before the batch; the host reads it back).  SC_CURSOR holds the link-arena cursor (u32) and the error word (int).
enum : int {
  ERR_ARENA_OVERFLOW = 1,
  ERR_TOO_MANY_REACTIONS = 2,
  ERR_FRONTIER_FULL = 4,
  ERR_TOO_MANY_LINKS = 8,
  ERR_LINE_MISMATCH = 16,  // sized and emitted line lengths disagree: never expected
  ERR_PAGE_OVERFLOW = 64,  // a page does not fit its result block: the host reruns it on the bulk pipeline
  SC_CHAN_TOTAL = 0, SC_LINE_TOTAL = 1, SC_CURSOR = 2, SC_NEW = 3, SC_FSIZE = 4, SC_LINK_TOTAL = 5, SC_LONG = 6,
  SC_URL_CURSOR = 7, SC_LANE_OUT = 8, SC_LANE_IN = 9, SC_LISTS = 10 /* 3 x u32 */, SC_COUNT = 12,
  PAGE_TRACE_AT = 16,  // page kernels: phase clock and slowest records behind the scalars (TGI_PAGE_TRACE)
};

DEVI int lane_id() { return (int)(threadIdx.x & 31); }

// ---- global byte / word loads (read-only path) ---------------------------------------------------
DEVI uint32_t ldb(const uint8_t* p) { return (uint32_t)__ldg(p); }

// 4 bytes at arbitrary alignment, little-endian; may touch up to 3 bytes past p+3 rounded to a
// word boundary (device blobs are padded by 32 zero bytes).
DEVI uint32_t ld_u32_unaligned(const uint8_t* p) {
  uintptr_t a = (uintptr_t)p;
  const uint32_t* q = (const uint32_t*)(a & ~(uintptr_t)3);
  uint32_t sh = (uint32_t)(a & 3) * 8;
  uint32_t lo = __ldg(q);
  if (sh == 0) return lo;
  uint32_t hi = __ldg(q + 1);
  return __funnelshift_r(lo, hi, sh);
}

// ---- character classes ---------------------------------------------------------------------------
DEVI bool is_letter(uint32_t c) { return ((c | 32u) - 'a') < 26u; }
DEVI bool is_word(uint32_t c) { return is_letter(c) || (c - '0') < 10u || c == '_'; }
DEVI uint32_t ascii_lower(uint32_t c) { return (c - 'A') < 26u ? c + 32u : c; }

// Go encoding/json (escapeHTML=true, go>=1.22) output length of one ASCII byte: 1, 2 or 6.
DEVI uint32_t ascii_esc_len(uint32_t b) {
  if (b >= 0x20) {
    if (b == '"' || b == '\\') return 2;
    if (b == '<' || b == '>' || b == '&') return 6;
    return 1;
  }
  const uint32_t two = (1u << 8) | (1u << 9) | (1u << 10) | (1u << 12) | (1u << 13);
  return ((two >> b) & 1u) ? 2u : 6u;
}

// ---- exact UTF-8 decoding rules of Go's unicode/utf8 (DecodeRuneInString) -----------------------
// returns the sequence length (2..4) if a VALID sequence starts at s[i], else 0.  s[i] >= 0x80.
__device__ __noinline__ int utf8_valid_lead(const uint8_t* s, int64_t i, int64_t n) {
  uint32_t b0 = ldb(s + i);
  if (b0 < 0xC2 || b0 > 0xF4) return 0;
  int need = b0 < 0xE0 ? 2 : (b0 < 0xF0 ? 3 : 4);
  if (i + need > n) return 0;
  uint32_t b1 = ldb(s + i + 1);
  uint32_t lo = 0x80, hi = 0xBF;
  if (b0 == 0xE0) lo = 0xA0;
  if (b0 == 0xED) hi = 0x9F;
  if (b0 == 0xF0) lo = 0x90;
  if (b0 == 0xF4) hi = 0x8F;
  if (b1 < lo || b1 > hi) return 0;
  if (need >= 3 && (ldb(s + i + 2) & 0xC0) != 0x80) return 0;
  if (need == 4 && (ldb(s + i + 3) & 0xC0) != 0x80) return 0;
  return need;
}

// Exact classification of byte i of string s[0..n):
//   esc : bytes this input byte contributes to the JSON-escaped output (0,1,2,6)
//   u16 : UTF-16 code units it contributes in utf16OffsetToBytes (tdutils.go:55-78) (0,1,2)
//   start: 1 if a rune starts here (Go's loop visits this index)
struct ByteInfo {
  uint32_t esc, u16, start;
};
__device__ __noinline__ ByteInfo byte_info_exact(const uint8_t* s, int64_t i, int64_t n) {
  ByteInfo r;
  uint32_t b = ldb(s + i);
  if (b < 0x80) {
    r.esc = ascii_esc_len(b);
    r.u16 = 1;
    r.start = 1;
    return r;
  }
  if ((b & 0xC0) == 0x80) {  // continuation byte: consumed iff a valid lead precedes it closely enough
    for (int d = 1; d <= 3; d++) {
      if (i - d < 0) break;
      uint32_t p = ldb(s + i - d);
      if ((p & 0xC0) == 0x80) continue;  // another continuation: keep looking back
      if (p >= 0xC2) {
        int need = utf8_valid_lead(s, i - d, n);
        if (need > d) {  // covered
          bool ls = (need == 3 && p == 0xE2 && ldb(s + i - d + 1) == 0x80 &&
                     (ldb(s + i - d + 2) | 1u) == 0xA9);  // U+2028 / U+2029
          r.esc = ls ? 0 : 1;
          r.u16 = 0;
          r.start = 0;
          return r;
        }
      }
      break;  // nearest non-continuation byte decides
    }
    r.esc = 6;
    r.u16 = 1;
    r.start = 1;
    return r;
  }
  int need = utf8_valid_lead(s, i, n);
  if (need == 0) {
    r.esc = 6;  // �
    r.u16 = 1;
    r.start = 1;
    return r;
  }
  bool ls = (need == 3 && b == 0xE2 && ldb(s + i + 1) == 0x80 && (ldb(s + i + 2) | 1u) == 0xA9);
  r.esc = ls ? 6 : 1;
  r.u16 = need == 4 ? 2 : 1;
  r.start = 1;
  return r;
}

// ---- warp scans / reductions ---------------------------------------------------------------------
DEVI uint32_t warp_incl_scan(uint32_t v) {
  int l = lane_id();
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(FULL, v, d);
    if (l >= d) v += t;
  }
  return v;
}
DEVI uint32_t warp_sum(uint32_t v) { return __reduce_add_sync(FULL, v); }

// ---- a strip = 128 consecutive bytes of a string, 4 per lane ------------------------------------
// Lane l owns bytes [base+4l, base+4l+4).  `w` holds them little-endian with bytes at index >= n
// forced to 0.  The fast path handles ASCII and every structurally valid UTF-8 sequence whose
// validity can be decided with SWAR tests (2/3/4-byte leads incl. the E0/ED/F0 second-byte ranges).
// What is left for the exact per-byte path (byte_info_exact): bytes >= 0xF4, C0/C1, E2 80 xx
// (U+2028/9 candidates) and any structural mismatch.  `exact` is warp-uniform.
struct Strip {
  uint32_t w;       // own 4 bytes
  uint32_t nvalid;  // how many of them are < n (0..4)
  bool exact;       // warp-uniform
  uint32_t cont;    // fast path: continuation-byte mask (bit 7 of each byte)
  uint32_t l4;      // fast path: 4-byte-lead mask (bit 7 of each byte)
};

DEVI uint32_t swar_has_byte(uint32_t w, uint32_t c) {  // bit7 of each byte equal to c
  uint32_t x = w ^ (c * 0x01010101u);
  return (x - 0x01010101u) & ~x & 0x80808080u;
}

// exact per-byte equality: bit 7 of every byte of w that equals c (swar_has_byte above is exact only
// as an "any" test: its borrow can flag the byte above a match)
DEVI uint32_t swar_eq(uint32_t w, uint32_t c) {
  const uint32_t x = w ^ (c * 0x01010101u);
  return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
}
DEVI uint32_t swar_movemask(uint32_t m) { return (((m >> 7) & 0x01010101u) * 0x01020408u) >> 24; }  // bit 7s -> 4 bits

// carry: structure flags of the previous strip's lane 31 (bit 0: previous strip was exact with a
// pending sequence, which forces this strip to be exact as well); 0 at string start
DEVI Strip warp_load_strip(const uint8_t* s, int64_t base, int64_t n, uint32_t& carry) {
  Strip st;
  int l = lane_id();
  int64_t p0 = base + 4 * l;
  int64_t rem = n - p0;
  st.nvalid = rem <= 0 ? 0u : (rem >= 4 ? 4u : (uint32_t)rem);
  uint32_t w = 0;
  if (st.nvalid) {
    w = ld_u32_unaligned(s + p0);
    if (st.nvalid < 4) w &= (1u << (8 * st.nvalid)) - 1u;
  }
  st.w = w;
  uint32_t hi = w & 0x80808080u;
  st.cont = 0;
  st.l4 = 0;
  if (__ballot_sync(FULL, hi != 0) == 0 && carry == 0) {
    st.exact = false;
    return st;
  }
  const uint32_t M = 0x80808080u;
  uint32_t c = w & ((~w) << 1) & M;   // 10xxxxxx
  uint32_t ld = w & (w << 1) & M;     // 11xxxxxx
  uint32_t l3 = ld & (w << 2);        // 111xxxxx
  uint32_t l4 = l3 & (w << 3);        // 1111xxxx
  uint32_t isF0 = swar_has_byte(w, 0xF0), isE2 = swar_has_byte(w, 0xE2), isE0 = swar_has_byte(w, 0xE0),
           isED = swar_has_byte(w, 0xED);
  uint32_t P = ld | (l3 >> 1) | (l4 >> 2) | (isF0 >> 3) | (isE2 >> 4) | (isE0 >> 5) | (isED >> 6);
  uint32_t Pp = __shfl_up_sync(FULL, P, 1);
  if (l == 0) Pp = carry & ~1u;
  uint32_t Q = __funnelshift_l(Pp, P, 8);  // byte i of Q = flags of byte i-1
  uint32_t e1 = Q & M;
  uint32_t e2 = (__funnelshift_l(Pp, P, 16) << 1) & M;
  uint32_t e3 = (__funnelshift_l(Pp, P, 24) << 2) & M;
  uint32_t expect = e1 | e2 | e3;
  uint32_t pF0 = (Q << 3) & M, pE2 = (Q << 4) & M, pE0 = (Q << 5) & M, pED = (Q << 6) & M;
  uint32_t b20 = (w << 2) & M;                                  // (b & 0x20) != 0
  uint32_t nz30 = ((w & 0x30303030u) + 0x70707070u) & M;        // (b & 0x30) != 0
  uint32_t geF4 = l4 & (((w & 0x0C0C0C0Cu) + 0x7C7C7C7Cu) & M);  // byte >= 0xF4
  // evaluate one virtual byte past the end too (a lead as the last byte must be flagged)
  uint32_t chk = st.nvalid >= 3 ? M : (((1u << (8 * (st.nvalid + 1))) - 1u) & M);
  if (rem < 0) chk = 0;
  uint32_t bad = ((c ^ expect) & chk) | geF4 | swar_has_byte(w & 0xFEFEFEFEu, 0xC0) | (pF0 & ~nz30) |
                 (pE0 & ~b20) | (pED & b20) | (pE2 & swar_has_byte(w, 0x80));
  if (l == 31 && (P & 0x80402000u)) {
    if (base + 128 >= n) {
      bad |= 1;  // string ends at the strip end: the open sequence is truncated
    } else {
      // a sequence starts in the last bytes of this strip and ends in the next one: its validity
      // (and the U+2028/9 special case) depends on bytes this strip does not hold -> check it now
      int64_t pos = p0 + ((P & 0x80000000u) ? 3 : ((P & 0x00400000u) ? 2 : 1));
      int v = utf8_valid_lead(s, pos, n);
      bool ls = v == 3 && ldb(s + pos) == 0xE2 && ldb(s + pos + 1) == 0x80 && (ldb(s + pos + 2) | 1u) == 0xA9;
      if (v == 0 || ls) bad |= 1;
    }
  }
  bool exact = __ballot_sync(FULL, bad != 0) != 0 || (carry & 1u);
  st.exact = exact;
  st.cont = c;
  st.l4 = l4;
  uint32_t tail = __shfl_sync(FULL, P, 31);
  // pending = the last bytes open a sequence that continues into the next strip
  carry = (tail & 0x80402000u) ? ((tail & ~1u) | (exact ? 1u : 0u)) : 0u;
  return st;
}

// per-lane totals for the strip: escaped bytes and UTF-16 units of the lane's valid bytes
DEVI void strip_lane_totals(const Strip& st, const uint8_t* s, int64_t base, int64_t n,
                            uint32_t& esc, uint32_t& u16) {
  esc = 0;
  u16 = 0;
  if (!st.nvalid) return;
  if (st.exact) {
    int64_t p0 = base + 4 * lane_id();
    for (uint32_t k = 0; k < st.nvalid; k++) {
      ByteInfo bi = byte_info_exact(s, p0 + k, n);
      esc += bi.esc;
      u16 += bi.u16;
    }
    return;
  }
  // SWAR: does any valid byte need escaping (< 0x20, '"', '\\', '<', '>', '&')?  Exact as an "any" test.
  uint32_t wt = st.nvalid < 4 ? (st.w | (0x20202020u << (8 * st.nvalid))) : st.w;
  uint32_t special = ((wt - 0x20202020u) & ~wt & 0x80808080u) | swar_has_byte(wt, 0x22) | swar_has_byte(wt, 0x5C) |
                     swar_has_byte(wt, 0x3C) | swar_has_byte(wt, 0x3E) | swar_has_byte(wt, 0x26);
  if (!special) {
    esc = st.nvalid;
  } else {
#pragma unroll
    for (uint32_t k = 0; k < 4; k++) {
      if (k < st.nvalid) {
        uint32_t b = (st.w >> (8 * k)) & 0xFF;
        esc += b < 0x80 ? ascii_esc_len(b) : 1u;
      }
    }
  }
  u16 = st.nvalid - __popc(st.cont) + __popc(st.l4);
}

// JSON-escaped length of s[0..n) (without the quotes).  *needs_exact (optional): some strip took the
// exact per-byte path, i.e. the string holds invalid UTF-8 or U+2028/9 candidates; if it stays false
// every non-ASCII byte is copied verbatim by the escaper (esc_ascii_to_global may be used).
__device__ __noinline__ uint32_t warp_esc_len(const uint8_t* s, int64_t n, bool* needs_exact = nullptr) {
  uint32_t tot = 0, carry = 0;
  bool ex = false;
  for (int64_t base = 0; base < n; base += 128) {
    Strip st = warp_load_strip(s, base, n, carry);
    uint32_t e, u;
    strip_lane_totals(st, s, base, n, e, u);
    tot += e;
    ex = ex || st.exact;
  }
  if (needs_exact) *needs_exact = ex;
  return warp_sum(tot);
}

// ---- single-thread number / time rendering (different lanes render different fields) ------------
DEVI uint32_t ndigits_u32(uint32_t v) {
  return 1u + (v >= 10u) + (v >= 100u) + (v >= 1000u) + (v >= 10000u) + (v >= 100000u) + (v >= 1000000u) +
         (v >= 10000000u) + (v >= 100000000u) + (v >= 1000000000u);
}
DEVI uint32_t ndigits_u64(uint64_t v) {
  if ((v >> 32) == 0) return ndigits_u32((uint32_t)v);
  uint32_t d = 10;
  uint64_t p = 10000000000ull;
  while (d < 20 && v >= p) {
    d++;
    p *= 10;
  }
  return d;
}
DEVI uint32_t ndigits_i64(int64_t v) { return v < 0 ? 1u + ndigits_u64((uint64_t)0 - (uint64_t)v) : ndigits_u64((uint64_t)v); }

__device__ __noinline__ int render_u64(uint8_t* dst, uint64_t v) {
  int n = (int)ndigits_u64(v);
  int k = n;
  while (v >> 32) {  // peel 9 digits at a time with one 64-bit division
    uint64_t q = v / 1000000000ull;
    uint32_t r = (uint32_t)(v - q * 1000000000ull);
#pragma unroll
    for (int j = 0; j < 9; j++) {
      uint32_t t = r / 10;
      dst[--k] = (uint8_t)('0' + (r - t * 10));
      r = t;
    }
    v = q;
  }
  uint32_t r = (uint32_t)v;
  while (k > 0) {
    uint32_t t = r / 10;
    dst[--k] = (uint8_t)('0' + (r - t * 10));
    r = t;
  }
  return n;
}
DEVI int render_i64(uint8_t* dst, int64_t v) {
  if (v < 0) {
    dst[0] = '-';
    return 1 + render_u64(dst + 1, (uint64_t)0 - (uint64_t)v);
  }
  return render_u64(dst, (uint64_t)v);
}
DEVI void put2(uint8_t* d, uint32_t v) {
  d[0] = (uint8_t)('0' + v / 10);
  d[1] = (uint8_t)('0' + v % 10);
}
// time.Time.MarshalJSON (RFC3339Nano, quoted) for a fixed-offset zone; returns 0 if the year is
// outside [0,9999] (Marshal error).  dst needs 40 bytes.
__device__ __noinline__ int render_time(uint8_t* dst, int64_t sec, int32_t nsec, int32_t tz) {
  int64_t t = sec + tz;
  int64_t days = t / 86400;
  int32_t rem = (int32_t)(t - days * 86400);
  if (rem < 0) {
    rem += 86400;
    days -= 1;
  }
  int64_t z = days + 719468;
  int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  uint32_t doe = (uint32_t)(z - era * 146097);
  uint32_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  int64_t y = (int64_t)yoe + era * 400;
  uint32_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  uint32_t mp = (5 * doy + 2) / 153;
  uint32_t d = doy - (153 * mp + 2) / 5 + 1;
  uint32_t m = mp < 10 ? mp + 3 : mp - 9;
  if (m <= 2) y += 1;
  if (y < 0 || y > 9999) return 0;
  int o = 0;
  dst[o++] = '"';
  put2(dst + o, (uint32_t)y / 100);
  put2(dst + o + 2, (uint32_t)y % 100);
  o += 4;
  dst[o++] = '-';
  put2(dst + o, m);
  o += 2;
  dst[o++] = '-';
  put2(dst + o, d);
  o += 2;
  dst[o++] = 'T';
  put2(dst + o, (uint32_t)rem / 3600);
  o += 2;
  dst[o++] = ':';
  put2(dst + o, (uint32_t)rem % 3600 / 60);
  o += 2;
  dst[o++] = ':';
  put2(dst + o, (uint32_t)rem % 60);
  o += 2;
  if (nsec != 0) {
    uint8_t f[9];
    uint32_t v = (uint32_t)nsec;
    for (int k = 8; k >= 0; k--) {
      f[k] = (uint8_t)('0' + v % 10);
      v /= 10;
    }
    int k = 9;
    while (k > 0 && f[k - 1] == '0') k--;
    dst[o++] = '.';
    for (int j = 0; j < k; j++) dst[o++] = f[j];
  }
  if (tz == 0) {
    dst[o++] = 'Z';
  } else {
    uint32_t a = (uint32_t)(tz < 0 ? -tz : tz);
    dst[o++] = tz < 0 ? '-' : '+';
    put2(dst + o, a / 3600);
    o += 2;
    dst[o++] = ':';
    put2(dst + o, a % 3600 / 60);
    o += 2;
  }
  dst[o++] = '"';
  return o;
}

// ---- shared-memory access by 32-bit shared-space address ------------------------------------------
DEVI uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
DEVI void sts8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v)); }
DEVI uint32_t lds8(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
DEVI uint32_t lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
DEVI uint32_t lds16(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
DEVI void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v)); }
DEVI uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}

// ---- single-thread JSON escaping (Go's sequential algorithm, for short strings such as map keys) --
DEVI uint32_t thread_esc_len(const uint8_t* s, uint32_t n) {
  uint32_t o = 0;
  for (uint32_t i = 0; i < n;) {
    if (i + 4 <= n) {  // four plain ASCII bytes at once (ids, handles and file names are mostly that)
      const uint32_t w = ld_u32_unaligned(s + i);
      const uint32_t odd = (w & 0x80808080u) | ((w - 0x20202020u) & ~w & 0x80808080u) | swar_has_byte(w, 0x22) |
                           swar_has_byte(w, 0x5C) | swar_has_byte(w, 0x3C) | swar_has_byte(w, 0x3E) | swar_has_byte(w, 0x26);
      if (!odd) {
        o += 4;
        i += 4;
        continue;
      }
    }
    uint32_t b = ldb(s + i);
    if (b < 0x80) {
      o += ascii_esc_len(b);
      i++;
      continue;
    }
    int need = utf8_valid_lead(s, i, n);
    if (need == 0) {
      o += 6;
      i++;
    } else {
      bool ls = need == 3 && b == 0xE2 && ldb(s + i + 1) == 0x80 && (ldb(s + i + 2) | 1u) == 0xA9;
      o += ls ? 6u : (uint32_t)need;
      i += (uint32_t)need;
    }
  }
  return o;
}
// ---- byte sinks ---------------------------------------------------------------------------------
// All emission writes straight into the output blob in HBM (DstG) at offsets that were fixed by the
// size + scan passes; the L2 merges the byte-granular stores of neighbouring lanes / instructions
// into full sectors.  DstS (shared memory) is used for small per-lane staging only.
struct DstG {
  uint8_t* p;
  DEVI void st(uint32_t off, uint32_t v) const { p[off] = (uint8_t)v; }
  DEVI DstG at(uint32_t off) const { return DstG{p + off}; }
};
struct DstS {
  uint32_t a;
  DEVI void st(uint32_t off, uint32_t v) const { sts8(a + off, v); }
  DEVI DstS at(uint32_t off) const { return DstS{a + off}; }
};

template <class D>
DEVI void put_escaped(const D& d, uint32_t o, uint32_t b, uint32_t len) {
  if (len == 1) {
    d.st(o, b);
  } else if (len == 2) {
    d.st(o, '\\');
    uint32_t c = b;
    if (b == '\b') c = 'b';
    else if (b == '\f') c = 'f';
    else if (b == '\n') c = 'n';
    else if (b == '\r') c = 'r';
    else if (b == '\t') c = 't';
    d.st(o + 1, c);
  } else {
    uint32_t h = b >> 4, l = b & 15;
    d.st(o, '\\'); d.st(o + 1, 'u'); d.st(o + 2, '0'); d.st(o + 3, '0');
    d.st(o + 4, h < 10 ? '0' + h : 'a' + h - 10);
    d.st(o + 5, l < 10 ? '0' + l : 'a' + l - 10);
  }
}
template <class D>
DEVI void put_u(const D& d, uint32_t o, uint32_t a, uint32_t b, uint32_t c, uint32_t e) {  // \uXXXX
  d.st(o, '\\'); d.st(o + 1, 'u'); d.st(o + 2, a); d.st(o + 3, b); d.st(o + 4, c); d.st(o + 5, e);
}

// JSON-escape s[0..n) to dst (no quotes); returns the bytes written.  128-byte strips, 4 bytes per
// lane; a warp scan over the per-lane output lengths places every lane's bytes.
template <class D>
__device__ __noinline__ uint32_t esc_to(D dst, const uint8_t* s, uint32_t n) {
  uint32_t carry = 0, out = 0;
  for (int64_t base = 0; base < (int64_t)n; base += 128) {
    Strip st = warp_load_strip(s, base, n, carry);
    uint32_t el, u;
    strip_lane_totals(st, s, base, n, el, u);
    uint32_t incl = warp_incl_scan(el);
    uint32_t tot = __shfl_sync(FULL, incl, 31);
    uint32_t d = out + (incl - el);
    if (st.nvalid) {
      if (!st.exact) {
        if (el == st.nvalid) {  // nothing to escape in this lane's bytes
#pragma unroll
          for (uint32_t k = 0; k < 4; k++)
            if (k < st.nvalid) dst.st(d + k, (st.w >> (8 * k)) & 0xFF);
        } else {
#pragma unroll
          for (uint32_t k = 0; k < 4; k++) {
            if (k < st.nvalid) {
              uint32_t b = (st.w >> (8 * k)) & 0xFF;
              uint32_t len = b < 0x80 ? ascii_esc_len(b) : 1u;
              put_escaped(dst, d, b, len);
              d += len;
            }
          }
        }
      } else {
        int64_t p0 = base + 4 * lane_id();
        for (uint32_t k = 0; k < st.nvalid; k++) {
          ByteInfo bi = byte_info_exact(s, p0 + k, n);
          uint32_t b = (st.w >> (8 * k)) & 0xFF;
          if (bi.esc == 6 && b >= 0x80) {
            if (b == 0xE2 && bi.start && utf8_valid_lead(s, p0 + k, n) == 3)  // U+2028/9
              put_u(dst, d, '2', '0', '2', ldb(s + p0 + k + 2) == 0xA8 ? '8' : '9');
            else  // invalid byte -> U+FFFD
              put_u(dst, d, 'f', 'f', 'f', 'd');
          } else if (bi.esc) {
            put_escaped(dst, d, b, bi.esc);
          }
          d += bi.esc;
        }
      }
    }
    out += tot;
  }
  return out;
}

// The same for a string whose non-ASCII bytes all pass through unchanged (warp_esc_len reported
// needs_exact == false): no UTF-8 bookkeeping, so a lane can own 16 bytes and a strip is 512 bytes.
template <class D>
__device__ __noinline__ uint32_t esc_ascii_to(D dst, const uint8_t* s, uint32_t n) {
  const uint32_t l = lane_id();
  const uint32_t M = 0x80808080u, L7 = 0x7F7F7F7Fu;
  uint32_t out = 0;
  for (uint32_t base = 0; base < n; base += 512) {
    const uint32_t p0 = base + 16u * l;
    const uint32_t nv = p0 >= n ? 0u : min(16u, n - p0);
    uint32_t w[4];
    uint32_t m2 = 0, m6 = 0;  // 16-bit masks: bytes that become 2 / 6 bytes (exact, branch-free: every lane of the
                              // warp does the same work whether or not it holds such a byte)
#pragma unroll
    for (uint32_t j = 0; j < 4; j++) {
      const uint32_t nj = nv > 4u * j ? min(4u, nv - 4u * j) : 0u;
      uint32_t x = nj ? ld_u32_unaligned(s + p0 + 4u * j) : 0u;
      if (nj < 4) x = (x & ((1u << (8u * nj)) - 1u)) | (0x20202020u << (8u * nj));  // fill with spaces
      w[j] = x;
      const uint32_t lo7 = x & L7;
      const uint32_t ctl = ~(((lo7 + 0x60606060u) | x)) & M;                              // < 0x20
      const uint32_t in8_13 = (lo7 + 0x78787878u) & ~(lo7 + 0x72727272u) & M;             // 0x08..0x0d (7-bit value)
      const uint32_t sctl = ctl & in8_13 & ~swar_eq(x, 0x0B);                              // \b \t \n \f \r
      const uint32_t s2 = sctl | swar_eq(x, 0x22) | swar_eq(x, 0x5C);
      const uint32_t s6 = (ctl & ~sctl) | swar_eq(x, 0x3C) | swar_eq(x, 0x3E) | swar_eq(x, 0x26);
      m2 |= swar_movemask(s2) << (4u * j);
      m6 |= swar_movemask(s6) << (4u * j);
    }
    const uint32_t el = nv + (uint32_t)__popc(m2) + 5u * (uint32_t)__popc(m6);
    const uint32_t incl = warp_incl_scan(el);
    const uint32_t d = out + incl - el;
    const uint32_t sp = m2 | m6;
    // plain bytes: byte k lands at d + k + (bytes inserted before it)
#pragma unroll
    for (uint32_t k = 0; k < 16; k++) {
      const uint32_t below = (1u << k) - 1u;
      if (k < nv && !((sp >> k) & 1u))
        dst.st(d + k + (uint32_t)__popc(m2 & below) + 5u * (uint32_t)__popc(m6 & below), (w[k >> 2] >> (8u * (k & 3u))) & 0xFFu);
    }
    // escaped bytes: one per lane and round
    uint32_t todo = sp;
    while (__any_sync(FULL, todo != 0)) {
      if (todo) {
        const uint32_t k = (uint32_t)__ffs(todo) - 1u;
        todo &= todo - 1u;
        const uint32_t below = (1u << k) - 1u;
        const uint32_t wk = k < 4 ? w[0] : k < 8 ? w[1] : k < 12 ? w[2] : w[3];
        put_escaped(dst, d + k + (uint32_t)__popc(m2 & below) + 5u * (uint32_t)__popc(m6 & below), (wk >> (8u * (k & 3u))) & 0xFFu,
                    ((m2 >> k) & 1u) ? 2u : 6u);
      }
    }
    out += __shfl_sync(FULL, incl, 31);
  }
  return out;
}

DEVI uint32_t esc_to_global(uint8_t* dstp, const uint8_t* s, uint32_t n) { return esc_to(DstG{dstp}, s, n); }
DEVI uint32_t esc_ascii_to_global(uint8_t* dstp, const uint8_t* s, uint32_t n) { return esc_ascii_to(DstG{dstp}, s, n); }

// single-thread escape of a short string into shared memory (map keys); ~0u if it does not fit
DEVI uint32_t thread_esc(const uint8_t* s, uint32_t n, uint32_t d, uint32_t cap) {
  DstS dst{d};
  uint32_t o = 0;
  for (uint32_t i = 0; i < n;) {
    uint32_t b = ldb(s + i);
    if (o + 6 > cap) return ~0u;
    if (b < 0x80) {
      uint32_t len = ascii_esc_len(b);
      put_escaped(dst, o, b, len);
      o += len;
      i++;
      continue;
    }
    int need = utf8_valid_lead(s, i, n);
    if (need == 0) {
      put_u(dst, o, 'f', 'f', 'f', 'd');
      o += 6;
      i++;
    } else if (need == 3 && b == 0xE2 && ldb(s + i + 1) == 0x80 && (ldb(s + i + 2) | 1u) == 0xA9) {
      put_u(dst, o, '2', '0', '2', ldb(s + i + 2) == 0xA8 ? '8' : '9');
      o += 6;
      i += 3;
    } else {
      for (int k = 0; k < need; k++) dst.st(o + k, ldb(s + i + k));
      o += (uint32_t)need;
      i += (uint32_t)need;
    }
  }
  return o;
}

// warp copies into the output blob (any length): global source / shared source / one or two bytes
DEVI void gcopy_g(uint8_t* dst, const uint8_t* src, uint32_t n) {
  uint32_t l = lane_id();
  uint8_t* d = dst + l;
  const uint8_t* s = src + l;
  uint32_t i = 0;
  for (; i + 128 <= n; i += 128) {
    uint32_t b0 = ldb(s + i), b1 = ldb(s + i + 32), b2 = ldb(s + i + 64), b3 = ldb(s + i + 96);
    d[i] = (uint8_t)b0; d[i + 32] = (uint8_t)b1; d[i + 64] = (uint8_t)b2; d[i + 96] = (uint8_t)b3;
  }
  for (; i + l < n; i += 32) d[i] = (uint8_t)ldb(s + i);
}
// warp memcpy for long strings: 16-byte stores to the aligned part of dst, the source read as aligned
// 16-byte blocks and funnel-shifted by its (warp-uniform) misalignment; <= 15 head and tail bytes
// go out as single bytes.  Reads up to 31 bytes past src + n (device blobs carry that slack).
__device__ __noinline__ void warp_copy_vec(uint8_t* dst, const uint8_t* src, uint32_t n) {
  const uint32_t l = lane_id();
  const uint32_t hh = min((16u - ((uint32_t)(uintptr_t)dst & 15u)) & 15u, n);
  if (l < hh) dst[l] = (uint8_t)ldb(src + l);
  dst += hh;
  src += hh;
  n -= hh;
  const uint32_t sa = (uint32_t)(uintptr_t)src & 15u, sh = (sa & 3u) * 8u, q = sa >> 2;
  const uint4* A = (const uint4*)(src - sa);
  const uint32_t nb = n >> 4;
  for (uint32_t i = l; i < nb; i += 32) {
    const uint4 a = __ldg(A + i), b = __ldg(A + i + 1);
    uint32_t w0, w1, w2, w3, w4;  // the five words that hold bytes [sa, sa + 16) of b:a
    if (q == 0) { w0 = a.x; w1 = a.y; w2 = a.z; w3 = a.w; w4 = b.x; }
    else if (q == 1) { w0 = a.y; w1 = a.z; w2 = a.w; w3 = b.x; w4 = b.y; }
    else if (q == 2) { w0 = a.z; w1 = a.w; w2 = b.x; w3 = b.y; w4 = b.z; }
    else { w0 = a.w; w1 = b.x; w2 = b.y; w3 = b.z; w4 = b.w; }
    *(uint4*)(dst + 16u * i) = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                                          __funnelshift_r(w3, w4, sh));
  }
  const uint32_t t0 = nb << 4;
  if (t0 + l < n) dst[t0 + l] = (uint8_t)ldb(src + t0 + l);
}
// JSON-escape s[0..n) to dst when only a FEW bytes need escaping (a message whose only specials are its line breaks):
// the text between two special bytes is a plain copy at a shifted position, so the string goes out segment by segment
// with the vector memcpy and the escapes themselves are written by lane 0.  The per-byte placement of esc_ascii_to
// (one store instruction per byte position, every lane on its own bytes) is only worth it for dense specials.
// Requires valid UTF-8 without U+2028 / U+2029 (non-ASCII bytes pass through).  Returns the bytes written.
__device__ __noinline__ uint32_t esc_sparse_to_global(uint8_t* dst, const uint8_t* s, uint32_t n) {
  const uint32_t l = lane_id();
  uint32_t cur = 0, out = 0;  // warp-uniform: next source byte to copy, next output byte
  for (uint32_t base = 0; base < n; base += 512) {
    const uint32_t p0 = base + 16u * l;
    const uint32_t nv = p0 >= n ? 0u : min(16u, n - p0);
    uint32_t m = 0;  // bit k: byte p0 + k needs escaping
#pragma unroll 1
    for (uint32_t j = 0; j < nv; j += 4) {
      const uint32_t nj = min(4u, nv - j);
      uint32_t x = ld_u32_unaligned(s + p0 + j);
      if (nj < 4) x = (x & ((1u << (8u * nj)) - 1u)) | (0x20202020u << (8u * nj));
      const uint32_t ctl = ~(((x & 0x7F7F7F7Fu) + 0x60606060u) | x) & 0x80808080u;  // < 0x20
      if (ctl | swar_has_byte(x & 0xFBFBFBFBu, 0x22) | swar_has_byte(x & 0xFDFDFDFDu, 0x3C) | swar_has_byte(x, 0x5C)) {
        for (uint32_t k = 0; k < nj; k++) {
          const uint32_t bt = (x >> (8u * k)) & 0xFFu;
          if (bt < 0x80u && ascii_esc_len(bt) != 1u) m |= 1u << (j + k);
        }
      }
    }
    uint32_t lanes = __ballot_sync(FULL, m != 0);
    while (lanes) {
      const int sl = __ffs(lanes) - 1;
      lanes &= lanes - 1;
      uint32_t mm = __shfl_sync(FULL, m, sl);
      while (mm) {
        const uint32_t p = base + 16u * (uint32_t)sl + (uint32_t)(__ffs(mm) - 1);
        mm &= mm - 1;
        const uint32_t seg = p - cur;
        if (seg >= 48) warp_copy_vec(dst + out, s + cur, seg);
        else if (seg) gcopy_g(dst + out, s + cur, seg);
        out += seg;
        const uint32_t bt = ldb(s + p), el = ascii_esc_len(bt);
        if (l == 0) put_escaped(DstG{dst}, out, bt, el);
        out += el;
        cur = p + 1;
      }
    }
  }
  const uint32_t seg = n - cur;
  if (seg >= 48) warp_copy_vec(dst + out, s + cur, seg);
  else if (seg) gcopy_g(dst + out, s + cur, seg);
  return out + seg;
}

// the same three through a byte sink (DstG: the output blob, DstS: a line being assembled in shared memory)
template <class D>
DEVI void copy_g(const D& d, const uint8_t* src, uint32_t n) {
  for (uint32_t i = lane_id(); i < n; i += 32) d.st(i, ldb(src + i));
}
template <class D>
DEVI void copy_s(const D& d, uint32_t src, uint32_t n) {
  for (uint32_t i = lane_id(); i < n; i += 32) d.st(i, lds8(src + i));
}
template <class D>
DEVI void put1(const D& d, uint32_t c) {
  if (lane_id() == 0) d.st(0, c);
}
template <class D>
DEVI void put2(const D& d, uint32_t c0, uint32_t c1) {
  if (lane_id() < 2) d.st(lane_id(), lane_id() ? c1 : c0);
}
DEVI void gcopy_s(uint8_t* dst, uint32_t src, uint32_t n) {
  for (uint32_t i = lane_id(); i < n; i += 32) dst[i] = (uint8_t)lds8(src + i);
}
DEVI void gput1(uint8_t* dst, uint32_t c) {
  if (lane_id() == 0) dst[0] = (uint8_t)c;
}
DEVI void gput2(uint8_t* dst, uint32_t c0, uint32_t c1) {
  if (lane_id() < 2) dst[lane_id()] = (uint8_t)(lane_id() ? c1 : c0);
}

}  // namespace tgi
