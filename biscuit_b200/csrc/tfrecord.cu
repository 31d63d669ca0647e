// TFRecord reading on the host: record framing with CRC32C verification, and the tf.train.Example wire format down to
// the byte ranges / values of the features a tile record carries (Slideflow: image_raw, slide, loc_x, loc_y).
#include <stdint.h>

#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/biscuit_b200.h"

namespace {

struct CrcTables {
  uint32_t t[8][256];
  CrcTables() {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c >> 1) ^ (0x82F63B78u & (0u - (c & 1)));
      t[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; ++i)
      for (int k = 1; k < 8; ++k) t[k][i] = (t[k - 1][i] >> 8) ^ t[0][t[k - 1][i] & 0xFF];
  }
};

uint32_t crc_table(uint32_t crc, const uint8_t* p, int64_t n) {
  static const CrcTables tabs;
  const auto& g_table = tabs.t;
  while (n >= 8) {                                   // slicing-by-8
    uint64_t v;
    memcpy(&v, p, 8);
    const uint32_t lo = (uint32_t)v ^ crc, hi = (uint32_t)(v >> 32);
    crc = g_table[7][lo & 0xFF] ^ g_table[6][(lo >> 8) & 0xFF] ^ g_table[5][(lo >> 16) & 0xFF] ^ g_table[4][lo >> 24] ^
          g_table[3][hi & 0xFF] ^ g_table[2][(hi >> 8) & 0xFF] ^ g_table[1][(hi >> 16) & 0xFF] ^ g_table[0][hi >> 24];
    p += 8;
    n -= 8;
  }
  while (n-- > 0) crc = (crc >> 8) ^ g_table[0][(crc ^ *p++) & 0xFF];
  return crc;
}

#if defined(__x86_64__)
__attribute__((target("sse4.2"))) uint32_t crc_sse42(uint32_t crc, const uint8_t* p, int64_t n) {
  uint64_t c = crc;
  while (n >= 8) {
    uint64_t v;
    memcpy(&v, p, 8);
    c = __builtin_ia32_crc32di(c, v);
    p += 8;
    n -= 8;
  }
  uint32_t c32 = (uint32_t)c;
  while (n-- > 0) c32 = __builtin_ia32_crc32qi(c32, *p++);
  return c32;
}
bool have_sse42() { return __builtin_cpu_supports("sse4.2"); }
#endif

uint32_t crc32c(const uint8_t* p, int64_t n) {
#if defined(__x86_64__)
  static const bool hw = have_sse42();
  if (hw) return ~crc_sse42(0xFFFFFFFFu, p, n);
#endif
  return ~crc_table(0xFFFFFFFFu, p, n);
}

uint32_t masked(uint32_t c) { return ((c >> 15) | (c << 17)) + 0xA282EAD8u; }

uint32_t le32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
uint64_t le64(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }

// protobuf wire format
bool varint(const uint8_t*& p, const uint8_t* e, uint64_t& v) {
  v = 0;
  for (int s = 0; s < 64 && p < e; s += 7) {
    const uint8_t b = *p++;
    v |= (uint64_t)(b & 0x7F) << s;
    if (!(b & 0x80)) return true;
  }
  return false;
}

// Skip a field of wire type wt; false on malformed input.
bool skip(const uint8_t*& p, const uint8_t* e, int wt) {
  uint64_t v;
  switch (wt) {
    case 0: return varint(p, e, v);
    case 1: if (e - p < 8) return false; p += 8; return true;
    case 5: if (e - p < 4) return false; p += 4; return true;
    case 2: if (!varint(p, e, v) || v > (uint64_t)(e - p)) return false; p += v; return true;
    default: return false;                         // groups are not used by tf.train.Example
  }
}

// Length-delimited field: [*b, *e) on success.
bool ld(const uint8_t*& p, const uint8_t* e, const uint8_t** b, const uint8_t** f) {
  uint64_t v;
  if (!varint(p, e, v) || v > (uint64_t)(e - p)) return false;
  *b = p;
  *f = p + v;
  p += v;
  return true;
}

// Feature message: first value of bytes_list (field 1) -> range, of int64_list (field 3) -> value.
bool feature(const uint8_t* p, const uint8_t* e, const uint8_t** bb, const uint8_t** be, bool* has_int, int64_t* iv) {
  while (p < e) {
    uint64_t key;
    if (!varint(p, e, key)) return false;
    const int fn = (int)(key >> 3), wt = (int)(key & 7);
    if ((fn == 1 || fn == 3) && wt == 2) {
      const uint8_t *lb, *le;
      if (!ld(p, e, &lb, &le)) return false;
      const uint8_t* q = lb;
      while (q < le) {
        uint64_t k2;
        if (!varint(q, le, k2)) return false;
        const int f2 = (int)(k2 >> 3), w2 = (int)(k2 & 7);
        if (f2 == 1 && fn == 1 && w2 == 2) {
          const uint8_t *vb, *ve;
          if (!ld(q, le, &vb, &ve)) return false;
          if (!*bb) { *bb = vb; *be = ve; }
        } else if (f2 == 1 && fn == 3 && w2 == 2) {        // packed int64
          const uint8_t *vb, *ve;
          if (!ld(q, le, &vb, &ve)) return false;
          uint64_t v;
          if (vb < ve && !*has_int) { if (!varint(vb, ve, v)) return false; *iv = (int64_t)v; *has_int = true; }
        } else if (f2 == 1 && fn == 3 && w2 == 0) {
          uint64_t v;
          if (!varint(q, le, v)) return false;
          if (!*has_int) { *iv = (int64_t)v; *has_int = true; }
        } else if (!skip(q, le, w2)) {
          return false;
        }
      }
    } else if (!skip(p, e, wt)) {
      return false;
    }
  }
  return true;
}

struct Want {
  const char* key;
  size_t len;
  const uint8_t *bb = nullptr, *be = nullptr;
  bool has_int = false;
  int64_t iv = 0;
};

// Example { Features features = 1 }  Features { map<string, Feature> feature = 1 }
bool example(const uint8_t* p, const uint8_t* e, Want* w, int nw) {
  while (p < e) {
    uint64_t key;
    if (!varint(p, e, key)) return false;
    if ((key >> 3) == 1 && (key & 7) == 2) {
      const uint8_t *fb, *fe;
      if (!ld(p, e, &fb, &fe)) return false;
      while (fb < fe) {
        uint64_t k1;
        if (!varint(fb, fe, k1)) return false;
        if ((k1 >> 3) == 1 && (k1 & 7) == 2) {         // one map entry
          const uint8_t *mb, *me;
          if (!ld(fb, fe, &mb, &me)) return false;
          const uint8_t *kb = nullptr, *ke = nullptr, *vb = nullptr, *ve = nullptr;
          while (mb < me) {
            uint64_t k2;
            if (!varint(mb, me, k2)) return false;
            if ((k2 >> 3) == 1 && (k2 & 7) == 2) { if (!ld(mb, me, &kb, &ke)) return false; }
            else if ((k2 >> 3) == 2 && (k2 & 7) == 2) { if (!ld(mb, me, &vb, &ve)) return false; }
            else if (!skip(mb, me, (int)(k2 & 7))) return false;
          }
          if (!kb || !vb) continue;
          for (int i = 0; i < nw; ++i)
            if (w[i].key && (size_t)(ke - kb) == w[i].len && memcmp(kb, w[i].key, w[i].len) == 0 &&
                !feature(vb, ve, &w[i].bb, &w[i].be, &w[i].has_int, &w[i].iv))
              return false;
        } else if (!skip(fb, fe, (int)(k1 & 7))) {
          return false;
        }
      }
    } else if (!skip(p, e, (int)(key & 7))) {
      return false;
    }
  }
  return true;
}

int fail(char* err, int64_t cap, const char* msg, int64_t rec, int64_t off) {
  if (err && cap > 0) snprintf(err, (size_t)cap, "TFRecord record %lld (byte %lld): %s", (long long)rec, (long long)off, msg);
  return BQ_ERR_DATA;
}

}  // namespace

extern "C" {

uint32_t bq_crc32c(const uint8_t* buf, int64_t len) { return crc32c(buf, len); }
uint32_t bq_crc32c_masked(const uint8_t* buf, int64_t len) { return masked(crc32c(buf, len)); }

int bq_tfrecord_scan(const uint8_t* buf, int64_t len, const char* image_key, const char* slide_key, const char* x_key,
                     const char* y_key, int64_t capacity, int64_t* n_records, int64_t* image, int64_t* slide,
                     int64_t* loc, char* err, int64_t err_capacity) {
  if (err && err_capacity > 0) err[0] = 0;
  if (len < 0 || (len > 0 && !buf) || !image_key || !n_records || capacity < 0 ||
      (capacity > 0 && (!image || !slide || !loc)))
    return BQ_ERR_ARG;
  Want w[4];
  const char* keys[4] = {image_key, slide_key, x_key, y_key};
  for (int i = 0; i < 4; ++i) { w[i].key = keys[i]; w[i].len = keys[i] ? strlen(keys[i]) : 0; }
  int64_t off = 0, r = 0;
  while (off < len) {
    if (len - off < 12) return fail(err, err_capacity, "truncated record header", r, off);
    const uint64_t n = le64(buf + off);
    if (masked(crc32c(buf + off, 8)) != le32(buf + off + 8)) {
      if (r == 0 && len >= 2 && buf[0] == 0x1F && buf[1] == 0x8B)
        return fail(err, err_capacity, "gzip-compressed TFRecord files are not supported (decompress first)", r, off);
      if (r == 0 && len >= 2 && (buf[0] & 0x0F) == 8 && ((buf[0] << 8) | buf[1]) % 31 == 0)
        return fail(err, err_capacity, "zlib-compressed TFRecord files are not supported (decompress first)", r, off);
      return fail(err, err_capacity, "length CRC mismatch (corrupt or not a TFRecord file)", r, off);
    }
    if (n > (uint64_t)(len - off - 12) || len - off - 12 - (int64_t)n < 4)
      return fail(err, err_capacity, "truncated record", r, off);
    const uint8_t* p = buf + off + 12;
    if (masked(crc32c(p, (int64_t)n)) != le32(p + n)) return fail(err, err_capacity, "payload CRC mismatch", r, off);
    if (r < capacity) {
      for (auto& x : w) { x.bb = x.be = nullptr; x.has_int = false; x.iv = 0; }
      if (!example(p, p + n, w, 4)) return fail(err, err_capacity, "malformed tf.train.Example", r, off);
      if (!w[0].bb) {
        std::string m = std::string("no bytes feature '") + image_key + "'";
        return fail(err, err_capacity, m.c_str(), r, off);
      }
      image[2 * r] = w[0].bb - buf;
      image[2 * r + 1] = w[0].be - buf;
      slide[2 * r] = w[1].bb ? w[1].bb - buf : -1;
      slide[2 * r + 1] = w[1].bb ? w[1].be - buf : -1;
      loc[2 * r] = w[2].has_int ? w[2].iv : INT64_MIN;
      loc[2 * r + 1] = w[3].has_int ? w[3].iv : INT64_MIN;
    }
    off += 12 + (int64_t)n + 4;
    ++r;
  }
  *n_records = r;
  return BQ_OK;
}

}  // extern "C"
