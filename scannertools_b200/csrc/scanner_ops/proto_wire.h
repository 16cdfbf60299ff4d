// Protobuf wire-format reader for the kernel classes whose args are a few scalar or string fields
// (ResizeArgs, BlurArgs; scannertools_imgproc.proto), so they do not need the generated scannertools_imgproc.pb.h.
#pragma once
#include <cstddef>
#include <vector>

#include "scanner/util/common.h"

namespace scanner {

inline bool read_varint(const u8*& p, const u8* end, u64& v) {
  v = 0;
  for (int shift = 0; p < end && shift < 64; shift += 7) {
    const u8 b = *p++;
    v |= (u64)(b & 0x7f) << shift;
    if (!(b & 0x80)) return true;
  }
  return false;
}

// One field of a message: `varint` for wire type 0; `data` / `len` for types 2 (the payload), 5 (4 bytes) and 1
// (8 bytes).
struct WireField {
  int field, wire;
  u64 varint;
  const u8* data;
  size_t len;
};

// Calls on_field(const WireField&) for every field of `buf` in order; false on a truncated field or a wire type
// other than 0, 1, 2 and 5 (groups are not used by these messages).
template <class OnField>
bool parse_wire_fields(const std::vector<u8>& buf, OnField on_field) {
  const u8* p = buf.data();
  const u8* end = p + buf.size();
  while (p < end) {
    u64 key;
    if (!read_varint(p, end, key)) return false;
    WireField f{(int)(key >> 3), (int)(key & 7), 0, nullptr, 0};
    if (f.wire == 0) {
      if (!read_varint(p, end, f.varint)) return false;
    } else if (f.wire == 2) {
      u64 len;
      if (!read_varint(p, end, len) || len > (u64)(end - p)) return false;
      f.len = (size_t)len;
    } else if (f.wire == 5) {
      if (end - p < 4) return false;
      f.len = 4;
    } else if (f.wire == 1) {
      if (end - p < 8) return false;
      f.len = 8;
    } else {
      return false;
    }
    if (f.wire != 0) {
      f.data = p;
      p += f.len;
    }
    on_field(f);
  }
  return true;
}

}  // namespace scanner
