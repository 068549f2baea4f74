// The byte-position rules of keccakSponge.Digest (keccakSponge.go:40-75) as a walk over segments, shared by the two
// duplex kernels in keccak.cu and compiled for the host by tests/host_harness/duplex_host.cc, which pins it against
// oracle/keccak.py's Sponge.  Nothing else in the kernels knows the rules.
//
// An op (Absorb(len) or Squeeze(len)) is cut into segments, each inside one rate block: "permute first (or not), then
// overwrite / emit `len` bytes of the rate starting at byte `rate_off`, taking / giving row bytes from `row_off` on".
//   Absorb:  a byte meets absorb_pos == 136 -> permute, absorb_pos = 0; write byte absorb_pos++.  After the op (len 0
//            included) squeeze_pos = 136, so the next Squeeze permutes first.
//   Squeeze: a byte meets squeeze_pos == 136 -> permute, squeeze_pos = absorb_pos = 0; emit byte squeeze_pos++.
// A permutation is only ever issued in front of a byte, so a full block absorbed last (absorb_pos == 136) stays
// unpermuted until the next byte or squeeze, in this call or a later one.
#pragma once
#include "ptx.cuh"

namespace b200 {

constexpr uint32_t DUPLEX_RATE = 136;

struct DuplexSeg {
  bool permute;       // run Keccak-f before touching the bytes
  uint32_t rate_off;  // first state byte of the segment (0 .. 135)
  uint32_t len;       // bytes in the segment (1 .. 136 - rate_off)
  uint64_t row_off;   // offset of its first byte in the sponge's input row (absorb) or output row (squeeze)
};

// Walk state of one sponge inside one op: the two Digest positions, the op's bytes still to go and where the next
// one sits in the row.
struct DuplexWalk {
  uint32_t absorb_pos, squeeze_pos;
  uint32_t left;
  uint64_t row_off;
};

// Start op (squeeze, len) whose first byte sits at row_off of its row.
B200_HD void duplex_op_begin(DuplexWalk& w, uint32_t len, uint64_t row_off) {
  w.left = len;
  w.row_off = row_off;
}

// The next segment of the current op (call while w.left > 0); advances the positions past it.
B200_HD DuplexSeg duplex_next(DuplexWalk& w, bool squeeze) {
  DuplexSeg s;
  s.row_off = w.row_off;
  if (squeeze) {
    s.permute = w.squeeze_pos == DUPLEX_RATE;
    if (s.permute) { w.squeeze_pos = 0; w.absorb_pos = 0; }
    s.rate_off = w.squeeze_pos;
  } else {
    s.permute = w.absorb_pos == DUPLEX_RATE;
    if (s.permute) w.absorb_pos = 0;
    s.rate_off = w.absorb_pos;
  }
  const uint32_t room = DUPLEX_RATE - s.rate_off;
  s.len = w.left < room ? w.left : room;
  if (squeeze) w.squeeze_pos += s.len;
  else w.absorb_pos += s.len;
  w.left -= s.len;
  w.row_off += s.len;
  return s;
}

// After the op's last segment (also for an op of length 0).
B200_HD void duplex_op_end(DuplexWalk& w, bool squeeze) {
  if (!squeeze) w.squeeze_pos = DUPLEX_RATE;
}

// The bytes of state lane l (bytes 8l .. 8l+7) that segment s covers: [*lo, *hi) within the lane; false if none.
B200_HD bool duplex_lane_span(const DuplexSeg& s, uint32_t l, uint32_t* lo, uint32_t* hi) {
  const uint32_t b0 = 8 * l, b1 = b0 + 8, e = s.rate_off + s.len;
  const uint32_t a = s.rate_off > b0 ? s.rate_off : b0, z = e < b1 ? e : b1;
  if (a >= z) return false;
  *lo = a - b0;
  *hi = z - b0;
  return true;
}

}  // namespace b200
