// Test harness (NOT part of libb200g16): compiles gnark_whir_b200/csrc/keccak_duplex.cuh for the host with g++ and
// applies its segments to a 200-byte state, with a plain Keccak-f here, so the CPU test-suite can pin the op walk the
// duplex kernels run against oracle/keccak.py's Sponge.
#include <cstring>

#include "keccak_duplex.cuh"

using namespace b200;

namespace {

const uint64_t RC[24] = {
    0x0000000000000001ull, 0x0000000000008082ull, 0x800000000000808aull, 0x8000000080008000ull,
    0x000000000000808bull, 0x0000000080000001ull, 0x8000000080008081ull, 0x8000000000008009ull,
    0x000000000000008aull, 0x0000000000000088ull, 0x0000000080008009ull, 0x000000008000000aull,
    0x000000008000808bull, 0x800000000000008bull, 0x8000000000008089ull, 0x8000000000008003ull,
    0x8000000000008002ull, 0x8000000000000080ull, 0x000000000000800aull, 0x800000008000000aull,
    0x8000000080008081ull, 0x8000000000008080ull, 0x0000000080000001ull, 0x8000000080008008ull};
const int ROT[25] = {0, 1, 62, 28, 27, 36, 44, 6, 55, 20, 3, 10, 43, 25, 39, 41, 45, 15, 21, 8, 18, 2, 61, 56, 14};

uint64_t rol(uint64_t v, int n) { return n ? (v << n) | (v >> (64 - n)) : v; }

// FIPS-202 Keccak-f[1600] on the state's bytes (lane x + 5y little-endian at byte 8(x + 5y))
void keccak_f(uint8_t* st) {
  uint64_t a[25], b[25], c[5];
  for (int i = 0; i < 25; i++) {
    a[i] = 0;
    for (int k = 0; k < 8; k++) a[i] |= (uint64_t)st[8 * i + k] << (8 * k);
  }
  for (int r = 0; r < 24; r++) {
    for (int x = 0; x < 5; x++) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
    for (int i = 0; i < 25; i++) a[i] ^= c[(i + 4) % 5] ^ rol(c[(i + 1) % 5], 1);
    for (int x = 0; x < 5; x++)
      for (int y = 0; y < 5; y++) b[y + 5 * ((2 * x + 3 * y) % 5)] = rol(a[x + 5 * y], ROT[x + 5 * y]);
    for (int i = 0; i < 25; i++) a[i] = b[i] ^ (~b[(i % 5 + 1) % 5 + 5 * (i / 5)] & b[(i % 5 + 2) % 5 + 5 * (i / 5)]);
    a[0] ^= RC[r];
  }
  for (int i = 0; i < 25; i++)
    for (int k = 0; k < 8; k++) st[8 * i + k] = (uint8_t)(a[i] >> (8 * k));
}

}  // namespace

extern "C" {

// Run the script ops[k] = (kind, len) (kind 0 absorb, 1 squeeze) on state (200 bytes) with positions pos[0] =
// absorb_pos, pos[1] = squeeze_pos, taking the absorbed bytes from `in` and writing the squeezed ones to `out` in
// script order; *n_perm counts the permutations.  Each segment is applied lane by lane through duplex_lane_span, as
// the kernels apply it.  Returns the number of segments.
long host_duplex(uint8_t* state, uint32_t* pos, const uint32_t* ops, size_t n_ops, const uint8_t* in, uint8_t* out,
                 uint64_t* n_perm) {
  DuplexWalk w;
  w.absorb_pos = pos[0];
  w.squeeze_pos = pos[1];
  uint64_t in_off = 0, out_off = 0;
  long segs = 0;
  for (size_t k = 0; k < n_ops; k++) {
    const bool sq = ops[2 * k] != 0;
    duplex_op_begin(w, ops[2 * k + 1], sq ? out_off : in_off);
    while (w.left) {
      const DuplexSeg s = duplex_next(w, sq);
      segs++;
      if (s.len == 0 || s.rate_off + s.len > DUPLEX_RATE) return -1;   // a segment stays inside one rate block
      if (s.permute) {
        keccak_f(state);
        ++*n_perm;
      }
      for (uint32_t l = 0; l < 17; l++) {
        uint32_t lo, hi;
        if (!duplex_lane_span(s, l, &lo, &hi)) continue;
        for (uint32_t b = lo; b < hi; b++) {
          const uint64_t row = s.row_off + 8 * l + b - s.rate_off;
          if (sq) out[row] = state[8 * l + b];
          else state[8 * l + b] = in[row];
        }
      }
    }
    duplex_op_end(w, sq);
    if (sq) out_off = w.row_off;
    else in_off = w.row_off;
  }
  pos[0] = w.absorb_pos;
  pos[1] = w.squeeze_pos;
  return segs;
}
}
