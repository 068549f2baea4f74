// Batched Keccak-f[1600], the reference's overwrite-mode duplex sponge, and Merkle-path
// recomputation, for sm_100a.
//
//   k_keccak_f_batch  <- gnark std/permutation/keccakf.Permute as called at
//                        /root/reference/keccakSponge/keccakSponge.go:48,69 (FIPS-202 permutation
//                        on 25 little-endian u64 lanes, lane index x + 5y)
//   k_sponge_batch    <- keccakSponge.Digest: NewKeccak / Absorb / Squeeze
//                        (keccakSponge.go:17-30, 40-56, 64-75): rate 136 B, OVERWRITE absorb,
//                        no padding, permute-on-full and permute-before-first-squeeze
//   k_duplex_thread,  <- the whole keccakSponge.Digest (keccakSponge.go:17-75): NewKeccakWithTag, Absorb /
//   k_duplex_warp        Squeeze in any order, the state carried across calls (byte rules: keccak_duplex.cuh)
//   k_merkle_paths    <- VerifyMerkleTreeProofs (/root/reference/mtUtilities.go:109-141): leaf hash,
//                        then per level pair with the sibling by the index bit (bit 0 uses
//                        LeafSiblingHashes, bit k>=1 uses AuthPaths[k-1]; set bit => current node
//                        is the right child), compare with the root.  The 2-to-1 hash is the
//                        Keccak duplex above, as BASELINE.json config 4 specifies.
//
// One thread owns one state: 25 lanes = 50 registers, 24 fully unrolled rounds; chi is a
// single LOP3 per 32-bit half and theta's 5-way XOR two LOP3s, so the kernel is LOP3/SHF
// (ALU-pipe) bound, not HBM bound (400 B of traffic per ~3.7k 64-bit logic ops).
#include <cstdlib>

#include "common.cuh"
#include "keccak_duplex.cuh"

namespace b200 {

constexpr int KECCAK_RATE = 136;
constexpr int KECCAK_RATE_LANES = 17;

__constant__ uint64_t kRC[24] = {
    0x0000000000000001ull, 0x0000000000008082ull, 0x800000000000808aull, 0x8000000080008000ull,
    0x000000000000808bull, 0x0000000080000001ull, 0x8000000080008081ull, 0x8000000000008009ull,
    0x000000000000008aull, 0x0000000000000088ull, 0x0000000080008009ull, 0x000000008000000aull,
    0x000000008000808bull, 0x800000000000008bull, 0x8000000000008089ull, 0x8000000000008003ull,
    0x8000000000008002ull, 0x8000000000000080ull, 0x000000000000800aull, 0x800000008000000aull,
    0x8000000080008081ull, 0x8000000000008080ull, 0x0000000080000001ull, 0x8000000080008008ull};

__device__ __forceinline__ uint64_t rol64(uint64_t v, int n) { return (v << n) | (v >> (64 - n)); }

// 2^k, read through the constant bank so ptxas cannot turn the multiplications below back into shifts
__constant__ uint32_t kPow2[32] = {1u << 0,  1u << 1,  1u << 2,  1u << 3,  1u << 4,  1u << 5,  1u << 6,  1u << 7,
                                   1u << 8,  1u << 9,  1u << 10, 1u << 11, 1u << 12, 1u << 13, 1u << 14, 1u << 15,
                                   1u << 16, 1u << 17, 1u << 18, 1u << 19, 1u << 20, 1u << 21, 1u << 22, 1u << 23,
                                   1u << 24, 1u << 25, 1u << 26, 1u << 27, 1u << 28, 1u << 29, 1u << 30, 1u << 31};

// 64-bit rotation on the FMA pipe: (x << k) = x * 2^k (IMAD), (x >> (32 - k)) = umulhi(x, 2^k) (IMAD.HI);
// the two parts of each half never overlap, so the OR is the multiply-add's addition.  Keccak-f is bound
// by the ALU pipe (LOP3 + SHF: 81% busy, FMA pipe 5% — profiles/r01b_ncu_full_summary.txt); moving part of
// the rotations over balances the two pipes.
template <int N>
__device__ __forceinline__ uint64_t rol64_fma(uint64_t v) {
  uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
  if (N >= 32) { uint32_t t = lo; lo = hi; hi = t; }
  constexpr int K = N & 31;
  if (K == 0) return ((uint64_t)hi << 32) | lo;
  const uint32_t m = kPow2[K];
  uint32_t nlo = lo * m + __umulhi(hi, m);
  uint32_t nhi = hi * m + __umulhi(lo, m);
  return ((uint64_t)nhi << 32) | nlo;
}

// rotation `IDX` (0..4: theta's rotations by 1, 5..28: the rho rotation of lane IDX-4) goes to the FMA
// pipe when bit IDX of MASK is set
template <uint32_t MASK, int IDX, int N>
__device__ __forceinline__ uint64_t rolx(uint64_t v) {
  if constexpr ((MASK >> IDX) & 1u) return rol64_fma<N>(v);
  else return rol64(v, N);
}

template <uint32_t MASK>
__device__ __forceinline__ void keccak_f1600_t(uint64_t (&a)[25]) {
#pragma unroll
  for (int rnd = 0; rnd < 24; rnd++) {
    uint64_t c0 = a[0] ^ a[5] ^ a[10] ^ a[15] ^ a[20];
    uint64_t c1 = a[1] ^ a[6] ^ a[11] ^ a[16] ^ a[21];
    uint64_t c2 = a[2] ^ a[7] ^ a[12] ^ a[17] ^ a[22];
    uint64_t c3 = a[3] ^ a[8] ^ a[13] ^ a[18] ^ a[23];
    uint64_t c4 = a[4] ^ a[9] ^ a[14] ^ a[19] ^ a[24];
    uint64_t d0 = c4 ^ rolx<MASK, 0, 1>(c1);
    uint64_t d1 = c0 ^ rolx<MASK, 1, 1>(c2);
    uint64_t d2 = c1 ^ rolx<MASK, 2, 1>(c3);
    uint64_t d3 = c2 ^ rolx<MASK, 3, 1>(c4);
    uint64_t d4 = c3 ^ rolx<MASK, 4, 1>(c0);
    // theta + rho + pi:  b[y + 5((2x+3y)%5)] = rol(a[x+5y] ^ d[x], ROT[x][y])
    uint64_t b0 = a[0] ^ d0;
    uint64_t b10 = rolx<MASK, 5, 1>(a[1] ^ d1);
    uint64_t b20 = rolx<MASK, 6, 62>(a[2] ^ d2);
    uint64_t b5 = rolx<MASK, 7, 28>(a[3] ^ d3);
    uint64_t b15 = rolx<MASK, 8, 27>(a[4] ^ d4);
    uint64_t b16 = rolx<MASK, 9, 36>(a[5] ^ d0);
    uint64_t b1 = rolx<MASK, 10, 44>(a[6] ^ d1);
    uint64_t b11 = rolx<MASK, 11, 6>(a[7] ^ d2);
    uint64_t b21 = rolx<MASK, 12, 55>(a[8] ^ d3);
    uint64_t b6 = rolx<MASK, 13, 20>(a[9] ^ d4);
    uint64_t b7 = rolx<MASK, 14, 3>(a[10] ^ d0);
    uint64_t b17 = rolx<MASK, 15, 10>(a[11] ^ d1);
    uint64_t b2 = rolx<MASK, 16, 43>(a[12] ^ d2);
    uint64_t b12 = rolx<MASK, 17, 25>(a[13] ^ d3);
    uint64_t b22 = rolx<MASK, 18, 39>(a[14] ^ d4);
    uint64_t b23 = rolx<MASK, 19, 41>(a[15] ^ d0);
    uint64_t b8 = rolx<MASK, 20, 45>(a[16] ^ d1);
    uint64_t b18 = rolx<MASK, 21, 15>(a[17] ^ d2);
    uint64_t b3 = rolx<MASK, 22, 21>(a[18] ^ d3);
    uint64_t b13 = rolx<MASK, 23, 8>(a[19] ^ d4);
    uint64_t b14 = rolx<MASK, 24, 18>(a[20] ^ d0);
    uint64_t b24 = rolx<MASK, 25, 2>(a[21] ^ d1);
    uint64_t b9 = rolx<MASK, 26, 61>(a[22] ^ d2);
    uint64_t b19 = rolx<MASK, 27, 56>(a[23] ^ d3);
    uint64_t b4 = rolx<MASK, 28, 14>(a[24] ^ d4);
    // chi
    a[0] = b0 ^ (~b1 & b2);   a[1] = b1 ^ (~b2 & b3);   a[2] = b2 ^ (~b3 & b4);
    a[3] = b3 ^ (~b4 & b0);   a[4] = b4 ^ (~b0 & b1);
    a[5] = b5 ^ (~b6 & b7);   a[6] = b6 ^ (~b7 & b8);   a[7] = b7 ^ (~b8 & b9);
    a[8] = b8 ^ (~b9 & b5);   a[9] = b9 ^ (~b5 & b6);
    a[10] = b10 ^ (~b11 & b12); a[11] = b11 ^ (~b12 & b13); a[12] = b12 ^ (~b13 & b14);
    a[13] = b13 ^ (~b14 & b10); a[14] = b14 ^ (~b10 & b11);
    a[15] = b15 ^ (~b16 & b17); a[16] = b16 ^ (~b17 & b18); a[17] = b17 ^ (~b18 & b19);
    a[18] = b18 ^ (~b19 & b15); a[19] = b19 ^ (~b15 & b16);
    a[20] = b20 ^ (~b21 & b22); a[21] = b21 ^ (~b22 & b23); a[22] = b22 ^ (~b23 & b24);
    a[23] = b23 ^ (~b24 & b20); a[24] = b24 ^ (~b20 & b21);
    // iota
    a[0] ^= kRC[rnd];
  }
}

// Which rotations run on the FMA pipe.  Measured on B200, 2^22 states (tools/gpu_probe9.py): none 2.81,
// all 29 2.86 (FMA-bound), theta's five 2.83, one rho rotation in three 2.91, every other 2.92, two in
// three 2.95 Gperm/s.  The gain is small because IMAD.HI issues at half rate and the two pipes overlap
// only partly (b200g16_pipe_probe mode 5), but it is free.
#ifndef B200_KECCAK_FMA_MASK
#define B200_KECCAK_FMA_MASK 0x1b6db6d0u
#endif
__device__ __forceinline__ void keccak_f1600(uint64_t (&a)[25]) { keccak_f1600_t<B200_KECCAK_FMA_MASK>(a); }

// ---- raw batch: states[i][25] permuted in place.  A warp stages its 32 states (6400
// contiguous bytes) through shared memory so the global accesses are fully coalesced.
constexpr int KF_THREADS = 128;
template <uint32_t MASK>
__global__ void __launch_bounds__(KF_THREADS) k_keccak_f_batch(uint64_t* __restrict__ states, size_t n) {
  __shared__ uint64_t sm[KF_THREADS / 32][32 * 25];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t warp_first = ((size_t)blockIdx.x * KF_THREADS + (size_t)warp * 32);
  if (warp_first >= n) return;
  const size_t in_warp = n - warp_first < 32 ? n - warp_first : 32;
  uint64_t* g = states + warp_first * 25;
  const uint32_t words = (uint32_t)in_warp * 25;
#pragma unroll
  for (int j = 0; j < 25; j++) {
    uint32_t w = lane + 32 * j;
    if (w < words) sm[warp][w] = g[w];
  }
  __syncwarp();
  uint64_t a[25];
  if (lane < in_warp) {
#pragma unroll
    for (int l = 0; l < 25; l++) a[l] = sm[warp][lane * 25 + l];
    keccak_f1600_t<MASK>(a);
#pragma unroll
    for (int l = 0; l < 25; l++) sm[warp][lane * 25 + l] = a[l];
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 25; j++) {
    uint32_t w = lane + 32 * j;
    if (w < words) g[w] = sm[warp][w];
  }
}

// ---- sponge helpers.  `len` bytes at `src` overwrite the first bytes of the rate, block by block.
__device__ __forceinline__ uint64_t load_le64_partial(const uint8_t* p, int nbytes) {
  uint64_t v = 0;
  for (int k = 0; k < nbytes; k++) v |= (uint64_t)p[k] << (8 * k);
  return v;
}

// absorb `len` bytes then permute once more (the permute Squeeze issues first): state after
// NewKeccak(); Absorb(src[:len]); and the permutation at the head of Squeeze.
template <bool ALIGNED8>
__device__ __forceinline__ void sponge_absorb_finish(uint64_t (&a)[25], const uint8_t* src, size_t len) {
  size_t off = 0;
  while (len - off > KECCAK_RATE) {  // full blocks followed by more data: overwrite + permute
#pragma unroll
    for (int l = 0; l < KECCAK_RATE_LANES; l++)
      a[l] = ALIGNED8 ? reinterpret_cast<const uint64_t*>(src + off)[l] : load_le64_partial(src + off + 8 * l, 8);
    keccak_f1600(a);
    off += KECCAK_RATE;
  }
  int rem = (int)(len - off);  // 0..136 bytes in the last block (0 only when len == 0)
#pragma unroll
  for (int l = 0; l < KECCAK_RATE_LANES; l++) {
    int nb = rem - 8 * l;
    if (nb >= 8) {
      a[l] = ALIGNED8 ? reinterpret_cast<const uint64_t*>(src + off)[l] : load_le64_partial(src + off + 8 * l, 8);
    } else if (nb > 0) {
      uint64_t mask = (1ull << (8 * nb)) - 1;
      a[l] = (a[l] & ~mask) | load_le64_partial(src + off + 8 * l, nb);
    }
  }
  keccak_f1600(a);
}

// squeeze out_len bytes (state already permuted once)
__device__ __forceinline__ void sponge_squeeze(uint64_t (&a)[25], uint8_t* dst, size_t out_len) {
  size_t done = 0;
  while (true) {
    size_t take = out_len - done < KECCAK_RATE ? out_len - done : KECCAK_RATE;
#pragma unroll
    for (int l = 0; l < KECCAK_RATE_LANES; l++) {
      long nb = (long)take - 8 * l;
      if (nb > 0) {
        uint64_t v = a[l];
        for (int k = 0; k < (nb < 8 ? nb : 8); k++) dst[done + 8 * l + k] = (uint8_t)(v >> (8 * k));
      }
    }
    done += take;
    if (done >= out_len) break;
    keccak_f1600(a);
  }
}

__global__ void __launch_bounds__(128) k_sponge_batch(const uint8_t* __restrict__ in, size_t in_len, size_t n,
                                                       uint8_t* __restrict__ out, size_t out_len, int aligned8) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t a[25];
#pragma unroll
  for (int l = 0; l < 25; l++) a[l] = 0;
  if (aligned8) sponge_absorb_finish<true>(a, in + i * in_len, in_len);
  else sponge_absorb_finish<false>(a, in + i * in_len, in_len);
  sponge_squeeze(a, out + i * out_len, out_len);
}

// ---- Merkle paths.  Digests are 32 bytes = lanes 0..3 of the squeezed state.
__global__ void __launch_bounds__(128) k_merkle_paths(const uint8_t* __restrict__ leaves, size_t leaf_len,
                                                       const uint64_t* __restrict__ leaf_siblings,
                                                       const uint64_t* __restrict__ auth_paths,
                                                       const uint64_t* __restrict__ indexes, unsigned height,
                                                       size_t n, const uint64_t* __restrict__ expected_root,
                                                       uint64_t* __restrict__ roots_out, uint8_t* __restrict__ ok_out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t a[25];
#pragma unroll
  for (int l = 0; l < 25; l++) a[l] = 0;
  sponge_absorb_finish<true>(a, leaves + i * leaf_len, leaf_len);
  uint64_t cur[4] = {a[0], a[1], a[2], a[3]};
  const uint64_t idx = indexes[i];
  const uint64_t* ap = auth_paths + i * (size_t)(height - 1) * 4;
  for (unsigned level = 0; level < height; level++) {
    const uint64_t* sp = level == 0 ? leaf_siblings + i * 4 : ap + (size_t)(level - 1) * 4;
    uint64_t s0 = sp[0], s1 = sp[1], s2 = sp[2], s3 = sp[3];
    bool right = (idx >> level) & 1;  // set bit: current node is the right child
#pragma unroll
    for (int l = 8; l < 25; l++) a[l] = 0;
    a[0] = right ? s0 : cur[0]; a[1] = right ? s1 : cur[1]; a[2] = right ? s2 : cur[2]; a[3] = right ? s3 : cur[3];
    a[4] = right ? cur[0] : s0; a[5] = right ? cur[1] : s1; a[6] = right ? cur[2] : s2; a[7] = right ? cur[3] : s3;
    keccak_f1600(a);
    cur[0] = a[0]; cur[1] = a[1]; cur[2] = a[2]; cur[3] = a[3];
  }
  if (roots_out) {
    roots_out[i * 4 + 0] = cur[0]; roots_out[i * 4 + 1] = cur[1];
    roots_out[i * 4 + 2] = cur[2]; roots_out[i * 4 + 3] = cur[3];
  }
  if (ok_out)
    ok_out[i] = expected_root && cur[0] == expected_root[0] && cur[1] == expected_root[1] &&
                cur[2] == expected_root[2] && cur[3] == expected_root[3];
}

// ---- the same path recompute for SMALL batches (one WHIR round opens 64..256 paths): one WARP per path.
// A path is 24 dependent permutations; one thread runs them in ~8 us each, so a round's paths take 0.2 ms however
// few they are.  Here lane l = x + 5y of a warp holds state lane A[x, y] (lanes 25..31 idle) and a round is a few
// exchange stages between the lanes.  Two exchange mechanisms (template parameter SMEM):
//   shuffles:       theta's column parities (4 independent 64-bit shuffles) and D (2), then rho + pi + chi as ONE stage
//                   (three independent shuffles fetch B[x, y], B[x+1, y], B[x+2, y] straight from the rotated pre-pi
//                   lanes): 18 SHFL in three dependent stages per round;
//   shared memory:  the warp parks the state in a 25-lane shared array; every lane reads the two neighbouring COLUMNS
//                   (10 independent LDS.64) and forms theta's D by itself, parks the rotated value in a second array
//                   and reads chi's three operands from their pre-pi slots: two store -> load round trips per round,
//                   one 64-bit access where the shuffle path needs two 32-bit ones.
struct KeccakLaneCtx {
  int l5, l10, l15, l20;   // lanes of the same column (theta parities)
  int xm1, xp1;            // a lane of column x-1 / x+1 (theta's D)
  int cm0, cp0;            // the row-0 lane of column x-1 / x+1 (shared-memory path)
  int rot;                 // rho rotation of THIS lane's value before it leaves (mod 32)
  bool swap;               // rho rotation >= 32: exchange the halves first
  int s0, s1, s2;          // rho + pi + chi in one stage: the lanes whose rotated values become B[x, y], B[x+1, y], B[x+2, y]
};

__device__ __forceinline__ uint64_t shfl64(uint64_t v, int src) {
  uint32_t lo = __shfl_sync(0xffffffffu, (uint32_t)v, src);
  uint32_t hi = __shfl_sync(0xffffffffu, (uint32_t)(v >> 32), src);
  return ((uint64_t)hi << 32) | lo;
}

__device__ __forceinline__ KeccakLaneCtx keccak_lane_ctx(int lane) {
  // rho offsets by lane index x + 5y (FIPS-202 table 2)
  const int kRot[25] = {0, 1, 62, 28, 27, 36, 44, 6, 55, 20, 3, 10, 43, 25, 39, 41, 45, 15, 21, 8, 18, 2, 61, 56, 14};
  KeccakLaneCtx c;
  const int l = lane < 25 ? lane : 0, x = l % 5, y = l / 5;
  c.l5 = (l + 5) % 25; c.l10 = (l + 10) % 25; c.l15 = (l + 15) % 25; c.l20 = (l + 20) % 25;
  c.cm0 = (x + 4) % 5; c.cp0 = (x + 1) % 5;
  c.xm1 = c.cm0 + 5 * y; c.xp1 = c.cp0 + 5 * y;
  c.rot = kRot[l] & 31; c.swap = kRot[l] >= 32;
  // pi: B[y', 2x' + 3y'] = A[x', y'];  lane (X, Y) receives from the (x', y') with y' = X, 2x' + 3y' = Y (mod 5);
  // chi reads B[x+1, y] and B[x+2, y] as well: fetch all three straight from their pre-pi lanes (one exchange stage
  // instead of the permuting exchange followed by chi's two)
  auto pi_src = [](int X, int Y) { const int yp = X, xp = ((Y - 3 * yp) % 5 + 5) * 3 % 5; return xp + 5 * yp; };   // 2^-1 = 3 (mod 5)
  c.s0 = pi_src(x, y); c.s1 = pi_src((x + 1) % 5, y); c.s2 = pi_src((x + 2) % 5, y);
  return c;
}

// rho on the two halves: optional swap (rotation >= 32), then two funnel shifts by rot mod 32
__device__ __forceinline__ uint64_t keccak_lane_rho(uint64_t a, const KeccakLaneCtx& c) {
  uint32_t lo = (uint32_t)a, hi = (uint32_t)(a >> 32);
  const uint32_t l2 = c.swap ? hi : lo, h2 = c.swap ? lo : hi;
  const uint32_t nh = __funnelshift_l(l2, h2, c.rot), nl = __funnelshift_l(h2, l2, c.rot);
  return ((uint64_t)nh << 32) | nl;
}

// sA, sB: this warp's two 32-lane exchange arrays (shared-memory path only)
template <bool SMEM>
__device__ __forceinline__ uint64_t keccak_f1600_warp(uint64_t a, const KeccakLaneCtx& c, int lane, uint64_t* sA,
                                                      uint64_t* sB) {
#pragma unroll 1
  for (int rnd = 0; rnd < 24; rnd++) {
    const uint64_t rc = lane == 0 ? kRC[rnd] : 0;
    uint64_t cm, cp;
    // theta
    if constexpr (SMEM) {
      sA[lane] = a;
      __syncwarp();
      cm = sA[c.cm0] ^ sA[c.cm0 + 5] ^ sA[c.cm0 + 10] ^ sA[c.cm0 + 15] ^ sA[c.cm0 + 20];
      cp = sA[c.cp0] ^ sA[c.cp0 + 5] ^ sA[c.cp0 + 10] ^ sA[c.cp0 + 15] ^ sA[c.cp0 + 20];
    } else {
      const uint64_t col = a ^ shfl64(a, c.l5) ^ shfl64(a, c.l10) ^ shfl64(a, c.l15) ^ shfl64(a, c.l20);
      cm = shfl64(col, c.xm1); cp = shfl64(col, c.xp1);
    }
    a ^= cm ^ ((cp << 1) | (cp >> 63));
    // rho (rotate own value), then pi and chi's operands as three independent fetches of the rotated lanes
    const uint64_t r = keccak_lane_rho(a, c);
    uint64_t b, b1, b2;
    if constexpr (SMEM) {
      sB[lane] = r;
      __syncwarp();
      b = sB[c.s0]; b1 = sB[c.s1]; b2 = sB[c.s2];
    } else {
      b = shfl64(r, c.s0); b1 = shfl64(r, c.s1); b2 = shfl64(r, c.s2);
    }
    a = b ^ (~b1 & b2) ^ rc;
  }
  return a;
}

constexpr size_t MERKLE_WARP_MAX = 8192;   // up to here a warp per path fits the machine in one wave (148 SMs x 64 warps)
template <int WARPS, bool SMEM>
__global__ void __launch_bounds__(32 * WARPS) k_merkle_paths_warp(const uint8_t* __restrict__ leaves, size_t leaf_len,
                                                                   const uint64_t* __restrict__ leaf_siblings,
                                                                   const uint64_t* __restrict__ auth_paths,
                                                                   const uint64_t* __restrict__ indexes, unsigned height,
                                                                   size_t n, const uint64_t* __restrict__ expected_root,
                                                                   uint64_t* __restrict__ roots_out,
                                                                   uint8_t* __restrict__ ok_out) {
  __shared__ uint64_t sx[SMEM ? WARPS : 1][2][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t i = (size_t)blockIdx.x * WARPS + warp;
  if (i >= n) return;   // whole warps leave together
  uint64_t* sA = sx[SMEM ? warp : 0][0];
  uint64_t* sB = sx[SMEM ? warp : 0][1];
  const KeccakLaneCtx c = keccak_lane_ctx(lane);
  // leaf: Absorb(leaf) block by block (overwrite the rate lanes, permute when more data follows), then the permutation
  // at the head of Squeeze.  leaf_len is a positive multiple of 8 (checked by the entry point).
  uint64_t a = 0;
  const uint64_t* leaf = reinterpret_cast<const uint64_t*>(leaves + i * leaf_len);
  const size_t words = leaf_len / 8;
  const uint64_t idx = indexes[i];
  const uint64_t* ap = auth_paths + i * (size_t)(height - 1) * 4;
  // the next block / sibling is fetched BEFORE the permutation in front of it, so its HBM latency hides behind it
  uint64_t nxt = (size_t)lane < words && lane < KECCAK_RATE_LANES ? leaf[lane] : 0;
  size_t off = 0;
  while (words - off > (size_t)KECCAK_RATE_LANES) {
    if (lane < KECCAK_RATE_LANES) a = nxt;
    off += KECCAK_RATE_LANES;
    nxt = (size_t)lane < words - off && lane < KECCAK_RATE_LANES ? leaf[off + lane] : 0;
    a = keccak_f1600_warp<SMEM>(a, c, lane, sA, sB);
  }
  if ((size_t)lane < words - off) a = nxt;
  uint64_t sib = (lane < 8 && height > 0) ? leaf_siblings[i * 4 + (lane & 3)] : 0;
  a = keccak_f1600_warp<SMEM>(a, c, lane, sA, sB);
  for (unsigned level = 0; level < height; level++) {
    const bool right = (idx >> level) & 1;       // set bit: current node is the right child
    const uint64_t cur = shfl64(a, lane & 3);    // lanes 0..7 see cur[lane & 3]
    uint64_t v = 0;
    if (lane < 8) v = ((lane < 4) == right) ? sib : cur;   // left half = sibling iff we are the right child
    if (lane < 8 && level + 1 < height) sib = ap[(size_t)level * 4 + (lane & 3)];
    a = keccak_f1600_warp<SMEM>(v, c, lane, sA, sB);
  }
  if (roots_out && lane < 4) roots_out[i * 4 + lane] = a;
  if (ok_out) {
    const bool eq = lane >= 4 || (expected_root && a == expected_root[lane]);
    const unsigned all = __ballot_sync(0xffffffffu, eq);
    if (lane == 0) ok_out[i] = (expected_root && all == 0xffffffffu) ? 1 : 0;
  }
}

// ---- Keccak duplex (b200g16_keccak_duplex_batch): keccakSponge.Digest with Absorb / Squeeze in any order and the
// state carried across calls.  A digest is 26 words: the 25 lanes, then absorb_pos (low half) and squeeze_pos (high
// half).  Every sponge runs the same op script (device memory, read uniformly); keccak_duplex.cuh cuts each op into
// segments that stay inside one rate block, and a segment touches the rate lanes it overlaps, byte by byte where it
// starts or ends inside a lane or the row is not 8-byte aligned, one 64-bit access otherwise.
constexpr int DIGEST_WORDS = 26;

struct DuplexTag {
  uint64_t lane[8];   // state lanes 17..24 of NewKeccakWithTag (the tag's bytes 136..199, zero-padded)
  int use;            // 1: start every sponge from this state, 0: continue from its digest
};

__device__ __forceinline__ uint64_t duplex_positions(uint32_t absorb_pos, uint32_t squeeze_pos) {
  return (uint64_t)absorb_pos | ((uint64_t)squeeze_pos << 32);
}

// bytes [lo, hi) of the lane whose byte 0 maps to p (only p[lo..hi) is touched)
__device__ __forceinline__ uint64_t duplex_load(const uint8_t* p, uint32_t lo, uint32_t hi) {
  if (lo == 0 && hi == 8 && ((uintptr_t)p & 7) == 0) return *reinterpret_cast<const uint64_t*>(p);
  uint64_t v = 0;
  for (uint32_t k = lo; k < hi; k++) v |= (uint64_t)p[k] << (8 * k);
  return v;
}

__device__ __forceinline__ void duplex_store(uint8_t* p, uint64_t v, uint32_t lo, uint32_t hi) {
  if (lo == 0 && hi == 8 && ((uintptr_t)p & 7) == 0) { *reinterpret_cast<uint64_t*>(p) = v; return; }
  for (uint32_t k = lo; k < hi; k++) p[k] = (uint8_t)(v >> (8 * k));
}

__device__ __forceinline__ uint64_t duplex_mask(uint32_t lo, uint32_t hi) {
  return (hi == 8 ? ~0ull : (1ull << (8 * hi)) - 1) & ~((1ull << (8 * lo)) - 1);
}

// One thread per sponge, 25 lanes in registers.  A warp stages its 32 digests (6656 contiguous bytes) through shared
// memory in and out, as k_keccak_f_batch does, so the digest traffic is coalesced.
constexpr int DUPLEX_THREADS = 128;
__global__ void __launch_bounds__(DUPLEX_THREADS) k_duplex_thread(uint64_t* __restrict__ digests, size_t n, DuplexTag tag,
                                                                  const b200g16_duplex_op* __restrict__ ops, size_t n_ops,
                                                                  const uint8_t* __restrict__ in, size_t in_stride,
                                                                  uint8_t* __restrict__ out, size_t out_stride) {
  __shared__ uint64_t sm[DUPLEX_THREADS / 32][32 * DIGEST_WORDS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t warp_first = (size_t)blockIdx.x * DUPLEX_THREADS + (size_t)warp * 32;
  if (warp_first >= n) return;   // whole warps leave together
  const uint32_t in_warp = n - warp_first < 32 ? (uint32_t)(n - warp_first) : 32;
  uint64_t* g = digests + warp_first * DIGEST_WORDS;
  const uint32_t words = in_warp * DIGEST_WORDS;
  uint64_t* mine = sm[warp] + lane * DIGEST_WORDS;
  if (!tag.use) {
#pragma unroll
    for (int j = 0; j < DIGEST_WORDS; j++) {
      const uint32_t w = lane + 32 * j;
      if (w < words) sm[warp][w] = g[w];
    }
    __syncwarp();
  }
  if ((uint32_t)lane < in_warp) {
    const size_t i = warp_first + lane;
    uint64_t a[25];
    DuplexWalk w;
    if (tag.use) {
#pragma unroll
      for (int l = 0; l < 25; l++) a[l] = l < KECCAK_RATE_LANES ? 0 : tag.lane[l - KECCAK_RATE_LANES];
      w.absorb_pos = 0;
      w.squeeze_pos = DUPLEX_RATE;
    } else {
#pragma unroll
      for (int l = 0; l < 25; l++) a[l] = mine[l];
      w.absorb_pos = (uint32_t)mine[25];
      w.squeeze_pos = (uint32_t)(mine[25] >> 32);
    }
    const uint8_t* in_row = in + i * in_stride;
    uint8_t* out_row = out + i * out_stride;
    uint64_t in_off = 0, out_off = 0;
    for (size_t k = 0; k < n_ops; k++) {
      const b200g16_duplex_op op = ops[k];
      const bool sq = op.squeeze != 0;
      duplex_op_begin(w, op.len, sq ? out_off : in_off);
      while (w.left) {
        const DuplexSeg s = duplex_next(w, sq);
        if (s.permute) keccak_f1600(a);
        // lane l's byte 0 sits at row byte s.row_off + 8l - s.rate_off (only its bytes inside the segment are touched)
        const long long base = (long long)s.row_off - (long long)s.rate_off;
#pragma unroll
        for (int l = 0; l < KECCAK_RATE_LANES; l++) {
          uint32_t lo, hi;
          if (!duplex_lane_span(s, l, &lo, &hi)) continue;
          if (sq) {
            duplex_store(out_row + base + 8 * l, a[l], lo, hi);
          } else {
            const uint64_t m = duplex_mask(lo, hi);
            a[l] = (a[l] & ~m) | (duplex_load(in_row + base + 8 * l, lo, hi) & m);
          }
        }
      }
      duplex_op_end(w, sq);
      if (sq) out_off = w.row_off;
      else in_off = w.row_off;
    }
#pragma unroll
    for (int l = 0; l < 25; l++) mine[l] = a[l];
    mine[25] = duplex_positions(w.absorb_pos, w.squeeze_pos);
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < DIGEST_WORDS; j++) {
    const uint32_t w = lane + 32 * j;
    if (w < words) g[w] = sm[warp][w];
  }
}

// One WARP per sponge, for the few sponges of a transcript replay: lane l = x + 5y holds state lane A[x, y] and the
// permutation is keccak_f1600_warp (as k_merkle_paths_warp runs it); lane l < 17 overwrites or emits the bytes of its
// lane that fall inside a segment.
template <int WARPS, bool SMEM>
__global__ void __launch_bounds__(32 * WARPS) k_duplex_warp(uint64_t* __restrict__ digests, size_t n, DuplexTag tag,
                                                             const b200g16_duplex_op* __restrict__ ops, size_t n_ops,
                                                             const uint8_t* __restrict__ in, size_t in_stride,
                                                             uint8_t* __restrict__ out, size_t out_stride) {
  __shared__ uint64_t sx[SMEM ? WARPS : 1][2][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t i = (size_t)blockIdx.x * WARPS + warp;
  if (i >= n) return;   // whole warps leave together
  uint64_t* sA = sx[SMEM ? warp : 0][0];
  uint64_t* sB = sx[SMEM ? warp : 0][1];
  const KeccakLaneCtx c = keccak_lane_ctx(lane);
  uint64_t* dg = digests + i * DIGEST_WORDS;
  uint64_t a;
  DuplexWalk w;
  if (tag.use) {
    a = 0;
#pragma unroll
    for (int j = 0; j < 8; j++)
      if (lane == KECCAK_RATE_LANES + j) a = tag.lane[j];
    w.absorb_pos = 0;
    w.squeeze_pos = DUPLEX_RATE;
  } else {
    a = lane < 25 ? dg[lane] : 0;
    const uint64_t pos = dg[25];
    w.absorb_pos = (uint32_t)pos;
    w.squeeze_pos = (uint32_t)(pos >> 32);
  }
  const uint8_t* in_row = in + i * in_stride;
  uint8_t* out_row = out + i * out_stride;
  uint64_t in_off = 0, out_off = 0;
  for (size_t k = 0; k < n_ops; k++) {
    const b200g16_duplex_op op = ops[k];
    const bool sq = op.squeeze != 0;
    duplex_op_begin(w, op.len, sq ? out_off : in_off);
    while (w.left) {
      const DuplexSeg s = duplex_next(w, sq);
      if (s.permute) a = keccak_f1600_warp<SMEM>(a, c, lane, sA, sB);
      uint32_t lo, hi;
      if (lane < KECCAK_RATE_LANES && duplex_lane_span(s, lane, &lo, &hi)) {
        const long long at = (long long)s.row_off - (long long)s.rate_off + 8 * lane;
        if (sq) {
          duplex_store(out_row + at, a, lo, hi);
        } else {
          const uint64_t m = duplex_mask(lo, hi);
          a = (a & ~m) | (duplex_load(in_row + at, lo, hi) & m);
        }
      }
    }
    duplex_op_end(w, sq);
    if (sq) out_off = w.row_off;
    else in_off = w.row_off;
  }
  if (lane < 25) dg[lane] = a;
  if (lane == 0) dg[25] = duplex_positions(w.absorb_pos, w.squeeze_pos);
}

// *bad = 1 if a digest holds a position above 136 (run before a continuing call changes any digest)
__global__ void __launch_bounds__(256) k_duplex_check(const uint64_t* __restrict__ digests, size_t n,
                                                      uint32_t* __restrict__ bad) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t pos = digests[i * DIGEST_WORDS + 25];
  if ((uint32_t)pos > DUPLEX_RATE || (uint32_t)(pos >> 32) > DUPLEX_RATE) *bad = 1;
}

// ------------------------------------------------------------------------------ host drivers
int keccak_f_batch_device(b200g16_ctx* ctx, uint64_t* d_states, size_t n) {
  if (n == 0) return 0;
  unsigned grid = (unsigned)((n + KF_THREADS - 1) / KF_THREADS);
  k_keccak_f_batch<B200_KECCAK_FMA_MASK><<<grid, KF_THREADS, 0, ctx->stream>>>(d_states, n);
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  return 0;
}

int sponge_batch_device(b200g16_ctx* ctx, const uint8_t* d_in, size_t in_len, size_t n, uint8_t* d_out,
                        size_t out_len) {
  if (n == 0) return 0;
  int aligned8 = (in_len % 8 == 0) && (((uintptr_t)d_in) % 8 == 0);
  k_sponge_batch<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(d_in, in_len, n, d_out, out_len, aligned8);
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  return 0;
}

int merkle_paths_device(b200g16_ctx* ctx, const uint8_t* d_leaves, size_t leaf_len, const uint64_t* d_sib,
                        const uint64_t* d_auth, const uint64_t* d_idx, unsigned height, size_t n,
                        const uint64_t* d_expected_root, uint64_t* d_roots, uint8_t* d_ok) {
  if (n == 0) return 0;
  if (n <= MERKLE_WARP_MAX) {   // latency-bound batch (a WHIR round's queries): one warp per path
    // experiment knob (tools/sweep.py --merkle): B200G16_MERKLE_WARP = 10*warps_per_cta + (1: shared memory, 0: shuffles)
    // Measured (profiles/r02n_merkle_warp_sweep.jsonl, height 20, 512 B leaves): 64..256 paths 0.071 ms with one warp
    // per CTA exchanging through shared memory (shuffles 0.077, four warps per CTA 0.079 / 0.094); from ~1000 paths the
    // SMs hold several warps each and two-warp CTAs with shuffles win (1024: 0.090 against 0.095; 4096: 0.190 / 0.314).
    const char* e = getenv("B200G16_MERKLE_WARP");
    const int cfg = e ? atoi(e) : (n <= 512 ? 11 : 20);
#define B200_MERKLE_LAUNCH(W, S)                                                                                     \
  k_merkle_paths_warp<W, S><<<(unsigned)((n + W - 1) / W), 32 * W, 0, ctx->stream>>>(                                \
      d_leaves, leaf_len, d_sib, d_auth, d_idx, height, n, d_expected_root, d_roots, d_ok)
    switch (cfg) {
      case 10: B200_MERKLE_LAUNCH(1, false); break;
      case 11: B200_MERKLE_LAUNCH(1, true); break;
      case 20: B200_MERKLE_LAUNCH(2, false); break;
      case 21: B200_MERKLE_LAUNCH(2, true); break;
      case 40: B200_MERKLE_LAUNCH(4, false); break;
      case 41: B200_MERKLE_LAUNCH(4, true); break;
      default: return B200G16_ERR_ARG;
    }
#undef B200_MERKLE_LAUNCH
    ctx->launches++;
    B200_CUDA(cudaGetLastError());
    return 0;
  }
  k_merkle_paths<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(d_leaves, leaf_len, d_sib, d_auth, d_idx,
                                                                        height, n, d_expected_root, d_roots, d_ok);
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  return 0;
}

// Up to here one warp per sponge; above, one thread per sponge.  Measured (profiles/r03c_keccak_duplex.jsonl, transcript
// script, 6 permutations per sponge, device path, median call): the warp form takes 0.078-0.080 ms from 1 to 1024
// sponges where the thread form takes 0.161-0.172 (one thread runs the 6 dependent permutations about twice as slowly
// as a warp), 0.107 against 0.164 ms at 4096, 0.150 against 0.160 at 8192; at 16384 the warps no longer fit one wave
// (148 SMs x 64 warps) and the thread form wins, 0.163 against 0.234 ms.
constexpr size_t DUPLEX_WARP_MAX = 8192;

// tag: NULL = continue from the digests, else tag_len (<= 64) bytes of NewKeccakWithTag.  d_ops in device memory.
int keccak_duplex_device(b200g16_ctx* ctx, uint64_t* d_digests, size_t n, const uint8_t* tag, size_t tag_len,
                         const b200g16_duplex_op* d_ops, size_t n_ops, const uint8_t* d_in, size_t in_stride,
                         uint8_t* d_out, size_t out_stride) {
  if (n == 0) return 0;
  DuplexTag t = {};
  t.use = tag != nullptr;
  for (size_t j = 0; tag && j < tag_len; j++) t.lane[j / 8] |= (uint64_t)tag[j] << (8 * (j % 8));
  // experiment knob (tools/duplex_bench.py): B200G16_DUPLEX_WARP = 1 forces the warp form, 0 the thread form
  const char* e = getenv("B200G16_DUPLEX_WARP");
  const bool warp = e && *e ? atoi(e) != 0 : n <= DUPLEX_WARP_MAX;
  if (warp) {
    // the exchange mechanism and CTA shape k_merkle_paths_warp measured best (profiles/r02o_merkle_warp_sweep.jsonl):
    // shared memory with one warp per CTA up to 512 sponges, shuffles with two warps per CTA above
    if (n <= 512)
      k_duplex_warp<1, true><<<(unsigned)n, 32, 0, ctx->stream>>>(d_digests, n, t, d_ops, n_ops, d_in, in_stride, d_out,
                                                                   out_stride);
    else
      k_duplex_warp<2, false><<<(unsigned)((n + 1) / 2), 64, 0, ctx->stream>>>(d_digests, n, t, d_ops, n_ops, d_in,
                                                                                in_stride, d_out, out_stride);
  } else {
    k_duplex_thread<<<(unsigned)((n + DUPLEX_THREADS - 1) / DUPLEX_THREADS), DUPLEX_THREADS, 0, ctx->stream>>>(
        d_digests, n, t, d_ops, n_ops, d_in, in_stride, d_out, out_stride);
  }
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  return 0;
}

// *bad = whether a digest holds a position above 136; d_flag: 4 bytes of device scratch.  Synchronises the stream.
int keccak_duplex_check_device(b200g16_ctx* ctx, const uint64_t* d_digests, size_t n, uint32_t* d_flag, bool* bad) {
  *bad = false;
  if (n == 0) return 0;
  B200_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(uint32_t), ctx->stream));
  k_duplex_check<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_digests, n, d_flag);
  ctx->launches++;
  B200_CUDA(cudaGetLastError());
  uint32_t h = 0;
  B200_CUDA(cudaMemcpyAsync(&h, d_flag, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  *bad = h != 0;
  return 0;
}

}  // namespace b200
