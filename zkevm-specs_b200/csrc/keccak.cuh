// keccak.cuh — Keccak-256 (original 0x01 padding, rate 136) on the device.
//
// The reference takes it from third-party packages (pycryptodome / eth_utils: src/zkevm_specs/util/hash.py:7-10,
// evm_circuit/instruction.py:1338-1340); the algorithm is the published Keccak-f[1600] sponge.  Used here by
// the BeginTx gate program (contract address = keccak(rlp([caller, nonce]))[12:], instruction.py:1338) and by
// the keccak-table / code-hash generation kernels (evm_circuit/typing.py:854-865, bytecode_circuit.py:182-186).
// One thread absorbs one message; the 25 lanes live in registers (the permutation is fully unrolled).
#pragma once
#include "fr.cuh"

namespace zk {

ZK_HD u64 rotl64(u64 v, int s) { return s ? (v << s) | (v >> (64 - s)) : v; }

#define ZK_KECCAK_RC                                                                                             \
  {0x0000000000000001ull, 0x0000000000008082ull, 0x800000000000808aull, 0x8000000080008000ull, 0x000000000000808bull, \
   0x0000000080000001ull, 0x8000000080008081ull, 0x8000000000008009ull, 0x000000000000008aull, 0x0000000000000088ull, \
   0x0000000080008009ull, 0x000000008000000aull, 0x000000008000808bull, 0x800000000000008bull, 0x8000000000008089ull, \
   0x8000000000008003ull, 0x8000000000008002ull, 0x8000000000000080ull, 0x000000000000800aull, 0x800000008000000aull, \
   0x8000000080008081ull, 0x8000000000008080ull, 0x0000000080000001ull, 0x8000000080008008ull}
#ifdef __CUDACC__
// round constants in constant memory: the round index is the same in every lane (a broadcast read), and a
// per-thread copy would be a 192-byte stack array indexed by the rolled round loop
__constant__ u64 kKeccakRC[24] = ZK_KECCAK_RC;
#endif

ZK_HD void keccak_f1600(u64 a[25]) {
#ifdef __CUDA_ARCH__
  const u64* RC = kKeccakRC;
#else
  const u64 RC[24] = ZK_KECCAK_RC;
#endif
#pragma unroll 1
  for (int round = 0; round < 24; round++) {
    u64 c[5], d[5], b[25];
#pragma unroll
    for (int x = 0; x < 5; x++) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
#pragma unroll
    for (int x = 0; x < 5; x++) d[x] = c[(x + 4) % 5] ^ rotl64(c[(x + 1) % 5], 1);
#pragma unroll
    for (int i = 0; i < 25; i++) a[i] ^= d[i % 5];
    // rho + pi: b[y + 5 * ((2x + 3y) % 5)] = rot(a[x + 5y], r[x][y])
    b[0] = a[0];
    b[10] = rotl64(a[1], 1);
    b[20] = rotl64(a[2], 62);
    b[5] = rotl64(a[3], 28);
    b[15] = rotl64(a[4], 27);
    b[16] = rotl64(a[5], 36);
    b[1] = rotl64(a[6], 44);
    b[11] = rotl64(a[7], 6);
    b[21] = rotl64(a[8], 55);
    b[6] = rotl64(a[9], 20);
    b[7] = rotl64(a[10], 3);
    b[17] = rotl64(a[11], 10);
    b[2] = rotl64(a[12], 43);
    b[12] = rotl64(a[13], 25);
    b[22] = rotl64(a[14], 39);
    b[23] = rotl64(a[15], 41);
    b[8] = rotl64(a[16], 45);
    b[18] = rotl64(a[17], 15);
    b[3] = rotl64(a[18], 21);
    b[13] = rotl64(a[19], 8);
    b[14] = rotl64(a[20], 18);
    b[24] = rotl64(a[21], 2);
    b[9] = rotl64(a[22], 61);
    b[19] = rotl64(a[23], 56);
    b[4] = rotl64(a[24], 14);
#pragma unroll
    for (int y = 0; y < 25; y += 5)
#pragma unroll
      for (int x = 0; x < 5; x++) a[y + x] = b[y + x] ^ (~b[y + (x + 1) % 5] & b[y + (x + 2) % 5]);
    a[0] ^= RC[round];
  }
}

// byte k of the padded message stream of `msg` (len bytes): data, then 0x01, zeros, 0x80 at the end of the block
ZK_HD u64 keccak_lane(const unsigned char* msg, u64 len, u64 off) {  // 8 message bytes at offset `off`, zero past the end
  u64 v = 0;
#pragma unroll
  for (int k = 0; k < 8; k++)
    if (off + k < len) v |= (u64)msg[off + k] << (8 * k);
  return v;
}
// out[0..3] = the 32 digest bytes as little-endian u64 lanes (digest byte j = (out[j / 8] >> 8 (j % 8)) & 0xFF)
ZK_HD void keccak256(const unsigned char* msg, u64 len, u64 out[4]) {
  u64 a[25];
#pragma unroll
  for (int i = 0; i < 25; i++) a[i] = 0;
  const u64 n_blocks = len / 136 + 1;  // the padding always adds at least one byte
#pragma unroll 1
  for (u64 blk = 0; blk < n_blocks; blk++) {
    const u64 base = blk * 136;
#pragma unroll
    for (int i = 0; i < 17; i++) {
      u64 v = keccak_lane(msg, len, base + 8 * i);
      const u64 lo = base + 8 * i;
      if (len >= lo && len < lo + 8) v |= 0x01ull << (8 * (len - lo));  // first padding byte
      if (blk == n_blocks - 1 && i == 16) v |= 0x80ull << 56;            // last byte of the last block
      a[i] ^= v;
    }
    keccak_f1600(a);
  }
  out[0] = a[0];
  out[1] = a[1];
  out[2] = a[2];
  out[3] = a[3];
}
// the digest as a 256-bit big-endian integer split into (lo, hi) 128-bit halves — Word(int.from_bytes(digest, "big"))
ZK_HD void keccak_digest_to_word(const u64 d[4], u64 lo[2], u64 hi[2]) {
  // integer limb k (little-endian) = bytes 31-8k .. 24-8k of the digest, i.e. lane 3-k byte-swapped
  u64 sw[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    u64 v = d[3 - k], r = 0;
#pragma unroll
    for (int b = 0; b < 8; b++) r |= ((v >> (8 * b)) & 0xFF) << (8 * (7 - b));
    sw[k] = r;
  }
  lo[0] = sw[0];
  lo[1] = sw[1];
  hi[0] = sw[2];
  hi[1] = sw[3];
}

// The keccak table's input_rlc column, RLC(reversed(msg), r) = sum msg[i] * r^(len-1-i), folded in chunks: one chunk gives
// (val, pow) = (Horner value of its bytes, r^(chunk length)); two adjacent chunks combine as val = l.val * r.pow + r.val.
// val is canonical, pow and r_mont are in Montgomery form (canonical x Montgomery -> canonical; Montgomery x Montgomery
// -> Montgomery).
ZK_HD void rlc_chunk(const unsigned char* msg, u64 lo, u64 hi, const Fr& r_mont, Fr& val, Fr& pow) {
  Fr acc = fr_u64(0), pw = fr_to_mont(fr_u64(1));
  for (u64 i = lo; i < hi; i++) {
    acc = fr_add_u64(fr_montmul(acc, r_mont), msg[i]);
    pw = fr_montmul(pw, r_mont);
  }
  val = acc;
  pow = pw;
}
ZK_HD void rlc_combine(Fr& lval, Fr& lpow, const Fr& rval, const Fr& rpow) {
  lval = fr_add(fr_montmul(lval, rpow), rval);
  lpow = fr_montmul(lpow, rpow);
}

}  // namespace zk
