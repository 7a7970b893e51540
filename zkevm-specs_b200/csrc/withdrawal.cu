// withdrawal.cu — withdrawal-circuit row checker (one thread per row) and its witness assignment.
//
// Replaces the loop of verify_circuit, src/zkevm_specs/withdrawal_circuit.py:127-201.  Row = 8 cells
// (include/zkcheck.h ZK_CIRCUIT_WITHDRAWAL): withdrawal_id, validator_id, address, amount, hash lo/hi, root lo/hi;
// rotations {-1, 0, +1} without wrap.  Per row: the next-id equality, the keccak-table membership of the row's RLP
// encoding, the 12-column MPT lookup; global row MAX - 1 also owns the block-table lookup that follows the loop.
// Algorithmic bytes: 8 x 32 B per row + the looked-up keccak row (5 x 32 B) and MPT row (12 x 32 B).
//
// The RLP encoding rlp.encode([id, validator_id, address, amount]) is never materialised: its bytes are streamed
// straight from the cell limbs (wd_rlp_emit).  Every byte is below 256, so the RLC sum_i byte_i * r^(len-1-i) is a
// sum of one-limb products byte * (r^k * 2^64) (fr_montmul1) against a table of r^0..r^133 staged in shared memory,
// instead of a chain of dependent 4-limb Horner steps (profiles/README.md, round 4, measures both).
#include "circuit.cuh"
#include "keccak.cuh"
#include "../../include/zk_constraints.h"
#include "../../include/zkcheck.h"

namespace zk {

enum { W_ID, W_VALIDATOR, W_ADDRESS, W_AMOUNT, W_HASH_LO, W_HASH_HI, W_ROOT_LO, W_ROOT_HI, WD_COLS };
#define WD_MAX_RLP 134                 // 2 header bytes + 4 x (1 + 32): one keccak rate block (136 bytes)
#define WD_TAG_WITHDRAWAL_ROOT 9       // BlockContextFieldTag.WithdrawalRoot (evm_circuit/table.py:144)
#define WD_PROOF_WITHDRAWAL_MOD 8      // MPTProofType.WithdrawalMod (evm_circuit/table.py:338)
#define WD_PROOF_NON_EXISTING 4        // MPTProofType.NonExistingAccountProof (evm_circuit/table.py:334)

ZK_HD u32 clz64(u64 v) {
#ifdef __CUDA_ARCH__
  return (u32)__clzll((long long)v);
#else
  return v ? (u32)__builtin_clzll(v) : 64u;
#endif
}
// minimal big-endian byte length of the integer v.n (0 for 0)
ZK_HD u32 wd_nbytes(const Fr& v) {
  const u32 L = v.l[3] ? 3 : v.l[2] ? 2 : v.l[1] ? 1 : 0;
  const u64 top = L == 3 ? v.l[3] : L == 2 ? v.l[2] : L == 1 ? v.l[1] : v.l[0];
  return top ? 8 * L + (71 - clz64(top)) / 8 : 0;
}
// rlp.encode of one integer: 0 -> 0x80, below 0x80 -> the byte itself, else 0x80 + nb then the nb bytes
ZK_HD bool wd_single(const Fr& v, u32 nb) { return nb <= 1 && v.l[0] < 0x80; }
ZK_HD u32 wd_field_len(const Fr& v, u32 nb) { return wd_single(v, nb) ? 1 : 1 + nb; }

struct WdRlp {
  u32 nb[4];    // byte length of each field
  u32 payload;  // list payload length
  u32 len;      // whole encoding: header (1 byte, or 0xf8 + length once the payload reaches 56) + payload
};
ZK_HD WdRlp wd_rlp_shape(const Fr& id, const Fr& vid, const Fr& addr, const Fr& amt) {
  WdRlp s;
  s.nb[0] = wd_nbytes(id);
  s.nb[1] = wd_nbytes(vid);
  s.nb[2] = wd_nbytes(addr);
  s.nb[3] = wd_nbytes(amt);
  s.payload = wd_field_len(id, s.nb[0]) + wd_field_len(vid, s.nb[1]) + wd_field_len(addr, s.nb[2]) + wd_field_len(amt, s.nb[3]);
  s.len = (s.payload < 56 ? 1 : 2) + s.payload;
  return s;
}
// emit(byte, pos) for the bytes of one field starting at `pos`, in positional order; returns the position after it
template <class E>
ZK_HD u32 wd_emit_field(const Fr& v, u32 nb, u32 pos, E& emit) {
  if (wd_single(v, nb)) {
    emit(nb ? (u32)v.l[0] : 0x80u, pos);
    return pos + 1;
  }
  emit(0x80u + nb, pos);
  const u32 end = pos + 1 + nb;  // little-endian byte k of v sits at position end - 1 - k
#pragma unroll
  for (int L = 3; L >= 0; L--)
#pragma unroll
    for (int b = 7; b >= 0; b--) {
      const u32 k = 8 * L + b;
      if (k < nb) emit((u32)(v.l[L] >> (8 * b)) & 0xFFu, end - 1 - k);
    }
  return end;
}
// every byte of rlp.encode([id, validator_id, address, amount]) in positional order, no byte array
template <class E>
ZK_HD void wd_rlp_emit(const WdRlp& s, const Fr& id, const Fr& vid, const Fr& addr, const Fr& amt, E& emit) {
  u32 pos = 0;
  if (s.payload < 56) {
    emit(0xC0u + s.payload, pos++);
  } else {
    emit(0xF8u, pos++);
    emit(s.payload, pos++);
  }
  pos = wd_emit_field(id, s.nb[0], pos, emit);
  pos = wd_emit_field(vid, s.nb[1], pos, emit);
  pos = wd_emit_field(addr, s.nb[2], pos, emit);
  wd_emit_field(amt, s.nb[3], pos, emit);
}

// RLC(bytes(reversed(enc)), r) = sum_i enc[i] * r^(len-1-i), each term one fr_montmul1 against rp[k] = r^k * 2^64 mod p
struct WdRlcSum {
  const Fr* rp;
  u32 len;
  Fr acc;
  ZK_HD void operator()(u32 byte, u32 pos) {
    if (byte) acc = fr_add(acc, fr_montmul1(byte, rp[len - 1 - pos]));
  }
};
// the same value as a Horner chain acc = acc * r + byte (r_mont: r in Montgomery form); kept for the A/B build
// (-DZK_WD_HORNER) that profiles/README.md round 4 compares against
struct WdRlcHorner {
  Fr r_mont;
  Fr acc;
  ZK_HD void operator()(u32 byte, u32) { acc = fr_add_u64(fr_montmul(acc, r_mont), byte); }
};
ZK_HD Fr wd_rlc(const WdRlp& s, const Fr& id, const Fr& vid, const Fr& addr, const Fr& amt, const Fr* rp) {
#ifdef ZK_WD_HORNER
  WdRlcHorner h{fr_to_mont(fr_montmul1(1, rp[1])), fr_u64(0)};  // rp[1] = r * 2^64: montmul1(1, .) = r
  wd_rlp_emit(s, id, vid, addr, amt, h);
  return h.acc;
#else
  WdRlcSum sum{rp, s.len, fr_u64(0)};
  wd_rlp_emit(s, id, vid, addr, amt, sum);
  return sum.acc;
#endif
}
// rp[k] = r^k * 2^64 mod p for k < WD_MAX_RLP (host side: the table the kernels stage into shared memory)
inline void wd_rpow_table(const Fr& r, Fr* rp) {
  const Fr r_mont = fr_to_mont(r);
  rp[0] = fr_u128(0, 1);  // 2^64 < p
  for (int k = 1; k < WD_MAX_RLP; k++) rp[k] = fr_montmul(rp[k - 1], r_mont);
}

#define WD_CHECK(id, cond)   \
  do {                       \
    if (!(cond)) {           \
      fail(res, (id), row);  \
      return;                \
    }                        \
  } while (0)

// rows [b, e) of a shard; `row` = global row = row_base + i; max = MAX_WITHDRAWALS.  The row body runs for global rows
// below max; the block lookup after the loop runs at global row max - 1 (row 0 when max == 0: the caller then holds
// rows[-1] there, the row the reference reads).
template <int LAYOUT>
ZK_HD void check_withdrawal_row(const WitnessDev& w, const CheckRange& rg, const IndexDev& kec_ix, const IndexDev& mpt_ix,
                                const IndexDev& blk_ix, const Fr* rp, u64 max, const ResultDev& res, u64 i) {
  const u64 row = rg.row_base + i;
#define C(c) wcell_l<LAYOUT>(w, (c), i)
  if (row == (max ? max - 1 : 0)) {  // :199-201  block_lookup(WithdrawalRoot, rows[MAX-1].root)
    Fr key[3] = {fr_u64(WD_TAG_WITHDRAWAL_ROOT), C(W_ROOT_LO), C(W_ROOT_HI)};
    u32 hit;
    const int n = lookup<3>(blk_ix, key, &hit);
    ZK_REQUIRE(res, WD_BLOCK_LOOKUP, row, n >= 1);
    ZK_REQUIRE(res, WD_BLOCK_AMBIG, row, n <= 1);
  }
  if (row >= max) return;
  const Fr id = C(W_ID), amount = C(W_AMOUNT), hlo = C(W_HASH_LO), hhi = C(W_HASH_HI);
  // :153-158
  if (row + 1 < max) WD_CHECK(WD_NEXT_ID, fr_eq(wcell_l<LAYOUT>(w, W_ID, i + 1), fr_add(id, fr_u64(1))));
  const bool pad = fr_is_zero(amount);  // :150  is_not_padding = FQ(amount != 0)
  {  // :169-181  (q, q * RLC, q * len, hash.select(q)) is a member of the keccak table
    Fr key[5] = {fr_u64(0), fr_u64(0), fr_u64(0), fr_u64(0), fr_u64(0)};
    if (!pad) {
      const Fr vid = C(W_VALIDATOR), addr = C(W_ADDRESS);
      const WdRlp s = wd_rlp_shape(id, vid, addr, amount);
      key[0] = fr_u64(1);
      key[1] = wd_rlc(s, id, vid, addr, amount, rp);
      key[2] = fr_u64(s.len);
      key[3] = hlo;
      key[4] = hhi;
      WD_CHECK(WD_HASH_WORD, fr_fits128(hlo) && fr_fits128(hhi));
    }
    u32 hit;
    WD_CHECK(WD_KECCAK_LOOKUP, lookup<5>(kec_ix, key, &hit) >= 1);
  }
  {  // :184-193  every column of MPTTableRow: (address, proof_type, storage_key, root, root_prev, value, value_prev)
    const bool first = row == 0;
    Fr key[12] = {C(W_ADDRESS), fr_u64(pad ? WD_PROOF_NON_EXISTING : WD_PROOF_WITHDRAWAL_MOD),
                  fr_u128(id.l[0], id.l[1]), fr_u128(id.l[2], id.l[3]),  // Word(withdrawal_id.n)
                  C(W_ROOT_LO), C(W_ROOT_HI),
                  first ? fr_u64(0) : wcell_l<LAYOUT>(w, W_ROOT_LO, i - 1), first ? fr_u64(0) : wcell_l<LAYOUT>(w, W_ROOT_HI, i - 1),
                  hlo, hhi,  // the unselected hash
                  fr_u64(0), fr_u64(0)};
    u32 hit;
    WD_CHECK(WD_MPT_LOOKUP, lookup<12>(mpt_ix, key, &hit) >= 1);
  }
#undef C
}

#ifdef __CUDACC__
template <int LAYOUT>
__global__ void __launch_bounds__(256)
k_check_withdrawal(const __grid_constant__ WitnessDev w, const __grid_constant__ CheckRange rg, const __grid_constant__ IndexDev kec_ix,
                   const __grid_constant__ IndexDev mpt_ix, const __grid_constant__ IndexDev blk_ix, const Fr* __restrict__ rpow,
                   u64 max, const __grid_constant__ ResultDev res) {
  __shared__ Fr rp[WD_MAX_RLP];
  for (u32 k = threadIdx.x; k < WD_MAX_RLP; k += blockDim.x) rp[k] = rpow[k];
  __syncthreads();
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = rg.row_begin + (u64)blockIdx.x * blockDim.x + threadIdx.x; i < rg.row_end; i += stride)
    check_withdrawal_row<LAYOUT>(w, rg, kec_ix, mpt_ix, blk_ix, rp, max, res, i);
}

// zk_assign_withdrawal_circuit: one thread per circuit row.  rows = canonical [8][max][4], keccak = canonical [5][n + 1][4]
// (row 0 the all-zero row), records = [n][5][4].  The RLP bytes go to the thread's slice of a shared buffer, which the
// keccak sponge reads; the RLC is streamed from the cells like the checker's.
#define WD_ASSIGN_THREADS 128
__global__ void __launch_bounds__(WD_ASSIGN_THREADS)
k_assign_withdrawal(const u64* __restrict__ records, u64 n, u64 max, const Fr* __restrict__ rpow, u64* __restrict__ rows,
                    u64* __restrict__ keccak) {
  __shared__ Fr rp[WD_MAX_RLP];
  __shared__ unsigned char msg[WD_ASSIGN_THREADS * 136];
  for (u32 k = threadIdx.x; k < WD_MAX_RLP; k += blockDim.x) rp[k] = rpow[k];
  __syncthreads();
  const u64 nk = n + 1;
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < max; i += stride) {
    Fr cell[WD_COLS];
#pragma unroll
    for (int c = 0; c < WD_COLS; c++) cell[c] = fr_u64(0);
    if (i < n) {
      const u64* rec = records + i * 20;
      const Fr id = ld_cell(rec), vid = ld_cell(rec + 4), addr = ld_cell(rec + 8), amt = ld_cell(rec + 12);
      const WdRlp s = wd_rlp_shape(id, vid, addr, amt);
      struct Put {
        unsigned char* buf;
        ZK_HD void operator()(u32 byte, u32 pos) { buf[pos] = (unsigned char)byte; }
      } put{msg + threadIdx.x * 136};
      wd_rlp_emit(s, id, vid, addr, amt, put);
      u64 d[4];
      keccak256(put.buf, s.len, d);
      const Fr rlc = wd_rlc(s, id, vid, addr, amt, rp);
      cell[W_ID] = id;
      cell[W_VALIDATOR] = vid;
      cell[W_ADDRESS] = addr;
      cell[W_AMOUNT] = amt;
      // Word(bytes(keccak(rlp))): lo = digest bytes 0..15, hi = bytes 16..31, each read little-endian
      cell[W_HASH_LO] = fr_u128(d[0], d[1]);
      cell[W_HASH_HI] = fr_u128(d[2], d[3]);
      const Fr root = ld_cell(rec + 16);
      cell[W_ROOT_LO] = fr_u128(root.l[0], root.l[1]);
      cell[W_ROOT_HI] = fr_u128(root.l[2], root.l[3]);
      const Fr krow[5] = {fr_u64(1), rlc, fr_u64(s.len), cell[W_HASH_LO], cell[W_HASH_HI]};
#pragma unroll
      for (int c = 0; c < 5; c++) {
        u64* p = keccak + ((u64)c * nk + i + 1) * 4;
        p[0] = krow[c].l[0], p[1] = krow[c].l[1], p[2] = krow[c].l[2], p[3] = krow[c].l[3];
      }
    } else if (n) {  // Row(0, 0, 0, 0, Word(0), last_root)
      const Fr root = ld_cell(records + (n - 1) * 20 + 16);
      cell[W_ROOT_LO] = fr_u128(root.l[0], root.l[1]);
      cell[W_ROOT_HI] = fr_u128(root.l[2], root.l[3]);
    }
    if (i == 0)
#pragma unroll
      for (int c = 0; c < 5; c++) {
        u64* p = keccak + (u64)c * nk * 4;
        p[0] = p[1] = p[2] = p[3] = 0;
      }
#pragma unroll
    for (int c = 0; c < WD_COLS; c++) {
      u64* p = rows + ((u64)c * max + i) * 4;
      p[0] = cell[c].l[0], p[1] = cell[c].l[1], p[2] = cell[c].l[2], p[3] = cell[c].l[3];
    }
  }
}
#endif

}  // namespace zk
