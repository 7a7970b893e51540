// tests/emu/withdrawal_emu.cc — TEST INFRASTRUCTURE: runs the withdrawal circuit's row body (csrc/withdrawal.cu:
// check_withdrawal_row, the __host__ __device__ function k_check_withdrawal calls) serially on the CPU over the lookup
// indexes of tests/emu/zk_emu.cu, in the canonical and the packed storage instance, so the CPU suite can diff it against
// the oracle.  Built by tests/test_emu_withdrawal.py with plain g++; never used by the product.
#include "zk_emu.cu"
#include "../../zkevm-specs_b200/csrc/withdrawal.cu"

extern "C" int emu_check_withdrawal(const uint64_t* rows, uint64_t n_rows, const uint64_t* keccak, uint64_t n_keccak,
                                    const uint64_t* mpt, uint64_t n_mpt, const uint64_t* block, uint64_t n_block,
                                    const uint64_t r[4], uint64_t max, uint64_t row_begin, uint64_t row_end, uint64_t row_base,
                                    const uint64_t challenge[4], uint32_t* first_fail, uint64_t* fail_count) {
  const Fr ch{{challenge[0], challenge[1], challenge[2], challenge[3]}};
  const u32 kk[5] = {0, 1, 2, 3, 4}, mk[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}, bk[3] = {0, 2, 3};
  IndexStore s1, s2, s3;
  IndexDev kix = build_index((const u64*)keccak, n_keccak, 5, kk, 5, ch, s1);
  IndexDev mix = build_index((const u64*)mpt, n_mpt, 12, mk, 12, ch, s2);
  IndexDev bix = build_index((const u64*)block, n_block, 4, bk, 3, ch, s3);
  Store ws;
  WitnessDev w = make_witness(ws, (const u64*)rows, n_rows, WD_COLS, nullptr);
  ResultDev res;
  init_result(res, first_fail, fail_count, WD_N_CONSTRAINTS);
  Fr rp[WD_MAX_RLP];
  wd_rpow_table(Fr{{r[0], r[1], r[2], r[3]}}, rp);
  CheckRange rg{row_begin, row_end, row_base, 0};
  bool canon = true;
  for (u32 c = 0; c < WD_COLS; c++) canon = canon && w.width[c] == 32;
  for (u64 i = row_begin; i < row_end; i++) {
    if (canon) check_withdrawal_row<L_CANON>(w, rg, kix, mix, bix, rp, max, res, i);
    else check_withdrawal_row<L_ANY>(w, rg, kix, mix, bix, rp, max, res, i);
  }
  return 0;
}

// the RLP bytes and the RLC of one row as the kernels stream them
extern "C" int emu_withdrawal_rlp(const uint64_t f[16], const uint64_t r[4], uint8_t out[140], uint64_t rlc[4]) {
  const u64* c = (const u64*)f;
  const Fr id = ld_cell(c), vid = ld_cell(c + 4), addr = ld_cell(c + 8), amt = ld_cell(c + 12);
  const WdRlp s = wd_rlp_shape(id, vid, addr, amt);
  struct Put {
    uint8_t* buf;
    void operator()(u32 byte, u32 pos) { buf[pos] = (uint8_t)byte; }
  } put{out};
  wd_rlp_emit(s, id, vid, addr, amt, put);
  Fr rp[WD_MAX_RLP];
  wd_rpow_table(Fr{{r[0], r[1], r[2], r[3]}}, rp);
  const Fr v = wd_rlc(s, id, vid, addr, amt, rp);
  memcpy(rlc, v.l, 32);
  return (int)s.len;
}
