// tests/emu/dense_verify_emu.cc — TEST INFRASTRUCTURE: runs the two forms of the ZK_POS_DENSE structure verify
// (lookup.cuh: pos_verify_dense_row, one row at a time, and pos_verify_dense_strip, the typed strip form the
// device uses for narrow rw tables) serially on the CPU over the same table, so the CPU suite can diff their
// flag and split row.  Built by tests/test_emu_dense_verify.py with plain g++; never used by the product.
#include <stdint.h>
#include <string.h>

#include "../../zkevm-specs_b200/csrc/lookup.cuh"

using namespace zk;

template <int WC, int WT>
static void run_strips(const IndexDev& d, u32* ok) {
  for (u64 r = 0; r < d.tab.n_rows; r += ZK_DENSE_STRIP) pos_verify_dense_strip<WC, WT>(d, ok, r);
}

// `buf`: the counter column (wc = 4 or 8 bytes per row) at off_counter, the tag column (wt = 1 byte per row, or
// 0: one constant 32-byte cell) at off_tag.  Returns -1 for a layout the strip form does not take.
extern "C" int emu_dense_verify(const unsigned char* buf, uint64_t off_counter, uint32_t wc, uint64_t off_tag, uint32_t wt,
                                uint64_t n_rows, int has_tail, uint32_t* ok_row, uint32_t* ok_strip) {
  IndexDev d;
  memset(&d, 0, sizeof(d));
  d.tab.base = buf;
  d.tab.n_rows = n_rows;
  d.tab.n_cols = 3;
  d.tab.flags = nullptr;
  for (u32 c = 0; c < ZK_MAX_TABLE_COLS; c++) d.tab.width[c] = 0;
  d.tab.off[0] = off_counter;
  d.tab.width[0] = (unsigned char)wc;
  d.tab.off[1] = off_tag;  // unused column
  d.tab.off[2] = off_tag;
  d.tab.width[2] = (unsigned char)wt;
  d.n_key = 5;
  for (u32 j = 0; j < 5; j++) d.key_cols[j] = j;
  d.pos_kind = ZK_POS_DENSE;
  d.tail_col = 2;
  d.tail_val = 1;
  d.tail_key = has_tail ? 2 : -1;
  ok_row[0] = ok_strip[0] = 1;
  ok_row[1] = ok_strip[1] = (u32)n_rows;
  for (u64 r = 0; r < n_rows; r++) pos_verify_dense_row(d, ok_row, r);
  if (wc == 4 && wt == 0) run_strips<4, 0>(d, ok_strip);
  else if (wc == 4 && wt == 1) run_strips<4, 1>(d, ok_strip);
  else if (wc == 8 && wt == 0) run_strips<8, 0>(d, ok_strip);
  else if (wc == 8 && wt == 1) run_strips<8, 1>(d, ok_strip);
  else return -1;
  return 0;
}
