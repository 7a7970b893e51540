// lookup.cuh — exact table lookups on the device.
//
// Replaces lookup()/TableRow.match (src/zkevm_specs/evm_circuit/table.py:864-884, 389-401):
// the reference scans a Python set linearly and counts rows whose queried (non-None)
// columns equal the query; 0 matches => LookupUnsatFailure, >1 => LookupAmbiguousFailure.
// That scan is >99 % of the reference's EVM/copy time (SURVEY.md §3.1).
//
// Here every (table, queried-column set) gets an open-addressing hash index built on the
// device.  The hash of a row is a keyed combination of its queried cells (rlc_term below; the keys
// come from ZK_CHALLENGE_LOOKUP); its low bits pick the bucket.  A probe recomputes h for the query,
// walks the bucket run, and CONFIRMS each candidate by comparing the queried cells exactly,
// so pass/fail never depends on r; it also counts distinct matching rows so ambiguity is
// reported exactly like the reference (rows identical in every column count once, the
// table being a set).
#pragma once
#include "fr.cuh"

namespace zk {

#define ZK_MAX_KEY 12
#define ZK_EMPTY_SLOT 0xFFFFFFFFFFFFFFFFull  // a slot is (fingerprint32 << 32) | row32

#define ZK_MAX_TABLE_COLS 16
struct TableDev {
  const unsigned char* base;  // column c: n_rows integers of width[c] bytes at base + off[c]
  u64 n_rows;
  u32 n_cols;
  const unsigned char* flags;  // optional per-row type flags (may be null)
  u64 off[ZK_MAX_TABLE_COLS];
  unsigned char width[ZK_MAX_TABLE_COLS];  // 0 (constant column), 1, 2, 4, 8, 16 or 32 (fr.cuh:ld_col)
};
// canonical layout: uint64[n_cols][n_rows][4]
ZK_HD void layout_canonical(u64* off, unsigned char* width, u32 n_cols, u64 n_rows) {
  for (u32 c = 0; c < n_cols; c++) {
    off[c] = (u64)c * n_rows * 32;
    width[c] = 32;
  }
}

// One entry of the heads index of a ZK_POS_RUNS table: the code hash of the run is stored INLINE, so a
// probe is one memory round trip (claim word + hash, two loads of the same 64-byte line) instead of
// "slot, then the table's hash cells".  Only runs whose hash cells fit 128 bits are indexed (others
// clear the positional flag), so the two low limbs of each half identify the hash exactly.
struct alignas(64) HeadEnt {
  u64 claim;  // (fingerprint32 << 32) | head row; ZK_EMPTY_SLOT = free
  u32 head;   // first row of the run (the Header row)
  u32 len;    // number of Byte rows of the run
  u64 pad[2];
  u64 h[4];   // hash_lo limbs 0,1; hash_hi limbs 0,1
};
struct IndexDev {
  TableDev tab;
  u64* slots;  // capacity = mask+1 slots, ZK_EMPTY_SLOT = free
  u32 mask;
  u32 n_key;
  u32 key_cols[ZK_MAX_KEY];
  u64 hm[ZK_MAX_KEY];  // odd per-position multipliers of the key hash (drawn from the lookup challenge)
  // Positional fast path (see "positional indexes" below).  pos_ok points at a device flag that the
  // verify kernel leaves at 1 iff the table has the regular structure `pos_kind` promises; the
  // hash index above is then not built and lookups go straight to the row.
  const u32* pos_ok;   // [0] the flag; [1] (ZK_POS_DENSE) the split row D between the dense head and the tail, see below
  u32 pos_kind;
  // ZK_POS_DENSE with a tail: rows [0, D) are one dense counter run; rows [D, n) are a second dense run whose
  // cell `tail_col` equals `tail_val` (and no head row's does) — the rw table's `Start` padding rows, whose
  // rw_counters restart at 1 (end_block.py:30-38).  `tail_key` = index of tail_col in the lookup key, or -1.
  u32 tail_col, tail_val;
  int tail_key;
  HeadEnt* heads;    // ZK_POS_RUNS: hash index over the first row of every run (one 64-byte entry each)
  u32 heads_mask;
  u64 hk[4];         // keyed multipliers of the heads hash (odd, derived from the lookup challenge)
  u32* heads_list;   // [heads_mask + 1] head rows in insertion order, heads_count[0] of them
  u32* heads_count;
  // [0] = number of heads entries claimed since the index was last cleared, [1..] their buckets: the next build
  // resets just those entries (k_pos_prep) instead of the whole heads array.  nullptr: not recorded.
  u32* heads_used = nullptr;
};
#define ZK_POS_NONE 0
#define ZK_POS_DENSE 1  // key column 0 is a counter: cell(row) == cell(0) + row   (rw table by rw_counter)
#define ZK_POS_RUNS 2   // bytecode table: runs [Header, Byte 0, Byte 1, ...] of one code hash each

ZK_HD Fr table_cell(const TableDev& t, u32 col, u64 row) {
  return ld_col(t.base + t.off[col], t.width[col], row);
}
// NARROW: the caller's kernel was launched for tables whose key columns the host found narrow (fr.cuh:ld_col_narrow)
template <bool NARROW>
ZK_HD Fr table_key_cell(const TableDev& t, u32 col, u64 row) {
  if (NARROW) return ld_col_narrow(t.base + t.off[col], t.width[col], row);
  return ld_col(t.base + t.off[col], t.width[col], row);
}

// 64-bit mix of the canonical RLC value: low bits pick the bucket, high 32 bits are the
// fingerprint stored in the slot (so a probe only touches table rows whose fingerprint matches)
ZK_HD u64 rlc_mix(const Fr& h) {
  u64 x = h.l[0] ^ (h.l[1] * 0x9E3779B97F4A7C15ull) ^ (h.l[2] * 0xC2B2AE3D27D4EB4Full) ^
          (h.l[3] * 0x165667B19E3779F9ull);
  x ^= x >> 32;
  x *= 0xD6E8FEB86659FD93ull;
  x ^= x >> 32;
  x *= 0xD6E8FEB86659FD93ull;
  x ^= x >> 32;
  return x;
}

// One term of the key hash.  Round 1 compressed a row into its random linear combination over Fr
// (one 254-bit Montgomery product per wide cell, ~100-400 instructions); matches are confirmed cell by
// cell anyway, so the hash only has to spread keys: a keyed multiply-add of the four limbs, times an odd
// per-position constant (keys drawn from ZK_CHALLENGE_LOOKUP after the witness is fixed), ~30 instructions.
ZK_HD Fr rlc_term(const IndexDev& ix, const Fr& cell, int j) {
  const u64 f = cell.l[0] * ix.hk[0] + cell.l[1] * ix.hk[1] + cell.l[2] * ix.hk[2] + cell.l[3] * ix.hk[3];
  return fr_u64(f * ix.hm[j]);
}
// h = key[0] + sum_{j>=1} term(key[j], j)
template <int NK>
ZK_HD Fr rlc_key(const IndexDev& ix, const Fr (&key)[NK]) {
  Fr h = key[0];
#pragma unroll
  for (int j = 1; j < NK; j++) h = fr_add(h, rlc_term(ix, key[j], j));
  return h;
}

// One thread per table row: compress the queried columns and claim a slot.
ZK_HD void index_insert_row(const IndexDev& ix, u64 row) {
  Fr h = table_cell(ix.tab, ix.key_cols[0], row);
  for (u32 j = 1; j < ix.n_key; j++) h = fr_add(h, rlc_term(ix, table_cell(ix.tab, ix.key_cols[j], row), (int)j));
  const u64 mix = rlc_mix(h);
  const u64 entry = (mix & 0xFFFFFFFF00000000ull) | (u64)(u32)row;
  u32 b = (u32)mix & ix.mask;
  for (;;) {
    const u64 old = atomic_cas_u64(&ix.slots[b], ZK_EMPTY_SLOT, entry);
    if (old == ZK_EMPTY_SLOT) break;
    b = (b + 1) & ix.mask;
  }
}


ZK_HD bool rows_identical(const TableDev& t, u32 a, u32 b) {
  for (u32 c = 0; c < t.n_cols; c++)
    if (!fr_eq(table_cell(t, c, a), table_cell(t, c, b))) return false;
  return true;
}

// Walk the bucket run starting at the bucket of h.  Returns the number of distinct matching
// rows, capped at 2; *row = the first match.
//
// WARP-SYNCHRONOUS form: every lane named in `mask` must call it together (lanes with nothing
// to look up pass active = false).  Lanes finish their bucket runs after different numbers of
// slots; the loop runs until every lane of the mask is done (warp-uniform trip count), so the
// warp leaves the loop CONVERGED.  With a plain data-dependent `break` each lane ran the rest
// of its gate program alone (measured: 1-2 active threads per instruction, profiles/r01_v4).
template <int NK>
ZK_HD int probe_slots(const IndexDev& ix, const u64* slots, u32 slot_mask, const Fr& h, const Fr (&key)[NK],
                      u32* row, unsigned mask, bool active, u32* slot_out = nullptr) {
  int found = 0;
  u32 first = 0, first_slot = 0;
  const u64 mix = rlc_mix(h);
  const u32 fp = (u32)(mix >> 32);
  u32 b = (u32)mix & slot_mask;
#ifdef __CUDA_ARCH__
#define ZK_GROUP_ANY(p) ((mask & (mask - 1)) ? __any_sync(mask, (p)) : (p))  /* a single-lane mask (lane-private lookups of the group kernels) needs no vote */
#else
#define ZK_GROUP_ANY(p) (p)
  (void)mask;
#endif
  bool done = !active;
  while (ZK_GROUP_ANY(!done)) {
    if (!done) {
      const u64 slot = ld_u64(&slots[b]);
      if (slot == ZK_EMPTY_SLOT) {
        done = true;
      } else {
        if ((u32)(slot >> 32) == fp) {
          const u32 cand = (u32)slot;
          // all key cells are loaded before any compare: NK independent loads in flight instead of
          // a chain of NK dependent round trips
          Fr cells[NK];
#pragma unroll
          for (int j = 0; j < NK; j++) cells[j] = table_cell(ix.tab, ix.key_cols[j], cand);
          bool eq = true;
#pragma unroll
          for (int j = 0; j < NK; j++) eq = eq && fr_eq(cells[j], key[j]);
          if (eq) {
            if (found == 0) {
              first = cand;
              first_slot = b;
              found = 1;
            } else if (!rows_identical(ix.tab, first, cand)) {
              found = 2;
              done = true;
            }
          }
        }
        b = (b + 1) & slot_mask;
      }
    }
  }
#undef ZK_GROUP_ANY
  *row = first;
  if (slot_out) *slot_out = first_slot;
  return found;
}
template <int NK>
ZK_HD int probe_hashed(const IndexDev& ix, const Fr& h, const Fr (&key)[NK], u32* row, unsigned mask,
                       bool active) {
  return probe_slots<NK>(ix, ix.slots, ix.mask, h, key, row, mask, active);
}

// ---- positional indexes ---------------------------------------------------------------------
// Witness generators emit some tables in a regular order (the rw table by rw_counter, the
// bytecode table as one run per contract).  A streaming verify kernel checks that structure
// exactly; if it holds, a lookup computes the only row that CAN match and confirms it cell by
// cell — same match count as the reference's scan (0 or 1: the structure implies key
// uniqueness) with no hash build, no slot probe and no RLC.  If it does not hold, the flag is 0
// and every lookup takes the generic hash path, so the result never depends on the layout.
ZK_HD bool pos_enabled(const IndexDev& ix) { return ix.pos_ok != nullptr && ld_u32(ix.pos_ok) != 0; }

// ZK_POS_DENSE: candidate = key[0] - cell(0).  Branch-free (candidate clamped, cells always
// loaded) so that it overlaps with neighbouring lookups; `base0` = limb 0 of cell(0) of the
// counter column, hoisted by callers that do many lookups (pass nullptr to read it here).
// The tail run (keys whose tail column holds tail_val: the rw table's Start padding rows, stored after the dense head)
// is the same computation on another window of rows — base, limit and row offset switch, the loads and compares are
// shared.  (Round 1 had the tail as an out-of-line function taking the key array by reference: that single call pinned
// every caller's key array in local memory — 160-750 B of stack traffic per row in every kernel with a positional
// lookup; profiles/README.md r02.)
template <int NK, bool NARROW = false>
ZK_HD int pos_lookup_dense(const IndexDev& ix, const Fr (&key)[NK], u32* row, bool active, const u64* base0 = nullptr,
                           int extra_col = -1, Fr* extra = nullptr, int extra_col2 = -1, Fr* extra2 = nullptr) {
  bool tail = false;  // key[ix.tail_key] == ix.tail_val, without indexing `key` by a run-time value
#pragma unroll
  for (int j = 0; j < NK; j++) {  // every cell compared unconditionally, combined without short-circuit: a conditional read
    const bool e = fr_eq_u64(key[j], ix.tail_val);  // of key[j] is turned back into key[tail_key] by the compiler, which
    tail |= (j == ix.tail_key) & e;                 // puts the caller's key array in local memory
  }
  const u64 split = ix.tail_key >= 0 ? (u64)ld_u32(ix.pos_ok + 1) : ix.tab.n_rows;  // dense head = rows [0, split)
  const u64 offset = tail ? split : 0;
  const u64 limit = tail ? ix.tab.n_rows - split : split;
  u64 base;
  if (tail) base = limit ? table_cell(ix.tab, ix.key_cols[0], split).l[0] : 0;
  else base = base0 ? *base0 : table_cell(ix.tab, ix.key_cols[0], 0).l[0];
  const bool in_range = fr_fits64(key[0]) && key[0].l[0] >= base && key[0].l[0] - base < limit;
  const bool valid = active && in_range;
  const u64 cand = valid ? offset + (key[0].l[0] - base) : 0;
  Fr cells[NK];  // independent loads first, compares after
#pragma unroll
  for (int j = 1; j < NK; j++) cells[j] = table_key_cell<NARROW>(ix.tab, ix.key_cols[j], cand);
  if (extra_col >= 0) *extra = table_cell(ix.tab, (u32)extra_col, cand);
  if (extra_col2 >= 0) *extra2 = table_cell(ix.tab, (u32)extra_col2, cand);
  bool eq = valid;
#pragma unroll
  for (int j = 1; j < NK; j++) eq = eq && fr_eq(cells[j], key[j]);
  *row = (u32)cand;
  return eq ? 1 : 0;
}
// ZK_POS_RUNS (bytecode table, key = hash_lo, hash_hi, tag, index, is_code): `head` is the first
// row of the run with this code hash and `len` its number of Byte rows (both from the heads index,
// whose probe CONFIRMS the two hash cells); Header row = head, Byte row k = head + 1 + k, k < len.
// The verify pass has pinned, for every row of a run, hash == the head's hash, tag (Header at the
// head, Byte after it) and index == position in the run, so the only row that can match the key
// is known and just ONE of its cells is still open: is_code.  A lookup therefore reads is_code
// (+ the looked-up value) — 2 narrow cells instead of 6 — and its verdict equals the reference's
// scan: 0 or 1 match, never 2 (distinct runs have distinct hashes, rows of a run distinct indices).
// Branch-free: the candidate row is clamped to a valid row and its cells are always loaded, so
// several lookups of one thread have all their loads in flight together; `extra_col` (or -1)
// names one more cell of the candidate row to fetch in the same batch (the looked-up value).
// TYPED: the table has the layout k_bytecode_table_expand writes (is_code 1 byte, value 4 bytes): plain typed loads
template <bool TYPED = false>
ZK_HD int pos_lookup_run(const IndexDev& ix, const Fr (&key)[5], int n_head, u32 head, u32 len, u32* row, bool active,
                         int extra_col = -1, Fr* extra = nullptr) {
  const bool is_hdr = fr_eq_u64(key[2], 1) && fr_is_zero(key[3]);
  const bool is_byte = fr_eq_u64(key[2], 2) && fr_fits64(key[3]) && key[3].l[0] < (u64)len;
  u64 cand = is_hdr ? (u64)head : (u64)head + 1 + (is_byte ? key[3].l[0] : 0);
  const bool valid = active && n_head == 1 && (is_hdr || is_byte) && cand < ix.tab.n_rows;
  if (!valid) cand = 0;
  Fr is_code;
  if (TYPED) {
    is_code = ld_col_c<1>(ix.tab.base + ix.tab.off[4], cand);
    if (extra_col >= 0) *extra = ld_col_c<4>(ix.tab.base + ix.tab.off[5], cand);  // the looked-up cell is `value`
  } else {
    is_code = table_cell(ix.tab, ix.key_cols[4], cand);
    if (extra_col >= 0) *extra = table_cell(ix.tab, (u32)extra_col, cand);
  }
  *row = (u32)cand;
  return valid && fr_eq(is_code, key[4]) ? 1 : 0;
}
// keyed 64-bit hash of a code hash held as two 128-bit halves: four multiplies by odd constants drawn
// from the lookup challenge + a finaliser (the RLC of the generic index would cost a 254-bit Montgomery
// product per probe; this hash only picks a bucket, matches are confirmed on all 256 bits)
ZK_HD u64 heads_mix(const IndexDev& ix, const Fr& hlo, const Fr& hhi) {
  u64 x = hlo.l[0] * ix.hk[0] + hlo.l[1] * ix.hk[1] + hhi.l[0] * ix.hk[2] + hhi.l[1] * ix.hk[3];
  x ^= x >> 32;
  x *= 0xD6E8FEB86659FD93ull;
  x ^= x >> 29;
  return x;
}
// 16-byte / 32-byte halves of a heads entry (written by an earlier kernel: read-only here)
ZK_HD void ld_head_ent(const HeadEnt* e, u64* claim, u32* head, u32* len, u64 h[4]) {
#ifdef __CUDA_ARCH__
  u64 hl;
  asm volatile("ld.global.nc.v2.u64 {%0,%1}, [%2];" : "=l"(*claim), "=l"(hl) : "l"(e));
  asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(h[0]), "=l"(h[1]), "=l"(h[2]), "=l"(h[3]) : "l"(e->h));
  *head = (u32)hl;
  *len = (u32)(hl >> 32);
#else
  *claim = e->claim;
  *head = e->head;
  *len = e->len;
  for (int k = 0; k < 4; k++) h[k] = e->h[k];
#endif
}
// heads index probe (warp-synchronous like probe_slots: lanes of `mask` call it together and leave
// converged).  Run heads are unique by construction (a duplicate code hash clears the positional
// flag), so the first confirmed entry is the only one: returns 0 or 1.
ZK_HD int heads_probe(const IndexDev& ix, const Fr& hlo, const Fr& hhi, u32* head, u32* len, unsigned mask, bool active) {
  const bool key_ok = fr_fits128(hlo) && fr_fits128(hhi);  // indexed hashes all fit 128-bit halves
  const u64 mix = heads_mix(ix, hlo, hhi);
  const u32 fp = (u32)(mix >> 32);
  u32 b = (u32)mix & ix.heads_mask;
  int found = 0;
  *head = 0;
  *len = 0;
#ifdef __CUDA_ARCH__
#define ZK_GROUP_ANY(p) ((mask & (mask - 1)) ? __any_sync(mask, (p)) : (p))  /* a single-lane mask (lane-private lookups of the group kernels) needs no vote */
#else
#define ZK_GROUP_ANY(p) (p)
  (void)mask;
#endif
  bool done = !(active && key_ok);
  while (ZK_GROUP_ANY(!done)) {
    if (!done) {
      u64 claim, h[4];
      u32 e_head, e_len;
      ld_head_ent(&ix.heads[b], &claim, &e_head, &e_len, h);
      if (claim == ZK_EMPTY_SLOT) {
        done = true;
      } else if ((u32)(claim >> 32) == fp && h[0] == hlo.l[0] && h[1] == hlo.l[1] && h[2] == hhi.l[0] && h[3] == hhi.l[1]) {
        *head = e_head;
        *len = e_len;
        found = 1;
        done = true;
      } else {
        b = (b + 1) & ix.heads_mask;
      }
    }
  }
#undef ZK_GROUP_ANY
  return found;
}

// verify kernels' row functions
ZK_HD void pos_fail(u32* ok) {
#ifdef __CUDA_ARCH__
  atomicExch(ok, 0u);
#else
  *ok = 0;
#endif
}
// ok[0] = flag, ok[1] = split row (initialised to n_rows).  Every row is checked against its predecessor:
// inside a run the counter grows by one; the one allowed change of run is head -> tail.
ZK_HD void pos_verify_dense_row(const IndexDev& ix, u32* ok, u64 row) {
  const TableDev& t = ix.tab;
  const Fr c = table_cell(t, ix.key_cols[0], row);
  const bool tail = ix.tail_key >= 0 && fr_eq_u64(table_cell(t, ix.tail_col, row), ix.tail_val);
  bool good = fr_fits64(c);
  if (row == 0) {
    if (tail) atomic_min_u32(ok + 1, 0u);
  } else {
    const Fr p = table_cell(t, ix.key_cols[0], row - 1);
    const bool ptail = ix.tail_key >= 0 && fr_eq_u64(table_cell(t, ix.tail_col, row - 1), ix.tail_val);
    if (tail == ptail) good = good && fr_fits64(p) && p.l[0] != ~0ull && c.l[0] == p.l[0] + 1;
    else if (tail) atomic_min_u32(ok + 1, (u32)row);
    else good = false;  // a head row after the tail
  }
  if (!good) pos_fail(ok);
}
// pos_verify_dense_row over a STRIP of ZK_DENSE_STRIP consecutive rows [row0, row0 + strip) ∩ [0, n), for the layout every
// packer gives the rw table: the counter (key column 0) stored in WC = 4 or 8 bytes, the tail column narrow in WT = 1
// byte or a constant cell (WT = 0; Matrix::narrow_mask: its value fits limb 0).  The strip's cells are loaded at once
// (on the device as 16-byte vectors: the host picks this form only for 16-byte aligned columns), each row is compared
// with its predecessor held in registers, and the strip's verdict goes out in at most two atomics.  Same flag and split
// row as pos_verify_dense_row on every row.
#define ZK_DENSE_STRIP 8
template <int WC, int WT>
ZK_HD void pos_verify_dense_strip(const IndexDev& ix, u32* ok, u64 row0) {
  static_assert((WC == 4 || WC == 8) && (WT == 0 || WT == 1), "typed dense verify: counter 4 / 8 bytes, tail 0 / 1 byte");
  const TableDev& t = ix.tab;
  const unsigned char* pc = t.base + t.off[ix.key_cols[0]];
  const unsigned char* pt = t.base + t.off[ix.tail_col];
  const bool has_tail = ix.tail_key >= 0;
  const u64 n = t.n_rows;
  u64 c[ZK_DENSE_STRIP];
  u32 tag[ZK_DENSE_STRIP];
  const u32 tag0 = has_tail && WT == 0 ? (u32)(ld_col_c<0>(pt, 0).l[0] == ix.tail_val) : 0u;  // constant column
#ifdef __CUDA_ARCH__
  if (row0 + ZK_DENSE_STRIP <= n) {
    const uint4* vc = (const uint4*)(pc + row0 * WC);
#pragma unroll
    for (int q = 0; q < ZK_DENSE_STRIP * WC / 16; q++) {
      const uint4 v = __ldg(vc + q);
      const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4 * 4 / WC; k++)
        c[q * (16 / WC) + k] = WC == 8 ? ((u64)w[2 * k + 1] << 32 | w[2 * k]) : (u64)w[k];
    }
    const u64 tb = (WT == 1 && has_tail) ? __ldg((const unsigned long long*)(pt + row0)) : 0ull;
#pragma unroll
    for (int j = 0; j < ZK_DENSE_STRIP; j++) tag[j] = WT == 1 ? (u32)((tb >> (8 * j)) & 0xFF) : 0u;
  } else
#endif
  {
#pragma unroll
    for (int j = 0; j < ZK_DENSE_STRIP; j++) {
      const u64 r = row0 + j < n ? row0 + j : row0;
      c[j] = ld_col_c<WC>(pc, r).l[0];
      tag[j] = (WT == 1 && has_tail) ? (u32)ld_col_c<1>(pt, r).l[0] : 0u;
    }
  }
  u64 p = 0;
  bool ptail = false;
  if (row0 > 0) {
    p = ld_col_c<WC>(pc, row0 - 1).l[0];
    ptail = has_tail && (WT == 0 ? tag0 != 0 : ld_col_c<1>(pt, row0 - 1).l[0] == ix.tail_val);
  }
  bool good = true;
  u32 split = ~0u;
#pragma unroll
  for (int j = 0; j < ZK_DENSE_STRIP; j++) {
    const u64 row = row0 + j;
    if (row < n) {
      const bool tail = has_tail && (WT == 0 ? tag0 != 0 : tag[j] == ix.tail_val);
      if (row == 0) {
        if (tail) split = 0;
      } else if (tail == ptail) {
        good = good && p != ~0ull && c[j] == p + 1;
      } else if (tail) {
        split = (u32)row < split ? (u32)row : split;
      } else {
        good = false;  // a head row after the tail
      }
      p = c[j];
      ptail = tail;
    }
  }
  if (split != ~0u) atomic_min_u32(ok + 1, split);
  if (!good) pos_fail(ok);
}
// Claim an entry of the heads index for the run that starts at `row` with code hash (hlo, hhi).
// `len` != nullptr: the run length is known (table unrolled by the library) and is stored at once;
// otherwise the head is listed for k_pos_runlen.  A duplicate hash, a hash cell beyond 128 bits or a
// full index clears the flag.
ZK_HD void heads_insert(const IndexDev& ix, u32* ok, u64 row, const Fr& hlo, const Fr& hhi, const u32* len) {
  const TableDev& t = ix.tab;
  if (!(fr_fits128(hlo) && fr_fits128(hhi))) {
    pos_fail(ok);
    return;
  }
  const u64 mix = heads_mix(ix, hlo, hhi);
  const u64 entry = (mix & 0xFFFFFFFF00000000ull) | (u64)(u32)row;
  u32 b = (u32)mix & ix.heads_mask;
  for (u32 tries = 0; tries <= ix.heads_mask; tries++) {
    HeadEnt* e = &ix.heads[b];
    const u64 old = atomic_cas_u64(&e->claim, ZK_EMPTY_SLOT, entry);
    if (old == ZK_EMPTY_SLOT) {  // payload: read only by later kernels
      if (ix.heads_used) ix.heads_used[1 + atomic_add_u32(ix.heads_used, 1u)] = b;  // one record per claimed bucket
      e->head = (u32)row;
      e->len = len ? *len : 0u;
      e->h[0] = hlo.l[0];
      e->h[1] = hlo.l[1];
      e->h[2] = hhi.l[0];
      e->h[3] = hhi.l[1];
      if (!len) {
        const u32 k = atomic_add_u32(ix.heads_count, 1u);  // k <= heads_mask: one entry per listed head
        ix.heads_list[k & ix.heads_mask] = (u32)row;
      }
      return;
    }
    if ((old >> 32) == (mix >> 32)) {  // the other claimant's payload may not be written yet: compare table cells
      const u32 other = (u32)old;
      if (fr_eq(table_cell(t, 0, other), hlo) && fr_eq(table_cell(t, 1, other), hhi)) break;  // duplicate hash
    }
    b = (b + 1) & ix.heads_mask;
  }
  pos_fail(ok);  // duplicate code hash, or more runs than the heads index holds
}
struct RunCells {
  Fr hlo, hhi, tag, index;
};
ZK_HD RunCells run_cells(const TableDev& t, u64 row) {
  return RunCells{table_cell(t, 0, row), table_cell(t, 1, row), table_cell(t, 2, row), table_cell(t, 3, row)};
}
// same cells when the four columns' widths are compile-time constants (hash lo / hi, tag, index)
template <int WH, int WT, int WI>
ZK_HD RunCells run_cells_c(const TableDev& t, u64 row) {
  return RunCells{ld_col_c<WH>(t.base + t.off[0], row), ld_col_c<WH>(t.base + t.off[1], row),
                  ld_col_c<WT>(t.base + t.off[2], row), ld_col_c<WI>(t.base + t.off[3], row)};
}
ZK_HD void pos_verify_run_cells(const IndexDev& ix, u32* ok, u64 row, const RunCells& cur, const RunCells& prev);
ZK_HD void pos_verify_run_row(const IndexDev& ix, u32* ok, u64 row) {
  const RunCells cur = run_cells(ix.tab, row);
  pos_verify_run_cells(ix, ok, row, cur, row > 0 ? run_cells(ix.tab, row - 1) : cur);
}
// `prev` = the cells of row - 1 (ignored for row 0)
ZK_HD void pos_verify_run_cells(const IndexDev& ix, u32* ok, u64 row, const RunCells& cur, const RunCells& prev) {
  const TableDev& t = ix.tab;
  const Fr hlo = cur.hlo, hhi = cur.hhi, tag = cur.tag, index = cur.index;
  bool head = row == 0;
  Fr ptag = fr_u64(0), pindex = fr_u64(0);
  if (row > 0) {
    head = !(fr_eq(hlo, prev.hlo) && fr_eq(hhi, prev.hhi));
    ptag = prev.tag;
    pindex = prev.index;
  }
  if (head) {
    if (!(fr_eq_u64(tag, 1) && fr_is_zero(index))) {
      pos_fail(ok);
      return;
    }
    // register the run head; a second run with the same code hash makes keys ambiguous -> irregular
    heads_insert(ix, ok, row, hlo, hhi, nullptr);
  } else {
    const bool byte_row = fr_eq_u64(tag, 2);
    const bool idx_ok = fr_eq_u64(ptag, 1) ? fr_is_zero(index)
                                           : (fr_eq_u64(ptag, 2) && fr_fits64(pindex) && fr_fits64(index) &&
                                              pindex.l[0] != ~0ull && index.l[0] == pindex.l[0] + 1);
    if (!(byte_row && idx_ok)) pos_fail(ok);
  }
}

// Second (tiny) pass over the listed heads: entry k < count closes the run that ends just before
// head k, entry k == count the run that ends at the last row.  The last row of a run gives its
// length directly (a Byte row's index is its position in the run, a Header-only run has none), and
// the run's head is that many rows back; its slot in the heads index receives the length.
// Only meaningful when the verify pass leaves the flag at 1 (otherwise nothing reads it).
ZK_HD void pos_runlen_entry(const IndexDev& ix, u32 k, u32 count) {
  const TableDev& t = ix.tab;
  u64 end;
  if (k < count) {
    const u32 h = ix.heads_list[k];
    if (h == 0) return;
    end = (u64)h - 1;
  } else {
    end = t.n_rows - 1;
  }
  const Fr tag = table_cell(t, 2, end), index = table_cell(t, 3, end);
  u64 len = 0;
  if (!fr_eq_u64(tag, 1)) {
    if (!fr_fits64(index) || index.l[0] >= end) return;  // irregular table: the flag is already 0
    len = index.l[0] + 1;
  }
  const u64 head = end - len;
  const Fr hlo = table_cell(t, 0, end), hhi = table_cell(t, 1, end);
  const u64 mix = heads_mix(ix, hlo, hhi);
  u32 b = (u32)mix & ix.heads_mask;
  for (u32 tries = 0; tries <= ix.heads_mask; tries++) {
    const u64 claim = ld_volatile_u64(&ix.heads[b].claim);
    if (claim == ZK_EMPTY_SLOT) return;
    if ((u32)claim == (u32)head) {
      ix.heads[b].len = (u32)len;
      return;
    }
    b = (b + 1) & ix.heads_mask;
  }
}

// warp-synchronous lookup (see probe_hashed)
template <int NK>
ZK_HD int lookup_sync(const IndexDev& ix, const Fr (&key)[NK], u32* row, unsigned mask, bool active) {
  if (ix.tab.n_rows == 0) return 0;  // uniform: the table is the same for every lane
  if (pos_enabled(ix)) {             // uniform: one flag per table
    if (ix.pos_kind == ZK_POS_DENSE) return pos_lookup_dense<NK>(ix, key, row, active);
    if constexpr (NK == 5) {
      if (ix.pos_kind == ZK_POS_RUNS) {
        u32 head = 0, len = 0;
        const int n_head = heads_probe(ix, key[0], key[1], &head, &len, mask, active);
        return pos_lookup_run(ix, key, n_head, head, len, row, active);
      }
    }
  }
  return probe_hashed<NK>(ix, rlc_key<NK>(ix, key), key, row, mask, active);
}
// single-thread lookup: the calling thread is its own group
template <int NK>
ZK_HD int lookup(const IndexDev& ix, const Fr (&key)[NK], u32* row) {
#ifdef __CUDA_ARCH__
  const unsigned self = 1u << (threadIdx.x & 31);
#else
  const unsigned self = 1u;
#endif
  return lookup_sync<NK>(ix, key, row, self, true);
}

#ifdef __CUDACC__
// the generic hash index is only needed when the table is NOT positional
__global__ void __launch_bounds__(256) k_index_build(IndexDev ix) {
  if (pos_enabled(ix)) return;
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 row = (u64)blockIdx.x * blockDim.x + threadIdx.x; row < ix.tab.n_rows; row += stride) index_insert_row(ix, row);
}
__global__ void __launch_bounds__(256) k_slots_clear(u64* slots, u64 n, const u32* skip_if_set) {
  if (skip_if_set && *skip_if_set) return;
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) slots[i] = ZK_EMPTY_SLOT;
}
// Everything a positional index needs before its verify pass, for every index a check is about to verify, in ONE
// launch (one block): flag = 1, split = n_rows, and the heads entries the previous build claimed back to free (the
// heads index is never cleared whole: a build claims one entry per run, a few hundred of its 65,536).
#define ZK_POS_PREP_MAX 2
struct PosPrep {
  u32 n;
  u32* flag[ZK_POS_PREP_MAX];
  u32 n_rows[ZK_POS_PREP_MAX];
  HeadEnt* heads[ZK_POS_PREP_MAX];   // nullptr: no heads index
  u32* heads_count[ZK_POS_PREP_MAX];
  u32* heads_used[ZK_POS_PREP_MAX];  // IndexDev::heads_used
  u32 heads_cap;
};
__global__ void __launch_bounds__(1024) k_pos_prep(PosPrep p) {
  for (u32 e = 0; e < p.n; e++) {
    if (threadIdx.x == 0) {
      p.flag[e][0] = 1u;
      p.flag[e][1] = p.n_rows[e];
    }
    if (p.heads[e]) {
      const u32 used = min(p.heads_used[e][0], p.heads_cap);
      for (u32 k = threadIdx.x; k < used; k += blockDim.x) p.heads[e][p.heads_used[e][1 + k]].claim = ZK_EMPTY_SLOT;
    }
  }
  __syncthreads();  // every thread has read the counts
  if (threadIdx.x == 0)
    for (u32 e = 0; e < p.n; e++)
      if (p.heads[e]) p.heads_used[e][0] = p.heads_count[e][0] = 0u;
}
// ZK_POS_DENSE verify in the typed strip form (pos_verify_dense_strip): one thread per ZK_DENSE_STRIP rows
template <int WC, int WT>
__global__ void __launch_bounds__(256) k_pos_verify_dense_typed(IndexDev ix, u32* ok) {
  const u64 strips = (ix.tab.n_rows + ZK_DENSE_STRIP - 1) / ZK_DENSE_STRIP, stride = (u64)gridDim.x * blockDim.x;
  for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < strips; s += stride)
    pos_verify_dense_strip<WC, WT>(ix, ok, s * ZK_DENSE_STRIP);
}
__global__ void __launch_bounds__(256) k_pos_runlen(IndexDev ix) {
  if (ix.tab.n_rows == 0) return;
  const u32 count = min(*ix.heads_count, ix.heads_mask + 1);
  for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k <= count; k += gridDim.x * blockDim.x) pos_runlen_entry(ix, k, count);
}
// A bytecode table unrolled by the library itself (zk_upload_bytecode_table_from_code) is regular
// by construction: its heads index is filled straight from the contract offsets — one thread per
// CONTRACT instead of a pass over every table row — and only duplicate code hashes (or more
// contracts than the heads index holds) still clear the flag.
__global__ void __launch_bounds__(256) k_heads_from_offsets(IndexDev ix, u32* ok, const u64* offsets, u64 n_contracts) {
  if (n_contracts > (u64)ix.heads_mask + 1) {
    if (blockIdx.x == 0 && threadIdx.x == 0) pos_fail(ok);
    return;
  }
  for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n_contracts; k += (u64)gridDim.x * blockDim.x) {
    const u64 start = offsets[k], row = start + k;
    const u32 len = (u32)(offsets[k + 1] - start);
    heads_insert(ix, ok, row, table_cell(ix.tab, 0, row), table_cell(ix.tab, 1, row), &len);
  }
}
__global__ void __launch_bounds__(256) k_pos_verify(IndexDev ix, u32* ok) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  if (ix.pos_kind == ZK_POS_DENSE) {
    for (u64 row = (u64)blockIdx.x * blockDim.x + threadIdx.x; row < ix.tab.n_rows; row += stride) pos_verify_dense_row(ix, ok, row);
    return;
  }
  // the two layouts a bytecode table normally arrives in get plain typed loads; anything else goes
  // through the generic per-column-width loader
  const unsigned char* wd = ix.tab.width;
  const u64 row0 = (u64)blockIdx.x * blockDim.x + threadIdx.x, n = ix.tab.n_rows;
  if (wd[0] == 16 && wd[1] == 16 && wd[2] == 1 && wd[3] == 4) {  // packing.TYPE_WIDTHS["bytecode_table"]
    for (u64 row = row0; row < n; row += stride)
      pos_verify_run_cells(ix, ok, row, run_cells_c<16, 1, 4>(ix.tab, row), run_cells_c<16, 1, 4>(ix.tab, row ? row - 1 : 0));
  } else if (wd[0] == 32 && wd[1] == 32 && wd[2] == 32 && wd[3] == 32) {  // canonical
    for (u64 row = row0; row < n; row += stride)
      pos_verify_run_cells(ix, ok, row, run_cells_c<32, 32, 32>(ix.tab, row), run_cells_c<32, 32, 32>(ix.tab, row ? row - 1 : 0));
  } else {
    for (u64 row = row0; row < n; row += stride) pos_verify_run_row(ix, ok, row);
  }
}
#endif

// ---- result recording -------------------------------------------------------------------
struct ResultDev {
  u32* first_fail;  // [n_constraints]
  u64* fail_count;  // [n_constraints]
};
ZK_HD void fail(const ResultDev& r, int id, u64 row) {
  atomic_min_u32(&r.first_fail[id], (u32)row);
  atomic_add_u64(&r.fail_count[id], 1ull);
}
#define ZK_REQUIRE(res, id, row, cond) \
  do {                                 \
    if (!(cond)) fail((res), (id), (row)); \
  } while (0)

}  // namespace zk
