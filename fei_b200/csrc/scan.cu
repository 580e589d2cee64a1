// K1/K2: the Memdir scan kernels (sm_100a).
//
// Replaces the per-record loops of the reference:
//   search_memories -> _memory_matches_query -> _get_field_value / _compare_values
//       (memdir_tools/search.py:361-367, :244-335, :97-139, :141-242)
//   FilterManager.process_memories -> MemoryFilter.matches      (memdir_tools/filter.py:229-233, :67-109)
//   parse_memory_content header parsing                          (memdir_tools/utils.py:113-118)
//
// k_head_meta / k_head_parse : meta predicates (flags / date / folder / status) over the 20-byte meta columns, four
//          records per thread; records that still need a header or name field go to a work list and get one thread
//          each in k_head_parse, which reads the record's header directory (hdir.cu: interned key + stripped value
//          span per header line; k_key_lut maps the corpus' distinct keys to the program's fields once per scan)
//          and applies the reference's dict semantics (a repeated key keeps its last value, a case-insensitive
//          field lookup takes the first matching spelling).  Headers the directory cannot address are split / stripped
//          here exactly like utils.py:113-118.  Every string condition is an output bit of a byte DFA; the program
//          head (conditions + small automata) is staged into shared memory by a TMA bulk copy per CTA.
//          Writes alive[i] = bitmask of queries whose non-content conditions all hold.
// k_body : one warp per group of 32 records in the warp-transposed body tiles (corpus.h): each
//          row is one contiguous coalesced request (ld.global.nc 16 B per lane); each lane walks
//          its own record through the multi-pattern DFA whose tables were staged into shared
//          memory with 1-D TMA bulk copies (cp.async.bulk + mbarrier).  Groups with no live
//          record are skipped without touching their bytes.  hits[i] = alive[i] & content bits.
// k_count / k_scan_blocks / k_emit : order-preserving compaction of hits[] into per-query lists
//          of global record indices (warp ballots + popc prefix, block offsets from a scan).
#include "corpus.h"
#include "../../include/feiscan_prog.h"
#include "pyws.cuh"
#include <string.h>
#include <stdlib.h>
#include <vector>
#include <algorithm>

namespace fei {

// ---------------------------------------------------------------- DFA view
struct DfaView {
  const uint16_t* trans;
  const uint32_t* out;
  const uint32_t* endout;
  const uint8_t* cls;
  uint32_t n_cols, stride, start, n_acc, empty_acc;
};

__device__ __forceinline__ DfaView dfa_view(const uint8_t* blob, uint32_t off) {
  const fei_prog_dfa* d = reinterpret_cast<const fei_prog_dfa*>(blob + off);
  DfaView v;
  v.trans = reinterpret_cast<const uint16_t*>(blob + d->off_trans);
  v.out = reinterpret_cast<const uint32_t*>(blob + d->off_out);
  v.endout = reinterpret_cast<const uint32_t*>(blob + d->off_endout);
  v.cls = blob + d->off_cls;
  v.n_cols = d->n_cols; v.stride = d->row_stride; v.start = d->start; v.n_acc = d->n_acc; v.empty_acc = d->empty_acc;
  return v;
}

// generic run over a byte span (tables in global memory or, for the head kernels, in the shared-memory copy of the
// program head: plain loads, the address space is resolved at run time); used on short fields
__device__ uint32_t dfa_run(const DfaView& d, const uint8_t* p, uint32_t len) {
  if (len == 0) return d.empty_acc;
  uint32_t s = d.start;
  uint32_t acc = s < d.n_acc ? d.out[s] : 0u;
  const bool direct = d.n_cols == 256;
  for (uint32_t i = 0; i < len; ++i) {
    uint32_t b = p[i];
    uint32_t col = direct ? b : d.cls[b];
    s = d.trans[s * d.stride + col];
    if (s < d.n_acc) acc |= d.out[s];
  }
  return acc | d.endout[s];
}

// The same run with the tables in the shared-memory copy of the program head (stage_prog_head): 32-bit shared
// addresses and ld.shared instead of generic 64-bit pointer arithmetic (the generic loop costs 29 instructions per
// byte in SASS, this one about 8).
struct DfaViewS { uint32_t trans, out, endout, cls, n_cols, stride2, start, n_acc, empty_acc; };
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) { uint32_t r; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(r) : "r"(a)); return r; }
__device__ __forceinline__ uint32_t lds_u16(uint32_t a) { uint32_t r; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r) : "r"(a)); return r; }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t r; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(a)); return r; }
__device__ __forceinline__ DfaViewS dfa_view_s(const uint8_t* sblob, uint32_t off) {
  const fei_prog_dfa* d = reinterpret_cast<const fei_prog_dfa*>(sblob + off);
  const uint32_t base = (uint32_t)__cvta_generic_to_shared(sblob);
  return DfaViewS{base + d->off_trans, base + d->off_out, base + d->off_endout, base + d->off_cls, d->n_cols, d->row_stride * 2u, d->start, d->n_acc, d->empty_acc};
}
// One automaton over a byte span in global memory.  out[] has an entry (0) for non-accepting states too, so there is no
// branch around the lookup and the byte loads of an unrolled group issue ahead of the table walk.  (Fetching the span as
// aligned 4- or 16-byte words was measured slower on the header workloads: per-lane skip / tail predicates diverge.)
struct DfaStepS {
  const DfaViewS& d; uint32_t s, acc; bool direct;
  __device__ __forceinline__ void step(uint32_t b) {
    const uint32_t col = direct ? b : lds_u8(d.cls + b);
    s = lds_u16(d.trans + s * d.stride2 + col * 2u);
    acc |= lds_u32(d.out + 4u * s);
  }
};
__device__ __forceinline__ uint32_t dfa_run_s(const DfaViewS& d, const uint8_t* p, uint32_t len) {
  if (len == 0) return d.empty_acc;
  DfaStepS r{d, d.start, lds_u32(d.out + 4u * d.start), d.n_cols == 256};
  uint32_t i = 0;
  for (; i + 4 <= len; i += 4) {
    const uint32_t b0 = p[i], b1 = p[i + 1], b2 = p[i + 2], b3 = p[i + 3];
    r.step(b0); r.step(b1); r.step(b2); r.step(b3);
  }
  for (; i < len; ++i) r.step(p[i]);
  return r.acc | lds_u32(d.endout + 4u * r.s);
}
// the same over up to 8 bytes held in a register (the flags string of a record: flags8)
__device__ __forceinline__ uint32_t dfa_run_s_u64(const DfaViewS& d, unsigned long long bytes, uint32_t len) {
  if (len == 0) return d.empty_acc;
  DfaStepS r{d, d.start, lds_u32(d.out + 4u * d.start), d.n_cols == 256};
#pragma unroll
  for (uint32_t k = 0; k < 8; ++k) if (k < len) r.step((uint32_t)(bytes >> (8 * k)) & 0xFFu);
  return r.acc | lds_u32(d.endout + 4u * r.s);
}
// the same over a column value: unit k (16 bytes) of the value at base + k * plane_stride (hdir.cu), LDG.128 per unit
__device__ __forceinline__ uint32_t dfa_run_units(const DfaViewS& d, const uint8_t* base, uint64_t plane_stride, uint32_t len) {
  if (len == 0) return d.empty_acc;
  DfaStepS r{d, d.start, lds_u32(d.out + 4u * d.start), d.n_cols == 256};
  for (uint32_t k = 0; k * 16 < len; ++k) {
    const uint4 c = *reinterpret_cast<const uint4*>(base + k * plane_stride);
    const uint32_t w[4] = {c.x, c.y, c.z, c.w};
    const uint32_t nb = len - k * 16;
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j) if (j < nb) r.step((w[j >> 2] >> (8 * (j & 3))) & 0xFFu);
  }
  return r.acc | lds_u32(d.endout + 4u * r.s);
}
__device__ uint32_t dfa_run_units_g(const DfaView& d, const uint8_t* base, uint64_t plane_stride, uint32_t len) {   // tables in global memory
  if (len == 0) return d.empty_acc;
  uint32_t s = d.start, acc = d.out[s];
  const bool direct = d.n_cols == 256;
  for (uint32_t i = 0; i < len; ++i) {
    const uint32_t b = base[(uint64_t)(i >> 4) * plane_stride + (i & 15)];
    s = d.trans[s * d.stride + (direct ? b : d.cls[b])];
    acc |= d.out[s];
  }
  return acc | d.endout[s];
}
// dispatch: `in_smem` is uniform for the grid (stage_prog_head either staged the head for every CTA or for none)
__device__ __forceinline__ uint32_t dfa_run_at(const uint8_t* blob, uint32_t off, bool in_smem, const uint8_t* p, uint32_t len) {
  if (in_smem) return dfa_run_s(dfa_view_s(blob, off), p, len);
  return dfa_run(dfa_view(blob, off), p, len);
}

// ---------------------------------------------------------------- head kernel
struct HeadArgs {
  const uint8_t* prog;         // device copy of the program blob
  const uint8_t* hdr; const uint64_t* hdr_off;
  const uint8_t* name; const uint64_t* name_off; const uint16_t* name_spans;
  const int64_t* wall; const uint64_t* flags8; const uint32_t* fsb;
  uint64_t n;
  uint32_t* alive;
  const uint2* hdir; const uint64_t* hdir_off;     // header directory (hdir.cu)
  const uint32_t* key_lut;                         // dictionary slot of a header key -> mask of the program's slots it names (k_key_lut)
  bool prog_in_smem;                               // set by the kernels after stage_prog_head
  const int8_t* slot_col;                          // per program slot: value column to read (k_slot_cols), -1 walk the directory, -2 no record has the field
  const uint16_t* col_len; const uint8_t* col_planes;   // header value columns (hdir.cu)
  const int64_t* ts;                               // filename timestamps (metadata "timestamp")
  const uint8_t* aux[FEI_MAX_AUX];                 // host-computed per-record verdict bytes (fei_corpus_set_aux)
};

constexpr int kHeadThreads = 256;

__device__ __forceinline__ bool cmp_i64(int64_t v, int64_t o, uint32_t op) {
  switch (op) {
    case FEI_CMP_GT: return v > o; case FEI_CMP_LT: return v < o;
    case FEI_CMP_GE: return v >= o; case FEI_CMP_LE: return v <= o;
    case FEI_CMP_EQ: return v == o; default: return v != o;
  }
}
__device__ __forceinline__ bool eval_meta_cond(const HeadArgs& a, uint64_t rec, const fei_prog_cond& cd, uint32_t flags_acc, int64_t wall, uint32_t fsb) {
  switch (cd.kind) {
    case FEI_C_RECBITS: {
      // selected, not indexed: a dynamic index into the by-value kernel argument makes ptxas copy the whole struct to local memory
      const uint32_t k = cd.ref & (FEI_MAX_AUX - 1);
      static_assert(FEI_MAX_AUX == 4, "aux column select below");
      const uint8_t* col = k == 0 ? a.aux[0] : k == 1 ? a.aux[1] : k == 2 ? a.aux[2] : a.aux[3];
      return (col[rec] != 0) != (cd.negate != 0);
    }
    case FEI_C_TS_CMP: return cmp_i64(a.ts[rec], cd.i64, cd.cmp_op);
    case FEI_C_CONST: return cd.bit != 0;
    case FEI_C_FLAGS: return ((flags_acc >> cd.bit) & 1u) != cd.negate;
    case FEI_C_DATE_CMP: {
      int64_t v = wall * 1000000ll, o = cd.i64;
      switch (cd.cmp_op) {
        case FEI_CMP_GT: return v > o; case FEI_CMP_LT: return v < o;
        case FEI_CMP_GE: return v >= o; case FEI_CMP_LE: return v <= o;
        case FEI_CMP_EQ: return v == o; default: return v != o;
      }
    }
    case FEI_C_FOLDER_SET: return (cd.set64 >> (fsb & 0xFFFFu) & 1ull) != 0;
    case FEI_C_STATUS_SET: return (cd.set64 >> ((fsb >> 16) & 0xFFu) & 1ull) != 0;
    default: return true;                                      // slot / name / body: decided later
  }
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count);
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes);
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar);
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity);

// str(int) of a non-negative integer; returns the length
__device__ __forceinline__ uint32_t format_u64(unsigned long long v, uint8_t* out) {
  uint8_t tmp[20]; int n = 0;
  do { tmp[n++] = (uint8_t)('0' + v % 10); v /= 10; } while (v);
  for (int i = 0; i < n; ++i) out[i] = tmp[n - 1 - i];
  return (uint32_t)n;
}
// str(datetime) of a naive wall-clock second count (no microseconds): "YYYY-MM-DD HH:MM:SS" (civil-from-days, proleptic Gregorian)
__device__ __forceinline__ uint32_t format_datetime(int64_t wall, uint8_t* out) {
  int64_t days = wall / 86400; int64_t rem = wall % 86400;
  if (rem < 0) { rem += 86400; --days; }
  const int64_t z = days + 719468;
  const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  const uint32_t doe = (uint32_t)(z - era * 146097);
  const uint32_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  int64_t y = (int64_t)yoe + era * 400;
  const uint32_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  const uint32_t mp = (5 * doy + 2) / 153;
  const uint32_t d = doy - (153 * mp + 2) / 5 + 1;
  const uint32_t m = mp < 10 ? mp + 3 : mp - 9;
  if (m <= 2) ++y;
  const uint32_t hh = (uint32_t)(rem / 3600), mi = (uint32_t)(rem % 3600 / 60), ss = (uint32_t)(rem % 60);
  uint32_t yy = (uint32_t)(y < 0 ? 0 : y > 9999 ? 9999 : y);
  out[0] = '0' + yy / 1000; out[1] = '0' + yy / 100 % 10; out[2] = '0' + yy / 10 % 10; out[3] = '0' + yy % 10; out[4] = '-';
  out[5] = '0' + m / 10; out[6] = '0' + m % 10; out[7] = '-'; out[8] = '0' + d / 10; out[9] = '0' + d % 10; out[10] = ' ';
  out[11] = '0' + hh / 10; out[12] = '0' + hh % 10; out[13] = ':'; out[14] = '0' + mi / 10; out[15] = '0' + mi % 10; out[16] = ':';
  out[17] = '0' + ss / 10; out[18] = '0' + ss % 10;
  return 19;
}

// File-name fields and the strings Python would format from the metadata (rare predicates): kept out of line so that their
// buffers and divisions do not cost the common header path registers.  (Arguments by value: a reference to the kernel's by-value
// HeadArgs, like a dynamic index into one of its arrays, makes ptxas copy the whole struct to local memory -- that, via the aux
// column array, took the cfg2 head pass from 0.18 to 0.41 ms before it was noticed in the bench.)
struct NameArgs { const uint8_t* prog; const uint8_t* name; const uint64_t* name_off; const uint16_t* name_spans; const int64_t* ts; const int64_t* wall; bool prog_in_smem; };
__device__ __noinline__ void eval_name_fields(const NameArgs a, const fei_prog_hdr* ph, uint64_t rec, uint32_t* name_acc) {
  for (int k = 0; k < 3; ++k) {
    if (!ph->off_name_dfa[k]) continue;
    const uint8_t* nb = a.name + a.name_off[rec];
    uint32_t nl = (uint32_t)(a.name_off[rec + 1] - a.name_off[rec]);
    if (k > 0) { const uint16_t* sp = a.name_spans + 4 * rec + 2 * (k - 1); nb += sp[0]; nl = sp[1]; }
    name_acc[k] = dfa_run_at(a.prog, ph->off_name_dfa[k], a.prog_in_smem, nb, nl);
  }
  // str(timestamp) and str(datetime.fromtimestamp(ts))
  if (ph->off_meta_dfa[0]) { uint8_t buf[24]; const uint32_t nl = format_u64(a.ts[rec] < 0 ? 0ull : (unsigned long long)a.ts[rec], buf); name_acc[3] = dfa_run_at(a.prog, ph->off_meta_dfa[0], a.prog_in_smem, buf, nl); }
  if (ph->off_meta_dfa[1]) { uint8_t buf[24]; const uint32_t nl = format_datetime(a.wall[rec], buf); name_acc[4] = dfa_run_at(a.prog, ph->off_meta_dfa[1], a.prog_in_smem, buf, nl); }
}

// Phase 2 for one record: header fields (if `parse`), name fields, evaluation of the queries left in `pre`.
__device__ void head_finish(const HeadArgs& a, uint64_t rec, uint32_t pre, uint32_t flags_acc, bool parse) {
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(a.prog);
  const fei_prog_cond* conds = reinterpret_cast<const fei_prog_cond*>(a.prog + ph->off_conds);
  const fei_prog_query* queries = reinterpret_cast<const fei_prog_query*>(a.prog + ph->off_queries);
  const fei_prog_slot* slots = reinterpret_cast<const fei_prog_slot*>(a.prog + ph->off_slots);
  const uint32_t nslots = ph->n_slots;
  uint32_t slot_acc[FEI_MAX_SLOTS];
  uint32_t present = 0;
  if (parse) {
    uint32_t first_off[FEI_MAX_SLOTS], first_len[FEI_MAX_SLOTS];
    uint32_t have_first = 0;
    // fields that have a value column: the record's value sits at plane k, offset 16 * rec -- consecutive threads read
    // consecutive units, and neither the directory nor the header text of the record is touched
    bool walk = false;
    for (uint32_t s = 0; s < nslots; ++s) {
      const int col = a.slot_col[s];
      if (col == -2) continue;                                 // no record of this corpus has the field
      if (col < 0) { walk = true; break; }
      const uint32_t len = a.col_len[(uint64_t)col * a.n + rec];
      if (len == kColAbsent) continue;
      if (len == kColWalk) { walk = true; break; }
      const uint8_t* unit = a.col_planes + (uint64_t)col * kColUnits * a.n * 16 + rec * 16;
      slot_acc[s] = a.prog_in_smem ? dfa_run_units(dfa_view_s(a.prog, slots[s].off_val_dfa), unit, a.n * 16, len)
                                   : dfa_run_units_g(dfa_view(a.prog, slots[s].off_val_dfa), unit, a.n * 16, len);
      present |= 1u << s;
    }
    if (walk) {
    present = 0;
    const uint64_t hoff = a.hdr_off[rec];
    const uint8_t* h = a.hdr + hoff;
    const uint32_t hlen = (uint32_t)(a.hdr_off[rec + 1] - hoff);
    const uint2* ent = a.hdir + a.hdir_off[rec];
    const uint32_t n_ent = (uint32_t)(a.hdir_off[rec + 1] - a.hdir_off[rec]);
    if (!(n_ent == 1 && ent[0].x == 0xFFFFFFFFu)) {
      // the usual case: walk the record's header directory (one entry per line with a colon: interned key, stripped value span)
      uint32_t first_key[FEI_MAX_SLOTS], val_off[FEI_MAX_SLOTS], val_len[FEI_MAX_SLOTS];
      uint32_t any_mask = 0;                                   // mode-2 slots ("any header value", utils.py:333-336) already accumulated
      for (uint32_t j = 0; j < n_ent; ++j) {
        const uint2 e = ent[j];
        const uint32_t kid = e.x & 0xFFFFu;
        uint32_t km = a.key_lut[kid];
        while (km) {
          int s = __ffs(km) - 1; km &= km - 1;
          if (slots[s].mode == 2) {
            // every value of the headers dict: a line counts unless a later line assigns the same key again
            bool overridden = false;
            for (uint32_t k = j + 1; k < n_ent && !overridden; ++k) overridden = (ent[k].x & 0xFFFFu) == kid;
            if (overridden) continue;
            const uint32_t acc = dfa_run_at(a.prog, slots[s].off_val_dfa, a.prog_in_smem, h + e.y, e.x >> 16);
            slot_acc[s] = (any_mask >> s & 1u) ? (slot_acc[s] | acc) : acc;
            any_mask |= 1u << s;
            continue;
          }
          if (slots[s].mode == 0) {                            // first key that lower()-equals the field (search.py:121-122)
            if (!(have_first >> s & 1)) { have_first |= 1u << s; first_key[s] = kid; }
            else if (first_key[s] != kid) continue;            // a different spelling of the key: not the dict entry we read
          }
          val_off[s] = e.y; val_len[s] = e.x >> 16;            // repeated key: last value wins (dict assignment)
          present |= 1u << s;
        }
      }
      for (uint32_t m = present; m;) {
        int s = __ffs(m) - 1; m &= m - 1;
        slot_acc[s] = dfa_run_at(a.prog, slots[s].off_val_dfa, a.prog_in_smem, h + val_off[s], val_len[s]);
      }
      present |= any_mask;
    } else {
    // header text longer than a directory span can address: split / strip it here
    DfaView keyd = dfa_view(a.prog, ph->off_key_dfa);
    const uint8_t* hend = h + hlen;
    const uint8_t* p = h;
    while (p < hend) {
      const uint8_t* eol = p; const uint8_t* colon = nullptr;
      while (eol < hend && *eol != '\n') { if (!colon && *eol == ':') colon = eol; ++eol; }
      if (colon) {                                             // `if ":" in line` (utils.py:116)
        const uint8_t* ka = p; const uint8_t* kb = colon; strip_span(ka, kb);
        const uint8_t* va = colon + 1; const uint8_t* vb = eol; strip_span(va, vb);
        uint32_t km = dfa_run(keyd, ka, (uint32_t)(kb - ka));
        while (km) {
          int s = __ffs(km) - 1; km &= km - 1;
          if (slots[s].mode == 2) {
            // every value of the headers dict: this line counts unless a later line assigns the same (stripped) key again
            bool overridden = false;
            for (const uint8_t* q = eol + 1; q < hend && !overridden;) {
              const uint8_t* e2 = q; const uint8_t* c2 = nullptr;
              while (e2 < hend && *e2 != '\n') { if (!c2 && *e2 == ':') c2 = e2; ++e2; }
              if (c2) {
                const uint8_t* k2a = q; const uint8_t* k2b = c2; strip_span(k2a, k2b);
                bool same = (k2b - k2a) == (kb - ka);
                for (uint32_t k = 0; same && k < (uint32_t)(kb - ka); ++k) same = k2a[k] == ka[k];
                overridden = same;
              }
              q = e2 + 1;
            }
            if (overridden) continue;
            const uint32_t acc = dfa_run(dfa_view(a.prog, slots[s].off_val_dfa), va, (uint32_t)(vb - va));
            slot_acc[s] = (present >> s & 1u) ? (slot_acc[s] | acc) : acc;
            present |= 1u << s;
            continue;
          }
          if (slots[s].mode == 0) {                            // first key that lower()-equals the field (search.py:121-122)
            if (!(have_first >> s & 1)) { have_first |= 1u << s; first_off[s] = (uint32_t)(ka - h); first_len[s] = (uint32_t)(kb - ka); }
            else {
              bool same = first_len[s] == (uint32_t)(kb - ka);
              for (uint32_t k = 0; same && k < first_len[s]; ++k) same = h[first_off[s] + k] == ka[k];
              if (!same) continue;                             // a different spelling of the key: not the dict entry we read
            }
          }
          DfaView vd = dfa_view(a.prog, slots[s].off_val_dfa);
          slot_acc[s] = dfa_run(vd, va, (uint32_t)(vb - va));   // repeated key: last value wins (dict assignment)
          present |= 1u << s;
        }
      }
      p = eol + 1;
    }
    }
    }
  }
  for (uint32_t s = 0; s < nslots; ++s)
    if (!(present >> s & 1) && slots[s].empty_if_missing) {   // headers.get("Status", "")
      slot_acc[s] = reinterpret_cast<const fei_prog_dfa*>(a.prog + slots[s].off_val_dfa)->empty_acc;
      present |= 1u << s;
    }
  uint32_t name_acc[FEI_NAME_FIELDS] = {0, 0, 0, 0, 0};
  if (pre & ph->name_mask) eval_name_fields(NameArgs{a.prog, a.name, a.name_off, a.name_spans, a.ts, a.wall, (bool)a.prog_in_smem}, ph, rec, name_acc);
  uint32_t alive = 0;
  for (uint32_t q = 0; q < ph->n_queries; ++q) {
    if (!(pre >> q & 1)) continue;
    bool ok = true;
    bool fallback = false;                                      // the condition is the fallback field of an absent header
    for (uint32_t c = queries[q].cond_begin; ok && c < queries[q].cond_end; ++c) {
      const fei_prog_cond& cd = conds[c];
      bool r;
      switch (cd.kind) {
        case FEI_C_BODY: continue;                              // evaluated by k_body
        case FEI_C_SLOT:
          if (present >> cd.ref & 1) { r = ((slot_acc[cd.ref] >> cd.bit) & 1u) != cd.negate; if (cd.if_missing == 2) ++c; }
          else if (cd.if_missing == 2) { fallback = true; continue; }   // header absent: the next condition is the fallback field
          else r = cd.if_missing != 0;
          break;
        case FEI_C_NAME: r = ((name_acc[cd.ref < FEI_NAME_FIELDS ? cd.ref : 0] >> cd.bit) & 1u) != cd.negate; break;
        default:
          // meta predicates of a query in `pre` already held in k_head_meta; only a fallback field (skipped there) is still open
          r = fallback ? eval_meta_cond(a, rec, cd, flags_acc, a.wall[rec], a.fsb[rec]) : true;
      }
      fallback = false;
      ok = r;
    }
    if (ok) alive |= 1u << q;
  }
  a.alive[rec] = alive;
}

// Per scan: run the key automaton over the corpus' distinct header keys (hdir.cu), one thread per dictionary slot.
__global__ void k_key_lut(const uint8_t* __restrict__ prog, const uint8_t* __restrict__ hdr, const unsigned long long* __restrict__ tag,
                          const unsigned long long* __restrict__ rep, const uint32_t* __restrict__ len, uint32_t* __restrict__ lut) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= kKeySlots) return;
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(prog);
  lut[s] = tag[s] ? dfa_run(dfa_view(prog, ph->off_key_dfa), hdr + rep[s], len[s]) : 0u;
}

// One warp, after k_key_lut: a program slot whose field is spelled exactly one way in the whole corpus can be read from that
// key's value column (if it has one); a field no record carries is absent everywhere; anything else walks the directory.
__global__ void k_slot_cols(const uint8_t* __restrict__ prog, const uint32_t* __restrict__ lut, const int8_t* __restrict__ kid_col,
                            uint32_t n_cols, uint32_t any_text, int8_t* __restrict__ slot_col) {
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(prog);
  const int lane = threadIdx.x & 31;
  for (uint32_t s = 0; s < ph->n_slots && s < FEI_MAX_SLOTS; ++s) {
    uint32_t count = 0, kid = 0;
    for (uint32_t k = lane; k < kKeySlots; k += 32) if (lut[k] >> s & 1u) { ++count; kid = k; }
    for (int o = 16; o; o >>= 1) { count += __shfl_xor_sync(0xffffffffu, count, o); kid = max(kid, __shfl_xor_sync(0xffffffffu, kid, o)); }
    // (records whose header is parsed from its text keep their keys out of the dictionary: with any of those, nothing is "absent everywhere")
    if (lane == 0) slot_col[s] = count == 0 ? (any_text ? (int8_t)-1 : (int8_t)-2) : (count == 1 && n_cols ? kid_col[kid] : (int8_t)-1);
  }
}

// Every CTA of the head kernels first copies the "head" of the program (header, conditions, queries, slots and all
// automata except the big content one: fei_prog_hdr.head_bytes, a few KB) into shared memory with one TMA bulk copy,
// so that the interpretive condition loops and the short automaton runs read LDS instead of chasing global pointers.
constexpr uint32_t kHeadProgSmem = 32 * 1024;
__device__ __forceinline__ const uint8_t* stage_prog_head(const uint8_t* gprog, uint8_t* sprog, uint64_t* bar) {
  const uint32_t head_bytes = reinterpret_cast<const fei_prog_hdr*>(gprog)->head_bytes;
  if (head_bytes == 0 || head_bytes > kHeadProgSmem) return gprog;           // uniform for the whole grid
  if (threadIdx.x == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  __syncthreads();
  if (threadIdx.x == 0) { mbar_expect_tx(bar, head_bytes); bulk_g2s(sprog, gprog, head_bytes, bar); }
  mbar_wait(bar, 0);
  return sprog;
}

// k_head_meta streams the 20-byte meta columns, finalises every record that needs no header text and appends
// the others to a work list; k_head_parse then gives each survivor its own thread at full occupancy (a survivor's
// serial header walk does not pin a CTA full of already-finished threads), and the dead records' headers are never read.
struct Survivor { uint32_t rec, pre, flags_acc; };

constexpr int kMetaPer = 4;     // records per thread: the (uniform) condition fetch / decode is paid once for four records

template <bool kFused>
__global__ void __launch_bounds__(256, 5) k_head_meta(HeadArgs a, Survivor* __restrict__ list, unsigned int* __restrict__ count) {
  __shared__ __align__(128) uint8_t sprog[kHeadProgSmem];
  __shared__ uint64_t bar;
  a.prog = stage_prog_head(a.prog, sprog, &bar);
  a.prog_in_smem = a.prog == sprog;
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(a.prog);
  const fei_prog_cond* conds = reinterpret_cast<const fei_prog_cond*>(a.prog + ph->off_conds);
  const fei_prog_query* queries = reinterpret_cast<const fei_prog_query*>(a.prog + ph->off_queries);
  const uint64_t base = blockIdx.x * (uint64_t)(256 * kMetaPer) + threadIdx.x;
  uint32_t fsb[kMetaPer], flags_acc[kMetaPer], pre[kMetaPer];
  int64_t wall[kMetaPer];
  uint64_t f8[kMetaPer];
  bool valid[kMetaPer];
#pragma unroll
  for (int r = 0; r < kMetaPer; ++r) {
    const uint64_t i = base + (uint64_t)r * 256;
    valid[r] = i < a.n;
    fsb[r] = valid[r] ? a.fsb[i] : 0u; wall[r] = valid[r] ? a.wall[i] : 0; f8[r] = valid[r] ? a.flags8[i] : 0ull;
    flags_acc[r] = 0; pre[r] = 0;
  }
  if (ph->off_flags_dfa) {                                     // flags string (search.py:105-106): up to 7 letters in flags8
#pragma unroll
    for (int r = 0; r < kMetaPer; ++r) {
      if (a.prog_in_smem) flags_acc[r] = dfa_run_s_u64(dfa_view_s(a.prog, ph->off_flags_dfa), f8[r], (uint32_t)(f8[r] >> 56));
      else {
        uint8_t fb[8];
        for (int k = 0; k < 7; ++k) fb[k] = (uint8_t)(f8[r] >> (8 * k));
        flags_acc[r] = dfa_run(dfa_view(a.prog, ph->off_flags_dfa), fb, (uint32_t)(f8[r] >> 56));
      }
    }
  }
  for (uint32_t q = 0; q < ph->n_queries; ++q) {
    bool ok[kMetaPer];
#pragma unroll
    for (int r = 0; r < kMetaPer; ++r) ok[r] = true;
    for (uint32_t c = queries[q].cond_begin; c < queries[q].cond_end; ++c) {
      const fei_prog_cond cd = conds[c];
      if (cd.kind == FEI_C_SLOT && cd.if_missing == 2) { ++c; continue; }     // header-or-fallback pair: decided in phase 2
#pragma unroll
      for (int r = 0; r < kMetaPer; ++r) ok[r] = ok[r] && (!valid[r] || eval_meta_cond(a, base + (uint64_t)r * 256, cd, flags_acc[r], wall[r], fsb[r]));
    }
#pragma unroll
    for (int r = 0; r < kMetaPer; ++r) if (ok[r]) pre[r] |= 1u << q;
  }
  const uint32_t later_mask = ph->slot_mask | ph->name_mask;
  if (kFused) {
    // header / name fields right here: with value columns a record's fields are a couple of coalesced loads and short
    // automaton runs, so there is no long per-record walk that would pin the CTA, and the work list is not needed
    for (int r = 0; r < kMetaPer; ++r) {
      const uint64_t i = base + (uint64_t)r * 256;
      if (!valid[r]) continue;
      if ((pre[r] & later_mask) == 0) a.alive[i] = pre[r];
      else head_finish(a, i, pre[r], flags_acc[r], (pre[r] & ph->slot_mask) != 0);
    }
    return;
  }
  const int lane = threadIdx.x & 31;
  // survivors: slots are reserved per warp in shared memory and per CTA with ONE global atomic (a global atomic per
  // warp put 260 k same-address atomics on the L2 for 10 M records: 130 us, more than streaming the columns)
  __shared__ unsigned int cta_count, cta_base;
  if (threadIdx.x == 0) cta_count = 0;
  __syncthreads();
  bool later[kMetaPer];
  uint32_t bal[kMetaPer];
  unsigned int warp_total = 0;
#pragma unroll
  for (int r = 0; r < kMetaPer; ++r) {
    const uint64_t i = base + (uint64_t)r * 256;
    later[r] = valid[r] && (pre[r] & later_mask) != 0;
    if (valid[r] && !later[r]) a.alive[i] = pre[r];            // no header / name condition left: pre is the verdict
    bal[r] = __ballot_sync(0xffffffffu, later[r]);
    warp_total += __popc(bal[r]);
  }
  unsigned int warp_base = 0;
  if (lane == 0 && warp_total) warp_base = atomicAdd(&cta_count, warp_total);
  warp_base = __shfl_sync(0xffffffffu, warp_base, 0);
  __syncthreads();
  if (threadIdx.x == 0 && cta_count) cta_base = atomicAdd(count, cta_count);
  __syncthreads();
  unsigned int slot = cta_base + warp_base;
#pragma unroll
  for (int r = 0; r < kMetaPer; ++r) {
    if (later[r]) list[slot + __popc(bal[r] & ((1u << lane) - 1u))] = Survivor{(uint32_t)(base + (uint64_t)r * 256), pre[r], flags_acc[r]};
    slot += __popc(bal[r]);
  }
}

__global__ void __launch_bounds__(256, 5) k_head_parse(HeadArgs a, const Survivor* __restrict__ list, const unsigned int* __restrict__ n_list) {
  __shared__ __align__(128) uint8_t sprog[kHeadProgSmem];
  __shared__ uint64_t bar;
  const unsigned int n_surv = *n_list;                         // written by k_head_meta earlier on this stream: no host round trip
  if (blockIdx.x * blockDim.x >= n_surv) return;               // the grid is sized for "every record survives"
  a.prog = stage_prog_head(a.prog, sprog, &bar);
  a.prog_in_smem = a.prog == sprog;
  const unsigned int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_surv) return;
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(a.prog);
  const Survivor sv = list[t];
  head_finish(a, sv.rec, sv.pre, sv.flags_acc, (sv.pre & ph->slot_mask) != 0);
}

// ---------------------------------------------------------------- body kernel
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  }
}
__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

struct BodyArgs {
  const uint8_t* prog;
  const uint8_t* tiles; const uint64_t* grp_base; const uint32_t* grp_rec; const uint32_t* grp_len;
  uint64_t n_groups;
  uint32_t* hits;              // in: alive masks (when has_alive), out: final hit masks
  int has_alive;
  unsigned long long* counter; // [1] = tile bytes of the groups entered, [3] = tile bytes requested, [4] = live records (gather)
  unsigned long long gather_max;   // k_body_sticky stands down (and k_body_gather runs) when 0 < counter[4] <= gather_max
  // one launch covers the groups [g_begin, n_groups): the scan is cut into chunks of whole windows so that the compaction
  // (and, multi-GPU, the all-gather) of a finished chunk overlaps the next chunk's scan; *next hands out the chunk's groups
  unsigned long long g_begin;
  unsigned long long* next;
  // window w (groups [w * kWindow / 32, (w + 1) * kWindow / 32)) is finished when win_done[w] reaches kWindow / 32: the side stream
  // waits on these counters (k_wait_windows) to compact / send a finished run of windows while this kernel is still scanning
  unsigned int* win_done;
  // multi-GPU, fused exchange: the warp that completes a window stores the window's 4096 hit masks into every rank's rank-major
  // mask buffer (peer memory over NVLink / NVSwitch, mapped with CUDA IPC) -- the transfer of a finished window runs under the scan
  // of the next ones, from inside the scan kernel.  push_peers is a DEVICE array (a dynamic index into this by-value struct would
  // make ptxas copy it to local memory).
  uint32_t* const* push_peers; uint32_t push_n; unsigned long long push_off, n_records;
};
constexpr uint32_t kGroupsPerWindow = kWindow / 32;
__device__ __noinline__ void publish_window(const uint32_t* __restrict__ hits, uint32_t* const* __restrict__ peers, uint32_t n_peers,
                                            unsigned long long off, unsigned long long n_records, unsigned long long w, int lane) {
  __threadfence();                                   // acquire side of the window counter: the other groups' masks are visible now
  const unsigned long long r0 = w * kWindow;
  const uint32_t cnt = (uint32_t)((n_records - r0) < kWindow ? (n_records - r0) : kWindow);
  const uint32_t* src = hits + r0;                   // 16 KiB aligned; the destination is 16-byte aligned too (n_max is a multiple of 4)
  for (uint32_t p = 0; p < n_peers; ++p) {
    uint32_t* dst = peers[(p + (uint32_t)w) % n_peers];        // successive windows start with different ranks
    if (!dst) continue;
    dst += off + r0;
    for (uint32_t i = lane * 4u; i < cnt; i += 128u) {
      if (i + 4u <= cnt) {
        const uint4 v = __ldcg(reinterpret_cast<const uint4*>(src + i));        // L2: another SM wrote them
        *reinterpret_cast<uint4*>(dst + i) = v;
      } else {
        for (uint32_t j = i; j < cnt; ++j) dst[j] = __ldcg(src + j);
      }
    }
  }
  __threadfence_system();                            // the remote stores are ordered before this kernel's completion is observed
}
// kPush: the multi-GPU instantiation; the single-GPU kernels do not carry the exchange code (it cost 0.5 % of the headline
// when it was compiled into the one kernel: a shuffle and a branch per group, and a different register allocation)
template <bool kPush>
__device__ __forceinline__ void signal_group_done(const BodyArgs& a, unsigned long long g, int lane) {
  if (!a.win_done) return;
  __threadfence();                                   // this lane's hit mask is visible device-wide ...
  __syncwarp();
  unsigned int old = 0;
  if (lane == 0) old = atomicAdd(a.win_done + g / kGroupsPerWindow, 1u);   // ... before the group counts as done
  if (kPush && a.push_n) {
    old = __shfl_sync(0xffffffffu, old, 0);
    if (old + 1u == kGroupsPerWindow) publish_window(a.hits, a.push_peers, a.push_n, a.push_off, a.n_records, g / kGroupsPerWindow, lane);
  }
}

constexpr int kBodyThreads = 1024;

__device__ __forceinline__ uint32_t shl_clamp(uint32_t v, uint32_t n) {   // PTX shl clamps: n >= 32 -> 0
  uint32_t r;
  asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n));
  return r;
}

// One DFA step.  kAcc selects how accepting states are recorded (they are numbered 0..n_acc-1):
//   1 / 2 : branch-free, bit k of (a0,a1) = "accepting state k was visited" (n_acc <= 32 / <= 64):
//           no second shared-memory lookup and no divergent branch in the byte loop; the pattern
//           masks out[k] are OR-ed once per record from the visited-state bits;
//   0     : generic: out[] lookup when the new state is accepting.
// Address arithmetic is written so that it lands on the FMA pipe (IMAD) and only the byte extract
// (PRMT) and the accept bits (SHL/LOP3) use the ALU pipe: the loop is ALU-pipe / LDS-wavefront bound.
template <bool kDirect, int kAcc>
struct BodyDfa {
  uint32_t trans_s;            // shared-space address of the transition table
  const uint32_t* out; const uint8_t* cls;
  uint32_t stride2, n_acc;     // stride2 = row stride in bytes
  uint32_t s, a0;
  unsigned long long a64;
  __device__ __forceinline__ void step(uint32_t b) {
    uint32_t col = kDirect ? b : cls[b];
    uint32_t t, addr;
    asm("mad.lo.u32 %0, %1, 2, %2;" : "=r"(t) : "r"(col), "r"(trans_s));        // IMAD (FMA pipe)
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(s), "r"(stride2), "r"(t));
    uint16_t nxt;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(nxt) : "r"(addr));
    s = nxt;
    if (kAcc == 1) a0 |= shl_clamp(1u, s);            // s >= 32 shifts out: no bit
    if (kAcc == 2) { unsigned long long bit; asm("shl.b64 %0, %1, %2;" : "=l"(bit) : "l"(1ull), "r"(s)); a64 |= bit; }   // s >= 64: no bit
    if (kAcc == 0) { if (s < n_acc) a0 |= out[s]; }
    // kAcc == 3 ("sticky" single-pattern automaton): nothing to record, the verdict is endout[final state]
  }
  __device__ __forceinline__ void word(uint32_t w) {
    step(__byte_perm(w, 0, 0x4440)); step(__byte_perm(w, 0, 0x4441)); step(__byte_perm(w, 0, 0x4442)); step(__byte_perm(w, 0, 0x4443));
  }
  __device__ __forceinline__ void word_partial(uint32_t w, int nbytes) {
#pragma unroll
    for (int j = 0; j < 4; ++j) if (j < nbytes) step((w >> (8 * j)) & 0xFFu);
  }
  __device__ __forceinline__ void reset(uint32_t start) {
    s = start; a0 = 0; a64 = 0;
    if (kAcc == 0) a0 = start < n_acc ? out[start] : 0u;
    if (kAcc == 1) a0 = shl_clamp(1u, start);
    if (kAcc == 2) a64 = start < 64 ? 1ull << start : 0ull;
  }
  __device__ __forceinline__ uint32_t finish(const uint32_t* endout) const {
    uint32_t acc = endout[s];
    if (kAcc == 3) return acc;
    if (kAcc == 0) return acc | a0;
    unsigned long long m = kAcc == 1 ? (unsigned long long)a0 : a64;
    if (n_acc < 64) m &= (1ull << n_acc) - 1ull;
    while (m) { int k = __ffsll((long long)m) - 1; m &= m - 1; acc |= out[k]; }
    return acc;
  }
};

template <bool kDirect, int kAcc, bool kPush>
__global__ void __launch_bounds__(kBodyThreads, 1) k_body(BodyArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bar;
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(a.prog);
  const fei_prog_dfa* dd = reinterpret_cast<const fei_prog_dfa*>(a.prog + ph->off_body_dfa);
  const uint32_t table_bytes = dd->table_bytes;
  // ---- stage the automaton into shared memory with TMA bulk copies (cp.async.bulk + mbarrier)
  if (threadIdx.x == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar, table_bytes);
    const uint8_t* src = a.prog + dd->off_trans;
    for (uint32_t o = 0; o < table_bytes; o += 32768u) {
      uint32_t nb = table_bytes - o < 32768u ? table_bytes - o : 32768u;
      bulk_g2s(smem + o, src + o, nb, &bar);
    }
  }
  mbar_wait(&bar, 0);
  const uint32_t* endout = reinterpret_cast<const uint32_t*>(smem + (dd->off_endout - dd->off_trans));
  const uint32_t start = dd->start;
  const fei_prog_cond* conds = reinterpret_cast<const fei_prog_cond*>(a.prog + ph->off_conds);
  const fei_prog_query* queries = reinterpret_cast<const fei_prog_query*>(a.prog + ph->off_queries);
  const uint32_t nq = ph->n_queries;
  const uint32_t all_q = nq >= 32 ? 0xFFFFFFFFu : ((1u << nq) - 1u);
  const int lane = threadIdx.x & 31;
  unsigned long long touched = 0, bytes_read = 0;
  BodyDfa<kDirect, kAcc> d;
  d.trans_s = smem_u32(smem);
  d.out = reinterpret_cast<const uint32_t*>(smem + (dd->off_out - dd->off_trans));
  d.cls = smem + (dd->off_cls - dd->off_trans);
  d.stride2 = dd->row_stride * 2u; d.n_acc = dd->n_acc;
  const uint32_t sticky_state = dd->sticky ? dd->sticky - 1u : 0xFFFFFFFFu;

  for (;;) {
    unsigned long long g = 0;
    if (lane == 0) g = a.g_begin + atomicAdd(a.next, 1ull);
    g = __shfl_sync(0xffffffffu, g, 0);
    if (g >= a.n_groups) break;
    const uint32_t rec = a.grp_rec[g * 32 + lane];
    const uint32_t len = a.grp_len[g * 32 + lane];
    const uint32_t units = (len + 15) >> 4;
    uint32_t alive = 0;
    if (rec != kInvalidRec) alive = a.has_alive ? a.hits[rec] : all_q;
    const bool live = alive != 0;
    if (__ballot_sync(0xffffffffu, live) == 0) {              // nobody in this group can still match: skip its bytes
      if (rec != kInvalidRec && !a.has_alive) a.hits[rec] = 0;
      signal_group_done<kPush>(a, g, lane);
      continue;
    }
    const uint8_t* row = a.tiles + a.grp_base[g] * 16;
    const uint32_t maxu = __shfl_sync(0xffffffffu, units, 0);
    if (lane == 0) touched += (a.grp_base[g + 1] - a.grp_base[g]) * 16;
    const uint8_t* const row0 = row;
    d.reset(start);
    // software pipeline: the next row's 16 bytes are in flight while this row runs through the DFA
    uint4 cur = make_uint4(0, 0, 0, 0);
    if (0 < units && live) cur = ldg_stream16(row + lane * 16);
    for (uint32_t k = 0; k < maxu; ++k) {
      const uint32_t m = __popc(__ballot_sync(0xffffffffu, k < units));
      const uint8_t* next_row = row + (uint64_t)m * 16;
      uint4 nxt = make_uint4(0, 0, 0, 0);
      if (k + 1 < units && live) nxt = ldg_stream16(next_row + lane * 16);
      if (k < units && live) {
        int nb = (int)len - (int)(k * 16);
        if (nb >= 16) { d.word(cur.x); d.word(cur.y); d.word(cur.z); d.word(cur.w); }
        else { d.word_partial(cur.x, nb); d.word_partial(cur.y, nb - 4); d.word_partial(cur.z, nb - 8); d.word_partial(cur.w, nb - 12); }
      }
      cur = nxt; row = next_row;
      // sticky automaton: stop reading this group as soon as every live lane has either matched or ended
      if (kAcc == 3 && __ballot_sync(0xffffffffu, live && k + 1 < units && d.s != sticky_state) == 0) break;
    }
    if (lane == 0) bytes_read += (unsigned long long)(row - row0);
    if (live) {
      const uint32_t acc = d.finish(endout);
      uint32_t hit = 0;
      for (uint32_t q = 0; q < nq; ++q) {
        if (!(alive >> q & 1)) continue;
        bool ok = true;
        for (uint32_t c = queries[q].cond_begin; ok && c < queries[q].cond_end; ++c) {
          const fei_prog_cond& cd = conds[c];
          if (cd.kind == FEI_C_BODY) ok = ((acc >> cd.bit) & 1u) != cd.negate;
        }
        if (ok) hit |= 1u << q;
      }
      a.hits[rec] = hit;
    } else if (rec != kInvalidRec && !a.has_alive) {
      a.hits[rec] = 0;
    }
    signal_group_done<kPush>(a, g, lane);
  }
  if (lane == 0 && touched) { atomicAdd(a.counter + 1, touched); atomicAdd(a.counter + 3, bytes_read); }
}

// ---------------------------------------------------------------- single-pattern content scan, small automaton
// k_body_sticky: the kAcc == 3 case of k_body when the whole byte-indexed table sits below shared address 64 Ki.
// The transition entries are rewritten in place, after staging, from "state index" to "shared address of that
// state's row", so one step is PRMT (byte extract) + IMAD (byte * 2 + row address) + LDS.U16: 3 issue slots per
// byte instead of 4, no second multiply on the dependent chain.  Rows that are full for all 32 lanes (all but the
// ragged tail of a group: the records of a group are length-sorted neighbours) run in a predicate-free loop, two
// rows per iteration with the loads for the next two already in flight.
__device__ __forceinline__ uint32_t sticky_step(uint32_t e, uint32_t b) {
  uint32_t addr;
  asm("mad.lo.u32 %0, %1, 2, %2;" : "=r"(addr) : "r"(b), "r"(e));
  uint16_t nxt;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(nxt) : "r"(addr));
  return nxt;
}
__device__ __forceinline__ uint32_t sticky_word(uint32_t e, uint32_t w) {
  e = sticky_step(e, __byte_perm(w, 0, 0x4440)); e = sticky_step(e, __byte_perm(w, 0, 0x4441));
  e = sticky_step(e, __byte_perm(w, 0, 0x4442)); return sticky_step(e, __byte_perm(w, 0, 0x4443));
}
__device__ __forceinline__ uint32_t sticky_row(uint32_t e, const uint4& v) {
  return sticky_word(sticky_word(sticky_word(sticky_word(e, v.x), v.y), v.z), v.w);
}
__device__ __forceinline__ uint32_t sticky_partial(uint32_t e, uint32_t w, int nbytes) {
#pragma unroll
  for (int j = 0; j < 4; ++j) if (j < nbytes) e = sticky_step(e, (w >> (8 * j)) & 0xFFu);
  return e;
}

constexpr int kStages = 2, kChunkRows = 2;        // per warp: 2 stages, each 2 rows (1 KiB) of each of two groups
constexpr uint32_t kChunkBytes = kChunkRows * 512u;
constexpr uint32_t kStageBytes = 2 * kChunkBytes;
constexpr uint32_t kWarpRingBytes = kStages * kStageBytes;
constexpr uint32_t kStickyRingBytes = (kWarpRingBytes + kStages * 8u) * (kBodyThreads / 32);
__device__ __forceinline__ uint4 lds128(uint32_t addr_s) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr_s));
  return r;
}
constexpr unsigned long long kGatherDiv = 16;       // k_body_gather takes over when at most 1 record in 16 is still alive
constexpr uint32_t kStickyAddrLimit = 65535u;
constexpr uint32_t kStickyAddrSlack = 4096u;     // head-room the host leaves for the shared-memory window base

template <bool kPush>
__global__ void __launch_bounds__(kBodyThreads, 1) k_body_sticky(BodyArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bar;
  if (a.gather_max && a.counter[4] <= a.gather_max) return;    // few live records: k_body_gather has them (uniform for the grid)
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(a.prog);
  const fei_prog_dfa* dd = reinterpret_cast<const fei_prog_dfa*>(a.prog + ph->off_body_dfa);
  const uint32_t table_bytes = dd->table_bytes;
  if (threadIdx.x == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar, table_bytes);
    const uint8_t* src = a.prog + dd->off_trans;
    for (uint32_t o = 0; o < table_bytes; o += 32768u) {
      uint32_t nb = table_bytes - o < 32768u ? table_bytes - o : 32768u;
      bulk_g2s(smem + o, src + o, nb, &bar);
    }
  }
  mbar_wait(&bar, 0);
  const uint32_t trans_s = smem_u32(smem), stride2 = dd->row_stride * 2u, n_entries = dd->n_states * dd->row_stride;
  // per-warp ring + its mbarriers, behind the table
  const uint32_t warp = threadIdx.x >> 5;
  uint8_t* ring = smem + ((table_bytes + 127u) & ~127u) + warp * kWarpRingBytes;
  const uint32_t ring_s = smem_u32(ring);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ((table_bytes + 127u) & ~127u) + (kBodyThreads / 32) * kWarpRingBytes) + warp * kStages;
  if ((threadIdx.x & 31) < kStages) mbar_init(&bars[threadIdx.x & 31], 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  uint32_t prod = 0, cons = 0;                       // chunks issued / consumed by this warp since kernel start (stage = count % kStages)
  if (trans_s + dd->n_states * stride2 > kStickyAddrLimit) __trap();      // host-side eligibility test left 4 KiB of slack
  {
    uint16_t* t = reinterpret_cast<uint16_t*>(smem);
    for (uint32_t i = threadIdx.x; i < n_entries; i += kBodyThreads) t[i] = (uint16_t)(trans_s + (uint32_t)t[i] * stride2);
  }
  __syncthreads();
  const uint32_t* endout = reinterpret_cast<const uint32_t*>(smem + (dd->off_endout - dd->off_trans));
  const uint32_t start_e = trans_s + dd->start * stride2;
  const uint32_t sticky_e = dd->sticky != 0xFFFFFFFFu ? trans_s + (dd->sticky - 1u) * stride2 : 0xFFFFFFFFu;
  const fei_prog_cond* conds = reinterpret_cast<const fei_prog_cond*>(a.prog + ph->off_conds);
  const fei_prog_query* queries = reinterpret_cast<const fei_prog_query*>(a.prog + ph->off_queries);
  const uint32_t nq = ph->n_queries;
  const uint32_t all_q = nq >= 32 ? 0xFFFFFFFFu : ((1u << nq) - 1u);
  const int lane = threadIdx.x & 31;
  unsigned long long touched = 0, bytes_read = 0;

  // One group of 32 records as this warp sees it.
  struct Grp {
    uint32_t rec, len, alive, maxu, full, k, e;
    bool live;
    const uint8_t* row;          // next unread row
  };
  auto open_group = [&](unsigned long long g, Grp& G) {
    G.rec = kInvalidRec; G.len = 0; G.alive = 0; G.maxu = 0; G.full = 0; G.k = 0; G.e = start_e; G.live = false; G.row = a.tiles;
    if (g >= a.n_groups) return;
    G.rec = a.grp_rec[g * 32 + lane];
    G.len = a.grp_len[g * 32 + lane];
    if (G.rec != kInvalidRec) G.alive = a.has_alive ? a.hits[G.rec] : all_q;
    G.live = G.alive != 0;
    const uint32_t live_mask = __ballot_sync(0xffffffffu, G.live);
    if (live_mask == 0) return;                                     // nobody in this group can still match: skip its bytes
    G.row = a.tiles + a.grp_base[g] * 16;
    G.maxu = __shfl_sync(0xffffffffu, (G.len + 15) >> 4, 0);
    // rows that are 16 full bytes for all 32 lanes form one contiguous run of 512-byte rows.  Lanes a header predicate
    // already rejected ride along in the absorbing state (they read zeros, never hold up the early stop, write nothing):
    // a half-alive group keeps the streaming path instead of falling back to the row-by-row loop.
    const uint32_t valid_mask = __ballot_sync(0xffffffffu, G.rec != kInvalidRec);
    G.full = valid_mask == 0xffffffffu ? __reduce_min_sync(0xffffffffu, G.len >> 4) : 0u;
    if (!G.live && sticky_e != 0xFFFFFFFFu) G.e = sticky_e;
    if (lane == 0) touched += (a.grp_base[g + 1] - a.grp_base[g]) * 16;
  };
  // Full rows of ONE group through the ring: kChunkRows rows per bulk copy, kStages copies in flight; a stage is refilled
  // as soon as its rows sit in registers.
  auto stream_single = [&](Grp& G) {
    if (G.k >= G.full) return;
    const uint32_t n_chunks = (G.full - G.k) / kChunkRows;
    if (!n_chunks) return;
    uint32_t issued = 0, c = 0;
    for (; issued < n_chunks && issued < (uint32_t)kStages; ++issued, ++prod)
      if (lane == 0) { mbar_expect_tx(&bars[prod % kStages], kChunkBytes); bulk_g2s(ring + (prod % kStages) * kStageBytes, G.row + (uint64_t)issued * kChunkBytes, kChunkBytes, &bars[prod % kStages]); }
    bool stop = false;
    for (; c < n_chunks && !stop; ++c) {
      const uint32_t st = cons % kStages;
      mbar_wait(&bars[st], (cons / kStages) & 1u);
      ++cons;
      uint4 v[kChunkRows];
#pragma unroll
      for (int r = 0; r < kChunkRows; ++r) v[r] = lds128(ring_s + st * kStageBytes + r * 512u + lane * 16u);
      if (G.e == sticky_e) {                         // matched lanes all look up the same word (a broadcast) from here on
#pragma unroll
        for (int r = 0; r < kChunkRows; ++r) v[r] = make_uint4(0, 0, 0, 0);
      }
      __syncwarp();                                  // every lane holds its rows: the stage may be overwritten
      if (issued < n_chunks) {
        if (lane == 0) { mbar_expect_tx(&bars[st], kChunkBytes); bulk_g2s(ring + st * kStageBytes, G.row + (uint64_t)issued * kChunkBytes, kChunkBytes, &bars[st]); }
        ++issued; ++prod;
      }
#pragma unroll
      for (int r = 0; r < kChunkRows; ++r) G.e = sticky_row(G.e, v[r]);
      stop = __ballot_sync(0xffffffffu, G.e != sticky_e) == 0;      // every lane has matched
    }
    for (; cons < prod; ++cons) mbar_wait(&bars[cons % kStages], (cons / kStages) & 1u);   // early stop: let the copies in flight land
    bytes_read += (unsigned long long)issued * kChunkBytes;
    G.row += (uint64_t)c * kChunkBytes;
    G.k = stop ? G.maxu : G.k + c * kChunkRows;
  };
  // The same for TWO groups in lock step: each lane runs two independent automaton chains, so the shared-memory
  // latency of one lookup is covered by the other chain's (the single chain is LDS-latency bound: 8 warps per scheduler).
  auto stream_pair = [&](Grp& A, Grp& B) {
    const uint32_t n_chunks = (A.full < B.full ? A.full : B.full) / kChunkRows;
    if (!n_chunks) return;
    uint32_t issued = 0, c = 0;
    auto issue = [&](uint32_t st) {
      if (lane == 0) {
        mbar_expect_tx(&bars[st], 2 * kChunkBytes);
        bulk_g2s(ring + st * kStageBytes, A.row + (uint64_t)issued * kChunkBytes, kChunkBytes, &bars[st]);
        bulk_g2s(ring + st * kStageBytes + kChunkBytes, B.row + (uint64_t)issued * kChunkBytes, kChunkBytes, &bars[st]);
      }
      ++issued; ++prod;
    };
    while (issued < n_chunks && issued < (uint32_t)kStages) issue(prod % kStages);
    bool stop_a = false, stop_b = false;
    for (; c < n_chunks && !stop_a && !stop_b; ++c) {
      const uint32_t st = cons % kStages;
      mbar_wait(&bars[st], (cons / kStages) & 1u);
      ++cons;
      uint4 va[kChunkRows], vb[kChunkRows];
#pragma unroll
      for (int r = 0; r < kChunkRows; ++r) {
        va[r] = lds128(ring_s + st * kStageBytes + r * 512u + lane * 16u);
        vb[r] = lds128(ring_s + st * kStageBytes + kChunkBytes + r * 512u + lane * 16u);
      }
      uint32_t ea = A.e, eb = B.e;
      // a lane that has matched stays in the absorbing state whatever it reads: give it zeros, so that all matched
      // lanes look up one and the same word (a broadcast) instead of spreading over the banks of the absorbing row
      if (ea == sticky_e) {
#pragma unroll
        for (int r = 0; r < kChunkRows; ++r) va[r] = make_uint4(0, 0, 0, 0);
      }
      if (eb == sticky_e) {
#pragma unroll
        for (int r = 0; r < kChunkRows; ++r) vb[r] = make_uint4(0, 0, 0, 0);
      }
      __syncwarp();
      if (issued < n_chunks) issue(st);
#pragma unroll
      for (int r = 0; r < kChunkRows; ++r) {
        const uint32_t wa[4] = {va[r].x, va[r].y, va[r].z, va[r].w}, wb[4] = {vb[r].x, vb[r].y, vb[r].z, vb[r].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          ea = sticky_step(ea, __byte_perm(wa[j], 0, 0x4440)); eb = sticky_step(eb, __byte_perm(wb[j], 0, 0x4440));
          ea = sticky_step(ea, __byte_perm(wa[j], 0, 0x4441)); eb = sticky_step(eb, __byte_perm(wb[j], 0, 0x4441));
          ea = sticky_step(ea, __byte_perm(wa[j], 0, 0x4442)); eb = sticky_step(eb, __byte_perm(wb[j], 0, 0x4442));
          ea = sticky_step(ea, __byte_perm(wa[j], 0, 0x4443)); eb = sticky_step(eb, __byte_perm(wb[j], 0, 0x4443));
        }
      }
      A.e = ea; B.e = eb;
      stop_a = __ballot_sync(0xffffffffu, ea != sticky_e) == 0;
      stop_b = __ballot_sync(0xffffffffu, eb != sticky_e) == 0;
    }
    for (; cons < prod; ++cons) mbar_wait(&bars[cons % kStages], (cons / kStages) & 1u);
    bytes_read += 2ull * issued * kChunkBytes;
    A.row += (uint64_t)c * kChunkBytes; B.row += (uint64_t)c * kChunkBytes;
    A.k = stop_a ? A.maxu : c * kChunkRows;
    B.k = stop_b ? B.maxu : c * kChunkRows;
  };
  // Ragged remainder of both groups (and groups with dead lanes), still two chains per lane: row k of a group holds
  // only the lanes that have a unit k (lane count from a ballot), every lane steps through all 16 bytes and keeps
  // the new state only for the bytes its record really has (nb), so there is no divergent branch between the chains.
  auto ragged_pair = [&](Grp& A, Grp& B) {
    const uint32_t rem_a = A.maxu - A.k, rem_b = B.maxu - B.k;       // k <= maxu always
    const uint32_t rounds = rem_a > rem_b ? rem_a : rem_b;
    if (!rounds) return;
    const uint32_t units_a = (A.len + 15) >> 4, units_b = (B.len + 15) >> 4;
    bool act_a = A.live && rem_a, act_b = B.live && rem_b;
    const uint8_t* row_a = A.row; const uint8_t* row_b = B.row;
    uint32_t ea = A.e, eb = B.e;
    uint4 cur_a = make_uint4(0, 0, 0, 0), cur_b = cur_a;
    if (act_a && A.k < units_a) cur_a = ldg_stream16(row_a + lane * 16);
    if (act_b && B.k < units_b) cur_b = ldg_stream16(row_b + lane * 16);
    for (uint32_t i = 0; i < rounds; ++i) {
      const uint32_t ka = A.k + i, kb = B.k + i;
      bytes_read += __popc(__ballot_sync(0xffffffffu, act_a && ka < units_a)) * 16 + __popc(__ballot_sync(0xffffffffu, act_b && kb < units_b)) * 16;
      row_a += (uint64_t)__popc(__ballot_sync(0xffffffffu, ka < units_a)) * 16;
      row_b += (uint64_t)__popc(__ballot_sync(0xffffffffu, kb < units_b)) * 16;
      uint4 nxt_a = make_uint4(0, 0, 0, 0), nxt_b = nxt_a;
      if (act_a && ka + 1 < units_a) nxt_a = ldg_stream16(row_a + lane * 16);
      if (act_b && kb + 1 < units_b) nxt_b = ldg_stream16(row_b + lane * 16);
      int nba = act_a ? (int)A.len - (int)(ka * 16) : 0, nbb = act_b ? (int)B.len - (int)(kb * 16) : 0;   // <= 0: no byte of this row
      const uint32_t wa[4] = {cur_a.x, cur_a.y, cur_a.z, cur_a.w}, wb[4] = {cur_b.x, cur_b.y, cur_b.z, cur_b.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t ta = sticky_step(ea, __byte_perm(wa[j], 0, 0x4440 + q)), tb = sticky_step(eb, __byte_perm(wb[j], 0, 0x4440 + q));
          ea = 4 * j + q < nba ? ta : ea;
          eb = 4 * j + q < nbb ? tb : eb;
        }
      }
      cur_a = nxt_a; cur_b = nxt_b;
      // a group is finished as soon as every live lane has either matched or ended
      if (__ballot_sync(0xffffffffu, act_a && ka + 1 < units_a && ea != sticky_e) == 0) act_a = false;
      if (__ballot_sync(0xffffffffu, act_b && kb + 1 < units_b && eb != sticky_e) == 0) act_b = false;
      if (__ballot_sync(0xffffffffu, act_a || act_b) == 0) break;
    }
    A.e = ea; B.e = eb;
  };
  auto close_group = [&](const Grp& G) {
    if (G.live) {
      const uint32_t acc = endout[(G.e - trans_s) / stride2];
      uint32_t hit = 0;
      for (uint32_t q = 0; q < nq; ++q) {
        if (!(G.alive >> q & 1)) continue;
        bool ok = true;
        for (uint32_t c = queries[q].cond_begin; ok && c < queries[q].cond_end; ++c) {
          const fei_prog_cond& cd = conds[c];
          if (cd.kind == FEI_C_BODY) ok = ((acc >> cd.bit) & 1u) != cd.negate;
        }
        if (ok) hit |= 1u << q;
      }
      a.hits[G.rec] = hit;
    } else if (G.rec != kInvalidRec && !a.has_alive) {
      a.hits[G.rec] = 0;
    }
  };

  for (;;) {
    unsigned long long g = 0;
    if (lane == 0) g = a.g_begin + atomicAdd(a.next, 2ull);
    g = __shfl_sync(0xffffffffu, g, 0);
    if (g >= a.n_groups) break;
    Grp A, B;
    open_group(g, A);
    open_group(g + 1, B);
    stream_pair(A, B);
    stream_single(A);
    stream_single(B);
    ragged_pair(A, B);
    close_group(A);
    close_group(B);
    signal_group_done<kPush>(a, g, lane);
    if (g + 1 < a.n_groups) signal_group_done<kPush>(a, g + 1, lane);
  }
  if (lane == 0 && touched) { atomicAdd(a.counter + 1, touched); atomicAdd(a.counter + 3, bytes_read); }
}

// ---------------------------------------------------------------- single-pattern scan of FEW surviving records
// After selective header predicates a group of 32 has at most a lane or two left alive; k_body_sticky then runs one
// serial automaton chain per group and the SM idles at 64 chains (measured 0.25 ms for 35 k survivors of 10 M records:
// the latency floor of that shape).  k_live_list compacts the survivors and k_body_gather gives every one its own
// thread: a lane walks its record through the tiles of its group (row k of a group starts 16 * sum_{j<k} m_j after the
// group base, m_j = lanes that still have a unit j, recovered from the group's sorted lengths), so a warp runs 32 chains.
__global__ void __launch_bounds__(256) k_live_list(const uint32_t* __restrict__ alive, uint64_t n, uint32_t* __restrict__ list,
                                                  unsigned long long* __restrict__ count, unsigned long long cap) {
  __shared__ unsigned int cta_count; __shared__ unsigned long long cta_base;
  if (threadIdx.x == 0) cta_count = 0;
  __syncthreads();
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const bool live = i < n && alive[i] != 0;
  const uint32_t bal = __ballot_sync(0xffffffffu, live);
  const int lane = threadIdx.x & 31;
  unsigned int wbase = 0;
  if (lane == 0 && bal) wbase = atomicAdd(&cta_count, (unsigned int)__popc(bal));
  wbase = __shfl_sync(0xffffffffu, wbase, 0);
  __syncthreads();
  if (threadIdx.x == 0 && cta_count) cta_base = atomicAdd(count, (unsigned long long)cta_count);
  __syncthreads();
  if (live) { const unsigned long long at = cta_base + wbase + __popc(bal & ((1u << lane) - 1u)); if (at < cap) list[at] = (uint32_t)i; }
}

__global__ void __launch_bounds__(kBodyThreads, 1) k_body_gather(BodyArgs a, const uint32_t* __restrict__ live, const uint32_t* __restrict__ rec_pos) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bar;
  const unsigned long long n_live = a.counter[4];
  if (n_live == 0 || n_live > a.gather_max) return;            // k_body_sticky takes the dense case (uniform for the grid)
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(a.prog);
  const fei_prog_dfa* dd = reinterpret_cast<const fei_prog_dfa*>(a.prog + ph->off_body_dfa);
  const uint32_t table_bytes = dd->table_bytes;
  if (threadIdx.x == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar, table_bytes);
    const uint8_t* src = a.prog + dd->off_trans;
    for (uint32_t o = 0; o < table_bytes; o += 32768u) {
      uint32_t nb = table_bytes - o < 32768u ? table_bytes - o : 32768u;
      bulk_g2s(smem + o, src + o, nb, &bar);
    }
  }
  mbar_wait(&bar, 0);
  const uint32_t trans_s = smem_u32(smem), stride2 = dd->row_stride * 2u, n_entries = dd->n_states * dd->row_stride;
  if (trans_s + dd->n_states * stride2 > kStickyAddrLimit) __trap();
  {
    uint16_t* t = reinterpret_cast<uint16_t*>(smem);
    for (uint32_t i = threadIdx.x; i < n_entries; i += kBodyThreads) t[i] = (uint16_t)(trans_s + (uint32_t)t[i] * stride2);
  }
  __syncthreads();
  const uint32_t* endout = reinterpret_cast<const uint32_t*>(smem + (dd->off_endout - dd->off_trans));
  const uint32_t start_e = trans_s + dd->start * stride2;
  const uint32_t sticky_e = dd->sticky != 0xFFFFFFFFu ? trans_s + (dd->sticky - 1u) * stride2 : 0xFFFFFFFFu;
  const fei_prog_cond* conds = reinterpret_cast<const fei_prog_cond*>(a.prog + ph->off_conds);
  const fei_prog_query* queries = reinterpret_cast<const fei_prog_query*>(a.prog + ph->off_queries);
  const uint32_t nq = ph->n_queries;
  unsigned long long bytes_read = 0;
  for (unsigned long long t = blockIdx.x * (unsigned long long)kBodyThreads + threadIdx.x; t < n_live; t += (unsigned long long)gridDim.x * kBodyThreads) {
    const uint32_t rec = live[t];
    const uint32_t pos = rec_pos[rec];
    const uint64_t g = pos >> 5; const uint32_t l = pos & 31u;
    const uint32_t* gl = a.grp_len + g * 32;
    const uint32_t len = gl[l];
    const uint32_t units = (len + 15) >> 4;
    const uint32_t alive = a.hits[rec];
    uint32_t m = 32;                                             // lanes of the group that have a unit k (lengths are sorted descending)
    uint32_t drop = (gl[31] + 15) >> 4;                          // the first row lane m-1 is missing from
    const uint8_t* p = a.tiles + a.grp_base[g] * 16 + l * 16;
    uint32_t e = start_e;
    for (uint32_t k = 0; k < units; ++k) {
      while (k >= drop) { --m; drop = m > l + 1 ? (gl[m - 1] + 15) >> 4 : 0xFFFFFFFFu; }
      const uint4 v = ldg_stream16(p);
      p += (uint64_t)m * 16;
      const int nb = (int)len - (int)(k * 16);
      if (nb >= 16) e = sticky_row(e, v);
      else { e = sticky_partial(e, v.x, nb); e = sticky_partial(e, v.y, nb - 4); e = sticky_partial(e, v.z, nb - 8); e = sticky_partial(e, v.w, nb - 12); }
      bytes_read += 16;
      if (e == sticky_e) break;                                  // matched: the verdict cannot change any more
    }
    const uint32_t acc = endout[(e - trans_s) / stride2];
    uint32_t hit = 0;
    for (uint32_t q = 0; q < nq; ++q) {
      if (!(alive >> q & 1)) continue;
      bool ok = true;
      for (uint32_t c = queries[q].cond_begin; ok && c < queries[q].cond_end; ++c) {
        const fei_prog_cond& cd = conds[c];
        if (cd.kind == FEI_C_BODY) ok = ((acc >> cd.bit) & 1u) != cd.negate;
      }
      if (ok) hit |= 1u << q;
    }
    a.hits[rec] = hit;
  }
  for (int o = 16; o; o >>= 1) bytes_read += __shfl_down_sync(0xffffffffu, bytes_read, o);
  if ((threadIdx.x & 31) == 0 && bytes_read) { atomicAdd(a.counter + 3, bytes_read); atomicAdd(a.counter + 1, bytes_read); }
}

template <bool kDirect, int kAcc>
static int launch_body(const BodyArgs& a, unsigned grid, size_t smem, cudaStream_t s) {
  if (a.push_n) {
    FEI_CUDA(cudaFuncSetAttribute(k_body<kDirect, kAcc, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_body<kDirect, kAcc, true><<<grid, kBodyThreads, smem, s>>>(a);
  } else {
    FEI_CUDA(cudaFuncSetAttribute(k_body<kDirect, kAcc, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_body<kDirect, kAcc, false><<<grid, kBodyThreads, smem, s>>>(a);
  }
  return FEI_OK;
}

// ---------------------------------------------------------------- compaction
constexpr int kCompactBlock = 256;          // threads
constexpr int kCompactPer = 8;              // records per thread -> 2048 records per block
constexpr uint64_t kCompactRecs = (uint64_t)kCompactBlock * kCompactPer;

// counts[block * nq + q] = records of this block that hit query q  (block = blk0 + blockIdx.x: a chunk of the scan
// compacts its own blocks while the next chunk is still being scanned)
__global__ void __launch_bounds__(kCompactBlock)
k_count(const uint32_t* __restrict__ hits, uint64_t n, uint32_t nq, uint64_t blk0, uint32_t* __restrict__ counts) {
  __shared__ uint32_t sh[32][8];
  const uint64_t blk = blk0 + blockIdx.x;
  uint64_t base = blk * kCompactRecs;
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t cnt = 0;                        // lane q accumulates query q
  for (int r = 0; r < kCompactPer; ++r) {
    uint64_t i = base + (uint64_t)(warp * kCompactPer + r) * 32 + lane;
    uint32_t m = i < n ? hits[i] : 0u;
    for (uint32_t q = 0; q < nq; ++q) {
      uint32_t b = __popc(__ballot_sync(0xffffffffu, (m >> q) & 1u));
      if (lane == (int)q) cnt += b;
    }
  }
  sh[lane][warp] = cnt;
  __syncthreads();
  if (threadIdx.x < 32 && threadIdx.x < nq) {
    uint32_t s = 0;
    for (int w = 0; w < 8; ++w) s += sh[threadIdx.x][w];
    counts[blk * nq + threadIdx.x] = s;
  }
}

// per query: exclusive scan over the blocks [blk0, blk0 + nblocks) (one thread block per query), continuing from
// carry[q] (the hits of the blocks before blk0) and leaving the new running total there
__global__ void k_scan_blocks(const uint32_t* __restrict__ counts, uint64_t blk0, uint64_t nblocks, uint32_t nq,
                              uint64_t* __restrict__ offsets, uint64_t* __restrict__ carry_io) {
  __shared__ uint64_t sh[1024];
  __shared__ uint64_t carry;
  uint32_t q = blockIdx.x;
  if (threadIdx.x == 0) carry = carry_io[q];
  __syncthreads();
  for (uint64_t base = 0; base < nblocks; base += blockDim.x) {
    uint64_t b = base + threadIdx.x;
    uint64_t v = b < nblocks ? counts[(blk0 + b) * nq + q] : 0;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < blockDim.x; o <<= 1) {
      uint64_t t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
      __syncthreads();
      sh[threadIdx.x] += t;
      __syncthreads();
    }
    uint64_t incl = sh[threadIdx.x];
    if (b < nblocks) offsets[(blk0 + b) * nq + q] = carry + incl - v;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry += incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) carry_io[q] = carry;
}

// ordered emit: lists[q * stride + rank] = global_base + i
// (32 registers: one CTA of it fits next to a 1024-thread scan CTA that leaves 8 K of the SM's registers free)
__global__ void __launch_bounds__(kCompactBlock, 8)
k_emit(const uint32_t* __restrict__ hits, uint64_t n, uint32_t nq, const uint64_t* __restrict__ offsets, uint64_t blk0,
       uint64_t global_base, uint64_t stride, uint64_t* __restrict__ lists) {
  __shared__ uint32_t wcnt[8][32];          // [warp][query] hits of this warp's records
  const uint64_t blk = blk0 + blockIdx.x;
  uint64_t base = blk * kCompactRecs;
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t m[kCompactPer];
  uint32_t cnt = 0;
  for (int r = 0; r < kCompactPer; ++r) {
    uint64_t i = base + (uint64_t)(warp * kCompactPer + r) * 32 + lane;
    m[r] = i < n ? hits[i] : 0u;
    for (uint32_t q = 0; q < nq; ++q) {
      uint32_t b = __popc(__ballot_sync(0xffffffffu, (m[r] >> q) & 1u));
      if (lane == (int)q) cnt += b;
    }
  }
  wcnt[warp][lane] = cnt;
  __syncthreads();
  for (uint32_t q = 0; q < nq; ++q) {
    uint64_t pos = offsets[blk * nq + q];
    for (int w = 0; w < warp; ++w) pos += wcnt[w][q];
    for (int r = 0; r < kCompactPer; ++r) {
      uint32_t bal = __ballot_sync(0xffffffffu, (m[r] >> q) & 1u);
      if ((m[r] >> q) & 1u) {
        uint64_t i = base + (uint64_t)(warp * kCompactPer + r) * 32 + lane;
        uint64_t rank = pos + __popc(bal & ((1u << lane) - 1u));
        if (rank < stride) lists[q * stride + rank] = global_base + i;
      }
      pos += __popc(bal);
    }
  }
}

// Side-stream gate of a pipelined scan: one warp spins until every window of [w0, w1) is finished (see BodyArgs::win_done).
// A warp that sleeps between polls costs the scan nothing; the time limit only guards against a scan kernel that died.
__global__ void k_wait_windows(const volatile unsigned int* __restrict__ win_done, uint64_t w0, uint64_t w1, unsigned long long* __restrict__ err) {
  const int lane = threadIdx.x & 31;
  const long long t0 = clock64();
  for (;;) {
    bool ok = true;
    for (uint64_t w = w0 + lane; w < w1; w += 32) ok = ok && win_done[w] >= kGroupsPerWindow;
    if (__all_sync(0xffffffffu, ok)) break;
    if (clock64() - t0 > 20000000000ll) { if (lane == 0) atomicExch(err, 1ull); break; }     // ~10 s
    __nanosleep(1000);
  }
  __threadfence();
}

__global__ void k_fill32(uint32_t* __restrict__ p, uint64_t n, uint32_t v) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// Order-sensitive checksum of an index list: sum_k (k + 1) * v[k] and sum_k v[k] (mod 2^64).  Two lists agree on both
// sums iff (with overwhelming probability) they hold the same indices in the same order; the pair (A, S) of the
// concatenation of two lists follows from the parts: A = A1 + A2 + len1 * S2.
__global__ void __launch_bounds__(256) k_list_checksum(const uint64_t* __restrict__ v, uint64_t n, unsigned long long* __restrict__ out) {
  unsigned long long a = 0, s = 0;
  for (uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) { a += (k + 1) * v[k]; s += v[k]; }
  for (int o = 16; o; o >>= 1) { a += __shfl_down_sync(0xffffffffu, a, o); s += __shfl_down_sync(0xffffffffu, s, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out, a); atomicAdd(out + 1, s); }
}

// ---------------------------------------------------------------- host side
static int check_prog(const uint8_t* prog, uint64_t len) {
  if (!prog || len < sizeof(fei_prog_hdr)) { set_error("program blob too small"); return FEI_E_BADARG; }
  fei_prog_hdr h; memcpy(&h, prog, sizeof(h));
  if (h.magic != FEI_PROG_MAGIC || h.version != FEI_PROG_VERSION) { set_error("bad program magic/version"); return FEI_E_BADARG; }
  if (h.total_bytes != len) { set_error("program length mismatch (%u vs %llu)", h.total_bytes, (unsigned long long)len); return FEI_E_BADARG; }
  if (h.n_queries == 0 || h.n_queries > FEI_MAX_QUERIES) { set_error("1..32 queries per program"); return FEI_E_BADARG; }
  if (h.n_slots > FEI_MAX_SLOTS) { set_error("at most %d header slots per program", FEI_MAX_SLOTS); return FEI_E_UNSUPPORTED; }
  auto in = [&](uint64_t off, uint64_t sz) { return off % 16 == 0 && off + sz <= len; };
  if (!in(h.off_conds, (uint64_t)h.n_conds * sizeof(fei_prog_cond)) || !in(h.off_queries, (uint64_t)h.n_queries * sizeof(fei_prog_query)) ||
      !in(h.off_slots, (uint64_t)h.n_slots * sizeof(fei_prog_slot))) { set_error("program section out of bounds"); return FEI_E_BADARG; }
  auto dfa_ok = [&](uint32_t off) {
    if (!off) return true;
    if (!in(off, sizeof(fei_prog_dfa))) return false;
    fei_prog_dfa d; memcpy(&d, prog + off, sizeof(d));
    return in(d.off_trans, d.table_bytes) && d.start < d.n_states && d.n_cols >= 1 && d.n_cols <= 256 &&
           d.off_out >= d.off_trans && d.off_endout >= d.off_trans && d.off_cls >= d.off_trans &&
           d.off_out + 4ull * d.n_states <= (uint64_t)d.off_trans + d.table_bytes &&
           d.off_endout + 4ull * d.n_states <= (uint64_t)d.off_trans + d.table_bytes &&
           d.row_stride >= d.n_cols && 2ull * d.n_states * d.row_stride <= d.trans_bytes && d.n_states <= 65535;
  };
  if (!dfa_ok(h.off_key_dfa) || !dfa_ok(h.off_body_dfa) || !dfa_ok(h.off_flags_dfa) || !dfa_ok(h.off_name_dfa[0]) ||
      !dfa_ok(h.off_name_dfa[1]) || !dfa_ok(h.off_name_dfa[2]) || !dfa_ok(h.off_meta_dfa[0]) || !dfa_ok(h.off_meta_dfa[1])) { set_error("bad DFA descriptor in program"); return FEI_E_BADARG; }
  const fei_prog_slot* sl = reinterpret_cast<const fei_prog_slot*>(prog + h.off_slots);
  for (uint32_t s = 0; s < h.n_slots; ++s) if (!sl[s].off_val_dfa || !dfa_ok(sl[s].off_val_dfa)) { set_error("bad slot DFA"); return FEI_E_BADARG; }
  if (h.n_slots && !h.off_key_dfa) { set_error("slots without a key DFA"); return FEI_E_BADARG; }
  if (h.head_bytes > h.total_bytes || (h.head_bytes & 15u)) { set_error("bad head_bytes in program"); return FEI_E_BADARG; }
  const fei_prog_query* qs = reinterpret_cast<const fei_prog_query*>(prog + h.off_queries);
  for (uint32_t q = 0; q < h.n_queries; ++q) if (qs[q].cond_begin > qs[q].cond_end || qs[q].cond_end > h.n_conds) { set_error("bad query range"); return FEI_E_BADARG; }
  return FEI_OK;
}


// ---- chunking: the body pass runs as up to kMaxChunks launches over runs of whole windows (a window = kWindow consecutive
// records = kWindow / 32 groups, so a chunk's hit masks are one contiguous record range).  The moment a chunk's masks are
// final its compaction (and the hook, e.g. the NCCL all-gather of comm.cu) is queued on the side stream and runs under the
// next chunk's scan: the 32-pattern scan is shared-memory bound and leaves three quarters of the HBM bandwidth idle.
constexpr uint32_t kMaxChunks = 16;
struct ChunkPlan { uint32_t n = 1; uint64_t g[kMaxChunks + 1] = {0}; uint64_t rec[kMaxChunks + 1] = {0}; };

static uint32_t chunk_count(uint64_t n_windows, bool allow, bool watermark) {
  uint32_t want = 0;
  if (const char* e = getenv("FEI_SCAN_CHUNKS")) want = (uint32_t)atoi(e);
  if (!allow) return 1;
  // logical chunks of a single launch are nearly free (a one-warp gate kernel each): ~300 k records and up, at most 16; separate
  // launches cost a kernel tail each, so without the window counters the scan stays in one piece unless asked otherwise
  if (!want) want = watermark ? (uint32_t)(n_windows / 80) : 1;
  if (want > kMaxChunks) want = kMaxChunks;
  if (want > n_windows) want = (uint32_t)n_windows;
  return want ? want : 1;
}
void plan_chunks(uint64_t n, uint32_t chunks, uint64_t* rec_bounds) {       // shared with comm.cu: every rank derives every rank's bounds
  const uint64_t n_windows = (n + kWindow - 1) / kWindow;
  for (uint32_t k = 0; k <= chunks; ++k) { uint64_t r = n_windows * k / chunks * kWindow; rec_bounds[k] = r < n ? r : n; }
  rec_bounds[chunks] = n;
}

static int ensure_side(fei_corpus* c) {
  if (!c->side) {                                              // highest priority: a finished chunk's compaction / all-gather gets the first SM that frees up
    int lo = 0, hi = 0;
    FEI_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    FEI_CUDA(cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, hi));
  }
  for (auto& e : c->ev_chunk) if (!e) FEI_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  if (!c->ev_side) FEI_CUDA(cudaEventCreateWithFlags(&c->ev_side, cudaEventDisableTiming));
  return FEI_OK;
}

enum { kCompactNone = kScanCompactNone, kCompactLists = kScanCompactLists };

// Everything is queued on the context stream (and the corpus' side stream); nothing here waits for the GPU.
int run_scan(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, int compact_mode, ChunkHook* hook, uint32_t force_chunks) {
  FEI_TRY(require_ready());
  if (!c || !c->loaded) { set_error("corpus not loaded"); return FEI_E_STATE; }
  FEI_TRY(check_prog(prog, prog_len));
  Context& cx = ctx();
  cudaStream_t s = cx.stream;
  fei_prog_hdr h; memcpy(&h, prog, sizeof(h));
  uint64_t n = c->n;
  c->timing = fei_scan_timing{};
  c->last_nq = h.n_queries;
  for (uint32_t q = 0; q < 32; ++q) c->last_counts[q] = 0;
  FEI_TRY(c->prog.ensure(prog_len + 16));
  FEI_TRY(c->hits.ensure((n ? n : 1) * sizeof(uint32_t)));
  FEI_TRY(c->work_counter.ensure((8 + kMaxChunks) * sizeof(unsigned long long)));
  FEI_TRY(ensure_side(c));
  FEI_CUDA(cudaEventRecord(c->ev[0], s));
  FEI_CUDA(cudaMemcpyAsync(c->prog.p, prog, prog_len, cudaMemcpyHostToDevice, s));
  FEI_CUDA(cudaMemsetAsync(c->work_counter.p, 0, (8 + kMaxChunks) * sizeof(unsigned long long), s));
  bool need_head = h.head_mask != 0;
  bool need_body = h.off_body_dfa != 0 && h.body_mask != 0;
  if ((h.off_name_dfa[0] || h.off_name_dfa[1] || h.off_name_dfa[2]) && !c->name.p) {
    set_error("program reads filename / id / hostname but the corpus was packed without names"); return FEI_E_STATE;
  }
  const uint32_t nq = h.n_queries;
  const uint64_t nblocks = (n + kCompactRecs - 1) / kCompactRecs;
  if (compact_mode == kCompactLists) {
    FEI_TRY(c->compact.blk_counts.ensure((nblocks ? nblocks : 1) * nq * sizeof(uint32_t)));
    FEI_TRY(c->compact.blk_offsets.ensure((nblocks ? nblocks : 1) * nq * sizeof(uint64_t)));
    FEI_TRY(c->compact.totals.ensure(32 * sizeof(uint64_t)));
    FEI_TRY(c->hit_lists.ensure((n ? n : 1) * nq * sizeof(uint64_t)));
    c->hit_list_stride = n ? n : 1;
    FEI_CUDA(cudaMemsetAsync(c->compact.totals.p, 0, 32 * sizeof(uint64_t), s));
  }
  FEI_CUDA(cudaEventRecord(c->ev[1], s));
  uint32_t launches = 0;
  if (n && need_head) {
    HeadArgs a{c->prog.as<uint8_t>(), c->hdr.as<uint8_t>(), c->hdr_off.as<uint64_t>(), c->name.as<uint8_t>(), c->name_off.as<uint64_t>(),
               c->name_spans.as<uint16_t>(), c->wall.as<int64_t>(), c->flags8.as<uint64_t>(), c->fsb.as<uint32_t>(), n, c->hits.as<uint32_t>(),
               c->hdir.as<uint2>(), c->hdir_off.as<uint64_t>(), c->key_lut.as<uint32_t>(), false,
               c->slot_col.as<int8_t>(), c->col_len.as<uint16_t>(), c->col_planes.as<uint8_t>(), c->ts.as<int64_t>(), {}};
    {
      const fei_prog_cond* cds = reinterpret_cast<const fei_prog_cond*>(prog + h.off_conds);
      for (uint32_t k = 0; k < h.n_conds; ++k)
        if (cds[k].kind == FEI_C_RECBITS) {
          const uint32_t x = cds[k].ref;
          if (x >= FEI_MAX_AUX || !c->aux[x].p || c->aux_n[x] != n) { set_error("program reads aux column %u, which is not set for this corpus state (fei_corpus_set_aux)", x); return FEI_E_STATE; }
        }
      for (int x = 0; x < FEI_MAX_AUX; ++x) a.aux[x] = c->aux[x].as<uint8_t>();
    }
    if (h.n_slots) {                                           // which of the program's fields does each distinct header key of the corpus name?
      FEI_TRY(c->key_lut.ensure(kKeySlots * sizeof(uint32_t)));
      a.key_lut = c->key_lut.as<uint32_t>();
      k_key_lut<<<kKeySlots / 128, 128, 0, s>>>(c->prog.as<uint8_t>(), c->hdr.as<uint8_t>(), c->key_tag.as<unsigned long long>(),
                                                c->key_rep.as<unsigned long long>(), c->key_len.as<uint32_t>(), c->key_lut.as<uint32_t>());
      FEI_TRY(c->slot_col.ensure(FEI_MAX_SLOTS));
      FEI_TRY(c->kid_col.ensure(kKeySlots));
      a.slot_col = c->slot_col.as<int8_t>();
      k_slot_cols<<<1, 32, 0, s>>>(c->prog.as<uint8_t>(), c->key_lut.as<uint32_t>(), c->kid_col.as<int8_t>(), c->n_cols, c->has_text_records ? 1u : 0u, c->slot_col.as<int8_t>());
      launches += 2;
    }
    // selective meta predicates first: stream the meta columns, collect survivors
    FEI_TRY(c->survivors.ensure((n + 32) * sizeof(Survivor)));
    unsigned int* d_count = reinterpret_cast<unsigned int*>(c->work_counter.as<unsigned long long>() + 2);
    const unsigned meta_grid = (unsigned)((n + 256 * kMetaPer - 1) / (256 * kMetaPer));
    // One fused kernel when no meta predicate can thin out the records that need header fields (then every one of them is
    // finished where it was read, no work list); otherwise the meta pass collects the survivors and k_head_parse runs them dense.
    bool fuse = !(getenv("FEI_HEAD_FUSE") && getenv("FEI_HEAD_FUSE")[0] == '0');
    {
      const fei_prog_cond* cds = reinterpret_cast<const fei_prog_cond*>(prog + h.off_conds);
      const fei_prog_query* qs = reinterpret_cast<const fei_prog_query*>(prog + h.off_queries);
      for (uint32_t q = 0; q < h.n_queries && fuse; ++q) {
        if (!((h.slot_mask | h.name_mask) >> q & 1u)) continue;
        for (uint32_t k = qs[q].cond_begin; k < qs[q].cond_end; ++k) {
          const uint8_t kind = cds[k].kind;
          if (kind == FEI_C_SLOT && cds[k].if_missing == 2) { ++k; continue; }      // the fallback field is decided with the header
          if (kind == FEI_C_FLAGS || kind == FEI_C_DATE_CMP || kind == FEI_C_FOLDER_SET || kind == FEI_C_STATUS_SET || kind == FEI_C_RECBITS || kind == FEI_C_TS_CMP) { fuse = false; break; }
        }
      }
    }
    if (fuse) {
      k_head_meta<true><<<meta_grid, 256, 0, s>>>(a, nullptr, nullptr);
      ++launches;
    } else {
      k_head_meta<false><<<meta_grid, 256, 0, s>>>(a, c->survivors.as<Survivor>(), d_count);
      ++launches;
      if (h.slot_mask | h.name_mask) {                         // somebody may need header text or name fields
        k_head_parse<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a, c->survivors.as<Survivor>(), d_count);
        ++launches;
      }
    }
  }
  FEI_CUDA(cudaEventRecord(c->ev[2], s));

  // ---- body pass, chunk by chunk
  fei_prog_dfa d; memset(&d, 0, sizeof(d));
  size_t smem = 0;
  int acc_mode = 0; bool direct = false, sticky_kernel = false, gather = false;
  if (n && need_body) {
    memcpy(&d, prog + h.off_body_dfa, sizeof(d));
    smem = d.table_bytes;
    if (smem > 220 * 1024) { set_error("content automaton needs %zu bytes of shared memory (limit 220 KiB)", smem); return FEI_E_UNSUPPORTED; }
    acc_mode = d.sticky ? 3 : d.n_acc <= 32 ? 1 : d.n_acc <= 64 ? 2 : 0;
    direct = d.n_cols == 256;
    sticky_kernel = direct && acc_mode == 3 && (uint64_t)d.n_states * d.row_stride * 2 + kStickyAddrSlack <= kStickyAddrLimit;
    gather = sticky_kernel && need_head && n >= 65536;         // few survivors of the header pass: one thread per record (device-side choice)
  } else if (n && !need_head) {
    // no condition reads the corpus at all (constant queries): every record gets the constant verdict
    // (program.py folds constants into head conditions, so this only happens for empty condition lists)
    uint32_t all_q = nq >= 32 ? 0xFFFFFFFFu : ((1u << nq) - 1u);
    k_fill32<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(c->hits.as<uint32_t>(), n, all_q);
    ++launches;
  }
  const uint64_t n_windows = (n + kWindow - 1) / kWindow;
  const bool side_work = (n && compact_mode != kCompactNone) || hook;
  BodyArgs a{c->prog.as<uint8_t>(), c->tiles.as<uint8_t>(), c->grp_base.as<uint64_t>(), c->grp_rec.as<uint32_t>(), c->grp_len.as<uint32_t>(),
             c->n_groups, c->hits.as<uint32_t>(), need_head ? 1 : 0, c->work_counter.as<unsigned long long>(), 0ull, 0ull, nullptr, nullptr};
  const unsigned grid = (unsigned)cx.sm_count;
  // One launch, logical chunks: with side work to overlap, the scan kernel is launched ONCE over all groups and publishes finished
  // windows (win_done); the side stream gates each chunk's compaction / exchange on them with k_wait_windows.  Cutting the scan into
  // several LAUNCHES instead (FEI_SCAN_CHUNK_LAUNCHES=1) costs ~0.2 ms of persistent-kernel tail per launch (measured on 10 M entries:
  // 14.3 ms in one launch, 15.8 ms in eight).
  const bool env_launches = getenv("FEI_SCAN_CHUNK_LAUNCHES") && getenv("FEI_SCAN_CHUNK_LAUNCHES")[0] == '1';
  const bool chunkable = n && need_body && !gather && side_work;
  const bool watermark = chunkable && !env_launches;
  ChunkPlan plan;
  plan.n = force_chunks ? force_chunks : chunk_count(n_windows, chunkable, watermark);
  if (plan.n > kMaxChunks) plan.n = kMaxChunks;
  if (plan.n < 1) plan.n = 1;
  plan_chunks(n, plan.n, plan.rec);
  for (uint32_t k = 0; k <= plan.n; ++k) plan.g[k] = (plan.rec[k] + kWindow - 1) / kWindow * (kWindow / 32);
  plan.g[plan.n] = c->n_groups;
  auto launch_body_range = [&](uint64_t g0, uint64_t g1, uint32_t slot) -> int {
    a.g_begin = g0; a.n_groups = g1; a.next = a.counter + 8 + slot;
    int rc = FEI_OK;
    if (sticky_kernel) {
      const size_t smem_sticky = ((smem + 127) & ~(size_t)127) + kStickyRingBytes;
      if (a.push_n) {
        FEI_CUDA(cudaFuncSetAttribute(k_body_sticky<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sticky));
        k_body_sticky<true><<<grid, kBodyThreads, smem_sticky, s>>>(a);
      } else {
        FEI_CUDA(cudaFuncSetAttribute(k_body_sticky<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sticky));
        k_body_sticky<false><<<grid, kBodyThreads, smem_sticky, s>>>(a);
      }
    } else if (direct) rc = acc_mode == 3 ? launch_body<true, 3>(a, grid, smem, s) : acc_mode == 1 ? launch_body<true, 1>(a, grid, smem, s) : acc_mode == 2 ? launch_body<true, 2>(a, grid, smem, s) : launch_body<true, 0>(a, grid, smem, s);
    else rc = acc_mode == 3 ? launch_body<false, 3>(a, grid, smem, s) : acc_mode == 1 ? launch_body<false, 1>(a, grid, smem, s) : acc_mode == 2 ? launch_body<false, 2>(a, grid, smem, s) : launch_body<false, 0>(a, grid, smem, s);
    FEI_TRY(rc);
    ++launches;
    return FEI_OK;
  };
  auto side_chunk = [&](uint32_t k) -> int {                    // compaction + hook of chunk k, queued on the side stream
    if (compact_mode == kCompactLists && plan.rec[k + 1] > plan.rec[k]) {
      const uint64_t b0 = plan.rec[k] / kCompactRecs, b1 = (plan.rec[k + 1] + kCompactRecs - 1) / kCompactRecs;   // chunk bounds are multiples of kWindow (= 2 blocks)
      k_count<<<(unsigned)(b1 - b0), kCompactBlock, 0, c->side>>>(c->hits.as<uint32_t>(), n, nq, b0, c->compact.blk_counts.as<uint32_t>());
      k_scan_blocks<<<nq, 256, 0, c->side>>>(c->compact.blk_counts.as<uint32_t>(), b0, b1 - b0, nq, c->compact.blk_offsets.as<uint64_t>(), c->compact.totals.as<uint64_t>());
      k_emit<<<(unsigned)(b1 - b0), kCompactBlock, 0, c->side>>>(c->hits.as<uint32_t>(), n, nq, c->compact.blk_offsets.as<uint64_t>(), b0, c->global_base,
                                                               c->hit_list_stride, c->hit_lists.as<uint64_t>());
      launches += 3;
    }
    if (hook) FEI_TRY(hook->on_chunk(k, plan.n, plan.rec[k], plan.rec[k + 1], c->side));
    return FEI_OK;
  };
  if (n && need_body && gather) {
    a.gather_max = n / kGatherDiv;
    FEI_TRY(c->live_list.ensure((a.gather_max + 1) * sizeof(uint32_t)));
    k_live_list<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(c->hits.as<uint32_t>(), n, c->live_list.as<uint32_t>(), a.counter + 4, a.gather_max);
    FEI_CUDA(cudaFuncSetAttribute(k_body_gather, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    a.next = a.counter + 8;
    k_body_gather<<<grid, kBodyThreads, smem, s>>>(a, c->live_list.as<uint32_t>(), c->rec_pos.as<uint32_t>());
    launches += 2;
  }
  const bool push = watermark && hook && hook->push_peers && hook->push_n;
  if (watermark && (plan.n > 1 || push)) {
    if (push) { a.push_peers = hook->push_peers; a.push_n = hook->push_n; a.push_off = hook->push_off; a.n_records = n; hook->pushed = true; }
    FEI_TRY(c->win_done.ensure((n_windows + 1) * sizeof(unsigned int)));
    FEI_CUDA(cudaMemsetAsync(c->win_done.p, 0, (n_windows + 1) * sizeof(unsigned int), s));
    a.win_done = c->win_done.as<unsigned int>();
    FEI_CUDA(cudaEventRecord(c->ev_chunk[0], s));              // head pass done, counters zeroed: the side stream may start polling
    FEI_CUDA(cudaStreamWaitEvent(c->side, c->ev_chunk[0], 0));
    FEI_TRY(launch_body_range(0, c->n_groups, 0));
    for (uint32_t k = 0; k < plan.n; ++k) {
      const uint64_t w0 = plan.rec[k] / kWindow, w1 = (plan.rec[k + 1] + kWindow - 1) / kWindow;
      if (w1 > w0) { k_wait_windows<<<1, 32, 0, c->side>>>(c->win_done.as<unsigned int>(), w0, w1, a.counter + 5); ++launches; }
      FEI_TRY(side_chunk(k));
    }
  } else {
    for (uint32_t k = 0; k < plan.n; ++k) {
      if (n && need_body && plan.g[k + 1] > plan.g[k]) FEI_TRY(launch_body_range(plan.g[k], plan.g[k + 1], k));
      if (!side_work) continue;
      FEI_CUDA(cudaEventRecord(c->ev_chunk[k], s));
      FEI_CUDA(cudaStreamWaitEvent(c->side, c->ev_chunk[k], 0));
      FEI_TRY(side_chunk(k));
    }
  }
  FEI_CUDA(cudaEventRecord(c->ev[3], s));
  if (side_work) {
    if (hook) FEI_TRY(hook->on_done(c->side));
    FEI_CUDA(cudaEventRecord(c->ev_side, c->side));
    FEI_CUDA(cudaStreamWaitEvent(s, c->ev_side, 0));
  }
  if (compact_mode == kCompactLists)
    FEI_CUDA(cudaMemcpyAsync(c->last_counts, c->compact.totals.p, nq * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaEventRecord(c->ev[4], s));
  FEI_CUDA(cudaGetLastError());
  c->timing.kernel_launches = launches;
  return FEI_OK;
}

int finish_timing(fei_corpus* c, bool compacted) {
  cudaStream_t s = ctx().stream;
  FEI_CUDA(cudaEventRecord(c->ev[5], s));
  FEI_CUDA(cudaStreamSynchronize(s));
  float t;
  FEI_CUDA(cudaEventElapsedTime(&t, c->ev[0], c->ev[1])); c->timing.h2d_ms = t;
  FEI_CUDA(cudaEventElapsedTime(&t, c->ev[1], c->ev[2])); c->timing.head_ms = t;
  FEI_CUDA(cudaEventElapsedTime(&t, c->ev[2], c->ev[3])); c->timing.body_ms = t;
  if (compacted) { FEI_CUDA(cudaEventElapsedTime(&t, c->ev[3], c->ev[4])); c->timing.compact_ms = t; }   // what is left after the last chunk's scan
  FEI_CUDA(cudaEventElapsedTime(&t, c->ev[4], c->ev[5])); c->timing.d2h_ms = t;
  FEI_CUDA(cudaEventElapsedTime(&t, c->ev[0], c->ev[5])); c->timing.total_ms = t;
  unsigned long long cnt[6] = {0, 0, 0, 0, 0, 0};
  FEI_CUDA(cudaMemcpy(cnt, c->work_counter.as<unsigned long long>(), sizeof(cnt), cudaMemcpyDeviceToHost));
  c->timing.body_bytes_touched = cnt[1];
  c->timing.body_bytes_read = cnt[3];
  if (cnt[5]) { set_error("pipelined scan: the side stream gave up waiting for the scan kernel's finished windows"); return FEI_E_CUDA; }
  return FEI_OK;
}

// Order-preserving compaction of a mask array into per-query lists of global indices (one shot, any stream; used for the
// rank segments of an all-gathered mask array).  counts_out[q] = hits of query q; when `lists` is given,
// lists[q * stride + k] = k-th hit (stride = max count).
int compact_masks(const uint32_t* masks, uint64_t n, uint32_t nq, uint64_t global_base, CompactScratch& sc,
                  uint64_t* counts_out, DevBuf* lists, uint64_t* stride_out, uint32_t* launches, cudaStream_t s) {
  uint64_t nblocks = (n + kCompactRecs - 1) / kCompactRecs;
  for (uint32_t q = 0; q < nq; ++q) counts_out[q] = 0;
  if (stride_out) *stride_out = 1;
  if (n == 0) return FEI_OK;
  FEI_TRY(sc.blk_counts.ensure(nblocks * nq * sizeof(uint32_t)));
  FEI_TRY(sc.blk_offsets.ensure(nblocks * nq * sizeof(uint64_t)));
  FEI_TRY(sc.totals.ensure(32 * sizeof(uint64_t)));
  FEI_CUDA(cudaMemsetAsync(sc.totals.p, 0, 32 * sizeof(uint64_t), s));
  k_count<<<(unsigned)nblocks, kCompactBlock, 0, s>>>(masks, n, nq, 0, sc.blk_counts.as<uint32_t>());
  k_scan_blocks<<<nq, 256, 0, s>>>(sc.blk_counts.as<uint32_t>(), 0, nblocks, nq, sc.blk_offsets.as<uint64_t>(), sc.totals.as<uint64_t>());
  if (launches) *launches += 2;
  FEI_CUDA(cudaMemcpyAsync(counts_out, sc.totals.p, nq * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaStreamSynchronize(s));
  if (lists) {
    uint64_t stride = 1;
    for (uint32_t q = 0; q < nq; ++q) if (counts_out[q] > stride) stride = counts_out[q];
    if (stride_out) *stride_out = stride;
    FEI_TRY(lists->ensure(stride * nq * sizeof(uint64_t)));
    k_emit<<<(unsigned)nblocks, kCompactBlock, 0, s>>>(masks, n, nq, sc.blk_offsets.as<uint64_t>(), 0, global_base, stride, lists->as<uint64_t>());
    if (launches) *launches += 1;
  }
  FEI_CUDA(cudaGetLastError());
  return FEI_OK;
}

// Global ordered lists from an all-gathered, rank-major mask array: segment r = masks[r * seg_stride .. + seg_n[r]), its
// record 0 is global index seg_base[r].  lists[q * stride + k]; totals_out[q] (host) after a final sync.
int compact_segments(const uint32_t* masks, uint64_t seg_stride, const uint64_t* seg_n, const uint64_t* seg_base, uint32_t n_seg, uint32_t nq,
                     CompactScratch& sc, uint64_t stride, uint64_t* lists, uint64_t* totals_out, cudaStream_t s) {
  uint64_t n_max = 0;
  for (uint32_t r = 0; r < n_seg; ++r) if (seg_n[r] > n_max) n_max = seg_n[r];
  const uint64_t nb_max = (n_max + kCompactRecs - 1) / kCompactRecs;
  FEI_TRY(sc.blk_counts.ensure((nb_max ? nb_max : 1) * nq * sizeof(uint32_t)));
  FEI_TRY(sc.blk_offsets.ensure((nb_max ? nb_max : 1) * nq * sizeof(uint64_t)));
  FEI_TRY(sc.totals.ensure(32 * sizeof(uint64_t)));
  FEI_CUDA(cudaMemsetAsync(sc.totals.p, 0, 32 * sizeof(uint64_t), s));
  for (uint32_t r = 0; r < n_seg; ++r) {
    const uint64_t n = seg_n[r], nb = (n + kCompactRecs - 1) / kCompactRecs;
    if (!n) continue;
    const uint32_t* m = masks + (size_t)r * seg_stride;
    k_count<<<(unsigned)nb, kCompactBlock, 0, s>>>(m, n, nq, 0, sc.blk_counts.as<uint32_t>());
    k_scan_blocks<<<nq, 256, 0, s>>>(sc.blk_counts.as<uint32_t>(), 0, nb, nq, sc.blk_offsets.as<uint64_t>(), sc.totals.as<uint64_t>());   // the carry runs on across segments
    k_emit<<<(unsigned)nb, kCompactBlock, 0, s>>>(m, n, nq, sc.blk_offsets.as<uint64_t>(), 0, seg_base[r], stride, lists);
  }
  if (totals_out) {
    FEI_CUDA(cudaMemcpyAsync(totals_out, sc.totals.p, nq * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    FEI_CUDA(cudaStreamSynchronize(s));
  }
  FEI_CUDA(cudaGetLastError());
  return FEI_OK;
}

// (A, S) checksums of `count` indices at `list` (device memory); see k_list_checksum
int list_checksum(const uint64_t* list, uint64_t count, DevBuf& tmp, uint64_t* a_out, uint64_t* s_out, cudaStream_t s) {
  FEI_TRY(tmp.ensure(16));
  FEI_CUDA(cudaMemsetAsync(tmp.p, 0, 16, s));
  if (count) k_list_checksum<<<(unsigned)std::min<uint64_t>((count + 255) / 256, 4096), 256, 0, s>>>(list, count, tmp.as<unsigned long long>());
  unsigned long long r[2];
  FEI_CUDA(cudaMemcpyAsync(r, tmp.p, 16, cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaStreamSynchronize(s));
  *a_out = r[0]; *s_out = r[1];
  return FEI_OK;
}

}  // namespace fei

using namespace fei;

extern "C" int fei_scan_masks(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint32_t* masks) {
  if (!c) { set_error("null corpus"); return FEI_E_BADARG; }
  std::lock_guard<std::mutex> lock(c->mu);
  FEI_TRY(run_scan(c, prog, prog_len, kCompactNone, nullptr, 0));
  if (masks && c->n) FEI_CUDA(cudaMemcpyAsync(masks, c->hits.p, c->n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx().stream));
  return finish_timing(c, false);
}

extern "C" int fei_scan_count(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint64_t* nhits) {
  if (!c) { set_error("null corpus"); return FEI_E_BADARG; }
  std::lock_guard<std::mutex> lock(c->mu);
  FEI_TRY(run_scan(c, prog, prog_len, kCompactLists, nullptr, 0));     // lists stay on the device (fei_comm_allgather_hits, fei_scan_list_checksum)
  FEI_TRY(finish_timing(c, true));
  if (nhits) for (uint32_t q = 0; q < c->last_nq; ++q) nhits[q] = c->last_counts[q];
  return FEI_OK;
}

extern "C" int fei_scan_hits(fei_corpus* c, const uint8_t* prog, uint64_t prog_len,
                             uint64_t* const* hits, const uint64_t* cap, uint64_t* nhits) {
  if (!c) { set_error("null corpus"); return FEI_E_BADARG; }
  std::lock_guard<std::mutex> lock(c->mu);
  if (!hits || !cap || !nhits) { set_error("null argument"); return FEI_E_BADARG; }
  FEI_TRY(run_scan(c, prog, prog_len, kCompactLists, nullptr, 0));
  cudaStream_t s = ctx().stream;
  FEI_CUDA(cudaStreamSynchronize(s));                                  // the counts decide how much of every list is copied
  bool truncated = false;
  for (uint32_t q = 0; q < c->last_nq; ++q) {
    nhits[q] = c->last_counts[q];
    uint64_t take = nhits[q] < cap[q] ? nhits[q] : cap[q];
    if (take < nhits[q]) truncated = true;
    if (take && hits[q]) FEI_CUDA(cudaMemcpyAsync(hits[q], c->hit_lists.as<uint64_t>() + q * c->hit_list_stride, take * 8, cudaMemcpyDeviceToHost, s));
  }
  FEI_TRY(finish_timing(c, true));
  if (truncated) { set_error("hit buffer too small for at least one query (see nhits)"); return FEI_E_CAPACITY; }
  return FEI_OK;
}

/* copies (a prefix of) the ordered lists the last fei_scan_count left on the device: no second scan */
extern "C" int fei_scan_fetch_hits(fei_corpus* c, uint32_t nq, uint64_t* const* hits, const uint64_t* cap) {
  if (!c || !hits || !cap) { set_error("null argument"); return FEI_E_BADARG; }
  std::lock_guard<std::mutex> lock(c->mu);
  if (nq == 0 || nq != c->last_nq || !c->hit_lists.p) { set_error("no matching scan result with lists on this corpus"); return FEI_E_STATE; }
  cudaStream_t s = ctx().stream;
  bool truncated = false;
  for (uint32_t q = 0; q < nq; ++q) {
    uint64_t take = c->last_counts[q] < cap[q] ? c->last_counts[q] : cap[q];
    if (take < c->last_counts[q]) truncated = true;
    if (take && hits[q]) FEI_CUDA(cudaMemcpyAsync(hits[q], c->hit_lists.as<uint64_t>() + q * c->hit_list_stride, take * 8, cudaMemcpyDeviceToHost, s));
  }
  FEI_CUDA(cudaStreamSynchronize(s));
  if (truncated) { set_error("hit buffer too small for at least one query"); return FEI_E_CAPACITY; }
  return FEI_OK;
}

/* (A, S) checksums of the ordered hit lists the last fei_scan_count / fei_scan_hits left on the device */
extern "C" int fei_scan_list_checksum(fei_corpus* c, uint32_t nq, uint64_t* a_out, uint64_t* s_out) {
  if (!c || !a_out || !s_out) { set_error("null argument"); return FEI_E_BADARG; }
  std::lock_guard<std::mutex> lock(c->mu);
  if (nq == 0 || nq != c->last_nq || !c->hit_lists.p) { set_error("no matching scan result with lists on this corpus"); return FEI_E_STATE; }
  for (uint32_t q = 0; q < nq; ++q)
    FEI_TRY(list_checksum(c->hit_lists.as<uint64_t>() + q * c->hit_list_stride, c->last_counts[q], c->scan_tmp, a_out + q, s_out + q, ctx().stream));
  return FEI_OK;
}

extern "C" int fei_scan_last_timing(const fei_corpus* c, fei_scan_timing* out) {
  if (!c || !out) { set_error("null argument"); return FEI_E_BADARG; }
  *out = c->timing;
  return FEI_OK;
}

// ---------------------------------------------------------------- token histogram of a header field ("next" row 4)
// MemdirFolderManager.get_folder_stats (memdir_tools/folders.py:286-292):
//     if "Tags" in memory["headers"]: for tag in [t.strip() for t in headers["Tags"].split(",")]: stats["tags"][tag] += 1
// One thread per selected record walks the record's header directory for the field (exact key: slot 0 of the program,
// last line wins), splits the value at `sep`, strips every piece with Python's whitespace set and counts it in a device
// hash table (64-bit hash, representative spelling = smallest header offset, every piece verified against it in a
// second pass).  `first` orders the tokens the way the reference's dict does (first record, then position in the value).
namespace fei {
constexpr uint32_t kTokSlots = 1u << 16;
struct TokTable { unsigned long long* tag; unsigned long long* rep; unsigned long long* first; uint32_t* len; uint32_t* count; uint32_t* flag; };

__device__ __forceinline__ unsigned long long tok_hash(const uint8_t* p, uint32_t n) {
  unsigned long long h = 0x9E3779B97F4A7C15ull;
  for (uint32_t i = 0; i < n; ++i) { h ^= p[i]; h *= 0x100000001b3ull; }
  h ^= h >> 31; h *= 0xD6E8FEB86659FD93ull; h ^= h >> 32;
  return h | 1ull;
}

template <int kPass>
__global__ void __launch_bounds__(256) k_tok_hist(const uint8_t* __restrict__ hdr, const uint64_t* __restrict__ hdr_off,
                                                  const uint2* __restrict__ hdir, const uint64_t* __restrict__ hdir_off,
                                                  const uint32_t* __restrict__ key_lut, const uint32_t* __restrict__ alive, uint64_t n,
                                                  uint8_t sep, TokTable t) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n || !(alive[i] & 1u)) return;
  const uint2* ent = hdir + hdir_off[i];
  const uint32_t n_ent = (uint32_t)(hdir_off[i + 1] - hdir_off[i]);
  if (n_ent == 1 && ent[0].x == 0xFFFFFFFFu) { atomicOr(t.flag, 4u); return; }      // header parsed from its text: not handled here
  int last = -1;
  for (uint32_t j = 0; j < n_ent; ++j) if (key_lut[ent[j].x & 0xFFFFu] & 1u) last = (int)j;      // slot 0, repeated key: last value
  if (last < 0) return;
  const uint8_t* v = hdr + hdr_off[i] + ent[last].y;
  const uint32_t vlen = ent[last].x >> 16;
  uint32_t pos = 0, idx = 0;
  for (;;) {                                                     // str.split(sep): k separators -> k + 1 pieces, empty ones included
    uint32_t end = pos;
    while (end < vlen && v[end] != sep) ++end;
    const uint8_t* a = v + pos; const uint8_t* b = v + end;
    strip_span(a, b);
    const uint32_t len = (uint32_t)(b - a);
    const unsigned long long h = tok_hash(a, len);
    uint32_t s = (uint32_t)(h >> 20) & (kTokSlots - 1);
    bool placed = false;
    for (uint32_t probe = 0; probe < kTokSlots / 2 && !placed; ++probe, s = (s + 1) & (kTokSlots - 1)) {
      unsigned long long cur = t.tag[s];
      if (cur == 0 && kPass == 0) cur = atomicCAS(t.tag + s, 0ull, h), cur = cur == 0 ? h : cur;
      if (cur == h) {
        placed = true;
        if (kPass == 0) {
          atomicAdd(t.count + s, 1u);
          atomicMin(t.rep + s, (unsigned long long)(a - hdr));
          atomicMin(t.first + s, (unsigned long long)i << 20 | (idx < 0xFFFFFu ? idx : 0xFFFFFu));
          t.len[s] = len;
        } else {
          bool same = t.len[s] == len;
          const uint8_t* r = hdr + t.rep[s];
          for (uint32_t k = 0; same && k < len; ++k) same = r[k] == a[k];
          if (!same) atomicOr(t.flag, 2u);                       // two different pieces with one 64-bit hash
        }
      } else if (cur == 0) break;                                // pass 1 only: cannot happen after pass 0
    }
    if (!placed) atomicOr(t.flag, 1u);                           // table over-full
    ++idx;
    if (end >= vlen) break;
    pos = end + 1;
  }
}

__global__ void k_tok_pack(const uint8_t* __restrict__ hdr, const unsigned long long* __restrict__ rep, const uint32_t* __restrict__ len,
                           const uint32_t* __restrict__ slots, const uint64_t* __restrict__ out_off, uint32_t n_tok, uint8_t* __restrict__ out) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_tok) return;
  const uint32_t s = slots[k];
  const uint8_t* p = hdr + rep[s];
  for (uint32_t b = 0; b < len[s]; ++b) out[out_off[k] + b] = p[b];
}
}  // namespace fei

extern "C" int fei_corpus_token_histogram(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint8_t sep,
                                          uint8_t* tok_blob, uint64_t blob_cap, uint64_t* tok_off, uint64_t* tok_count, uint64_t* tok_first,
                                          uint64_t cap, uint64_t* n_tokens) {
  if (!c || !n_tokens || !tok_off) { set_error("null argument"); return FEI_E_BADARG; }
  std::lock_guard<std::mutex> lock(c->mu);
  *n_tokens = 0; tok_off[0] = 0;
  FEI_TRY(run_scan(c, prog, prog_len, kCompactNone, nullptr, 0));
  fei_prog_hdr h; memcpy(&h, prog, sizeof(h));
  if (h.n_queries != 1 || h.n_slots < 1) { set_error("token histogram wants one query whose first header field names the column"); return FEI_E_BADARG; }
  if (c->n == 0) return finish_timing(c, false);
  if (c->has_text_records || !c->hdir.p) { set_error("corpus holds records whose header is parsed from its text; the token histogram does not handle them"); return FEI_E_UNSUPPORTED; }
  cudaStream_t s = ctx().stream;
  DevBuf& tb = c->scan_tmp;
  const size_t bytes = (size_t)kTokSlots * (8 + 8 + 8 + 4 + 4) + 16;
  FEI_TRY(tb.ensure(bytes));
  uint8_t* base = tb.as<uint8_t>();
  TokTable t{reinterpret_cast<unsigned long long*>(base), reinterpret_cast<unsigned long long*>(base) + kTokSlots, reinterpret_cast<unsigned long long*>(base) + 2 * kTokSlots,
             reinterpret_cast<uint32_t*>(base + (size_t)kTokSlots * 24), reinterpret_cast<uint32_t*>(base + (size_t)kTokSlots * 28), reinterpret_cast<uint32_t*>(base + (size_t)kTokSlots * 32)};
  FEI_CUDA(cudaMemsetAsync(base, 0, bytes, s));
  FEI_CUDA(cudaMemsetAsync(t.rep, 0xFF, (size_t)kTokSlots * 16, s));           // rep and first: ~0 so that atomicMin works
  const unsigned grid = (unsigned)((c->n + 255) / 256);
  k_tok_hist<0><<<grid, 256, 0, s>>>(c->hdr.as<uint8_t>(), c->hdr_off.as<uint64_t>(), c->hdir.as<uint2>(), c->hdir_off.as<uint64_t>(), c->key_lut.as<uint32_t>(),
                                     c->hits.as<uint32_t>(), c->n, sep, t);
  k_tok_hist<1><<<grid, 256, 0, s>>>(c->hdr.as<uint8_t>(), c->hdr_off.as<uint64_t>(), c->hdir.as<uint2>(), c->hdir_off.as<uint64_t>(), c->key_lut.as<uint32_t>(),
                                     c->hits.as<uint32_t>(), c->n, sep, t);
  std::vector<unsigned long long> tag(kTokSlots), first(kTokSlots);
  std::vector<uint32_t> len(kTokSlots), count(kTokSlots);
  uint32_t flag = 0;
  FEI_CUDA(cudaMemcpyAsync(tag.data(), t.tag, kTokSlots * 8, cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaMemcpyAsync(first.data(), t.first, kTokSlots * 8, cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaMemcpyAsync(len.data(), t.len, kTokSlots * 4, cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaMemcpyAsync(count.data(), t.count, kTokSlots * 4, cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaMemcpyAsync(&flag, t.flag, 4, cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaStreamSynchronize(s));
  FEI_CUDA(cudaGetLastError());
  if (flag & 4u) { set_error("a selected record's header is parsed from its text; the token histogram does not handle it"); return FEI_E_UNSUPPORTED; }
  if (flag) { set_error(flag & 1u ? "more than 32768 distinct tokens" : "64-bit hash collision between two tokens"); return FEI_E_UNSUPPORTED; }
  std::vector<uint32_t> slots;
  for (uint32_t k = 0; k < kTokSlots; ++k) if (tag[k]) slots.push_back(k);
  std::sort(slots.begin(), slots.end(), [&](uint32_t a, uint32_t b) { return first[a] < first[b]; });   // the order a dict filled record by record has
  if (slots.size() > cap) { set_error("token table too small: need %zu entries", slots.size()); return FEI_E_CAPACITY; }
  std::vector<uint64_t> off(slots.size() + 1, 0);
  for (size_t k = 0; k < slots.size(); ++k) off[k + 1] = off[k] + len[slots[k]];
  if (off.back() > blob_cap) { set_error("token buffer too small: need %llu bytes", (unsigned long long)off.back()); return FEI_E_CAPACITY; }
  if (!slots.empty()) {
    DevBuf d_slots, d_off, d_out;
    FEI_TRY(d_slots.ensure(slots.size() * 4)); FEI_TRY(d_off.ensure(off.size() * 8)); FEI_TRY(d_out.ensure(off.back() + 16));
    FEI_CUDA(cudaMemcpyAsync(d_slots.p, slots.data(), slots.size() * 4, cudaMemcpyHostToDevice, s));
    FEI_CUDA(cudaMemcpyAsync(d_off.p, off.data(), off.size() * 8, cudaMemcpyHostToDevice, s));
    k_tok_pack<<<(unsigned)((slots.size() + 127) / 128), 128, 0, s>>>(c->hdr.as<uint8_t>(), t.rep, t.len, d_slots.as<uint32_t>(), d_off.as<uint64_t>(), (uint32_t)slots.size(), d_out.as<uint8_t>());
    if (off.back() && tok_blob) FEI_CUDA(cudaMemcpyAsync(tok_blob, d_out.p, off.back(), cudaMemcpyDeviceToHost, s));
    FEI_CUDA(cudaStreamSynchronize(s));
    FEI_CUDA(cudaGetLastError());
  }
  for (size_t k = 0; k < slots.size(); ++k) {
    tok_off[k + 1] = off[k + 1];
    if (tok_count) tok_count[k] = count[slots[k]];
    if (tok_first) tok_first[k] = (first[slots[k]] >> 20) + c->global_base;
  }
  *n_tokens = slots.size();
  return finish_timing(c, false);
}


// ---------------------------------------------------------------- header values of one field, record by record
// For conditions only Python can judge value by value (search.py:126-130: Due / Created / Modified / DeletedDate go through
// dateutil.parser.parse per record), the host needs the VALUE the reference would read for every record: slot 0 of the program
// resolved with the reference's dict semantics (mode 0: first key whose lower() equals the field, last line of that exact key;
// mode 1: exact key).  k_slot_spans finds the value's span in the header blob (directory walk, or the text for headers the
// directory cannot address), k_slot_gather packs the values into one blob that goes back to the host.  The sort keys of
// fei_sort_rows (order.cu) read the same spans for a list of records (slot_spans_rows).
namespace fei {
// rows == nullptr: records 0 .. m-1; else records rows[0 .. m).  Out: len_out[i], src_out[i] (offset into the header blob, ~0: absent).
__global__ void __launch_bounds__(256) k_slot_spans(HeadArgs a, const uint64_t* __restrict__ rows, uint64_t m, uint32_t* __restrict__ len_out,
                                                   uint64_t* __restrict__ src_out) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const uint64_t rec = rows ? rows[i] : i;
  const fei_prog_hdr* ph = reinterpret_cast<const fei_prog_hdr*>(a.prog);
  const fei_prog_slot* slots = reinterpret_cast<const fei_prog_slot*>(a.prog + ph->off_slots);
  const uint32_t mode = slots[0].mode;
  const uint64_t hoff = a.hdr_off[rec];
  const uint8_t* h = a.hdr + hoff;
  const uint32_t hlen = (uint32_t)(a.hdr_off[rec + 1] - hoff);
  const uint2* ent = a.hdir + a.hdir_off[rec];
  const uint32_t n_ent = (uint32_t)(a.hdir_off[rec + 1] - a.hdir_off[rec]);
  bool have = false, have_first = false;
  uint32_t voff = 0, vlen = 0;
  if (!(n_ent == 1 && ent[0].x == 0xFFFFFFFFu)) {
    uint32_t first_key = 0;
    for (uint32_t j = 0; j < n_ent; ++j) {
      const uint2 e = ent[j];
      const uint32_t kid = e.x & 0xFFFFu;
      if (!(a.key_lut[kid] & 1u)) continue;
      if (mode == 0) {
        if (!have_first) { have_first = true; first_key = kid; }
        else if (first_key != kid) continue;
      }
      voff = e.y; vlen = e.x >> 16; have = true;
    }
  } else {
    DfaView keyd = dfa_view(a.prog, ph->off_key_dfa);
    const uint8_t* hend = h + hlen;
    const uint8_t* p = h;
    uint32_t first_off = 0, first_len = 0;
    while (p < hend) {
      const uint8_t* eol = p; const uint8_t* colon = nullptr;
      while (eol < hend && *eol != '\n') { if (!colon && *eol == ':') colon = eol; ++eol; }
      if (colon) {
        const uint8_t* ka = p; const uint8_t* kb = colon; strip_span(ka, kb);
        const uint8_t* va = colon + 1; const uint8_t* vb = eol; strip_span(va, vb);
        if (dfa_run(keyd, ka, (uint32_t)(kb - ka)) & 1u) {
          bool take = true;
          if (mode == 0) {
            if (!have_first) { have_first = true; first_off = (uint32_t)(ka - h); first_len = (uint32_t)(kb - ka); }
            else {
              bool same = first_len == (uint32_t)(kb - ka);
              for (uint32_t k = 0; same && k < first_len; ++k) same = h[first_off + k] == ka[k];
              take = same;
            }
          }
          if (take) { voff = (uint32_t)(va - h); vlen = (uint32_t)(vb - va); have = true; }
        }
      }
      p = eol + 1;
    }
  }
  len_out[i] = have ? vlen : 0u;
  src_out[i] = have ? hoff + voff : ~0ull;                       // ~0: the record has no such header
}

__global__ void __launch_bounds__(256) k_slot_gather(const uint8_t* __restrict__ hdr, const uint32_t* __restrict__ len, const uint64_t* __restrict__ src,
                                                    const uint64_t* __restrict__ off, uint64_t n, uint8_t* __restrict__ out, uint8_t* __restrict__ present) {
  const uint64_t rec = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (rec >= n) return;
  const bool have = src[rec] != ~0ull;
  present[rec] = have ? 1 : 0;
  if (!have) return;
  const uint8_t* p = hdr + src[rec];
  uint8_t* d = out + off[rec];
  for (uint32_t k = 0; k < len[rec]; ++k) d[k] = p[k];
}
}  // namespace fei

namespace fei {
int slot_spans_rows(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, const uint64_t* d_rows, uint64_t m, uint32_t* d_len, uint64_t* d_src,
                    cudaStream_t s) {
  FEI_TRY(check_prog(prog, prog_len));
  fei_prog_hdr h; memcpy(&h, prog, sizeof(h));
  if (h.n_slots < 1) { set_error("program has no header field"); return FEI_E_BADARG; }
  if (m == 0) return FEI_OK;
  FEI_TRY(c->prog.ensure(prog_len + 16));
  FEI_CUDA(cudaMemcpyAsync(c->prog.p, prog, prog_len, cudaMemcpyHostToDevice, s));
  FEI_TRY(c->key_lut.ensure(kKeySlots * sizeof(uint32_t)));
  k_key_lut<<<kKeySlots / 128, 128, 0, s>>>(c->prog.as<uint8_t>(), c->hdr.as<uint8_t>(), c->key_tag.as<unsigned long long>(),
                                            c->key_rep.as<unsigned long long>(), c->key_len.as<uint32_t>(), c->key_lut.as<uint32_t>());
  HeadArgs a{c->prog.as<uint8_t>(), c->hdr.as<uint8_t>(), c->hdr_off.as<uint64_t>(), nullptr, nullptr, nullptr, c->wall.as<int64_t>(), c->flags8.as<uint64_t>(),
             c->fsb.as<uint32_t>(), c->n, nullptr, c->hdir.as<uint2>(), c->hdir_off.as<uint64_t>(), c->key_lut.as<uint32_t>(), false, nullptr, nullptr, nullptr, c->ts.as<int64_t>(), {}};
  k_slot_spans<<<(unsigned)((m + 255) / 256), 256, 0, s>>>(a, d_rows, m, d_len, d_src);
  FEI_CUDA(cudaGetLastError());
  return FEI_OK;
}
}  // namespace fei

/* prog: any program whose slot 0 names the field (conditions are ignored).  Out: present[n], off[n+1] (value i =
 * blob[off[i] .. off[i+1]), empty for absent headers).  FEI_E_CAPACITY with the needed size in off[n] when blob_cap is too small. */
extern "C" int fei_corpus_slot_values(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint8_t* present, uint64_t* off,
                                      uint8_t* blob, uint64_t blob_cap) {
  if (!c || !prog || !present || !off) { set_error("null argument"); return FEI_E_BADARG; }
  std::lock_guard<std::mutex> lock(c->mu);
  FEI_TRY(require_ready());
  if (!c->loaded) { set_error("corpus not loaded"); return FEI_E_STATE; }
  const uint64_t n = c->n;
  cudaStream_t s = ctx().stream;
  DevBuf d_len, d_src, d_off, d_present, d_out;
  FEI_TRY(d_len.alloc(n * 4 + 4)); FEI_TRY(d_src.alloc(n * 8 + 8)); FEI_TRY(d_off.alloc((n + 1) * 8)); FEI_TRY(d_present.alloc(n + 1));
  FEI_TRY(slot_spans_rows(c, prog, prog_len, nullptr, n, d_len.as<uint32_t>(), d_src.as<uint64_t>(), s));
  off[0] = 0;
  if (n == 0) return FEI_OK;
  const unsigned grid = (unsigned)((n + 255) / 256);
  FEI_TRY(exclusive_scan_u32_u64(d_len.as<uint32_t>(), n, d_off.as<uint64_t>(), c->scan_tmp, s));
  FEI_CUDA(cudaMemcpyAsync(off, d_off.p, (n + 1) * 8, cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaStreamSynchronize(s));
  FEI_TRY(d_out.alloc(off[n] + 16));
  k_slot_gather<<<grid, 256, 0, s>>>(c->hdr.as<uint8_t>(), d_len.as<uint32_t>(), d_src.as<uint64_t>(), d_off.as<uint64_t>(), n, d_out.as<uint8_t>(), d_present.as<uint8_t>());
  FEI_CUDA(cudaMemcpyAsync(present, d_present.p, n, cudaMemcpyDeviceToHost, s));
  const bool fits = blob && off[n] <= blob_cap;
  if (fits && off[n]) FEI_CUDA(cudaMemcpyAsync(blob, d_out.p, off[n], cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaStreamSynchronize(s));
  FEI_CUDA(cudaGetLastError());
  if (!fits) { set_error("value buffer too small: need %llu bytes", (unsigned long long)off[n]); return FEI_E_CAPACITY; }
  return FEI_OK;
}

/* Aux column k (0 .. FEI_MAX_AUX-1): one verdict byte per record, read by FEI_C_RECBITS conditions of later scans.  n must be the
 * corpus' record count; bytes == NULL drops the column.                                                                         */
extern "C" int fei_corpus_set_aux(fei_corpus* c, uint32_t k, const uint8_t* bytes, uint64_t n) {
  if (!c || k >= FEI_MAX_AUX) { set_error("bad argument"); return FEI_E_BADARG; }
  std::lock_guard<std::mutex> lock(c->mu);
  FEI_TRY(require_ready());
  if (!bytes) { c->aux[k].release(); c->aux_n[k] = 0; return FEI_OK; }
  if (n != c->n) { set_error("aux column has %llu entries, the corpus %llu records", (unsigned long long)n, (unsigned long long)c->n); return FEI_E_BADARG; }
  cudaStream_t s = ctx().stream;
  FEI_TRY(c->aux[k].ensure(n + 16));
  if (n) FEI_CUDA(cudaMemcpyAsync(c->aux[k].p, bytes, n, cudaMemcpyHostToDevice, s));
  FEI_CUDA(cudaStreamSynchronize(s));
  c->aux_n[k] = n;
  return FEI_OK;
}
