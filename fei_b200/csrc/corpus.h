// Device-resident packed Memdir corpus (see DESIGN.md "data layout in HBM").
//
//   headers : canonical blob  hdr[hdr_off[i] .. hdr_off[i+1])           (4% of the bytes)
//   meta    : SoA  ts[n], wall[n], flags8[n], fsb[n]
//   names   : canonical blob (optional)
//   bodies  : warp-transposed, length-sorted, ragged tiles:
//       records are taken in windows of kWindow consecutive records; inside a window they
//       are sorted by body length (16-byte units, descending, stable) and cut into groups
//       of 32.  A group stores unit k of every member that still has a unit k, members in
//       sorted order, as one contiguous row of m_k * 16 bytes, rows back to back:
//           row_k = grp_base[g] + 16 * sum_{j<k} m_j ,   lane l's unit k at row_k + 16*l
//       so a warp reading "unit k of its 32 records" issues ONE contiguous coalesced
//       request of m_k*16 bytes, every lane gets the next 16 bytes of its own record in
//       registers, and (lengths being sorted) lanes finish together.  No padding except the
//       last unit of each record (<= 15 bytes, zero filled).
//       grp_rec[g*32 + l] = record index (kInvalidRec for padding lanes), grp_len[...] = byte length.
#pragma once
#include "common.h"
#include <mutex>

namespace fei {
// Body tiles store every byte b as  b ^ ((b >> 1) & 0x20)  (an involution: bit 5 ^= bit 6).  The scan tables are
// indexed by the stored value (program.py permutes their columns), so nothing changes for the result; what changes
// is which shared-memory bank a byte selects: plain ASCII puts lower-case letters (0x60-0x7F) and space / digits /
// punctuation (0x20-0x3F) on the SAME 16 banks (bank = (row + byte/2) mod 32), so lanes sitting in the same automaton
// state collided whenever one read a letter and another a space; after the swap letters use banks 0-15 and
// space / punctuation banks 16-31 (measured: 2.0 -> see DESIGN.md wavefronts per lookup on single-pattern scans).
#ifdef __CUDACC__
__host__ __device__ __forceinline__ uint32_t tile_byte_perm4(uint32_t w) { return w ^ ((w >> 1) & 0x20202020u); }
#endif
constexpr int kWindow = 4096;
constexpr uint32_t kKeySlots = 4096;       // header-key dictionary slots (hdir.cu); at most half may fill
constexpr uint32_t kMaxCols = 8;           // header value columns kept per corpus
constexpr uint32_t kColUnits = 4;          // 16-byte units per column value (longer values: directory walk)
constexpr uint16_t kColAbsent = 0xFFFF, kColWalk = 0xFFFE;
constexpr uint32_t kInvalidRec = 0xFFFFFFFFu;
#define FEI_MAX_AUX 4
}

namespace fei {
struct CompactScratch { DevBuf blk_counts, blk_offsets, totals; };
}

struct fei_corpus {
  std::mutex mu;                         // one scan / load at a time per handle (callers may be concurrent threads)
  uint64_t n = 0, global_base = 0;
  uint64_t hdr_bytes = 0, body_bytes = 0, name_bytes = 0, tile_bytes = 0;
  uint64_t n_groups = 0;
  bool loaded = false;
  fei::DevBuf hdr, hdr_off, name, name_off, name_spans, ts, wall, flags8, fsb;
  fei::DevBuf tiles, grp_base, grp_rec, grp_len, rec_pos;
  fei::DevBuf hdir, hdir_off;            // header directory (hdir.cu): uint2 entries, u64 offsets [n+1]
  fei::DevBuf key_tag, key_rep, key_len, key_lut;   // dictionary of the corpus' distinct header keys + per-scan key -> slot-mask table
  uint64_t hdir_entries = 0;
  // header value columns (hdir.cu): for the few keys almost every record carries, the stripped value of the record's LAST
  // line with that exact key, as 16-byte units in unit-major planes (unit k of record i at plane k, offset 16 * i): a
  // thread-per-record scan reads them fully coalesced.  col_len[c * n + i]: 0xFFFF absent, 0xFFFE walk the directory.
  fei::DevBuf col_len, col_planes, kid_col, slot_col;
  uint32_t n_cols = 0;
  bool has_text_records = false;         // some record's header is parsed from its text (keys not in the dictionary)
  fei::DevBuf stage_body, stage_body_off, tmp_len, tmp_gunits;   // reused by repeated loads (no cudaMalloc per batch)
  fei::DevBuf aux[FEI_MAX_AUX]; uint64_t aux_n[FEI_MAX_AUX] = {0};   // host-computed per-record verdict bytes (fei_corpus_set_aux, FEI_C_RECBITS)
  fei::DevBuf stage_raw, stage_raw_off, stage_ms, stage_hlen, stage_blen;   // raw ingest staging (ingest.cu)
  // scan scratch (grown on demand, reused across scans)
  fei::DevBuf prog, hits, hit_lists, work_counter, scan_tmp, survivors, live_list, win_done;
  fei::CompactScratch compact;
  uint64_t hit_list_stride = 0;          // entries per query in hit_lists (last fei_scan_hits)
  uint32_t last_nq = 0;
  uint64_t last_counts[32] = {0};
  fei_scan_timing timing = {};
  cudaEvent_t ev[8] = {nullptr};
  // chunked scans: compaction / all-gather of a finished chunk run on `side` under the next chunk's scan (scan.cu)
  cudaStream_t side = nullptr;
  cudaEvent_t ev_load[3] = {nullptr, nullptr, nullptr};   // load_raw: before / after the text copy, end of the pack kernels
  bool load_timed = false; uint64_t load_raw_bytes = 0;
  uint64_t staged_text_bytes = ~0ull;    // size of the text fei_corpus_stage_text is filling stage_raw with (~0: none)
  cudaStream_t load_stream = nullptr;    // loads of this handle (H2D + pack kernels): own stream, so that batches streamed through several handles overlap
  cudaEvent_t ev_chunk[16] = {nullptr};
  cudaEvent_t ev_side = nullptr;
};

namespace fei {
// builds tiles from a canonical body blob already on the device (body has >= 32 bytes of slack)
int corpus_load_events(fei_corpus* c);              // ev_load[], created on first use
cudaStream_t corpus_load_stream(fei_corpus* c);   // created on first use; falls back to the context's copy stream
int build_tiles(fei_corpus* c, const uint8_t* d_body, const uint64_t* d_body_off, cudaStream_t s);
// builds the header directory from hdr / hdr_off already on the device (hdir.cu)
int build_header_dir(fei_corpus* c, cudaStream_t s);
// spans of the header value slot 0 of `prog` names (dict semantics of search.py:121-132) for records d_rows[0 .. m) (device array;
// nullptr: records 0 .. m-1): d_len[i] bytes at offset d_src[i] of the header blob, d_src[i] = ~0 when absent.  Caller holds c->mu.
int slot_spans_rows(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, const uint64_t* d_rows, uint64_t m, uint32_t* d_len, uint64_t* d_src,
                    cudaStream_t s);
int exclusive_scan_u32_u64(const uint32_t* in, uint64_t n, uint64_t* out, DevBuf& tmp, cudaStream_t s);
// Hook of a chunked scan: on_chunk is called on the host right after the work that makes the hit masks of records
// [rec_begin, rec_end) final has been queued, with `side` already waiting for it; on_done after the last chunk.
struct ChunkHook {
  // multi-GPU: if set, the scan kernel itself stores every finished window's hit masks into these peer buffers (device array of
  // push_n pointers, one per rank incl. this one; this rank's records start at element push_off of each).  run_scan sets `pushed`
  // when the launch it queued does that (k_body / k_body_sticky with window counters); otherwise on_chunk must move the masks.
  uint32_t* const* push_peers = nullptr; uint32_t push_n = 0; uint64_t push_off = 0; bool pushed = false;
  virtual int on_chunk(uint32_t k, uint32_t n_chunks, uint64_t rec_begin, uint64_t rec_end, cudaStream_t side) = 0;
  virtual int on_done(cudaStream_t side) { return FEI_OK; }
  virtual ~ChunkHook() {}
};
enum { kScanCompactNone = 0, kScanCompactLists = 1 };
// queues a whole scan (nothing waits for the GPU); force_chunks = 0 lets the scan pick its chunking.  Caller holds c->mu.
int run_scan(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, int compact_mode, ChunkHook* hook, uint32_t force_chunks);
int finish_timing(fei_corpus* c, bool compacted);
void plan_chunks(uint64_t n, uint32_t chunks, uint64_t* rec_bounds /* chunks + 1 */);
int compact_segments(const uint32_t* masks, uint64_t seg_stride, const uint64_t* seg_n, const uint64_t* seg_base, uint32_t n_seg, uint32_t nq,
                     CompactScratch& sc, uint64_t stride, uint64_t* lists, uint64_t* totals_out, cudaStream_t s);
int list_checksum(const uint64_t* list, uint64_t count, DevBuf& tmp, uint64_t* a_out, uint64_t* s_out, cudaStream_t s);
int compact_masks(const uint32_t* masks, uint64_t n, uint32_t nq, uint64_t global_base, CompactScratch& sc,
                  uint64_t* counts_out, DevBuf* lists, uint64_t* stride_out, uint32_t* launches, cudaStream_t s);
}
