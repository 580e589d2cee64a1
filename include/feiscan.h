/*
 * feiscan.h — C ABI of libfeiscan.so, the sm_100a scan engine behind Fei's Memdir
 * search / filter pipeline and Memorychain validation.
 *
 * The reference (david-strejc/fei) is pure Python and has no FFI of its own; each
 * entry point below names the reference interface whose inner loop it replaces.
 * The Python host layer (fei_b200/memdir_tools/) binds these with ctypes and keeps
 * the reference's signatures; INTEGRATION.md shows the stub a maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative FEI_E_* code; the message is
 *     available from fei_last_error() (thread local);
 *   - plain pointers and sizes only; the caller owns all host arrays for the duration
 *     of a call, the library copies what it keeps; device memory lives behind opaque
 *     handles; outputs go to caller-provided buffers with explicit capacities;
 *   - there is no CPU implementation behind any of the compute entry points: without
 *     a usable CUDA device they fail with FEI_E_CUDA.
 */
#ifndef FEISCAN_H_
#define FEISCAN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FEI_ABI_VERSION 1

enum {
  FEI_OK = 0,
  FEI_E_CUDA = -1,        /* CUDA runtime / driver error, or no device          */
  FEI_E_NCCL = -2,        /* NCCL error or NCCL not loadable                    */
  FEI_E_CAPACITY = -3,    /* caller buffer too small (required size is reported) */
  FEI_E_UNSUPPORTED = -4, /* program uses a feature the kernels do not implement */
  FEI_E_BADARG = -5,
  FEI_E_STATE = -6        /* call sequence error (e.g. scan before load)         */
};

int fei_abi_version(void);
const char* fei_last_error(void);

/* ---- process / device ------------------------------------------------------ */
/* One process drives one GPU (rank-local device index).                         */
int fei_init(int device);
int fei_shutdown(void);
int fei_device_info(int* sm_count, uint64_t* hbm_bytes, int* cc_major, int* cc_minor);
/* Page-lock a caller-owned host buffer so fei_corpus_load / fei_scan_hits copy at full PCIe
 * speed and asynchronously (cudaHostRegister / cudaHostUnregister).                        */
int fei_host_register(void* p, uint64_t bytes);
int fei_host_unregister(void* p);
/* Measured copy bandwidth (GB/s, best of reps) of a caller buffer to the device and back. */
int fei_host_copy_bench(void* host, uint64_t bytes, int reps, float* h2d_gbs, float* d2h_gbs);

/* Measured integer-issue peak of the chip (the roofline of the SHA-256 kernel, which is not HBM bound): tera lane-operations
 * per second of LOP3 / SHF (ALU pipe; IADD3 issues at the same rate), best of `reps` launches; ms = that launch's duration. */
int fei_microbench_alu(int reps, float* tera_lane_ops, float* ms);

/* ---- packed Memdir corpus ---------------------------------------------------
 * Replaces the per-query file walk of memdir_tools.utils.list_memories
 * (memdir_tools/utils.py:202-253): records are packed once, in the reference's
 * listing order, and stay resident in HBM.
 *
 * Host-side canonical form (what the packer produces, struct of arrays):
 *   hdr / hdr_off[n+1]    header text of record i = text before the first "---"
 *                         (parse_memory_content, utils.py:105-118), newline-normalised
 *   body / body_off[n+1]  body of record i, already .strip()ped (utils.py:120)
 *   name / name_off[n+1]  file name "ts.uid.host:2,FLAGS" (utils.py:74-95); may be NULL
 *   name_spans[4n]        where unique_id and hostname sit inside the name (the packer runs
 *                         the reference's filename regex, utils.py:81); NULL iff name is NULL
 *   ts[n]                 filename timestamp (utils.py:90)
 *   wall[n]               datetime.fromtimestamp(ts) as naive wall-clock seconds (utils.py:94)
 *   flags8[n]             flag letters, byte k = k-th letter, byte 7 = count (<= 7)
 *   fsb[n]                folder_id (bits 0-15) | status_id (16-23) | record bits (24-31)
 */
typedef struct fei_corpus fei_corpus;

#define FEI_REC_NO_SEPARATOR  0x01u  /* no "---": headers = {}, body = whole text (utils.py:107-109) */
#define FEI_REC_NONASCII      0x02u  /* record contains non-ASCII bytes                               */
#define FEI_REC_HAS_SIGMA     0x04u  /* record holds U+03A3: its str.lower() depends on the context (final sigma, search.py:148-163)  */
#define FEI_REC_HAS_IDOT      0x08u  /* record holds U+0130, whose lower() is two characters (the automata expand it)               */

typedef struct fei_corpus_host {
  uint64_t n;
  uint64_t global_base;      /* index of record 0 in the unsharded corpus (hits are global indices) */
  const uint8_t* hdr;   const uint64_t* hdr_off;
  const uint8_t* body;  const uint64_t* body_off;
  const uint8_t* name;  const uint64_t* name_off;
  const uint16_t* name_spans; /* 4 per record: unique_id start, length, hostname start, length inside the name */
  const int64_t* ts;
  const int64_t* wall;
  const uint64_t* flags8;
  const uint32_t* fsb;
} fei_corpus_host;

int fei_corpus_create(fei_corpus** out);
int fei_corpus_destroy(fei_corpus* c);
/* Copies the canonical arrays to HBM (pageable or pinned host memory), builds the
 * warp-transposed body tiles (DESIGN.md "data layout") and drops the canonical body. */
int fei_corpus_load(fei_corpus* c, const fei_corpus_host* h);
/* Raw ingest: like fei_corpus_load, but the text work of utils.list_memories / parse_memory_content
 * (memdir_tools/utils.py:229-232, :105-120) runs on the GPU.  raw/raw_off[n+1] = file contents as read from disk
 * (bytes); h->hdr / h->body (+ offsets) are ignored.  The kernels validate UTF-8 strictly (what open(path,"r")
 * would decode), fold "\r\n" / "\r" to "\n", split at the first "---", .strip() the body with Python's whitespace
 * set and set the record bits.  valid_out[n] (may be NULL) receives 1 for decodable files; if any file is not,
 * nothing is loaded and FEI_E_BADARG is returned so the caller can drop them (the reference reports and skips
 * such files, utils.py:247-248) and call again.                                                                */
int fei_corpus_load_raw(fei_corpus* c, const fei_corpus_host* h, const uint8_t* raw, const uint64_t* raw_off, uint8_t* valid_out);
/* Uploads raw[offset .. offset + bytes) of a text of total_bytes ahead of fei_corpus_load_raw[_spans], which is then called with
 * raw == NULL: lets a caller that produces the text piece by piece (one directory at a time) overlap the upload with producing
 * the next piece.  One stretch at a time per handle; fei_corpus_load_raw fails with FEI_E_STATE if the sizes do not agree. */
int fei_corpus_stage_text(fei_corpus* c, uint64_t total_bytes, const uint8_t* src, uint64_t offset, uint64_t bytes);
/* The same with file i at raw[begin[i] .. begin[i] + len[i]) (any order, gaps allowed: what fei_read_dir_packed leaves in its arena);
 * raw_bytes = the extent of raw to upload. */
int fei_corpus_load_raw_spans(fei_corpus* c, const fei_corpus_host* h, const uint8_t* raw, uint64_t raw_bytes, const uint64_t* begin,
                              const uint64_t* len, uint8_t* valid_out);
/* Device-side stage times (ms) of the last fei_corpus_load_raw on this handle, CUDA events on its load stream:
 * out[0] = host-to-device copy of the file text, out[1] = the pack kernels after it (measure, offsets, normalise, tiling,
 * header directory), out[2] = that copy's rate in GB/s.  Waits for the load to finish on the device. */
int fei_corpus_last_load_timing(fei_corpus* c, float* out);
/* Fills the corpus with records [first, first+n) of the deterministic synthetic
 * Memdir (fei_b200/csrc/synth.cuh), generated on the GPU.                           */
int fei_corpus_synth(fei_corpus* c, uint64_t seed, uint64_t first, uint64_t n);

/* ---- native directory listing / file reads (host only; the one-time pack of utils.list_memories, utils.py:202-253) ----
 * fei_dir_list: the entries of one cur/new/tmp directory whose names match the listing grammar `\d+\.[a-z0-9]+\.[^:]+:2,[A-Z]*`
 * (utils.py:223), newest filename timestamp first, ties in readdir (= os.listdir) order (utils.py:251), with what
 * parse_memory_filename (utils.py:74-95) extracts and a stat of every file (inode / size / mtime: the change detector of the
 * incremental sync).  status[i]: 1 = parsed natively; 2 = a name only Python's re / int() / datetime can judge (non-ASCII leading
 * digits, more than 18 digits, years past 9999, a file that vanished): listed last, the caller decides.  A missing directory
 * lists as empty (utils.py:216-217).                                                                                        */
typedef struct fei_dirlist fei_dirlist;
typedef struct fei_dirlist_view {
  uint64_t n;
  const uint8_t* names; const uint64_t* name_off;      /* n + 1 offsets */
  const int64_t* ts; const int64_t* wall; const int64_t* mtime_ns;
  const uint64_t* ino; const uint64_t* size; const uint64_t* flags8;
  const uint16_t* spans;                               /* 4 per entry, like fei_corpus_host.name_spans */
  const uint8_t* status; const int64_t* flags_len;
} fei_dirlist_view;
int fei_dir_list(const char* path, fei_dirlist** out);
/* The same listing without the per-entry stat: ino comes from the directory entry, size = 0 and mtime_ns = -1 until
 * fei_read_dir_packed has opened the file. */
int fei_dir_list_names(const char* path, fei_dirlist** out);
int fei_dirlist_view_get(const fei_dirlist* l, fei_dirlist_view* v);
void fei_dirlist_free(fei_dirlist* l);
/* n files of one directory read by `threads` workers into dst[dst_off[i] .. dst_off[i+1]) (capacities from the listing's sizes);
 * got[i] = bytes read (at most the listed size), err[i] = errno.  dst may be pinned (fei_host_register).                          */
int fei_read_files(const char* dir, const uint8_t* names, const uint64_t* name_off, uint64_t n, uint8_t* dst, const uint64_t* dst_off,
                   int threads, uint64_t* got, int32_t* err);
/* Cold read without a stat pass (open, fstat, read, close per file): the files' bytes go into a caller arena at positions handed out
 * by an atomic add on *cursor (start it at 0 and pass the same cursor for every directory of a tree); begin[i] / len[i] locate file
 * i, ino[i] / mtime_ns[i] come from the open file.  err[i] = errno; EFBIG = larger than max_file_bytes (len[i] = its size, not
 * read), ENOMEM = the arena is full.  fei_host_arena_alloc maps address space without committing memory (MAP_NORESERVE): size it
 * for the largest tree, only the bytes read become resident.                                                                  */
int fei_host_arena_alloc(uint64_t bytes, int huge_pages, void** out);   /* huge_pages: madvise(MADV_HUGEPAGE) on the mapping */
int fei_host_arena_free(void* p, uint64_t bytes);
int fei_read_dir_packed(const char* dir, const uint8_t* names, const uint64_t* name_off, uint64_t n, uint8_t* arena, uint64_t arena_cap,
                        uint64_t* cursor, uint64_t max_file_bytes, int threads, uint64_t* begin, uint64_t* len, uint64_t* ino,
                        int64_t* mtime_ns, int32_t* err);
/* tooling: write n files into an existing directory with `threads` workers (synthetic trees for tests and the bench).          */
int fei_write_files(const char* dir, const uint8_t* names, const uint64_t* name_off, const uint8_t* blob, const uint64_t* off, uint64_t n, int threads);

typedef struct fei_corpus_stats {
  uint64_t n, global_base;
  uint64_t hdr_bytes, body_bytes, tile_bytes, name_bytes;
  uint64_t n_groups;
  uint64_t device_bytes;     /* total HBM held by this corpus */
} fei_corpus_stats;
int fei_corpus_stats_get(const fei_corpus* c, fei_corpus_stats* out);

/* Debug / materialisation: copy the canonical pieces of records [first, first+n) back
 * to the host.  Bodies are un-tiled on the device first.  Any pointer may be NULL. */
int fei_corpus_fetch(fei_corpus* c, uint64_t first, uint64_t n,
                     uint8_t* hdr, uint64_t hdr_cap, uint64_t* hdr_off,
                     uint8_t* body, uint64_t body_cap, uint64_t* body_off,
                     int64_t* ts, int64_t* wall, uint64_t* flags8, uint32_t* fsb);

/* Header text and body of the m records idx[0..m) (any order), for materialising hits without keeping file contents on the host.
 * hdr_off / body_off get m + 1 offsets; hdr / body may be NULL to only size the buffers; FEI_E_CAPACITY if a blob is too small.  */
int fei_corpus_fetch_records(fei_corpus* c, const uint64_t* idx, uint64_t m, uint8_t* hdr, uint64_t hdr_cap, uint64_t* hdr_off,
                             uint8_t* body, uint64_t body_cap, uint64_t* body_off);
/* Snapshot of the packed corpus (everything fei_corpus_load* built) in one file, and its restore: the file is streamed through a
 * ring of pinned buffers, reader threads ahead of the copy engine; gbs = bytes restored per second (CUDA events).  A process
 * restart then costs a file read instead of a walk + pack of the Memdir tree (utils.py:202-253 re-reads every file per query). */
int fei_corpus_save(fei_corpus* c, const char* path);
int fei_corpus_load_snapshot(fei_corpus* c, const char* path, float* gbs);

/* ---- scan ---------------------------------------------------------------------
 * Replaces the hot loops of memdir_tools.search.search_memories
 * (memdir_tools/search.py:361-367 -> _memory_matches_query :244-335) and of
 * FilterManager.process_memories / MemoryFilter.matches (memdir_tools/filter.py:229-233,
 * :67-109).  `prog` is a compiled predicate program (fei_b200/program.py documents the
 * binary layout; include/feiscan_prog.h declares it): up to 32 queries evaluated in one
 * pass, each the AND of header/meta/content conditions.
 *
 * fei_scan_masks : mask[i] bit q = record i satisfies query q.  `masks` may be a host
 *                  pointer (n entries) or NULL to keep the result on the device only.
 * fei_scan_hits  : per query, the ordered list of matching GLOBAL record indices
 *                  (ascending = the reference's listing order).  hits[q] has room for
 *                  cap[q] entries; nhits[q] receives the true count; returns
 *                  FEI_E_CAPACITY if any list was truncated.
 */
int fei_scan_masks(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint32_t* masks);
int fei_scan_hits(fei_corpus* c, const uint8_t* prog, uint64_t prog_len,
                  uint64_t* const* hits, const uint64_t* cap, uint64_t* nhits);
/* Counts on the host, the ordered lists stay on the device: nhits[q] for every query.
 * Big content scans run as a few chunks of whole 4096-record windows; the compaction of a
 * finished chunk runs on a second stream under the next chunk's scan.                  */
int fei_scan_count(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint64_t* nhits);
/* Copies the lists the last fei_scan_count left on the device (hits[q] has room for cap[q]
 * entries; FEI_E_CAPACITY if one is shorter than its list): the second half of fei_scan_hits
 * for callers that size their buffers from the counts.                                     */
int fei_scan_fetch_hits(fei_corpus* c, uint32_t nq, uint64_t* const* hits, const uint64_t* cap);
/* Order-sensitive checksums of the lists the last fei_scan_count / fei_scan_hits left on the
 * device: a[q] = sum_k (k+1) * list_q[k], s[q] = sum_k list_q[k] (mod 2^64).  A sharded scan
 * reports the same numbers for the gathered global lists (fei_comm_gathered_checksum).  */
int fei_scan_list_checksum(fei_corpus* c, uint32_t nq, uint64_t* a, uint64_t* s);

/* Per-call timing of the last scan on this corpus, measured with CUDA events on the
 * launching stream: ms spent in the head kernel, body kernel, compaction, copies.    */
typedef struct fei_scan_timing {
  float head_ms, body_ms, compact_ms, h2d_ms, d2h_ms, total_ms;
  uint32_t kernel_launches;
  uint64_t body_bytes_touched;   /* tile bytes of groups that had at least one live record */
  uint64_t body_bytes_read;      /* tile bytes the body kernel really requested (a single-pattern scan stops reading a
                                    group once all of its records have matched; copies already in flight are counted) */
} fei_scan_timing;
int fei_scan_last_timing(const fei_corpus* c, fei_scan_timing* out);

/* Token histogram of one header field over the records a program selects -- the tag statistics of
 * MemdirFolderManager.get_folder_stats (memdir_tools/folders.py:286-292):
 *     if "Tags" in memory["headers"]: for tag in [t.strip() for t in memory["headers"]["Tags"].split(",")]: tags[tag] += 1
 * prog: ONE query; its conditions select the records, its first header field (slot 0; use an exact-key slot with an
 * always-true pattern) names the column.  sep: the separator byte.  Out, ordered like a dict filled record by record
 * (first record carrying the token, then position inside the value): token k = tok_blob[tok_off[k] .. tok_off[k+1]),
 * tok_count[k] occurrences, tok_first[k] = global index of the first record with it.  *n_tokens = entries written.
 * FEI_E_CAPACITY when cap / blob_cap are too small; FEI_E_UNSUPPORTED for corpora with headers over 64 KiB, more than
 * 32768 distinct tokens or a 64-bit hash collision (callers then count on the host). */
int fei_corpus_token_histogram(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint8_t sep,
                               uint8_t* tok_blob, uint64_t blob_cap, uint64_t* tok_off, uint64_t* tok_count, uint64_t* tok_first,
                               uint64_t cap, uint64_t* n_tokens);

/* The header value the reference would read for one field, for every record (slot 0 of `prog` resolved with the dict semantics of
 * search.py:121-132 / filter.py:90-91): present[n], off[n+1], blob.  For conditions whose verdict only Python can compute value by
 * value: the per-record dateutil parses of Due / Created / Modified / DeletedDate (search.py:126-130).  The host judges the DISTINCT
 * values and hands the verdicts back as an aux column (fei_corpus_set_aux) that FEI_C_RECBITS conditions read in the scan.   */
int fei_corpus_slot_values(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint8_t* present, uint64_t* off,
                           uint8_t* blob, uint64_t blob_cap);
int fei_corpus_set_aux(fei_corpus* c, uint32_t k, const uint8_t* bytes, uint64_t n);

/* ---- result order --------------------------------------------------------------
 * Replaces the sort and the slice of memdir_tools.search.search_memories (memdir_tools/search.py:370-388):
 *     results.sort(key=lambda x: _get_field_value(x, sort_by) or "", reverse=sort_reverse)   (keys: search.py:97-139)
 *     results = results[offset : offset + limit]
 * for the keys whose order the device can decide.  Row i is record row_rec[i] of corpora[row_corpus[i]] (a base corpus and the
 * delta of an incremental sync can be mixed); rows [0, m) are in the order the hits were found.  The sort is stable, also when
 * descending (as CPython's reverse=True: equal keys keep their order).  out[0 .. min(count, m - first)) receives the row
 * indices at sorted positions [first, first + count).  Key sources (spec->source):
 *   FEI_SORT_SLOT        the header value slot 0 of spec->prog names (mode 0: first key whose lower() equals the field, dict
 *                        semantics; mode 1: exact key); an absent header reads as spec->fallback: FEI_SORT_NONE (the empty
 *                        string), FEI_SORT_NAME_UID or FEI_SORT_NAME_HOST (the metadata of search.py:134-137)
 *   FEI_SORT_NAME        the file name; FEI_SORT_NAME_UID / _HOST its unique_id / hostname (corpora loaded with names)
 *   FEI_SORT_FLAGS       the flag letters joined;  FEI_SORT_BODY the stripped body
 *   FEI_SORT_TS / _WALL  the filename timestamp / datetime.fromtimestamp(ts) (naive wall clock)
 *   FEI_SORT_KEYS        spec->keys[i], unsigned (values the caller ranked)
 * Strings compare by unsigned byte (= code point order for UTF-8), a proper prefix first.  info (may be NULL): rounds = sort
 * rounds (one per 7 bytes of the longest common prefix still tied), radix_passes, refined_rows = rows re-sorted after round 0,
 * ms = device time from the first to the last kernel (CUDA events).  FEI_E_BADARG for a bad spec or row.          */
enum { FEI_SORT_NONE = 0, FEI_SORT_SLOT = 1, FEI_SORT_NAME = 2, FEI_SORT_NAME_UID = 3, FEI_SORT_NAME_HOST = 4, FEI_SORT_FLAGS = 5,
       FEI_SORT_BODY = 6, FEI_SORT_TS = 7, FEI_SORT_WALL = 8, FEI_SORT_KEYS = 9 };
typedef struct fei_sort_spec {
  uint32_t source;
  uint32_t fallback;            /* FEI_SORT_SLOT only */
  const uint8_t* prog;          /* FEI_SORT_SLOT: compiled program (fei_b200/program.py), slot 0 names the header */
  uint64_t prog_len;
  const uint64_t* keys;         /* FEI_SORT_KEYS: m keys */
} fei_sort_spec;
typedef struct fei_sort_info {
  uint32_t rounds, radix_passes;
  uint64_t refined_rows;
  float ms;
} fei_sort_info;
int fei_sort_rows(fei_corpus* const* corpora, uint32_t n_corpora, const uint32_t* row_corpus, const uint64_t* row_rec, uint64_t m,
                  const fei_sort_spec* spec, int descending, uint64_t first, uint64_t count, uint64_t* out, fei_sort_info* info);

/* ---- Memorychain validation -----------------------------------------------------
 * Replaces the loop of MemoryChain.validate_chain (memdir_tools/memorychain.py:596-618)
 * and its inline copy in receive_chain_update (:1059-1078):
 *   for i in 1..n-1:  hash[i] == sha256(canonical_json(block i))   else "invalid hash"
 *                     prev[i] == hash[i-1]                          else "broken link"
 * first_bad = smallest failing i (or -1), bad_kind = 1 (invalid hash) / 2 (broken link).
 * Block 0 (genesis) is never checked, exactly as in the reference.
 *
 * fei_chain_validate_msgs takes the canonical JSON texts (MemoryBlock.calculate_hash,
 * memorychain.py:117-128) already serialised:
 *   msgs/msg_off[n+1], stored hash strings hash/hash_off[n+1], previous_hash strings
 *   prev/prev_off[n+1]; digests (32*n bytes, may be NULL) receives the raw SHA-256.
 */
int fei_chain_validate_msgs(const uint8_t* msgs, const uint64_t* msg_off,
                            const uint8_t* hash, const uint64_t* hash_off,
                            const uint8_t* prev, const uint64_t* prev_off,
                            uint64_t n, uint64_t first_index,
                            int64_t* first_bad, int32_t* bad_kind, uint8_t* digests);

/* Column form: the ten hashed fields of every block as typed JSON scalars; the library
 * serialises them to canonical JSON (json.dumps(sort_keys=True), memorychain.py:117-128)
 * in C++ and validates on the GPU.  Field order in `cols` is the sorted key order:
 * difficulty, index, memory_id, nonce, previous_hash, proposer_node, responsible_node,
 * solver_node, task_state, timestamp.                                                */
enum { FEI_J_NULL = 0, FEI_J_STR = 1, FEI_J_INT = 2, FEI_J_FLOAT = 3, FEI_J_TRUE = 4, FEI_J_FALSE = 5,
       FEI_J_BIGINT = 6 /* decimal digits in the string blob */ };
typedef struct fei_json_col {
  const uint8_t* tag;        /* n tags, or NULL when every value has tag `uniform_tag` */
  int32_t uniform_tag;
  const uint64_t* num;       /* n entries: int64 or IEEE double bit patterns            */
  const uint8_t* str;        /* UTF-8 blob                                              */
  const uint64_t* str_off;   /* n+1 offsets                                             */
} fei_json_col;
#define FEI_CHAIN_NCOLS 10
int fei_chain_validate_cols(const fei_json_col* cols /*[FEI_CHAIN_NCOLS]*/,
                            const uint8_t* hash, const uint64_t* hash_off,
                            uint64_t n, uint64_t first_index,
                            int64_t* first_bad, int32_t* bad_kind, uint8_t* digests,
                            uint8_t* msgs_out, uint64_t msgs_cap, uint64_t* msg_off_out);

/* Resident form for benchmarking / streaming: messages and stored hashes uploaded
 * once, validated repeatedly.                                                         */
typedef struct fei_chain fei_chain;
int fei_chain_create(fei_chain** out);
int fei_chain_destroy(fei_chain* ch);
int fei_chain_load_msgs(fei_chain* ch, const uint8_t* msgs, const uint64_t* msg_off,
                        const uint8_t* hash, const uint64_t* hash_off,
                        const uint8_t* prev, const uint64_t* prev_off, uint64_t n, uint64_t first_index);
/* The same from the column form: typed columns go up (~100 B per block), the canonical JSON texts (incl. Python's shortest
 * round-trip float repr) are produced by a GPU kernel, then hashed in place.  previous_hash must be all strings.                 */
int fei_chain_load_cols(fei_chain* ch, const fei_json_col* cols /*[FEI_CHAIN_NCOLS]*/, const uint8_t* hash, const uint64_t* hash_off,
                        uint64_t n, uint64_t first_index);
/* Synthetic chain blocks [first, first+n) (synth.cuh gen_block): canonical JSON and
 * the SHA-256 links are produced on the GPU; `corrupt_at` >= 0 flips one stored digest. */
int fei_chain_synth(fei_chain* ch, uint64_t seed, uint64_t first, uint64_t n, int64_t corrupt_at);
int fei_chain_validate(fei_chain* ch, int64_t* first_bad, int32_t* bad_kind, uint8_t* digests, float* kernel_ms);
int fei_chain_fetch(fei_chain* ch, uint64_t first, uint64_t n, uint8_t* msgs, uint64_t msgs_cap, uint64_t* msg_off,
                    uint8_t* hash_hex /*64*n*/, uint8_t* prev_hex /*64*n*/);

/* Proof of work, MemoryBlock.mine_block (memdir_tools/memorychain.py:132-143): the block's canonical text is
 * prefix + decimal(nonce) + suffix; finds the smallest nonce >= start_nonce whose SHA-256 hexdigest starts with
 * `difficulty` zeros (FEI_E_CAPACITY if none within max_tries).  digest_out (32 bytes, may be NULL) = its digest. */
int fei_chain_mine(const uint8_t* prefix, uint32_t prefix_len, const uint8_t* suffix, uint32_t suffix_len,
                   uint64_t start_nonce, uint32_t difficulty, uint64_t max_tries,
                   uint64_t* nonce_out, uint8_t* digest_out, uint64_t* tried_out);

/* Host-only helper (no GPU): canonical JSON of the column form, for tests of the
 * serialiser against json.dumps.                                                      */
int fei_chain_serialize_cols(const fei_json_col* cols, uint64_t n,
                             uint8_t* msgs_out, uint64_t msgs_cap, uint64_t* msg_off_out);

/* ---- synthetic data on the host (same generator as the device one) --------------- */
int fei_synth_record_host(uint64_t seed, uint64_t i,
                          uint8_t* hdr, uint32_t hdr_cap, uint32_t* hdr_len,
                          uint8_t* body, uint32_t body_cap, uint32_t* body_len,
                          int64_t* ts, char* uid8, char* flags4, uint8_t* nflags, uint8_t* status, uint8_t* folder);
int fei_synth_block_host(uint64_t seed, uint64_t i, double* timestamp, char* memory_id8,
                         uint8_t* task_state, uint8_t* difficulty, uint8_t* is_task);

/* tooling: records [first, first+n) of the synthetic Memdir written as Maildir files under base (directories must exist).          */
int fei_synth_write_tree(const char* base, const char* hostname, uint64_t seed, uint64_t first, uint64_t n, int threads);

/* ---- multi-GPU (one process per GPU; NCCL is dlopen()ed at first use) ------------- */
#define FEI_NCCL_ID_BYTES 128
int fei_comm_unique_id(uint8_t* id /*[FEI_NCCL_ID_BYTES]*/);
int fei_comm_init(const uint8_t* id, int nranks, int rank);
int fei_comm_destroy(void);
/* all-gatherv of the per-query ordered hit lists left on the device by the last
 * fei_scan_hits / fei_scan_count(keep) on this corpus: rank-order concatenation is the
 * global listing order.  counts_out[r*nq + q] = hits of query q on rank r.             */
int fei_comm_allgather_hits(fei_corpus* c, uint32_t nq, uint64_t* const* hits, const uint64_t* cap,
                            uint64_t* nhits_total, uint64_t* counts_out);
/* Collective: every rank names the shard it is going to scan.  The ranks exchange (record count,
 * first global index), allocate the rank-major buffer that receives the hit masks of all shards
 * and map each other's buffer (CUDA IPC: NVLink / NVSwitch peer memory); FEI_COMM_P2P=0, or a
 * failed mapping on any rank, keeps the exchange on NCCL.  fei_comm_is_p2p() says which.        */
int fei_comm_bind_corpus(fei_corpus* c);
int fei_comm_is_p2p(void);
int fei_comm_last_exchange_in_kernel(void);   /* 1: the last fei_comm_scan_gather stored its masks into the peers from inside the scan kernel */
/* Collective: the scan of fei_scan_count (masks + ordered local lists) with the hit all-gather
 * folded in: the scan runs in chunks, and the masks of a finished chunk are written into every
 * peer's buffer by copy-engine transfers (or a grouped ncclBroadcast) while the next chunk is
 * scanned.  On return every rank holds the masks of ALL shards, rank-major = global listing
 * order, and nhits_total[q] = global hits of query q.  The buffers are overwritten as soon as
 * any rank enters the next gather.                                                            */
int fei_comm_scan_gather(fei_corpus* c, const uint8_t* prog, uint64_t prog_len, uint64_t* nhits_total);
/* Lengths and order-sensitive checksums (see fei_scan_list_checksum) of the GLOBAL ordered hit
 * lists the last gather on this rank stands for (fei_comm_scan_gather / fei_comm_allgather_hits). */
int fei_comm_gathered_checksum(uint32_t nq, uint64_t* totals, uint64_t* a, uint64_t* s);
/* Materialises those global ordered lists on this rank's device from the gathered masks
 * (dense results); ms = device time of the build.                                            */
int fei_comm_global_lists(uint32_t nq, uint64_t* totals, float* ms);
/* min-reduce of (first_bad, kind) over ranks for a range-sharded chain.               */
int fei_comm_allreduce_first_bad(int64_t* first_bad, int32_t* bad_kind);

#ifdef __cplusplus
}
#endif
#endif /* FEISCAN_H_ */
