// Result ordering of search_memories (memdir_tools/search.py:370-388) on the device: fei_sort_rows.
//
//   results.sort(key=lambda x: _get_field_value(x, sort_by) or "", reverse=sort_reverse); results[offset : offset + limit]
//
// The rows are (corpus, record) pairs in the hit order the scan returned.  Every key the sort can see is turned into 64-bit words
// whose unsigned order is the key's order:
//   - byte strings (header values, file names and their unique_id / hostname spans, bodies): word r holds bytes [7r, 7r+7)
//     zero-padded, big-endian in the top 7 bytes, and in the low byte the number of those bytes that exist (0..7), or 8 when more
//     bytes follow.  Code-point order of strictly decoded UTF-8 is unsigned byte order with a proper prefix first, and this word
//     order is exactly that, embedded NUL bytes included (a padding zero and a real zero differ in the count byte);
//   - flags8 is already that word for the joined flag letters (at most 7, so one word);
//   - ts / wall: the int64 with the sign bit flipped;  caller keys (host-ranked values): as given.
// Descending order complements the words: CPython's reverse=True keeps equal keys in their original order, which a stable
// ascending sort of the complemented keys does too.
//
// Round 0 sorts all rows by word 0 (stable LSD radix sort, 8-bit digits, digits on which every key agrees are skipped).  A run
// of equal words whose count byte is 8 is a segment whose order is not decided yet; round r re-sorts only the rows of such
// segments by (segment, word r): a radix sort by the word, then a stable one by the segment id, and writes them back into the
// positions their segment occupies.  Rounds stop when no such segment is left.
#include "corpus.h"
#include <string.h>
#include <algorithm>
#include <mutex>
#include <vector>

namespace fei {
namespace {
constexpr int kSortThreads = 256;
constexpr int kSortItems = 16;                               // keys per thread and pass
constexpr uint32_t kSortTile = kSortThreads * kSortItems;    // keys per block
constexpr int kSortWarps = kSortThreads / 32;
constexpr uint32_t kWarpSpan = kSortTile / kSortWarps;       // consecutive keys of one warp

struct SrcPtrs {                                             // one corpus' device columns
  const uint8_t* hdr; const uint8_t* name; const uint64_t* name_off; const uint16_t* name_spans;
  const uint8_t* tiles; const uint64_t* grp_base; const uint32_t* grp_len; const uint32_t* rec_pos;
  const int64_t* ts; const int64_t* wall; const uint64_t* flags8;
};
enum : uint8_t { kStrHdr = 0, kStrName = 1, kStrBody = 2 };

// Where row i's byte string lives: kind, offset (hdr / name blob; rec_pos entry for bodies), length.
__global__ void k_str_prep(const SrcPtrs* __restrict__ cp, const uint32_t* __restrict__ row_c, const uint64_t* __restrict__ row_r, uint32_t m,
                           uint32_t source, uint32_t fallback, const uint32_t* __restrict__ slot_len, const uint64_t* __restrict__ slot_src,
                           uint8_t* __restrict__ kind, uint64_t* __restrict__ off, uint32_t* __restrict__ len) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const SrcPtrs c = cp[row_c[i]];
  const uint64_t r = row_r[i];
  uint32_t src = source;
  if (src == FEI_SORT_SLOT) {
    if (slot_src[i] != ~0ull) { kind[i] = kStrHdr; off[i] = slot_src[i]; len[i] = slot_len[i]; return; }
    src = fallback;
  }
  if (src == FEI_SORT_BODY) {
    const uint32_t pos = c.rec_pos[r];
    kind[i] = kStrBody; off[i] = pos; len[i] = c.grp_len[pos];
    return;
  }
  kind[i] = kStrName;
  if (src == FEI_SORT_NAME) { off[i] = c.name_off[r]; len[i] = (uint32_t)(c.name_off[r + 1] - c.name_off[r]); return; }
  if (src == FEI_SORT_NAME_UID || src == FEI_SORT_NAME_HOST) {
    const int k = src == FEI_SORT_NAME_UID ? 0 : 2;
    off[i] = c.name_off[r] + c.name_spans[4 * r + k]; len[i] = c.name_spans[4 * r + k + 1];
    return;
  }
  off[i] = 0; len[i] = 0;                                    // FEI_SORT_NONE: the empty string
}

__device__ __forceinline__ uint8_t body_byte(const SrcPtrs& c, uint32_t pos, uint32_t o) {
  // unit u of the record at tile position pos: grp_base + sum over the group's lanes of min(units, u), then this lane (corpus.h)
  const uint64_t g = pos >> 5;
  const uint32_t u = o >> 4;
  const uint32_t* gl = c.grp_len + g * 32;
  uint64_t before = 0;
  for (int l = 0; l < 32; ++l) { const uint32_t n = (gl[l] + 15) >> 4; before += n < u ? n : u; }
  const uint8_t t = c.tiles[(c.grp_base[g] + before) * 16 + (pos & 31) * 16 + (o & 15)];
  return (uint8_t)(t ^ ((t >> 1) & 0x20));                   // undo the tile byte permutation
}

// Word `round` of the key of item j (row order[pos[j]]); complemented for a descending sort.  Also seeds the payload j.
__global__ void k_words(const SrcPtrs* __restrict__ cp, const uint32_t* __restrict__ row_c, const uint64_t* __restrict__ row_r,
                        const uint64_t* __restrict__ host_keys, uint32_t source, const uint8_t* __restrict__ kind,
                        const uint64_t* __restrict__ off, const uint32_t* __restrict__ len, const uint32_t* __restrict__ order,
                        const uint32_t* __restrict__ pos, uint32_t k, uint32_t round, int desc, uint64_t* __restrict__ w0,
                        uint64_t* __restrict__ key, uint32_t* __restrict__ val) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= k) return;
  const uint32_t i = order[pos ? pos[j] : j];
  uint64_t w;
  if (source == FEI_SORT_TS || source == FEI_SORT_WALL) {
    const SrcPtrs c = cp[row_c[i]];
    w = (uint64_t)(source == FEI_SORT_TS ? c.ts : c.wall)[row_r[i]] ^ (1ull << 63);
  } else if (source == FEI_SORT_FLAGS) {
    const uint64_t f = cp[row_c[i]].flags8[row_r[i]];
    const uint32_t n = (uint32_t)(f >> 56);
    w = n;
    for (uint32_t b = 0; b < n; ++b) w |= ((f >> (8 * b)) & 0xFF) << (56 - 8 * b);
  } else if (source == FEI_SORT_KEYS) {
    w = host_keys[i];
  } else {
    const uint32_t o = round * 7, L = len[i];
    const uint32_t avail = L > o ? L - o : 0;
    const uint32_t n = avail < 7 ? avail : 7;
    w = avail > 7 ? 8 : n;
    const uint8_t kd = kind[i];
    if (kd == kStrBody) {
      const SrcPtrs c = cp[row_c[i]];
      for (uint32_t b = 0; b < n; ++b) w |= (uint64_t)body_byte(c, (uint32_t)off[i], o + b) << (56 - 8 * b);
    } else {
      const SrcPtrs& c = cp[row_c[i]];
      const uint8_t* p = (kd == kStrHdr ? c.hdr : c.name) + off[i] + o;
      for (uint32_t b = 0; b < n; ++b) w |= (uint64_t)p[b] << (56 - 8 * b);
    }
  }
  if (desc) w = ~w;
  w0[j] = w; key[j] = w; val[j] = j;
}

// out[0] |= key, out[1] &= key over keys[0..k): the bits on which the keys differ are out[0] ^ out[1].
__global__ void k_or_and(const uint64_t* __restrict__ keys, uint32_t k, unsigned long long* __restrict__ out) {
  unsigned long long o = 0, a = ~0ull;
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < k; j += gridDim.x * blockDim.x) { o |= keys[j]; a &= keys[j]; }
  for (int d = 16; d; d >>= 1) { o |= __shfl_xor_sync(0xffffffffu, o, d); a &= __shfl_xor_sync(0xffffffffu, a, d); }
  if ((threadIdx.x & 31) == 0) { atomicOr(out, o); atomicAnd(out + 1, a); }
}

__global__ void __launch_bounds__(kSortThreads) k_digit_hist(const uint64_t* __restrict__ keys, uint32_t k, int sh, uint32_t nb,
                                                             uint32_t* __restrict__ counts) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t base = blockIdx.x * kSortTile;
  for (uint32_t t = threadIdx.x; t < kSortTile; t += kSortThreads) {
    const uint32_t j = base + t;
    if (j < k) atomicAdd(&h[(keys[j] >> sh) & 0xFF], 1u);
  }
  __syncthreads();
  counts[threadIdx.x * nb + blockIdx.x] = h[threadIdx.x];    // digit-major: one exclusive scan gives every block's bucket offsets
}

// Stable scatter of one 8-bit digit: warp w of block b owns keys [b*tile + w*span, +span), 32 at a time in lane order; equal
// digits inside a 32-key step are ranked with __match_any_sync, so the relative order of equal digits is kept everywhere.
__global__ void __launch_bounds__(kSortThreads) k_digit_scatter(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint32_t k,
                                                                int sh, uint32_t nb, const uint64_t* __restrict__ offs,
                                                                uint64_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out) {
  __shared__ uint32_t wh[kSortWarps][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = threadIdx.x; t < kSortWarps * 256; t += kSortThreads) (&wh[0][0])[t] = 0;
  __syncthreads();
  const uint32_t wbase = blockIdx.x * kSortTile + warp * kWarpSpan;
  const uint32_t lt = (1u << lane) - 1;
  uint32_t dg[kWarpSpan / 32];
#pragma unroll
  for (int s = 0; s < (int)(kWarpSpan / 32); ++s) {
    const uint32_t j = wbase + s * 32 + lane;
    dg[s] = j < k ? (uint32_t)((keys[j] >> sh) & 0xFF) : 256u + lane;
    const uint32_t peers = __match_any_sync(0xffffffffu, dg[s]);
    if (dg[s] < 256 && (peers & lt) == 0) wh[warp][dg[s]] += __popc(peers);
  }
  __syncthreads();
  {
    const int d = threadIdx.x;                               // kSortThreads == 256 digits
    uint32_t run = (uint32_t)offs[(uint64_t)d * nb + blockIdx.x];
    for (int w = 0; w < kSortWarps; ++w) { const uint32_t t = wh[w][d]; wh[w][d] = run; run += t; }
  }
  __syncthreads();
#pragma unroll
  for (int s = 0; s < (int)(kWarpSpan / 32); ++s) {
    const uint32_t j = wbase + s * 32 + lane;
    const uint32_t peers = __match_any_sync(0xffffffffu, dg[s]);
    uint32_t at = 0;
    if (dg[s] < 256) {
      at = wh[warp][dg[s]] + __popc(peers & lt);
      keys_out[at] = keys[j]; vals_out[at] = vals[j];
    }
    __syncwarp();
    if (dg[s] < 256 && (peers & lt) == 0) wh[warp][dg[s]] += __popc(peers);
    __syncwarp();
  }
}

__global__ void k_seg_keys(const uint32_t* __restrict__ seg, const uint32_t* __restrict__ val, uint32_t k, uint64_t* __restrict__ key) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < k) key[j] = seg[val[j]];
}

// Sorted item t is item val[t]: its row goes to position pos[t] (the positions of the items, ascending, cover their segments).
__global__ void k_apply_gather(const uint32_t* __restrict__ val, uint32_t k, const uint32_t* __restrict__ order, const uint32_t* __restrict__ pos,
                               const uint64_t* __restrict__ w0, const uint32_t* __restrict__ seg, uint32_t* __restrict__ rows_tmp,
                               uint64_t* __restrict__ sw, uint32_t* __restrict__ ss) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= k) return;
  const uint32_t j = val[t];
  rows_tmp[t] = order[pos ? pos[j] : j];
  sw[t] = w0[j];
  ss[t] = seg ? seg[j] : 0u;
}
__global__ void k_apply_scatter(const uint32_t* __restrict__ rows_tmp, uint32_t k, const uint32_t* __restrict__ pos, uint32_t* __restrict__ order) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < k) order[pos ? pos[t] : t] = rows_tmp[t];
}

// head[t]: sorted item t starts a run of equal (segment, word); cont[t]: its run has >= 2 items and bytes left (count byte 8).
__global__ void k_runs(const uint64_t* __restrict__ sw, const uint32_t* __restrict__ ss, uint32_t k, int desc, uint32_t* __restrict__ head,
                       uint32_t* __restrict__ cont) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= k) return;
  const bool h = t == 0 || sw[t] != sw[t - 1] || ss[t] != ss[t - 1];
  const bool next_same = t + 1 < k && sw[t + 1] == sw[t] && ss[t + 1] == ss[t];
  const uint64_t w = desc ? ~sw[t] : sw[t];
  head[t] = h ? 1u : 0u;
  cont[t] = ((w & 0xFF) == 8 && (!h || next_same)) ? 1u : 0u;
}
__global__ void k_next_items(const uint32_t* __restrict__ head, const uint32_t* __restrict__ cont, const uint64_t* __restrict__ hoff,
                             const uint64_t* __restrict__ coff, const uint32_t* __restrict__ pos, uint32_t k, uint32_t* __restrict__ pos_out,
                             uint32_t* __restrict__ seg_out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= k || !cont[t]) return;
  const uint64_t d = coff[t];
  pos_out[d] = pos ? pos[t] : t;
  seg_out[d] = (uint32_t)(hoff[t] + head[t] - 1);
}

__global__ void k_scatter_spans(const uint32_t* __restrict__ idx, uint32_t mk, const uint32_t* __restrict__ len_in, const uint64_t* __restrict__ src_in,
                                uint32_t* __restrict__ len, uint64_t* __restrict__ src) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < mk) { len[idx[t]] = len_in[t]; src[idx[t]] = src_in[t]; }
}

inline unsigned blocks(uint64_t n, unsigned t) { return (unsigned)((n + t - 1) / t); }

struct Sorter {
  cudaStream_t s;
  DevBuf counts, offs, scan_tmp, orand;
  unsigned long long* h_orand = nullptr;
  uint32_t passes = 0;
  // Stable sort of (key, val)[0..k) by key; the result is in (key, val) on return (the alt buffers are scratch).
  int sort(uint64_t*& key, uint32_t*& val, uint64_t*& key_alt, uint32_t*& val_alt, uint32_t k) {
    if (k < 2) return FEI_OK;
    const unsigned long long init[2] = {0ull, ~0ull};
    FEI_CUDA(cudaMemcpyAsync(orand.p, init, 16, cudaMemcpyHostToDevice, s));
    k_or_and<<<std::min(blocks(k, 256), 1024u), 256, 0, s>>>(key, k, orand.as<unsigned long long>());
    FEI_CUDA(cudaMemcpyAsync(h_orand, orand.p, 16, cudaMemcpyDeviceToHost, s));
    FEI_CUDA(cudaStreamSynchronize(s));
    const uint64_t diff = h_orand[0] ^ h_orand[1];
    const uint32_t nb = blocks(k, kSortTile);
    for (int sh = 0; sh < 64; sh += 8) {
      if (!((diff >> sh) & 0xFF)) continue;
      k_digit_hist<<<nb, kSortThreads, 0, s>>>(key, k, sh, nb, counts.as<uint32_t>());
      FEI_TRY(exclusive_scan_u32_u64(counts.as<uint32_t>(), (uint64_t)nb * 256, offs.as<uint64_t>(), scan_tmp, s));
      k_digit_scatter<<<nb, kSortThreads, 0, s>>>(key, val, k, sh, nb, offs.as<uint64_t>(), key_alt, val_alt);
      std::swap(key, key_alt); std::swap(val, val_alt);
      ++passes;
    }
    FEI_CUDA(cudaGetLastError());
    return FEI_OK;
  }
};

bool is_string_source(uint32_t s) {
  return s == FEI_SORT_SLOT || s == FEI_SORT_NAME || s == FEI_SORT_NAME_UID || s == FEI_SORT_NAME_HOST || s == FEI_SORT_BODY || s == FEI_SORT_NONE;
}
bool uses_names(const fei_sort_spec* sp) {
  const uint32_t s = sp->source == FEI_SORT_SLOT ? sp->fallback : sp->source;
  return s == FEI_SORT_NAME || s == FEI_SORT_NAME_UID || s == FEI_SORT_NAME_HOST;
}
}  // namespace
}  // namespace fei

using namespace fei;

extern "C" int fei_sort_rows(fei_corpus* const* corpora, uint32_t n_corpora, const uint32_t* row_corpus, const uint64_t* row_rec, uint64_t m,
                             const fei_sort_spec* spec, int descending, uint64_t first, uint64_t count, uint64_t* out, fei_sort_info* info) {
  if (!spec || (m && (!corpora || !n_corpora || !row_corpus || !row_rec))) { set_error("null argument"); return FEI_E_BADARG; }
  const uint32_t src = spec->source;
  if (src > FEI_SORT_KEYS) { set_error("unknown sort source %u", src); return FEI_E_BADARG; }
  if (src == FEI_SORT_SLOT && (!spec->prog || (spec->fallback != FEI_SORT_NONE && spec->fallback != FEI_SORT_NAME_UID && spec->fallback != FEI_SORT_NAME_HOST))) {
    set_error("a header sort needs a program and a fallback of none / unique_id / hostname"); return FEI_E_BADARG;
  }
  if (src == FEI_SORT_KEYS && m && !spec->keys) { set_error("FEI_SORT_KEYS without keys"); return FEI_E_BADARG; }
  if (m >= 0xFFFFFFFFull) { set_error("at most 2^32 - 2 rows"); return FEI_E_BADARG; }
  const uint64_t lo = std::min(first, m), n_out = std::min(count, m - lo);
  if (n_out && !out) { set_error("null output"); return FEI_E_BADARG; }
  for (uint32_t k = 0; k < n_corpora; ++k) if (!corpora[k]) { set_error("null corpus"); return FEI_E_BADARG; }
  for (uint64_t i = 0; i < m; ++i) if (row_corpus[i] >= n_corpora) { set_error("row %llu names corpus %u of %u", (unsigned long long)i, row_corpus[i], n_corpora); return FEI_E_BADARG; }

  // every distinct corpus locked, in address order (deadlock-free against any other caller doing the same)
  std::vector<fei_corpus*> uniq(corpora, corpora + (m ? n_corpora : 0));
  std::sort(uniq.begin(), uniq.end());
  uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
  std::vector<std::unique_lock<std::mutex>> locks;
  for (fei_corpus* c : uniq) locks.emplace_back(c->mu);
  FEI_TRY(require_ready());
  if (info) memset(info, 0, sizeof(*info));
  if (m == 0) return FEI_OK;
  for (fei_corpus* c : uniq) if (!c->loaded) { set_error("corpus not loaded"); return FEI_E_STATE; }
  for (uint64_t i = 0; i < m; ++i) {
    const fei_corpus* c = corpora[row_corpus[i]];
    if (row_rec[i] >= c->n) { set_error("row %llu: record %llu out of range", (unsigned long long)i, (unsigned long long)row_rec[i]); return FEI_E_BADARG; }
    if (uses_names(spec) && !c->name.p) { set_error("corpus has no file names"); return FEI_E_BADARG; }
  }

  cudaStream_t s = ctx().stream;
  const uint32_t mm = (uint32_t)m;
  std::vector<SrcPtrs> hp(n_corpora);
  for (uint32_t k = 0; k < n_corpora; ++k) {
    fei_corpus* c = corpora[k];
    hp[k] = {c->hdr.as<uint8_t>(), c->name.as<uint8_t>(), c->name_off.as<uint64_t>(), c->name_spans.as<uint16_t>(), c->tiles.as<uint8_t>(),
             c->grp_base.as<uint64_t>(), c->grp_len.as<uint32_t>(), c->rec_pos.as<uint32_t>(), c->ts.as<int64_t>(), c->wall.as<int64_t>(),
             c->flags8.as<uint64_t>()};
  }
  DevBuf d_cp, d_rc, d_rr, d_keys, d_kind, d_off, d_len, d_order, d_pos[2], d_seg[2], d_w0, d_key[2], d_val[2], d_tmp, d_sw, d_ss, d_head, d_cont, d_hoff, d_coff;
  Sorter so; so.s = s;
  FEI_TRY(d_cp.alloc(sizeof(SrcPtrs) * n_corpora)); FEI_TRY(d_rc.alloc(m * 4)); FEI_TRY(d_rr.alloc(m * 8)); FEI_TRY(d_order.alloc(m * 4));
  FEI_TRY(d_w0.alloc(m * 8)); FEI_TRY(d_key[0].alloc(m * 8)); FEI_TRY(d_key[1].alloc(m * 8)); FEI_TRY(d_val[0].alloc(m * 4)); FEI_TRY(d_val[1].alloc(m * 4));
  FEI_TRY(d_tmp.alloc(m * 4)); FEI_TRY(d_sw.alloc(m * 8)); FEI_TRY(d_ss.alloc(m * 4));
  FEI_TRY(so.counts.alloc((uint64_t)blocks(m, kSortTile) * 256 * 4)); FEI_TRY(so.offs.alloc(((uint64_t)blocks(m, kSortTile) * 256 + 1) * 8)); FEI_TRY(so.orand.alloc(16));
  unsigned long long orand_host[2];
  so.h_orand = orand_host;
  FEI_CUDA(cudaMemcpyAsync(d_cp.p, hp.data(), sizeof(SrcPtrs) * n_corpora, cudaMemcpyHostToDevice, s));
  FEI_CUDA(cudaMemcpyAsync(d_rc.p, row_corpus, m * 4, cudaMemcpyHostToDevice, s));
  FEI_CUDA(cudaMemcpyAsync(d_rr.p, row_rec, m * 8, cudaMemcpyHostToDevice, s));
  if (src == FEI_SORT_KEYS) { FEI_TRY(d_keys.alloc(m * 8)); FEI_CUDA(cudaMemcpyAsync(d_keys.p, spec->keys, m * 8, cudaMemcpyHostToDevice, s)); }

  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  FEI_CUDA(cudaEventCreate(&ev0)); FEI_CUDA(cudaEventCreate(&ev1));
  struct EvFree { cudaEvent_t a, b; ~EvFree() { cudaEventDestroy(a); cudaEventDestroy(b); } } evf{ev0, ev1};
  FEI_CUDA(cudaEventRecord(ev0, s));

  const bool strings = is_string_source(src);
  if (strings) {
    FEI_TRY(d_kind.alloc(m)); FEI_TRY(d_off.alloc(m * 8)); FEI_TRY(d_len.alloc(m * 4));
    DevBuf slot_len, slot_src;
    if (src == FEI_SORT_SLOT) {                              // the header value's span, per corpus (the key dictionary is per corpus)
      FEI_TRY(slot_len.alloc(m * 4)); FEI_TRY(slot_src.alloc(m * 8));
      for (uint32_t k = 0; k < n_corpora; ++k) {
        std::vector<uint32_t> idx; std::vector<uint64_t> rec;
        for (uint64_t i = 0; i < m; ++i) if (row_corpus[i] == k) { idx.push_back((uint32_t)i); rec.push_back(row_rec[i]); }
        if (idx.empty()) continue;
        const uint32_t mk = (uint32_t)idx.size();
        DevBuf d_idx, d_rec, l_k, s_k;
        FEI_TRY(d_idx.alloc(mk * 4ull)); FEI_TRY(d_rec.alloc(mk * 8ull)); FEI_TRY(l_k.alloc(mk * 4ull)); FEI_TRY(s_k.alloc(mk * 8ull));
        FEI_CUDA(cudaMemcpyAsync(d_idx.p, idx.data(), mk * 4ull, cudaMemcpyHostToDevice, s));
        FEI_CUDA(cudaMemcpyAsync(d_rec.p, rec.data(), mk * 8ull, cudaMemcpyHostToDevice, s));
        FEI_TRY(slot_spans_rows(corpora[k], spec->prog, spec->prog_len, d_rec.as<uint64_t>(), mk, l_k.as<uint32_t>(), s_k.as<uint64_t>(), s));
        k_scatter_spans<<<blocks(mk, 256), 256, 0, s>>>(d_idx.as<uint32_t>(), mk, l_k.as<uint32_t>(), s_k.as<uint64_t>(), slot_len.as<uint32_t>(), slot_src.as<uint64_t>());
        FEI_CUDA(cudaStreamSynchronize(s));                  // idx / rec are host vectors of this iteration
      }
    }
    k_str_prep<<<blocks(m, 256), 256, 0, s>>>(d_cp.as<SrcPtrs>(), d_rc.as<uint32_t>(), d_rr.as<uint64_t>(), mm, src, spec->fallback,
                                              slot_len.as<uint32_t>(), slot_src.as<uint64_t>(), d_kind.as<uint8_t>(), d_off.as<uint64_t>(), d_len.as<uint32_t>());
    FEI_CUDA(cudaStreamSynchronize(s));                      // slot_len / slot_src go out of scope
  }

  // order = identity; round 0 sorts every row (pos / seg == nullptr: item j is position j, one segment)
  std::vector<uint32_t> iota(m);
  for (uint32_t i = 0; i < mm; ++i) iota[i] = i;
  FEI_CUDA(cudaMemcpyAsync(d_order.p, iota.data(), m * 4, cudaMemcpyHostToDevice, s));
  uint32_t k = mm, rounds = 0;
  uint64_t refined = 0;
  uint32_t* pos = nullptr; uint32_t* seg = nullptr;
  int cur = 0;
  for (uint32_t round = 0; k > 0; ++round) {
    ++rounds;
    if (round) refined += k;
    uint64_t* key = d_key[0].as<uint64_t>(); uint64_t* key_alt = d_key[1].as<uint64_t>();
    uint32_t* val = d_val[0].as<uint32_t>(); uint32_t* val_alt = d_val[1].as<uint32_t>();
    k_words<<<blocks(k, 256), 256, 0, s>>>(d_cp.as<SrcPtrs>(), d_rc.as<uint32_t>(), d_rr.as<uint64_t>(), d_keys.as<uint64_t>(), src, d_kind.as<uint8_t>(),
                                           d_off.as<uint64_t>(), d_len.as<uint32_t>(), d_order.as<uint32_t>(), pos, k, round, descending ? 1 : 0,
                                           d_w0.as<uint64_t>(), key, val);
    FEI_TRY(so.sort(key, val, key_alt, val_alt, k));
    if (seg) {                                               // then stably by segment: equal words stay in the order just made
      k_seg_keys<<<blocks(k, 256), 256, 0, s>>>(seg, val, k, key);
      FEI_TRY(so.sort(key, val, key_alt, val_alt, k));
    }
    k_apply_gather<<<blocks(k, 256), 256, 0, s>>>(val, k, d_order.as<uint32_t>(), pos, d_w0.as<uint64_t>(), seg, d_tmp.as<uint32_t>(), d_sw.as<uint64_t>(), d_ss.as<uint32_t>());
    k_apply_scatter<<<blocks(k, 256), 256, 0, s>>>(d_tmp.as<uint32_t>(), k, pos, d_order.as<uint32_t>());
    if (!strings) break;
    if (!d_head.p) {
      FEI_TRY(d_head.alloc(m * 4)); FEI_TRY(d_cont.alloc(m * 4)); FEI_TRY(d_hoff.alloc((m + 1) * 8)); FEI_TRY(d_coff.alloc((m + 1) * 8));
      for (int b = 0; b < 2; ++b) { FEI_TRY(d_pos[b].alloc(m * 4)); FEI_TRY(d_seg[b].alloc(m * 4)); }
    }
    k_runs<<<blocks(k, 256), 256, 0, s>>>(d_sw.as<uint64_t>(), d_ss.as<uint32_t>(), k, descending ? 1 : 0, d_head.as<uint32_t>(), d_cont.as<uint32_t>());
    FEI_TRY(exclusive_scan_u32_u64(d_head.as<uint32_t>(), k, d_hoff.as<uint64_t>(), so.scan_tmp, s));
    FEI_TRY(exclusive_scan_u32_u64(d_cont.as<uint32_t>(), k, d_coff.as<uint64_t>(), so.scan_tmp, s));
    uint32_t* npos = d_pos[cur].as<uint32_t>(); uint32_t* nseg = d_seg[cur].as<uint32_t>();
    k_next_items<<<blocks(k, 256), 256, 0, s>>>(d_head.as<uint32_t>(), d_cont.as<uint32_t>(), d_hoff.as<uint64_t>(), d_coff.as<uint64_t>(), pos, k, npos, nseg);
    uint64_t next = 0;
    FEI_CUDA(cudaMemcpyAsync(&next, d_coff.as<uint64_t>() + k, 8, cudaMemcpyDeviceToHost, s));
    FEI_CUDA(cudaStreamSynchronize(s));
    pos = npos; seg = nseg; cur ^= 1;
    k = (uint32_t)next;
  }
  FEI_CUDA(cudaEventRecord(ev1, s));
  std::vector<uint32_t> page(n_out);
  if (n_out) FEI_CUDA(cudaMemcpyAsync(page.data(), d_order.as<uint32_t>() + lo, n_out * 4, cudaMemcpyDeviceToHost, s));
  FEI_CUDA(cudaStreamSynchronize(s));
  FEI_CUDA(cudaGetLastError());
  for (uint64_t t = 0; t < n_out; ++t) out[t] = page[t];
  if (info) {
    info->rounds = rounds; info->radix_passes = so.passes; info->refined_rows = refined;
    FEI_CUDA(cudaEventElapsedTime(&info->ms, ev0, ev1));
  }
  return FEI_OK;
}
