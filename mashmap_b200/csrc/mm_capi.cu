/*
 * mm_capi.cu -- implementation of the C ABI declared in include/mashmap_b200.h.
 *
 * Owns the device context: the index blob (one arena, see mm_internal.h), the per-batch buffers,
 * the stream and the stage timers, and drives K1 (mm_sketch.cu) -> K2 (mm_l1.cu) -> K3 (mm_l2.cu).
 * There is no CPU implementation behind any entry point: without a usable sm_100 device every call
 * fails with MM_ENODEVICE.
 */
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "mm_index_build.h"
#include "mm_internal.h"
#include <chrono>

static thread_local std::string g_create_error;

namespace {

int fail(mm_ctx *c, int code, const char *fmt, ...);

/* A device array that frees itself: the context's batch buffers and the temporaries of the index builders. */
template <typename T>
struct dev_array {
  T *p = nullptr;
  uint64_t cap = 0; /* elements */
  dev_array() = default;
  dev_array(const dev_array &) = delete;
  dev_array &operator=(const dev_array &) = delete;
  ~dev_array() { release(); }
  void release() { cudaFree(p); p = nullptr; cap = 0; }
  /* room for `need` elements: kept if it has them, else replaced (contents lost) by `new_cap` elements, *fresh = true.
   * The capacity changes only once the allocation has succeeded, and a failed one is not left as the last error. */
  int reserve(mm_ctx *c, uint64_t need, uint64_t new_cap, bool *fresh = nullptr)
  {
    if (fresh) *fresh = false;
    if (p && need <= cap) return MM_OK;
    release();
    const cudaError_t e = cudaMalloc((void **)&p, new_cap * sizeof(T));
    if (e != cudaSuccess) {
      p = nullptr;
      cudaGetLastError();
      return fail(c, e == cudaErrorMemoryAllocation ? MM_ENOMEM : MM_ECUDA, "cannot allocate %llu bytes of device memory: %s",
                  (unsigned long long)(new_cap * sizeof(T)), cudaGetErrorString(e));
    }
    cap = new_cap;
    if (fresh) *fresh = true;
    return MM_OK;
  }
};

/* the context's timing events (mm_last_stage_ms, mm_last_pack_ms); EV_BEGIN is in front of K0 (pack) / K1, EV_PREP_* around
 * the L2 record-preparation kernel */
enum stage_event { EV_BEGIN, EV_K1_BEGIN, EV_K1_END, EV_K2_END, EV_K3_BEGIN, EV_K3_END, EV_PREP_BEGIN, EV_PREP_END,
                   EV_H2D_BEGIN, EV_H2D_END, EV_D2H_BEGIN, EV_D2H_END, EV_COUNT };
struct event_set {
  cudaEvent_t ev[EV_COUNT] = {};
  event_set() = default;
  event_set(const event_set &) = delete;
  event_set &operator=(const event_set &) = delete;
  ~event_set() { for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e); }
  cudaEvent_t operator[](stage_event i) const { return ev[i]; }
};

constexpr uint32_t L2_LOCI_PER_CAND = 2; /* fixed locus slots per candidate of the stream kernels; more -> general kernel */

} // namespace

struct mm_ctx {
  int device = -1;
  int sm_count = 0;
  mm_params params{};
  cudaStream_t stream = nullptr;
  std::string error;
  uint64_t launches = 0;
  uint64_t diag[8] = {0}; /* mm_ctx_diag: how often the rare paths ran (cumulative) */

  /* index blob */
  unsigned char *blob = nullptr;
  uint64_t blob_bytes = 0;
  bool blob_owned = false;
  bool blob_ready = false;
  mm_blob_header hdr{};
  mm_dev_index ix{};
  std::vector<int32_t> cutoffs, min_hits;

  /* batch */
  dev_array<uint8_t> d_bases; uint64_t n_bases = 0;
  dev_array<uint8_t> d_packed; /* nibbles */
  mm_built_index built{}; /* lookup arrays of an index built on the device, kept for mm_index_download (keep_lookup) */
  bool built_kept = false;
  bool batch_is_ascii = false; /* the resident batch came in as text: K0 (pack) runs in front of K1 */
  float pack_ms = 0;
  dev_array<mm_segment> d_segs; uint64_t n_segs = 0;
  dev_array<uint64_t> d_sk_hash, d_sk_val; dev_array<int2> d_sk_pos; dev_array<int8_t> d_sk_strand;
  dev_array<mm_segment_result> d_seg_res;
  dev_array<uint32_t> d_sk_reject;
  int sk_mode = 0; /* 0 = fast sketch kernel + general kernel over its rejects; 1 = general kernel only (MM_SKETCH_TABLE=1) */
  dev_array<mm_l1_candidate> d_cands;
  dev_array<mm_l2_locus> d_loci;
  dev_array<uint32_t> d_counters;
  bool blocking_wait = false;       /* MM_BLOCKING_WAIT=1: host waits block on an event instead of spinning (experiment) */
  cudaEvent_t ev_wait = nullptr;
  const mm_ctx *share_src = nullptr; /* mm_ctx_share_index: the context whose index image this one reads */
  mm_phase_hook hook = nullptr;
  void *hook_user = nullptr;
  uint32_t *h_pub = nullptr; /* pinned, device-mapped: kernels publish counters here (no copy engine involved) */
  dev_array<uint64_t> d_scratch; uint64_t scratch_slice = 0; uint64_t scratch_pool = 0;
  uint64_t l1_pool0 = 32ULL << 20; /* interval points the bump pool holds at first (grown on demand; MM_L1_POOL_ELEMS) */
  uint32_t l1_grid = 0;
  uint64_t n_cands = 0, n_loci = 0;
  /* per-candidate L2 work areas, grown together: l2_cand_cap is recorded once all four are allocated */
  dev_array<mm_l2_range> d_l2_ranges; dev_array<uint64_t> d_l2_rec_off; uint64_t l2_cand_cap = 0;
  dev_array<uint8_t> d_scan_tmp;
  dev_array<uint8_t> d_l2_order; /* work area of the candidate ordering (mm_launch_l2_order) */
  dev_array<uint2> d_l2_recs;
  dev_array<uint32_t> d_l1_slow;
  int l1_warp = 1; /* 1 = warp-per-segment fast path + CTA path for big segments; 0 = CTA path only (MM_L1_CTA=1) */
  int l2_mode = 1; /* 1 = stream kernels (mm_l2_stream.cu), 0 = general kernel only (MM_L2_GENERAL=1) */
  bool batch_mapped = false;

  event_set ev;
  float stage_ms[8]{};
};

namespace {

int fail(mm_ctx *c, int code, const char *fmt, ...)
{
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->error = buf; else g_create_error = buf;
  return code;
}

#define CU(c, call)                                                                              \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return fail(c, e_ == cudaErrorMemoryAllocation ? MM_ENOMEM : MM_ECUDA, "%s: %s", #call,    \
                  cudaGetErrorString(e_));                                                       \
  } while (0)

uint64_t align_up(uint64_t x, uint64_t a) { return (x + a - 1) / a * a; }

void resolve_index(mm_ctx *c)
{
  const mm_blob_header &h = c->hdr;
  unsigned char *b = c->blob;
  mm_dev_index &ix = c->ix;
  ix.idx_hash = (const uint64_t *)(b + h.off_idx_hash);
  ix.idx_wpos = (const int32_t *)(b + h.off_idx_wpos);
  ix.idx_wend = (const int32_t *)(b + h.off_idx_wend);
  ix.idx_strand = (const int8_t *)(b + h.off_idx_strand);
  ix.contig_start = (const uint64_t *)(b + h.off_contig_start);
  ix.idx2_hash = (const uint64_t *)(b + h.off_idx2_hash);
  ix.idx2_wend = (const int32_t *)(b + h.off_idx2_wend);
  ix.tab = (const mm_tab_slot *)(b + h.off_tab);
  ix.pts = (const uint64_t *)(b + h.off_pts);
  ix.contig_len = (const int32_t *)(b + h.off_contig_len);
  ix.contig_name_id = (const int32_t *)(b + h.off_contig_name_id);
  ix.contig_group = (const int32_t *)(b + h.off_contig_group);
  ix.cutoffs = (const int32_t *)(b + h.off_cutoffs);
  ix.min_hits = (const int32_t *)(b + h.off_min_hits);
  ix.n_minmers = h.n_minmers;
  ix.n_contigs = h.n_contigs;
  ix.tab_log2 = h.tab_log2;
  ix.n_cutoffs = h.n_cutoffs;
  ix.n_min_hits = h.n_min_hits;
}

constexpr uint64_t TABLE_REGION_BYTES = 64 * 1024; /* room reserved for each of cutoffs / min_hits */

int write_tables(mm_ctx *c)
{
  if (!c->blob || c->cutoffs.empty() || c->min_hits.empty()) return MM_OK;
  if (c->cutoffs.size() * 4 > TABLE_REGION_BYTES || c->min_hits.size() * 4 > TABLE_REGION_BYTES)
    return fail(c, MM_EINVAL, "lookup tables too large");
  c->hdr.n_cutoffs = (int32_t)c->cutoffs.size();
  c->hdr.n_min_hits = (int32_t)c->min_hits.size();
  CU(c, cudaMemcpyAsync(c->blob + c->hdr.off_cutoffs, c->cutoffs.data(), c->cutoffs.size() * 4, cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaMemcpyAsync(c->blob + c->hdr.off_min_hits, c->min_hits.data(), c->min_hits.size() * 4, cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaMemcpyAsync(c->blob, &c->hdr, sizeof(c->hdr), cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  resolve_index(c);
  return MM_OK;
}

/* The index image's layout (mm_internal.h): the header, then each region at the next 256-byte boundary. */
mm_blob_header blob_layout(uint64_t n_minmers, uint64_t n_keys, uint64_t n_points, int32_t n_contigs)
{
  mm_blob_header h{};
  h.magic = MM_BLOB_MAGIC;
  h.n_minmers = n_minmers; h.n_keys = n_keys; h.n_points = n_points;
  h.n_contigs = n_contigs;
  h.tab_log2 = 4;
  while ((1ULL << h.tab_log2) < 2 * n_keys + 2) h.tab_log2++;
  uint64_t o = align_up(sizeof(mm_blob_header), 256);
  auto place = [&](uint64_t bytes) { uint64_t at = o; o = align_up(o + bytes, 256); return at; };
  h.off_idx_hash = place((n_minmers + 1) * 8);
  h.off_idx_wpos = place((n_minmers + 1) * 4);
  h.off_idx_wend = place((n_minmers + 1) * 4);
  h.off_idx_strand = place(n_minmers + 1);
  h.off_contig_start = place(((uint64_t)n_contigs + 1) * 8);
  h.off_idx2_hash = place((n_minmers + 1) * 8);
  h.off_idx2_wend = place((n_minmers + 1) * 4);
  h.off_tab = place((1ULL << h.tab_log2) * sizeof(mm_tab_slot));
  h.off_pts = place((n_points + 1) * 8);
  h.off_contig_len = place((uint64_t)n_contigs * 4);
  h.off_contig_name_id = place((uint64_t)n_contigs * 4);
  h.off_contig_group = place((uint64_t)n_contigs * 4);
  h.off_cutoffs = place(TABLE_REGION_BYTES);
  h.off_min_hits = place(TABLE_REGION_BYTES);
  h.total_bytes = o;
  return h;
}

/* the context no longer has an index image; it is freed if the context owns it */
void release_blob(mm_ctx *c)
{
  if (c->blob && c->blob_owned) { cudaSetDevice(c->device); cudaFree(c->blob); }
  c->blob = nullptr; c->blob_bytes = 0; c->blob_ready = false;
}

/* a new index image of h.total_bytes bytes, owned by the context, in place of the old one; it is not ready until
 * finish_blob, and a blob_guard frees it on every return before that */
int replace_blob(mm_ctx *c, const mm_blob_header &h)
{
  release_blob(c);
  const cudaError_t e = cudaMalloc((void **)&c->blob, h.total_bytes);
  if (e != cudaSuccess) {
    c->blob = nullptr;
    cudaGetLastError();
    return fail(c, e == cudaErrorMemoryAllocation ? MM_ENOMEM : MM_ECUDA, "cannot allocate the index image (%llu bytes): %s",
                (unsigned long long)h.total_bytes, cudaGetErrorString(e));
  }
  c->blob_bytes = h.total_bytes; c->blob_owned = true; c->hdr = h; c->share_src = nullptr;
  return MM_OK;
}

struct blob_guard {
  mm_ctx *c;
  ~blob_guard() { if (!c->blob_ready) release_blob(c); }
};

/* the last writes of an index image: the contig tables (name ids default to -1, groups to 0) and the header; then the
 * image is ready and the threshold tables go in */
int finish_blob(mm_ctx *c, const int32_t *contig_len, const int32_t *contig_name_id, const int32_t *contig_group)
{
  const mm_blob_header &h = c->hdr;
  const size_t n = (size_t)h.n_contigs;
  std::vector<int32_t> tmp(n, -1);
  CU(c, cudaMemcpyAsync(c->blob + h.off_contig_len, contig_len, n * 4, cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaMemcpyAsync(c->blob + h.off_contig_name_id, contig_name_id ? contig_name_id : tmp.data(), n * 4, cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaStreamSynchronize(c->stream)); /* tmp is rewritten below */
  std::fill(tmp.begin(), tmp.end(), 0);
  CU(c, cudaMemcpyAsync(c->blob + h.off_contig_group, contig_group ? contig_group : tmp.data(), n * 4, cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaMemcpyAsync(c->blob, &c->hdr, sizeof(c->hdr), cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  resolve_index(c);
  c->blob_ready = true;
  return write_tables(c);
}

/* wait for the context's stream. Default: cudaStreamSynchronize (spins, lowest latency). With MM_BLOCKING_WAIT=1 the
 * thread sleeps on a blocking event instead -- for hosts with fewer usable CPUs than pipeline threads (DESIGN section 9). */
cudaError_t wait_stream(mm_ctx *c)
{
  if (!c->blocking_wait) return cudaStreamSynchronize(c->stream);
  const cudaError_t e = cudaEventRecord(c->ev_wait, c->stream);
  return e != cudaSuccess ? e : cudaEventSynchronize(c->ev_wait);
}

int check_ready(mm_ctx *c)
{
  if (!c) return MM_EINVAL;
  if (c->share_src) { /* follow the owner: its image may have been replaced since (new upload / adopted blob / new tables) */
    const mm_ctx *s = c->share_src;
    if (c->blob != s->blob || c->blob_bytes != s->blob_bytes || c->hdr.n_cutoffs != s->hdr.n_cutoffs ||
        c->hdr.n_min_hits != s->hdr.n_min_hits || c->blob_ready != s->blob_ready) {
      c->blob = s->blob; c->blob_bytes = s->blob_bytes; c->hdr = s->hdr; c->blob_ready = s->blob_ready;
      resolve_index(c);
    }
  }
  if (!c->blob_ready) return fail(c, MM_ESTATE, "reference index not uploaded");
  if (c->hdr.n_cutoffs <= 0 || c->hdr.n_min_hits <= 0) return fail(c, MM_ESTATE, "threshold tables not uploaded");
  return MM_OK;
}

int validate_segments(mm_ctx *c, const mm_segment *segs, uint64_t n_segs, uint64_t n_bases)
{
  if (n_segs >= (1ULL << 31)) return fail(c, MM_EINVAL, "too many segments in one batch");
  for (uint64_t i = 0; i < n_segs; i++) {
    const mm_segment &s = segs[i];
    if (s.length < 1 || s.length > c->params.seg_length)
      return fail(c, MM_EINVAL, "segment %llu: length %d outside [1, seg_length=%d] (unsplit reads longer than "
                  "seg_length are not supported)", (unsigned long long)i, s.length, c->params.seg_length);
    if (s.offset + (uint64_t)s.length > n_bases) return fail(c, MM_EINVAL, "segment %llu exceeds the base buffer", (unsigned long long)i);
  }
  return MM_OK;
}

/* batch buffers that do not depend on the input format */
int prepare_batch_buffers(mm_ctx *c, uint64_t n_bases, uint64_t n_segs)
{
  int rc;
  /* nibbles: n_bases/2 rounded up to 8-byte groups of 16 bases, + 256 so that the 16-byte-granular bulk copies of the
   * sketch kernel never leave the allocation */
  const uint64_t pbytes = (n_bases + 15) / 16 * 8 + 256;
  bool fresh = false;
  if ((rc = c->d_packed.reserve(c, pbytes, pbytes, &fresh))) return rc;
  if (fresh) CU(c, cudaMemsetAsync(c->d_packed.p, 0x88, c->d_packed.cap, c->stream));
  const uint64_t n = n_segs * (uint64_t)c->params.sketch_size + 1;
  if ((rc = c->d_segs.reserve(c, n_segs + 1, n_segs + 1)) || (rc = c->d_sk_hash.reserve(c, n, n)) ||
      (rc = c->d_sk_val.reserve(c, n, n)) || (rc = c->d_sk_pos.reserve(c, n, n)) || (rc = c->d_sk_strand.reserve(c, n, n)) ||
      (rc = c->d_seg_res.reserve(c, n_segs + 1, n_segs + 1)) || (rc = c->d_sk_reject.reserve(c, n_segs + 1, n_segs + 1)) ||
      (rc = c->d_counters.reserve(c, 16, 16)))
    return rc;
  return MM_OK;
}

/* host -> device copy of `bytes` bytes, in <= 16 MiB pieces when a phase hook is installed (MM_PHASE_UPLOAD_CHUNK) */
int copy_in(mm_ctx *c, uint8_t *dst, const void *src, uint64_t bytes)
{
  if (!c->hook) {
    CU(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return MM_OK;
  }
  const uint64_t CH = 16ULL << 20;
  for (uint64_t at = 0; at < bytes; at += CH) {
    const uint64_t n = std::min(CH, bytes - at);
    c->hook(c->hook_user, MM_PHASE_UPLOAD_CHUNK, 1);
    cudaError_t e = cudaMemcpyAsync(dst + at, (const uint8_t *)src + at, n, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = wait_stream(c);
    c->hook(c->hook_user, MM_PHASE_UPLOAD_CHUNK, 0);
    CU(c, e);
  }
  return MM_OK;
}

/* packed != 0: `bases` holds nibbles (mm_batch_upload_packed) */
int upload_batch(mm_ctx *c, const void *bases, uint64_t n_bases, const mm_segment *segs, uint64_t n_segs, int packed)
{
  int rc = validate_segments(c, segs, n_segs, n_bases);
  if (rc) return rc;
  CU(c, cudaSetDevice(c->device));
  if ((rc = prepare_batch_buffers(c, n_bases, n_segs))) return rc;
  CU(c, cudaEventRecord(c->ev[EV_H2D_BEGIN], c->stream));
  if (packed) {
    const uint64_t pbytes = (n_bases + 1) / 2;
    if ((rc = copy_in(c, c->d_packed.p, bases, pbytes))) return rc;
    CU(c, cudaMemsetAsync(c->d_packed.p + pbytes, 0x88, 64, c->stream));
    if (n_bases & 1) { /* the unused high nibble of the last byte is whatever the caller had there: irrelevant (never a k-mer) */ }
  } else {
    if ((rc = c->d_bases.reserve(c, n_bases + 256, n_bases + 256))) return rc;
    if ((rc = copy_in(c, c->d_bases.p, bases, n_bases))) return rc;
    CU(c, cudaMemsetAsync(c->d_bases.p + n_bases, 'N', 256, c->stream));
  }
  CU(c, cudaMemcpyAsync(c->d_segs.p, segs, n_segs * sizeof(mm_segment), cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaEventRecord(c->ev[EV_H2D_END], c->stream));
  c->n_bases = n_bases;
  c->n_segs = n_segs;
  c->batch_is_ascii = !packed;
  c->batch_mapped = false;
  return MM_OK;
}

/* K0 in front of K1 when the resident batch is text */
int launch_pack_if_ascii(mm_ctx *c)
{
  if (!c->batch_is_ascii) { c->pack_ms = 0; return MM_OK; }
  CU(c, mm_launch_pack_bases(c->d_bases.p, c->d_packed.p, c->n_bases, c->stream, c->sm_count));
  c->launches++;
  return MM_OK;
}

mm_dev_batch make_batch(mm_ctx *c)
{
  mm_dev_batch b{};
  b.bases = c->d_bases.p; b.packed = c->d_packed.p; b.segs = c->d_segs.p; b.n_segs = (uint32_t)c->n_segs;
  b.sk_hash = c->d_sk_hash.p; b.sk_val = c->d_sk_val.p; b.sk_pos = c->d_sk_pos.p; b.sk_strand = c->d_sk_strand.p;
  b.seg_res = c->d_seg_res.p; b.sk_reject = c->d_sk_reject.p;
  b.cands = c->d_cands.p; b.cand_cap = (uint32_t)std::min<uint64_t>(c->d_cands.cap, 0xffffffffu);
  b.loci = c->d_loci.p; b.loci_cap = (uint32_t)std::min<uint64_t>(c->d_loci.cap, 0xffffffffu);
  b.counters = c->d_counters.p;
  b.scratch = c->d_scratch.p; b.scratch_slice = c->scratch_slice; b.scratch_pool_off = c->scratch_pool;
  b.scratch_cap = c->d_scratch.cap;
  b.l2_ranges = c->d_l2_ranges.p; b.l2_rec_off = c->d_l2_rec_off.p; b.l2_recs = c->d_l2_recs.p; b.l2_recs_cap = c->d_l2_recs.cap;
  b.l2_loci_per_cand = L2_LOCI_PER_CAND;
  return b;
}

int ensure_scratch(mm_ctx *c, uint64_t pool_elems)
{
  if (c->l1_grid == 0) {
    c->l1_grid = mm_l1_grid_size(c->params, c->sm_count);
    if (c->l1_grid == 0) return fail(c, MM_ECUDA, "cannot size the L1 grid");
  }
  const uint64_t slice = 3ULL << 16; /* 65536 points per CTA slice */
  const uint64_t need = slice * c->l1_grid + pool_elems;
  if (int rc = c->d_scratch.reserve(c, need, need)) return rc;
  c->scratch_slice = slice;
  c->scratch_pool = slice * c->l1_grid;
  return MM_OK;
}

/* Small device->host readbacks do not go through a copy engine: a DMA queued while another context's batch upload
 * (hundreds of MB) is in flight waits for it. A one-warp kernel stores the words into pinned, device-mapped host memory. */
__global__ void k_publish(const uint32_t *__restrict__ src, volatile uint32_t *dst, int n)
{
  if ((int)threadIdx.x < n) dst[threadIdx.x] = src[threadIdx.x];
  __threadfence_system();
}
__global__ void k_set_u32(uint32_t *dst, uint32_t v) { *dst = v; }
/* cudaMemsetAsync of a few words may be executed by a copy engine too: zero them with a kernel */
__global__ void k_zero_words(uint32_t *dst, int n) { if ((int)threadIdx.x < n) dst[threadIdx.x] = 0; }
#define ZERO_WORDS(c, ptr, n) do { k_zero_words<<<1, 32, 0, (c)->stream>>>((uint32_t *)(ptr), (n)); (c)->launches++; CU((c), cudaGetLastError()); } while (0)

int read_words(mm_ctx *c, const void *dev, uint32_t *out, int n_words)
{
  k_publish<<<1, 32, 0, c->stream>>>((const uint32_t *)dev, c->h_pub, n_words);
  c->launches++;
  CU(c, cudaGetLastError());
  CU(c, wait_stream(c));
  for (int i = 0; i < n_words; i++) out[i] = c->h_pub[i];
  return MM_OK;
}
#define RD(c, dev, out, n) do { int rc__ = read_words((c), (dev), (out), (n)); if (rc__) return rc__; } while (0)

/* K3's general kernel (mm_l2.cu), over every candidate or (only_flagged) over the ones the stream kernels flagged, whose
 * loci it appends after the fixed slots. The counters come back in h_cnt. *grown: the locus buffer was too small and has
 * been grown; the caller runs the kernel again. */
int run_l2_general(mm_ctx *c, bool only_flagged, uint32_t *h_cnt, bool *grown)
{
  const mm_dev_batch b = make_batch(c);
  const uint32_t nc = (uint32_t)c->n_cands;
  *grown = false;
  if (only_flagged) { /* counter 1 was zeroed in front of the stream kernels */
    k_set_u32<<<1, 1, 0, c->stream>>>(c->d_counters.p + 6, nc * L2_LOCI_PER_CAND);
    c->launches++;
    CU(c, mm_launch_l2_overflow(c->params, c->ix, b, nc, c->stream, c->sm_count));
    c->launches++;
  } else {
    ZERO_WORDS(c, c->d_counters.p + 1, 1);
    ZERO_WORDS(c, c->d_counters.p + 6, 2);
    CU(c, cudaEventRecord(c->ev[EV_K3_BEGIN], c->stream));
    CU(c, mm_launch_l2(c->params, c->ix, b, nc, c->stream, c->sm_count));
    CU(c, cudaEventRecord(c->ev[EV_K3_END], c->stream));
    if (nc) c->launches++;
  }
  RD(c, c->d_counters.p, h_cnt, 16);
  if (h_cnt[1] == 2) return fail(c, MM_ECUDA, "L2 live-set overflow in the general kernel: the reference index has more than "
                                 "sketch_size+64 overlapping minmer windows at one position");
  if (h_cnt[1] == 1 || h_cnt[6] > c->d_loci.cap) {
    if (int rc = c->d_loci.reserve(c, h_cnt[6], (uint64_t)h_cnt[6] + h_cnt[6] / 4 + 1024)) return rc;
    *grown = true;
  }
  return MM_OK;
}

/* K3 fast path (mm_l2_stream.cu): ranges+scan -> records -> lane-per-candidate scan -> general kernel for the
 * candidates that need more locus slots. Returns MM_ENOMEM if the record buffer cannot be allocated. */
int run_l2_stream(mm_ctx *c, uint32_t *h_cnt)
{
  const uint64_t nc = c->n_cands;
  int rc;
  CU(c, cudaEventRecord(c->ev[EV_K3_BEGIN], c->stream));
  if (nc == 0) {
    CU(c, cudaEventRecord(c->ev[EV_K3_END], c->stream));
    CU(c, wait_stream(c));
    c->n_loci = 0;
    return MM_OK;
  }
  if (nc + 1 > c->l2_cand_cap) {
    const uint64_t cap = nc + nc / 8 + 1024;
    const uint64_t scan_bytes = mm_l2_scan_tmp_bytes((uint32_t)cap) + 256, order_bytes = mm_l2_order_bytes((uint32_t)cap);
    if ((rc = c->d_l2_ranges.reserve(c, cap, cap)) || (rc = c->d_l2_rec_off.reserve(c, cap + 1, cap + 1)) ||
        (rc = c->d_scan_tmp.reserve(c, scan_bytes, scan_bytes)) || (rc = c->d_l2_order.reserve(c, order_bytes, order_bytes)))
      return rc;
    c->l2_cand_cap = cap;
  }
  if ((rc = c->d_loci.reserve(c, nc * L2_LOCI_PER_CAND + 1024, nc * L2_LOCI_PER_CAND + nc / 8 + 4096))) return rc;
  mm_dev_batch b = make_batch(c);
  const auto tk0 = std::chrono::steady_clock::now();
  ZERO_WORDS(c, c->d_l2_rec_off.p + nc, 2);
  CU(c, mm_launch_l2_ranges(c->params, c->ix, b, (uint32_t)nc, c->d_scan_tmp.p, c->d_scan_tmp.cap, c->stream));
  uint64_t total = 0;
  RD(c, c->d_l2_rec_off.p + nc, (uint32_t *)&total, 2);
  const auto tk1 = std::chrono::steady_clock::now();
  c->stage_ms[6] = std::chrono::duration<float, std::milli>(tk1 - tk0).count(); /* host view: ranges + scan + readback */
  /* the scan's record readers run up to 2 * RING_CHUNKS + 2 records past a stream's end */
  const uint64_t want = total + total / 16 + 1024;
  if (c->d_l2_recs.reserve(c, total + 64, want))
    return fail(c, MM_ENOMEM, "cannot allocate %llu L2 operation records", (unsigned long long)want);
  for (int attempt = 0; attempt < 4; attempt++) {
    b = make_batch(c);
    ZERO_WORDS(c, c->d_counters.p + 1, 1);
    ZERO_WORDS(c, c->d_counters.p + 6, 2);
    /* the record-preparation kernel is the bandwidth-bound one: no PCIe upload next to it (MM_PHASE_L2) */
    {
      struct phase_guard { /* the hook is always closed, whatever fails in between */
        mm_ctx *c; bool open;
        explicit phase_guard(mm_ctx *cc) : c(cc), open(cc->hook != nullptr) { if (open) c->hook(c->hook_user, MM_PHASE_L2, 1); }
        void close() { if (open) { c->hook(c->hook_user, MM_PHASE_L2, 0); open = false; } }
        ~phase_guard() { close(); }
      } guard(c);
      CU(c, cudaEventRecord(c->ev[EV_PREP_BEGIN], c->stream));
      CU(c, mm_launch_l2_prep(c->params, c->ix, b, (uint32_t)nc, c->stream, c->sm_count));
      CU(c, cudaEventRecord(c->ev[EV_PREP_END], c->stream));
      if (guard.open && c->blocking_wait) CU(c, cudaEventRecord(c->ev_wait, c->stream));
      uint32_t *perm = nullptr;
      CU(c, mm_launch_l2_order(b, (uint32_t)nc, c->d_l2_order.p, c->d_l2_order.cap, &perm, c->stream));
      b.l2_perm = perm;
      CU(c, mm_launch_l2_scan(c->params, c->ix, b, (uint32_t)nc, c->stream, c->sm_count));
      /* the scan is already queued behind it: waiting for the end of the preparation kernel costs no bubble */
      if (guard.open) CU(c, cudaEventSynchronize(c->blocking_wait ? c->ev_wait : c->ev[EV_PREP_END]));
    }
    c->launches += 4; /* own kernels: ranges, prep, order keys, scan (the prefix sum and the sort are library calls, not counted) */
    RD(c, c->d_counters.p, h_cnt, 16);
    uint64_t extent = nc * L2_LOCI_PER_CAND;
    if (h_cnt[7] > 0) { /* candidates with more than L2_LOCI_PER_CAND loci: general kernel, loci appended after the fixed slots */
      c->diag[MM_DIAG_L2_GENERAL_CANDS] += h_cnt[7];
      bool grown = false;
      if ((rc = run_l2_general(c, true, h_cnt, &grown))) return rc;
      if (grown) { /* redo prep+scan+overflow */
        c->diag[MM_DIAG_L2_LOCI_REGROW]++;
        continue;
      }
      extent = h_cnt[6];
    }
    CU(c, cudaEventRecord(c->ev[EV_K3_END], c->stream));
    CU(c, wait_stream(c));
    cudaEventElapsedTime(&c->stage_ms[6], c->ev[EV_PREP_BEGIN], c->ev[EV_PREP_END]); /* k_l2_prep */
    cudaEventElapsedTime(&c->stage_ms[7], c->ev[EV_PREP_END], c->ev[EV_K3_END]);     /* k_l2_scan (+ overflow kernel) */
    c->n_loci = extent;
    return MM_OK;
  }
  return fail(c, MM_ECUDA, "locus buffer kept overflowing");
}

/* K3: the stream kernels, or the general kernel alone (MM_L2_GENERAL, large sketches, or no memory for the stream
 * kernels' records), retried alone while the locus buffer is too small (it is idempotent) */
int run_l2(mm_ctx *c)
{
  uint32_t h_cnt[16];
  if (c->l2_mode == 1) {
    const int rc = run_l2_stream(c, h_cnt);
    if (rc != MM_ENOMEM) return rc;
    /* not enough memory for the operation records: fall through to the general kernel */
  }
  for (int attempt = 0; attempt < 4; attempt++) {
    bool grown = false;
    if (int rc = run_l2_general(c, false, h_cnt, &grown)) return rc;
    if (!grown) {
      c->n_loci = h_cnt[6];
      return MM_OK;
    }
  }
  return fail(c, MM_ECUDA, "locus buffer kept overflowing");
}

/* stage_ms / pack_ms of the batch run_pipeline has just mapped */
void record_stage_times(mm_ctx *c)
{
  if (c->batch_is_ascii) cudaEventElapsedTime(&c->pack_ms, c->ev[EV_BEGIN], c->ev[EV_K1_BEGIN]);
  cudaEventElapsedTime(&c->stage_ms[0], c->ev[EV_K1_BEGIN], c->ev[EV_K1_END]);
  cudaEventElapsedTime(&c->stage_ms[1], c->ev[EV_K1_END], c->ev[EV_K2_END]);
  cudaEventElapsedTime(&c->stage_ms[2], c->ev[EV_K3_BEGIN], c->ev[EV_K3_END]);
  cudaEventElapsedTime(&c->stage_ms[5], c->ev[EV_BEGIN], c->ev[EV_K3_END]); /* first launch -> last kernel end, incl. host gaps */
}

/* K1 -> K2 -> K3 on the resident batch, growing output buffers and retrying on overflow */
int run_pipeline(mm_ctx *c)
{
  int rc = check_ready(c);
  if (rc) return rc;
  CU(c, cudaSetDevice(c->device));
  const uint64_t n_segs = c->n_segs;
  if ((rc = c->d_cands.reserve(c, 2 * n_segs + 1024, 2 * n_segs + 1024)) ||
      (rc = c->d_loci.reserve(c, 2 * c->d_cands.cap, 2 * c->d_cands.cap)) ||
      (rc = ensure_scratch(c, c->d_scratch.cap ? c->d_scratch.cap - c->scratch_pool : c->l1_pool0)) ||
      (rc = c->d_l1_slow.reserve(c, n_segs + 1, n_segs + n_segs / 8 + 1024)))
    return rc;

  uint32_t h_cnt[16];
  for (int attempt = 0; attempt < 6; attempt++) {
    mm_dev_batch b = make_batch(c);
    ZERO_WORDS(c, c->d_counters.p, 16);
    CU(c, cudaEventRecord(c->ev[EV_BEGIN], c->stream));
    if ((rc = launch_pack_if_ascii(c))) return rc;
    CU(c, cudaEventRecord(c->ev[EV_K1_BEGIN], c->stream));
    CU(c, mm_launch_sketch(c->params, b, c->stream, c->sm_count, c->sk_mode));
    CU(c, cudaEventRecord(c->ev[EV_K1_END], c->stream));
    int l1_launches = 0;
    CU(c, mm_launch_l1(c->params, c->ix, b, c->stream, c->sm_count, c->d_l1_slow.p, c->l1_warp, &l1_launches));
    CU(c, cudaEventRecord(c->ev[EV_K2_END], c->stream));
    c->launches += (c->sk_mode ? 1 : 2) + (uint64_t)l1_launches;
    RD(c, c->d_counters.p, h_cnt, 16);
    const uint64_t need_cands = h_cnt[0];
    bool retry = false;
    c->diag[MM_DIAG_L1_CTA_SEGMENTS] += h_cnt[8];
    c->diag[MM_DIAG_SKETCH_GENERAL_SEGMENTS] += h_cnt[9];
    if (h_cnt[3] || need_cands > c->d_cands.cap) {
      c->diag[MM_DIAG_CAND_REGROW]++;
      if ((rc = c->d_cands.reserve(c, need_cands, need_cands + need_cands / 4 + 1024))) return rc;
      retry = true;
    }
    if (h_cnt[2]) { /* scratch pool exhausted: quadruple it */
      c->diag[MM_DIAG_L1_POOL_REGROW]++;
      if ((rc = ensure_scratch(c, (c->d_scratch.cap - c->scratch_pool) * 4))) return rc;
      retry = true;
    }
    if (retry) continue;
    c->n_cands = need_cands;
    if ((rc = run_l2(c))) return rc;
    record_stage_times(c);
    c->batch_mapped = true;
    return MM_OK;
  }
  return fail(c, MM_ECUDA, "candidate/scratch buffers kept overflowing");
}

} // namespace

extern "C" {

int mm_params_check(const mm_params *params)
{
  if (!params) return fail(nullptr, MM_EINVAL, "null params");
  if (!mm_sketch_kmer_supported(params->kmer_size))
    return fail(nullptr, MM_EINVAL, "k-mer size %d is not compiled in (8..32)", params->kmer_size);
  if (params->sketch_size < 1 || params->seg_length < params->kmer_size)
    return fail(nullptr, MM_EINVAL, "bad sketch_size / seg_length");
  if (mm_sketch_smem_bytes(params->seg_length, params->sketch_size, params->kmer_size, nullptr, nullptr) == 0)
    return fail(nullptr, MM_EINVAL, "seg_length %d / sketch_size %d exceed the shared-memory budget of the sketch kernel",
                params->seg_length, params->sketch_size);
  return MM_OK;
}

int mm_ctx_create(int device, const mm_params *params, mm_ctx **out)
{
  if (!params || !out) return fail(nullptr, MM_EINVAL, "null argument");
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return fail(nullptr, MM_ENODEVICE, "no CUDA device: %s (this library has no CPU path)", cudaGetErrorString(e));
  if (device < 0 || device >= n_dev) return fail(nullptr, MM_ENODEVICE, "device %d out of range (%d devices)", device, n_dev);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, MM_ENODEVICE, "cannot query device");
  if (prop.major != 10) return fail(nullptr, MM_ENODEVICE, "device %d is sm_%d%d; this build is sm_100a only", device, prop.major, prop.minor);
  if (int rc = mm_params_check(params)) return rc;
  mm_ctx *c = new mm_ctx();
  c->device = device;
  c->params = *params;
  c->sm_count = prop.multiProcessorCount;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return fail(nullptr, MM_ECUDA, "cannot create stream");
  }
  for (cudaEvent_t &ev : c->ev.ev) cudaEventCreate(&ev);
  if (cudaHostAlloc((void **)&c->h_pub, 256, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
    cudaStreamDestroy(c->stream);
    delete c;
    return fail(nullptr, MM_ENOMEM, "cannot allocate the pinned counter page");
  }
  if (const char *g = getenv("MM_BLOCKING_WAIT")) {
    if (g[0] == '1' && cudaEventCreateWithFlags(&c->ev_wait, cudaEventBlockingSync | cudaEventDisableTiming) == cudaSuccess)
      c->blocking_wait = true;
  }
  if (const char *g = getenv("MM_L2_GENERAL")) c->l2_mode = (g[0] == '1') ? 0 : 1; /* test hook: general kernel only */
  if (const char *g = getenv("MM_SKETCH_TABLE")) c->sk_mode = (g[0] == '1') ? 1 : 0; /* test hook: general sketch kernel only */
  if (const char *g = getenv("MM_L1_CTA")) c->l1_warp = (g[0] == '1') ? 0 : 1; /* test hook: general L1 path only */
  if (const char *g = getenv("MM_L1_POOL_ELEMS")) c->l1_pool0 = std::max<uint64_t>(1024, strtoull(g, nullptr, 10)); /* test hook: force the pool regrow */
  if (params->sketch_size > 1000) c->l2_mode = 0; /* the stream kernel packs its counters in 11 bits */
  *out = c;
  return MM_OK;
}

int mm_ctx_destroy(mm_ctx *c)
{
  if (!c) return MM_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  release_blob(c);
  mm_built_index_free(&c->built);
  if (c->h_pub) cudaFreeHost(c->h_pub);
  if (c->ev_wait) cudaEventDestroy(c->ev_wait);
  cudaStreamDestroy(c->stream);
  delete c; /* the batch buffers and the timing events go with it */
  return MM_OK;
}

const char *mm_last_error(const mm_ctx *c) { return c ? c->error.c_str() : g_create_error.c_str(); }
int mm_ctx_diag(const mm_ctx *ctx, uint64_t out[8])
{
  if (!ctx || !out) return MM_EINVAL;
  memcpy(out, ctx->diag, sizeof(ctx->diag));
  return MM_OK;
}
int mm_ctx_device(const mm_ctx *c) { return c ? c->device : -1; }
uint64_t mm_kernel_launches(const mm_ctx *c) { return c ? c->launches : 0; }

int mm_index_upload(mm_ctx *c, const mm_minmer *mi, uint64_t n_mi, const uint64_t *keys, const uint64_t *offsets,
                    uint64_t n_keys, const mm_ipoint *points, uint64_t n_points, const uint8_t *key_is_freq,
                    const int32_t *contig_len, const int32_t *contig_name_id, const int32_t *contig_group,
                    int32_t n_contigs)
{
  if (!c) return MM_EINVAL;
  if (n_contigs < 1 || !contig_len) return fail(c, MM_EINVAL, "no contigs");
  if (n_keys && (!keys || !offsets || !key_is_freq)) return fail(c, MM_EINVAL, "null lookup arrays");
  if (n_keys && offsets[n_keys] != n_points) return fail(c, MM_EINVAL, "offsets[n_keys] != n_points");
  CU(c, cudaSetDevice(c->device));
  release_blob(c);

  /* contig_start: first index entry of each contig; the index must be ordered by (seqId, wpos) */
  std::vector<uint64_t> cstart((size_t)n_contigs + 1, 0);
  {
    int32_t prev_seq = 0, prev_pos = -0x7fffffff;
    for (uint64_t i = 0; i < n_mi; i++) {
      const int32_t s = mi[i].seqId;
      if (s < 0 || s >= n_contigs) return fail(c, MM_EINVAL, "minmer %llu: seqId %d out of range", (unsigned long long)i, s);
      if (s < prev_seq || (s == prev_seq && mi[i].wpos < prev_pos))
        return fail(c, MM_EINVAL, "minmer index not sorted by (seqId, wpos) at entry %llu", (unsigned long long)i);
      if (s != prev_seq) prev_pos = -0x7fffffff;
      prev_seq = s; prev_pos = mi[i].wpos;
      cstart[(size_t)s + 1]++;
    }
    for (int32_t s = 0; s < n_contigs; s++) cstart[(size_t)s + 1] += cstart[(size_t)s];
  }
  const mm_blob_header h = blob_layout(n_mi, n_keys, n_points, n_contigs);
  const uint64_t tab_slots = 1ULL << h.tab_log2;
  int rc = replace_blob(c, h);
  if (rc) return rc;
  blob_guard guard{c}; /* every early return below also releases the temporaries (dev_array) */

  /* AoS records go up in chunks and are re-laid out on the device (SoA index, packed points, hash table) */
  {
    const uint64_t CH = 1ULL << 24;
    dev_array<uint8_t> stage;
    if ((rc = stage.reserve(c, CH * 24, CH * 24))) return rc;
    for (uint64_t at = 0; at < n_mi; at += CH) {
      const uint64_t n = std::min(CH, n_mi - at);
      CU(c, cudaMemcpyAsync(stage.p, mi + at, n * sizeof(mm_minmer), cudaMemcpyHostToDevice, c->stream));
      CU(c, mm_upload_split_minmers((const mm_minmer *)stage.p, n, (uint64_t *)(c->blob + h.off_idx_hash) + at,
                                    (int32_t *)(c->blob + h.off_idx_wpos) + at, (int32_t *)(c->blob + h.off_idx_wend) + at,
                                    (int8_t *)(c->blob + h.off_idx_strand) + at, c->stream));
      CU(c, cudaStreamSynchronize(c->stream));
    }
    CU(c, cudaMemcpyAsync(c->blob + h.off_contig_start, cstart.data(), cstart.size() * 8, cudaMemcpyHostToDevice, c->stream));
    /* the same entries per contig in wpos_end order (device sort), for the L2 stream merge */
    CU(c, mm_build_death_order((const uint64_t *)(c->blob + h.off_idx_hash), (const int32_t *)(c->blob + h.off_idx_wend),
                               (const uint64_t *)(c->blob + h.off_contig_start), n_contigs, n_mi,
                               (uint64_t *)(c->blob + h.off_idx2_hash), (int32_t *)(c->blob + h.off_idx2_wend), c->stream));
    dev_array<uint32_t> d_err;
    if ((rc = d_err.reserve(c, 1, 1))) return rc;
    CU(c, cudaMemsetAsync(d_err.p, 0, 4, c->stream));
    for (uint64_t at = 0; at < n_points; at += CH) {
      const uint64_t n = std::min(CH, n_points - at);
      CU(c, cudaMemcpyAsync(stage.p, points + at, n * sizeof(mm_ipoint), cudaMemcpyHostToDevice, c->stream));
      CU(c, mm_upload_pack_points((const mm_ipoint *)stage.p, n, n_contigs, (uint64_t *)(c->blob + h.off_pts) + at, d_err.p, c->stream));
      CU(c, cudaStreamSynchronize(c->stream));
    }
    stage.release();
    /* open-addressing table, filled on the device */
    CU(c, cudaMemsetAsync(c->blob + h.off_tab, 0, tab_slots * sizeof(mm_tab_slot), c->stream));
    if (n_keys) {
      dev_array<uint64_t> d_keys, d_offs;
      dev_array<uint8_t> d_freq;
      if ((rc = d_keys.reserve(c, n_keys, n_keys)) || (rc = d_offs.reserve(c, n_keys + 1, n_keys + 1)) ||
          (rc = d_freq.reserve(c, n_keys, n_keys)))
        return rc;
      CU(c, cudaMemcpyAsync(d_keys.p, keys, n_keys * 8, cudaMemcpyHostToDevice, c->stream));
      CU(c, cudaMemcpyAsync(d_offs.p, offsets, (n_keys + 1) * 8, cudaMemcpyHostToDevice, c->stream));
      CU(c, cudaMemcpyAsync(d_freq.p, key_is_freq, n_keys, cudaMemcpyHostToDevice, c->stream));
      CU(c, mm_upload_build_table(d_keys.p, d_offs.p, d_freq.p, n_keys, (mm_tab_slot *)(c->blob + h.off_tab), h.tab_log2, d_err.p, c->stream));
      CU(c, cudaStreamSynchronize(c->stream));
    }
    uint32_t err = 0;
    CU(c, cudaMemcpyAsync(&err, d_err.p, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (err & 1) return fail(c, MM_EINVAL, "an interval point has a bad seqId or a negative position");
    if (err & 2) return fail(c, MM_EINVAL, "a key has no or too many (>= 2^24) interval points, or offsets overflow");
    if (err & 4) return fail(c, MM_EINVAL, "duplicate key in the lookup index");
  }
  return finish_blob(c, contig_len, contig_name_id, contig_group);
}

int mm_tables_upload(mm_ctx *c, const int32_t *cut, int32_t n_cut, const int32_t *mh, int32_t n_mh)
{
  if (!c || !cut || !mh || n_cut < 1 || n_mh < 1) return fail(c, MM_EINVAL, "bad tables");
  c->cutoffs.assign(cut, cut + n_cut);
  c->min_hits.assign(mh, mh + n_mh);
  CU(c, cudaSetDevice(c->device));
  return write_tables(c);
}

int mm_index_blob(mm_ctx *c, void **blob, uint64_t *n_bytes)
{
  if (!c || !blob || !n_bytes) return MM_EINVAL;
  if (!c->blob_ready) return fail(c, MM_ESTATE, "no index");
  *blob = c->blob; *n_bytes = c->blob_bytes;
  return MM_OK;
}

int mm_index_blob_alloc(mm_ctx *c, uint64_t n_bytes, void **blob)
{
  if (!c || !blob || n_bytes < sizeof(mm_blob_header)) return MM_EINVAL;
  CU(c, cudaSetDevice(c->device));
  mm_blob_header h{}; /* the real one arrives with the image (mm_index_adopt_blob) */
  h.total_bytes = n_bytes;
  if (int rc = replace_blob(c, h)) return rc;
  *blob = c->blob;
  return MM_OK;
}

int mm_index_adopt_blob(mm_ctx *c)
{
  if (!c || !c->blob) return fail(c, MM_ESTATE, "no blob allocated");
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaMemcpyAsync(&c->hdr, c->blob, sizeof(c->hdr), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  if (c->hdr.magic != MM_BLOB_MAGIC || c->hdr.total_bytes != c->blob_bytes) return fail(c, MM_EINVAL, "blob header mismatch");
  resolve_index(c);
  c->blob_ready = true;
  return MM_OK;
}

int mm_ctx_share_index(mm_ctx *c, const mm_ctx *src)
{
  if (!c || !src) return MM_EINVAL;
  if (!src->blob_ready) return fail(c, MM_ESTATE, "source context has no index");
  if (c->device != src->device) return fail(c, MM_EINVAL, "contexts are on different devices");
  release_blob(c);
  c->blob = src->blob; c->blob_bytes = src->blob_bytes; c->blob_owned = false;
  c->hdr = src->hdr;
  c->cutoffs = src->cutoffs; c->min_hits = src->min_hits;
  c->share_src = src;
  resolve_index(c);
  c->blob_ready = true;
  return MM_OK;
}

static int batch_upload_any(mm_ctx *c, const void *bases, uint64_t n_bases, const mm_segment *segs, uint64_t n_segs, int packed)
{
  if (!c || (!bases && n_bases) || (!segs && n_segs)) return fail(c, MM_EINVAL, "null argument");
  int rc = upload_batch(c, bases, n_bases, segs, n_segs, packed);
  if (rc) return rc;
  CU(c, wait_stream(c));
  cudaEventElapsedTime(&c->stage_ms[3], c->ev[EV_H2D_BEGIN], c->ev[EV_H2D_END]);
  return MM_OK;
}
int mm_batch_upload(mm_ctx *c, const char *bases, uint64_t n_bases, const mm_segment *segs, uint64_t n_segs)
{
  return batch_upload_any(c, bases, n_bases, segs, n_segs, 0);
}
int mm_batch_upload_packed(mm_ctx *c, const uint8_t *nibbles, uint64_t n_bases, const mm_segment *segs, uint64_t n_segs)
{
  return batch_upload_any(c, nibbles, n_bases, segs, n_segs, 1);
}

int mm_map_resident(mm_ctx *c, uint64_t *n_candidates, uint64_t *n_loci)
{
  if (!c) return MM_EINVAL;
  int rc = run_pipeline(c);
  if (rc) return rc;
  if (n_candidates) *n_candidates = c->n_cands;
  if (n_loci) *n_loci = c->n_loci;
  return MM_OK;
}

int mm_batch_fetch(mm_ctx *c, mm_segment_result *seg_results, mm_l1_candidate *cands, uint64_t cand_cap,
                   mm_l2_locus *loci, uint64_t loci_cap)
{
  if (!c || !c->batch_mapped) return fail(c, MM_ESTATE, "no mapped batch");
  if (cand_cap < c->n_cands || loci_cap < c->n_loci) return fail(c, MM_ECAPACITY, "output capacity too small");
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaEventRecord(c->ev[EV_D2H_BEGIN], c->stream));
  if (seg_results) CU(c, cudaMemcpyAsync(seg_results, c->d_seg_res.p, c->n_segs * sizeof(mm_segment_result), cudaMemcpyDeviceToHost, c->stream));
  if (cands && c->n_cands) CU(c, cudaMemcpyAsync(cands, c->d_cands.p, c->n_cands * sizeof(mm_l1_candidate), cudaMemcpyDeviceToHost, c->stream));
  if (loci && c->n_loci) CU(c, cudaMemcpyAsync(loci, c->d_loci.p, c->n_loci * sizeof(mm_l2_locus), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaEventRecord(c->ev[EV_D2H_END], c->stream));
  CU(c, wait_stream(c));
  cudaEventElapsedTime(&c->stage_ms[4], c->ev[EV_D2H_BEGIN], c->ev[EV_D2H_END]);
  return MM_OK;
}

int mm_batch_fetch_sketch(mm_ctx *c, mm_minmer *out, int32_t *out_count)
{
  if (!c || !c->batch_mapped || !out || !out_count) return fail(c, MM_ESTATE, "no mapped batch");
  CU(c, cudaSetDevice(c->device));
  const uint64_t S = (uint64_t)c->params.sketch_size, n = c->n_segs * S;
  std::vector<uint64_t> hh(n);
  std::vector<int2> pp(n);
  std::vector<int8_t> ss(n);
  std::vector<mm_segment_result> sr(c->n_segs);
  std::vector<mm_segment> sg(c->n_segs);
  CU(c, cudaMemcpyAsync(hh.data(), c->d_sk_hash.p, n * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaMemcpyAsync(pp.data(), c->d_sk_pos.p, n * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaMemcpyAsync(ss.data(), c->d_sk_strand.p, n, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaMemcpyAsync(sr.data(), c->d_seg_res.p, c->n_segs * sizeof(mm_segment_result), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaMemcpyAsync(sg.data(), c->d_segs.p, c->n_segs * sizeof(mm_segment), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  for (uint64_t s = 0; s < c->n_segs; s++) {
    out_count[s] = sr[s].sketch_size;
    for (int j = 0; j < sr[s].sketch_size; j++) {
      mm_minmer &m = out[s * S + j];
      m.hash = hh[s * S + j]; m.wpos = pp[s * S + j].x; m.wpos_end = pp[s * S + j].y;
      m.seqId = sg[s].seq_counter; m.strand = ss[s * S + j]; m._pad = 0;
    }
  }
  return MM_OK;
}

int mm_sketch_segments(mm_ctx *c, const char *bases, uint64_t n_bases, const mm_segment *segs, uint64_t n_segs,
                       mm_minmer *out, int32_t *out_count)
{
  if (!c || !out || !out_count) return fail(c, MM_EINVAL, "null argument");
  int rc = upload_batch(c, bases, n_bases, segs, n_segs, 0);
  if (rc) return rc;
  mm_dev_batch b = make_batch(c);
  if ((rc = launch_pack_if_ascii(c))) return rc;
  ZERO_WORDS(c, c->d_counters.p, 16);
  CU(c, cudaEventRecord(c->ev[EV_K1_BEGIN], c->stream));
  CU(c, mm_launch_sketch(c->params, b, c->stream, c->sm_count, c->sk_mode));
  CU(c, cudaEventRecord(c->ev[EV_K1_END], c->stream));
  c->launches += c->sk_mode ? 1 : 2;
  CU(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->stage_ms[0], c->ev[EV_K1_BEGIN], c->ev[EV_K1_END]);
  {
    uint32_t h9 = 0;
    if (cudaMemcpy(&h9, c->d_counters.p + 9, 4, cudaMemcpyDeviceToHost) == cudaSuccess) c->diag[MM_DIAG_SKETCH_GENERAL_SEGMENTS] += h9;
  }
  c->batch_mapped = true; /* sketches only; fetch_sketch reads sketch_size == raw count */
  rc = mm_batch_fetch_sketch(c, out, out_count);
  c->batch_mapped = false;
  return rc;
}

static int map_segments_any(mm_ctx *c, const void *bases, uint64_t n_bases, const mm_segment *segs, uint64_t n_segs,
                            mm_segment_result *seg_results, mm_l1_candidate *cands, uint64_t cand_cap, uint64_t *n_candidates,
                            mm_l2_locus *loci, uint64_t loci_cap, uint64_t *n_loci, int packed)
{
  if (!c || !seg_results || !n_candidates || !n_loci) return fail(c, MM_EINVAL, "null argument");
  int rc = upload_batch(c, bases, n_bases, segs, n_segs, packed);
  if (rc) return rc;
  if ((rc = run_pipeline(c))) return rc;
  cudaEventElapsedTime(&c->stage_ms[3], c->ev[EV_H2D_BEGIN], c->ev[EV_H2D_END]);
  *n_candidates = c->n_cands;
  *n_loci = c->n_loci;
  if (cand_cap < c->n_cands || loci_cap < c->n_loci) return fail(c, MM_ECAPACITY, "need %llu candidates, %llu loci", (unsigned long long)c->n_cands, (unsigned long long)c->n_loci);
  return mm_batch_fetch(c, seg_results, cands, cand_cap, loci, loci_cap);
}
int mm_map_segments(mm_ctx *c, const char *bases, uint64_t n_bases, const mm_segment *segs, uint64_t n_segs,
                    mm_segment_result *seg_results, mm_l1_candidate *cands, uint64_t cand_cap, uint64_t *n_candidates,
                    mm_l2_locus *loci, uint64_t loci_cap, uint64_t *n_loci)
{
  return map_segments_any(c, bases, n_bases, segs, n_segs, seg_results, cands, cand_cap, n_candidates, loci, loci_cap, n_loci, 0);
}
int mm_map_segments_packed(mm_ctx *c, const uint8_t *nibbles, uint64_t n_bases, const mm_segment *segs, uint64_t n_segs,
                           mm_segment_result *seg_results, mm_l1_candidate *cands, uint64_t cand_cap, uint64_t *n_candidates,
                           mm_l2_locus *loci, uint64_t loci_cap, uint64_t *n_loci)
{
  return map_segments_any(c, nibbles, n_bases, segs, n_segs, seg_results, cands, cand_cap, n_candidates, loci, loci_cap, n_loci, 1);
}

int mm_ctx_set_wait_mode(mm_ctx *c, int blocking)
{
  if (!c) return MM_EINVAL;
  if (blocking && !c->ev_wait) {
    cudaSetDevice(c->device);
    if (cudaEventCreateWithFlags(&c->ev_wait, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess) {
      c->ev_wait = nullptr;
      return fail(c, MM_ECUDA, "cannot create the blocking event");
    }
  }
  c->blocking_wait = blocking != 0;
  return MM_OK;
}

int mm_ctx_set_phase_hook(mm_ctx *c, mm_phase_hook hook, void *user)
{
  if (!c) return MM_EINVAL;
  c->hook = hook; c->hook_user = user;
  return MM_OK;
}

int mm_last_stage_ms(const mm_ctx *c, float ms[8])
{
  if (!c || !ms) return MM_EINVAL;
  for (int i = 0; i < 8; i++) ms[i] = c->stage_ms[i];
  return MM_OK;
}
int mm_last_pack_ms(const mm_ctx *c, float *ms)
{
  if (!c || !ms) return MM_EINVAL;
  *ms = c->pack_ms;
  return MM_OK;
}

/* pinned host memory for the caller's batch buffers (H2D/D2H at full PCIe rate) */
int mm_host_alloc(void **ptr, uint64_t bytes)
{
  if (!ptr) return MM_EINVAL;
  return cudaHostAlloc(ptr, bytes, cudaHostAllocPortable) == cudaSuccess ? MM_OK : MM_ENOMEM; /* pinned for every device of the process */
}
int mm_host_free(void *ptr) { return cudaFreeHost(ptr) == cudaSuccess ? MM_OK : MM_ECUDA; }

} // extern "C"

namespace {
__global__ void k_count_seq(uint64_t n, const int32_t *__restrict__ seq, unsigned long long *cnt)
{
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&cnt[seq[i]], 1ULL);
}
__global__ void k_unpack_points(uint64_t n, const uint64_t *__restrict__ pts, const uint64_t *__restrict__ keys, const uint64_t *__restrict__ offs,
                                uint64_t n_keys, mm_ipoint *out)
{ /* packed point -> skch::IntervalPoint (the hash comes from the key whose list the point is in) */
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t lo = 0, hi = n_keys; /* last key with offs <= i */
  while (lo + 1 < hi) { const uint64_t mid = (lo + hi) >> 1; if (offs[mid] <= i) lo = mid; else hi = mid; }
  mm_ipoint p;
  memset(&p, 0, sizeof p);
  p.pos = mm_point_pos(pts[i]); p.hash = keys[lo]; p.seqId = mm_point_seq(pts[i]); p.side = mm_point_open(pts[i]) ? 1 : -1;
  out[i] = p;
}
} // namespace

extern "C" {

/* skch::Sketch's build + index + computeFreqHist + dropFreqSeedSet on the device (mm_index_build.cu) */
int mm_index_build(mm_ctx *c, const char *seqs, int seqs_on_device, const uint64_t *contig_offsets, int32_t n_contigs,
                   const int32_t *contig_name_id, const int32_t *contig_group, float kmer_pct_threshold, int keep_lookup,
                   mm_index_stats *stats)
{
  if (!c) return MM_EINVAL;
  if (n_contigs < 1 || !contig_offsets || !seqs) return fail(c, MM_EINVAL, "no contigs");
  CU(c, cudaSetDevice(c->device));
  const auto t0 = std::chrono::steady_clock::now();
  release_blob(c);
  mm_built_index_free(&c->built);
  c->built_kept = false;
  /* every early return below releases the temporaries: the staged text, the builder's arrays, the counters */
  struct built_guard {
    mm_built_index b;
    ~built_guard() { mm_built_index_free(&b); }
  } built;
  mm_built_index &B = built.b;
  int rc;
  {
    const uint64_t total = contig_offsets[n_contigs];
    const uint8_t *d_seq = (const uint8_t *)seqs;
    dev_array<uint8_t> staged;
    if (!seqs_on_device) {
      if ((rc = staged.reserve(c, total + 64, total + 64))) return rc;
      CU(c, cudaMemcpyAsync(staged.p, seqs, total, cudaMemcpyHostToDevice, c->stream));
      d_seq = staged.p;
    }
    std::string err;
    rc = mm_build_index_device(c->params, d_seq, contig_offsets, n_contigs, kmer_pct_threshold, c->stream, c->sm_count, &B, err);
    if (rc != MM_OK) return fail(c, rc, "index build: %s", err.c_str());
  }
  c->launches += 12;

  const uint64_t n_mi = B.n_minmers, n_keys = B.n_keys, n_points = B.n_points;
  if (n_mi >= (1ULL << 32)) return fail(c, MM_EINVAL, "more than 2^32 minmers");
  /* contig_start from the seqId column */
  std::vector<uint64_t> cstart((size_t)n_contigs + 1, 0);
  if (n_mi) {
    dev_array<unsigned long long> d_cnt;
    if ((rc = d_cnt.reserve(c, (size_t)n_contigs + 1, (size_t)n_contigs + 1))) return rc;
    CU(c, cudaMemsetAsync(d_cnt.p, 0, ((size_t)n_contigs + 1) * 8, c->stream));
    k_count_seq<<<(uint32_t)((n_mi + 255) / 256), 256, 0, c->stream>>>(n_mi, B.seq, d_cnt.p);
    std::vector<unsigned long long> cnt((size_t)n_contigs + 1);
    CU(c, cudaMemcpyAsync(cnt.data(), d_cnt.p, ((size_t)n_contigs + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    for (int32_t q = 0; q < n_contigs; q++) cstart[(size_t)q + 1] = cstart[(size_t)q] + cnt[(size_t)q];
  }
  const mm_blob_header h = blob_layout(n_mi, n_keys, n_points, n_contigs);
  if ((rc = replace_blob(c, h))) return rc;
  blob_guard guard{c};
  if (n_mi) {
    CU(c, cudaMemcpyAsync(c->blob + h.off_idx_hash, B.hash, n_mi * 8, cudaMemcpyDeviceToDevice, c->stream));
    CU(c, cudaMemcpyAsync(c->blob + h.off_idx_wpos, B.wpos, n_mi * 4, cudaMemcpyDeviceToDevice, c->stream));
    CU(c, cudaMemcpyAsync(c->blob + h.off_idx_wend, B.wend, n_mi * 4, cudaMemcpyDeviceToDevice, c->stream));
    CU(c, cudaMemcpyAsync(c->blob + h.off_idx_strand, B.strand, n_mi, cudaMemcpyDeviceToDevice, c->stream));
  }
  CU(c, cudaMemcpyAsync(c->blob + h.off_contig_start, cstart.data(), cstart.size() * 8, cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  cudaFree(B.hash); cudaFree(B.wpos); cudaFree(B.wend); cudaFree(B.seq); cudaFree(B.strand);
  B.hash = nullptr; B.wpos = nullptr; B.wend = nullptr; B.seq = nullptr; B.strand = nullptr;
  CU(c, mm_build_death_order((const uint64_t *)(c->blob + h.off_idx_hash), (const int32_t *)(c->blob + h.off_idx_wend),
                             (const uint64_t *)(c->blob + h.off_contig_start), n_contigs, n_mi,
                             (uint64_t *)(c->blob + h.off_idx2_hash), (int32_t *)(c->blob + h.off_idx2_wend), c->stream));
  if (n_points) CU(c, cudaMemcpyAsync(c->blob + h.off_pts, B.pts, n_points * 8, cudaMemcpyDeviceToDevice, c->stream));
  CU(c, cudaMemsetAsync(c->blob + h.off_tab, 0, (1ULL << h.tab_log2) * sizeof(mm_tab_slot), c->stream));
  if (n_keys) {
    dev_array<uint32_t> d_err;
    if ((rc = d_err.reserve(c, 1, 1))) return rc;
    CU(c, cudaMemsetAsync(d_err.p, 0, 4, c->stream));
    CU(c, mm_upload_build_table(B.keys, B.offs, B.is_freq, n_keys, (mm_tab_slot *)(c->blob + h.off_tab), h.tab_log2, d_err.p, c->stream));
    uint32_t e = 0;
    CU(c, cudaMemcpyAsync(&e, d_err.p, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (e) return fail(c, MM_EINVAL, "lookup table build failed (code %u)", e);
  }
  std::vector<int32_t> clen((size_t)n_contigs);
  for (int32_t q = 0; q < n_contigs; q++) clen[(size_t)q] = (int32_t)(contig_offsets[q + 1] - contig_offsets[q]);
  if ((rc = finish_blob(c, clen.data(), contig_name_id, contig_group))) return rc;
  if (stats) {
    memset(stats, 0, sizeof *stats);
    stats->n_minmers = n_mi; stats->n_minmers_before_filter = B.n_minmers_before_filter; stats->n_keys = n_keys; stats->n_points = n_points;
    stats->freq_threshold = B.freq_threshold; stats->n_chunks = B.n_chunks; stats->n_fixed_chunks = B.n_fixed_chunks; stats->fix_rounds = B.fix_rounds;
    stats->hist_min_count = B.hist_min_count; stats->hist_max_count = B.hist_max_count; stats->hist_min_keys = B.hist_min_keys;
    stats->hist_max_keys = B.hist_max_keys; stats->ms_scan = B.ms_scan; stats->ms_post = B.ms_post; stats->ms_lookup = B.ms_lookup;
    stats->ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  }
  if (keep_lookup) {
    c->built = B;
    c->built_kept = true;
    B = mm_built_index{};
  }
  return MM_OK;
}

/* host copies of what mm_index_build left on the device (needs keep_lookup); any output may be NULL */
int mm_index_download(mm_ctx *c, mm_minmer *mi, uint64_t *keys, uint64_t *offsets, mm_ipoint *points, uint8_t *is_freq)
{
  if (!c || !c->blob_ready) return fail(c, MM_ESTATE, "no index");
  if ((keys || offsets || points || is_freq) && !c->built_kept) return fail(c, MM_ESTATE, "the lookup arrays were not kept (keep_lookup)");
  CU(c, cudaSetDevice(c->device));
  const mm_blob_header &h = c->hdr;
  if (mi && h.n_minmers) {
    const uint64_t n = h.n_minmers;
    std::vector<uint64_t> hh(n), cs((size_t)h.n_contigs + 1);
    std::vector<int32_t> a(n), b(n);
    std::vector<int8_t> st(n);
    CU(c, cudaMemcpy(hh.data(), c->blob + h.off_idx_hash, n * 8, cudaMemcpyDeviceToHost));
    CU(c, cudaMemcpy(a.data(), c->blob + h.off_idx_wpos, n * 4, cudaMemcpyDeviceToHost));
    CU(c, cudaMemcpy(b.data(), c->blob + h.off_idx_wend, n * 4, cudaMemcpyDeviceToHost));
    CU(c, cudaMemcpy(st.data(), c->blob + h.off_idx_strand, n, cudaMemcpyDeviceToHost));
    CU(c, cudaMemcpy(cs.data(), c->blob + h.off_contig_start, cs.size() * 8, cudaMemcpyDeviceToHost));
    int32_t q = 0;
    for (uint64_t i = 0; i < n; i++) {
      while (i >= cs[(size_t)q + 1]) q++;
      mi[i].hash = hh[i]; mi[i].wpos = a[i]; mi[i].wpos_end = b[i]; mi[i].seqId = q; mi[i].strand = st[i]; mi[i]._pad = 0;
    }
  }
  const mm_built_index &B = c->built;
  if (keys && B.n_keys) CU(c, cudaMemcpy(keys, B.keys, B.n_keys * 8, cudaMemcpyDeviceToHost));
  if (offsets) CU(c, cudaMemcpy(offsets, B.offs, (B.n_keys + 1) * 8, cudaMemcpyDeviceToHost));
  if (is_freq && B.n_keys) CU(c, cudaMemcpy(is_freq, B.is_freq, B.n_keys, cudaMemcpyDeviceToHost));
  if (points && B.n_points) {
    dev_array<mm_ipoint> d;
    if (int rc = d.reserve(c, B.n_points, B.n_points)) return rc;
    k_unpack_points<<<(uint32_t)((B.n_points + 255) / 256), 256, 0, c->stream>>>(B.n_points, (const uint64_t *)(c->blob + h.off_pts), B.keys, B.offs, B.n_keys, d.p);
    CU(c, cudaMemcpyAsync(points, d.p, B.n_points * sizeof(mm_ipoint), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
  }
  return MM_OK;
}

} // extern "C"
