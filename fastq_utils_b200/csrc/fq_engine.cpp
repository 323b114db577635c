/*
 * fq_engine.cpp — host orchestration of the fastq_info hot path on one GPU (see fq_engine.h).
 *
 * Reference control flow being replaced: src/fastq_info.c:57-176 (three loops), :273-362 (dispatch, index loop
 * call, mate loop) and src/fastq.c:396-439 (index loop).  The reference walks records one by one and stops at the
 * first failing check; here every record of a chunk is checked at once and each failure becomes an *event key*
 * (step << 6 | rank) ordered exactly like the reference's sequential execution; the smallest key wins.
 */
#include "fq_engine.h"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

static const uint32_t kPad = 64;                 /* readable bytes after every chunk */
static const size_t kMaxChunk = 1ull << 31;      /* bytes per chunk: offsets are 32-bit */
/* test hook: FQG_MAX_CHUNK_BYTES (a multiple of 16) cuts what is fed into smaller chunks, so that chunk boundaries inside records,
 * bridges and every starting phase are reached with small inputs */
static size_t feed_chunk() { const char* e = getenv("FQG_MAX_CHUNK_BYTES"); size_t v = e ? strtoull(e, nullptr, 10) & ~(size_t)15 : 0; return v >= 4096 && v < kMaxChunk ? v : kMaxChunk; }
static const uint32_t kNone32 = 0xFFFFFFFFu;
static const double kLanesTile = 31744.0;        /* bytes of a tile of the per-line clean-data pass (fq_lanes.cuh: LS_TILE): sizes the arena */
/* device words: [0] equal hashes that tuples alone could not judge, [1] claimed by the mate loop, [2] table full, [3] the owner's earliest
 * name event, [4] names that met ANOTHER name with their hash (diagnostics), [5] units measured for an arena, [6] arena cursor */
static const int kCounters = 12; /* [8] names claimed / [9] mates without a (fresh) partner at the owner (pipelined routing of paired files) */

static uint64_t pow2_at_least(uint64_t x) { uint64_t p = 1; while (p < x) p <<= 1; return p; }

FqEngine::FqEngine(const fqg_config& cfg, FqDevice* dev) : cfg_(cfg), dev_(dev) {
  if (cfg_.mode == FQG_MODE_READER) { reader_ = true; cfg_.mode = FQG_MODE_SINGLE; } /* same chunks, segments, tails and events; only the per-record verdict differs */
  key_ = (unsigned long long*)dev_->alloc(sizeof(unsigned long long));
  counters_ = (unsigned long long*)dev_->alloc(kCounters * sizeof(unsigned long long));
  streaming_ = (cfg_.mode == FQG_MODE_SINGLE || cfg_.mode == FQG_MODE_INDEX || cfg_.mode == FQG_MODE_INDEX_PAIR) && !(cfg_.flags & FQG_FLAG_KEEP_CHUNKS);
  scratch_ = (uint32_t*)dev_->alloc(64 * sizeof(uint32_t));
  recout_ = (FqRecOut*)dev_->alloc(sizeof(FqRecOut));
  tile_out_ = (uint32_t*)dev_->alloc(32 * sizeof(uint32_t));
  route_cursors_ = (unsigned long long*)dev_->alloc(2 * FQ_SHARD_MAX_SRC * sizeof(unsigned long long));
  for (int f = 0; f < 2; f++) {
    f_[f].stats = (FqStats*)dev_->alloc(sizeof(FqStats));
    f_[f].hist = (unsigned long long*)dev_->alloc((size_t)FQ_MAX_READ_LENGTH * sizeof(unsigned long long));
    f_[f].stats_open = (FqStats*)dev_->alloc(sizeof(FqStats));
    f_[f].hist_open = (unsigned long long*)dev_->alloc((size_t)FQ_MAX_READ_LENGTH * sizeof(unsigned long long));
  }
  if (cfg_.index_capacity_hint && (cfg_.mode == FQG_MODE_INDEX || cfg_.mode == FQG_MODE_INDEX_PAIR)) {
    table_cap_ = pow2_at_least(std::max<uint64_t>(1u << 16, cfg_.index_capacity_hint * 2));
    slots_ = (FqSlot*)dev_->alloc(table_cap_ * sizeof(FqSlot));
  }
  reset();
}

void FqEngine::free_file(FqFile& F) {
  for (auto& s : F.segs) { if (s.names) dev_->release(s.names); if (s.lines_dev) dev_->release(s.lines_dev); if (s.arena) dev_->release(s.arena); }
  for (auto& b : F.bufs) { if (b.owned && b.data) dev_->release(b.data); if (b.line_end) dev_->release(b.line_end); }
  if (F.pend) dev_->release(F.pend);
  if (F.dir_dev) dev_->release(F.dir_dev);
  for (auto& ps : F.prescans) dev_->release(ps.line_end);
  FqStats* st = F.stats; unsigned long long* h = F.hist; FqStats* so = F.stats_open; unsigned long long* ho = F.hist_open;
  F = FqFile();
  F.stats = st; F.hist = h; F.stats_open = so; F.hist_open = ho;
}

FqEngine::~FqEngine() {
  dev_->sync();
  if (pre_.valid) { try { lanes_discard(&pre_); } catch (...) {} }
  for (int f = 0; f < 2; f++) { free_file(f_[f]); dev_->release(f_[f].stats); dev_->release(f_[f].hist); dev_->release(f_[f].stats_open); dev_->release(f_[f].hist_open); }
  if (slots_) dev_->release(slots_);
  dev_->release(key_); dev_->release(counters_); dev_->release(scratch_); dev_->release(recout_); dev_->release(tile_out_);
  dev_->release(route_cursors_);
}

/* forget input and results; the index keeps its allocation */
void FqEngine::reset() {
  dev_->sync();
  if (pre_.valid) { try { lanes_discard(&pre_); } catch (...) {} }
  for (int f = 0; f < 2; f++) free_file(f_[f]);
  for (auto& c : path_counts) c = 0;
  seed_ = 0; finished_ = false; total0_set_ = false; total0_ = 0; fused_ok_ = !(cfg_.flags & FQG_FLAG_TWO_PASS);
  { const char* e = getenv("FQG_FUSED_MIN_BYTES"); fused_min_ = e ? (uint32_t)strtoul(e, nullptr, 10) : (1u << 20); } /* test hook */
  { const char* e = getenv("FQG_NO_LANES"); lanes_ok_ = !(e && *e && *e != '0'); }                                  /* test hook */
  { const char* e = getenv("FQG_TEST_WEAK_HASH"); if (e && *e && *e != '0') seed_ = FQ_SEED_WEAK; }                 /* test hook: 12-bit name hashes, so that equal hashes of different names are common */
  for (auto& m : mem_stats) m = 0;
  open_ = streaming_; add_depth_ = 0; open_dirty_ = false;
  /* results */
  dev_->fill(key_, 0xFF, sizeof(unsigned long long));
  dev_->fill(counters_, 0, kCounters * sizeof(unsigned long long));
  for (int f = 0; f < 2; f++) {
    FqStats init; memset(&init, 0, sizeof init);
    init.min_rl = 0xFFFFFFFFu; init.min_q = 255u;
    dev_->upload(f_[f].stats, &init, sizeof init);
    dev_->fill(f_[f].hist, 0, (size_t)FQ_MAX_READ_LENGTH * sizeof(unsigned long long));
    dev_->sync(); /* `init` is a stack object */
  }
  clear_open();
  if (slots_) dev_->fill_index(slots_, 0xFF, table_cap_ * sizeof(FqSlot)); /* on the index kernels' stream: beside the first chunk's pass */
  table_names_ = 0;
}

int FqEngine::loop_of(int file) const {
  switch (cfg_.mode) {
    case FQG_MODE_SINGLE: return reader_ ? FQ_LOOP_READER : FQ_LOOP_SINGLE;
    case FQG_MODE_INDEX: return FQ_LOOP_INDEX;
    case FQG_MODE_INDEX_PAIR: return file == 0 ? FQ_LOOP_INDEX : FQ_LOOP_MATE;
    case FQG_MODE_INTERLEAVED: return FQ_LOOP_INTERLEAVED;
    default: return file == 0 ? FQ_LOOP_SORTED1 : FQ_LOOP_SORTED2;
  }
}
static uint64_t eff_records(const FqFile& F) { return std::min<uint64_t>(F.nrec, F.limit); }
/* records the index loop read from file 1 (over all ranks in a sharded run) */
uint64_t FqEngine::total0() const { return total0_set_ ? total0_ : eff_records(f_[0]); }
uint64_t FqEngine::step_base(int file) const { return loop_of(file) == FQ_LOOP_MATE ? total0() + 1 : 0; }

FqRecCtx FqEngine::make_ctx(int file) const {
  FqRecCtx cx; memset(&cx, 0, sizeof cx);
  cx.loop = loop_of(file);
  cx.fmt_key = fq_fmt_of_sniff(f_[file].sniff_fmt);
  cx.pe_key = (cfg_.mode == FQG_MODE_INDEX && !(cfg_.flags & FQG_FLAG_PAIRED_NAMES)) ? 0 : 1; /* fastq_info.c:63,112-113,158,290,327 */
  if (cx.loop == FQ_LOOP_MATE) { /* fastq_info.c:345: file-2 records are validated against file 1's state */
    cx.fmt_val = fq_fmt_of_sniff(f_[0].sniff_fmt); cx.pe_val = 1; cx.space = f_[0].sniff_color;
  } else { cx.fmt_val = cx.fmt_key; cx.pe_val = cx.pe_key; cx.space = f_[file].sniff_color; }
  cx.weight = cx.loop == FQ_LOOP_INDEX ? 2 : 1; /* fastq.c:241 + :344 */
  cx.seed = seed_;
  return cx;
}

/* ------------------------------------------------------------------------------------------------ feeding */
void FqEngine::feed_host(int file, const void* bytes, size_t n, bool last) {
  const uint8_t* p = (const uint8_t*)bytes;
  if (n == 0) { add_buffer(file, nullptr, 0, last, false); return; }
  const size_t maxc = feed_chunk();
  while (n) {
    size_t k = std::min(n, maxc);
    uint8_t* d = (uint8_t*)dev_->alloc(k + kPad);
    dev_->upload(d, p, k);
    dev_->fill(d + k, 0, kPad);
    add_buffer(file, d, (uint32_t)k, last && k == n, true);
    p += k; n -= k;
  }
}
void FqEngine::feed_device(int file, const void* dptr, size_t n, bool last) {
  uint8_t* p = (uint8_t*)dptr;
  if (n == 0) { add_buffer(file, nullptr, 0, last, false); return; }
  const size_t maxc = std::min(feed_chunk(), kMaxChunk - 16);
  FqFile& F = f_[file];
  while (n) {
    size_t k = std::min(n, maxc);
    /* the kernels read 16 bytes at a time: a chunk that starts at an unaligned address is handed over from the boundary below
     * it, with the bytes in between marked as not its own (they are readable: same allocation) */
    const uint32_t lead = (uint32_t)((uintptr_t)p & 15u);
    const bool whole_records = F.pend_n == 0; /* nothing carried over: the chunk starts at a record start */
    hook_fired_ = false;
    next_.valid = whole_records && n > k; next_.file = file; next_.ptr = p + k; next_.remaining = n - k; next_.last = last;
    add_buffer(file, p - lead, (uint32_t)(k + lead), last && k == n, false, true, lead);
    next_.valid = false;
    if (hook_ && !hook_fired_) hook_(hook_user_, file); /* the chunk did not take the clean-data pass: its hook call comes after it */
    p += k; n -= k;
    /* A record cut by the end of the chunk normally travels on as pending bytes and is finished in a bridge chunk.  The bytes are
     * still here, so the next chunk simply starts at that record instead: no bridge, no second pass over its lines. */
    if (n && whole_records && !F.ended && F.pend_n > 0 && F.pend_n < k / 2) {
      p -= F.pend_n; n += F.pend_n;
      F.pend_n = 0; F.pend_lfs = 0;
    }
  }
  if (cfg_.flags & FQG_FLAG_BORROW_FOR_CALL) {
    /* the caller wants its buffer back now: chunks that could not be settled (an event fired; or a loop kind that keeps its chunks)
     * move into memory of our own */
    for (auto& B : F.bufs) {
      if (B.released || B.owned || !B.data) continue;
      uint8_t* d = (uint8_t*)dev_->alloc((size_t)B.n + kPad);
      dev_->copy(d, B.data, B.n); dev_->fill(d + B.n, 0, kPad);
      B.data = d; B.owned = true;
    }
    dev_->sync_main();
  }
}

/* a borrowed chunk with bytes in front of its data that the clean-data pass did not take: the other kernels want the data at
 * offset 0 of an aligned buffer */
void FqEngine::realign(FqBuffer& B) {
  if (!B.lead) return;
  uint32_t k = B.n - B.lead;
  uint8_t* d = (uint8_t*)dev_->alloc((size_t)k + kPad);
  dev_->copy(d, B.data + B.lead, k);
  dev_->fill(d + k, 0, kPad);
  if (B.owned && B.data) dev_->release(B.data);
  B.data = d; B.n = k; B.lead = 0; B.owned = true;
}

/* the fused pass stores only the line ends the host normally needs; anything else rebuilds the index with K1 */
void FqEngine::ensure_full_index(FqBuffer& b) {
  if (!b.index_partial) return;
  uint32_t cap = b.n / 32 + 4096; /* the capacity the fused pass allocated and did not overflow */
  dev_->scan_lines(b.data, b.n, b.index_virtual_end ? 1 : 0, b.line_end, cap, scratch_, b.lead);
  dev_->sync();
  b.index_partial = false;
}
uint32_t FqEngine::line_end_at(FqBuffer& b, uint32_t idx) {
  if (idx >= b.tail_from && idx < b.tail_from + b.tail_n) return b.tail_ends[idx - b.tail_from];
  if (b.index_partial && idx >= 8 && idx < b.index_from) ensure_full_index(b);
  uint32_t v; dev_->download(&v, b.line_end + idx, sizeof v); return v;
}

void FqEngine::append_pending(int file, const uint8_t* src, size_t n, uint32_t lfs) {
  FqFile& F = f_[file];
  if (F.pend_n + n + kPad > F.pend_cap) {
    size_t cap = std::max<size_t>((F.pend_n + n + kPad) * 2, 1 << 16);
    uint8_t* np = (uint8_t*)dev_->alloc(cap);
    if (F.pend_n) dev_->copy(np, F.pend, F.pend_n);
    if (F.pend) { dev_->sync(); dev_->release(F.pend); }
    F.pend = np; F.pend_cap = cap;
  }
  dev_->copy(F.pend + F.pend_n, src, n);
  F.pend_n += n; F.pend_lfs += lfs;
}

/* The file ended while bytes were still waiting for the rest of their record: what is left may still split into
 * a complete record (over-long lines), so it goes through the normal path as the file's final chunk. */
void FqEngine::flush_pending_as_last(int file) {
  FqFile& F = f_[file];
  if (F.pend_n == 0) { end_file(file, nullptr, 0); return; }
  size_t bn = F.pend_n;
  uint8_t* bd = (uint8_t*)dev_->alloc(bn + kPad);
  dev_->copy(bd, F.pend, bn);
  dev_->fill(bd + bn, 0, kPad);
  F.pend_n = 0; F.pend_lfs = 0;
  add_buffer(file, bd, (uint32_t)bn, true, true);
}

/* K1: line index.  Capacity is a guess (one line per 32 bytes); on overflow rescan with the exact count. */
void FqEngine::scan_buffer(FqBuffer& B, bool last) {
  uint32_t cap = B.n / 32 + 4096;
  for (;;) {
    B.line_end = (uint32_t*)dev_->alloc((size_t)cap * sizeof(uint32_t) + kPad);
    dev_->scan_lines(B.data, B.n, last ? 1 : 0, B.line_end, cap, scratch_);
    uint32_t out2[2]; dev_->download(out2, scratch_, sizeof out2);
    B.nlines = out2[0];
    if (!out2[1]) break;
    dev_->release(B.line_end); cap = B.nlines;
  }
}

/* Sniff the first record of a file from a short prefix so that the fused pass knows the read-name format and colour space
 * before it runs.  False when the prefix does not hold the two lines (the two-pass path sniffs later). */
bool FqEngine::presniff(int file, const uint8_t* data, uint32_t n, uint32_t skip, bool short_only) {
  FqFile& F = f_[file];
  if (F.sniff_fmt >= 0) return true;
  uint32_t pn = std::min<uint32_t>(n, 1u << 16), cap = 4096;
  uint32_t* le = (uint32_t*)dev_->alloc((size_t)cap * sizeof(uint32_t) + kPad);
  dev_->scan_lines(data, pn, 0, le, cap, scratch_);
  uint32_t out2[2]; dev_->download(out2, scratch_, sizeof out2);
  bool ok = false;
  if (out2[0] >= skip + 2 && skip + 2 <= cap) {
    uint32_t e[3] = {0, 0, 0};
    if (skip) dev_->download(e, le + skip - 1, 3 * sizeof(uint32_t)); else dev_->download(e + 1, le, 2 * sizeof(uint32_t));
    FqLine h, q; h.off = e[0]; h.len = e[1] - e[0]; q.off = e[1]; q.len = e[2] - e[1];
    if (!short_only || (h.len < FQ_MAX_LABEL_LENGTH && q.len < 2048)) { /* fused pass: short reads only, long records do not fit its window */
      dev_->sniff(data, h, q, (int32_t*)scratch_);
      int32_t o2[2]; dev_->download(o2, scratch_, sizeof o2);
      F.sniff_fmt = o2[0]; F.sniff_color = o2[1];
      F.first_seq_len = q.len; F.first_hdr_len = h.len;
      ok = true;
    }
  }
  dev_->release(le);
  return ok;
}

/* K1+K2 fused over buffer b.  Returns false (nothing launched, or results discarded) when the two-pass path must be used. */
/* Everything a fused pass over one chunk needs, and the launch of the clean-data pass when the chunk may take it.  Split from the
 * collection of its results so that the pass of chunk k+1 can be launched as soon as the pass of chunk k has said where chunk k+1
 * starts — before the host has done its bookkeeping for chunk k (segments, name kernels, settling), which then runs beside it. */
void FqEngine::lanes_prepare(int file, uint8_t* data, uint32_t n, uint32_t lead, bool last, uint32_t j0, uint64_t g0_local, bool skip_lanes, LanesLaunch* L) {
  FqFile& F = f_[file];
  const int loop = loop_of(file);
  *L = LanesLaunch();
  L->valid = true; L->file = file; L->data = data; L->n = n; L->lead = lead; L->last = last; L->j0 = j0;
  L->cap = n / 32 + 4096;
  L->line_end = (uint32_t*)dev_->alloc((size_t)L->cap * sizeof(uint32_t) + kPad);
  L->ncap = L->cap / 4 + 1;
  /* (16 bytes per record: with the lengths of the file's first record known, room for a third more records than such records would
   * fill the chunk with — a chunk with more hands itself on, see fq_lanes_post_kernel, and the next one asks for the full bound) */
  if (lanes_ok_ && !names_cap_full_ && F.first_hdr_len && F.first_seq_len)
    L->ncap = std::min<uint32_t>(L->ncap, (uint32_t)((double)n / (0.75 * (F.first_hdr_len + 2.0 * F.first_seq_len + 2))) + 4096);
  L->routed = F.route_world > 0 && lanes_ok_ && !skip_lanes && f_[loop == FQ_LOOP_MATE ? 0 : file].sniff_color != FQ_SPACE_COLOR; /* the pass routes the names itself: no descriptors, no arena */
  L->names = (loop != FQ_LOOP_SINGLE && loop != FQ_LOOP_READER && !L->routed) ? (FqName*)dev_->alloc((size_t)L->ncap * sizeof(FqName)) : nullptr;
  FqTileArgs& a = L->a; memset(&a, 0, sizeof a);
  a.data = data; a.n = n; a.virtual_end = last ? 1 : 0; a.line_end = L->line_end; a.cap = L->cap; a.out5 = tile_out_;
  a.j0 = j0; a.max_rec = kNone32; a.g0 = g0_local + F.g_base; a.step_base = step_base(file); a.cx = make_ctx(file);
  const int target = a.cx.loop == FQ_LOOP_MATE ? 0 : file;
  a.stats = f_[target].stats_open; a.hist = f_[target].hist_open; a.stats_range = f_[file].stats_open; a.key = key_; a.names = L->names; a.names_cap = L->ncap;
  a.hint_line_len = F.first_seq_len;
  a.lead = lead;
  /* first choice: the clean-data pass.  It commits nothing unless the whole chunk is clean; otherwise the per-record kernels
   * decide (they own the reference's first-error semantics). */
  if (!(lanes_ok_ && !skip_lanes && a.cx.space != FQ_SPACE_COLOR)) return;
  L->tried = true;
  uint32_t linit[FQ_LANES_OUT_WORDS]; memset(linit, 0, sizeof linit);
  linit[2] = kNone32; linit[5] = kNone32; linit[6] = kNone32; linit[8] = kNone32;
  dev_->set_words(tile_out_, linit, FQ_LANES_OUT_WORDS);
  /* room for the names of the chunk (the per-line mode of the pass copies them out of the window itself): what the chunks before
   * it needed per byte and a quarter more; a pass that runs out of room hands the chunk on like any other anomaly */
  if (L->names) {
    double rate = F.arena_rate;
    if (rate <= 0 && F.first_hdr_len >= 3 && F.first_seq_len) rate = 1.2 * (double)((F.first_hdr_len - 2 + 15) >> 4) / (double)(F.first_hdr_len + 2.0 * F.first_seq_len + 2);
    if (rate <= 0) rate = 1.0 / 64;
    /* (every tile of the pass gets the same stretch of the block: what the fullest tile needed so far, a quarter more, and a little) */
    const uint64_t ntiles = ((uint64_t)n + (uint64_t)kLanesTile - 1) / (uint64_t)kLanesTile;
    L->arena_units = std::min<uint64_t>(((uint64_t)(rate * 1.25 * kLanesTile) + 16) * ntiles, (1ull << 28) - 1);
    L->arena = (uint8_t*)dev_->alloc((size_t)L->arena_units * 16 + kPad);
  }
  a.arena = L->arena; a.arena_units = (uint32_t)L->arena_units;
  if (L->routed) {
    a.route_world = F.route_world; a.route_stride = F.route_stride; a.route_units = F.route_units;
    for (uint32_t o = 0; o < F.route_world; o++) a.route_region[o] = F.route_region[o] + (size_t)(F.route_chunks % F.route_depth) * F.route_bytes;
  }
  /* While every chunk so far is final and no bytes wait for the rest of their record, an accepted clean-data pass is final too: its
   * statistics go straight into the main set (a chunk the pass hands on leaves no trace in either set). */
  L->direct = open_ && add_depth_ == 1 && F.pend_n == 0 && !open_dirty_;
  if (L->direct) { a.stats = f_[target].stats; a.hist = f_[target].hist; a.stats_range = f_[file].stats; }
  L->launched = dev_->lanes_pass(a, &L->self_judged);
  if (L->launched && hook_) { /* the pass is running: the caller routes the names of the chunks before this one beside it */
    in_beside_hook_ = true; L->hooked = true;
    try { hook_(hook_user_, file); } catch (...) { in_beside_hook_ = false; throw; }
    in_beside_hook_ = false;
  }
}

/* a pass launched ahead whose chunk never came (it cannot happen for the chunks of one fqg_feed_device call: the start of the next
 * chunk was taken from the pass's own line ends; a caller may stop feeding, though) */
void FqEngine::lanes_discard(LanesLaunch* L) {
  if (!L->valid) return;
  dev_->sync();
  if (L->launched) {
    uint32_t o[FQ_LANES_OUT_WORDS]; dev_->download(o, tile_out_, sizeof o);
    const bool pass_ok = !o[1] && o[2] == kNone32 && !o[3] && !o[4];
    const bool accepted = L->self_judged ? o[25] != 0 : false;
    if (!L->self_judged && pass_ok) dev_->lanes_commit(L->a, true);
    if (accepted) { L->valid = false; throw std::runtime_error("internal: a clean-data pass launched ahead of its chunk was never collected"); }
  }
  if (L->line_end) dev_->release(L->line_end);
  if (L->names) dev_->release(L->names);
  if (L->arena) dev_->release(L->arena);
  L->valid = false;
}

/* K1+K2 fused over buffer b.  Returns false (nothing launched, or results discarded) when the two-pass path must be used. */
bool FqEngine::try_fused_pass(int file, int b, bool last, uint32_t j0, uint64_t g0_local, FqName** names_out, uint32_t* names_cap, bool skip_lanes) {
  FqFile& F = f_[file];
  FqBuffer& B = F.bufs[b];
  int loop = loop_of(file);
  LanesLaunch L;
  if (pre_.valid) { /* this chunk's pass may be running already */
    if (pre_.file == file && pre_.data == B.data && pre_.n == B.n && pre_.lead == B.lead && pre_.j0 == j0 && pre_.last == last && !skip_lanes) { L = pre_; pre_.valid = false; }
    else lanes_discard(&pre_);
  }
  if (!L.valid) {
    if (loop == FQ_LOOP_MATE && total0() == 0) return false;
    if (F.limit != ~0ull) return false;
    if (F.sniff_fmt < 0) {
      if (F.nrec != 0 || F.pend_n != 0) return false;
      if (!presniff(file, B.data, B.n, j0, !lanes_ok_)) return false; /* the clean-data pass has no record-length limit */
    }
    lanes_prepare(file, B.data, B.n, B.lead, last, j0, g0_local, skip_lanes, &L);
  }
  if (L.hooked) hook_fired_ = true;
  B.line_end = L.line_end;
  uint32_t cap = L.cap, ncap = L.ncap;
  FqName* names = L.names;
  FqTileArgs a = L.a;
  const bool routed = L.routed, direct = L.direct, self_judged = L.self_judged;
  uint8_t* arena = L.arena; const uint64_t arena_units = L.arena_units;
  const int target = a.cx.loop == FQ_LOOP_MATE ? 0 : file;
  (void)cap;
  if (L.tried) {
    if (L.launched) {
      uint32_t o[FQ_LANES_OUT_WORDS];
      dev_->download(o, tile_out_, sizeof o);
      bool pass_ok = !o[1] && o[2] == kNone32 && !o[3] && !o[4];
      if (getenv("FQG_DEBUG")) fprintf(stderr, "[fqg] clean-data pass: n=%u j0=%u lines=%u capovf=%u overlong=%u anomaly=0x%x internal=%u virt=%u q=%u..%u rl=%u..%u recbad=%u | polls=%u lookback_rounds=%u waited=%u | arena %u of %llu units, accepted=%u, staged=%u\n",
                                       B.n, j0, o[0], o[1], o[2], o[3], o[4], o[5], o[6], o[7], o[8], o[9], o[10], o[11], o[12], o[13], o[24], (unsigned long long)arena_units, o[25], o[27]);
      bool accepted = self_judged ? o[25] != 0 : (pass_ok && !o[10]);
      if (routed && !(accepted && self_judged)) F.route_broken = true; /* names of this chunk did not reach the regions: the caller repeats the job */
      if (accepted && routed) F.route_chunks++;
      if (accepted) {
        if (!self_judged) dev_->lanes_commit(a, false);
        path_counts[0]++; fused_lanes_ = true;
        if (!direct) open_dirty_ = true;
        fused_direct_ = direct;
        B.nlines = o[0]; B.index_partial = self_judged; B.index_from = self_judged ? o[26] : 0; B.index_virtual_end = last;
        B.tail_from = o[0] > 8 ? o[0] - 8 : 0; B.tail_n = o[0] - B.tail_from;
        for (uint32_t i = 0; i < B.tail_n; i++) B.tail_ends[i] = o[16 + i];
        if (self_judged && arena) {
          fused_arena_ = arena; mem_stats[2] += arena_units * 16;
          F.arena_rate = std::max(F.arena_rate, (double)o[24] / kLanesTile); /* (the fullest tile's units: every tile gets the same stretch) */
        } else if (arena) dev_->release(arena);
        *names_out = names; *names_cap = ncap;
        launch_ahead(file, B, j0, g0_local); /* the next chunk's pass, before this chunk's bookkeeping */
        return true;
      }
      path_counts[1]++;
      if (self_judged && o[4] == 3) names_cap_full_ = true; /* (perhaps) more records than name descriptors */
      if (!self_judged && pass_ok) dev_->lanes_commit(a, true); /* counters went in before a record broke a length rule: take them back */
      if (self_judged && (o[3] & 16u) && arena) F.arena_rate = std::max(F.arena_rate, 1.5 * (double)o[24] / kLanesTile); /* (perhaps) ran out of arena: what the fullest tile asked for, and half as much again */
    } else { dev_->sync(); if (routed) F.route_broken = true; }
    if (arena) dev_->release(arena);
    a.arena = nullptr; a.arena_units = 0; a.route_world = 0;
    a.stats = f_[target].stats_open; a.hist = f_[target].hist_open; a.stats_range = f_[file].stats_open; /* the per-record kernels count into the open set */
    if (routed) { /* the per-record kernels deliver name descriptors: the caller packs them (fqg_names_pack_slots) */
      names = (FqName*)dev_->alloc((size_t)ncap * sizeof(FqName));
      a.names = names;
    }
  }
  if (B.lead) { /* the per-record kernels want the chunk's data at offset 0: the caller copies it and comes back */
    if (names) dev_->release(names);
    dev_->release(B.line_end); B.line_end = nullptr;
    return false;
  }
  uint32_t init[6] = {0, 0, kNone32, 0, 0, 0};
  dev_->upload(tile_out_, init, sizeof init);
  fused_lanes_ = false; fused_direct_ = false; open_dirty_ = true;
  bool launched = dev_->tile_pass(a);
  uint32_t out5[6] = {0, 0, kNone32, 0, 0, 0};
  if (launched) dev_->download(out5, tile_out_, sizeof out5); else dev_->sync();
  if (launched && !out5[1] && out5[2] == kNone32 && !out5[3] && !out5[4]) {
    B.nlines = out5[0]; B.index_partial = true; B.index_from = out5[5]; B.index_virtual_end = last;
    *names_out = names; *names_cap = ncap;
    path_counts[2]++;
    return true;
  }
  /* not usable: a line gzgets would split, a record longer than the window, more lines than guessed, or no such kernel */
  if (names) dev_->release(names);
  bool keep_index = launched && !out5[1] && !out5[4];
  if (keep_index) { B.nlines = out5[0]; B.index_partial = true; B.index_from = out5[5]; B.index_virtual_end = last; }
  else { dev_->release(B.line_end); B.line_end = nullptr; }
  if (launched) fused_fallback();
  else fused_ok_ = false;
  return false;
}

/* The pass of chunk k has told where its last complete record ends: chunk k+1 of the same fqg_feed_device call starts there (see
 * feed_device) and its pass is launched now, while the host still has chunk k's segment, name kernels and settling to do.  Only when
 * nothing can move that start: what is left behind the last record must be a plain partial record (no line gzgets would split). */
void FqEngine::launch_ahead(int file, const FqBuffer& B, uint32_t j0, uint64_t g0_local) {
  if (!next_.valid || next_.file != file) return;
  next_.valid = false;
  FqFile& F = f_[file];
  if (hook_ && F.route_world == 0) return; /* a caller that packs the name descriptors of finished chunks from its hook wants this chunk's segment first */
  if (B.nlines < j0 + 4u || !fused_ok_ || F.limit != ~0ull) return;
  const uint32_t nrec = (B.nlines - j0) / 4, idx = j0 + 4 * nrec - 1;
  if (idx < B.tail_from || idx >= B.tail_from + B.tail_n) return;
  const uint32_t end_off = B.tail_ends[idx - B.tail_from];
  uint32_t start = end_off;
  for (uint32_t i = idx + 1, c = 0; i <= B.nlines; i++, c++) { /* the lines behind the last record, and the bytes behind the last line */
    const uint32_t end = i < B.nlines ? B.tail_ends[i - B.tail_from] : B.n;
    if (end - start >= ((c & 1u) == 0 ? FQ_MAX_LABEL_LENGTH : FQ_MAX_READ_LENGTH)) return;
    start = end;
  }
  const size_t pend = B.n - end_off, own = B.n - B.lead;
  if (pend >= own / 2) return;
  uint8_t* p = next_.ptr - pend;
  const size_t rem = next_.remaining + pend;
  if (rem == 0) return;
  const size_t maxc = std::min(feed_chunk(), kMaxChunk - 16), k = std::min(rem, maxc);
  if (k < fused_min_) return;
  const uint32_t lead = (uint32_t)((uintptr_t)p & 15u);
  lanes_prepare(file, p - lead, (uint32_t)(k + lead), lead, next_.last && k == rem, 0, g0_local + nrec, false, &pre_);
  if (!pre_.tried) lanes_discard(&pre_);
}

/* the fused pass touched the global statistics / event key with results we cannot use: redo everything seen so far two-pass */
void FqEngine::fused_fallback() {
  fused_ok_ = false;
  path_counts[3]++;
  reprocess();
}

void FqEngine::add_buffer(int file, uint8_t* data, uint32_t n, bool last, bool owned, bool allow_fused, uint32_t lead) {
  FqFile& F = f_[file];
  if (F.ended) throw std::runtime_error("fqg_feed after the end of the file");
  if (cfg_.mode == FQG_MODE_INDEX_PAIR && file == 1 && !f_[0].ended) throw std::runtime_error("INDEX_PAIR: file 1 fed before file 0 ended");
  if (file >= nfiles()) throw std::runtime_error("file index out of range for this mode");
  F.fed = true;
  if (n == 0) {
    if (owned && data) dev_->release(data);
    if (last) flush_pending_as_last(file);
    return;
  }
  struct Depth { FqEngine* e; int file; Depth(FqEngine* e_, int f_) : e(e_), file(f_) { e->add_depth_++; } ~Depth() { e->add_depth_--; } } depth_guard(this, file);
  struct Settle { FqEngine* e; int file; ~Settle() { if (e->add_depth_ == 1 && !std::uncaught_exceptions()) e->try_settle(file); } } settle_guard{this, file};
  int b = (int)F.bufs.size();
  F.bufs.push_back(FqBuffer());
  mem_stats[0] += n;
  bool fused = false; uint32_t fused_j0 = 0, fused_ncap = 0; uint64_t fused_g0 = 0; FqName* fused_names = nullptr;
  {
    FqBuffer& B = F.bufs[b];
    B.data = data; B.n = n; B.owned = owned; B.lead = lead;
    bool cached = false;
    for (size_t i = 0; i < F.prescans.size(); i++) {
      FqFile::Prescan& ps = F.prescans[i];
      if (ps.data == data && ps.n == n && ps.last == last) { B.line_end = ps.line_end; B.nlines = ps.nlines; F.prescans.erase(F.prescans.begin() + i); cached = true; break; }
    }
    if (B.lead && (cached || !allow_fused || !fused_ok_ || n < fused_min_ || F.sniff_fmt < 0 || !F.started || F.pend_n > 0)) realign(B); /* a lead-in only where the clean-data pass may take it */
    if (!cached && allow_fused && fused_ok_ && n >= fused_min_) {
      fused_j0 = F.pend_n > 0 ? 4 - std::min<uint32_t>(F.pend_lfs, 3) : (F.started ? 0 : F.start_skip);
      fused_g0 = F.nrec + (F.pend_n > 0 ? 1 : 0);
      fused = try_fused_pass(file, b, last, fused_j0, fused_g0, &fused_names, &fused_ncap);
      if (!fused && F.bufs[b].lead) { /* only the clean-data pass takes a chunk with a lead-in: copy it, then the per-record kernels */
        realign(F.bufs[b]);
        if (fused_ok_) fused = try_fused_pass(file, b, last, fused_j0, fused_g0, &fused_names, &fused_ncap, true);
      }
    }
    if (!fused) realign(F.bufs[b]); /* (no fused pass at all) */
    if (!fused && !cached && !F.bufs[b].line_end) scan_buffer(F.bufs[b], last);
  }
  uint32_t pos = F.bufs[b].lead, j = 0;
  if (!F.started) { /* multi-GPU: the first lines of a range belong to the previous range's last record */
    F.started = true;
    if (F.start_skip) {
      if (F.bufs[b].nlines < F.start_skip) throw std::runtime_error("fqg_set_stream_start: the first buffer holds fewer lines than skip_lines");
      j = F.start_skip; pos = line_end_at(F.bufs[b], j - 1);
    }
  }
  /* bridge: finish the record that straddles the previous chunk boundary in a small chunk of its own */
  while (F.pend_n > 0 && !F.ended) {
    const FqBuffer B = F.bufs[b];
    uint32_t need = 4 - std::min<uint32_t>(F.pend_lfs, 3);
    uint32_t avail = B.nlines - j;
    if (avail >= need) {
      uint32_t cut = line_end_at(F.bufs[b], j + need - 1);
      size_t bn = F.pend_n + (cut - pos);
      uint8_t* bd = (uint8_t*)dev_->alloc(bn + kPad);
      dev_->copy(bd, F.pend, F.pend_n);
      dev_->copy(bd + F.pend_n, B.data + pos, cut - pos);
      dev_->fill(bd + bn, 0, kPad);
      F.pend_n = 0; F.pend_lfs = 0;
      bool blast = last && cut == B.n;
      pos = cut; j += need;
      add_buffer(file, bd, (uint32_t)bn, blast, true, false); /* may leave a new remainder in F.pend (over-long lines) */
    } else {
      append_pending(file, B.data + pos, B.n - pos, avail);
      pos = B.n; j = B.nlines;
      if (last) flush_pending_as_last(file);
      return;
    }
  }
  if (F.ended) return;
  if (fused) {
    /* the fused pass assumed: records start at line fused_j0 and the first one is record fused_g0 of the file */
    const FqBuffer B = F.bufs[b];
    if (j == fused_j0 && F.nrec == fused_g0 && F.pend_n == 0) {
      uint32_t nrec = (B.nlines - j) / 4;
      if (nrec > fused_ncap) nrec = fused_ncap; /* cannot happen: ncap = cap/4+1 and lines <= cap */
      if (nrec) {
        FqSegment s; s.buf = b; s.q = pos; s.j0 = j; s.nrec = nrec; s.fused = true;
        j += 4 * nrec;
        uint32_t end = line_end_at(F.bufs[b], j - 1);
        s.span = end - pos; pos = end;
        s.g0 = F.nrec; F.nrec += nrec; s.names = fused_names; s.lanes = fused_lanes_;
        if (fused_lanes_ && fused_direct_) { s.settled = true; mem_stats[3] += nrec; } /* (its statistics are in the main set already) */
        s.arena = fused_arena_; fused_arena_ = nullptr; /* the per-line mode of the clean-data pass put the names there itself */
        F.segs.push_back(s);
        if (s.arena) set_dir(file, F.segs.size() - 1); else gather_segment(file, F.segs.size() - 1, nrec);
        launch_names(file, F.segs.size() - 1, nrec);
      } else { if (fused_names) dev_->release(fused_names); if (fused_arena_) { dev_->release(fused_arena_); fused_arena_ = nullptr; } }
      segmentize(file, b, pos, j, last); /* what is left: fewer than four lines (over-long check, pending bytes / end of file) */
      return;
    }
    /* the bridge did not behave as assumed (over-long lines around the chunk boundary): discard the fused results */
    if (fused_names) dev_->release(fused_names);
    if (fused_arena_) { dev_->release(fused_arena_); fused_arena_ = nullptr; }
    fused_fallback();
  }
  segmentize(file, b, pos, j, last);
}

void FqEngine::segmentize(int file, int b, uint32_t pos, uint32_t j, bool last) {
  FqFile& F = f_[file];
  for (;;) {
    const FqBuffer B = F.bufs[b];
    uint32_t avail = B.nlines - j, nrec = avail / 4;
    uint32_t a = kNone32;
    if (B.index_partial && !(j >= 1 && j - 1 >= B.index_from) && !(B.nlines <= 8)) { ensure_full_index(F.bufs[b]); }
    if (avail <= 3 && B.tail_n && (avail == 0 || (j >= B.tail_from && j + avail <= B.tail_from + B.tail_n))) {
      /* the lines after the last complete record: their ends came back with the pass's result words */
      uint32_t total = avail + (last ? 0u : 1u), start = pos;
      for (uint32_t i = 0; i < total; i++) {
        uint32_t end = i < avail ? B.tail_ends[j + i - B.tail_from] : B.n;
        uint32_t lim = (i & 1u) == 0 ? FQ_MAX_LABEL_LENGTH : FQ_MAX_READ_LENGTH;
        if (end - start >= lim) { a = j + i; break; }
        start = end;
      }
    } else if (avail > 0 || (!last && pos < B.n)) {
      dev_->fill(scratch_, 0xFF, sizeof(uint32_t));
      dev_->find_overlong(B.line_end, pos, j, avail, B.n, last ? 0 : 1, scratch_);
      dev_->download(&a, scratch_, sizeof a);
    }
    uint32_t nfast = a == kNone32 ? nrec : std::min(nrec, (a - j) / 4);
    if (nfast) {
      FqSegment s; s.buf = b; s.q = pos; s.j0 = j; s.nrec = nfast;
      j += 4 * nfast;
      pos = line_end_at(F.bufs[b], j - 1);
      s.span = pos - s.q;
      add_segment(file, s);
    }
    if (a == kNone32) break;
    /* the record starting at pos holds a line that gzgets would split: emulate the four reads serially */
    FqLine* ld = (FqLine*)dev_->alloc(4 * sizeof(FqLine));
    dev_->split_serial(B.data, B.n, pos, last ? 1 : 0, ld, scratch_);
    uint32_t out3[3]; dev_->download(out3, scratch_, sizeof out3);
    if (out3[1] != 4) { dev_->release(ld); break; }
    FqSegment s; s.buf = b; s.q = pos; s.j0 = j; s.nrec = 1; s.explicit_lines = true; s.lines_dev = ld;
    dev_->download(s.lines_host, ld, 4 * sizeof(FqLine));
    s.span = out3[0] - pos;
    add_segment(file, s);
    pos = out3[0]; j += out3[2];
  }
  const FqBuffer B = F.bufs[b];
  if (last) end_file(file, B.data + pos, B.n - pos);
  else if (pos < B.n) append_pending(file, B.data + pos, B.n - pos, B.nlines - j);
}

/* The file ended; [tail, tail+n) holds fewer than four gz-lines.  Split them the way gzgets would. */
void FqEngine::end_file(int file, const uint8_t* dev_tail, size_t n) {
  FqFile& F = f_[file];
  F.tail.assign(n, 0);
  if (n) dev_->download(F.tail.data(), dev_tail, n);
  F.tail_lines.clear();
  size_t p = 0; int i = 0;
  while (p < n) {
    size_t maxb = ((i & 1) == 0 ? FQ_MAX_LABEL_LENGTH : FQ_MAX_READ_LENGTH) - 1, k = 0;
    while (k < maxb && p + k < n) { k++; if (F.tail[p + k - 1] == '\n') break; }
    FqTailLine tl; tl.off = (uint32_t)p; tl.len = (uint32_t)k;
    F.tail_lines.push_back(tl);
    p += k; i++;
  }
  F.ended = true;
}

/* ------------------------------------------------------------------------------------------------ name arena, settling */
/* the names of segment si leave their chunk (names_gather); the directory entry of the segment points at the copy */
void FqEngine::gather_segment(int file, size_t si, uint32_t nrec) {
  FqFile& F = f_[file];
  FqSegment& s = F.segs[si];
  if (s.names) {
    if (s.arena) { dev_->sync(); dev_->release(s.arena); s.arena = nullptr; } /* (a re-run: kernels of the side stream may still read the old copy) */
    dev_->fill(counters_ + 5, 0, 2 * sizeof(unsigned long long));
    dev_->names_measure(s.names, nrec, counters_ + 5);
    unsigned long long units = 0; dev_->download(&units, counters_ + 5, sizeof units);
    if (units * 16ull >= (1ull << 32)) throw std::runtime_error("internal: more than 4 GiB of read names in one chunk");
    s.arena = (uint8_t*)dev_->alloc((size_t)units * 16 + kPad);
    mem_stats[2] += units * 16;
    dev_->names_gather(s.names, F.bufs[s.buf].data, nrec, s.arena, counters_ + 6);
  }
  set_dir(file, si);
}
void FqEngine::set_dir(int file, size_t si) {
  FqFile& F = f_[file];
  const FqSegment& s = F.segs[si];
  if (F.dir_host.size() <= si) F.dir_host.resize(si + 1);
  FqDirEntry de; de.g0 = s.g0; de.names = s.names; de.data = s.arena;
  F.dir_host[si] = de;
  if (F.dir_synced > si) F.dir_synced = si;
}
void FqEngine::fold_open() {
  FqStats* m[2] = {f_[0].stats, f_[1].stats}; FqStats* o[2] = {f_[0].stats_open, f_[1].stats_open};
  unsigned long long* h[2] = {f_[0].hist, f_[1].hist}; unsigned long long* ho[2] = {f_[0].hist_open, f_[1].hist_open};
  dev_->stats_fold(m, o, h, ho);
}
void FqEngine::clear_open() {
  for (int f = 0; f < 2; f++) {
    FqStats init; memset(&init, 0, sizeof init);
    init.min_rl = 0xFFFFFFFFu; init.min_q = 255u;
    dev_->upload(f_[f].stats_open, &init, sizeof init);
    dev_->fill(f_[f].hist_open, 0, (size_t)FQ_MAX_READ_LENGTH * sizeof(unsigned long long));
    dev_->sync(); /* `init` is a stack object */
  }
}
/* main + open set of one file */
FqStats FqEngine::read_stats(int file) {
  FqStats m, o;
  dev_->download(&m, f_[file].stats, sizeof m); dev_->download(&o, f_[file].stats_open, sizeof o);
  m.num_rds += o.num_rds; m.mem_sum += o.mem_sum; m.n_names += o.n_names;
  m.min_rl = std::min(m.min_rl, o.min_rl); m.max_rl = std::max(m.max_rl, o.max_rl);
  m.min_q = std::min(m.min_q, o.min_q); m.max_q = std::max(m.max_q, o.max_q);
  return m;
}
void FqEngine::release_buffer(FqBuffer& B) {
  if (B.released) return;
  /* stream-ordered: every kernel that reads the chunk runs on the main stream and has been queued (the index kernels of the side
   * stream read names and arenas only) */
  if (B.owned && B.data) dev_->release(B.data);
  if (B.line_end) dev_->release(B.line_end);
  mem_stats[0] -= B.n; mem_stats[1] += B.n;
  B.data = nullptr; B.line_end = nullptr; B.owned = false; B.released = true;
}
/* The outermost add_buffer is done with its chunk.  While no event has fired, what was validated is final: the open statistics are
 * folded into the main set and the chunk's bytes go (the reference keeps nothing of a record but its name either,
 * src/fastq.c:396-439).  A chunk of the per-record kernels costs one look at the event key; a chunk of the clean-data pass, which
 * can raise none, costs nothing.  The first chunk that cannot be settled ends this: it and everything after it stay resident. */
void FqEngine::try_settle(int file) {
  if (!open_) return;
  FqFile& F = f_[file];
  bool look = false;
  for (size_t si = F.n_settled; si < F.segs.size(); si++) if (!F.segs[si].lanes) look = true;
  if (look) {
    unsigned long long k = 0; dev_->download(&k, key_, sizeof k);
    if (k != FQ_KEY_NONE || f_[0].limit != ~0ull || f_[1].limit != ~0ull) { open_ = false; return; }
  }
  if (open_dirty_) { fold_open(); open_dirty_ = false; }
  for (size_t si = F.n_settled; si < F.segs.size(); si++) if (!F.segs[si].settled) { F.segs[si].settled = true; mem_stats[3] += F.segs[si].nrec; }
  F.n_settled = F.segs.size();
  for (auto& B : F.bufs) release_buffer(B);
}
/* bytes of the normalised name of a record, from the arena (message details of the name events) */
void FqEngine::fetch_name(int file, uint64_t g, char* dst, uint32_t* len_out) {
  FqFile& F = f_[file];
  dst[0] = 0; *len_out = 0;
  if (F.segs.empty()) return;
  size_t lo = 0, hi = F.segs.size();
  while (hi - lo > 1) { size_t mid = (lo + hi) / 2; if (F.segs[mid].g0 <= g) lo = mid; else hi = mid; }
  const FqSegment& s = F.segs[lo];
  if (!s.names || !s.arena || g - s.g0 >= s.nrec) return;
  FqName nm; dev_->download(&nm, s.names + (g - s.g0), sizeof nm);
  uint32_t n = std::min<uint32_t>(nm.len, 1023);
  std::vector<uint8_t> tmp(n);
  if (n) dev_->download(tmp.data(), s.arena + nm.off, n);
  uint32_t k = 0; while (k < n && tmp[k] != 0) k++; /* (printed with %s by the reference) */
  memcpy(dst, tmp.data(), k); dst[k] = 0; *len_out = k;
}

void FqEngine::sync_dir(int file) {
  FqFile& F = f_[file];
  if (F.dir_synced == F.dir_host.size()) return;
  if (F.dir_host.size() > F.dir_cap) {
    size_t cap = std::max<size_t>(F.dir_host.size() * 2, 64);
    FqDirEntry* nd = (FqDirEntry*)dev_->alloc(cap * sizeof(FqDirEntry));
    if (F.dir_dev) { dev_->sync(); dev_->release(F.dir_dev); }
    F.dir_dev = nd; F.dir_cap = cap; F.dir_synced = 0;
  }
  dev_->upload(F.dir_dev + F.dir_synced, F.dir_host.data() + F.dir_synced, (F.dir_host.size() - F.dir_synced) * sizeof(FqDirEntry));
  /* no wait: a copy from pageable host memory has left the source buffer when cudaMemcpyAsync returns (it is staged), so dir_host
   * may grow or move afterwards */
  F.dir_synced = F.dir_host.size();
}

void FqEngine::add_segment(int file, FqSegment s) {
  FqFile& F = f_[file];
  s.g0 = F.nrec; F.nrec += s.nrec;
  if (loop_of(file) != FQ_LOOP_SINGLE && loop_of(file) != FQ_LOOP_READER) s.names = (FqName*)dev_->alloc((size_t)s.nrec * sizeof(FqName));
  F.segs.push_back(s);
  launch_segment(file, F.segs.size() - 1);
}

void FqEngine::record_lines(int file, uint64_t g, FqLine out[4], const uint8_t** data) {
  FqFile& F = f_[file];
  size_t lo = 0, hi = F.segs.size();
  while (hi - lo > 1) { size_t mid = (lo + hi) / 2; if (F.segs[mid].g0 <= g) lo = mid; else hi = mid; }
  const FqSegment& s = F.segs[lo];
  if (F.bufs[s.buf].released) throw std::runtime_error("internal: the lines of a record whose chunk has been released");
  ensure_full_index(F.bufs[s.buf]);
  const FqBuffer& B = F.bufs[s.buf];
  if (data) *data = B.data;
  if (s.explicit_lines) { memcpy(out, s.lines_host, 4 * sizeof(FqLine)); return; }
  uint32_t k = (uint32_t)(g - s.g0), j = s.j0 + 4 * k;
  uint32_t e[5];
  if (j == 0 || k == 0) { e[0] = s.q; dev_->download(e + 1, B.line_end + j, 4 * sizeof(uint32_t)); }
  else dev_->download(e, B.line_end + j - 1, 5 * sizeof(uint32_t));
  for (int i = 0; i < 4; i++) { out[i].off = e[i]; out[i].len = e[i + 1] - e[i]; }
}

void FqEngine::sniff_if_needed(int file, const FqSegment& s) {
  FqFile& F = f_[file];
  if (F.sniff_fmt >= 0 || s.g0 != 0) return;
  FqLine L[4]; const uint8_t* data;
  record_lines(file, 0, L, &data);
  dev_->sniff(data, L[0], L[1], (int32_t*)scratch_);
  int32_t out2[2]; dev_->download(out2, scratch_, sizeof out2);
  F.sniff_fmt = out2[0]; F.sniff_color = out2[1];
}

void FqEngine::ensure_table(uint64_t names_total) {
  if (slots_ && names_total * 2 <= table_cap_) return;
  uint64_t cap = pow2_at_least(std::max<uint64_t>(1u << 16, names_total * 4));
  if (slots_) { dev_->sync(); dev_->release(slots_); }
  slots_ = (FqSlot*)dev_->alloc(cap * sizeof(FqSlot));
  table_cap_ = cap;
  dev_->fill(slots_, 0xFF, cap * sizeof(FqSlot));
  /* re-insert what the smaller table held */
  uint64_t done = table_names_; table_names_ = 0;
  FqFile& F = f_[0];
  for (size_t si = 0; si < F.segs.size() && table_names_ < done; si++) {
    uint64_t lim = eff_records(F);
    if (F.segs[si].g0 >= lim) break;
    launch_names(0, si, (uint32_t)std::min<uint64_t>(F.segs[si].nrec, lim - F.segs[si].g0));
  }
}

void FqEngine::launch_names(int file, size_t si, uint32_t nrec) {
  FqFile& F = f_[file];
  const FqSegment& s = F.segs[si];
  int loop = loop_of(file);
  if (loop != FQ_LOOP_INDEX && loop != FQ_LOOP_MATE) return;
  if (cfg_.flags & FQG_FLAG_EXTERNAL_INDEX) return; /* the names go to the owners of their hashes instead (fqg_names_pack) */
  FqTableArgs t; memset(&t, 0, sizeof t);
  t.names = s.names; t.data = s.arena; t.nrec = nrec; t.g0 = s.g0; t.step_base = step_base(file);
  t.key = key_; t.counters = counters_;
  sync_dir(0);
  t.dir1 = f_[0].dir_dev; t.ndir1 = (uint32_t)f_[0].dir_host.size();
  if (loop == FQ_LOOP_INDEX) {
    ensure_table(table_names_ + nrec);
    t.slots = slots_; t.mask = table_cap_ - 1;
    dev_->index_insert(t);
    table_names_ += nrec;
  } else {
    ensure_table(table_names_);
    t.slots = slots_; t.mask = table_cap_ - 1;
    dev_->mate_claim(t);
  }
}

void FqEngine::launch_segment(int file, size_t si) {
  FqFile& F = f_[file];
  const FqSegment& s = F.segs[si];
  uint64_t lim = F.limit;
  if (s.g0 >= lim) return;
  if (loop_of(file) == FQ_LOOP_MATE && total0() == 0) return; /* "No reads found": file 2 is never opened */
  uint32_t nrec = (uint32_t)std::min<uint64_t>(s.nrec, lim - s.g0);
  if (s.fused || s.settled) { launch_names(file, si, nrec); return; } /* only reached when a table rebuild replays the name step */
  ensure_full_index(F.bufs[s.buf]);
  sniff_if_needed(file, s);
  const FqBuffer& B = F.bufs[s.buf];
  FqRecordsArgs a; memset(&a, 0, sizeof a);
  a.data = B.data; a.line_end = B.line_end; a.lines = s.explicit_lines ? s.lines_dev : nullptr;
  a.q = s.q; a.j0 = s.j0; a.nrec = nrec; a.span_bytes = s.span; a.g0 = s.g0 + F.g_base; a.step_base = step_base(file);
  a.cx = make_ctx(file);
  int target = a.cx.loop == FQ_LOOP_MATE ? 0 : file;
  a.stats = f_[target].stats_open; a.hist = f_[target].hist_open; a.stats_range = f_[file].stats_open;
  a.key = key_; a.names = s.names;
  open_dirty_ = true;
  dev_->records(a);
  gather_segment(file, si, nrec);
  launch_names(file, si, nrec);
}

/* interleaved mates and sorted pairs: compare the two names of every pair (fastq_info.c:86-91, :133-138) */
void FqEngine::launch_pairs() {
  if (cfg_.mode == FQG_MODE_INTERLEAVED) {
    FqFile& F = f_[0];
    uint64_t N = eff_records(F);
    const uint64_t gb = F.g_base; /* even: the pairs of this stream are records (2k, 2k + 1) of it, pair numbers continue at gb / 2 */
    for (size_t si = 0; si < F.segs.size(); si++) {
      const FqSegment& s = F.segs[si];
      if (s.g0 >= N) break;
      uint64_t end = std::min<uint64_t>(s.g0 + s.nrec, N);
      uint64_t e0 = s.g0 + (s.g0 & 1);
      const uint8_t* d = s.arena;
      if (e0 + 1 < end) {
        FqPairArgs p; memset(&p, 0, sizeof p);
        p.a = s.names + (e0 - s.g0); p.b = p.a + 1; p.da = p.db = d; p.stride_a = p.stride_b = 2;
        p.npairs = (uint32_t)((end - e0) / 2); p.p0 = (gb + e0) / 2; p.rank = FQ_RI_UNPAIRED; p.key = key_;
        dev_->pair_compare(p);
      }
      /* a pair split across two segments */
      if (((s.g0 + s.nrec) & 1) && s.g0 + s.nrec < N && si + 1 < F.segs.size()) {
        const FqSegment& t = F.segs[si + 1];
        FqPairArgs p; memset(&p, 0, sizeof p);
        p.a = s.names + (s.nrec - 1); p.da = d; p.b = t.names; p.db = t.arena; p.stride_a = p.stride_b = 1;
        p.npairs = 1; p.p0 = (gb + s.g0 + s.nrec - 1) / 2; p.rank = FQ_RI_UNPAIRED; p.key = key_;
        dev_->pair_compare(p);
      }
    }
  } else if (cfg_.mode == FQG_MODE_SORTED_PAIR) {
    uint64_t N = std::min(eff_records(f_[0]), eff_records(f_[1]));
    size_t i = 0, k = 0;
    while (i < f_[0].segs.size() && k < f_[1].segs.size()) {
      const FqSegment& s = f_[0].segs[i]; const FqSegment& t = f_[1].segs[k];
      uint64_t lo = std::max(s.g0, t.g0), hi = std::min<uint64_t>(std::min(s.g0 + s.nrec, t.g0 + t.nrec), N);
      if (lo < hi) {
        FqPairArgs p; memset(&p, 0, sizeof p);
        p.a = s.names + (lo - s.g0); p.da = s.arena; p.b = t.names + (lo - t.g0); p.db = t.arena;
        p.stride_a = p.stride_b = 1; p.npairs = (uint32_t)(hi - lo); p.p0 = lo; p.rank = FQ_RS_MISMATCH; p.key = key_;
        dev_->pair_compare(p);
      }
      if (s.g0 + s.nrec <= t.g0 + t.nrec) i++; else k++;
    }
  }
}

/* run every kernel again over the resident chunks (after a limit or the hash seed changed) */
void FqEngine::reprocess() {
  dev_->sync();
  /* limits changed: the two-pass kernels redo every segment that is not final; the final ones (their statistics are in the main set,
   * their chunks may be gone) only replay their name step into the cleared index */
  for (int f = 0; f < 2; f++) for (auto& s : f_[f].segs) if (!s.settled) { s.fused = false; s.lanes = false; }
  dev_->fill(key_, 0xFF, sizeof(unsigned long long));
  dev_->fill(counters_, 0, kCounters * sizeof(unsigned long long));
  clear_open();
  if (slots_) dev_->fill(slots_, 0xFF, table_cap_ * sizeof(FqSlot));
  table_names_ = 0;
  for (int f = 0; f < nfiles(); f++)
    for (size_t si = 0; si < f_[f].segs.size(); si++) launch_segment(f, si);
}

/* first byte of the gz-line with this index inside the file; -1 when the file has no such line */
int FqEngine::first_byte_of_line(int file, uint64_t gl) {
  FqFile& F = f_[file];
  uint64_t r = gl / 4;
  if (r < F.nrec) {
    {
      size_t lo = 0, hi = F.segs.size();
      while (hi - lo > 1) { size_t mid = (lo + hi) / 2; if (F.segs[mid].g0 <= r) lo = mid; else hi = mid; }
      if (F.segs[lo].settled) return '@'; /* a final record raised no reader event: none of its lines starts with NUL; only that is asked */
    }
    FqLine L[4]; const uint8_t* data;
    record_lines(file, r, L, &data);
    if (L[gl & 3].len == 0) return -1;
    uint8_t c; dev_->download(&c, data + L[gl & 3].off, 1);
    return c;
  }
  uint64_t ti = gl - 4 * F.nrec;
  if (ti < F.tail_lines.size() && F.tail_lines[ti].len) return F.tail[F.tail_lines[ti].off];
  return -1;
}

/* ------------------------------------------------------------------------------------------------ finish */
namespace {
struct HostEvent { uint64_t key; int code; int file; uint64_t line; uint64_t a; };
enum { PEEK_NONE = 0, PEEK_TRUNC = 1, PEEK_RECORD = 2 };
}

void FqEngine::finish(fqg_report* rep) {
  memset(rep, 0, sizeof *rep);
  rep->mode = cfg_.mode;
  for (int f = 0; f < nfiles(); f++)
    if (!f_[f].ended) {
      if (f == 1 && cfg_.mode == FQG_MODE_INDEX_PAIR && f_[0].ended) continue; /* caller stopped after file 1: allowed when file 1 failed */
      throw std::runtime_error("fqg_finish before the end of every file");
    }
  auto peek_record = [&](int file, uint64_t first_line) -> int { /* what fastq_read_entry would do from this line on */
    int b0 = first_byte_of_line(file, first_line);
    if (b0 <= 0) return PEEK_NONE;
    for (int i = 1; i < 4; i++) if (first_byte_of_line(file, first_line + i) <= 0) return PEEK_TRUNC;
    return PEEK_RECORD;
  };
  auto tail_first = [&](int file) -> int { /* -1 nothing left, else first byte of what is left */
    FqFile& F = f_[file];
    if (F.limit < F.nrec) return -1;
    return F.tail_lines.empty() ? -1 : (int)F.tail[0];
  };

  HostEvent ev; uint64_t dev_key = FQ_KEY_NONE; unsigned long long ctr[4] = {0, 0, 0, 0};
  bool sorted_end_f1 = false; uint64_t sorted_end_step = 0; bool have_end = false;
  bool sorted_validated[2] = {false, false};
  for (int attempt = 0;; attempt++) {
    if (attempt > 16) throw std::runtime_error("finish: too many reprocessing rounds");
    launch_pairs();
    dev_->sync(); /* the index kernels run on their own stream */
    dev_->download(&dev_key, key_, sizeof dev_key);
    dev_->download(ctr, counters_, sizeof ctr);
    if (ctr[2]) throw std::runtime_error("index table overflow");
    /* (two different names with one 64-bit hash are no event: the index kernels compare the bytes behind every equal hash and walk on) */
    /* events only the host can see: what is left at the end of each file */
    ev.key = FQ_KEY_NONE; ev.code = 0; ev.file = 0; ev.line = 0; ev.a = 0;
    auto offer = [&](uint64_t key, int code, int file, uint64_t line, uint64_t a) {
      if (key < ev.key) { ev.key = key; ev.code = code; ev.file = file; ev.line = line; ev.a = a; }
    };
    uint64_t N0 = eff_records(f_[0]), N1 = eff_records(f_[1]);
    int t0 = tail_first(0), t1 = nfiles() > 1 && f_[1].ended ? tail_first(1) : -1;
    have_end = false;
    switch (cfg_.mode) {
      case FQG_MODE_SINGLE: case FQG_MODE_INDEX:
        if (t0 > 0) offer(FQ_KEY(f_[0].g_base + N0, FQ_R_TRUNC), FQ_E_TRUNC, 0, 4 * (f_[0].g_base + N0), 0);
        break;
      case FQG_MODE_INDEX_PAIR:
        if (t0 > 0) offer(FQ_KEY(f_[0].g_base + N0, FQ_R_TRUNC), FQ_E_TRUNC, 0, 4 * (f_[0].g_base + N0), 0);
        if (total0() > 0 && f_[1].ended) {
          uint64_t S1 = total0() + 1;
          if (t1 > 0) offer(FQ_KEY(S1 + f_[1].g_base + N1, FQ_R_TRUNC), FQ_E_TRUNC, 1, 4 * (f_[1].g_base + N1), 0);
          if (!(cfg_.flags & FQG_FLAG_EXTERNAL_INDEX)) { /* sharded runs count the leftovers at the owners */
            FqStats st = read_stats(0);
            uint64_t left = st.n_names - ctr[1];
            if (left > 0) offer(FQ_KEY(S1 + N1 + 1, 0), FQ_E_LEFTOVER, 0, 0, left);
          }
        }
        break;
      case FQG_MODE_INTERLEAVED:
        if (f_[0].limit >= f_[0].nrec) {
          const uint64_t G0 = f_[0].g_base + N0; /* records of the file in front of what is left */
          if ((N0 & 1) == 0) { if (t0 > 0) offer(FQ_KEY(G0 / 2, FQ_RI_TRUNC1), FQ_E_TRUNC, 0, 4 * G0, 0); }
          else if (t0 > 0) offer(FQ_KEY(G0 / 2, FQ_RI_TRUNC2), FQ_E_TRUNC, 0, 4 * G0, 0);
          else offer(FQ_KEY(G0 / 2, FQ_RI_NOM2), FQ_E_TRUNC_PE, 0, 4 * G0, 0);
        }
        break;
      default: { /* sorted pair: the loop ends at the first file that runs out (fastq_info.c:121-141) */
        uint64_t k1 = t0 > 0 ? FQ_KEY_NONE : FQ_KEY(N0, FQ_RS_STOP1), k2 = t1 > 0 ? FQ_KEY_NONE : FQ_KEY(N1, FQ_RS_STOP2);
        if (t0 > 0) offer(FQ_KEY(N0, FQ_RS_TRUNC1), FQ_E_TRUNC, 0, 4 * N0, 0);
        if (t1 > 0) offer(FQ_KEY(N1, FQ_RS_TRUNC2), FQ_E_TRUNC, 1, 4 * N1, 0);
        uint64_t first_err = std::min(ev.key, dev_key);
        uint64_t kend = std::min(k1, k2);
        if (kend < first_err) { have_end = true; sorted_end_f1 = k1 < k2; sorted_end_step = sorted_end_f1 ? N0 : N1; }
        break;
      }
    }
    /* a record whose first line starts with NUL ends its file early (fastq.c:248): restrict and run again */
    uint64_t first = std::min(ev.key, dev_key);
    if (dev_key != FQ_KEY_NONE && dev_key == first && !(have_end)) {
      uint64_t step = FQ_KEY_STEP(dev_key); uint32_t rank = FQ_KEY_RANK(dev_key);
      bool restricted = false;
      switch (cfg_.mode) {
        case FQG_MODE_SINGLE: case FQG_MODE_INDEX:
          if (rank == FQ_R_STOP) { f_[0].limit = step - f_[0].g_base; restricted = true; }
          break;
        case FQG_MODE_INDEX_PAIR:
          if (rank == FQ_R_STOP) {
            if (step < total0() + 1) f_[0].limit = step - f_[0].g_base; else f_[1].limit = step - (total0() + 1) - f_[1].g_base;
            restricted = true;
          }
          break;
        case FQG_MODE_INTERLEAVED:
          if (rank == FQ_RI_STOP1) { f_[0].limit = 2 * step - f_[0].g_base; restricted = true; }
          break;
        default:
          if (rank == FQ_RS_STOP1) { f_[0].limit = step; f_[1].limit = std::min<uint64_t>(f_[1].limit, step); restricted = true; }
          else if (rank == FQ_RS_STOP2) { f_[1].limit = step; f_[0].limit = std::min<uint64_t>(f_[0].limit, step + 1); restricted = true; }
          break;
      }
      if (restricted) { reprocess(); continue; }
    }
    break;
  }

  uint64_t first = std::min(ev.key, dev_key);
  uint64_t N0 = eff_records(f_[0]), N1 = eff_records(f_[1]);
  /* sorted pair: the two reads after the loop (fastq_info.c:142-149) */
  if (cfg_.mode == FQG_MODE_SORTED_PAIR && have_end) {
    uint64_t k = sorted_end_step;
    /* a file that stopped on a NUL-led line has consumed only that line */
    bool f1_nul = sorted_end_f1 && first_byte_of_line(0, 4 * k) == 0;
    bool f2_nul = !sorted_end_f1 && first_byte_of_line(1, 4 * k) == 0;
    uint64_t next1 = sorted_end_f1 ? (f1_nul ? 4 * k + 1 : 4 * k + 4) : 4 * (k + 1);
    uint64_t next2 = sorted_end_f1 ? 4 * k : (f2_nul ? 4 * k + 1 : 4 * k + 4);
    uint64_t read1 = sorted_end_f1 ? k : k + 1; /* records file 1 has read */
    first = FQ_KEY_NONE; ev.key = FQ_KEY_NONE; dev_key = FQ_KEY_NONE;
    int p1 = peek_record(0, next1);
    if (p1 == PEEK_TRUNC) { ev.key = 0; ev.code = FQ_E_TRUNC; ev.file = 0; ev.line = 4 * read1; }
    else if (p1 == PEEK_RECORD) { ev.key = 0; ev.code = FQ_E_EOF2; ev.file = 0; }
    else {
      int p2 = peek_record(1, next2);
      if (p2 == PEEK_TRUNC) { ev.key = 0; ev.code = FQ_E_TRUNC; ev.file = 1; ev.line = 4 * k; }
      else if (p2 == PEEK_RECORD) { ev.key = 0; ev.code = FQ_E_EOF1; ev.file = 1; }
    }
    first = ev.key;
    if (first == FQ_KEY_NONE) { /* success: statistics cover exactly the records the loop validated */
      uint64_t l0 = read1, l1 = k;
      if (l0 < N0 || l1 < N1) { f_[0].limit = l0; f_[1].limit = l1; reprocess(); launch_pairs(); dev_->sync(); }
    }
    rep->reads_before_error[0] = k; rep->reads_before_error[1] = k;
    sorted_validated[0] = read1 >= 1; sorted_validated[1] = k >= 1;
    N0 = eff_records(f_[0]); N1 = eff_records(f_[1]);
  }

  rep->file[0].n_records = N0; rep->file[1].n_records = N1;
  for (int f = 0; f < 2; f++) { rep->file[f].sniff_format = -1; rep->file[f].color_space = -1; }
  if (first == FQ_KEY_NONE) {
    rep->error.code = FQG_OK;
    if (cfg_.mode != FQG_MODE_SORTED_PAIR) { rep->reads_before_error[0] = N0; rep->reads_before_error[1] = N1; }
    if (cfg_.mode == FQG_MODE_INTERLEAVED) rep->reads_before_error[0] = N0 / 2;
  } else if (first == ev.key) {
    fill_error(rep, FQ_KEY_NONE, ev.code, ev.file, ev.line, ev.a);
    if (cfg_.mode != FQG_MODE_SORTED_PAIR || !have_end) {
      uint64_t step = FQ_KEY_STEP(ev.key);
      if (cfg_.mode == FQG_MODE_INDEX_PAIR) {
        if (step <= N0) { rep->reads_before_error[0] = step; rep->reads_before_error[1] = 0; }
        else { rep->reads_before_error[0] = N0; rep->reads_before_error[1] = std::min<uint64_t>(step - (N0 + 1), N1); }
      } else { rep->reads_before_error[0] = step; rep->reads_before_error[1] = step; }
    }
  } else {
    fill_error(rep, dev_key, 0, 0, 0, 0);
  }
  rep->error.event_key = first;
  fill_stats(rep);
  /* which sniff lines the reference had printed by the time it stopped (SURVEY.md appendix A) */
  {
    uint64_t k = first;
    auto sniffed = [&](int f, uint64_t sniff_key) {
      if (f_[f].sniff_fmt < 0 || eff_records(f_[f]) == 0) return;
      if (k > sniff_key) { rep->file[f].sniff_format = f_[f].sniff_fmt; rep->file[f].color_space = f_[f].sniff_color; }
    };
    if (cfg_.mode == FQG_MODE_SORTED_PAIR && have_end) { /* the loop itself completed: a file was sniffed iff one of its records was validated */
      for (int f = 0; f < 2; f++)
        if (sorted_validated[f] && f_[f].sniff_fmt >= 0) { rep->file[f].sniff_format = f_[f].sniff_fmt; rep->file[f].color_space = f_[f].sniff_color; }
      k = 0;
    }
    switch (cfg_.mode) {
      case FQG_MODE_SINGLE: if (!reader_) sniffed(0, FQ_KEY(0, FQ_R_V0 + FQ_V_PLUS)); break; /* the reader tools never sniff */
      case FQG_MODE_INDEX: sniffed(0, FQ_KEY(0, FQ_R_WRONGHDR)); break;
      case FQG_MODE_INDEX_PAIR: sniffed(0, FQ_KEY(0, FQ_R_WRONGHDR)); sniffed(1, FQ_KEY(total0() + 1, FQ_R_WRONGHDR)); break;
      case FQG_MODE_INTERLEAVED: sniffed(0, FQ_KEY(0, FQ_RI_WRONGHDR1)); break;
      default: sniffed(0, FQ_KEY(0, FQ_RS_V1 + FQ_V_PLUS)); sniffed(1, FQ_KEY(0, FQ_RS_V2 + FQ_V_PLUS)); break;
    }
  }
  finished_ = true;
}

static void copy_cstr(char* dst, uint32_t* len_out, const std::vector<uint8_t>& src) {
  size_t n = 0;
  while (n < src.size() && n < 1023 && src[n] != 0) n++;
  memcpy(dst, src.data(), n); dst[n] = 0; *len_out = (uint32_t)n;
}

/* Build the error part of the report.  key != NONE: an event found on the device (needs the record's details). */
void FqEngine::fill_error(fqg_report* rep, uint64_t key, int host_code, int host_file, uint64_t host_line, uint64_t host_a) {
  fqg_error& e = rep->error;
  if (key == FQ_KEY_NONE) {
    e.code = host_code; e.file = host_file; e.msg_file = host_file; e.line = host_line; e.a = host_a;
    e.record = host_file == 0 ? eff_records(f_[0]) : eff_records(f_[1]);
    return;
  }
  uint64_t step = FQ_KEY_STEP(key); uint32_t rank = FQ_KEY_RANK(key);
  uint64_t N0 = cfg_.mode == FQG_MODE_INDEX_PAIR ? total0() : eff_records(f_[0]);
  int file = 0; uint64_t g = 0, L = 0; int code = 0; int vrank = -1; int msg_file = 0;
  switch (cfg_.mode) {
    case FQG_MODE_SINGLE: case FQG_MODE_INDEX: case FQG_MODE_INDEX_PAIR: {
      bool mate = cfg_.mode == FQG_MODE_INDEX_PAIR && step >= N0 + 1;
      file = mate ? 1 : 0; g = mate ? step - (N0 + 1) : step; msg_file = file;
      L = 4 * (g + 1); /* g is global here; made local below for the lookup */
      if (rank == FQ_R_TRUNC) { code = FQ_E_TRUNC; L = 4 * g; }
      else if (rank == FQ_R_WRONGHDR) code = FQ_E_WRONGHDR;
      else if (rank == FQ_R_NAME) code = mate ? FQ_E_UNPAIRED : FQ_E_DUP;
      else { vrank = (int)rank - FQ_R_V0; if (mate) { msg_file = 0; L = 4 * N0; } }
      rep->reads_before_error[0] = mate ? N0 : g; rep->reads_before_error[1] = mate ? g : 0;
      break;
    }
    case FQG_MODE_INTERLEAVED: {
      uint64_t p = step; L = 8 * (p + 1); g = 2 * p;
      if (rank == FQ_RI_TRUNC1) { code = FQ_E_TRUNC; L = 8 * p; }
      else if (rank == FQ_RI_NOM2) { code = FQ_E_TRUNC_PE; L = 8 * p + 4; g = 2 * p + 1; }
      else if (rank == FQ_RI_TRUNC2) { code = FQ_E_TRUNC; L = 8 * p + 4; g = 2 * p + 1; }
      else if (rank == FQ_RI_WRONGHDR1) code = FQ_E_WRONGHDR;
      else if (rank == FQ_RI_WRONGHDR2) { code = FQ_E_WRONGHDR; g = 2 * p + 1; }
      else if (rank == FQ_RI_UNPAIRED) code = FQ_E_UNPAIRED;
      else if (rank >= FQ_RI_V2) { vrank = (int)rank - FQ_RI_V2; g = 2 * p + 1; }
      else vrank = (int)rank - FQ_RI_V1;
      rep->reads_before_error[0] = p;
      break;
    }
    default: {
      uint64_t k = step; g = k; L = 4 * (k + 1);
      if (rank == FQ_RS_TRUNC1) { code = FQ_E_TRUNC; L = 4 * k; }
      else if (rank == FQ_RS_TRUNC2) { code = FQ_E_TRUNC; L = 4 * k; file = 1; }
      else if (rank == FQ_RS_MISMATCH) { code = FQ_E_MISMATCH; e.a = k + 2; }
      else if (rank >= FQ_RS_V2) { vrank = (int)rank - FQ_RS_V2; file = 1; }
      else vrank = (int)rank - FQ_RS_V1;
      msg_file = file;
      rep->reads_before_error[0] = k; rep->reads_before_error[1] = k;
      break;
    }
  }
  e.file = file; e.msg_file = msg_file; e.record = g;
  if (vrank < 0 && (code == FQ_E_DUP || code == FQ_E_UNPAIRED || code == FQ_E_MISMATCH)) {
    /* a name event: the message quotes the normalised name only, which lives in the arena (the record's chunk may be gone) */
    e.code = code; e.line = L;
    if (code != FQ_E_MISMATCH) fetch_name(file, g - f_[file].g_base, e.name, &e.name_len);
    return;
  }
  /* details from the record itself */
  FqLine Ls[4]; const uint8_t* data;
  record_lines(file, g - f_[file].g_base, Ls, &data);
  FqRecCtx cx = make_ctx(file);
  dev_->explain(data, Ls, cx, recout_);
  FqRecOut o; dev_->download(&o, recout_, sizeof o);
  if (vrank >= 0) {
    code = (int)o.code;
    if (code == FQ_E_BADCHAR) { L += 1; e.chr = (int32_t)o.bad; }
    else if (code == FQ_E_UT) L -= 2;
    else if (code == FQ_E_SHORT) { L += 1; e.a = o.slen; }
    else if (code == FQ_E_PLUS) L += 2;
    else if (code == FQ_E_LEN || code == FQ_E_LEN_CS) { e.a = o.slen; e.b = o.qlen; }
  }
  e.code = code; e.line = L;
  std::vector<uint8_t> tmp;
  auto fetch = [&](uint32_t off, uint32_t len, char* dst, uint32_t* lo) {
    tmp.assign(std::min<uint32_t>(len, 1023), 0);
    if (!tmp.empty()) dev_->download(tmp.data(), data + off, tmp.size());
    copy_cstr(dst, lo, tmp);
  };
  fetch(Ls[0].off, Ls[0].len, e.hdr1, &e.hdr1_len);
  fetch(Ls[2].off, Ls[2].len, e.hdr2, &e.hdr2_len);
  fetch(o.name_off, o.name_len, e.name, &e.name_len);
}

void FqEngine::fill_stats(fqg_report* rep) {
  dev_->sync();
  FqStats st[2];
  for (int f = 0; f < 2; f++) st[f] = read_stats(f);
  unsigned long long ctr[4]; dev_->download(ctr, counters_, sizeof ctr);
  for (int f = 0; f < 2; f++) {
    fqg_file_report& r = rep->file[f];
    r.num_rds = st[f].num_rds;
    r.min_rl = std::min<uint64_t>(FQ_MAX_READ_LENGTH, st[f].min_rl);
    r.max_rl = st[f].max_rl;
    /* (unsigned int)(char)c, fastq.c:374: bytes >= 0x80 become 0xFFFFFFxx */
    uint64_t mn = st[f].min_q >= 0x80 ? (0xFFFFFF00ull | st[f].min_q) : st[f].min_q;
    uint64_t mx = st[f].max_q >= 0x80 ? (0xFFFFFF00ull | st[f].max_q) : st[f].max_q;
    r.min_qual = std::min<uint64_t>(FQ_MAX_PHRED, mn);
    r.max_qual = mx;
  }
  rep->n_index_entries = st[0].n_names;
  rep->n_index_left = st[0].n_names - ctr[1];
  rep->index_mem = 8 + st[0].mem_sum + st[0].n_names * (16 + 1 + 24); /* fastq.c:609, fastq_info.c:293 */
  /* median_rl, fastq_info.c:39-55: file 1's histogram (the mate loop also counts into it) */
  const FqStats& s = st[0];
  bool fd2_null = cfg_.mode != FQG_MODE_INDEX_PAIR || !f_[1].fed || eff_records(f_[0]) == 0;
  uint64_t med = 1;
  if (s.num_rds == 1 && fd2_null) med = std::min<uint64_t>(FQ_MAX_READ_LENGTH, s.min_rl);
  else if (s.num_rds <= 1) med = FQ_MAX_READ_LENGTH;
  else {
    uint32_t lo = s.min_rl, hi = s.max_rl;
    if (cfg_.mode == FQG_MODE_INDEX_PAIR && st[1].max_rl > 0) { lo = std::min(lo, st[1].min_rl); hi = std::max(hi, st[1].max_rl); }
    std::vector<unsigned long long> h(hi - lo + 1), ho(hi - lo + 1);
    dev_->download(h.data(), f_[0].hist + lo, h.size() * sizeof(unsigned long long));
    dev_->download(ho.data(), f_[0].hist_open + lo, ho.size() * sizeof(unsigned long long));
    for (size_t i = 0; i < h.size(); i++) h[i] += ho[i];
    unsigned long long c = 0; med = FQ_MAX_READ_LENGTH;
    for (uint32_t l = lo; l <= hi; l++) { c += h[l - lo]; if (c > s.num_rds / 2) { med = l; break; } }
  }
  rep->median_rl = med;
}

/* The four gz-lines of the first `want` records the reader loop delivered (after fqg_finish, single-file loops fed as ONE chunk with
 * FQG_FLAG_KEEP_CHUNKS): offsets into that chunk.  For the tools that write records (src/fastq_truncate.c, src/fastq_filter_n.c). */
void FqEngine::record_table(uint64_t want, std::vector<FqLine>* lines4, const uint8_t** data) {
  FqFile& F = f_[0];
  lines4->clear(); *data = nullptr;
  uint64_t lim = std::min<uint64_t>(eff_records(F), want);
  if (lim == 0) return;
  if (F.bufs.empty()) return;
  for (auto& sg : F.segs) if (sg.buf != F.segs[0].buf) throw std::runtime_error("fqg_reader_tool_mem: the record-writing tools take the stream as one chunk");
  *data = F.bufs[F.segs[0].buf].data;
  lines4->reserve((size_t)lim * 4);
  for (auto& sg : F.segs) {
    if (sg.g0 >= lim) break;
    uint64_t nrec = std::min<uint64_t>(sg.nrec, lim - sg.g0);
    FqBuffer& B = F.bufs[sg.buf];
    if (sg.explicit_lines) { for (int i = 0; i < 4; i++) lines4->push_back(sg.lines_host[i]); continue; }
    ensure_full_index(B);
    std::vector<uint32_t> e((size_t)nrec * 4);
    dev_->download(e.data(), B.line_end + sg.j0, e.size() * sizeof(uint32_t));
    uint32_t start = sg.q;
    for (size_t i = 0; i < e.size(); i++) { FqLine L; L.off = start; L.len = e[i] - start; lines4->push_back(L); start = e[i]; }
  }
}
void FqEngine::count_n(const uint8_t* data, const std::vector<FqLine>& seq_lines, std::vector<uint32_t>* out2) {
  out2->assign(seq_lines.size() * 2, 0);
  if (seq_lines.empty()) return;
  FqLine* d = (FqLine*)dev_->alloc(seq_lines.size() * sizeof(FqLine));
  uint32_t* o = (uint32_t*)dev_->alloc(seq_lines.size() * 2 * sizeof(uint32_t));
  dev_->upload(d, seq_lines.data(), seq_lines.size() * sizeof(FqLine));
  dev_->count_n(data, d, (uint32_t)seq_lines.size(), o);
  dev_->download(out2->data(), o, out2->size() * sizeof(uint32_t));
  dev_->release(d); dev_->release(o);
}

FqName* FqEngine::header_names(const uint8_t* data, const std::vector<FqLine>& hdr_lines, int fmt, int is_pe) {
  if (hdr_lines.empty()) return nullptr;
  FqLine* d = (FqLine*)dev_->alloc(hdr_lines.size() * sizeof(FqLine));
  FqName* o = (FqName*)dev_->alloc(hdr_lines.size() * sizeof(FqName));
  dev_->upload(d, hdr_lines.data(), hdr_lines.size() * sizeof(FqLine));
  dev_->header_names(data, d, (uint32_t)hdr_lines.size(), fmt, is_pe, seed_, o);
  dev_->sync();
  dev_->release(d);
  return o;
}
void FqEngine::sniff_first(const uint8_t* data, FqLine hdr1, FqLine seq, int32_t* sniff_fmt, int32_t* color) {
  dev_->sniff(data, hdr1, seq, (int32_t*)scratch_);
  int32_t o2[2]; dev_->download(o2, scratch_, sizeof o2);
  *sniff_fmt = o2[0]; *color = o2[1];
}
void FqEngine::lookup_names(const FqName* dev_names, const uint8_t* data, uint32_t n, std::vector<unsigned long long>* idx) {
  idx->assign(n, FQ_IDX_NONE);
  if (!n || !slots_) return; /* (an empty index holds nothing) */
  FqTableArgs t; memset(&t, 0, sizeof t);
  t.names = dev_names; t.data = data; t.nrec = n; t.key = key_; t.counters = counters_;
  sync_dir(0);
  t.dir1 = f_[0].dir_dev; t.ndir1 = (uint32_t)f_[0].dir_host.size();
  t.slots = slots_; t.mask = table_cap_ - 1;
  unsigned long long* o = (unsigned long long*)dev_->alloc((size_t)n * sizeof(unsigned long long));
  dev_->names_lookup(t, o);
  dev_->download(idx->data(), o, (size_t)n * sizeof(unsigned long long));
  dev_->release(o);
}
void FqEngine::poly_at(const uint8_t* data, const std::vector<FqLine>& seq_lines, std::vector<uint32_t>* out3) {
  out3->assign(seq_lines.size() * 3, 0);
  if (seq_lines.empty()) return;
  FqLine* d = (FqLine*)dev_->alloc(seq_lines.size() * sizeof(FqLine));
  uint32_t* o = (uint32_t*)dev_->alloc(seq_lines.size() * 3 * sizeof(uint32_t));
  dev_->upload(d, seq_lines.data(), seq_lines.size() * sizeof(FqLine));
  dev_->poly_at(data, d, (uint32_t)seq_lines.size(), o);
  dev_->download(out3->data(), o, out3->size() * sizeof(uint32_t));
  dev_->release(d); dev_->release(o);
}

void FqEngine::index_records(const void* host_bytes, size_t n, uint64_t* starts, size_t cap, uint64_t* n_records) {
  if (n > kMaxChunk) throw std::runtime_error("fqg_index_records: at most 2 GiB per call");
  uint8_t* d = (uint8_t*)dev_->alloc(n + kPad);
  dev_->upload(d, host_bytes, n); dev_->fill(d + n, 0, kPad);
  uint32_t lcap = (uint32_t)(n / 32 + 4096); uint32_t* le; uint32_t out2[2];
  for (;;) {
    le = (uint32_t*)dev_->alloc((size_t)lcap * 4 + kPad);
    dev_->scan_lines(d, (uint32_t)n, 1, le, lcap, scratch_);
    dev_->download(out2, scratch_, sizeof out2);
    if (!out2[1]) break;
    dev_->release(le); lcap = out2[0];
  }
  uint64_t nrec = out2[0] / 4;
  *n_records = nrec;
  std::vector<uint32_t> h(out2[0]);
  if (out2[0]) dev_->download(h.data(), le, (size_t)out2[0] * 4);
  for (uint64_t i = 0; i < nrec && i < cap; i++) starts[i] = i == 0 ? 0 : h[4 * i - 1];
  dev_->release(le); dev_->release(d);
}

/* ------------------------------------------------------------------------------------------------ multi-GPU building blocks */
void FqEngine::prescan_device(int file, const void* dptr, size_t n, bool at_eof, uint64_t* n_lines, int32_t* ends_lf, uint64_t first_ends[4]) {
  FqFile& F = f_[file];
  const uint8_t* p = (const uint8_t*)dptr;
  for (int i = 0; i < 4; i++) first_ends[i] = ~0ull;
  uint8_t lastc = 0; dev_->download(&lastc, p + n - 1, 1);
  *ends_lf = lastc == '\n';
  if (fused_ok_ && n >= fused_min_) {
    /* the fused pass will build what it needs later: here only the LF count and the first line ends are wanted */
    {
      FqBuffer B; B.data = (uint8_t*)p; B.n = (uint32_t)std::min<size_t>(n, 1u << 20);
      scan_buffer(B, at_eof && B.n == n);
      uint32_t e[4]; uint32_t take = std::min<uint32_t>(4, B.nlines);
      if (take) dev_->download(e, B.line_end, take * sizeof(uint32_t));
      for (uint32_t i = 0; i < take; i++) first_ends[i] = e[i];
      /* any three lines in a row hold a sequence or a quality line: their longest is the line-length hint of this range
       * (a performance hint only: it picks the mode of the clean-data pass) */
      if (take == 4 && F.first_seq_len == 0) F.first_seq_len = std::max(std::max(e[1] - e[0], e[2] - e[1]), e[3] - e[2]);
      dev_->release(B.line_end);
      if (take < 4 && B.n < n) goto full_scan; /* very long first lines: take the exact path */
    }
    {
      unsigned long long* d = (unsigned long long*)dev_->alloc(sizeof(unsigned long long));
      dev_->fill(d, 0, sizeof(unsigned long long));
      size_t left = n; const uint8_t* q = p;
      while (left) { size_t k = std::min(left, kMaxChunk); dev_->count_lines(q, (uint32_t)k, d); q += k; left -= k; }
      unsigned long long total = 0; dev_->download(&total, d, sizeof total);
      dev_->release(d);
      *n_lines = total + ((at_eof && lastc != '\n') ? 1 : 0);
      return;
    }
  }
full_scan:
  {
    uint64_t total = 0, off = 0; int got = 0;
    for (int i = 0; i < 4; i++) first_ends[i] = ~0ull;
    while (n) {
      size_t k = std::min(n, kMaxChunk);
      FqBuffer B; B.data = (uint8_t*)p; B.n = (uint32_t)k;
      bool last = at_eof && k == n;
      scan_buffer(B, last);
      if (got < 4 && B.nlines) {
        uint32_t e[4]; uint32_t take = std::min<uint32_t>(4 - got, B.nlines);
        dev_->download(e, B.line_end, take * sizeof(uint32_t));
        for (uint32_t i = 0; i < take; i++) first_ends[got++] = off + e[i];
      }
      FqFile::Prescan ps; ps.data = p; ps.n = (uint32_t)k; ps.last = last; ps.line_end = B.line_end; ps.nlines = B.nlines;
      F.prescans.push_back(ps);
      total += B.nlines; p += k; n -= k; off += k;
    }
    *n_lines = total;
  }
}

void FqEngine::set_stream_start(int file, uint32_t skip_lines, uint64_t first_record) {
  FqFile& F = f_[file];
  if (F.started) throw std::runtime_error("fqg_set_stream_start after the first feed");
  /* (interleaved: a range starts with the first mate of a pair, so the offset is even; a pair never straddles two ranks) */
  if (first_record && !(cfg_.mode == FQG_MODE_SINGLE || (cfg_.mode == FQG_MODE_INTERLEAVED && (first_record & 1) == 0) ||
                        ((cfg_.mode == FQG_MODE_INDEX || cfg_.mode == FQG_MODE_INDEX_PAIR) && (cfg_.flags & FQG_FLAG_EXTERNAL_INDEX))))
    throw std::runtime_error("fqg_set_stream_start: a record offset needs FQG_MODE_SINGLE, FQG_MODE_INTERLEAVED with an even offset, or an index mode with FQG_FLAG_EXTERNAL_INDEX");
  F.start_skip = skip_lines; F.g_base = first_record;
}

void FqEngine::names_count(int file, uint32_t world, uint64_t* counts, uint64_t* bytes) {
  if (world == 0 || world > FQ_SHARD_MAX_SRC) throw std::runtime_error("fqg_names_count: world out of range");
  FqFile& F = f_[file];
  unsigned long long* d = (unsigned long long*)dev_->alloc(2 * world * sizeof(unsigned long long));
  dev_->fill(d, 0, 2 * world * sizeof(unsigned long long));
  uint64_t lim = eff_records(F);
  for (auto& s : F.segs) {
    if (s.g0 >= lim || !s.names) continue;
    dev_->names_count(s.names, (uint32_t)std::min<uint64_t>(s.nrec, lim - s.g0), world, d);
  }
  std::vector<unsigned long long> h(2 * world);
  dev_->download(h.data(), d, h.size() * sizeof(unsigned long long));
  for (uint32_t o = 0; o < world; o++) { counts[o] = h[2 * o]; bytes[o] = h[2 * o + 1]; }
  for (uint32_t o = 0; o < world; o++)
    if (bytes[o] >= (1ull << 32)) { dev_->release(d); throw std::runtime_error("fqg_names_count: more than 4 GiB of read-name bytes for one owner (the packed offsets are 32-bit): use more ranks or the pipelined routing"); }
  dev_->release(d);
}

void FqEngine::names_pack(int file, uint32_t world, void* meta, void* blob, const uint64_t* meta_base, const uint64_t* blob_base) {
  if (world == 0 || world > FQ_SHARD_MAX_SRC) throw std::runtime_error("fqg_names_pack: world out of range");
  FqFile& F = f_[file];
  std::vector<unsigned long long> h(2 * world);
  for (uint32_t o = 0; o < world; o++) { h[2 * o] = meta_base[o]; h[2 * o + 1] = blob_base[o]; }
  unsigned long long* base = (unsigned long long*)dev_->alloc(4 * world * sizeof(unsigned long long));
  unsigned long long* cursor = base + 2 * world;
  dev_->upload(base, h.data(), 2 * world * sizeof(unsigned long long));
  dev_->fill(cursor, 0, 2 * world * sizeof(unsigned long long));
  uint64_t lim = eff_records(F);
  for (auto& s : F.segs) {
    if (s.g0 >= lim || !s.names) continue;
    dev_->names_pack(s.names, s.arena, (uint32_t)std::min<uint64_t>(s.nrec, lim - s.g0), s.g0 + F.g_base, world,
                     (FqPackedName*)meta, (uint8_t*)blob, base, cursor);
  }
  dev_->sync(); /* h is a local */
  dev_->release(base);
}

uint64_t FqEngine::names_new(int file) {
  FqFile& F = f_[file];
  uint64_t lim = eff_records(F), n = 0;
  for (size_t si = F.routed_segs; si < F.segs.size(); si++) {
    const FqSegment& s = F.segs[si];
    if (s.g0 >= lim || !s.names) continue;
    n += std::min<uint64_t>(s.nrec, lim - s.g0);
  }
  return n;
}

void FqEngine::names_pack_slots(int file, uint32_t world, void* const* region_ptrs, uint64_t cap, uint32_t units) {
  if (world == 0 || world > FQ_SHARD_MAX_SRC) throw std::runtime_error("fqg_names_pack_slots: world out of range");
  if (!(cfg_.flags & FQG_FLAG_EXTERNAL_INDEX)) throw std::runtime_error("fqg_names_pack_slots needs FQG_FLAG_EXTERNAL_INDEX");
  if (units > 62) throw std::runtime_error("fqg_names_pack_slots: at most 62 name units (a read name is shorter than 1000 bytes)");
  FqFile& F = f_[file];
  FqRegionPtrs R; memset(&R, 0, sizeof R);
  for (uint32_t o = 0; o < world; o++) { if (!region_ptrs[o]) throw std::runtime_error("fqg_names_pack_slots: null region"); R.region[o] = (uint8_t*)region_ptrs[o]; }
  const bool beside = in_beside_hook_;
  dev_->route_begin(route_cursors_, world, beside);
  uint64_t lim = eff_records(F);
  for (size_t si = F.routed_segs; si < F.segs.size(); si++) {
    const FqSegment& s = F.segs[si];
    if (s.g0 >= lim || !s.names) continue;
    dev_->names_pack_slots(s.names, s.arena, (uint32_t)std::min<uint64_t>(s.nrec, lim - s.g0), s.g0 + F.g_base, world, R, cap, units, route_cursors_);
  }
  dev_->route_end(route_cursors_, world, R, cap);
  F.routed_segs = F.segs.size();
}

void FqEngine::shard_reserve(uint64_t n_names) {
  if (table_names_) throw std::runtime_error("fqg_shard_reserve after the first insert");
  ensure_table(std::max<uint64_t>(n_names, 1));
}

void FqEngine::shard_insert_slots(const void* regions, uint32_t n_src, size_t region_bytes, uint32_t nblocks, uint64_t stride, uint32_t units, bool beside, const void* flags, uint64_t expect) {
  if (n_src == 0 || n_src > FQ_SHARD_MAX_SRC) throw std::runtime_error("fqg_shard_insert_slots: n_src out of range");
  if (!slots_) ensure_table(1);
  dev_->shard_insert_slots((const uint8_t*)regions, n_src, region_bytes, nblocks, stride, units, slots_, table_cap_ - 1, counters_, beside, (const unsigned long long*)flags, expect);
  table_names_ = 1; /* the table holds names the engine cannot re-insert: it must not grow any more */
}
void FqEngine::shard_claim_slots(const void* regions, uint32_t n_src, size_t region_bytes, uint32_t nblocks, uint64_t stride, uint32_t units, bool beside, const void* flags, uint64_t expect) {
  if (n_src == 0 || n_src > FQ_SHARD_MAX_SRC) throw std::runtime_error("fqg_shard_claim_slots: n_src out of range");
  if (!units) throw std::runtime_error("fqg_shard_claim_slots: the mate loop compares names, the slots must carry their bytes");
  if (!slots_) ensure_table(1);
  dev_->shard_claim_slots((const uint8_t*)regions, n_src, region_bytes, nblocks, stride, units, slots_, table_cap_ - 1, counters_, beside, (const unsigned long long*)flags, expect);
}
/* sharded runs: the clean-data pass of every chunk of `file` writes the names straight into per-owner regions (include/fastq_gpu.h) */
void FqEngine::set_route(int file, uint32_t world, void* const* region_ptrs, size_t region_bytes, uint32_t depth, uint32_t stride, uint32_t units) {
  if (!(cfg_.flags & FQG_FLAG_EXTERNAL_INDEX)) throw std::runtime_error("fqg_set_route needs FQG_FLAG_EXTERNAL_INDEX");
  if (world > FQ_ROUTE_MAX_WORLD) throw std::runtime_error("fqg_set_route: too many owners for the pass to write to directly");
  if (units > 62) throw std::runtime_error("fqg_set_route: at most 62 name units");
  FqFile& F = f_[file];
  F.route_world = world; F.route_bytes = region_bytes; F.route_depth = depth ? depth : 1; F.route_stride = stride; F.route_units = units;
  for (uint32_t o = 0; o < world; o++) { if (!region_ptrs[o]) throw std::runtime_error("fqg_set_route: null region"); F.route_region[o] = (uint8_t*)region_ptrs[o]; }
}

void FqEngine::shard_slots_result(uint64_t* inserted, uint64_t* equal_hashes, int32_t* overflow, uint64_t* claimed, uint64_t* unpaired) {
  dev_->sync();
  unsigned long long ctr[kCounters]; dev_->download(ctr, counters_, sizeof ctr);
  *inserted = ctr[1]; *equal_hashes = ctr[0]; *claimed = ctr[8]; *unpaired = ctr[9];
  *overflow = (ctr[2] != 0 || ctr[1] * 2 > table_cap_) ? 1 : 0; /* above half full the probe sequences get long: let the exact path size the table */
}

void FqEngine::shard_insert(const void* meta, uint64_t n, const void* blob, uint32_t n_src, const uint64_t* meta_start, const uint64_t* blob_start) {
  if (n_src == 0 || n_src > FQ_SHARD_MAX_SRC) throw std::runtime_error("fqg_shard_insert: n_src out of range");
  if (n >= (1ull << FQ_SHARD_POS_BITS)) throw std::runtime_error("fqg_shard_insert: more than 2^28 names for one owner");
  dev_->fill(counters_ + 3, 0xFF, sizeof(unsigned long long));
  shard_meta_ = (const FqPackedName*)meta; shard_n_ = n; shard_blob_ = (const uint8_t*)blob; shard_nsrc_ = n_src;
  for (uint32_t i = 0; i <= n_src; i++) shard_meta_start_[i] = meta_start[i];
  for (uint32_t i = 0; i < n_src; i++) shard_blob_start_[i] = blob_start[i];
  if (!n) return;
  table_names_ = 0;
  ensure_table(n);
  FqShardArgs a; memset(&a, 0, sizeof a);
  a.meta = shard_meta_; a.n = n; a.blob = shard_blob_; a.n_src = n_src;
  memcpy(a.meta_start, shard_meta_start_, sizeof(unsigned long long) * (n_src + 1));
  memcpy(a.blob_start, shard_blob_start_, sizeof(unsigned long long) * n_src);
  a.slots = slots_; a.mask = table_cap_ - 1; a.dup_key = counters_ + 3; a.counters = counters_;
  dev_->shard_insert(a);
  table_names_ = n;
}

void FqEngine::shard_result(uint64_t* key, uint64_t* record, char* name, uint32_t* name_len, uint64_t* collisions) {
  dev_->sync();
  unsigned long long ctr[4]; dev_->download(ctr, counters_, sizeof ctr);
  if (ctr[2]) throw std::runtime_error("index table overflow");
  *collisions = ctr[0]; *key = ctr[3]; *record = 0; *name_len = 0; name[0] = 0;
  if (ctr[3] == FQ_KEY_NONE || !shard_n_) return;
  *record = FQ_KEY_STEP(ctr[3]);
  unsigned long long* d = (unsigned long long*)dev_->alloc(sizeof(unsigned long long));
  dev_->fill(d, 0xFF, sizeof(unsigned long long));
  dev_->shard_find(shard_meta_, shard_n_, *record, d);
  unsigned long long pos; dev_->download(&pos, d, sizeof pos);
  dev_->release(d);
  if (pos == ~0ull) return;
  FqPackedName pn; dev_->download(&pn, shard_meta_ + pos, sizeof pn);
  uint32_t src = 0; while (src + 1 < shard_nsrc_ && pos >= shard_meta_start_[src + 1]) src++;
  uint32_t len = std::min<uint32_t>(pn.len, 1023);
  if (len) dev_->download(name, shard_blob_ + shard_blob_start_[src] + pn.off, len);
  name[len] = 0; *name_len = len;
}

void FqEngine::hist_range(int file, uint64_t lo, uint64_t hi, uint64_t* out) {
  if (hi < lo || hi >= FQ_MAX_READ_LENGTH) throw std::runtime_error("fqg_hist_range: bad range");
  dev_->download(out, f_[file].hist + lo, (hi - lo + 1) * sizeof(unsigned long long));
  std::vector<unsigned long long> ho(hi - lo + 1);
  dev_->download(ho.data(), f_[file].hist_open + lo, ho.size() * sizeof(unsigned long long));
  for (size_t i = 0; i < ho.size(); i++) out[i] += ho[i];
}

void FqEngine::set_file_total(int file, uint64_t total) {
  if (file != 0) throw std::runtime_error("fqg_set_file_total: only file 0 has a total that other loops depend on");
  total0_set_ = true; total0_ = total;
}
uint64_t FqEngine::collisions_walked() { dev_->sync(); unsigned long long v = 0; dev_->download(&v, counters_ + 4, sizeof v); return v; }
void FqEngine::set_sniff(int file, int fmt, int color) { f_[file].sniff_fmt = fmt; f_[file].sniff_color = color; }
void FqEngine::sniff_device(int file, const void* dptr, size_t n, uint32_t skip, int32_t* fmt, int32_t* color) {
  FqFile& F = f_[file];
  int sf = F.sniff_fmt, sc = F.sniff_color;
  F.sniff_fmt = -1; F.sniff_color = -1;
  presniff(file, (const uint8_t*)dptr, (uint32_t)std::min<size_t>(n, kMaxChunk), skip, false);
  *fmt = F.sniff_fmt; *color = F.sniff_color;
  F.sniff_fmt = sf; F.sniff_color = sc;
}

void FqEngine::shard_claim(const void* meta, uint64_t n, const void* blob, uint32_t n_src, const uint64_t* meta_start, const uint64_t* blob_start, uint64_t sb) {
  if (n_src == 0 || n_src > FQ_SHARD_MAX_SRC) throw std::runtime_error("fqg_shard_claim: n_src out of range");
  dev_->sync();
  dev_->fill(counters_ + 3, 0xFF, sizeof(unsigned long long));
  dev_->fill(counters_ + 1, 0, sizeof(unsigned long long));
  claim_meta_ = (const FqPackedName*)meta; claim_n_ = n; claim_blob_ = (const uint8_t*)blob; claim_nsrc_ = n_src;
  for (uint32_t i = 0; i <= n_src; i++) claim_meta_start_[i] = meta_start[i];
  for (uint32_t i = 0; i < n_src; i++) claim_blob_start_[i] = blob_start[i];
  if (!n) return;
  ensure_table(table_names_);
  FqShardArgs a; memset(&a, 0, sizeof a);
  a.meta = claim_meta_; a.n = n; a.blob = claim_blob_; a.n_src = n_src;
  memcpy(a.meta_start, claim_meta_start_, sizeof(unsigned long long) * (n_src + 1));
  memcpy(a.blob_start, claim_blob_start_, sizeof(unsigned long long) * n_src);
  a.slots = slots_; a.mask = table_cap_ - 1; a.dup_key = counters_ + 3; a.counters = counters_;
  /* the names the slots point at: the tuples inserted before */
  FqShardArgs ins; memset(&ins, 0, sizeof ins);
  ins.meta = shard_meta_; ins.n = shard_n_; ins.blob = shard_blob_; ins.n_src = shard_nsrc_;
  memcpy(ins.meta_start, shard_meta_start_, sizeof(unsigned long long) * (shard_nsrc_ + 1));
  memcpy(ins.blob_start, shard_blob_start_, sizeof(unsigned long long) * shard_nsrc_);
  claim_sb_ = sb;
  dev_->shard_claim(a, ins, sb);
}

void FqEngine::shard_claim_result(uint64_t* key, uint64_t* record, char* name, uint32_t* name_len, uint64_t* claimed, uint64_t* collisions) {
  dev_->sync();
  unsigned long long ctr[4]; dev_->download(ctr, counters_, sizeof ctr);
  *collisions = ctr[0]; *claimed = ctr[1]; *key = ctr[3]; *record = 0; *name_len = 0; name[0] = 0;
  if (ctr[3] == FQ_KEY_NONE || !claim_n_) return;
  *record = FQ_KEY_STEP(ctr[3]) - claim_sb_; /* index of the unpaired record inside file 2 */
  unsigned long long* d = (unsigned long long*)dev_->alloc(sizeof(unsigned long long));
  dev_->fill(d, 0xFF, sizeof(unsigned long long));
  dev_->shard_find(claim_meta_, claim_n_, *record, d);
  unsigned long long pos; dev_->download(&pos, d, sizeof pos);
  dev_->release(d);
  if (pos == ~0ull) return;
  FqPackedName pn; dev_->download(&pn, claim_meta_ + pos, sizeof pn);
  uint32_t src = 0; while (src + 1 < claim_nsrc_ && pos >= claim_meta_start_[src + 1]) src++;
  uint32_t len = std::min<uint32_t>(pn.len, 1023);
  if (len) dev_->download(name, claim_blob_ + claim_blob_start_[src] + pn.off, len);
  name[len] = 0; *name_len = len;
}
