/*
 * fq_engine.h — host side of libfastq_gpu: turns a stream of byte chunks per file into kernel launches and the
 * kernels' results into the report of include/fastq_gpu.h.  No FASTQ byte is interpreted on the host except the
 * (< 1 record) tail left at the end of a file, which is what the reference's reader sees when it hits EOF.
 */
#ifndef FQ_ENGINE_H
#define FQ_ENGINE_H
#include <stdexcept>
#include <string>
#include <vector>
#include "../../include/fastq_gpu.h"
#include "fq_device.h"

struct FqBuffer {
  uint8_t* data = nullptr;   /* device */
  uint32_t n = 0;
  uint32_t lead = 0;         /* bytes in front of the chunk's own data (a chunk borrowed at an unaligned address starts at the 16-byte boundary below it) */
  bool owned = false;
  uint32_t* line_end = nullptr;
  uint32_t nlines = 0;       /* lines with an end inside the buffer (a final LF-less line counts when the file ended here) */
  bool index_partial = false; /* fused pass: only line ends [0,8) and [index_from, nlines) are stored */
  uint32_t index_from = 0;
  bool index_virtual_end = false;
  /* the last line ends of the chunk, read back together with the pass's result words: the host needs only these (where the last
   * complete record ends, how long the lines after it are) and would otherwise fetch them one synchronising copy at a time */
  uint32_t tail_from = 0, tail_n = 0, tail_ends[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  bool released = false;     /* every record of the chunk is final and its names live in the arena: the bytes and the line index are gone */
};

struct FqSegment {
  int buf = -1;
  uint32_t q = 0, j0 = 0, nrec = 0;
  uint64_t span = 0;
  bool explicit_lines = false;
  bool fused = false;        /* validated by the fused pass already: only the name step remains */
  FqLine lines_host[4];
  FqLine* lines_dev = nullptr;
  uint64_t g0 = 0;
  FqName* names = nullptr;   /* device, nrec entries (NULL for the single loop) */
  uint8_t* arena = nullptr;  /* device: the bytes of the segment's names, copied out of the chunk (names[k].off points in here) */
  bool settled = false;      /* final: validated without an event, statistics in the main set; the chunk's bytes are not needed again */
  bool lanes = false;        /* validated by the clean-data pass (`fused` says: by one of the two fused passes) */
};

struct FqTailLine { uint32_t off, len; };

struct FqFile {
  std::vector<FqBuffer> bufs;
  std::vector<FqSegment> segs;
  uint64_t nrec = 0;
  /* bytes after the last complete record of the buffers seen so far (device) */
  uint8_t* pend = nullptr; size_t pend_n = 0, pend_cap = 0; uint32_t pend_lfs = 0;
  bool fed = false, ended = false;
  /* what is left when the file ended: < 4 gz-lines, interpreted on the host like the reference's reader at EOF */
  std::vector<uint8_t> tail;
  std::vector<FqTailLine> tail_lines;
  int sniff_fmt = -1, sniff_color = -1;
  uint32_t first_seq_len = 0; /* raw length of the first record's sequence line (0: not seen by this context) */
  uint32_t first_hdr_len = 0; /* ... and of its header line */
  double arena_rate = 0;      /* 16-byte arena units per input byte the chunks so far needed (sizes the next chunk's block) */
  FqStats* stats = nullptr; unsigned long long* hist = nullptr; /* device: records that are final */
  FqStats* stats_open = nullptr; unsigned long long* hist_open = nullptr; /* device: records a later event may still exclude (DESIGN.md §3) */
  size_t n_settled = 0;     /* segments [0, n_settled) are final */
  FqDirEntry* dir_dev = nullptr; size_t dir_cap = 0; std::vector<FqDirEntry> dir_host; size_t dir_synced = 0;
  uint64_t limit = ~0ull;   /* records at or beyond this index are never read (early clean end of file) */
  /* multi-GPU: this context holds a range of the file */
  uint64_t g_base = 0;      /* index (inside the whole file) of the first record of this stream */
  uint32_t start_skip = 0;  /* lines of the first buffer that belong to the previous range */
  bool started = false;
  size_t routed_segs = 0;   /* pipelined routing: segments [0, routed_segs) have been packed by names_pack_slots */
  /* pipelined routing by the clean-data pass itself: chunk n of the file writes into region_o + (n % depth) * bytes */
  uint32_t route_world = 0, route_depth = 1, route_stride = 0, route_units = 0; size_t route_bytes = 0;
  uint8_t* route_region[FQ_ROUTE_MAX_WORLD] = {nullptr};
  uint64_t route_chunks = 0; bool route_broken = false;
  struct Prescan { const uint8_t* data; uint32_t n; bool last; uint32_t* line_end; uint32_t nlines; };
  std::vector<Prescan> prescans;
};

/* a clean-data pass that has been prepared (buffers) and perhaps launched, not collected yet */
struct LanesLaunch {
  bool valid = false; int file = 0; uint8_t* data = nullptr; uint32_t n = 0, lead = 0, j0 = 0; bool last = false;
  uint32_t cap = 0, ncap = 0; uint32_t* line_end = nullptr; FqName* names = nullptr; uint8_t* arena = nullptr; uint64_t arena_units = 0;
  FqTileArgs a; bool tried = false, launched = false, self_judged = false, routed = false, direct = false, hooked = false;
};

class FqEngine {
 public:
  FqEngine(const fqg_config& cfg, FqDevice* dev);
  ~FqEngine();
  void feed_host(int file, const void* bytes, size_t n, bool last);
  void feed_device(int file, const void* dptr, size_t n, bool last);
  void finish(fqg_report* rep);
  void reset();
  void index_records(const void* host_bytes, size_t n, uint64_t* starts, size_t cap, uint64_t* n_records);
  void record_table(uint64_t want, std::vector<FqLine>* lines4, const uint8_t** data);
  void count_n(const uint8_t* data, const std::vector<FqLine>& seq_lines, std::vector<uint32_t>* out2);
  void poly_at(const uint8_t* data, const std::vector<FqLine>& seq_lines, std::vector<uint32_t>* out3);
  /* fastq_filterpair: the names of header lines of a resident chunk (device descriptors, released by the caller through device()),
   * the sniff of a file's first record, and the record this engine's index holds for each name (FQ_IDX_NONE: none) */
  FqName* header_names(const uint8_t* data, const std::vector<FqLine>& hdr_lines, int fmt, int is_pe);
  void sniff_first(const uint8_t* data, FqLine hdr1, FqLine seq, int32_t* sniff_fmt, int32_t* color);
  void lookup_names(const FqName* dev_names, const uint8_t* data, uint32_t n, std::vector<unsigned long long>* idx);
  void prescan_device(int file, const void* dptr, size_t n, bool at_eof, uint64_t* n_lines, int32_t* ends_lf, uint64_t first_ends[4]);
  void set_stream_start(int file, uint32_t skip_lines, uint64_t first_record);
  void names_count(int file, uint32_t world, uint64_t* counts, uint64_t* bytes);
  void names_pack(int file, uint32_t world, void* meta, void* blob, const uint64_t* meta_base, const uint64_t* blob_base);
  void shard_insert(const void* meta, uint64_t n, const void* blob, uint32_t n_src, const uint64_t* meta_start, const uint64_t* blob_start);
  void shard_result(uint64_t* key, uint64_t* record, char* name, uint32_t* name_len, uint64_t* collisions);
  void hist_range(int file, uint64_t lo, uint64_t hi, uint64_t* out);
  void set_file_total(int file, uint64_t total);
  uint64_t records_fed(int file) const { return f_[file].nrec; }
  void set_hash_seed(uint32_t seed) { if (f_[0].fed || f_[1].fed) throw std::runtime_error("fqg_set_hash_seed after the first feed"); seed_ = seed; }
  uint64_t collisions_walked();
  void set_sniff(int file, int fmt, int color);
  void set_line_hint(int file, uint32_t len) { if (len && !f_[file].first_seq_len) f_[file].first_seq_len = len; }
  void sniff_device(int file, const void* dptr, size_t n, uint32_t skip, int32_t* fmt, int32_t* color);
  void shard_claim(const void* meta, uint64_t n, const void* blob, uint32_t n_src, const uint64_t* meta_start, const uint64_t* blob_start, uint64_t step_base);
  void shard_claim_result(uint64_t* key, uint64_t* record, char* name, uint32_t* name_len, uint64_t* claimed, uint64_t* collisions);
  /* pipelined routing (include/fastq_gpu.h) */
  void set_chunk_hook(fqg_chunk_hook hook, void* user) { hook_ = hook; hook_user_ = user; }
  uint64_t names_new(int file);
  void names_pack_slots(int file, uint32_t world, void* const* region_ptrs, uint64_t cap, uint32_t units);
  void shard_reserve(uint64_t n_names);
  void shard_insert_slots(const void* regions, uint32_t n_src, size_t region_bytes, uint32_t nblocks, uint64_t stride, uint32_t units, bool beside, const void* flags, uint64_t expect);
  void shard_claim_slots(const void* regions, uint32_t n_src, size_t region_bytes, uint32_t nblocks, uint64_t stride, uint32_t units, bool beside, const void* flags, uint64_t expect);
  void set_route(int file, uint32_t world, void* const* region_ptrs, size_t region_bytes, uint32_t depth, uint32_t stride, uint32_t units);
  uint64_t route_chunks(int file, int* broken) const { *broken = f_[file].route_broken ? 1 : 0; return f_[file].route_chunks; }
  void shard_slots_result(uint64_t* inserted, uint64_t* equal_hashes, int32_t* overflow, uint64_t* claimed, uint64_t* unpaired);
  FqDevice* device() { return dev_; }
  std::string last_error;
  uint64_t mem_stats[4] = {0, 0, 0, 0};   /* chunk bytes held, chunk bytes released, arena bytes, records that are final */
  uint64_t path_counts[4] = {0, 0, 0, 0}; /* lanes accepted, lanes handed on, fused per-record accepted, two-pass fallbacks */

 private:
  fqg_config cfg_;
  bool reader_ = false;      /* FQG_MODE_READER: the single-file loop without validation (everything else as FQG_MODE_SINGLE) */
  FqDevice* dev_;
  FqFile f_[2];
  unsigned long long* key_ = nullptr;       /* device: global minimum event key */
  unsigned long long* counters_ = nullptr;  /* device: [0] collisions, [1] claimed, [2] table full */
  uint32_t* scratch_ = nullptr;             /* device: small result words */
  FqRecOut* recout_ = nullptr;              /* device: explain result */
  FqSlot* slots_ = nullptr; uint64_t table_cap_ = 0; uint64_t table_names_ = 0;
  uint32_t seed_ = 0;
  fqg_chunk_hook hook_ = nullptr; void* hook_user_ = nullptr;
  bool hook_fired_ = false;                 /* the chunk being fed has called the hook already */
  bool in_beside_hook_ = false;             /* the hook runs while a clean-data pass occupies the main stream */
  unsigned long long* route_cursors_ = nullptr; /* device: FQ_SHARD_MAX_SRC per-owner tuple counts of the round being packed */
  const FqPackedName* shard_meta_ = nullptr; uint64_t shard_n_ = 0; const uint8_t* shard_blob_ = nullptr;
  uint32_t shard_nsrc_ = 0; uint64_t shard_meta_start_[FQ_SHARD_MAX_SRC + 1], shard_blob_start_[FQ_SHARD_MAX_SRC];
  void scan_buffer(FqBuffer& B, bool last);
  bool finished_ = false;
  /* Streaming (single / index loops): a chunk whose records raised no event is final — its statistics are folded into the main set,
   * its names are in the arena, its bytes are released.  open_ turns false with the first chunk that cannot be settled; from there
   * on everything is kept and counted in the open set, which reprocess() can clear and recount. */
  bool streaming_ = false, open_ = false;
  bool open_dirty_ = false;                 /* a kernel has counted into the open set since the last fold */
  int add_depth_ = 0;
  uint8_t* fused_arena_ = nullptr;          /* ... and it put the names of the chunk into this block */
  bool names_cap_full_ = false;             /* size the name descriptors of a chunk by the line bound, not by the first record's lengths */
  bool fused_direct_ = false;               /* ... and counted into the main set directly */
  bool fused_lanes_ = false;                /* the fused pass that validated the chunk being added was the clean-data pass */
  void try_settle(int file);
  void release_buffer(FqBuffer& B);
  void gather_segment(int file, size_t si, uint32_t nrec);
  void set_dir(int file, size_t si);
  void fold_open();
  void clear_open();
  void fetch_name(int file, uint64_t g_local, char* dst, uint32_t* len_out);
  FqStats read_stats(int file);
  bool total0_set_ = false; uint64_t total0_ = 0; /* multi-GPU: records of file 1 over all ranks */
  uint64_t total0() const;
  const FqPackedName* claim_meta_ = nullptr; uint64_t claim_n_ = 0; const uint8_t* claim_blob_ = nullptr;
  uint64_t claim_sb_ = 0; uint32_t claim_nsrc_ = 0; uint64_t claim_meta_start_[FQ_SHARD_MAX_SRC + 1], claim_blob_start_[FQ_SHARD_MAX_SRC];
  bool fused_ok_ = true;     /* cleared for the rest of the job once a chunk needed the two-pass path */
  uint32_t* tile_out_ = nullptr;
  bool lanes_ok_ = true;     /* FQG_NO_LANES=1 (test hook) skips the clean-data pass */
  uint32_t fused_min_ = 1u << 20; /* chunks smaller than this always take the two-pass path */

  int nfiles() const { return cfg_.mode == FQG_MODE_INDEX_PAIR || cfg_.mode == FQG_MODE_SORTED_PAIR ? 2 : 1; }
  int loop_of(int file) const;
  uint64_t step_base(int file) const;
  FqRecCtx make_ctx(int file) const;
  void add_buffer(int file, uint8_t* data, uint32_t n, bool last, bool owned, bool allow_fused = true, uint32_t lead = 0);
  void realign(FqBuffer& B);
  bool try_fused_pass(int file, int b, bool last, uint32_t j0, uint64_t g0_local, FqName** names_out, uint32_t* names_cap, bool skip_lanes = false);
  void lanes_prepare(int file, uint8_t* data, uint32_t n, uint32_t lead, bool last, uint32_t j0, uint64_t g0_local, bool skip_lanes, LanesLaunch* L);
  void lanes_discard(LanesLaunch* L);
  void launch_ahead(int file, const FqBuffer& B, uint32_t j0, uint64_t g0_local);
  LanesLaunch pre_;                         /* the pass of the next chunk, launched ahead */
  struct { bool valid = false; int file = 0; uint8_t* ptr = nullptr; size_t remaining = 0; bool last = false; } next_; /* what follows the chunk being added (fqg_feed_device) */
  bool presniff(int file, const uint8_t* data, uint32_t n, uint32_t skip, bool short_only = true);
  void fused_fallback();
  void segmentize(int file, int b, uint32_t pos, uint32_t j, bool last);
  void flush_pending_as_last(int file);
  void end_file(int file, const uint8_t* dev_tail, size_t n);
  void append_pending(int file, const uint8_t* dev_src, size_t n, uint32_t lfs);
  void add_segment(int file, FqSegment s);
  void launch_segment(int file, size_t si);
  void launch_names(int file, size_t si, uint32_t nrec);
  void ensure_table(uint64_t names_total);
  void sync_dir(int file);
  void sniff_if_needed(int file, const FqSegment& s);
  uint32_t line_end_at(FqBuffer& b, uint32_t idx);
  void ensure_full_index(FqBuffer& b);
  void record_lines(int file, uint64_t g, FqLine out[4], const uint8_t** data);
  int first_byte_of_line(int file, uint64_t global_line);
  void launch_pairs();
  void reprocess();
  void fill_error(fqg_report* rep, uint64_t key, int host_code, int host_file, uint64_t host_line, uint64_t host_a);
  void fill_stats(fqg_report* rep);
  void free_file(FqFile& f);
};

#endif
