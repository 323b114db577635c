/*
 * fq_render.cpp — turns a finished report into the text and exit status the reference's fastq_info produces
 * (stdout / stderr split, message wording, blank lines: src/fastq_info.c:190-396, src/fastq.h:69-82), and the main() of
 * each reference tool on inflated streams: fastq_info (fqg_fastq_info_mem / _stream), fastq_num_reads, fastq_not_empty,
 * fastq_truncate and fastq_filter_n (fqg_reader_tool_mem), fastq_filterpair (fqg_filterpair_mem) and fastq_trim_poly_at
 * (fqg_trim_poly_at_stream).  They share one skeleton: options through the C library's getopt as the reference parses them,
 * early exits that only print, and the engines run on a device by on_device(), which turns an exception into a status.
 */
#include <getopt.h>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include "fq_engine.h"

FqDevice* fq_default_device(int ordinal); /* fq_abi.cpp (CUDA) or the test stand-in */

namespace {

struct Text {
  std::string out, err;
  int rc = 0;
  void o(const char* fmt, ...) { va_list ap; va_start(ap, fmt); vput(out, fmt, ap); va_end(ap); }
  void e(const char* fmt, ...) { va_list ap; va_start(ap, fmt); vput(err, fmt, ap); va_end(ap); }
  void error(const char* fmt, ...) { err += "\nERROR: "; va_list ap; va_start(ap, fmt); vput(err, fmt, ap); va_end(ap); err += "\n"; } /* PRINT_ERROR */
  static void vput(std::string& s, const char* fmt, va_list ap) {
    va_list ap2; va_copy(ap2, ap);
    int k = vsnprintf(nullptr, 0, fmt, ap2); va_end(ap2);
    std::vector<char> buf((size_t)k + 1);
    vsnprintf(buf.data(), buf.size(), fmt, ap);
    s.append(buf.data(), (size_t)k);
  }
};
/* PRINT_ERROR, src/fastq.h:69, around a message that is put together piece by piece */
#define ERR_BEGIN(t) (t).err += "\nERROR: "
#define ERR_END(t) (t).err += "\n"

void banner(Text& t) { t.e("fastq_utils %s\n", "0.25.3"); } /* fastq_print_version */
void mode_line(Text& t, int mode) { /* the line fastq_info prints for a mode that has one, before it reads a file */
  switch (mode) {
    case FQG_MODE_INTERLEAVED: t.e("Paired-end interleaved\n"); break;
    case FQG_MODE_SORTED_PAIR: t.e("-s option used: assuming that reads have the same ordering in both files\n"); break;
    case FQG_MODE_SINGLE: t.e("Skipping check for duplicated read names\n"); break;
    default: break;
  }
}
/* the length the caller passes for an input it could not open */
const size_t UNOPENABLE = (size_t)-1;
void unable_to_open(Text& t, const char* name) { t.error("Unable to open %s", name); } /* src/fastq.c:651-655 */
/* the records the reader loop delivered: those before a record without all four lines, else all of them */
uint64_t records_delivered(const fqg_report& r) { return r.error.code == FQG_E_TRUNC ? r.reads_before_error[0] : r.file[0].n_records; }
/* fastq_write_entry2stdout (src/fastq.c:81-86): four `%s` of the line buffers, so a line ends at its first NUL */
void write_record(std::string& out, const char* bytes, const FqLine* l) {
  for (int i = 0; i < 4; i++) out.append(bytes + l[i].off, strnlen(bytes + l[i].off, l[i].len));
}

/* The C library's getopt keeps its state in globals: one parse at a time, started over (optind = 0, the GNU way) and silent
 * (opterr = 0: the tools print their own message).  getopt permutes the words it is given, so it gets a copy of the pointers;
 * after the loop the options (and a "--") stand in front of the operands, as the reference sees them. */
std::mutex getopt_mu;
struct Getopt {
  std::lock_guard<std::mutex> lk{getopt_mu};
  std::vector<char*> argv;
  Getopt(int argc, const char** a) {
    for (int i = 0; i < argc; i++) argv.push_back(const_cast<char*>(a[i]));
    argv.push_back(nullptr);
    optind = 0; opterr = 0;
  }
};

const char* qual_range2enc(unsigned int lo, unsigned int hi) { /* fastq_qualRange2enc, src/fastq.c:274-297 */
  static const char* names[] = {"33", "64", "solexa", "33 *", "sanger"};
  int enc;
  if (lo >= 33 && lo < 59 && hi >= 90) enc = 4;
  else if (lo >= 33 && hi <= 73) enc = 0;
  else if (lo < 59) enc = 0;
  else if (lo >= 64 && hi > 74) enc = 1;
  else if (lo >= 59 && hi > 74) enc = 2;
  else enc = 3;
  if (hi > FQ_MAX_PHRED) return nullptr;
  if (enc != 4 && hi > lo + 60) return nullptr;
  return names[enc];
}

void sniff_lines(Text& t, const fqg_file_report& f) { /* src/fastq.c:459-485 */
  if (f.sniff_format == FQ_SNIFF_CASAVA) t.e("CASAVA=1.8\n");
  else if (f.sniff_format == FQ_SNIFF_INT) t.e("Read name provided as an integer\n");
  else if (f.sniff_format == FQ_SNIFF_NOSUFFIX) t.e("Read name provided with no suffix\n");
  if (f.color_space == 1) t.e("Color space\n");
}
/* PRINT_READS_PROCESSED after each of `iters` loop iterations; the counter advances by `per_iter` */
void progress(Text& t, uint64_t iters, uint64_t per_iter) {
  uint64_t every = 100000 / per_iter;
  for (uint64_t c = every; c <= iters; c += every) t.e("\b\b\b\b\b\b\b\b\b\b\b\b\b\b\b%lu", (unsigned long)(c * per_iter));
}

void error_text(Text& t, const fqg_error& e, const char* n1, const char* n2) {
  const char* F = e.msg_file == 0 ? n1 : n2;
  unsigned long L = (unsigned long)e.line;
  ERR_BEGIN(t);
  switch (e.code) {
    case FQG_E_TRUNC: t.e("Error in file %s: line %lu: file truncated", F, L); break;
    case FQG_E_TRUNC_PE: t.e("Error in file %s: line %lu: file truncated?", F, L); break;
    case FQG_E_WRONGHDR: t.e("Error in file %s: line %lu: wrong header ", F, L); t.err.append(e.hdr1, e.hdr1_len); break;
    case FQG_E_AT: t.e("Error in file %s: line %lu: sequence identifier should start with an @ - ", F, L); t.err.append(e.hdr1, e.hdr1_len); break;
    case FQG_E_IDLEN: t.e("Error in file %s: line %lu: sequence identifier should be longer than 1", F, L); break;
    case FQG_E_BADCHAR:
      t.e("Error in file %s: line %lu: invalid character '", F, L);
      t.err.push_back((char)e.chr);
      t.e("' (hex. code:'%x'), expected ACGTUacgtu0123nN.", (int)(signed char)e.chr);
      break;
    case FQG_E_UT: t.e("Error in file %s: line %lu: read contains both U and T bases", F, L); break;
    case FQG_E_SHORT: t.e("Error in file %s: line %lu: read length too small - %lu", F, L, (unsigned long)e.a); break;
    case FQG_E_PLUS: t.e("Error in file %s: line %lu:  header2 wrong. The line should contain only '+' followed by a newline or read name (header1).", F, L); break;
    case FQG_E_HDR2:
      t.e("Error in file %s: line %lu:  header2 differs from header1\nheader 1 \"", F, L);
      t.err.append(e.hdr1, e.hdr1_len); t.err += "\"\nheader 2 \""; t.err.append(e.hdr2, e.hdr2_len); t.err += "\"";
      break;
    case FQG_E_LEN: t.e("Error in file %s: line %lu: sequence and quality don't have the same length %lu!=%lu", F, L, (unsigned long)e.a, (unsigned long)e.b); break;
    case FQG_E_LEN_CS: t.e("Error in file %s: line %lu: sequence and quality length don't match %lu!=%lu", F, L, (unsigned long)e.a, (unsigned long)e.b); break;
    case FQG_E_DUP: t.e("Error in file %s: line %lu: duplicated sequence ", F, L); t.err.append(e.name, e.name_len); break;
    case FQG_E_UNPAIRED: t.e("Error in file %s: line %lu: unpaired read - ", F, L); t.err.append(e.name, e.name_len); break;
    case FQG_E_LEFTOVER: t.e("Error in file %s: found %llu unpaired reads", n1, (unsigned long long)e.a); break;
    case FQG_E_MISMATCH: t.e("Readnames do not match across files (read #%ld)", (long)e.a); break;
    case FQG_E_EOF1: t.e("Premature end of file1"); break;
    case FQG_E_EOF2: t.e("Premature end of file2"); break;
    default: t.e("internal: unknown error code %d", e.code);
  }
  ERR_END(t);
  t.rc = e.code == FQG_E_TRUNC ? 1 : 3;
}

/* Everything after the banner, for a run whose files could be opened.  Returns false when the text is complete
 * (an error was printed). */
void render_run(Text& t, const fqg_report& r, const fqg_render_opts& o, bool f2_unopenable = false) {
  const char* n1 = o.name1 ? o.name1 : "";
  const char* n2 = o.name2 ? o.name2 : "";
  const fqg_error& e = r.error;
  bool failed = e.code != FQG_OK;
  unsigned long num_reads1 = 0;
  bool mate_pass = false;
  switch (r.mode) {
    case FQG_MODE_INTERLEAVED:
      sniff_lines(t, r.file[0]);
      progress(t, r.reads_before_error[0], 2);
      if (failed) { error_text(t, e, n1, n2); return; }
      t.o("\n");
      num_reads1 = (unsigned long)r.file[0].num_rds;
      break;
    case FQG_MODE_SORTED_PAIR:
      sniff_lines(t, r.file[0]); sniff_lines(t, r.file[1]);
      progress(t, r.reads_before_error[0], 2);
      if (failed) { error_text(t, e, n1, n2); return; }
      t.o("\n");
      num_reads1 = (unsigned long)r.file[0].num_rds;
      break;
    case FQG_MODE_SINGLE:
      sniff_lines(t, r.file[0]);
      progress(t, r.reads_before_error[0], 1);
      if (failed) { error_text(t, e, n1, n2); return; }
      t.o("\n");
      num_reads1 = (unsigned long)r.file[0].num_rds;
      break;
    default: { /* index loop, then the mate loop */
      t.e("DEFAULT_HASHSIZE=%lu\n", 39000001UL);
      t.e("Scanning and indexing all reads from %s\n", n1);
      sniff_lines(t, r.file[0]);
      progress(t, r.reads_before_error[0], 1);
      bool in_index_loop = failed && e.file == 0 && e.code != FQG_E_LEFTOVER;
      if (in_index_loop) { error_text(t, e, n1, n2); return; }
      t.e("Scanning complete.\n");
      num_reads1 = (unsigned long)r.n_index_entries;
      t.e("\n");
      t.e("Reads processed: %llu\n", (unsigned long long)r.n_index_entries);
      t.e("Memory used in indexing: ~%ld MB\n", (long)(r.index_mem / 1024 / 1024));
      mate_pass = r.mode == FQG_MODE_INDEX_PAIR;
    }
  }
  if (num_reads1 == 0) { /* src/fastq_info.c:304-314 */
    if (o.empty_ok) {
      t.o("Number of reads: %lu\n", 0L);
      t.o("Quality encoding range: %lu %lu\n", 0L, 0L);
      t.o("Quality encoding: %s\n", "");
      t.o("Read length: %lu %lu %u\n", 0L, 0L, 0);
      t.rc = 0; return;
    }
    t.error("No reads found in %s.", n1);
    t.rc = 3; return;
  }
  if (mate_pass) {
    t.e("File %s processed\n", n1);
    t.e("Next file %s\n", n2);
    if (o.name2 == nullptr) { t.rc = FQG_ERR_USAGE; return; }
    if (f2_unopenable) { unable_to_open(t, n2); t.rc = 1; return; }
    sniff_lines(t, r.file[1]);
    progress(t, r.reads_before_error[1], 1);
    if (failed && e.code != FQG_E_LEFTOVER) { error_text(t, e, n1, n2); return; }
    t.o("\n");
    if (failed) { error_text(t, e, n1, n2); return; }
  }
  const fqg_file_report& f = r.file[0];
  t.e("------------------------------------\n");
  t.e("Number of reads: %lu\n", num_reads1);
  const char* enc = qual_range2enc((unsigned int)f.min_qual, (unsigned int)f.max_qual);
  if (!enc && !o.no_enc_ok) {
    if (f.max_qual > FQ_MAX_PHRED) t.error("Unable to determine quality encoding - unknown range [%lu,>%u]", (unsigned long)f.min_qual, FQ_MAX_PHRED);
    else t.error("Unable to determine quality encoding - unknown range [%lu,%lu]", (unsigned long)f.min_qual, (unsigned long)f.max_qual);
    t.rc = 3; return;
  }
  t.e("Quality encoding range: %lu %lu\n", (unsigned long)f.min_qual, (unsigned long)f.max_qual);
  if (!enc) t.e("Quality encoding: NA\n"); else t.e("Quality encoding: %s\n", enc);
  t.e("Read length: %lu %lu %u\n", (unsigned long)(f.min_rl - 1), (unsigned long)(f.max_rl - 1), (unsigned int)(r.median_rl - 1));
  t.e("OK\n");
  t.rc = 0;
}

void usage(Text& t, bool verbose) { /* src/fastq_info.c:178-188 */
  t.o("Usage: fastq_info [-r -e -s -q -h] fastq1 [fastq2 file|pe]\n");
  if (verbose) {
    t.o(" -h  : print this help message\n");
    t.o(" -s  : the reads in the two fastq files have the same ordering\n");
    t.o(" -e  : do not fail with empty files\n");
    t.o(" -q  : do not fail if quality encoding cannot be determined\n");
    t.o(" -r  : skip check for duplicated readnames\n");
  }
}

void to_transcript(const Text& t, fqg_transcript* tr) {
  tr->rc = t.rc;
  tr->out = (char*)malloc(t.out.size() + 1); memcpy(tr->out, t.out.data(), t.out.size()); tr->out[t.out.size()] = 0; tr->out_len = t.out.size();
  tr->err = (char*)malloc(t.err.size() + 1); memcpy(tr->err, t.err.data(), t.err.size()); tr->err[t.err.size()] = 0; tr->err_len = t.err.size();
}
/* the tool exits here with status rc: what it printed so far is the whole transcript */
int stop(Text& t, fqg_transcript* tr, int rc) { t.rc = rc; to_transcript(t, tr); return 0; }

/* body(device) on a device of its own, released after everything body made (its engines), also when body throws.  An exception
 * becomes the entry point's status, with its message on stderr. */
template <class Body>
int on_device(int device, Body body) {
  try {
    std::unique_ptr<FqDevice> dev(fq_default_device(device));
    body(dev.get());
  } catch (const std::bad_alloc&) { return FQG_ERR_OOM;
  } catch (const std::exception& ex) {
    fprintf(stderr, "libfastq_gpu: %s\n", ex.what());
    return strstr(ex.what(), "CUDA") ? (strstr(ex.what(), "no CUDA") ? FQG_ERR_NO_DEVICE : FQG_ERR_CUDA) : FQG_ERR_INTERNAL;
  }
  return 0;
}

void feed_all(FqEngine& eng, int file, const void* p, size_t n, size_t chunk) {
  if (chunk == 0 || n <= chunk) { eng.feed_host(file, p, n, true); return; }
  const uint8_t* b = (const uint8_t*)p;
  for (size_t off = 0; off < n; off += chunk) {
    size_t k = n - off < chunk ? n - off : chunk;
    eng.feed_host(file, b + off, k, off + k == n);
  }
}

/* where the inflated bytes of the file operands come from */
struct Source {
  virtual ~Source() {}
  virtual bool open(int file, const char* name) = 0; /* false: the reference's "Unable to open" (src/fastq.c:651-655) */
  virtual void feed(FqEngine& eng, int file) = 0;    /* everything of an opened file; the last piece is marked */
};
struct MemSource : Source {
  const void* p[2]; size_t n[2]; size_t chunk;
  bool open(int file, const char*) override { return n[file] != UNOPENABLE; }
  void feed(FqEngine& eng, int file) override { feed_all(eng, file, p[file], n[file], chunk); }
};
/* The caller's reader (zlib in the CLI) fills one pinned buffer on a helper thread while the engine takes the other: inflating,
 * the copy to the device and the kernels overlap, and the host never holds more than two pieces of the file (the reference's own
 * loop is gzbuffer + gzgets, src/fastq.c:631-661: it holds one line). */
struct StreamSource : Source {
  const fqg_stream_io* io; void* h[2] = {nullptr, nullptr}; size_t piece;
  bool open(int file, const char* name) override { h[file] = io->open ? io->open(io->user, name) : nullptr; return h[file] != nullptr; }
  ~StreamSource() override { for (int f = 0; f < 2; f++) if (h[f] && io->close) io->close(io->user, h[f]); }
  void feed(FqEngine& eng, int file) override {
    FqDevice* dev = eng.device();
    uint8_t* buf[2] = {(uint8_t*)dev->host_alloc(piece), (uint8_t*)dev->host_alloc(piece)};
    struct Slot { long n = 0; bool full = false; } slot[2];
    std::mutex mu; std::condition_variable cv; bool failed = false, quit = false;
    std::thread reader([&] {
      for (int k = 0;; k ^= 1) {
        { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return !slot[k].full || quit; }); if (quit) return; }
        size_t got = 0; long r = 1;
        while (got < piece && (r = io->read(io->user, h[file], buf[k] + got, piece - got)) > 0) got += (size_t)r; /* whole pieces: fewer, larger chunks */
        { std::lock_guard<std::mutex> lk(mu); slot[k].n = r < 0 ? -1 : (long)got; slot[k].full = true; }
        cv.notify_all();
        if (r <= 0) return; /* the end of the stream (or an error): this piece is the last one */
      }
    });
    try {
      for (int k = 0;; k ^= 1) {
        long n;
        { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return slot[k].full; }); n = slot[k].n; }
        if (n < 0) { failed = true; break; }
        const bool last = (size_t)n < piece;
        eng.feed_host(file, buf[k], (size_t)n, last);
        { std::lock_guard<std::mutex> lk(mu); slot[k].full = false; }
        cv.notify_all();
        if (last) break;
      }
    } catch (...) {
      { std::lock_guard<std::mutex> lk(mu); quit = true; slot[0].full = slot[1].full = false; }
      cv.notify_all(); reader.join(); dev->host_release(buf[0]); dev->host_release(buf[1]);
      throw;
    }
    { std::lock_guard<std::mutex> lk(mu); quit = true; }
    cv.notify_all(); reader.join();
    dev->host_release(buf[0]); dev->host_release(buf[1]);
    if (failed) throw std::runtime_error("fqg_fastq_info_stream: the read callback reported an error");
  }
};

int fastq_info_run(int argc, const char** argv_in, Source& src, int device, fqg_transcript* tr) {
  Text t;
  bool is_paired = false, is_interleaved = false, is_sorted = false, empty_ok = false, no_enc_ok = false, skip_names = false;
  int nopt = 0; /* option characters, not words: "-rs" counts 2 */
  const char *a1, *a2 = nullptr;
  banner(t);
  {
    Getopt g(argc, argv_in);
    for (int c; (c = getopt(argc, g.argv.data(), "esfrhq")) != -1; ++nopt) {
      switch (c) {
        case 'q': no_enc_ok = true; break;
        case 'e': empty_ok = true; break;
        case 's': is_sorted = true; break;
        case 'r': skip_names = true; break;
        case 'h': usage(t, true); return stop(t, tr, 0);
        case 'f':
          t.e("Fixing (-f) enabled: Replacing . by N (creating .fix.gz files)\n");
          t.error("-f option is no longer valid.");
          return stop(t, tr, 1);
        default: t.error("Option -%c invalid", optopt); return stop(t, tr, 1); /* "--help" is the unknown option '-' */
      }
    }
    if (argc - nopt < 2 || argc - nopt > 3) {
      t.error("Invalid number of arguments");
      usage(t, false);
      return stop(t, tr, 1);
    }
    a1 = g.argv[1 + nopt];
    if (argc - nopt == 3) a2 = g.argv[2 + nopt];
  }
  if (a2) { is_paired = true; is_interleaved = strncmp(a2, "pe", 2) == 0; }

  fqg_config cfg; memset(&cfg, 0, sizeof cfg); cfg.device = device;
  if (is_interleaved) cfg.mode = FQG_MODE_INTERLEAVED;
  else if (is_paired && is_sorted && skip_names) cfg.mode = FQG_MODE_SORTED_PAIR;
  else if (!is_paired && skip_names) cfg.mode = FQG_MODE_SINGLE;
  else {
    cfg.mode = is_paired && !is_sorted ? FQG_MODE_INDEX_PAIR : FQG_MODE_INDEX;
    if (is_paired) cfg.flags |= FQG_FLAG_PAIRED_NAMES;
  }
  mode_line(t, cfg.mode);
  if (!src.open(0, a1)) { unable_to_open(t, a1); return stop(t, tr, 1); }
  if (cfg.mode == FQG_MODE_SORTED_PAIR && !src.open(1, a2)) { unable_to_open(t, a2); return stop(t, tr, 1); }
  fqg_report rep;
  bool f2_unopenable = false;
  const int st = on_device(device, [&](FqDevice* dev) {
      FqEngine eng(cfg, dev);
      src.feed(eng, 0);
      if (cfg.mode == FQG_MODE_INDEX_PAIR) {
        /* the reference opens file 2 only after file 1 was indexed without error and holds reads */
        fqg_report r1; eng.finish(&r1);
        bool stop_after_1 = (r1.error.code != FQG_OK && r1.error.file == 0) || r1.n_index_entries == 0;
        if (!stop_after_1) { if (src.open(1, a2)) src.feed(eng, 1); else f2_unopenable = true; }
      } else if (cfg.mode == FQG_MODE_SORTED_PAIR) src.feed(eng, 1);
      eng.finish(&rep);
  });
  if (st) return st;
  fqg_render_opts o; o.empty_ok = empty_ok; o.no_enc_ok = no_enc_ok; o.name1 = a1; o.name2 = a2;
  render_run(t, rep, o, f2_unopenable);
  if (t.rc < 0) return t.rc;
  to_transcript(t, tr);
  return 0;
}

}  // namespace

extern "C" int fqg_render(const fqg_report* rep, const fqg_render_opts* opts, fqg_transcript* tr) {
  if (!rep || !opts || !tr) return FQG_ERR_USAGE;
  Text t;
  banner(t);
  mode_line(t, rep->mode);
  render_run(t, *rep, *opts);
  if (t.rc < 0) return t.rc;
  to_transcript(t, tr);
  return 0;
}

extern "C" void fqg_transcript_free(fqg_transcript* t) {
  if (!t) return;
  free(t->out); free(t->err); t->out = t->err = nullptr;
}

extern "C" int fqg_fastq_info_mem(int argc, const char** argv_in, const void* f1, size_t n1, const void* f2, size_t n2,
                                  int device, size_t chunk_bytes, fqg_transcript* tr) {
  if (!tr || argc < 1 || !argv_in) return FQG_ERR_USAGE;
  MemSource src; src.p[0] = f1; src.n[0] = n1; src.p[1] = f2; src.n[1] = n2; src.chunk = chunk_bytes;
  return fastq_info_run(argc, argv_in, src, device, tr);
}
extern "C" int fqg_fastq_info_stream(int argc, const char** argv_in, const fqg_stream_io* io, int device, size_t piece_bytes, fqg_transcript* tr) {
  if (!tr || argc < 1 || !argv_in || !io || !io->read) return FQG_ERR_USAGE;
  StreamSource src; src.io = io; src.piece = piece_bytes ? piece_bytes : ((size_t)64 << 20);
  return fastq_info_run(argc, argv_in, src, device, tr);
}

namespace {
/* main() of the reader tools that WRITE records: src/fastq_truncate.c:32-57 (the first num_reads entries) and src/fastq_filter_n.c:33-93
 * (entries whose share of N bases is within -n percent).  Both are the fastq_read_entry loop (src/fastq.c:245-261) followed by
 * fastq_write_entry2stdout (:81-86: four `%s` of the line buffers, so a line ends at its first NUL).  The records are delimited on the
 * device (FQG_MODE_READER, the stream in windows of one chunk each: reader_windows), fastq_filter_n's predicate is evaluated there (count_n); the host writes the
 * chosen byte ranges of the stream it was given. */
/* The reader loop (FQG_MODE_READER) over a stream of any size, for the tools that write records.  The stream is taken in windows, each
 * one chunk of its own that starts at a record start; a window that is not the last one ends where the data was cut, so its last record
 * is trusted only when the engine saw all four of its lines AND the window ends behind a line feed — otherwise the next window starts at
 * that record.  A window that does not even hold its first record grows (a record is at most two lines of 2 499 999 bytes and two of
 * 999: a window of 6 MiB that still shows a broken first record shows a broken FILE).  visit(engine, lines of the window's records,
 * device bytes, host bytes, number of the first record) → false: the tool has what it wants. */
struct WindowsResult { bool truncated = false; fqg_error error; uint64_t records = 0; };
template <class Visit>
WindowsResult reader_windows(FqDevice* dev, int device, const char* p, size_t n, uint64_t want, Visit visit) {
  WindowsResult R; memset(&R.error, 0, sizeof R.error);
  if (want == 0) return R;
  const size_t CAP = ((size_t)1 << 31) - 64, MAXREC = 6u << 20;
  size_t window = (size_t)1 << 30;
  if (const char* e = getenv("FQG_TOOL_WINDOW_BYTES")) { const unsigned long long v = strtoull(e, nullptr, 10); if (v >= 64) window = (size_t)std::min<unsigned long long>(v, CAP); } /* tests */
  fqg_config cfg; memset(&cfg, 0, sizeof cfg); cfg.device = device; cfg.mode = FQG_MODE_READER; cfg.flags = FQG_FLAG_KEEP_CHUNKS;
  size_t pos = 0;
  for (;;) {
    const size_t len = std::min(window, n - pos);
    const bool final = pos + len == n;
    FqEngine eng(cfg, dev);
    eng.feed_host(0, p + pos, len, true);
    fqg_report rep; eng.finish(&rep);
    const bool trunc = rep.error.code == FQG_E_TRUNC; /* the loop met a record without all four lines */
    uint64_t nrec = records_delivered(rep);
    const bool cut_line = !final && len > 0 && p[pos + len - 1] != '\n';
    if (!final && !trunc && cut_line && nrec > 0) nrec--; /* its fourth line is where the window was cut */
    if (!final && nrec == 0 && (trunc || cut_line)) {
      if (len < MAXREC && window < CAP) { window = std::min(CAP, window * 2); continue; } /* the first record does not fit: a larger window */
      R.truncated = true; R.error = rep.error; R.error.line = 4 * R.records; /* (a broken record in the middle of the file) */
      return R;
    }
    const uint64_t take = std::min<uint64_t>(nrec, want - R.records);
    std::vector<FqLine> L; const uint8_t* ddata = nullptr;
    eng.record_table(take, &L, &ddata);
    const bool more = visit(eng, L, ddata, p + pos, R.records);
    R.records += take;
    if (!more || R.records >= want) return R; /* (the broken record, if there is one, was not reached) */
    if (final) {
      if (trunc) { R.truncated = true; R.error = rep.error; R.error.line = 4 * R.records; } /* fd->cline before the increment, src/fastq.c:254 */
      return R;
    }
    const size_t consumed = nrec ? (size_t)L[4 * nrec - 1].off + L[4 * nrec - 1].len : 0; /* (take == nrec here) */
    if (!trunc && !cut_line) {
      if (consumed < len) return R; /* a NUL-led header line ended the file quietly (src/fastq.c:248) */
      pos += len;
    } else pos += consumed;
  }
}

int writer_tool(bool filter_n, int argc, const char** argv_in, const void* f1, size_t n1, int device, fqg_transcript* tr) {
  Text t;
  banner(t);
  const char* fname = nullptr; long num_reads = 0; unsigned max_n = 0;
  if (!filter_n) {
    if (argc != 3) { t.e("Usage: fastq_truncate fastq1 num_reads\n"); return stop(t, tr, 1); }
    fname = argv_in[1]; num_reads = atol(argv_in[2]);
  } else {
    Getopt g(argc, argv_in);
    int nopt = 0;
    for (int c; (c = getopt(argc, g.argv.data(), "n:")) != -1;) {
      if (c != 'n') { t.error("Option -%c invalid", optopt); return stop(t, tr, 1); } /* "-n" without its argument too */
      max_n = (unsigned)atoi(optarg); if (max_n > 100) max_n = 100;
      nopt += 2; /* also for "-n10" */
    }
    if (argc - nopt < 2 || argc - nopt > 3) { t.error("Usage: fastq_filter_n [ -n 0 ] fastq1"); return stop(t, tr, 1); }
    if (max_n > 0) t.e("Discard reads with more than %d%% of Ns\n", (int)max_n); else t.e("Discard reads with at least one N\n");
    fname = g.argv[nopt + 1];
  }
  if (n1 == UNOPENABLE) { unable_to_open(t, fname); return stop(t, tr, 1); }
  if (!f1 && n1) return FQG_ERR_USAGE;
  const int st = on_device(device, [&](FqDevice* dev) {
      const uint64_t want = (filter_n || num_reads < 0) ? ~0ull : (uint64_t)num_reads;
      WindowsResult W = reader_windows(dev, device, (const char*)f1, n1, want, [&](FqEngine& eng, const std::vector<FqLine>& L, const uint8_t* ddata, const char* bytes, uint64_t g0) {
        std::vector<uint32_t> nn;
        if (filter_n && !L.empty()) {
          std::vector<FqLine> seq(L.size() / 4);
          for (size_t r = 0; r < seq.size(); r++) seq[r] = L[4 * r + 1];
          eng.count_n(ddata, seq, &nn);
        }
        for (size_t r = 0; r < L.size() / 4; r++) {
          if (filter_n) {
            const unsigned long read_len = nn[2 * r + 1];
            const unsigned max_num_n = (unsigned)(read_len * max_n / 100);
            const bool keep = nn[2 * r] <= max_num_n;
            if (keep) write_record(t.out, bytes, &L[4 * r]);
            const unsigned long cline = 4ul * (unsigned long)(g0 + r + 1);
            if (cline % 100000 == 0) t.e("\b\b\b\b\b\b\b\b\b\b\b\b\b\b\b%lu", cline);
          } else write_record(t.out, bytes, &L[4 * r]);
        }
        return true;
      });
      /* the loop met the broken record only if it went on reading that far (src/fastq_truncate.c:47-49) */
      if (W.truncated) { error_text(t, W.error, fname, fname); t.rc = 1; }
      else t.rc = 0;
  });
  if (st) return st;
  to_transcript(t, tr);
  return 0;
}
}  // namespace

/* main() of fastq_filterpair (src/fastq_filterpair.c:38-240) on two inflated streams.  File 1 goes through the index loop
 * (fastq_index_readnames, src/fastq.c:396-439: validation, duplicate check — FQG_MODE_INDEX with paired names); the records of both files
 * are delimited by the reader loop (FQG_MODE_READER), their names hashed on the device (fq_header_name) and looked up in the index there
 * (names_lookup: exact byte compare behind an equal hash).  What is left for the host is what the reference does one record at a time:
 * lookup-then-delete decides that the FIRST record of file 2 with a name gets the mate; the copies out of file 1 count seeks against the
 * reader's position; the last loop over file 1 starts where the last copy left the reader, not at the start of the file.  The three
 * gzip files the reference writes come back inflated. */
namespace {
struct PairFile { /* one input: its records (reader loop) on the device and on the host */
  FqEngine* rd = nullptr; std::vector<FqLine> L; const uint8_t* ddata = nullptr; const char* bytes = nullptr; uint64_t nrec = 0; fqg_report rep;
  void load(const fqg_config& base, FqDevice* dev, const void* p, size_t n) {
    fqg_config cfg = base; cfg.mode = FQG_MODE_READER; cfg.flags = FQG_FLAG_KEEP_CHUNKS;
    rd = new FqEngine(cfg, dev);
    rd->feed_host(0, p, n, true);
    rd->finish(&rep);
    nrec = records_delivered(rep);
    rd->record_table(nrec, &L, &ddata);
    bytes = (const char*)p;
  }
  ~PairFile() { delete rd; }
  std::vector<FqLine> headers() const { std::vector<FqLine> h(L.size() / 4); for (size_t r = 0; r < h.size(); r++) h[r] = L[4 * r]; return h; }
  void write(std::string& out, size_t r) const { write_record(out, bytes, &L[4 * r]); }
  uint32_t raw_len(size_t r) const { return L[4 * r].len + L[4 * r + 1].len + L[4 * r + 2].len + L[4 * r + 3].len; }
};
/* the index loop over one file (fastq_index_readnames and the lines fastq_filterpair prints around it); false: it ended the run */
bool index_file(Text& t, FqEngine& ix, const void* p, size_t n, const char* name, unsigned long* index_mem, fqg_report* rep) {
  t.e("Scanning and indexing all reads from %s\n", name);
  ix.feed_host(0, p, n, true);
  ix.finish(rep);
  sniff_lines(t, rep->file[0]);
  progress(t, rep->reads_before_error[0], 1);
  if (rep->error.code != FQG_OK) { error_text(t, rep->error, name, name); return false; }
  t.e("Scanning complete.\n");
  *index_mem += (unsigned long)rep->index_mem; /* (sizeof(hashtable) and the entries, src/fastq_filterpair.c:70, src/fastq.c:609) */
  t.e("Reads indexed: %llu\n", (unsigned long long)rep->n_index_entries);
  t.e("Memory used in indexing: %ld MB\n", (long)(*index_mem / 1024 / 1024));
  return true;
}
}  // namespace
extern "C" int fqg_filterpair_mem(int argc, const char** argv, const void* f1, size_t n1, const void* f2, size_t n2, int device,
                                  fqg_transcript* tr, char* outs[3], size_t lens[3], int32_t* created) {
  if (argc < 1 || !argv || !tr || !outs || !lens || !created) return FQG_ERR_USAGE;
  for (int i = 0; i < 3; i++) { outs[i] = nullptr; lens[i] = 0; }
  *created = 0;
  Text t;
  banner(t);
  if (argc != 6 && argc != 7) { t.e("Usage: filterpair fastq1 fastq2 paired1 paired2 unpaired [sorted]\n"); return stop(t, tr, 1); }
  t.e("%d", argc);
  if (n1 == UNOPENABLE) { unable_to_open(t, argv[1]); return stop(t, tr, 1); }
  if (n2 == UNOPENABLE) { unable_to_open(t, argv[2]); return stop(t, tr, 1); }
  if ((!f1 && n1) || (!f2 && n2)) return FQG_ERR_USAGE;
  const size_t LIMIT = ((size_t)1 << 31) - 64; /* one chunk per file: the record-writing tools take streams below 2 GiB */
  if (n1 > LIMIT || n2 > LIMIT) return FQG_ERR_USAGE;
  const bool sorted = argc == 7 && !strcmp(argv[6], "sorted");
  t.e("HASHSIZE=%u\n", 100000001u);
  if (sorted) t.e("Assuming sorted fastq files\n");
  std::string out[3]; /* paired1, paired2, unpaired */
  fqg_config cfg; memset(&cfg, 0, sizeof cfg); cfg.device = device; cfg.mode = FQG_MODE_INDEX; cfg.flags = FQG_FLAG_PAIRED_NAMES;
  const int st = on_device(device, [&](FqDevice* dev) {
      unsigned long index_mem = 0;
      fqg_report rep1, rep2;
      FqEngine ix1(cfg, dev);
      bool go = index_file(t, ix1, f1, n1, argv[1], &index_mem, &rep1);
      if (go) {
        *created = 1; /* the three output files exist from here on (src/fastq_filterpair.c:83-92) */
        PairFile A, B;
        A.load(cfg, dev, f1, n1);
        const int fmt1 = fq_fmt_of_sniff(rep1.file[0].sniff_format);
        unsigned long paired = 0, up2 = 0;
        if (sorted) {
          FqEngine ix2(cfg, dev);
          go = index_file(t, ix2, f2, n2, argv[2], &index_mem, &rep2);
          if (go) {
            B.load(cfg, dev, f2, n2);
            const int fmt2 = fq_fmt_of_sniff(rep2.file[0].sniff_format);
            /* both files hold every name once (the index loop saw to that): a record has its mate iff the other index holds its name */
            std::vector<unsigned long long> in2, in1;
            FqName* na = ix2.header_names(A.ddata, A.headers(), fmt1, 1);
            ix2.lookup_names(na, A.ddata, (uint32_t)A.nrec, &in2);
            if (na) dev->release(na);
            FqName* nb = ix1.header_names(B.ddata, B.headers(), fmt2, 1);
            ix1.lookup_names(nb, B.ddata, (uint32_t)B.nrec, &in1);
            if (nb) dev->release(nb);
            t.e("Filtering %s...\n", argv[1]);
            for (size_t r = 0; r < A.nrec; r++) {
              if (in2[r] == FQ_IDX_NONE) { ++up2; A.write(out[2], r); } else { ++paired; A.write(out[0], r); }
              if ((r + 1) % 10000 == 0) t.e("\b\b\b\b\b\b\b\b\b\b\b\b\b\b\b%lu", (unsigned long)(r + 1)); /* cline = 1 + 4(r+1) after the rewind */
            }
            t.e("Filtering %s...\n", argv[2]);
            for (size_t r = 0; r < B.nrec; r++) {
              if (in1[r] == FQ_IDX_NONE) { ++up2; B.write(out[2], r); } else B.write(out[1], r);
              if ((r + 1) % 10000 == 0) t.e("\b\b\b\b\b\b\b\b\b\b\b\b\b\b\b%lu", (unsigned long)(r + 1));
            }
          }
        } else {
          t.e("Processing %s\n", argv[2]);
          B.load(cfg, dev, f2, n2);
          int32_t sf2 = FQ_SNIFF_DEFAULT, col2 = 0;
          std::vector<unsigned long long> hit; std::vector<FqName> names2;
          if (B.nrec) {
            B.rd->sniff_first(B.ddata, B.L[0], B.L[1], &sf2, &col2);
            const int fmt2 = fq_fmt_of_sniff(sf2);
            FqName* nb = ix1.header_names(B.ddata, B.headers(), fmt2, 1);
            ix1.lookup_names(nb, B.ddata, (uint32_t)B.nrec, &hit);
            names2.resize(B.nrec);
            dev->download(names2.data(), nb, B.nrec * sizeof(FqName));
            dev->release(nb);
          }
          std::vector<uint8_t> gone(A.nrec, 0); /* fastq_index_delete: a name is found once */
          unsigned long ctr_seek = 0, ctr_noseek = 0;
          uint64_t pos1 = 0; /* where the reader of file 1 stands (inflated offset; 0 after the rewind) */
          for (size_t r = 0; r < B.nrec && go; r++) {
            if (names2[r].len == 0xFFFFFFFFu) { /* fastq_get_readname: src/fastq.c:448 */
              const FqLine& l = B.L[4 * r];
              ERR_BEGIN(t); t.e("Error in file %s: line %lu: wrong header ", argv[2], 4ul * (unsigned long)(r + 1)); t.err.append(B.bytes + l.off, strnlen(B.bytes + l.off, l.len)); ERR_END(t);
              t.rc = 3; go = false; break;
            }
            if (r == 0) { fqg_file_report fr; memset(&fr, 0, sizeof fr); fr.sniff_format = sf2; fr.color_space = col2; sniff_lines(t, fr); }
            const unsigned long long a = hit[r];
            if (a == FQ_IDX_NONE || a >= A.nrec || gone[a]) { ++up2; B.write(out[2], r); }
            else {
              ++paired;
              B.write(out[1], r);
              const uint64_t offset = A.L[4 * a].off; /* fastq_quick_copy_entry, src/fastq.c:122-159 */
              if (pos1 != offset) ++ctr_seek; else ++ctr_noseek;
              t.e("%lu / %lu\n", ctr_seek, ctr_noseek);
              A.write(out[0], (size_t)a);
              pos1 = offset + A.raw_len((size_t)a);
              gone[a] = 1;
            }
            if ((r + 1) % 10000 == 0) t.e("\b\b\b\b\b\b\b\b\b\b\b\b\b\b\b%lu", (unsigned long)(r + 1));
          }
          if (go && B.rep.error.code == FQG_E_TRUNC) { error_text(t, B.rep.error, argv[2], argv[2]); go = false; } /* the reader met the broken record after those */
          if (go) {
            t.e("\n");
            const unsigned long long left = rep1.n_index_entries - paired;
            t.e("Recording %llu unpaired reads from %s\n", left, argv[1]);
            unsigned long long remaining = left;
            size_t j = 0;
            while (j < A.nrec && A.L[4 * j].off < pos1) j++; /* the reader stands behind the last record it copied */
            for (unsigned long m = 1; j < A.nrec && remaining; j++, m++) {
              if (!gone[j]) { A.write(out[2], j); remaining--; }
              if (m % 100000 == 0) t.e("\b\b\b\b\b\b\b\b\b\b\b\b\b\b\b%lu", m); /* cline = 1 + 4m */
            }
            t.e("Unpaired from %s: %llu\n", argv[1], left);
            t.e("Unpaired from %s: %ld\n", argv[2], (long)up2);
          }
        }
        if (go) {
          t.e("\n");
          t.e("Paired: %ld\n", (long)paired);
          if (paired == 0) { t.e("!!!WARNING!!! 0 paired reads! are the headers ok?\n"); t.rc = 3; } else t.rc = 0;
        }
      }
  });
  if (st) return st;
  for (int i = 0; i < 3; i++) {
    outs[i] = (char*)malloc(out[i].size() + 1);
    if (!outs[i]) return FQG_ERR_OOM;
    memcpy(outs[i], out[i].data(), out[i].size()); outs[i][out[i].size()] = 0; lens[i] = out[i].size();
  }
  to_transcript(t, tr);
  return 0;
}

/* main() of fastq_trim_poly_at (src/fastq_trim_poly_at.c:121-233).  The options go through the C library's getopt_long, as the reference
 * calls it (long options and their unambiguous prefixes, `--opt=value`, the short forms a: b: c: d:, unknown words ignored); the input
 * is read through the caller's callbacks into one chunk, the records are delimited on the device (the bare fastq_read_next_entry loop,
 * FQG_MODE_READER) and the two scans of trim_poly_at run there too (fq_poly_at, one result triple per record).  The host then does what
 * the reference does to its line buffers: the buffers of a FASTQ_ENTRY live across records, and the trimming writes and reads at indices
 * taken from the SEQUENCE line into the QUALITY buffer too (:92-95, :108-111) — with a quality line shorter than its sequence line what
 * is printed depends on what an earlier record left there, so the two buffers are kept exactly as the reference keeps them.  What the
 * reference gzips into --outfile comes back inflated. */
extern "C" int fqg_trim_poly_at_stream(int argc, const char** argv_in, const fqg_stream_io* io, int device, fqg_transcript* tr,
                                       char** outfile, size_t* outfile_len, const char** outfile_name) {
  if (argc < 1 || !argv_in || !io || !tr || !outfile || !outfile_len || !outfile_name) return FQG_ERR_USAGE;
  *outfile = nullptr; *outfile_len = 0; *outfile_name = nullptr;
  Text t;
  const char* file = nullptr; const char* ofile = nullptr; int min_poly = 10; long min_len = 10;
  int help = 0;
  {
    const struct option long_options[] = {{"help", no_argument, &help, 1}, {"min_poly_at_len", required_argument, 0, 'a'}, {"file", required_argument, 0, 'b'},
                                          {"outfile", required_argument, 0, 'c'}, {"min_len", required_argument, 0, 'd'}, {0, 0, 0, 0}};
    Getopt g(argc, argv_in);
    for (int c; (c = getopt_long(argc, g.argv.data(), "a:b:c:d:", long_options, nullptr)) != -1;) {
      switch (c) {
        case 'a': min_poly = (int)atol(optarg); break;
        case 'b': file = optarg; break;
        case 'c': ofile = optarg; break;
        case 'd': min_len = atol(optarg); break;
        default: break;
      }
    }
  }
  banner(t);
  if (help) {
    t.o("usage: fastq_trim_poly_at --file fastq_file --outfile out_file [optional parameters]");
    t.o("%s", "\n  --help       :print the usage\n  --file <filename> :fastq (optional gzipped) file name \n  --ofile <filename> : fastq file name where the processed reads will be written \n"
              "  --min_poly_at_len integer     : minimum length of poly-A|T sequence to remove.\n  --min_len integer     : minimum read length.\n");
    return stop(t, tr, 0);
  }
  t.e("INFO:Validating options...\n");
  if (!file) { t.error("missing input file (--file)"); return stop(t, tr, 1); }
  if (!ofile) { t.error("missing output file name (--outfile)"); return stop(t, tr, 1); }
  t.e("INFO:Options OK.\n");
  void* h = io->open ? io->open(io->user, file) : nullptr;
  if (!h) { unable_to_open(t, file); return stop(t, tr, 1); }
  std::vector<char> in;
  {
    std::vector<char> piece(8u << 20);
    long r;
    while ((r = io->read(io->user, h, piece.data(), piece.size())) > 0) in.insert(in.end(), piece.data(), piece.data() + r);
    if (io->close) io->close(io->user, h);
    if (r < 0) return FQG_ERR_USAGE;
  }
  *outfile_name = ofile; /* from here on the reference has created the file */
  std::string out;
  const int st = on_device(device, [&](FqDevice* dev) {
      std::vector<char> sbuf(4, 0), qbuf(4, 0); /* the entry's seq and qual buffers: they outlive a record (and a window) */
      unsigned long trimmed = 0, discarded = 0, processed = 0;
      WindowsResult W = reader_windows(dev, device, in.data(), in.size(), ~0ull, [&](FqEngine& eng, const std::vector<FqLine>& L, const uint8_t* ddata, const char* bytes, uint64_t g0) {
        std::vector<FqLine> seq(L.size() / 4);
        uint32_t longest = 0;
        for (size_t r = 0; r < seq.size(); r++) { seq[r] = L[4 * r + 1]; longest = std::max(longest, std::max(L[4 * r + 1].len, L[4 * r + 3].len)); }
        std::vector<uint32_t> pa;
        eng.poly_at(ddata, seq, &pa);
        if (sbuf.size() < (size_t)longest + 4) { sbuf.resize((size_t)longest + 4, 0); qbuf.resize((size_t)longest + 4, 0); }
        for (size_t r = 0; r < seq.size(); r++) {
          const FqLine &lh = L[4 * r], &ls = L[4 * r + 1], &lp = L[4 * r + 2], &lq = L[4 * r + 3];
          memcpy(sbuf.data(), bytes + ls.off, ls.len); sbuf[ls.len] = 0; /* gzgets: the line's bytes and a NUL behind them */
          memcpy(qbuf.data(), bytes + lq.off, lq.len); qbuf[lq.len] = 0;
          ++processed;
          unsigned long read_len = pa[3 * r];
          const long tail = pa[3 * r + 1], head = pa[3 * r + 2];
          if (min_poly > 0) {
            if (tail >= min_poly) { /* the 3' end (:79-96) */
              const long x = (long)read_len - 2 - tail;
              read_len -= (unsigned long)tail;
              sbuf[x + 1] = '\n'; sbuf[x + 2] = 0; qbuf[x + 1] = '\n'; qbuf[x + 2] = 0;
              ++trimmed;
            } else if (head >= min_poly) { /* the 5' end (:99-113) */
              for (long x = 0; x <= (long)read_len - head; ++x) { sbuf[x] = sbuf[x + head]; qbuf[x] = qbuf[x + head]; }
              read_len -= (unsigned long)head;
              ++trimmed;
            }
          }
          if (read_len >= (unsigned long)min_len) {
            out.append(bytes + lh.off, strnlen(bytes + lh.off, lh.len));
            out.append(sbuf.data(), strlen(sbuf.data()));
            out.append(bytes + lp.off, strnlen(bytes + lp.off, lp.len));
            out.append(qbuf.data(), strlen(qbuf.data()));
          } else ++discarded;
          const unsigned long c = (unsigned long)(g0 + r + 1);
          if (c % 100000 == 0) t.e("\b\b\b\b\b\b\b\b\b\b\b\b\b\b\b%lu", c);
        }
        return true;
      });
      if (W.truncated) { error_text(t, W.error, file, file); t.rc = 1; }
      else {
        t.e("INFO:Reads processed: %ld\n", (long)processed); t.e("INFO:Reads trimmed: %ld\n", (long)trimmed); t.e("INFO:Reads discarded: %ld\n", (long)discarded);
        t.rc = 0;
      }
  });
  if (st) return st;
  *outfile = (char*)malloc(out.size() + 1);
  if (!*outfile) return FQG_ERR_OOM;
  memcpy(*outfile, out.data(), out.size()); (*outfile)[out.size()] = 0; *outfile_len = out.size();
  to_transcript(t, tr);
  return 0;
}
extern "C" void fqg_buffer_free(void* p) { free(p); }

/* main() of the reader-style tools on an inflated stream: src/fastq_num_reads.c:32-50, src/fastq_not_empty.c:32-47.  Both are
 * the bare fastq_read_next_entry loop (src/fastq.c:237-261): records are delimited, a NUL-led header line ends the file quietly,
 * a record with fewer than four lines is "file truncated" (exit 1); nothing is validated. */
extern "C" int fqg_reader_tool_mem(int argc, const char** argv, const void* f1, size_t n1, int device, size_t chunk_bytes, fqg_transcript* tr) {
  if (argc < 1 || !argv || !argv[0] || !tr) return FQG_ERR_USAGE;
  Text t;
  const char* tool = strrchr(argv[0], '/'); tool = tool ? tool + 1 : argv[0];
  const bool num_reads = !strcmp(tool, "fastq_num_reads"), not_empty = !strcmp(tool, "fastq_not_empty");
  if (!strcmp(tool, "fastq_truncate") || !strcmp(tool, "fastq_filter_n")) return writer_tool(!strcmp(tool, "fastq_filter_n"), argc, argv, f1, n1, device, tr);
  if (!num_reads && !not_empty) return FQG_ERR_USAGE;
  if (num_reads) banner(t); /* src/fastq_num_reads.c:34; fastq_not_empty prints none */
  if (argc != 2) {
    if (num_reads) t.e("Usage: fastq_num_reads fastq_file\n");
    else t.e("Usage: fastq_not_empty fastq_file\nExit status of 0 if it is not empty, 0 otherwise. The fastq file may be compressed with gzip.");
    return stop(t, tr, 1);
  }
  if (n1 == UNOPENABLE) { unable_to_open(t, argv[1]); return stop(t, tr, 1); }
  if (!f1 && n1) return FQG_ERR_USAGE;
  fqg_config cfg; memset(&cfg, 0, sizeof cfg); cfg.device = device; cfg.mode = FQG_MODE_READER;
  fqg_report rep;
  const int st = on_device(device, [&](FqDevice* dev) {
      FqEngine eng(cfg, dev);
      feed_all(eng, 0, f1, n1, chunk_bytes);
      eng.finish(&rep);
  });
  if (st) return st;
  const uint64_t n = rep.file[0].n_records;
  if (not_empty) { /* only the first entry is ever read: an error further down does not exist for this tool */
    if (rep.reads_before_error[0] >= 1) t.rc = 0;
    else if (rep.error.code == FQG_E_TRUNC) { error_text(t, rep.error, argv[1], argv[1]); t.rc = 1; }
    else t.rc = 1;
  } else if (rep.error.code == FQG_E_TRUNC) { error_text(t, rep.error, argv[1], argv[1]); t.rc = 1; }
  else { t.o("%lu\n", (unsigned long)n); t.rc = 0; }
  to_transcript(t, tr);
  return 0;
}
