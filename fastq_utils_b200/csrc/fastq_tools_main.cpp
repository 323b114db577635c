/*
 * fastq_tools_gpu — the reference's command lines on top of libfastq_gpu: fastq_info (src/fastq_info.c:190-396), fastq_num_reads,
 * fastq_not_empty, fastq_truncate, fastq_filter_n (src/fastq_num_reads.c, src/fastq_not_empty.c, src/fastq_truncate.c,
 * src/fastq_filter_n.c), fastq_trim_poly_at (src/fastq_trim_poly_at.c) and fastq_filterpair (src/fastq_filterpair.c).  One binary: the
 * tool is the name it is called by (symbolic links <tool>_gpu next to it) or, called as fastq_tools_gpu, its first argument.  Same
 * arguments, same stdout / stderr text, same exit status, same output files.  The host inflates the inputs (zlib, like the reference's
 * gzopen / gzgets: gzip members are concatenated, plain text passes through, `-` is standard input), gzips what the writers return with
 * the reference's compression levels, and prints; every FASTQ byte is checked, records are delimited, names indexed and looked up, reads
 * scanned on the GPU.  fastq_info streams its files: the library asks for the operands it would open (fqg_fastq_info_stream) and reads
 * them piece by piece (FQG_PIECE_BYTES, default 64 MiB) through the callbacks below, inflating one piece on a helper thread while the
 * previous one is copied to the device and validated.
 */
#include <zlib.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "../../include/fastq_gpu.h"

static void* gz_open(void*, const char* name) {
  gzFile fd = strcmp(name, "-") == 0 ? gzdopen(fileno(stdin), "r") : gzopen(name, "r");
  if (fd) gzbuffer(fd, 1 << 20);
  return fd;
}
static long gz_read(void*, void* h, void* buf, size_t cap) { return gzread((gzFile)h, buf, cap > (1u << 30) ? (1u << 30) : (unsigned)cap); }
static void gz_close(void*, void* h) { gzclose((gzFile)h); }

/* a whole file inflated; false: it cannot be opened */
static bool slurp(const char* name, std::vector<char>* out) {
  gzFile fd = (gzFile)gz_open(nullptr, name);
  if (!fd) return false;
  std::vector<char> piece(8u << 20);
  int k;
  while ((k = gzread(fd, piece.data(), (unsigned)piece.size())) > 0) out->insert(out->end(), piece.data(), piece.data() + k);
  gzclose(fd);
  return true;
}
static bool gz_write_file(const char* name, const char* mode, const char* p, size_t n) {
  gzFile fd = strcmp(name, "-") == 0 ? gzdopen(fileno(stdout), "wb") : gzopen(name, mode);
  if (!fd) return false;
  gzbuffer(fd, 128000);
  for (size_t off = 0; off < n;) { const unsigned k = (unsigned)(n - off > (1u << 30) ? (1u << 30) : n - off); if (gzwrite(fd, p + off, k) <= 0) break; off += k; }
  gzclose(fd);
  return true;
}
static int finish(fqg_transcript& t) {
  fwrite(t.out, 1, t.out_len, stdout);
  fwrite(t.err, 1, t.err_len, stderr);
  const int rc = t.rc;
  fqg_transcript_free(&t);
  return rc;
}
static int failed(int st) { fprintf(stderr, "\nERROR: libfastq_gpu failed (%d)\n", st); return 2; } /* SYS_INT_ERROR_EXIT_STATUS */

int main(int argc, char** argv) {
  const char* dev_s = getenv("FQG_DEVICE");
  const int dev = dev_s ? atoi(dev_s) : 0;
  std::string tool = argv[0];
  if (tool.rfind('/') != std::string::npos) tool = tool.substr(tool.rfind('/') + 1);
  if (tool.size() > 4 && tool.compare(tool.size() - 4, 4, "_gpu") == 0) tool.resize(tool.size() - 4);
  if (tool == "fastq_tools") {
    if (argc < 2) { fprintf(stderr, "usage: fastq_tools_gpu <fastq_info|fastq_num_reads|fastq_not_empty|fastq_truncate|fastq_filter_n|fastq_trim_poly_at|fastq_filterpair> arguments...\n"); return 1; }
    tool = argv[1]; argv++; argc--;
  }
  std::vector<const char*> av(argv, argv + argc);
  av[0] = tool.c_str();
  fqg_transcript t; memset(&t, 0, sizeof t);
  fqg_stream_io io; io.user = nullptr; io.open = gz_open; io.read = gz_read; io.close = gz_close;
  if (tool == "fastq_info") {
    const char* piece = getenv("FQG_PIECE_BYTES");
    const int st = fqg_fastq_info_stream(argc, av.data(), &io, dev, piece ? (size_t)strtoull(piece, nullptr, 10) : 0, &t);
    if (st) return failed(st);
    return finish(t);
  }
  if (tool == "fastq_trim_poly_at") {
    char* data = nullptr; size_t n = 0; const char* oname = nullptr;
    const int st = fqg_trim_poly_at_stream(argc, av.data(), &io, dev, &t, &data, &n, &oname);
    if (st) return failed(st);
    if (oname && !gz_write_file(oname, "w4", data, n)) { fprintf(stderr, "\nERROR: Unable to open %s\n", oname); return 1; } /* src/fastq.c:651-655 */
    fqg_buffer_free(data);
    return finish(t);
  }
  if (tool == "fastq_filterpair") {
    std::vector<char> a, b;
    const bool oa = argc >= 2 && slurp(argv[1], &a), ob = argc >= 3 && slurp(argv[2], &b);
    char* outs[3]; size_t lens[3]; int32_t created = 0;
    const int st = fqg_filterpair_mem(argc, av.data(), a.data(), oa ? a.size() : (size_t)-1, b.data(), ob ? b.size() : (size_t)-1, dev, &t, outs, lens, &created);
    if (st) return failed(st);
    if (created) for (int i = 0; i < 3; i++) if (!gz_write_file(argv[3 + i], "w3", outs[i], lens[i])) { fprintf(stderr, "Unable to create output files\n"); return 1; }
    for (int i = 0; i < 3; i++) fqg_buffer_free(outs[i]);
    return finish(t);
  }
  /* the tools of fqg_reader_tool_mem take the one file the reference would open: its first operand (fastq_filter_n: behind its options) */
  std::vector<char> a; bool opened = false;
  bool dashes = false; /* fastq_filter_n takes argv[1 + options] for its file: after "--" that is the "--" itself, which cannot be opened */
  for (int i = 1; i < argc; i++) if (tool == "fastq_filter_n" && !strcmp(argv[i], "--")) dashes = true;
  for (int i = 1; i < argc && !opened && !dashes; i++) {
    if (tool == "fastq_filter_n" && argv[i][0] == '-' && argv[i][1] != '\0') { if (!strcmp(argv[i], "-n")) i++; continue; }
    opened = slurp(argv[i], &a);
    break;
  }
  const int st = fqg_reader_tool_mem(argc, av.data(), a.data(), opened ? a.size() : (size_t)-1, dev, 0, &t);
  if (st) return failed(st);
  return finish(t);
}
