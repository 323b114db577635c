/*
 * fq_types.h — plain-data types shared by the host engine and the CUDA kernels of libfastq_gpu.
 *
 * Vocabulary follows the reference (fastq_utils 0.25.3): a *record* is four gz-lines (hdr1, seq, hdr2, qual;
 * src/fastq.h:97-108), a *file* is a FASTQ stream (src/fastq.h:110-131), the *index* is the read-name
 * uniqueness table (src/hash.c + src/fastq.c:529-611).  A *chunk* is a contiguous piece of one file's
 * decompressed byte stream resident in HBM (≤ 4 GiB so that byte offsets are 32-bit).
 */
#ifndef FQ_TYPES_H
#define FQ_TYPES_H
#include <stdint.h>

#if defined(__CUDACC__)
#define FQ_HD __host__ __device__ __forceinline__
#else
#define FQ_HD inline
#endif

/* gzgets limits, src/fastq.h:30-37 */
#define FQ_MAX_READ_LENGTH 2500000u
#define FQ_MAX_LABEL_LENGTH 1000u
#define FQ_MAX_PHRED 126u

/* read-name formats, src/fastq.h:25-28 (INTEGERNAME and NOP share the value 2) */
enum { FQ_FMT_UNDEF = -1, FQ_FMT_DEFAULT = 0, FQ_FMT_CASAVA = 1, FQ_FMT_INT = 2 };
/* what the format sniff found (decides which info line is printed, src/fastq.c:459-478) */
enum { FQ_SNIFF_DEFAULT = 0, FQ_SNIFF_CASAVA = 1, FQ_SNIFF_INT = 2, FQ_SNIFF_NOSUFFIX = 3 };
/* the read-name format a file's sniff selects */
FQ_HD int fq_fmt_of_sniff(int s) { return s == FQ_SNIFF_DEFAULT ? FQ_FMT_DEFAULT : s == FQ_SNIFF_CASAVA ? FQ_FMT_CASAVA : FQ_FMT_INT; }
enum { FQ_SPACE_UNDEF = -1, FQ_SPACE_SEQ = 0, FQ_SPACE_COLOR = 1 };

/* per-record validation outcome: the first failing step of fastq_validate_entry (src/fastq.c:300-392) */
enum {
  FQ_V_AT = 0,     /* :306  hdr1[0] != '@'                        */
  FQ_V_IDLEN = 1,  /* :310  identifier not longer than 1          */
  FQ_V_SEQ = 2,    /* :317-341 invalid character / both U and T   */
  FQ_V_SHORT = 3,  /* :346  read length too small                 */
  FQ_V_PLUS = 4,   /* :355  hdr2[0] != '+'                        */
  FQ_V_HDR2 = 5,   /* :363-370 header2 differs from header1       */
  FQ_V_LEN = 6,    /* :380-390 seq/qual length                    */
  FQ_V_OK = 7
};

/* record-level flags produced by the reader step (src/fastq.c:245-261) */
#define FQ_RF_STOP 1u    /* hdr1[0]==NUL: fastq_read_entry returns 0 (clean end of file) */
#define FQ_RF_TRUNC 2u   /* one of the other three lines is empty: "file truncated", exit 1 */
#define FQ_RF_NOTAT 4u   /* hdr1[0] != '@' (fastq_get_readname's "wrong header", src/fastq.c:448) */

/* error codes of the report (SURVEY.md appendix B) */
enum {
  FQ_OK = 0,
  FQ_E_TRUNC, FQ_E_TRUNC_PE, FQ_E_WRONGHDR, FQ_E_AT, FQ_E_IDLEN, FQ_E_BADCHAR, FQ_E_UT, FQ_E_SHORT, FQ_E_PLUS,
  FQ_E_HDR2, FQ_E_LEN, FQ_E_LEN_CS, FQ_E_DUP, FQ_E_UNPAIRED, FQ_E_LEFTOVER, FQ_E_MISMATCH, FQ_E_EOF1, FQ_E_EOF2,
  FQ_E_EMPTY, FQ_E_ENC, FQ_E_STOP /* internal: clean early end of file */
};

/* loop kinds (fastq_info.c:57-176, :322-362 and fastq.c:396-439) */
enum {
  FQ_LOOP_SINGLE = 0,      /* validate_single_fastq_file            (-r, one file)          */
  FQ_LOOP_INDEX = 1,       /* fastq_index_readnames                 (default, file 1)       */
  FQ_LOOP_MATE = 2,        /* main()'s mate loop                    (default, file 2)       */
  FQ_LOOP_INTERLEAVED = 3, /* validate_interleaved                  (pe)                    */
  FQ_LOOP_SORTED1 = 4,     /* validate_paired_sorted_fastq_file, file 1 (-r -s)             */
  FQ_LOOP_SORTED2 = 5,     /* validate_paired_sorted_fastq_file, file 2                     */
  FQ_LOOP_READER = 6       /* fastq_read_next_entry loops without validation (src/fastq_num_reads.c:43-45, fastq_not_empty.c:41-43) */
};

/* One raw gz-line inside a chunk: bytes [off, off+len), '\n' included when the line has one. */
typedef struct { uint32_t off, len; } FqLine;

/* What the record kernel needs to know about the file the records belong to. */
typedef struct {
  int32_t loop;      /* FQ_LOOP_*                                                                     */
  int32_t fmt_key;   /* read-name format used for the index/mate key (the record's own file)           */
  int32_t pe_key;    /* is_pe of that file                                                             */
  int32_t fmt_val;   /* format used by fastq_validate_entry's header2 comparison (file 1's in the mate loop, fastq_info.c:345) */
  int32_t pe_val;
  int32_t space;     /* FQ_SPACE_* used by the length check (again file 1's in the mate loop)          */
  uint32_t weight;   /* how many times fastq_new_entry_stats runs per record (2 for the index loop)    */
  uint32_t seed;     /* name-hash seed (changed only after a detected 64-bit collision)                */
} FqRecCtx;

/* Per-record result of the reader + validator steps. */
typedef struct {
  uint32_t flags;     /* FQ_RF_*                                     */
  uint32_t vrank;     /* FQ_V_*                                      */
  uint32_t code;      /* FQ_E_* of the validation failure (0 if ok)  */
  uint32_t read_len;  /* strlen(seq), terminators included           */
  uint32_t slen, qlen;
  uint32_t qmin, qmax; /* unsigned-byte min/max over the quality string; qmin>qmax when it is empty */
  uint32_t bad;       /* offending byte for FQ_E_BADCHAR              */
  uint32_t name_off, name_len; /* normalised read name (key) inside the chunk */
  uint64_t mem_len;   /* the `len` fastq_get_readname reports (feeds index_mem, fastq.c:609) */
} FqRecOut;

/* Per-file running statistics (src/fastq.c:97-110, :373-378).  Lives in device memory; histogram separate. */
typedef struct {
  unsigned long long num_rds;   /* with the reference's multiplicity */
  unsigned long long mem_sum;   /* Σ mem_len over indexed records    */
  unsigned long long n_names;   /* records that reached the index / mate key step */
  unsigned int min_rl, max_rl;  /* over read_len (terminators included) */
  unsigned int min_q, max_q;    /* unsigned-byte domain; mapped to the reference's sign-extended value on the host */
  unsigned int pad[2];
} FqStats;

/* name descriptor written by the record kernel, consumed by the index / mate / pair kernels */
typedef struct {
  uint64_t hash;   /* FQ_HASH_SKIP when the record never reaches the name step */
  uint32_t off;    /* name bytes: chunk data + off, len bytes */
  uint32_t len;
} FqName;
/* test mode (seed bit 31, fqg_set_hash_seed / FQG_TEST_WEAK_HASH): only 12 bits of the hash survive, so that different names with
 * EQUAL hashes are common and the byte compare behind every equal hash (and the walk past a slot that holds another name) is exercised */
#define FQ_SEED_WEAK 0x80000000u
#define FQ_HASH_EMPTY 0xFFFFFFFFFFFFFFFFull
#define FQ_HASH_SKIP 0xFFFFFFFFFFFFFFFEull
#define FQ_KEY_NONE 0xFFFFFFFFFFFFFFFFull
#define FQ_IDX_NONE 0xFFFFFFFFFFFFFFFFull

/* index slot: one 32-byte DRAM sector */
typedef struct {
  unsigned long long hash;   /* FQ_HASH_EMPTY = free                                   */
  unsigned long long idx1;   /* smallest file-1 record index carrying this name        */
  unsigned long long claim2; /* smallest file-2 record index that claimed it           */
  unsigned long long pad;
} FqSlot;

/* event key: (step << 6) | rank; smaller = earlier in the reference's sequential execution */
#define FQ_KEY(step, rank) ((((uint64_t)(step)) << 6) | (uint64_t)(rank))
#define FQ_KEY_STEP(k) ((k) >> 6)
#define FQ_KEY_RANK(k) ((uint32_t)((k) & 63u))

/* ranks inside one step, per loop kind (order of checks: SURVEY.md §8 a-9) */
enum { /* single / index / mate loops: one record per step */
  FQ_R_STOP = 0, FQ_R_TRUNC = 1, FQ_R_WRONGHDR = 2, FQ_R_NAME = 3 /* duplicated / unpaired */, FQ_R_V0 = 4 /* + FQ_V_* */
};
enum { /* interleaved: one pair per step */
  FQ_RI_STOP1 = 0, FQ_RI_TRUNC1 = 1, FQ_RI_NOM2 = 2, FQ_RI_TRUNC2 = 3, FQ_RI_WRONGHDR1 = 4, FQ_RI_WRONGHDR2 = 5,
  FQ_RI_UNPAIRED = 6, FQ_RI_V1 = 7, FQ_RI_V2 = 14
};
enum { /* sorted pair: one pair per step */
  FQ_RS_STOP1 = 0, FQ_RS_TRUNC1 = 1, FQ_RS_V1 = 2, FQ_RS_STOP2 = 9, FQ_RS_TRUNC2 = 10, FQ_RS_V2 = 11, FQ_RS_MISMATCH = 18
};

#endif
