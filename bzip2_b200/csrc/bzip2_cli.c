/*
 * bzip2_cli.c -- `bzip2` command-line front end over the GPU library.
 *
 * Mirrors the user-visible behaviour of the reference CLI
 * (bzip2.c: flag parsing :1870-1934, compressStream :328-427, compress() :1132-1309,
 *  uncompressStream :432-553, testStream :557-642, uncompress() :1313-1507):
 *   -1..-9 / --fast / --best, -z, -c, -k, -f, -q, -v, -s (clamps the level to 2,
 *   bzip2.c:1937-1938), BZIP2 / BZIP environment flags, "file" -> "file.bz2", refusal to
 *   overwrite without -f, refusal to write compressed data to a terminal, input removed
 *   after success unless -k / -c.
 * It feeds the libbz2-compatible stdio API (BZ2_bzWriteOpen / BZ2_bzWrite /
 * BZ2_bzWriteClose64), with 4 MiB reads instead of the reference's 5000-byte trickle
 * (bzip2.c:350-358) -- the stream bytes do not depend on the chunking.
 * -d / -t (and the bunzip2 / bzcat program names) run the library's host decoder
 * (BZ2_bzReadOpen / BZ2_bzRead / BZ2_bzReadGetUnused): concatenated streams are decoded
 * back to back, trailing garbage after a complete stream is ignored with a warning,
 * exit status 2 reports corrupt input (bzip2.c:432-553).
 */
#include "../../include/bzlib.h"
#include "../../include/bz2_b200.h"
#include <errno.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>
#include <time.h>
#include <stdint.h>

enum { OP_COMPRESS, OP_DECOMPRESS, OP_TEST };
static int level = 9, to_stdout = 0, keep = 0, force = 0, quiet = 0, verbose = 0, small = 0, op = OP_COMPRESS;
static const char* prog = "bzip2";

static void usage(void)
{
   fprintf(stderr,
      "bzip2-b200, a GPU (sm_100a) block-sorting file compressor, stream-compatible with bzip2 1.0.6.\n\n"
      "   usage: %s [flags and input files in any order]\n\n"
      "   -z --compress       compress on the GPU (default)\n"
      "   -d --decompress     decompress (host decoder)\n"
      "   -t --test           test compressed file integrity\n"
      "   -k --keep           keep (don't delete) input files\n"
      "   -f --force          overwrite existing output files\n"
      "   -c --stdout         output to standard out\n"
      "   -q --quiet          suppress noncritical error messages\n"
      "   -v --verbose        be verbose\n"
      "   -s --small          use block size 200k at most\n"
      "   -1 .. -9            set block size to 100k .. 900k\n"
      "   --fast / --best     alias for -1 / -9\n\n"
      "   If no file names are given, compresses standard input to standard output.\n", prog);
}

static double now_s(void)
{
   struct timespec ts;
   clock_gettime(CLOCK_MONOTONIC, &ts);
   return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* Regular files of up to 3 GiB are read whole and compressed with ONE call of the engine's one-shot entry point instead
 * of the reference's read-a-bit / BZ2_bzWrite loop (bzip2.c:350-358): the size is known, so a small file gets an engine
 * sized to it (no ~9 GB of HBM for a 100 kB file; the engines are kept for the next file of the invocation), and a large
 * one can be spread over several GPUs / engines (BZ2_B200_DEVICES).  BZ2B200_TAIL_STREAMED keeps the bytes those of the
 * streaming loop (every input byte arrives in BZ_RUN mode there, bzlib.c:276-308).  BZ2_B200_CLI_STREAM=1 forces the loop. */
#define ONE_SHOT_MAX ((unsigned long long)3 << 30)
#define SMALL_FILE   ((size_t)8 << 20)
static struct { bz2b200_engine* e; int level; size_t cap; } small_eng, big_eng;
static struct { bz2b200_multi* m; int level; } multi_eng;

static int parse_device_list(const char* v, int* out, int max)
{
   int n = 0;
   while (v && *v && n < max) {
      char* end;
      long d = strtol(v, &end, 10);
      if (end == v) break;
      out[n++] = (int)d;
      if (*end != ',') break;
      v = end + 1;
   }
   return n;
}

static int compress_whole_file(FILE* in, FILE* out, const char* name, size_t size, int lvl,
                               unsigned long long* nin, unsigned long long* nout)
{
   const size_t cap = size + size / 50 + 24576 * (size / (100000 * (size_t)lvl - 19) + 2) + 1024;
   unsigned char* src = (unsigned char*)malloc(size ? size : 1);
   unsigned char* dst = (unsigned char*)malloc(cap);
   size_t dlen = cap, got;
   int rc, devs[16], ndev;
   if (!src || !dst) { free(src); free(dst); return -1; }             /* fall back to the streaming loop */
   got = fread(src, 1, size, in);
   if (ferror(in)) { fprintf(stderr, "%s: %s: read error: %s\n", prog, name, strerror(errno)); free(src); free(dst); return 1; }
   if (got != size || fgetc(in) != EOF) { free(src); free(dst); if (fseek(in, 0, SEEK_SET) != 0) return 1; return -1; }   /* the file changed size */
   ndev = parse_device_list(getenv("BZ2_B200_DEVICES"), devs, 16);
   if (size <= SMALL_FILE) {
      size_t want = (size_t)1 << 20;
      while (want < size) want <<= 1;
      if (small_eng.e && (small_eng.level != lvl || small_eng.cap < size)) { bz2b200_engine_destroy(small_eng.e); small_eng.e = NULL; }
      rc = small_eng.e ? 0 : bz2b200_engine_create_bounded(&small_eng.e, getenv("BZ2_B200_DEVICE") ? atoi(getenv("BZ2_B200_DEVICE")) : 0, lvl, want);
      if (rc == 0) { small_eng.level = lvl; small_eng.cap = want; bz2b200_engine_set_verbosity(small_eng.e, verbose);
                     rc = bz2b200_compress_host(small_eng.e, src, size, dst, &dlen, BZ2B200_TAIL_STREAMED, NULL); }
   } else if (ndev >= 2) {
      if (multi_eng.m && multi_eng.level != lvl) { bz2b200_multi_destroy(multi_eng.m); multi_eng.m = NULL; }
      rc = multi_eng.m ? 0 : bz2b200_multi_create(&multi_eng.m, devs, ndev, lvl, 0);
      if (rc == 0) { multi_eng.level = lvl; rc = bz2b200_multi_compress(multi_eng.m, src, NULL, size, dst, &dlen, BZ2B200_TAIL_STREAMED, NULL); }
   } else {
      if (big_eng.e && big_eng.level != lvl) { bz2b200_engine_destroy(big_eng.e); big_eng.e = NULL; }
      rc = big_eng.e ? 0 : bz2b200_engine_create(&big_eng.e, getenv("BZ2_B200_DEVICE") ? atoi(getenv("BZ2_B200_DEVICE")) : 0, lvl, 0);
      if (rc == 0) { big_eng.level = lvl; bz2b200_engine_set_verbosity(big_eng.e, verbose);
                     rc = bz2b200_compress_host(big_eng.e, src, size, dst, &dlen, BZ2B200_TAIL_STREAMED, NULL); }
   }
   free(src);
   if (rc) {
      fprintf(stderr, "%s: %s: the GPU compressor failed (%d: %s)%s\n", prog, name, rc, bz2b200_last_error(),
              rc == BZ2B200_ENODEV ? "; this build has no CPU path" : "");
      free(dst);
      return 1;
   }
   if (fwrite(dst, 1, dlen, out) != dlen || fflush(out) != 0) { fprintf(stderr, "%s: write error: %s\n", prog, strerror(errno)); free(dst); return 1; }
   free(dst);
   *nin = size; *nout = dlen;
   return 0;
}

static int compress_stream(FILE* in, FILE* out, const char* name, unsigned long long* nin, unsigned long long* nout)
{
   const int timing = getenv("BZ2_B200_CLI_TIMING") != NULL;     /* phase times on stderr */
   {
      struct stat sb;
      const char* force = getenv("BZ2_B200_CLI_STREAM");
      if (!(force && *force == '1') && fstat(fileno(in), &sb) == 0 && S_ISREG(sb.st_mode) && (unsigned long long)sb.st_size <= ONE_SHOT_MAX
          && ftell(in) == 0) {
         const int r = compress_whole_file(in, out, name, (size_t)sb.st_size, small && level > 2 ? 2 : level, nin, nout);
         if (r >= 0) return r;
      }
   }
   double t0 = now_s(), t_open, t_read = 0, t_write = 0, t_loop;
   enum { CHUNK = 4 << 20 };
   int bzerr = BZ_OK;
   unsigned int in_lo = 0, in_hi = 0, out_lo = 0, out_hi = 0;
   char* buf = (char*)malloc(CHUNK);
   BZFILE* bz;
   if (!buf) { fprintf(stderr, "%s: out of memory\n", prog); return 1; }
   bz = BZ2_bzWriteOpen(&bzerr, out, small && level > 2 ? 2 : level, verbose, 30);
   if (bzerr != BZ_OK) {
      fprintf(stderr, "%s: cannot start the GPU compressor (libbz2 error %d%s)\n", prog, bzerr,
              bzerr == BZ_CONFIG_ERROR ? ": no usable CUDA device; this build has no CPU path" : "");
      free(buf);
      return 1;
   }
   t_open = now_s();
   for (;;) {
      double ta = now_s(), tb;
      size_t n = fread(buf, 1, CHUNK, in);
      tb = now_s(); t_read += tb - ta;
      if (ferror(in)) { fprintf(stderr, "%s: %s: read error: %s\n", prog, name, strerror(errno)); BZ2_bzWriteClose64(&bzerr, bz, 1, 0, 0, 0, 0); free(buf); return 1; }
      if (n > 0) {
         ta = now_s();
         BZ2_bzWrite(&bzerr, bz, buf, (int)n);
         t_write += now_s() - ta;
         if (bzerr != BZ_OK) { fprintf(stderr, "%s: %s: compression failed (libbz2 error %d)\n", prog, name, bzerr); BZ2_bzWriteClose64(&bzerr, bz, 1, 0, 0, 0, 0); free(buf); return 1; }
      }
      if (n < CHUNK) break;
   }
   t_loop = now_s();
   BZ2_bzWriteClose64(&bzerr, bz, 0, &in_lo, &in_hi, &out_lo, &out_hi);
   if (timing)
      fprintf(stderr, "%s: open %.3f s, loop %.3f s (fread %.3f, bzWrite %.3f), close %.3f s\n", prog, t_open - t0, t_loop - t_open,
              t_read, t_write, now_s() - t_loop);
   free(buf);
   if (bzerr != BZ_OK) { fprintf(stderr, "%s: %s: compression failed (libbz2 error %d)\n", prog, name, bzerr); return 1; }
   if (fflush(out) != 0) { fprintf(stderr, "%s: write error: %s\n", prog, strerror(errno)); return 1; }
   *nin = ((unsigned long long)in_hi << 32) | in_lo;
   *nout = ((unsigned long long)out_hi << 32) | out_lo;
   return 0;
}

/* Decodes every stream in `in`; out == NULL only tests.  0 ok, 1 i/o trouble, 2 corrupt input. */
static int expand_stream(FILE* in, FILE* out, const char* name)
{
   enum { CHUNK = 1 << 16 };
   static char obuf[CHUNK];
   char carry[BZ_MAX_UNUSED];
   int ncarry = 0, streams = 0, bzerr = BZ_OK;
   for (;;) {
      void* un; int nun, c;
      BZFILE* bz = BZ2_bzReadOpen(&bzerr, in, verbose, small, carry, ncarry);
      if (bz == NULL || bzerr != BZ_OK) { fprintf(stderr, "%s: %s: cannot start the decoder (libbz2 error %d)\n", prog, name, bzerr); return 1; }
      streams++;
      while (bzerr == BZ_OK) {
         int n = BZ2_bzRead(&bzerr, bz, obuf, CHUNK);
         if (bzerr == BZ_DATA_ERROR_MAGIC) break;
         if ((bzerr == BZ_OK || bzerr == BZ_STREAM_END) && n > 0 && out) {
            if (fwrite(obuf, 1, (size_t)n, out) != (size_t)n || ferror(out)) {
               fprintf(stderr, "%s: %s: write error: %s\n", prog, name, strerror(errno));
               BZ2_bzReadClose(&bzerr, bz);
               return 1;
            }
         }
      }
      if (bzerr != BZ_STREAM_END) {
         int e = bzerr;
         BZ2_bzReadClose(&bzerr, bz);
         if (e == BZ_DATA_ERROR_MAGIC) {
            if (streams == 1) { fprintf(stderr, "%s: %s is not a bzip2 file.\n", prog, name); return 2; }
            if (!quiet) fprintf(stderr, "\n%s: %s: trailing garbage after EOF ignored\n", prog, name);
            break;
         }
         if (e == BZ_IO_ERROR) { fprintf(stderr, "%s: %s: read error: %s\n", prog, name, strerror(errno)); return 1; }
         if (e == BZ_UNEXPECTED_EOF) fprintf(stderr, "%s: %s: file ends unexpectedly\n", prog, name);
         else if (e == BZ_MEM_ERROR) { fprintf(stderr, "%s: out of memory\n", prog); return 1; }
         else fprintf(stderr, "%s: %s: data integrity (CRC) error in data\n", prog, name);
         return 2;
      }
      BZ2_bzReadGetUnused(&bzerr, bz, &un, &nun);
      ncarry = nun;
      if (nun > 0) memcpy(carry, un, (size_t)nun);
      BZ2_bzReadClose(&bzerr, bz);
      if (ncarry == 0) {
         c = fgetc(in);
         if (c == EOF) break;
         ungetc(c, in);
      }
   }
   if (ferror(in)) { fprintf(stderr, "%s: %s: read error: %s\n", prog, name, strerror(errno)); return 1; }
   if (out && fflush(out) != 0) { fprintf(stderr, "%s: write error: %s\n", prog, strerror(errno)); return 1; }
   if (verbose) fprintf(stderr, "  %s: %s\n", name, out ? "done" : "ok");
   return 0;
}

/* "x.bz2" -> "x", "x.tbz2" -> "x.tar", anything else -> "x.out" (bzip2.c:1313-1345). */
static int expanded_name(const char* name, char* dst, size_t cap)
{
   static const char* const from[] = { ".bz2", ".bz", ".tbz2", ".tbz" };
   static const char* const to[] = { "", "", ".tar", ".tar" };
   size_t L = strlen(name), k;
   for (k = 0; k < 4; k++) {
      size_t fl = strlen(from[k]);
      if (L > fl && strcmp(name + L - fl, from[k]) == 0) {
         snprintf(dst, cap, "%.*s%s", (int)(L - fl), name, to[k]);
         return 1;
      }
   }
   snprintf(dst, cap, "%s.out", name);
   return 0;
}

static int expand_file(const char* name)
{
   char outname[4096];
   struct stat st;
   FILE *in, *out;
   int rc;
   if (strlen(name) + 5 > sizeof outname) { fprintf(stderr, "%s: file name too long: %s\n", prog, name); return 1; }
   if (stat(name, &st) != 0) { fprintf(stderr, "%s: Can't open input file %s: %s.\n", prog, name, strerror(errno)); return 1; }
   if (S_ISDIR(st.st_mode)) { fprintf(stderr, "%s: Input file %s is a directory.\n", prog, name); return 1; }
   in = fopen(name, "rb");
   if (!in) { fprintf(stderr, "%s: Can't open input file %s: %s.\n", prog, name, strerror(errno)); return 1; }
   if (op == OP_TEST || to_stdout) {
      rc = expand_stream(in, op == OP_TEST ? NULL : stdout, name);
      fclose(in);
      return rc;
   }
   if (!expanded_name(name, outname, sizeof outname) && !quiet)
      fprintf(stderr, "%s: Can't guess original name for %s -- using %s\n", prog, name, outname);
   if (!force && access(outname, F_OK) == 0) {
      fprintf(stderr, "%s: Output file %s already exists.\n", prog, outname);
      fclose(in);
      return 1;
   }
   out = fopen(outname, "wb");
   if (!out) { fprintf(stderr, "%s: Can't create output file %s: %s.\n", prog, outname, strerror(errno)); fclose(in); return 1; }
   rc = expand_stream(in, out, name);
   fclose(in);
   if (fclose(out) != 0 && !rc) rc = 1;
   if (rc) { remove(outname); return rc; }
   chmod(outname, st.st_mode & 07777);
   if (!keep) remove(name);
   return 0;
}

static void report(const char* name, unsigned long long nin, unsigned long long nout)
{
   if (!verbose) return;
   if (nin == 0) { fprintf(stderr, "  %s: no data compressed.\n", name); return; }
   fprintf(stderr, "  %s: %6.3f:1, %6.3f bits/byte, %5.2f%% saved, %llu in, %llu out.\n", name,
           (double)nin / (double)nout, 8.0 * (double)nout / (double)nin, 100.0 * (1.0 - (double)nout / (double)nin), nin, nout);
}

/* Consecutive small regular files are compressed together: one bz2b200_compress_batch_host call per batch of up to
 * BATCH_BYTES of input or BATCH_FILES files, on one engine kept for the invocation, instead of a whole set of kernel
 * launches and host round trips per file.  Every file still becomes its own stream with the bytes a call of its own
 * gives.  The batch is finished -- files written, closed, chmod-ed, removed unless -k, reported -- in argument order,
 * and before anything is printed about a later file or a later file is handled another way, so stderr and the output
 * files keep the order of one file at a time.  Not used with -vv and above (the per-block trace) or under
 * BZ2_B200_CLI_STREAM=1. */
#define BATCH_BYTES ((size_t)32 << 20)
#define BATCH_FILES 1024
static struct {
   unsigned char* buf; size_t len, cap;
   int n;
   char* name[BATCH_FILES];
   mode_t mode[BATCH_FILES];
   uint64_t offs[BATCH_FILES + 1];
} pend;
static struct { bz2b200_engine* e; int level; } batch_eng;
static int full_batch_rc;          /* exit code of batches flushed because they were full */

static int batch_usable(void)
{
   const char* force_stream = getenv("BZ2_B200_CLI_STREAM");
   return verbose < 2 && !(force_stream && *force_stream == '1');
}

/* Compress and finish every pending file.  Returns the largest exit code among them. */
static int flush_batch(void)
{
   const int lvl = small && level > 2 ? 2 : level;
   int rc = 0, k, r;
   size_t cap = 0;
   unsigned char* dst;
   uint64_t out_offs[BATCH_FILES + 1];
   if (pend.n == 0) return 0;
   for (k = 0; k < pend.n; k++) cap += bz2b200_compress_bound(lvl, (size_t)(pend.offs[k + 1] - pend.offs[k]));
   dst = (unsigned char*)malloc(cap ? cap : 1);
   if (batch_eng.e && batch_eng.level != lvl) { bz2b200_engine_destroy(batch_eng.e); batch_eng.e = NULL; }
   r = !dst ? BZ2B200_ENOMEM
       : batch_eng.e ? 0
       : bz2b200_engine_create_batch(&batch_eng.e, getenv("BZ2_B200_DEVICE") ? atoi(getenv("BZ2_B200_DEVICE")) : 0, lvl,
                                     BATCH_BYTES, BATCH_FILES);
   if (r == 0) {
      batch_eng.level = lvl;
      bz2b200_engine_set_verbosity(batch_eng.e, verbose);
      r = bz2b200_compress_batch_host(batch_eng.e, pend.buf, pend.offs, (size_t)pend.n, dst, cap, out_offs, NULL,
                                      BZ2B200_TAIL_STREAMED, NULL);
   }
   for (k = 0; k < pend.n; k++) {
      const char* name = pend.name[k];
      const unsigned long long nin = pend.offs[k + 1] - pend.offs[k];
      unsigned long long nout;
      char outname[4096];
      FILE* out;
      if (r) {
         fprintf(stderr, "%s: %s: the GPU compressor failed (%d: %s)%s\n", prog, name, r, bz2b200_last_error(),
                 r == BZ2B200_ENODEV ? "; this build has no CPU path" : "");
         rc = 1;
         continue;
      }
      nout = out_offs[k + 1] - out_offs[k];
      if (to_stdout) {
         if (fwrite(dst + out_offs[k], 1, nout, stdout) != nout || fflush(stdout) != 0) {
            fprintf(stderr, "%s: write error: %s\n", prog, strerror(errno));
            rc = 1;
            continue;
         }
         report(name, nin, nout);
         continue;
      }
      snprintf(outname, sizeof outname, "%s.bz2", name);
      out = fopen(outname, "wb");
      if (!out) { fprintf(stderr, "%s: Can't create output file %s: %s.\n", prog, outname, strerror(errno)); rc = 1; continue; }
      if (fwrite(dst + out_offs[k], 1, nout, out) != nout || fflush(out) != 0) {
         fprintf(stderr, "%s: write error: %s\n", prog, strerror(errno));
         fclose(out);
         remove(outname);
         rc = 1;
         continue;
      }
      if (fclose(out) != 0) { remove(outname); rc = 1; continue; }
      chmod(outname, pend.mode[k] & 07777);
      if (!keep) remove(name);
      report(name, nin, nout);
   }
   free(dst);
   for (k = 0; k < pend.n; k++) free(pend.name[k]);
   pend.n = 0; pend.len = 0;
   return rc;
}

/* Queue `name` for the next batch if it is a small regular file that would be compressed without a word on stderr.
 * 1: queued; 0: the caller flushes the batch and handles the file one at a time. */
static int queue_small_file(const char* name)
{
   struct stat st;
   size_t L = strlen(name), size, got;
   FILE* in;
   char outname[4096];
   int k;
   if (!batch_usable() || L + 5 > sizeof outname || stat(name, &st) != 0 || !S_ISREG(st.st_mode)) return 0;
   if ((unsigned long long)st.st_size > SMALL_FILE) return 0;
   if (L > 4 && strcmp(name + L - 4, ".bz2") == 0 && !force) return 0;
   snprintf(outname, sizeof outname, "%s.bz2", name);
   if (!to_stdout && !force && access(outname, F_OK) == 0) return 0;
   size = (size_t)st.st_size;
   for (k = 0; k < pend.n; k++) if (!strcmp(pend.name[k], name)) return 0;          /* the same file twice */
   if (pend.n == BATCH_FILES || pend.len + size > BATCH_BYTES) { const int r = flush_batch(); if (r > full_batch_rc) full_batch_rc = r; }
   if (pend.len + size > pend.cap) {
      size_t nc = pend.cap ? pend.cap : ((size_t)1 << 20);
      unsigned char* nb;
      while (nc < pend.len + size) nc *= 2;
      nb = (unsigned char*)realloc(pend.buf, nc);
      if (!nb) return 0;
      pend.buf = nb; pend.cap = nc;
   }
   in = fopen(name, "rb");
   if (!in) return 0;
   got = fread(pend.buf + pend.len, 1, size, in);
   if (ferror(in) || got != size || fgetc(in) != EOF) { fclose(in); return 0; }    /* the file changed: one at a time */
   fclose(in);
   pend.name[pend.n] = strdup(name);
   if (!pend.name[pend.n]) return 0;
   pend.mode[pend.n] = st.st_mode;
   pend.offs[pend.n] = pend.len;
   pend.len += size;
   pend.n++;
   pend.offs[pend.n] = pend.len;
   return 1;
}

static int do_file_now(const char* name);

static int do_file(const char* name)
{
   int r, r2;
   if (op != OP_COMPRESS) return expand_file(name);
   if (queue_small_file(name)) return 0;
   r = flush_batch();
   r2 = do_file_now(name);
   return r > r2 ? r : r2;
}

static int do_file_now(const char* name)
{
   char outname[4096];
   struct stat st;
   FILE *in, *out;
   unsigned long long nin = 0, nout = 0;
   int rc;
   size_t L = strlen(name);
   if (L + 5 > sizeof outname) { fprintf(stderr, "%s: file name too long: %s\n", prog, name); return 1; }
   if (stat(name, &st) != 0) { fprintf(stderr, "%s: Can't open input file %s: %s.\n", prog, name, strerror(errno)); return 1; }
   if (S_ISDIR(st.st_mode)) { fprintf(stderr, "%s: Input file %s is a directory.\n", prog, name); return 1; }
   if (L > 4 && strcmp(name + L - 4, ".bz2") == 0 && !force) {
      if (!quiet) fprintf(stderr, "%s: Input file %s already has .bz2 suffix.\n", prog, name);
      return 1;
   }
   in = fopen(name, "rb");
   if (!in) { fprintf(stderr, "%s: Can't open input file %s: %s.\n", prog, name, strerror(errno)); return 1; }
   if (to_stdout) {
      rc = compress_stream(in, stdout, name, &nin, &nout);
      fclose(in);
      if (!rc) report(name, nin, nout);
      return rc;
   }
   snprintf(outname, sizeof outname, "%s.bz2", name);
   if (!force && access(outname, F_OK) == 0) {
      fprintf(stderr, "%s: Output file %s already exists.\n", prog, outname);
      fclose(in);
      return 1;
   }
   out = fopen(outname, "wb");
   if (!out) { fprintf(stderr, "%s: Can't create output file %s: %s.\n", prog, outname, strerror(errno)); fclose(in); return 1; }
   rc = compress_stream(in, out, name, &nin, &nout);
   fclose(in);
   if (fclose(out) != 0) rc = 1;
   if (rc) { remove(outname); return rc; }
   chmod(outname, st.st_mode & 07777);
   if (!keep) remove(name);
   report(name, nin, nout);
   return 0;
}

static int handle_flag(const char* a)
{
   if (a[1] == '-') {
      if (!strcmp(a, "--stdout")) to_stdout = 1;
      else if (!strcmp(a, "--compress")) op = OP_COMPRESS;
      else if (!strcmp(a, "--decompress")) op = OP_DECOMPRESS;
      else if (!strcmp(a, "--test")) op = OP_TEST;
      else if (!strcmp(a, "--keep")) keep = 1;
      else if (!strcmp(a, "--force")) force = 1;
      else if (!strcmp(a, "--quiet")) quiet = 1;
      else if (!strcmp(a, "--verbose")) verbose++;
      else if (!strcmp(a, "--small")) small = 1;
      else if (!strcmp(a, "--fast")) level = 1;
      else if (!strcmp(a, "--best")) level = 9;
      else if (!strcmp(a, "--repetitive-fast") || !strcmp(a, "--repetitive-best") || !strcmp(a, "--exponential")) {}
      else if (!strcmp(a, "--help")) { usage(); exit(0); }
      else { fprintf(stderr, "%s: Bad flag `%s'\n", prog, a); usage(); exit(1); }
      return 0;
   }
   for (const char* p = a + 1; *p; p++) {
      switch (*p) {
         case 'c': to_stdout = 1; break;
         case 'z': op = OP_COMPRESS; break;
         case 'd': op = OP_DECOMPRESS; break;
         case 't': op = OP_TEST; break;
         case 'k': keep = 1; break;
         case 'f': force = 1; break;
         case 'q': quiet = 1; break;
         case 'v': verbose++; break;
         case 's': small = 1; break;
         case 'h': usage(); exit(0);
         case '1': case '2': case '3': case '4': case '5': case '6': case '7': case '8': case '9': level = *p - '0'; break;
         default: fprintf(stderr, "%s: Bad flag `%s'\n", prog, a); usage(); exit(1);
      }
   }
   return 0;
}

static void env_flags(const char* var)
{
   const char* v = getenv(var);
   char tmp[1024];
   char* tok;
   if (!v) return;
   snprintf(tmp, sizeof tmp, "%s", v);
   for (tok = strtok(tmp, " \t"); tok; tok = strtok(NULL, " \t")) if (tok[0] == '-' && tok[1]) handle_flag(tok);
}

static int run(int argc, char** argv)
{
   int i, nfiles = 0, rc = 0, dashdash = 0;
   const char* slash = strrchr(argv[0], '/');
   prog = slash ? slash + 1 : argv[0];
   if (strstr(prog, "unzip") || strstr(prog, "UNZIP")) op = OP_DECOMPRESS;
   if (strstr(prog, "z2cat") || strstr(prog, "Z2CAT") || strstr(prog, "zcat") || strstr(prog, "ZCAT")) { op = OP_DECOMPRESS; to_stdout = 1; }
   env_flags("BZIP2");
   env_flags("BZIP");
   for (i = 1; i < argc; i++) {
      if (!dashdash && !strcmp(argv[i], "--")) { dashdash = 1; continue; }
      if (!dashdash && argv[i][0] == '-' && argv[i][1]) handle_flag(argv[i]); else nfiles++;
   }
   if (verbose > 4) verbose = 4;
   if (nfiles == 0 && op != OP_COMPRESS) {
      if (op == OP_DECOMPRESS && isatty(fileno(stdin)) && !force) {
         fprintf(stderr, "%s: I won't read compressed data from a terminal.\n%s: For help, type: `%s --help'.\n", prog, prog, prog);
         return 1;
      }
      return expand_stream(stdin, op == OP_TEST ? NULL : stdout, "(stdin)");
   }
   if (nfiles == 0) {
      unsigned long long nin = 0, nout = 0;
      if (isatty(fileno(stdout)) && !force) {
         fprintf(stderr, "%s: I won't write compressed data to a terminal.\n%s: For help, type: `%s --help'.\n", prog, prog, prog);
         return 1;
      }
      rc = compress_stream(stdin, stdout, "(stdin)", &nin, &nout);
      if (!rc) report("(stdin)", nin, nout);
      return rc;
   }
   dashdash = 0;
   for (i = 1; i < argc; i++) {
      if (!dashdash && !strcmp(argv[i], "--")) { dashdash = 1; continue; }
      if (!dashdash && argv[i][0] == '-' && argv[i][1]) continue;
      { int r = do_file(argv[i]); if (r > rc) rc = r; }
   }
   { int r = flush_batch(); if (r > rc) rc = r; }
   return rc > full_batch_rc ? rc : full_batch_rc;
}

/* Everything is flushed and closed by the time run() returns; leaving through _exit skips the CUDA
 * runtime's exit handlers (freeing several GB of device and pinned memory allocation by allocation
 * costs more than the whole compression of a 2 GB file) and lets the driver reclaim the context. */
int main(int argc, char** argv)
{
   const double t0 = now_s();
   const int rc = run(argc, argv);
   fflush(stdout);
   fflush(stderr);
   if (getenv("BZ2_B200_CLI_TIMING")) { fprintf(stderr, "%s: main returned after %.3f s\n", argv[0], now_s() - t0); fflush(stderr); }
   if (getenv("BZ2_B200_CLI_SLOWEXIT")) return rc;
   _exit(rc);
}
