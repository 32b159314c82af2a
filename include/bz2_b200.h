/*
 * bz2_b200.h -- C ABI of the B200 (sm_100a) bzip2 compression engine.
 *
 * This is the boundary the libbz2-compatible front end (include/bzlib.h,
 * bzip2_b200/csrc/bzlib_api.c) sits on, and what a maintainer of the reference
 * would bind instead of its CPU block codec.  Plain pointers and sizes only.
 *
 * What each entry point replaces in the reference (aeb1787/bzip2):
 *   bz2b200_engine_create / _destroy   the allocation half of BZ2_bzCompressInit /
 *                                      BZ2_bzCompressEnd            (bzlib.c:144-207, :458-474)
 *   bz2b200_compress_host              handle_compress driven to completion: RLE1 + CRC
 *                                      (copy_input_until_stop, bzlib.c:211-315) and
 *                                      BZ2_compressBlock per block (compress.c:822-881),
 *                                      i.e. the body of BZ2_bzBuffToBuffCompress (bzlib.c:1309-1357)
 *   bz2b200_compress_device            same, input and output resident in HBM
 *   bz2b200_compress_batch_*           the same for many inputs at once, one stream each
 *   bz2b200_stream_*                   the same work fed in pieces (BZ2_bzCompress with
 *                                      BZ_RUN / BZ_FLUSH / BZ_FINISH, bzlib.c:400-454)
 *   bz2b200_debug_*                    per-stage intermediates for parity tests (the
 *                                      reference exposes these only as EState fields,
 *                                      bzlib_private.h:226-288)
 *
 * All functions return 0 on success or a negative BZ2B200_E* code; the text of
 * the last error is available from bz2b200_last_error().  There is no CPU
 * fallback: without a usable CUDA device every call fails with BZ2B200_ENODEV.
 */
#ifndef BZ2_B200_H
#define BZ2_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define BZ2B200_OK        0
#define BZ2B200_EPARAM   (-1)
#define BZ2B200_ENODEV   (-2)   /* no CUDA device / driver: the product has no CPU path  */
#define BZ2B200_ENOMEM   (-3)
#define BZ2B200_ECUDA    (-4)
#define BZ2B200_EOUTFULL (-5)   /* destination too small                                  */
#define BZ2B200_EINTERNAL (-6)

typedef struct bz2b200_engine bz2b200_engine;

/* Flags for the one-shot calls. */
#define BZ2B200_TAIL_STREAMED 1u  /* last input byte was handed over in BZ_RUN mode (CLI-style
                                     streaming); default is BuffToBuff semantics, where a lone
                                     final byte joins a block that has just filled
                                     (bzlib.c:276-308)                                         */

/* Segment mode (one stream sharded by block over several GPUs, see bz2b200_scan_*): the call
 * emits only its blocks, starting at bit 0 of the destination; the caller places the pieces. */
#define BZ2B200_NO_HEADER     2u
#define BZ2B200_NO_TRAILER    4u

typedef struct {
   uint64_t in_bytes, out_bytes;
   uint32_t n_blocks, n_windows;
   uint64_t sum_nblock;          /* post-RLE1 bytes  (rho = sum_nblock / in_bytes)           */
   uint64_t sum_nmtf;            /* MTF symbols      (mu  = sum_nmtf / sum_nblock)           */
   uint32_t n_power_blocks;      /* blocks that were an exact power u^q                      */
   uint32_t combined_crc;
   float    ms_total, ms_s1, ms_s2, ms_s3, ms_s4;   /* CUDA-event times, summed over windows */
   uint32_t bwt_rounds;          /* prefix-doubling rounds, summed over windows              */
   uint32_t kernel_launches;
   uint64_t out_bits;            /* exact bit length of what was produced (segment mode: not padded)   */
   float    ms_span;             /* bz2b200_multi_compress: duration of the job ON THE DEVICES -- CUDA events on every
                                    engine's stream at the start of the job and after its last copy, max over engines */
} bz2b200_stats;

int  bz2b200_device_count(void);
const char* bz2b200_last_error(void);
const char* bz2b200_version(void);

/* window_bytes = 0 picks the default (96 MiB of input per window; at most 100 MiB, at least one block of pure runs). */
int  bz2b200_engine_create(bz2b200_engine** out, int device, int block_size_100k, size_t window_bytes);
/* An engine for one-shot calls on inputs of at most max_input_bytes: its window is the input, so a 100 kB call does not
 * reserve the ~9 GB of HBM a full window needs (the default window must hold a whole block of pure runs: 46 MB at -9). */
int  bz2b200_engine_create_bounded(bz2b200_engine** out, int device, int block_size_100k, size_t max_input_bytes);
void bz2b200_engine_destroy(bz2b200_engine* e);
/* Run on the caller's CUDA stream (a cudaStream_t); NULL restores the engine's own stream. */
int  bz2b200_engine_set_stream(bz2b200_engine* e, void* cuda_stream);

/* The reference's `verbosity` (bzlib.c:144; 0-4): at >= 2 one line per block with its CRC, the combined CRC and its
 * size, and the final combined CRC; at >= 3 also nblock / nMTF / symbols in use -- same text as compress.c:831-834,
 * :259-262, :877-878, on stderr.  (The per-pass coding-table statistics of compress.c:304-308, :544-550 are not kept.) */
int  bz2b200_engine_set_verbosity(bz2b200_engine* e, int verbosity);

/* Whole-stream compression, host buffers.  *dst_len: capacity in, bytes written out. */
int  bz2b200_compress_host(bz2b200_engine* e, const void* src, size_t src_len,
                           void* dst, size_t* dst_len, unsigned flags, bz2b200_stats* stats);

/* Whole-stream compression, device buffers (d_dst must be 4-byte aligned and is cleared). */
int  bz2b200_compress_device(bz2b200_engine* e, const void* d_src, size_t src_len,
                             void* d_dst, size_t dst_cap, size_t* dst_len, unsigned flags,
                             bz2b200_stats* stats);

/* ---- many independent inputs in one call ---------------------------------------------------------
 * Consecutive items are packed into windows; no run, chunk or block crosses from one item into the next, and each
 * item is framed as its own stream.  An item too large for one window goes through the single-stream window loop. */

/* Worst-case size of one stream: the reference's documented BuffToBuff bound (1% + 600 bytes). */
size_t bz2b200_compress_bound(int block_size_100k, size_t n);

/* An engine whose windows can hold up to max_items inputs of a batch (block slots = full blocks of a window +
 * max_items, at most 4096).  Each extra slot costs about hist_stride*4 + 280*nmax/1024 + 25 KB of HBM (~1.3 MB at -9). */
int  bz2b200_engine_create_batch(bz2b200_engine** out, int device, int block_size_100k, size_t window_bytes, size_t max_items);

/* Item k is src[offs[k], offs[k+1]) (offs: host array of n_items+1, non-decreasing, offs[0] = 0).  Each item becomes its
 * own complete .bz2 stream, byte-identical to bz2b200_compress_host(e, item, flags) on that item alone.  The streams are
 * written back to back: stream k is dst[out_offs[k], out_offs[k+1]), so dst[0, out_offs[n]) is a valid multi-stream
 * .bz2 file and out_offs is its index.  stream_crcs (optional, n_items) receives each stream's combined CRC.
 * flags: 0 or BZ2B200_TAIL_STREAMED, applied to every item; NO_HEADER / NO_TRAILER are EPARAM.
 * dst too small: BZ2B200_EOUTFULL, and nothing is written past dst_cap.  Any engine but a bounded one accepts a batch;
 * one from bz2b200_engine_create_batch packs more items per window.  Stats are summed over the call; combined_crc is 0
 * and out_bits is 8 x the bytes written. */
int  bz2b200_compress_batch_host(bz2b200_engine* e, const void* src, const uint64_t* offs, size_t n_items,
                                 void* dst, size_t dst_cap, uint64_t* out_offs, uint32_t* stream_crcs,
                                 unsigned flags, bz2b200_stats* stats);
/* The same with src and dst in device memory (offs, out_offs and stream_crcs stay host arrays; no alignment needed). */
int  bz2b200_compress_batch_device(bz2b200_engine* e, const void* d_src, const uint64_t* offs, size_t n_items,
                                   void* d_dst, size_t dst_cap, uint64_t* out_offs, uint32_t* stream_crcs,
                                   unsigned flags, bz2b200_stats* stats);

/* Streaming: feed input in pieces; compressed bytes are handed to `sink`.
 * end_mode: 0 = more input will follow (BZ_RUN), 1 = flush (BZ_FLUSH: close the open
 * block, no trailer), 2 = finish (BZ_FINISH: trailer + padding). */
typedef int (*bz2b200_sink)(void* user, const void* bytes, size_t n);
int  bz2b200_stream_begin(bz2b200_engine* e);
int  bz2b200_stream_feed(bz2b200_engine* e, const void* src, size_t n, int end_mode,
                         bz2b200_sink sink, void* user);

/* ---- sharding one stream by block over several GPUs (SURVEY 8e) --------------------------------
 * Blocks are independent once their boundaries are known, and boundaries are a greedy chain over
 * the RLE1 chunk structure (bzlib.c:227, :383).  Each GPU scans its shard (plus a halo of the next
 * shard) in parallel; the chain itself is one integer handed from GPU g to GPU g+1.
 *   scan_create   chunk structure of d_src[0,n).  prev_byte / prev_run: the byte before d_src[0]
 *                 and the length of the run it ends (256 / 0 at the start of the stream);
 *                 input_ends: the stream ends at n.
 *   scan_rescan   the same for a new region of at most the size the scan was created for, reusing
 *                 its buffers (a step loop pays no allocation).
 *   scan_boundary first block boundary >= limit when blocks are laid from the boundary `start`;
 *                 also the number of blocks in [start, boundary).
 *   concat_bits   S5: OR `nbits` bits of d_src (from bit 0) into d_dst at bit offset dst_bit.     */
typedef struct bz2b200_scan bz2b200_scan;
int  bz2b200_scan_create(bz2b200_scan** out, int device, int block_size_100k, const void* d_src, size_t n,
                         int prev_byte, uint64_t prev_run, int input_ends);
int  bz2b200_scan_rescan(bz2b200_scan* s, const void* d_src, size_t n, int prev_byte, uint64_t prev_run, int input_ends);
int  bz2b200_scan_boundary(bz2b200_scan* s, size_t start, size_t limit, unsigned flags,
                           size_t* boundary, uint32_t* n_blocks);
void bz2b200_scan_destroy(bz2b200_scan* s);
int  bz2b200_concat_bits(int device, void* d_dst, uint64_t dst_bit, const void* d_src, uint64_t nbits);

/* ---- several engines on one stream (multi.cu) ---------------------------------------------------
 * Consecutive windows (~100 blocks each) of ONE stream go round-robin to n_engines engines, each on
 * its own thread and CUDA stream; devices[k] is the GPU of engine k.  Different GPUs: the stream is
 * sharded by block over them with a host-side gather (SURVEY 8e; replaces nothing in the reference,
 * which is single-threaded -- the unit of work is still BZ2_compressBlock, compress.c:822-881).  The
 * same GPU listed twice: two windows in flight on it.  Windows are chained by two host integers (where
 * the next window starts, bzlib.c:227/:383; at which bit its output starts, compress.c:37-86), every
 * engine copies its own input and writes its own output into the caller's buffer; no collective.
 * The result is byte-identical to bz2b200_compress_host on one engine.
 *   multi_compress   src: host pointer to the whole input -- or NULL with d_srcs[k] = device pointer,
 *                    on engine k's GPU, to a resident copy of the whole input.  dst: host memory,
 *                    *dst_len capacity in / bytes out.  flags: BZ2B200_TAIL_STREAMED.            */
typedef struct bz2b200_multi bz2b200_multi;
int  bz2b200_multi_create(bz2b200_multi** out, const int* devices, int n_engines, int block_size_100k, size_t window_bytes);
void bz2b200_multi_destroy(bz2b200_multi* m);
int  bz2b200_multi_engines(const bz2b200_multi* m);
int  bz2b200_multi_compress(bz2b200_multi* m, const void* src, const void* const* d_srcs, size_t n,
                            void* dst, size_t* dst_len, unsigned flags, bz2b200_stats* stats);

/* Per-stage intermediates of the LAST window processed (tests only).
 * name: "X" "P" "crc" "origptr" "power_q" "inuse" "ninuse" "nmtf" "mtffreq" "bits" "bitoff"
 *       "enc" "bwt" "z" "mtfv" "sa" "sel" "hlen" "ngroups" */
int  bz2b200_debug_keep(bz2b200_engine* e, int on);
int  bz2b200_debug_fetch(bz2b200_engine* e, const char* name, void* dst, size_t cap, size_t* got);

#ifdef __cplusplus
}
#endif
#endif
