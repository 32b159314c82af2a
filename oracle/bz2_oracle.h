/*
 * oracle/bz2_oracle.h -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * A plain-C, single-threaded restatement of the reference's compression path
 * (aeb1787/bzip2: bzlib.c copy_input_until_stop, blocksort.c BZ2_blockSort,
 * compress.c generateMTFValues / sendMTFValues / BZ2_compressBlock,
 * huffman.c BZ2_hbMakeCodeLengths / BZ2_hbAssignCodes).  It exists so the
 * CUDA path can be checked stage by stage on a box that has no /root/reference.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference
 * legs may load this.  The product (libbz2_b200.so) never links or calls it.
 *
 * Parity pin: validated against (a) the reference's own known-answer vectors
 * sample{1,2,3}.ref -> sample{1,2,3}.bz2 (Makefile:58-66) and (b) the reference
 * itself compiled as oracle/_ref/libbz2_ref.so (differential fuzz in
 * tests/test_oracle_vs_ref.py, tests/test_tie_order.py).  On blocks that are an
 * exact power u^q (q >= 2) the reference's origPtr is an artefact of
 * divsufsort's internal order (SURVEY.md section 7 #1); tie_order.c replays the
 * part of the reference's sorter that decides it, so origPtr is exact there too.
 */
#ifndef BZ2_ORACLE_H
#define BZ2_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
   uint64_t in_begin;   /* first input byte covered by this block             */
   uint64_t in_end;     /* one past the last input byte covered               */
   int32_t  nblock;     /* post-RLE1 length                                   */
   uint32_t crc;        /* finalised CRC-32/BZIP2 of in[in_begin, in_end)     */
} orc_block;

/* CRC-32/BZIP2 (crctable.c:29-99, bzlib_private.h:187-202). */
uint32_t orc_crc(const uint8_t* p, uint64_t n);

/* RLE1 block split (bzlib.c:211-315).  tail_merge: the last input byte was
 * consumed in FINISH/FLUSH mode (true for BZ2_bzBuffToBuffCompress). */
int64_t orc_rle1_split(const uint8_t* in, uint64_t n, int level, int tail_merge,
                       orc_block* blocks, int64_t max_blocks);

/* RLE1-encode in[begin,end) from a fresh run state; fills in_use[256]. */
int32_t orc_rle1_emit(const uint8_t* in, uint64_t begin, uint64_t end,
                      uint8_t* out, uint8_t* in_use);

/* Cyclic-rotation BWT (blocksort.c:1534-1545 contract).  Returns the period
 * class count: 1 if all rotations are distinct, q >= 2 if blk == u^q.
 * *orig_ptr is the reference's value in both cases: when q >= 2 it is
 * lo + orc_tie_offset(), lo being the smallest rank among the q equal copies
 * of rotation 0 (SURVEY.md 7#1). */
int32_t orc_bwt(const uint8_t* blk, int32_t n, uint8_t* bwt, int32_t* orig_ptr);

/* Exact power blk = u^q (q >= 2): g in [0,q) with origPtr_ref = lo + g, obtained by replaying the
 * reference's B*-suffix sort (tie_order.c; blocksort.c:1316-1401).  orc_bstar_ranks is the replay
 * itself: work = n + 256 ints, bstar = 65536 ints, T[n] == T[0]; returns the number m of B*
 * suffixes and leaves their ranks in work[m .. 2m). */
int32_t orc_tie_offset(const uint8_t* blk, int32_t n, int32_t q);
int32_t orc_bstar_ranks(const uint8_t* T, int32_t n, int32_t* work, int32_t* bstar);

/* MTF + zero-run coding (compress.c:93-229). Returns nMTF. */
int32_t orc_mtf(const uint8_t* bwt, int32_t n, const uint8_t* in_use,
                uint16_t* mtfv, int32_t* mtf_freq /*258*/, int32_t* n_in_use);

/* huffman.c:63-148 and :152-166 */
void orc_make_code_lengths(int32_t* len, const int32_t* freq, int32_t alpha, int32_t max_len);
void orc_assign_codes(int32_t* code, const int32_t* len, int32_t min_len, int32_t max_len, int32_t alpha);

/* Table selection + emission of one block's coded section (compress.c:250-818),
 * appended MSB-first at bit position *bitpos of out. */
void orc_send_mtf(const uint16_t* mtfv, int32_t n_mtf, const uint8_t* in_use,
                  const int32_t* mtf_freq, uint8_t* out, uint64_t* bitpos);

/* The same computation, returning what it decided instead of the bits: nGroups (the return value), the final
 * selector of every 50-symbol group (sel: (n_mtf + 49) / 50 entries), the final code lengths of every table
 * (len; tables >= nGroups and symbols >= nInUse + 2 are 0), how many times each of the 4 passes halved each
 * table's weights to meet the 17-bit limit, and the bit length of the coded section (symbol map onwards). */
int32_t orc_send_mtf_tables(const uint16_t* mtfv, int32_t n_mtf, const uint8_t* in_use, const int32_t* mtf_freq,
                            uint8_t* sel, int32_t len[6][258], int32_t halvings[4][6], uint64_t* coded_bits);

/* Whole stream (compress.c:822-881 framing).  force_orig_ptr: optional array
 * (one per block, or NULL) overriding origPtr where >= 0 (used to inject the
 * reference's tie-break on exact-power blocks). Returns bytes written or <0. */
int64_t orc_compress(const uint8_t* in, uint64_t n, int level, int tail_merge,
                     const int32_t* force_orig_ptr,
                     uint8_t* out, uint64_t out_cap);

/* Segment form of orc_compress (flags: 2 = no header, 4 = no trailer) and the block-boundary
 * chain, used to check the multi-GPU sharding logic on the CPU. */
int64_t orc_compress_ex(const uint8_t* in, uint64_t n, int level, int tail_merge, unsigned flags,
                        const int32_t* force_orig_ptr, uint8_t* out, uint64_t out_cap,
                        uint64_t* bits_out, uint32_t* fold_out, uint32_t* nblocks_out);
uint64_t orc_find_boundary(const uint8_t* in, uint64_t n, uint64_t start, uint64_t limit, int level,
                           int tail_merge, int input_ends, uint32_t* n_blocks);

#ifdef __cplusplus
}
#endif
#endif
