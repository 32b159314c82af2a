// engine.h -- internal C++ view of the compression engine (one per bz_stream / per GPU).
//
// A "window" is a slice of the input resident in HBM.  One window is cut into
// bzip2 blocks by stage 1 and all of its complete blocks go through stages 2-5
// together, so every kernel launch covers hundreds of blocks.
//
// HBM layout for a window (E = encoded bytes of the window, <= 1.25 * W):
//   enc   u8 [E]    RLE1 output of the whole window; block b is enc[X[b], X[b+1])
//   cend  u8 [E]    1 where an RLE1 chunk ends (block boundaries may only fall there)
//   sa    u32[E]    per block: rotation start indices in sorted order (block-local)
//   rank  u64[E]    per block: group-start rank of each rotation, two generations per word
//   keyA/keyB/idxB  u32[E] scratch for the large-segment radix path
//   bwt   u8 [E]    last column;   z u8[E]  MTF positions;   mtfv u16[E + 2*nb]
//   hist  u32[nb*hist_stride]  k-gram bucket histogram / cursors
#pragma once
#include "common.cuh"

namespace bz {

constexpr int N_SMALL_CLASSES = 5;          // segment lengths 2, 3-4, 5-8, 9-16, 17-32
constexpr int N_BIG_CLASSES = 7;            // u64 worklists
constexpr int CLS_W256 = 5;                 // 33..256    one warp, registers + shuffles
constexpr int CLS_C512 = 6;                 // 257..512   CTA of 64
constexpr int CLS_C1K = 7;                  // 513..1024  CTA of 128
constexpr int CLS_C2K = 8;                  // 1025..2048 CTA of 256
constexpr int CLS_C4K = 9;                  // 2049..4096 CTA of 512
constexpr int CLS_C8K = 10;                 // 4097..8192 CTA of 1024
constexpr int CLS_LARGE = 11;               // > 8192     CTA of 1024, radix passes in HBM
constexpr int N_CLASSES = 12;
constexpr u32 MED_MAX = 8192;
constexpr u32 MAX_BLOCKS = 4096;            // block id must fit 12 bits in a segment entry
constexpr u32 MAX_ENC = 1u << 27;           // flat position must fit 27 bits in a small entry

constexpr int MTF_TILE = 1024;              // symbols per MTF tile (one warp each)

// Segment worklists, double buffered.  Small classes hold u32 entries
// (pos | (len-1) << 27); medium/large hold u64 entries (pos << 32 | blk << 20 | len).
struct SegLists {
   u32* small_items[2][N_SMALL_CLASSES];
   u64* big_items[2][N_BIG_CLASSES];
   u32* counts[2];                          // [N_CLASSES] each, device
   u32  small_cap[N_SMALL_CLASSES];
   u32  big_cap[N_BIG_CLASSES];
};

struct BlockTables {                        // per-window block metadata (device arrays, nb+1 or nb long)
   u32* X;          // [nb+1] encoded start offset of each block
   u32* P;          // [nb+1] input start offset of each block
   u32* crc;        // [nb]   finalised block CRC
   u32* origptr;    // [nb]
   u32* power_q;    // [nb]   0, or q if the block is an exact power u^q
   u32* tie_flag;   // [nb]   1: exact power whose origPtr needs the tie-order replay (stage2_tie.cu)
   u32* tie_lo;     // [nb]   start of rotation 0's tie group (kept only when the replay is forced)
   u8*  inuse;      // [nb*256]
   u32* ninuse;     // [nb]
   u32* nmtf;       // [nb]
   i32* mtffreq;    // [nb*258]
   u32* mtfbase;    // [nb]   start of block's symbols in mtfv (u16 units)
   u64* bits;       // [nb]   total bits of the coded block (header + tables + payload)
   u64* bitoff;     // [nb+1] absolute stream bit offset of each block
};

// Batch windows (batch.cu): many independent inputs packed into one window, each becoming its own stream.
struct ItemTables {                         // device arrays, [blk_cap + 1] or [blk_cap]
   u32* start;      // [n+1] window-relative input start of each item (start[n] = W)
   u32* enc;        // [n]   encoded start of each item
   u32* cnt;        // [n]   blocks of each item
   u32* first;      // [n+1] first block of each item (first[n] = blocks of the window)
   u64* byteoff;    // [n+1] byte offset of each item's stream in the window's output (byteoff[n] = window bytes)
   u32* crc;        // [n]   combined CRC of each item's stream
};

struct Engine;

// One shard's chunk structure for the multi-GPU boundary chain (stage1_rle.cu)
struct ScanState {
   int device; u32 nmax; cudaStream_t st;
   const u8* in; u32 W; u32 input_ends;
   u32 prev_byte, carry0;
   u32 ntiles, enc_total;
   u32 *tile_len, *tile_ext, *tile_carry, *tile_size, *tile_base;
   u8* cend; size_t cend_cap;
   u32* scal;     // [16] device scalars
   u32* q;        // [2] device queries
   u32* h_scal;   // [16] pinned
};
int scan_build(ScanState* s, u32 prev_byte, u32 carry0);
int scan_boundary(ScanState* s, u32 start, u32 limit, u32 tail_merge, u32* boundary, u32* nblocks);

// ---- stage launchers (each returns 0 or a negative error; all work on e->stream) ----
int stage1_run(Engine* e, const u8* d_in, u32 W, bool is_final, bool tail_merge, u32* nb_out, u32* consumed_out, u32* enc_total_out);
int stage1_items_run(Engine* e, const u8* d_in, u32 W, u32 n_items, u32 nb_ub, bool tail_merge,
                     u32* nb_out, u32* enc_total_out, u32* max_blk_out);
int stage2_init();
int stage2_run(Engine* e, u32 nb, u32 E, u32 max_blk = 0);
u32 s2_batch_stride(const Engine* e, u32 max_blk);
int stage2_power_origptr(Engine* e, u32 b0, u32 g);
int stage3_run(Engine* e, u32 nb, u32 E);
// n_items != 0: a batch window; blocks are framed per item (e->it) from bit 0 and origin_bit / start_bit are unused
int stage4_run(Engine* e, u32 nb, u32 E, u8* d_out, u64 origin_bit, u64 start_bit, u64* end_bit_out, u32 n_items = 0);
int stage4_empty_items(Engine* e, u32 n_items, u8* d_out, u64* end_bit_out);
int put_bits_device(Engine* e, u8* d_out, u64 origin_bit, u64 bitpos, u64 value, int nbits);
int concat_bits_device(u8* d_dst, u64 dst_bit, const u8* d_src, u64 nbits);

struct Engine {
   int device;
   int level;
   u32 nmax;               // 100000*level - 19   (bzlib.c:190)
   cudaStream_t stream;
   cudaStream_t own_stream;   // created by the engine; `stream` may be replaced by the caller's
   int num_sms;
   u32 launches;              // kernels launched since the stream was reset
   u32 bwt_rounds;            // prefix-doubling rounds since the stream was reset

   // capacities
   u32 win_cap;            // max input bytes per window
   u32 enc_cap;            // max encoded bytes per window
   u32 blk_cap;            // max blocks per window

   // window buffers
   u8  *enc, *cend;
   u32 *sa, *keyA, *keyB, *idxB;
   u64 *rank;              // [E] tagged rank words (two generations per word)
   u8  *bwt, *z;
   u16 *mtfv;
   u32 *hist;
   u32 s2_group;           // blocks sorted per BWT sub-batch (0 = whole window)
   u32 hist_stride;        // k-gram bins reserved per block (power of two, 2^16..2^18)
   u32 hist_log2;          // the k-gram budget asked for (BZ2_B200_HIST_LOG2, default 18)
   u8  *code;              // [blk_cap*256]
   u32 *kk, *nbins, *hh, *kbits, *ksym;   // [blk_cap]
   u64 *K, *kscrA, *kscrB; // [E] packed text keys; 64-bit key scratch of the large path
   u32 chain;              // follow repeat chains: sort a segment by the rank at the end of its chain (default on)
   u32 chain_min_round;    // first refinement round that may use chains
   cudaStream_t aux[3];    // side streams of the BWT rounds
   cudaEvent_t ev_fork, ev_join[3];
   cudaEvent_t ev_s1, ev_s1b; // stage 1: the scalars of the window have reached the host; the stage is complete
   cudaStream_t s1_stream;    // high-priority stream of stage 1 (set by multi.cu), or null
   u32 hp_late;               // stages 3 and 4 also run on it
   // stage 1 may report the window's consumed bytes before it has finished (fast split of run-free windows, stage1_rle.cu)
   void (*s1_early)(Engine*, u32 consumed);
   bool s1_early_done;
   cudaEvent_t ev_fast;
   u32 *blockmap;          // [enc_cap/4096 + 2] block id of each 4 KiB chunk of enc
   u32 *tie_tmp;           // [blk_cap*256] side buffers of the tie-order replay
   u32 tie_force;          // BZ2_B200_TIE_FORCE=1: replay every exact-power block (tests: closed form == replay)
   SegLists lists;
   BlockTables bt;
   ItemTables it;          // allocated by the first batch call

   // stage-1 tile scratch
   u32 *tile_len, *tile_ext, *tile_carry, *tile_size, *tile_base;
   u32 *s1_scalars;        // [8]: nb, consumed, enc_total, ...

   // stage-3 scratch
   u8  *mtf_summary;       // [tiles*256] recency lists per tile, then start lists
   u32 *mtf_tilemeta;      // [blk_cap*tiles_max*5] lead, trail, inner, out_base | carry
   u32 *mtf_mode;          // [blk_cap] which MTF kernel handles the block
   u32 *mtf_tilecnt;       // [blk_cap*tiles_max] distinct symbols per tile
   // stage-4 scratch
   u8  *sel;               // [E/50 + nb] selectors
   u32 *selbase;           // [nb+1]
   u8  *hlen;              // [nb*6*258] code lengths
   i32 *hfreq;             // [nb*6*258] per-table frequencies
   u32 *hcode;             // [nb*6*258]
   u32 *grpbits;           // [nsel] bits per group, then exclusive offsets
   u8  *pre;               // [nb*PRE_STRIDE] per-block preamble bits
   u32 *prebits;           // [nb]
   u32 *ngroups;           // [nb]

   // device staging for the host API
   u8  *d_in;              // [win_cap + 64]
   u8  *d_out;             // [out_cap]
   size_t out_cap;

   // pinned host mirrors
   u32 *h_scalars;         // [64]
   u32 *h_counts;          // [N_CLASSES]
   u32 *h_blk;             // [blk_cap*4] per-block results (crc, nmtf, power_q, X)
   u32 *h_trace;           // [blk_cap] alphabet sizes for the verbosity >= 3 trace
   int verbosity;          // the reference's trace levels: >= 2 one line per block, >= 3 block statistics (compress.c:831-834, :259-262)
   u32 trace_block0;       // blocks of the stream handled by other engines before this window (multi.cu)
   u8  *h_in;              // [win_cap] pinned staging for streamed input
   u8  *h_out;             // [out_cap] pinned staging for compressed bytes

   char err[256];
};

int engine_fail(Engine* e, cudaError_t c, const char* file, int line);

#define BZ_CUDA(e, call) do { cudaError_t c_ = (call); if (c_ != cudaSuccess) return engine_fail((e), c_, __FILE__, __LINE__); } while (0)
#define BZ_KCHECK(e) do { (e)->launches++; BZ_CUDA(e, cudaGetLastError()); } while (0)

} // namespace bz
