// batch.cu -- many independent inputs in one call, each compressed to its own complete .bz2 stream.
//
// Consecutive items are packed into windows.  Stage 1 runs in its item mode (stage1_items_run): no run, chunk or
// block crosses an item start, so blocks are exactly those of a single-stream call on each item.  Stages 2 and 3 do not
// care which stream a block belongs to; stage 4 frames every item as its own stream (header, its blocks, trailer,
// padding) from bit 0 of the window's output.  Every stream ends on a byte boundary, so a window's output is a whole
// number of bytes and windows carry no bit state.  An item too large for one window takes the single-stream path.
#include "engine_full.h"
#include <stdlib.h>
#include <string.h>

namespace bz {

// block slots an item of n bytes may need: the bound stage1_run sizes its grids by
static u64 item_slots(const EngineFull* e, u64 n) { return (n + n / 4 + 64) / e->nmax + 1; }

static bool item_large(const EngineFull* e, u64 n) { return n > e->win_cap || item_slots(e, n) > e->blk_cap; }

// The next unit of work from item k: one large item (returns false), or the window [k, *k1) (returns true).
// A window closes before the item that would exceed win_cap input bytes or blk_cap block slots.
static bool plan_window(const EngineFull* e, const uint64_t* offs, size_t n_items, size_t k, size_t* k1, u32* slots)
{
   if (item_large(e, offs[k + 1] - offs[k])) { *k1 = k + 1; *slots = 0; return false; }
   u64 W = 0, s = 0;
   size_t j = k;
   while (j < n_items) {
      const u64 len = offs[j + 1] - offs[j];
      if (item_large(e, len) || W + len > e->win_cap || s + item_slots(e, len) > e->blk_cap) break;
      W += len; s += item_slots(e, len); j++;
   }
   *k1 = j; *slots = (u32)s;
   return true;
}

static int ensure_items(EngineFull* e)
{
   if (e->h_items) return 0;
   const size_t n = (size_t)e->blk_cap + 1;
   cudaError_t c = cudaMalloc(reinterpret_cast<void**>(&e->it.start), n * sizeof(u32));
   if (c == cudaSuccess) c = cudaMalloc(reinterpret_cast<void**>(&e->it.enc), n * sizeof(u32));
   if (c == cudaSuccess) c = cudaMalloc(reinterpret_cast<void**>(&e->it.cnt), n * sizeof(u32));
   if (c == cudaSuccess) c = cudaMalloc(reinterpret_cast<void**>(&e->it.first), n * sizeof(u32));
   if (c == cudaSuccess) c = cudaMalloc(reinterpret_cast<void**>(&e->it.byteoff), n * sizeof(u64));
   if (c == cudaSuccess) c = cudaMalloc(reinterpret_cast<void**>(&e->it.crc), n * sizeof(u32));
   if (c == cudaSuccess) c = cudaMallocHost(reinterpret_cast<void**>(&e->h_items), 5 * n * sizeof(u32));
   if (c != cudaSuccess) return engine_fail(e, c, __FILE__, __LINE__);
   return 0;
}

// pinned host mirrors of the item tables: byte offsets (u64) first, then starts, first blocks and CRCs
static u64* h_byteoff(EngineFull* e) { return reinterpret_cast<u64*>(e->h_items); }
static u32* h_start(EngineFull* e) { return e->h_items + 2 * ((size_t)e->blk_cap + 1); }
static u32* h_first(EngineFull* e) { return e->h_items + 3 * ((size_t)e->blk_cap + 1); }
static u32* h_icrc(EngineFull* e) { return e->h_items + 4 * ((size_t)e->blk_cap + 1); }

static void stats_add(bz2b200_stats& a, const bz2b200_stats& b)
{
   a.n_blocks += b.n_blocks; a.n_windows += b.n_windows;
   a.sum_nblock += b.sum_nblock; a.sum_nmtf += b.sum_nmtf; a.n_power_blocks += b.n_power_blocks;
   a.ms_total += b.ms_total; a.ms_s1 += b.ms_s1; a.ms_s2 += b.ms_s2; a.ms_s3 += b.ms_s3; a.ms_s4 += b.ms_s4;
   a.bwt_rounds += b.bwt_rounds; a.kernel_launches += b.kernel_launches;
}

// One batch window: items [k0, k1), whose input is d_in[0, offs[k1] - offs[k0]).  Their streams are written back to
// back from bit 0 of e->d_out; h_byteoff(e)[0..n] and h_icrc(e)[0..n) receive their offsets and combined CRCs.
static int batch_window(EngineFull* e, const u8* d_in, const uint64_t* offs, size_t k0, size_t k1, u32 slots,
                        bool tail_merge, bz2b200_stats& acc)
{
   cudaStream_t st = e->stream;
   const u32 n = (u32)(k1 - k0);
   const u32 W = (u32)(offs[k1] - offs[k0]);
   const u32 launches0 = e->launches, rounds0 = e->bwt_rounds;
   u32* hs = h_start(e);
   for (u32 i = 0; i <= n; i++) hs[i] = (u32)(offs[k0 + i] - offs[k0]);
   cudaEventRecord(e->ev[0], st);
   BZ_CUDA(e, cudaMemcpyAsync(e->it.start, hs, sizeof(u32) * (n + 1), cudaMemcpyHostToDevice, st));
   u32 nb = 0, E = 0, max_blk = 0;
   int rc = 0;
   if (W) rc = stage1_items_run(e, d_in, W, n, slots, tail_merge, &nb, &E, &max_blk);
   else BZ_CUDA(e, cudaMemsetAsync(e->it.first, 0, sizeof(u32) * (n + 1), st));     // only empty items: no blocks
   if (rc) { set_err_text(e->err); return rc; }
   cudaEventRecord(e->ev[1], st);
   e->last_nb = nb; e->last_E = E;
   // what the window can write: the blocks' bound of the single-stream path plus header, trailer and padding per item
   size_t clear = (size_t)E + E / 32 + (size_t)nb * 24576 + 16 * (size_t)n + 4096;
   if (clear > e->out_cap) clear = e->out_cap;
   BZ_CUDA(e, cudaMemsetAsync(e->d_out, 0, clear, st));
   u64 end_bit = 0;
   if (nb) {
      if ((rc = stage2_run(e, nb, E, max_blk))) { set_err_text(e->err); return rc; }
      cudaEventRecord(e->ev[2], st);
      if ((rc = stage3_run(e, nb, E))) { set_err_text(e->err); return rc; }
      cudaEventRecord(e->ev[3], st);
      if ((rc = stage4_run(e, nb, E, e->d_out, 0, 0, &end_bit, n))) { set_err_text(e->err); return rc; }
   } else {
      cudaEventRecord(e->ev[2], st);
      cudaEventRecord(e->ev[3], st);
      if ((rc = stage4_empty_items(e, n, e->d_out, &end_bit))) { set_err_text(e->err); return rc; }
   }
   cudaEventRecord(e->ev[4], st);
   if ((end_bit >> 3) > clear) return set_err(BZ2B200_EINTERNAL, "batch window output exceeds its staging bound");
   // per-block results for the statistics and the trace, per-item results for the index
   if (nb) {
      BZ_CUDA(e, cudaMemcpyAsync(e->h_blk, e->bt.crc, sizeof(u32) * nb, cudaMemcpyDeviceToHost, st));
      BZ_CUDA(e, cudaMemcpyAsync(e->h_blk + e->blk_cap, e->bt.nmtf, sizeof(u32) * nb, cudaMemcpyDeviceToHost, st));
      BZ_CUDA(e, cudaMemcpyAsync(e->h_blk + 2 * (size_t)e->blk_cap, e->bt.power_q, sizeof(u32) * nb, cudaMemcpyDeviceToHost, st));
      if (e->verbosity >= 2) {
         BZ_CUDA(e, cudaMemcpyAsync(e->h_blk + 3 * (size_t)e->blk_cap, e->bt.X, sizeof(u32) * (nb + 1), cudaMemcpyDeviceToHost, st));
         BZ_CUDA(e, cudaMemcpyAsync(e->h_trace, e->bt.ninuse, sizeof(u32) * nb, cudaMemcpyDeviceToHost, st));
      }
   }
   BZ_CUDA(e, cudaMemcpyAsync(h_first(e), e->it.first, sizeof(u32) * (n + 1), cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaMemcpyAsync(h_icrc(e), e->it.crc, sizeof(u32) * n, cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaMemcpyAsync(h_byteoff(e), e->it.byteoff, sizeof(u64) * (n + 1), cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaStreamSynchronize(st));
   const u32* first = h_first(e);
   for (u32 b = 0; b < nb; b++) {
      acc.sum_nmtf += e->h_blk[e->blk_cap + b];
      if (e->h_blk[2 * (size_t)e->blk_cap + b]) acc.n_power_blocks++;
   }
   if (e->verbosity >= 2) {
      // the text of one single-stream call per item: block numbers restart, every item has its final CRC line
      const u32* X = e->h_blk + 3 * (size_t)e->blk_cap;
      for (u32 i = 0; i < n; i++) {
         u32 c = 0;
         for (u32 b = first[i]; b < first[i + 1]; b++) {
            c = ((c << 1) | (c >> 31)) ^ e->h_blk[b];
            fprintf(stderr, "    block %d: crc = 0x%08x, combined CRC = 0x%08x, size = %d\n",
                    (int)(b - first[i] + 1), e->h_blk[b], c, (int)(X[b + 1] - X[b]));
            if (e->verbosity >= 3)
               fprintf(stderr, "      %d in block, %d after MTF & 1-2 coding, %d+2 syms in use\n",
                       (int)(X[b + 1] - X[b]), (int)e->h_blk[e->blk_cap + b], (int)e->h_trace[b]);
         }
         fprintf(stderr, "    final combined CRC = 0x%08x\n   ", c);
      }
   }
   acc.n_blocks += nb; acc.n_windows++; acc.sum_nblock += E;
   acc.kernel_launches += e->launches - launches0;
   acc.bwt_rounds += e->bwt_rounds - rounds0;
   float ms;
   cudaEventElapsedTime(&ms, e->ev[0], e->ev[1]); acc.ms_s1 += ms;
   cudaEventElapsedTime(&ms, e->ev[1], e->ev[2]); acc.ms_s2 += ms;
   cudaEventElapsedTime(&ms, e->ev[2], e->ev[3]); acc.ms_s3 += ms;
   cudaEventElapsedTime(&ms, e->ev[3], e->ev[4]); acc.ms_s4 += ms;
   cudaEventElapsedTime(&ms, e->ev[0], e->ev[4]); acc.ms_total += ms;
   return 0;
}

static int batch_call(bz2b200_engine* h, const void* src, bool dev_src, const uint64_t* offs, size_t n_items,
                      void* dst, bool dev_dst, size_t dst_cap, uint64_t* out_offs, uint32_t* stream_crcs,
                      unsigned flags, bz2b200_stats* stats)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e || !offs || !out_offs) return set_err(BZ2B200_EPARAM, "bad argument");
   if (flags & ~BZ2B200_TAIL_STREAMED) return set_err(BZ2B200_EPARAM, "a batch call takes no flag but BZ2B200_TAIL_STREAMED");
   if (offs[0] != 0) return set_err(BZ2B200_EPARAM, "offs[0] must be 0");
   for (size_t k = 0; k < n_items; k++) if (offs[k + 1] < offs[k]) return set_err(BZ2B200_EPARAM, "offs must not decrease");
   if ((!src && offs[n_items]) || (!dst && n_items)) return set_err(BZ2B200_EPARAM, "bad argument");
   if (e->bounded) return set_err(BZ2B200_EPARAM, "a bounded engine serves single-input calls only");
   const u8* in = static_cast<const u8*>(src);
   u8* out = static_cast<u8*>(dst);
   bz2b200_stats acc;
   memset(&acc, 0, sizeof acc);
   out_offs[0] = 0;
   if (n_items == 0) { if (stats) *stats = acc; return 0; }
   DeviceGuard guard(e->device);
   int rc = ensure_staging(e, false);
   if (rc) return rc;
   if ((rc = ensure_items(e))) return rc;
   feed_reset(e);
   stream_reset(e);
   e->after_s1 = nullptr;
   const bool tail_merge = !(flags & BZ2B200_TAIL_STREAMED);
   // host input from pinned memory: the next window's H2D runs on the copy stream while this window is compressed
   bool pinned = false;
   if (!dev_src && offs[n_items]) {
      cudaPointerAttributes at;
      if (cudaPointerGetAttributes(&at, src) == cudaSuccess) pinned = (at.type == cudaMemoryTypeHost);
      else cudaGetLastError();
   }
   u8* dbuf[2] = { e->d_in, e->d_in2 };
   int cur = 0;
   bool prefetched = false;
   struct BigBuf { u8* p = nullptr; size_t cap = 0; ~BigBuf() { if (p) cudaFree(p); } } big;   // device calls: a large item's stream
   size_t pos = 0, k = 0;
   while (k < n_items) {
      size_t k1 = 0; u32 slots = 0;
      if (!plan_window(e, offs, n_items, k, &k1, &slots)) {
         // an item larger than a window: the single-stream window loop, its stream placed at out_offs[k]
         const u64 len = offs[k + 1] - offs[k];
         bz2b200_stats s1;
         size_t got = 0;
         if (!dev_dst) {
            got = dst_cap - pos;
            rc = bz2b200_compress_host(h, in + offs[k], len, out + pos, &got, flags, &s1);
            if (rc) break;
         } else {
            const size_t need = len + len / 64 + (len / e->nmax + 2) * 24576 + 64;
            if (need > big.cap) {
               if (big.p) cudaFree(big.p);
               big.p = nullptr; big.cap = 0;
               cudaError_t c = cudaMalloc(reinterpret_cast<void**>(&big.p), need);
               if (c != cudaSuccess) { rc = engine_fail(e, c, __FILE__, __LINE__); break; }
               big.cap = need;
            }
            rc = bz2b200_compress_device(h, in + offs[k], len, big.p, big.cap, &got, flags, &s1);
            if (rc) break;
            if (got > dst_cap - pos) { rc = set_err(BZ2B200_EOUTFULL, "batch destination too small"); break; }
            cudaError_t c = cudaMemcpyAsync(out + pos, big.p, got, cudaMemcpyDeviceToDevice, e->stream);
            if (c == cudaSuccess) c = cudaStreamSynchronize(e->stream);
            if (c != cudaSuccess) { rc = engine_fail(e, c, __FILE__, __LINE__); break; }
            if (e->verbosity >= 2) fprintf(stderr, "    final combined CRC = 0x%08x\n   ", s1.combined_crc);   // as the host call
         }
         stats_add(acc, s1);
         if (stream_crcs) stream_crcs[k] = s1.combined_crc;
         pos += got;
         out_offs[k + 1] = pos;
         k = k1;
         continue;
      }
      const size_t W = (size_t)(offs[k1] - offs[k]);
      const u8* d_in = nullptr;
      if (dev_src) d_in = in + offs[k];
      else {
         d_in = dbuf[cur];
         if (prefetched) BZ_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_h2d[cur], 0));
         else if (W) BZ_CUDA(e, cudaMemcpyAsync(dbuf[cur], in + offs[k], W, cudaMemcpyHostToDevice, e->stream));
         prefetched = false;
         size_t k2 = 0; u32 s2 = 0;
         if (pinned && k1 < n_items && plan_window(e, offs, n_items, k1, &k2, &s2) && offs[k2] > offs[k1]) {
            BZ_CUDA(e, cudaMemcpyAsync(dbuf[cur ^ 1], in + offs[k1], (size_t)(offs[k2] - offs[k1]), cudaMemcpyHostToDevice, e->copy_stream));
            BZ_CUDA(e, cudaEventRecord(e->ev_h2d[cur ^ 1], e->copy_stream));
            prefetched = true;
         }
      }
      rc = batch_window(e, d_in, offs, k, k1, slots, tail_merge, acc);
      if (rc) break;
      const u64* boff = h_byteoff(e);
      const size_t nbytes = (size_t)boff[k1 - k];
      if (nbytes > dst_cap - pos) { rc = set_err(BZ2B200_EOUTFULL, "batch destination too small"); break; }
      BZ_CUDA(e, cudaMemcpyAsync(out + pos, e->d_out, nbytes, dev_dst ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, e->stream));
      BZ_CUDA(e, cudaStreamSynchronize(e->stream));
      for (size_t i = k; i < k1; i++) {
         out_offs[i + 1] = pos + boff[i + 1 - k];
         if (stream_crcs) stream_crcs[i] = h_icrc(e)[i - k];
      }
      pos += nbytes;
      if (prefetched) cur ^= 1;
      k = k1;
   }
   if (prefetched) cudaStreamSynchronize(e->copy_stream);
   if (rc) return rc;
   acc.in_bytes = offs[n_items]; acc.out_bytes = pos; acc.out_bits = (u64)pos * 8; acc.combined_crc = 0;
   if (stats) *stats = acc;
   return 0;
}

} // namespace bz

using namespace bz;

extern "C" {

size_t bz2b200_compress_bound(int block_size_100k, size_t n)
{
   if (block_size_100k < 1 || block_size_100k > 9) return 0;
   return n + (n + 99) / 100 + 600;
}

int bz2b200_engine_create_batch(bz2b200_engine** out, int device, int block_size_100k, size_t window_bytes, size_t max_items)
{
   if (!out) return set_err(BZ2B200_EPARAM, "null out pointer");
   int prev = -1;
   cudaGetDevice(&prev);
   EngineFull* e = nullptr;
   int rc = engine_new(&e, device, block_size_100k, window_bytes, false, max_items);
   if (prev >= 0) cudaSetDevice(prev);
   if (rc) return rc;
   stream_reset(e);
   *out = reinterpret_cast<bz2b200_engine*>(e);
   return 0;
}

int bz2b200_compress_batch_host(bz2b200_engine* e, const void* src, const uint64_t* offs, size_t n_items,
                                void* dst, size_t dst_cap, uint64_t* out_offs, uint32_t* stream_crcs,
                                unsigned flags, bz2b200_stats* stats)
{
   return batch_call(e, src, false, offs, n_items, dst, false, dst_cap, out_offs, stream_crcs, flags, stats);
}

int bz2b200_compress_batch_device(bz2b200_engine* e, const void* d_src, const uint64_t* offs, size_t n_items,
                                  void* d_dst, size_t dst_cap, uint64_t* out_offs, uint32_t* stream_crcs,
                                  unsigned flags, bz2b200_stats* stats)
{
   return batch_call(e, d_src, true, offs, n_items, d_dst, true, dst_cap, out_offs, stream_crcs, flags, stats);
}

} // extern "C"
