// engine.cu -- window orchestration and the C ABI declared in include/bz2_b200.h.
//
// Host-side driver of the five stages.  The path it replaces in the reference is
// handle_compress (bzlib.c:361-396) looping copy_input_until_stop + BZ2_compressBlock
// one 900 kB block at a time; here a window of up to ~100 blocks is taken through each
// stage with one set of kernel launches.
#include "engine_full.h"
#include <stdlib.h>
#include <string.h>
#include <new>
#include <pthread.h>

namespace bz {

static thread_local char g_err[256] = "";

int engine_fail(Engine* e, cudaError_t c, const char* file, int line)
{
   const char* base = strrchr(file, '/');
   snprintf(g_err, sizeof g_err, "CUDA error %d (%s) at %s:%d", (int)c, cudaGetErrorString(c), base ? base + 1 : file, line);
   if (e) snprintf(e->err, sizeof e->err, "%s", g_err);
   return BZ2B200_ECUDA;
}

void set_err_text(const char* msg) { snprintf(g_err, sizeof g_err, "%s", msg); }

int set_err(int code, const char* msg)
{
   snprintf(g_err, sizeof g_err, "%s", msg);
   return code;
}

template <typename T>
static cudaError_t dalloc(T** p, size_t count)
{
   return cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T));
}

#define ALLOC(ptr, count) do { cudaError_t c_ = dalloc(&(ptr), (size_t)(count)); if (c_ != cudaSuccess) { rc = engine_fail(e, c_, __FILE__, __LINE__); goto fail; } } while (0)

static void feed_shutdown(EngineFull* e);

void engine_free(EngineFull* e)
{
   if (!e) return;
   feed_shutdown(e);
   cudaSetDevice(e->device);
   void* dev[] = { e->enc, e->cend, e->sa, e->rank, e->keyA, e->keyB, e->idxB, e->bwt, e->z, e->mtfv, e->hist,
                   e->blockmap, e->code, e->kk, e->nbins, e->hh, e->kbits, e->ksym, e->K, e->kscrA, e->kscrB, e->tile_len, e->tile_ext, e->tile_carry, e->tile_size, e->tile_base, e->s1_scalars,
                   e->mtf_summary, e->mtf_tilemeta, e->mtf_tilecnt, e->mtf_mode, e->sel, e->hlen, e->hfreq, e->hcode, e->grpbits,
                   e->pre, e->prebits, e->ngroups, e->d_in, e->d_out,
                   e->bt.X, e->bt.P, e->bt.crc, e->bt.origptr, e->bt.power_q, e->bt.inuse, e->bt.ninuse, e->bt.nmtf,
                   e->bt.mtffreq, e->bt.bits, e->bt.bitoff, e->lists.counts[0], e->lists.counts[1],
                   e->tie_tmp, e->bt.tie_flag, e->bt.tie_lo,
                   e->it.start, e->it.enc, e->it.cnt, e->it.first, e->it.byteoff, e->it.crc };
   for (void* p : dev) if (p) cudaFree(p);
   for (int w = 0; w < 2; w++) {
      for (int c = 0; c < N_SMALL_CLASSES; c++) if (e->lists.small_items[w][c]) cudaFree(e->lists.small_items[w][c]);
      for (int c = 0; c < N_BIG_CLASSES; c++) if (e->lists.big_items[w][c]) cudaFree(e->lists.big_items[w][c]);
   }
   if (e->h_scalars) cudaFreeHost(e->h_scalars);
   if (e->h_counts) cudaFreeHost(e->h_counts);
   if (e->h_blk) cudaFreeHost(e->h_blk);
   if (e->h_trace) cudaFreeHost(e->h_trace);
   if (e->h_items) cudaFreeHost(e->h_items);
   if (e->h_in) cudaFreeHost(e->h_in);
   if (e->h_out) cudaFreeHost(e->h_out);
   if (e->d_in2) cudaFree(e->d_in2);
   if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
   for (int i = 0; i < 2; i++) if (e->ev_h2d[i]) cudaEventDestroy(e->ev_h2d[i]);
   for (int i = 0; i < 6; i++) if (e->ev[i]) cudaEventDestroy(e->ev[i]);
   for (int i = 0; i < 3; i++) { if (e->aux[i]) cudaStreamDestroy(e->aux[i]); if (e->ev_join[i]) cudaEventDestroy(e->ev_join[i]); }
   if (e->ev_fork) cudaEventDestroy(e->ev_fork);
   if (e->own_stream) cudaStreamDestroy(e->own_stream);
   free(e);
}

int engine_new(EngineFull** out, int device, int level, size_t window_bytes, bool bounded, size_t extra_slots)
{
   int ndev = 0;
   cudaError_t ce = cudaGetDeviceCount(&ndev);
   if (ce != cudaSuccess || ndev == 0) return set_err(BZ2B200_ENODEV, "no CUDA device available (this library has no CPU path)");
   if (device < 0 || device >= ndev) return set_err(BZ2B200_EPARAM, "bad device index");
   if (level < 1 || level > 9) return set_err(BZ2B200_EPARAM, "block_size_100k must be 1..9");
   EngineFull* e = static_cast<EngineFull*>(calloc(1, sizeof(EngineFull)));
   if (!e) return set_err(BZ2B200_ENOMEM, "out of host memory");
   int rc = 0;
   e->device = device; e->level = level; e->nmax = 100000u * (u32)level - 19u;
   if (cudaSetDevice(device) != cudaSuccess) { free(e); return set_err(BZ2B200_ENODEV, "cudaSetDevice failed"); }
   {
      cudaDeviceProp prop;
      cudaGetDeviceProperties(&prop, device);
      e->num_sms = prop.multiProcessorCount;
   }
   {
      const char* g = getenv("BZ2_B200_S2_GROUP");
      e->s2_group = g ? (u32)atoi(g) : 0;
      const char* ch = getenv("BZ2_B200_CHAIN");
      e->chain = ch ? (u32)atoi(ch) : 1;
      const char* tf2 = getenv("BZ2_B200_TIE_FORCE");
      e->tie_force = tf2 ? (u32)atoi(tf2) : 0;
      const char* cr = getenv("BZ2_B200_CHAIN_MIN_ROUND");
      e->chain_min_round = cr ? (u32)atoi(cr) : 2;
   }
   if (window_bytes == 0) window_bytes = (size_t)96 << 20;
   // a window must be able to hold the input of one full block of pure runs (255 -> 5 bytes)
   // ... unless the caller bounds the whole input (one-shot calls on small inputs): then the input itself is the window
   const size_t min_win = bounded ? ((size_t)64 << 10) : (size_t)(e->nmax + 16) * 52;
   e->bounded = bounded;
   if (window_bytes < min_win) window_bytes = min_win;
   if (window_bytes > ((size_t)100 << 20)) window_bytes = (size_t)100 << 20;   // 1.25*W must stay below 2^27
   e->win_cap = (u32)window_bytes;
   e->enc_cap = (u32)(window_bytes + window_bytes / 4 + 4096);
   e->blk_cap = e->enc_cap / e->nmax + 2;
   // batch engines: one slot more per item a window may hold (every item, however small, ends its own block)
   e->blk_cap = (u32)((size_t)e->blk_cap + (extra_slots < MAX_BLOCKS ? extra_slots : MAX_BLOCKS));
   if (e->blk_cap > MAX_BLOCKS) e->blk_cap = MAX_BLOCKS;
   {
      const size_t E = e->enc_cap, B = e->blk_cap;
      const size_t tiles_max = (e->nmax + 16 + MTF_TILE - 1) / MTF_TILE;
      const size_t ntiles = window_bytes / 4096 + 4;
      cudaError_t c0 = cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking);
      if (c0 != cudaSuccess) { rc = engine_fail(e, c0, __FILE__, __LINE__); goto fail; }
      e->stream = e->own_stream;
      for (int i = 0; i < 6; i++) cudaEventCreate(&e->ev[i]);
      for (int i = 0; i < 3; i++) {
         c0 = cudaStreamCreateWithFlags(&e->aux[i], cudaStreamNonBlocking);
         if (c0 == cudaSuccess) c0 = cudaEventCreateWithFlags(&e->ev_join[i], cudaEventDisableTiming);
         if (c0 != cudaSuccess) { rc = engine_fail(e, c0, __FILE__, __LINE__); goto fail; }
      }
      if (stage2_init() != 0) { rc = engine_fail(e, cudaGetLastError(), __FILE__, __LINE__); goto fail; }
      c0 = cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming);
      if (c0 == cudaSuccess) c0 = cudaEventCreateWithFlags(&e->ev_s1, cudaEventDisableTiming);
      if (c0 == cudaSuccess) c0 = cudaEventCreateWithFlags(&e->ev_s1b, cudaEventDisableTiming);
      if (c0 == cudaSuccess) c0 = cudaEventCreateWithFlags(&e->ev_fast, cudaEventDisableTiming);
      if (c0 != cudaSuccess) { rc = engine_fail(e, c0, __FILE__, __LINE__); goto fail; }
      ALLOC(e->enc, E + 64); ALLOC(e->cend, E + 64);
      ALLOC(e->sa, E + 64); ALLOC(e->rank, E + 64);
      ALLOC(e->keyA, E + 64); ALLOC(e->keyB, E + 64); ALLOC(e->idxB, E + 64);
      ALLOC(e->bwt, E + 64); ALLOC(e->z, E + 64); ALLOC(e->mtfv, E + B + 64);
      u32 hist_log2 = 18;
      { const char* hl = getenv("BZ2_B200_HIST_LOG2"); if (hl) { const int v = atoi(hl); if (v >= 16 && v <= 22) hist_log2 = (u32)v; } }
      e->hist_log2 = hist_log2;
      e->hist_stride = 1u << 16;
      while (e->hist_stride < (1u << hist_log2) && e->hist_stride < e->nmax / 4) e->hist_stride <<= 1;
      if (hist_log2 > 18 && e->hist_stride < e->nmax * 2u) e->hist_stride = 1u << hist_log2;
      ALLOC(e->hist, B * e->hist_stride);
      ALLOC(e->code, B * 256); ALLOC(e->kk, B); ALLOC(e->nbins, B); ALLOC(e->hh, B); ALLOC(e->kbits, B); ALLOC(e->ksym, B);
      ALLOC(e->K, E + 64); ALLOC(e->kscrA, E + 64); ALLOC(e->kscrB, E + 64);
      ALLOC(e->blockmap, E / 4096 + 4);
      ALLOC(e->tie_tmp, B * 256); ALLOC(e->bt.tie_flag, B); ALLOC(e->bt.tie_lo, B);
      ALLOC(e->tile_len, ntiles); ALLOC(e->tile_ext, ntiles); ALLOC(e->tile_carry, ntiles);
      ALLOC(e->tile_size, ntiles); ALLOC(e->tile_base, ntiles);
      ALLOC(e->s1_scalars, 16);
      ALLOC(e->mtf_summary, B * tiles_max * 256);
      ALLOC(e->mtf_tilemeta, B * tiles_max * 5);
      ALLOC(e->mtf_tilecnt, B * tiles_max); ALLOC(e->mtf_mode, B);
      ALLOC(e->sel, E / 50 + 2 * B + 64);
      ALLOC(e->grpbits, E / 50 + 2 * B + 64);
      ALLOC(e->hlen, B * 6 * BZ_MAX_ALPHA); ALLOC(e->hfreq, B * 6 * BZ_MAX_ALPHA); ALLOC(e->hcode, B * 6 * BZ_MAX_ALPHA);
      ALLOC(e->pre, B * 24576); ALLOC(e->prebits, B); ALLOC(e->ngroups, B);
      ALLOC(e->bt.X, B + 2); ALLOC(e->bt.P, B + 2); ALLOC(e->bt.crc, B); ALLOC(e->bt.origptr, B); ALLOC(e->bt.power_q, B);
      ALLOC(e->bt.inuse, B * 256); ALLOC(e->bt.ninuse, B); ALLOC(e->bt.nmtf, B); ALLOC(e->bt.mtffreq, B * BZ_MAX_ALPHA);
      ALLOC(e->bt.bits, B); ALLOC(e->bt.bitoff, B + 2);
      static const u32 minlen[N_SMALL_CLASSES] = {2, 3, 5, 9, 17};
      for (int c = 0; c < N_SMALL_CLASSES; c++) e->lists.small_cap[c] = (u32)(E / minlen[c] + 1024);
      static const u32 bigmin[N_BIG_CLASSES] = {33, 257, 513, 1025, 2049, 4097, 8193};
      for (int c = 0; c < N_BIG_CLASSES; c++) e->lists.big_cap[c] = (u32)(E / bigmin[c] + 1024);
      for (int w = 0; w < 2; w++) {
         for (int c = 0; c < N_SMALL_CLASSES; c++) ALLOC(e->lists.small_items[w][c], e->lists.small_cap[c]);
         for (int c = 0; c < N_BIG_CLASSES; c++) ALLOC(e->lists.big_items[w][c], e->lists.big_cap[c]);
         ALLOC(e->lists.counts[w], N_CLASSES);
      }
      e->out_cap = E + E / 32 + B * 24576 + 4096;
      e->out_cap = (e->out_cap + 255) & ~(size_t)255;
      // device/host staging is allocated lazily by the host and stream paths
   }
   {
      cudaError_t c1 = cudaMallocHost(reinterpret_cast<void**>(&e->h_scalars), 64 * sizeof(u32));
      cudaError_t c2 = cudaMallocHost(reinterpret_cast<void**>(&e->h_counts), 32 * sizeof(u32));
      cudaError_t c3 = cudaMallocHost(reinterpret_cast<void**>(&e->h_blk), (size_t)e->blk_cap * 4 * sizeof(u32) + 64);
      if (c3 == cudaSuccess) c3 = cudaMallocHost(reinterpret_cast<void**>(&e->h_trace), (size_t)e->blk_cap * sizeof(u32) + 64);
      if (c1 != cudaSuccess || c2 != cudaSuccess || c3 != cudaSuccess) { rc = set_err(BZ2B200_ENOMEM, "pinned host allocation failed"); goto fail; }
   }
   *out = e;
   return 0;
fail:
   engine_free(e);
   return rc ? rc : BZ2B200_ENOMEM;
}

int ensure_staging(EngineFull* e, bool need_hin)
{
   if (!e->d_in)  { cudaError_t c = cudaMalloc(reinterpret_cast<void**>(&e->d_in), (size_t)e->win_cap + 64); if (c != cudaSuccess) return engine_fail(e, c, __FILE__, __LINE__); }
   if (!e->d_out) { cudaError_t c = cudaMalloc(reinterpret_cast<void**>(&e->d_out), e->out_cap); if (c != cudaSuccess) return engine_fail(e, c, __FILE__, __LINE__); }
   if (!e->h_out) { cudaError_t c = cudaMallocHost(reinterpret_cast<void**>(&e->h_out), e->out_cap); if (c != cudaSuccess) return engine_fail(e, c, __FILE__, __LINE__); }
   if (!e->d_in2) { cudaError_t c = cudaMalloc(reinterpret_cast<void**>(&e->d_in2), (size_t)e->win_cap + 64); if (c != cudaSuccess) return engine_fail(e, c, __FILE__, __LINE__); }
   if (!e->copy_stream) {
      cudaError_t c = cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking);
      if (c != cudaSuccess) return engine_fail(e, c, __FILE__, __LINE__);
      for (int i = 0; i < 2; i++) cudaEventCreateWithFlags(&e->ev_h2d[i], cudaEventDisableTiming);
   }
   if (need_hin && !e->h_in) {
      e->af.cap = (size_t)e->win_cap + (size_t)e->win_cap / 2;
      cudaError_t c = cudaMallocHost(reinterpret_cast<void**>(&e->h_in), e->af.cap);
      if (c != cudaSuccess) return engine_fail(e, c, __FILE__, __LINE__);
   }
   return 0;
}

void stream_reset(EngineFull* e)
{
   memset(&e->ss, 0, sizeof e->ss);
   e->launches = 0;
   e->bwt_rounds = 0;
}

// One window through all stages.  d_in: device input; writes coded blocks into d_out at
// their absolute bit positions (relative to origin_bit) and advances ss.bits.
static void s1_early_trampoline(Engine* b, u32 consumed)
{
   EngineFull* f = static_cast<EngineFull*>(b);
   f->after_s1(f, consumed, f->after_s1_ctx);
}

int run_window(EngineFull* e, const u8* d_in, u32 W, bool is_final, bool tail_merge,
                      u8* d_out, u64 origin_bit, u32* consumed, u32* nb_out)
{
   cudaStream_t st = e->stream;
   u32 nb = 0, cons = 0, E = 0;
   StreamState& ss = e->ss;
   cudaEventRecord(e->ev[0], st);
   // several engines on one stream of data: stage 1 may hand the window's end to the next engine before it is done
   e->s1_early_done = false;
   e->s1_early = (e->after_s1 && e->s1_stream) ? s1_early_trampoline : nullptr;
   int rc = stage1_run(e, d_in, W, is_final, tail_merge, &nb, &cons, &E);
   e->s1_early = nullptr;
   if (rc) { snprintf(g_err, sizeof g_err, "%s", e->err); return rc; }
   cudaEventRecord(e->ev[1], st);
   if (e->after_s1 && !e->s1_early_done) e->after_s1(e, cons, e->after_s1_ctx);
   *consumed = cons; *nb_out = nb;
   e->last_nb = nb; e->last_E = E;
   if (nb == 0) return 0;
   rc = stage2_run(e, nb, E);
   if (rc) { snprintf(g_err, sizeof g_err, "%s", e->err); return rc; }
   cudaEventRecord(e->ev[2], st);
   // With several windows in flight on this GPU (multi.cu) the thin, latency-bound stages 3 and 4 also go to the engine's
   // high-priority stream: their CTAs are scheduled ahead of the register-hungry sort CTAs of the other windows instead
   // of waiting for a whole grid of them to drain, and the window leaves the GPU sooner.
   cudaStream_t hp = (e->s1_stream && e->hp_late) ? e->s1_stream : nullptr;
   if (hp) {
      BZ_CUDA(e, cudaStreamWaitEvent(hp, e->ev[2], 0));
      e->stream = hp;
   }
   rc = stage3_run(e, nb, E);
   if (rc) { e->stream = st; snprintf(g_err, sizeof g_err, "%s", e->err); return rc; }
   cudaEventRecord(e->ev[3], e->stream);
   u64 end_bit = 0;
   rc = stage4_run(e, nb, E, d_out, origin_bit, ss.bits, &end_bit);
   e->stream = st;
   if (rc) { snprintf(g_err, sizeof g_err, "%s", e->err); return rc; }
   cudaEventRecord(e->ev[4], hp ? hp : st);
   if (hp) BZ_CUDA(e, cudaStreamWaitEvent(st, e->ev[4], 0));
   // per-block results for the combined CRC and the statistics
   BZ_CUDA(e, cudaMemcpyAsync(e->h_blk, e->bt.crc, sizeof(u32) * nb, cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaMemcpyAsync(e->h_blk + e->blk_cap, e->bt.nmtf, sizeof(u32) * nb, cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaMemcpyAsync(e->h_blk + 2 * (size_t)e->blk_cap, e->bt.power_q, sizeof(u32) * nb, cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaStreamSynchronize(st));
   if (e->verbosity >= 2) {
      // the block sizes and alphabet sizes for the per-block trace lines (compress.c:831-834, :259-262)
      BZ_CUDA(e, cudaMemcpyAsync(e->h_blk + 3 * (size_t)e->blk_cap, e->bt.X, sizeof(u32) * (nb + 1), cudaMemcpyDeviceToHost, st));
      BZ_CUDA(e, cudaMemcpyAsync(e->h_trace, e->bt.ninuse, sizeof(u32) * nb, cudaMemcpyDeviceToHost, st));
      BZ_CUDA(e, cudaStreamSynchronize(st));
   }
   for (u32 b = 0; b < nb; b++) {
      ss.combined_crc = ((ss.combined_crc << 1) | (ss.combined_crc >> 31)) ^ e->h_blk[b];
      ss.st.sum_nmtf += e->h_blk[e->blk_cap + b];
      if (e->h_blk[2 * (size_t)e->blk_cap + b]) ss.st.n_power_blocks++;
      if (e->verbosity >= 2) {
         const u32* X = e->h_blk + 3 * (size_t)e->blk_cap;
         fprintf(stderr, "    block %d: crc = 0x%08x, combined CRC = 0x%08x, size = %d\n",
                 (int)(e->trace_block0 + ss.block_no + b + 1), e->h_blk[b], ss.combined_crc, (int)(X[b + 1] - X[b]));
         if (e->verbosity >= 3)
            fprintf(stderr, "      %d in block, %d after MTF & 1-2 coding, %d+2 syms in use\n",
                    (int)(X[b + 1] - X[b]), (int)e->h_blk[e->blk_cap + b], (int)e->h_trace[b]);
      }
   }
   ss.block_no += nb;
   ss.bits = end_bit;
   ss.st.n_blocks += nb; ss.st.n_windows++; ss.st.sum_nblock += E;
   ss.st.kernel_launches = e->launches;
   ss.st.bwt_rounds = e->bwt_rounds;
   float ms;
   cudaEventElapsedTime(&ms, e->ev[0], e->ev[1]); ss.st.ms_s1 += ms;
   cudaEventElapsedTime(&ms, e->ev[1], e->ev[2]); ss.st.ms_s2 += ms;
   cudaEventElapsedTime(&ms, e->ev[2], e->ev[3]); ss.st.ms_s3 += ms;
   cudaEventElapsedTime(&ms, e->ev[3], e->ev[4]); ss.st.ms_s4 += ms;
   cudaEventElapsedTime(&ms, e->ev[0], e->ev[4]); ss.st.ms_total += ms;
   return 0;
}

// ---- host-side bit carry helpers ----------------------------------------------------------
struct Sink {
   bz2b200_sink fn; void* user;
   u8* dst; size_t cap, len;      // used when fn == nullptr
   int put(const u8* p, size_t n)
   {
      if (fn) return fn(user, p, n);
      if (len + n > cap) return BZ2B200_EOUTFULL;
      memcpy(dst + len, p, n);
      len += n;
      return 0;
   }
};

static int host_put_bits(EngineFull* e, Sink& sk, u64 value, int nbits)
{
   StreamState& ss = e->ss;
   for (int k = nbits - 1; k >= 0; k--) {
      ss.carry = (u8)(ss.carry | (((value >> k) & 1) << (7 - ss.ncarry)));
      ss.ncarry++;
      if (ss.ncarry == 8) { int rc = sk.put(&ss.carry, 1); if (rc) return rc; ss.carry = 0; ss.ncarry = 0; }
   }
   ss.bits += (u64)nbits;
   return 0;
}

// Process one window whose input is already in device memory at d_in; compressed bytes go to the sink.
static int window_to_sink(EngineFull* e, const u8* d_in, u32 W, bool is_final, bool tail_merge, Sink& sk, u32* consumed)
{
   StreamState& ss = e->ss;
   cudaStream_t st = e->stream;
   const u64 bits_before = ss.bits;
   const u64 origin_bit = (bits_before >> 5) << 5;
   BZ_CUDA(e, cudaMemsetAsync(e->d_out, 0, e->out_cap, st));
   u32 nb = 0;
   int rc = run_window(e, d_in, W, is_final, tail_merge, e->d_out, origin_bit, consumed, &nb);
   if (rc) return rc;
   if (nb == 0) return 0;
   const u64 end_bit = ss.bits;
   const size_t nbytes = (size_t)((end_bit - origin_bit + 7) >> 3);
   if (nbytes > e->out_cap) return set_err(BZ2B200_EINTERNAL, "window output exceeds staging capacity");
   const size_t skip = (size_t)((bits_before >> 3) - (origin_bit >> 3));
   const size_t full_end = (size_t)((end_bit >> 3) - (origin_bit >> 3));     // first byte that is not complete
   if (!sk.fn) {
      // memory sink: copy straight into the caller's buffer, then patch the carried bits
      const size_t nfull = full_end - skip;
      if (sk.len + nfull > sk.cap) return BZ2B200_EOUTFULL;
      if (nfull) BZ_CUDA(e, cudaMemcpyAsync(sk.dst + sk.len, e->d_out + skip, nfull, cudaMemcpyDeviceToHost, st));
      BZ_CUDA(e, cudaMemcpyAsync(e->h_out, e->d_out + full_end, 1, cudaMemcpyDeviceToHost, st));
      BZ_CUDA(e, cudaStreamSynchronize(st));
      if (nfull) {
         if (ss.ncarry) sk.dst[sk.len] |= ss.carry;
         sk.len += nfull;
         ss.ncarry = (u32)(end_bit & 7);
         ss.carry = ss.ncarry ? e->h_out[0] : 0;
      } else {
         // the window ended inside the byte it started in
         ss.carry = (u8)(ss.carry | e->h_out[0]);
         ss.ncarry = (u32)(end_bit & 7);
      }
      return 0;
   }
   BZ_CUDA(e, cudaMemcpyAsync(e->h_out, e->d_out, nbytes, cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaStreamSynchronize(st));
   if (ss.ncarry) e->h_out[skip] |= ss.carry;
   if (full_end > skip) { rc = sk.put(e->h_out + skip, full_end - skip); if (rc) return rc; }
   else { ss.carry = e->h_out[skip]; ss.ncarry = (u32)(end_bit & 7); return 0; }
   ss.ncarry = (u32)(end_bit & 7);
   ss.carry = ss.ncarry ? e->h_out[full_end] : 0;
   if (full_end == skip && (bits_before & 7)) { /* still inside the same partial byte */ }
   return 0;
}

static int finish_stream(EngineFull* e, Sink& sk)
{
   StreamState& ss = e->ss;
   int rc;
   if (e->verbosity >= 2) fprintf(stderr, "    final combined CRC = 0x%08x\n   ", ss.combined_crc);      // compress.c:877-878
   if ((rc = host_put_bits(e, sk, 0x177245385090ULL, 48))) return rc;     // compress.c:874-875
   if ((rc = host_put_bits(e, sk, ss.combined_crc, 32))) return rc;       // :876
   if (ss.ncarry) { rc = sk.put(&ss.carry, 1); if (rc) return rc; ss.bits += 8 - ss.ncarry; ss.carry = 0; ss.ncarry = 0; }   // :879
   return 0;
}

static int begin_stream(EngineFull* e, Sink& sk)
{
   StreamState& ss = e->ss;
   if (ss.header_done) return 0;
   ss.header_done = true;
   return host_put_bits(e, sk, 0x425A6830u + (u32)e->level, 32);            // compress.c:841-845  "BZh" '0'+level
}

// ---- asynchronous streaming feed -----------------------------------------------------------------
static int feed_queue_sink(void* user, const void* bytes, size_t n)
{
   EngineFull* e = static_cast<EngineFull*>(user);
   AsyncFeed& a = e->af;
   pthread_mutex_lock(&a.mu);
   if (a.out_len + n > a.out_cap) {
      size_t nc = a.out_cap ? a.out_cap : ((size_t)1 << 20);
      while (nc < a.out_len + n) nc *= 2;
      u8* nb = static_cast<u8*>(realloc(a.outq, nc));
      if (!nb) { pthread_mutex_unlock(&a.mu); return BZ2B200_ENOMEM; }
      a.outq = nb; a.out_cap = nc;
   }
   memcpy(a.outq + a.out_len, bytes, n);
   a.out_len += n;
   pthread_mutex_unlock(&a.mu);
   return 0;
}

// stage 1 has fixed how much of the window this pass consumes and the H2D copy is complete: release the ring space
static void feed_after_s1(EngineFull* e, u32 consumed, void*)
{
   AsyncFeed& a = e->af;
   pthread_mutex_lock(&a.mu);
   a.head += consumed;
   a.hook_advanced = true;
   pthread_cond_broadcast(&a.cv_space);
   pthread_mutex_unlock(&a.mu);
}

static int feed_run_window(EngineFull* e, u64 head, u32 W, bool closing, int end_mode, bool tail_running, u32* cons)
{
   AsyncFeed& a = e->af;
   Sink sk; sk.fn = feed_queue_sink; sk.user = e; sk.dst = nullptr; sk.cap = 0; sk.len = 0;
   int rc = begin_stream(e, sk);
   if (rc) return rc;
   if (W) {
      const size_t pos = (size_t)(head % a.cap);
      const size_t first = (W < a.cap - pos) ? W : a.cap - pos;
      BZ_CUDA(e, cudaMemcpyAsync(e->d_in, e->h_in + pos, first, cudaMemcpyHostToDevice, e->stream));
      if (W > first) BZ_CUDA(e, cudaMemcpyAsync(e->d_in + first, e->h_in, W - first, cudaMemcpyHostToDevice, e->stream));
      e->after_s1 = feed_after_s1;
      e->after_s1_ctx = nullptr;
      rc = window_to_sink(e, e->d_in, W, closing, closing && !tail_running, sk, cons);
      e->after_s1 = nullptr;
      if (rc) return rc;
      if (*cons == 0 && !closing) return set_err(BZ2B200_EINTERNAL, "window made no progress");
   }
   if (closing && end_mode == 2) rc = finish_stream(e, sk);
   return rc;
}

static void* feed_worker(void* arg)
{
   EngineFull* e = static_cast<EngineFull*>(arg);
   AsyncFeed& a = e->af;
   cudaSetDevice(e->device);
   pthread_mutex_lock(&a.mu);
   for (;;) {
      while (!a.quit && (a.err || !((a.tail - a.head >= e->win_cap) || (a.pending_end && !a.closing_done))))
         pthread_cond_wait(&a.cv_work, &a.mu);
      if (a.quit) break;
      const u64 avail = a.tail - a.head;
      const int end_mode = a.pending_end;
      const bool closing = end_mode != 0 && avail <= e->win_cap;
      const u32 W = (u32)(avail < e->win_cap ? avail : e->win_cap);
      const u64 head = a.head;
      const bool tail_running = e->ss.tail_running;
      a.busy = true;
      a.hook_advanced = false;
      pthread_mutex_unlock(&a.mu);
      u32 cons = 0;
      const int rc = feed_run_window(e, head, W, closing, end_mode, tail_running, &cons);
      pthread_mutex_lock(&a.mu);
      if (!a.hook_advanced) a.head += cons;
      a.busy = false;
      if (rc) { a.err = rc; snprintf(a.errtext, sizeof a.errtext, "%s", g_err[0] ? g_err : e->err); }   // g_err is this thread's copy
      if (closing || rc) a.closing_done = true;
      pthread_cond_broadcast(&a.cv_space);
      pthread_cond_broadcast(&a.cv_done);
   }
   pthread_mutex_unlock(&a.mu);
   return nullptr;
}

static int feed_start(EngineFull* e)
{
   AsyncFeed& a = e->af;
   if (!a.inited) {
      pthread_mutex_init(&a.mu, nullptr);
      pthread_cond_init(&a.cv_work, nullptr);
      pthread_cond_init(&a.cv_space, nullptr);
      pthread_cond_init(&a.cv_done, nullptr);
      a.inited = true;
   }
   if (!a.th_started) {
      a.quit = false;
      if (pthread_create(&a.th, nullptr, feed_worker, e) != 0) return set_err(BZ2B200_ENOMEM, "cannot start the feed thread");
      a.th_started = true;
   }
   return 0;
}

static void feed_shutdown(EngineFull* e)
{
   AsyncFeed& a = e->af;
   if (a.th_started) {
      pthread_mutex_lock(&a.mu);
      a.quit = true;
      pthread_cond_broadcast(&a.cv_work);
      pthread_mutex_unlock(&a.mu);
      pthread_join(a.th, nullptr);
      a.th_started = false;
   }
   if (a.inited) {
      pthread_mutex_destroy(&a.mu);
      pthread_cond_destroy(&a.cv_work); pthread_cond_destroy(&a.cv_space); pthread_cond_destroy(&a.cv_done);
      a.inited = false;
   }
   free(a.outq);
   a.outq = nullptr; a.out_len = a.out_cap = 0;
}

// a new stream starts: wait for a window the previous (abandoned) stream may still have in flight, then forget it
void feed_reset(EngineFull* e)
{
   AsyncFeed& a = e->af;
   if (!a.inited) return;
   pthread_mutex_lock(&a.mu);
   while (a.busy) pthread_cond_wait(&a.cv_done, &a.mu);
   a.head = a.tail = 0;
   a.pending_end = 0; a.closing_done = false; a.err = 0; a.out_len = 0;
   pthread_mutex_unlock(&a.mu);
}

// hand the compressed bytes the worker has produced so far to the caller's sink (on the caller's thread)
static int feed_drain(EngineFull* e, bz2b200_sink sink, void* user)
{
   AsyncFeed& a = e->af;
   pthread_mutex_lock(&a.mu);
   u8* buf = a.outq; const size_t n = a.out_len;
   if (n == 0) { pthread_mutex_unlock(&a.mu); return 0; }
   a.outq = nullptr; a.out_len = a.out_cap = 0;          // the worker starts a fresh queue
   pthread_mutex_unlock(&a.mu);
   const int rc = sink(user, buf, n);
   free(buf);
   return rc;
}

} // namespace bz

using namespace bz;

extern "C" {

const char* bz2b200_last_error(void) { return g_err; }
const char* bz2b200_version(void) { return "bzip2-b200 0.1 (sm_100a), stream-compatible with libbzip2 1.0.6x"; }

int bz2b200_device_count(void)
{
   int n = 0;
   if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
   return n;
}

int bz2b200_engine_create(bz2b200_engine** out, int device, int block_size_100k, size_t window_bytes)
{
   if (!out) return set_err(BZ2B200_EPARAM, "null out pointer");
   int prev = -1;
   cudaGetDevice(&prev);
   EngineFull* e = nullptr;
   int rc = engine_new(&e, device, block_size_100k, window_bytes, false);
   if (prev >= 0) cudaSetDevice(prev);
   if (rc) return rc;
   stream_reset(e);
   *out = reinterpret_cast<bz2b200_engine*>(e);
   return 0;
}

int bz2b200_engine_create_bounded(bz2b200_engine** out, int device, int block_size_100k, size_t max_input_bytes)
{
   if (!out || max_input_bytes == 0) return set_err(BZ2B200_EPARAM, "bad argument");
   int prev = -1;
   cudaGetDevice(&prev);
   EngineFull* e = nullptr;
   int rc = engine_new(&e, device, block_size_100k, max_input_bytes, true);
   if (prev >= 0) cudaSetDevice(prev);
   if (rc) return rc;
   stream_reset(e);
   *out = reinterpret_cast<bz2b200_engine*>(e);
   return 0;
}

void bz2b200_engine_destroy(bz2b200_engine* h)
{
   if (!h) return;
   DeviceGuard guard(reinterpret_cast<EngineFull*>(h)->device);
   engine_free(reinterpret_cast<EngineFull*>(h));
}

int bz2b200_compress_host(bz2b200_engine* h, const void* src, size_t src_len, void* dst, size_t* dst_len,
                          unsigned flags, bz2b200_stats* stats)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e || !dst || !dst_len || (!src && src_len)) return set_err(BZ2B200_EPARAM, "bad argument");
   if (e->bounded && src_len > e->win_cap) return set_err(BZ2B200_EPARAM, "input larger than this bounded engine was created for");
   DeviceGuard guard(e->device);
   int rc = ensure_staging(e, false);
   if (rc) return rc;
   feed_reset(e);                 // a stream abandoned on this (pooled) engine may still have a window in flight
   stream_reset(e);
   Sink sk; sk.fn = nullptr; sk.user = nullptr; sk.dst = static_cast<u8*>(dst); sk.cap = *dst_len; sk.len = 0;
   if ((rc = begin_stream(e, sk))) return rc;
   const u8* in = static_cast<const u8*>(src);
   const bool tail_merge = !(flags & BZ2B200_TAIL_STREAMED);
   // Pinned (or registered) source: the next window's H2D is issued as soon as stage 1 has fixed
   // where it starts, on a second stream, so it overlaps stages 2-4 of the current window.
   bool pinned = false;
   if (src_len) {
      cudaPointerAttributes at;
      if (cudaPointerGetAttributes(&at, src) == cudaSuccess) pinned = (at.type == cudaMemoryTypeHost);
      else cudaGetLastError();
   }
   struct Prefetch { const u8* in; size_t n, pos; int buf; bool issued; u8* dbuf[2]; } pf;
   pf.in = in; pf.n = src_len; pf.pos = 0; pf.buf = 0; pf.issued = false; pf.dbuf[0] = e->d_in; pf.dbuf[1] = e->d_in2;
   e->after_s1 = nullptr; e->after_s1_ctx = &pf;
   if (pinned) {
      e->after_s1 = [](EngineFull* ee, u32 cons, void* ctx) {
         Prefetch* p = static_cast<Prefetch*>(ctx);
         const size_t next = p->pos + cons;
         p->issued = false;
         if (cons == 0 || next >= p->n) return;
         const size_t W2 = (p->n - next < ee->win_cap) ? (p->n - next) : ee->win_cap;
         const int nb = p->buf ^ 1;
         if (cudaMemcpyAsync(p->dbuf[nb], p->in + next, W2, cudaMemcpyHostToDevice, ee->copy_stream) != cudaSuccess) { cudaGetLastError(); return; }
         cudaEventRecord(ee->ev_h2d[nb], ee->copy_stream);
         p->issued = true;
      };
   }
   size_t pos = 0;
   while (pos < src_len) {
      const size_t W = (src_len - pos < e->win_cap) ? (src_len - pos) : e->win_cap;
      const bool fin = (pos + W == src_len);
      pf.pos = pos;
      u8* dcur = pf.dbuf[pf.buf];
      if (pf.issued) BZ_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_h2d[pf.buf], 0));
      else BZ_CUDA(e, cudaMemcpyAsync(dcur, in + pos, W, cudaMemcpyHostToDevice, e->stream));
      pf.issued = false;
      u32 cons = 0;
      rc = window_to_sink(e, dcur, (u32)W, fin, tail_merge, sk, &cons);
      if (rc) { e->after_s1 = nullptr; cudaStreamSynchronize(e->copy_stream); return rc; }
      if (cons == 0) { e->after_s1 = nullptr; cudaStreamSynchronize(e->copy_stream); return set_err(BZ2B200_EINTERNAL, "window made no progress"); }
      pos += cons;
      if (pf.issued) pf.buf ^= 1;
   }
   e->after_s1 = nullptr;
   if ((rc = finish_stream(e, sk))) return rc;
   *dst_len = sk.len;
   e->ss.st.in_bytes = src_len; e->ss.st.out_bytes = sk.len; e->ss.st.combined_crc = e->ss.combined_crc;
   if (stats) *stats = e->ss.st;
   return 0;
}

int bz2b200_compress_device(bz2b200_engine* h, const void* d_src, size_t src_len, void* d_dst, size_t dst_cap,
                            size_t* dst_len, unsigned flags, bz2b200_stats* stats)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e || !d_dst || !dst_len || (!d_src && src_len) || ((uintptr_t)d_dst & 3)) return set_err(BZ2B200_EPARAM, "bad argument");
   DeviceGuard guard(e->device);
   feed_reset(e);
   e->after_s1 = nullptr;
   stream_reset(e);
   StreamState& ss = e->ss;
   u8* out = static_cast<u8*>(d_dst);
   // worst case: incompressible data grows by < 1% plus per-block tables
   const size_t need = src_len + src_len / 64 + (src_len / e->nmax + 2) * 24576 + 64;
   if (dst_cap < need) return set_err(BZ2B200_EOUTFULL, "device destination too small (need src_len*1.016 + 24 KiB per block)");
   BZ_CUDA(e, cudaMemsetAsync(out, 0, dst_cap & ~(size_t)3, e->stream));
   int rc = 0;
   if (!(flags & BZ2B200_NO_HEADER)) {
      rc = put_bits_device(e, out, 0, 0, 0x425A6830u + (u32)e->level, 32);
      if (rc) return rc;
      ss.bits = 32;
   }
   ss.header_done = true;
   const u8* in = static_cast<const u8*>(d_src);
   const bool tail_merge = !(flags & BZ2B200_TAIL_STREAMED);
   size_t pos = 0;
   while (pos < src_len) {
      const size_t W = (src_len - pos < e->win_cap) ? (src_len - pos) : e->win_cap;
      const bool fin = (pos + W == src_len);
      u32 cons = 0, nb = 0;
      rc = run_window(e, in + pos, (u32)W, fin, tail_merge, out, 0, &cons, &nb);
      if (rc) return rc;
      if (cons == 0) return set_err(BZ2B200_EINTERNAL, "window made no progress");
      pos += cons;
   }
   if (!(flags & BZ2B200_NO_TRAILER)) {
      if ((rc = put_bits_device(e, out, 0, ss.bits, 0x177245385090ULL, 48))) return rc;
      ss.bits += 48;
      if ((rc = put_bits_device(e, out, 0, ss.bits, ss.combined_crc, 32))) return rc;
      ss.bits += 32;
   }
   ss.st.out_bits = ss.bits;
   BZ_CUDA(e, cudaStreamSynchronize(e->stream));
   *dst_len = (size_t)((ss.bits + 7) >> 3);
   ss.st.in_bytes = src_len; ss.st.out_bytes = *dst_len; ss.st.combined_crc = ss.combined_crc;
   if (stats) *stats = ss.st;
   return 0;
}

int bz2b200_stream_begin(bz2b200_engine* h)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e) return set_err(BZ2B200_EPARAM, "null engine");
   if (e->bounded) return set_err(BZ2B200_EPARAM, "a bounded engine serves one-shot calls only");
   DeviceGuard guard(e->device);
   int rc = ensure_staging(e, true);
   if (rc) return rc;
   feed_reset(e);
   stream_reset(e);
   return 0;
}

int bz2b200_stream_feed(bz2b200_engine* h, const void* src, size_t n, int end_mode, bz2b200_sink sink, void* user)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e || !sink || (!src && n) || end_mode < 0 || end_mode > 2) return set_err(BZ2B200_EPARAM, "bad argument");
   if (!e->h_in) return set_err(BZ2B200_EPARAM, "bz2b200_stream_begin was not called");
   int rc = feed_start(e);
   if (rc) return rc;
   AsyncFeed& a = e->af;
   if ((rc = feed_drain(e, sink, user))) return rc;
   const u8* in = static_cast<const u8*>(src);
   size_t off = 0;
   while (off < n) {
      pthread_mutex_lock(&a.mu);
      while (!a.err && a.tail - a.head >= a.cap) pthread_cond_wait(&a.cv_space, &a.mu);
      if (a.err) { rc = a.err; set_err_text(a.errtext); pthread_mutex_unlock(&a.mu); return rc; }
      const size_t space = a.cap - (size_t)(a.tail - a.head);
      const size_t take = (n - off < space) ? (n - off) : space;
      const size_t pos = (size_t)(a.tail % a.cap);
      pthread_mutex_unlock(&a.mu);
      // [tail, tail + take) is not visible to the worker until tail moves
      const size_t first = (take < a.cap - pos) ? take : a.cap - pos;
      memcpy(e->h_in + pos, in + off, first);
      if (take > first) memcpy(e->h_in, in + off + first, take - first);
      pthread_mutex_lock(&a.mu);
      a.tail += take;
      e->ss.tail_running = (end_mode == 0);
      e->ss.st.in_bytes += take;
      pthread_cond_signal(&a.cv_work);
      pthread_mutex_unlock(&a.mu);
      off += take;
      if ((rc = feed_drain(e, sink, user))) return rc;
   }
   if (end_mode != 0) {
      pthread_mutex_lock(&a.mu);
      a.pending_end = end_mode;
      a.closing_done = false;
      pthread_cond_signal(&a.cv_work);
      while (!a.closing_done && !a.err) pthread_cond_wait(&a.cv_done, &a.mu);
      a.pending_end = 0;
      rc = a.err;
      if (rc) set_err_text(a.errtext);
      pthread_mutex_unlock(&a.mu);
      if (rc) return rc;
   }
   return feed_drain(e, sink, user);
}

int bz2b200_engine_set_stream(bz2b200_engine* h, void* cuda_stream)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e) return set_err(BZ2B200_EPARAM, "null engine");
   e->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : e->own_stream;
   return 0;
}

struct bz2b200_scan { ScanState s; size_t cap; };

void bz2b200_scan_destroy(bz2b200_scan* h)
{
   if (!h) return;
   ScanState& s = h->s;
   DeviceGuard guard(s.device);
   void* dev[] = { s.tile_len, s.tile_ext, s.tile_carry, s.tile_size, s.tile_base, s.cend, s.scal, s.q };
   for (void* p : dev) if (p) cudaFree(p);
   if (s.h_scal) cudaFreeHost(s.h_scal);
   if (s.st) cudaStreamDestroy(s.st);
   free(h);
}

static void scan_set_input(ScanState& s, const void* d_src, size_t n, int prev_byte, uint64_t prev_run, int input_ends)
{
   s.in = static_cast<const u8*>(d_src); s.W = (u32)n; s.input_ends = input_ends ? 1u : 0u;
   s.prev_byte = (prev_byte >= 0 && prev_byte < 256 && prev_run) ? (u32)prev_byte : 256u;
   s.carry0 = (s.prev_byte < 256) ? (u32)(prev_run % 255u) : 0u;
}

int bz2b200_scan_create(bz2b200_scan** out, int device, int level, const void* d_src, size_t n,
                        int prev_byte, uint64_t prev_run, int input_ends)
{
   if (!out || level < 1 || level > 9 || (!d_src && n) || n >= 0xfff00000ull) return set_err(BZ2B200_EPARAM, "bad argument");
   int ndev = 0;
   if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return set_err(BZ2B200_ENODEV, "no such CUDA device");
   bz2b200_scan* h = static_cast<bz2b200_scan*>(calloc(1, sizeof(bz2b200_scan)));
   if (!h) return set_err(BZ2B200_ENOMEM, "out of host memory");
   ScanState& s = h->s;
   DeviceGuard guard(device);
   s.device = device; s.nmax = 100000u * (u32)level - 19u;
   scan_set_input(s, d_src, n, prev_byte, prev_run, input_ends);
   const size_t nt = n / 4096 + 4;
   h->cap = n;
   s.cend_cap = n + n / 4 + 4096;
   bool ok = cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking) == cudaSuccess;
   ok = ok && cudaMalloc(reinterpret_cast<void**>(&s.tile_len), nt * 4) == cudaSuccess;
   ok = ok && cudaMalloc(reinterpret_cast<void**>(&s.tile_ext), nt * 4) == cudaSuccess;
   ok = ok && cudaMalloc(reinterpret_cast<void**>(&s.tile_carry), nt * 4) == cudaSuccess;
   ok = ok && cudaMalloc(reinterpret_cast<void**>(&s.tile_size), nt * 4) == cudaSuccess;
   ok = ok && cudaMalloc(reinterpret_cast<void**>(&s.tile_base), nt * 4) == cudaSuccess;
   ok = ok && cudaMalloc(reinterpret_cast<void**>(&s.cend), s.cend_cap) == cudaSuccess;
   ok = ok && cudaMalloc(reinterpret_cast<void**>(&s.scal), 16 * 4) == cudaSuccess;
   ok = ok && cudaMalloc(reinterpret_cast<void**>(&s.q), 2 * 4) == cudaSuccess;
   ok = ok && cudaMallocHost(reinterpret_cast<void**>(&s.h_scal), 16 * 4) == cudaSuccess;
   if (!ok) { cudaGetLastError(); bz2b200_scan_destroy(h); return set_err(BZ2B200_ENOMEM, "scan allocation failed"); }
   cudaMemsetAsync(s.scal, 0, 16 * 4, s.st);
   const int rc = n ? scan_build(&s, s.prev_byte, s.carry0) : 0;
   if (rc) { bz2b200_scan_destroy(h); return set_err(BZ2B200_ECUDA, "shard scan failed"); }
   *out = h;
   return 0;
}

int bz2b200_scan_rescan(bz2b200_scan* h, const void* d_src, size_t n, int prev_byte, uint64_t prev_run, int input_ends)
{
   if (!h || (!d_src && n)) return set_err(BZ2B200_EPARAM, "bad argument");
   if (n > h->cap) return set_err(BZ2B200_EOUTFULL, "region larger than the scan was created for");
   ScanState& s = h->s;
   DeviceGuard guard(s.device);
   scan_set_input(s, d_src, n, prev_byte, prev_run, input_ends);
   cudaMemsetAsync(s.scal, 0, 16 * 4, s.st);
   const int rc = n ? scan_build(&s, s.prev_byte, s.carry0) : 0;
   if (rc) return set_err(BZ2B200_ECUDA, "shard scan failed");
   return 0;
}

int bz2b200_scan_boundary(bz2b200_scan* h, size_t start, size_t limit, unsigned flags, size_t* boundary, uint32_t* n_blocks)
{
   if (!h || !boundary || start > h->s.W) return set_err(BZ2B200_EPARAM, "bad argument");
   ScanState& s = h->s;
   DeviceGuard guard(s.device);
   if (limit > s.W) limit = s.W;
   if (start >= limit) { *boundary = start; if (n_blocks) *n_blocks = 0; return 0; }
   u32 b = 0, nb = 0;
   const int rc = scan_boundary(&s, (u32)start, (u32)limit, (flags & BZ2B200_TAIL_STREAMED) ? 0u : 1u, &b, &nb);
   if (rc == -3) return set_err(BZ2B200_EOUTFULL, "block chain ran past the scanned data (halo too small)");
   if (rc) return set_err(BZ2B200_ECUDA, "boundary chain failed");
   *boundary = b;
   if (n_blocks) *n_blocks = nb;
   return 0;
}

int bz2b200_concat_bits(int device, void* d_dst, uint64_t dst_bit, const void* d_src, uint64_t nbits)
{
   if (!d_dst || (!d_src && nbits) || ((uintptr_t)d_dst & 3) || ((uintptr_t)d_src & 3)) return set_err(BZ2B200_EPARAM, "bad argument");
   DeviceGuard guard(device);
   const int rc = concat_bits_device(static_cast<u8*>(d_dst), dst_bit, static_cast<const u8*>(d_src), nbits);
   if (rc) return set_err(BZ2B200_ECUDA, "concat_bits failed");
   return 0;
}

int bz2b200_engine_set_verbosity(bz2b200_engine* h, int verbosity)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e) return set_err(BZ2B200_EPARAM, "null engine");
   e->verbosity = verbosity;
   return 0;
}

int bz2b200_debug_keep(bz2b200_engine* h, int on)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e) return BZ2B200_EPARAM;
   e->debug_keep = on != 0;
   return 0;
}

int bz2b200_debug_fetch(bz2b200_engine* h, const char* name, void* dst, size_t cap, size_t* got)
{
   EngineFull* e = reinterpret_cast<EngineFull*>(h);
   if (!e || !name || !dst || !got) return set_err(BZ2B200_EPARAM, "bad argument");
   DeviceGuard guard(e->device);
   const size_t nb = e->last_nb, E = e->last_E;
   const void* src = nullptr; size_t bytes = 0;
   struct { const char* n; const void* p; size_t b; } tab[] = {
      {"X", e->bt.X, (nb + 1) * 4}, {"P", e->bt.P, (nb + 1) * 4}, {"crc", e->bt.crc, nb * 4},
      {"origptr", e->bt.origptr, nb * 4}, {"power_q", e->bt.power_q, nb * 4}, {"inuse", e->bt.inuse, nb * 256},
      {"ninuse", e->bt.ninuse, nb * 4}, {"nmtf", e->bt.nmtf, nb * 4}, {"mtffreq", e->bt.mtffreq, nb * BZ_MAX_ALPHA * 4},
      {"bits", e->bt.bits, nb * 8}, {"bitoff", e->bt.bitoff, (nb + 1) * 8},
      {"enc", e->enc, E}, {"bwt", e->bwt, E}, {"z", e->z, E}, {"mtfv", e->mtfv, (E + nb) * 2}, {"sa", e->sa, E * 4},
      {"rank", e->rank, E * 8},
      {"sel", e->sel, E / 50 + 2 * nb + 8}, {"hlen", e->hlen, nb * 6 * BZ_MAX_ALPHA}, {"ngroups", e->ngroups, nb * 4},
      {"prebits", e->prebits, nb * 4},
   };
   for (auto& t : tab) if (!strcmp(t.n, name)) { src = t.p; bytes = t.b; }
   if (!src) return set_err(BZ2B200_EPARAM, "unknown debug buffer name");
   if (bytes > cap) return set_err(BZ2B200_EOUTFULL, "debug destination too small");
   if (bytes) BZ_CUDA(e, cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
   *got = bytes;
   return 0;
}

} // extern "C"
