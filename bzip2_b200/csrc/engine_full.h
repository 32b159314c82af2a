// engine_full.h -- the engine with its per-stream state, shared by engine.cu (one engine, one stream) and multi.cu
// (several engines -- on one or several GPUs -- working on consecutive windows of one stream).
#pragma once
#include "engine.h"
#include "../../include/bz2_b200.h"
#include <pthread.h>

namespace bz {

// ---- stream state kept between windows -----------------------------------------------------
struct StreamState {
   u64 bits;            // absolute stream bits produced so far
   u32 combined_crc;    // compress.c:826-828
   u32 block_no;
   bool header_done;
   bool tail_running;   // last byte arrived in BZ_RUN mode
   // host-side bit carry for the host/stream paths
   u8  carry; u32 ncarry;
   size_t h_fill;       // bytes waiting in h_in
   bz2b200_stats st;
};

// Streaming feed (bz2b200_stream_feed): the caller's thread only copies input into a pinned ring; a worker
// thread owned by the engine cuts windows out of it and runs them, so feeding (fread / memcpy in the client)
// overlaps the GPU work (SURVEY 8(f)1: the reference's BZ2_bzWrite trickle, bzlib.c:1049-1066).
struct AsyncFeed {
   pthread_t th;
   pthread_mutex_t mu;
   pthread_cond_t cv_work, cv_space, cv_done;
   bool inited, th_started;
   size_t cap;                 // ring capacity in bytes (the ring is h_in)
   u64 head, tail;             // absolute byte counters: the ring holds stream bytes [head, tail)
   int pending_end;            // closing request posted by the feeding thread: 1 = flush, 2 = finish
   bool closing_done, busy, quit, hook_advanced;
   int err; char errtext[256]; // first failure of the worker and its text (the worker's thread-local message does not travel)
   u8* outq; size_t out_len, out_cap;   // compressed bytes produced by the worker, drained by the feeding thread
};

struct EngineFull : Engine {
   StreamState ss;
   AsyncFeed af;
   bool debug_keep;
   bool bounded;               // created for inputs of at most win_cap bytes (one-shot calls): no minimum window
   u32 last_nb, last_E;
   cudaEvent_t ev[6];
   // host path: double-buffered input so the next window's H2D overlaps this window's kernels
   u8* d_in2;
   cudaStream_t copy_stream;
   cudaEvent_t ev_h2d[2];
   void (*after_s1)(EngineFull*, u32 consumed, void* ctx);
   void* after_s1_ctx;
   u32* h_items;               // batch calls: pinned [4 * (blk_cap + 1)] u32 -- item starts, first blocks, CRCs, byte offsets
};

// engine.cu
int  engine_new(EngineFull** out, int device, int level, size_t window_bytes, bool bounded = false, size_t extra_slots = 0);
void engine_free(EngineFull* e);
int  ensure_staging(EngineFull* e, bool need_hin);
void stream_reset(EngineFull* e);
void feed_reset(EngineFull* e);
int  run_window(EngineFull* e, const u8* d_in, u32 W, bool is_final, bool tail_merge,
                u8* d_out, u64 origin_bit, u32* consumed, u32* nb_out);
int  set_err(int code, const char* msg);
void set_err_text(const char* msg);

// Makes the engine's device current for the duration of a C-ABI call and restores the caller's.
struct DeviceGuard {
   int prev;
   explicit DeviceGuard(int dev) : prev(-1) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
   ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

} // namespace bz
