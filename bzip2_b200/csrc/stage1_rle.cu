// stage1_rle.cu -- S1: initial run-length coding, block split and block CRCs.
//
// Replaces copy_input_until_stop (reference bzlib.c:211-315) and the per-byte
// BZ_UPDATE_CRC (bzlib_private.h:197-202, crctable.c:29-99).
//
// The reference walks the input one byte at a time.  Restated for a parallel
// machine: the input is a sequence of "chunks" (maximal runs cut every 255
// bytes); a chunk of length L costs min(L,4) + (L>=4) encoded bytes; a block
// closes at the first chunk end where its encoded size reaches nblockMAX.
// Everything except that greedy chain is a scan:
//   k_tile<AGG>      per 4 KiB tile: (trailing run length, tile-is-one-run) aggregate
//   k_scan_runs      segmented scan of the aggregates -> run length entering each tile
//   k_tile<COUNT>    encoded bytes produced by each tile
//   k_scan_u32       exclusive scan -> encoded offset of each tile
//   k_tile<SCATTER>  write enc[] and the chunk-end flags cend[]
//   k_chain          one warp follows the greedy block chain through cend[]
//   k_tile<FIND>     map each block's encoded start back to its input position
//   k_crc            block CRCs: per-thread table CRC, GF(2) shift-combine, atomicXor
#include "engine.h"
#include <string.h>

namespace bz {

constexpr int S1_THREADS = 256;
constexpr int S1_BPT = 16;
constexpr int S1_TILE = S1_THREADS * S1_BPT;   // 4096
constexpr int S1_STAGE = S1_TILE + S1_TILE / 4 + 48;   // worst case 5 output bytes per 4 input bytes, + alignment slack

enum { S1_AGG = 0, S1_COUNT = 1, S1_SCATTER = 2, S1_FIND = 3, S1_LOCATE = 4 };

struct RunAgg { u32 len; u32 ext; };   // ext: every position so far continues the run entering the range
__device__ __forceinline__ RunAgg run_comb(RunAgg a, RunAgg b)
{
   RunAgg r;
   r.len = b.ext ? a.len + b.len : b.len;
   r.ext = a.ext & b.ext;
   return r;
}

// Exclusive block scan of RunAgg (identity = {0,1}); also returns the block aggregate.
__device__ __forceinline__ RunAgg run_block_excl(RunAgg v, RunAgg* wsm, RunAgg* total)
{
   const u32 l = lane_id(), w = threadIdx.x >> 5;
   RunAgg inc = v;
#pragma unroll
   for (int d = 1; d < 32; d <<= 1) {
      RunAgg t;
      t.len = __shfl_up_sync(FULL, inc.len, d);
      t.ext = __shfl_up_sync(FULL, inc.ext, d);
      if (l >= (u32)d) inc = run_comb(t, inc);
   }
   __syncthreads();
   if (l == 31) wsm[w] = inc;
   __syncthreads();
   RunAgg pre; pre.len = 0; pre.ext = 1;
   for (u32 k = 0; k < w; k++) pre = run_comb(pre, wsm[k]);
   RunAgg tot = pre;
   for (u32 k = w; k < S1_THREADS / 32; k++) tot = run_comb(tot, wsm[k]);
   if (total) *total = tot;
   // exclusive within warp
   RunAgg ex;
   ex.len = __shfl_up_sync(FULL, inc.len, 1);
   ex.ext = __shfl_up_sync(FULL, inc.ext, 1);
   if (l == 0) { ex.len = 0; ex.ext = 1; }
   return run_comb(pre, ex);
}

struct S1Params {
   const u8* in;        // window base (any alignment)
   u32 W;               // window length
   u32 is_final;
   u32* tile_len; u32* tile_ext; u32* tile_carry; u32* tile_size; u32* tile_base;
   u8* enc; u8* cend;
   const u32* X; u32* P; u32 nb_find;   // FIND mode: encoded offsets X[1..] -> input positions P[1..]
   const u32* scalars;                   // [2] = enc_total
   u32 prev_byte;       // byte before in[0] (256: none) and the length of the run it ends,
   u32 carry0;          // when the window does not start at a chunk boundary (shard scans)
   const u32* Q; u32* EQ;                // LOCATE mode: input positions Q[k] -> encoded offsets EQ[k]
   const u32* seams; u32 nseams;         // batch windows: sorted item starts; no run continues into one (0: none)
};

template <int MODE>
__global__ void __launch_bounds__(S1_THREADS) k_tile(S1Params p)
{
   __shared__ RunAgg wsm[S1_THREADS / 32];
   __shared__ u32 ssm[34];
   __shared__ u32 s_tile;
   const u32 align = (u32)((uintptr_t)p.in & 15);
   const u8* base = p.in - align;
   u32 tile = blockIdx.x;
   u32 findX = 0;
   if (MODE == S1_FIND) {
      // one CTA per boundary: locate the tile whose encoded range contains X[b]
      const u32 b = blockIdx.x + 1;
      if (p.nb_find && blockIdx.x >= p.scalars[0]) return;      // grid sized by an upper bound; scalars[0] = blocks found
      findX = p.X[b];
      const u32 ntiles = (p.W + align + S1_TILE - 1) / S1_TILE;
      if (findX >= p.scalars[2]) { if (threadIdx.x == 0) p.P[b] = p.W; return; }
      if (threadIdx.x == 0) {
         u32 lo = 0, hi = ntiles - 1;          // largest t with tile_base[t] <= X and tile non-empty beyond
         while (lo < hi) {
            u32 mid = (lo + hi + 1) >> 1;
            if (p.tile_base[mid] <= findX) lo = mid; else hi = mid - 1;
         }
         // step back over empty tiles that share the same base
         while (lo > 0 && p.tile_size[lo] == 0) lo--;
         s_tile = lo;
      }
      __syncthreads();
      tile = s_tile;
   }
   u32 locQ = 0;
   if (MODE == S1_LOCATE) {
      locQ = p.Q[blockIdx.x];
      if (locQ >= p.W) { if (threadIdx.x == 0) p.EQ[blockIdx.x] = p.scalars[2]; return; }
      tile = (locQ + align) / S1_TILE;
   }
   const i64 pos0 = (i64)tile * S1_TILE + (i64)threadIdx.x * S1_BPT - (i64)align;   // window position of c[0]
   u8 c[S1_BPT];
   {
      const u8* src = base + (size_t)tile * S1_TILE + (size_t)threadIdx.x * S1_BPT;
      if (pos0 >= 0 && pos0 + S1_BPT <= (i64)p.W) {
         uint4 v = *reinterpret_cast<const uint4*>(src);
         u32 w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
         for (int k = 0; k < 16; k++) c[k] = (u8)(w4[k >> 2] >> ((k & 3) * 8));
      } else {
#pragma unroll
         for (int k = 0; k < 16; k++) { i64 q = pos0 + k; c[k] = (q >= 0 && q < (i64)p.W) ? src[k] : 0; }
      }
   }
   u32 prevb = 256, nextb = 256;
   if (pos0 >= 1 && pos0 - 1 < (i64)p.W) prevb = p.in[pos0 - 1];
   else if (pos0 == 0) prevb = p.prev_byte;
   if (pos0 + S1_BPT >= 0 && pos0 + S1_BPT < (i64)p.W) nextb = p.in[pos0 + S1_BPT];
   // Batch windows hold many independent inputs: an item start behaves like a window start (the byte before it is
   // "none"), so no run, chunk or block crosses from one item into the next and the last byte of every item ends a chunk.
   u32 seam = 0;                                            // bit k: position pos0 + k starts an item (k = 0..16)
   if (p.nseams) {
      u32 lo = 0, hi = p.nseams;
      while (lo < hi) { const u32 mid = (lo + hi) >> 1; if ((i64)p.seams[mid] < pos0) lo = mid + 1; else hi = mid; }
      for (u32 s = lo; s < p.nseams && (i64)p.seams[s] <= pos0 + S1_BPT; s++) seam |= 1u << (u32)((i64)p.seams[s] - pos0);
      if (seam & 1u) prevb = 256;
      if (seam & (1u << S1_BPT)) nextb = 256;
   }

   // per-position "continues the run" flags and the thread aggregate
   u32 eqmask = 0, vmask = 0;
   RunAgg agg; agg.len = 0; agg.ext = 1;
#pragma unroll
   for (int k = 0; k < 16; k++) {
      i64 q = pos0 + k;
      bool valid = (q >= 0 && q < (i64)p.W);
      u32 pb = (k == 0) ? prevb : (u32)c[k - 1];
      if (k > 0 && q == 0) pb = p.prev_byte;               // 256 unless the window continues a run (shard scans)
      if ((seam >> k) & 1u) pb = 256;
      bool eq = valid && (pb == (u32)c[k]);
      if (valid) {
         vmask |= 1u << k;
         if (eq) { eqmask |= 1u << k; agg.len += 1; } else { agg.len = 1; agg.ext = 0; }
      }
   }
   RunAgg tot;
   RunAgg pre = run_block_excl(agg, wsm, &tot);
   if (MODE == S1_AGG) {
      if (threadIdx.x == 0) { p.tile_len[tile] = tot.len; p.tile_ext[tile] = tot.ext; }
      return;
   }
   const u32 carry = p.tile_carry[tile];
   u32 rbefore = pre.ext ? carry + pre.len : pre.len;      // run length ending just before c[0]

   // phases and emitted byte counts
   u32 j = 0;                                               // phase of current position
   u32 emitted = 0;
   u32 ph[16];
#pragma unroll
   for (int k = 0; k < 16; k++) {
      if (!((vmask >> k) & 1)) { ph[k] = 0xffff; continue; }
      if ((eqmask >> k) & 1) {
         if (k == 0 || pos0 + k == 0) j = rbefore % 255u; else { j = j + 1; if (j == 255) j = 0; }
      } else j = 0;
      // careful: when k>0 and previous position was invalid (before window) j restarts at 0 via eq=false
      ph[k] = j;
      emitted += (j < 3) ? 1u : (j == 3 ? 2u : 0u);
   }
   u32 ttotal;
   u32 off = block_excl_sum<S1_THREADS>(emitted, ssm, &ttotal);
   if (MODE == S1_COUNT) {
      if (threadIdx.x == 0) p.tile_size[tile] = ttotal;
      return;
   }
   if (MODE == S1_FIND || MODE == S1_LOCATE) {
      u32 E = p.tile_base[tile] + off;
#pragma unroll
      for (int k = 0; k < 16; k++) {
         if (ph[k] == 0xffff) continue;
         const u32 jj = ph[k];
         const i64 q = pos0 + k;
         if (MODE == S1_FIND) { if (jj == 0 && E == findX) p.P[blockIdx.x + 1] = (u32)q; }
         else if ((u32)q == locQ) p.EQ[blockIdx.x] = E;
         E += (jj < 3) ? 1u : (jj == 3 ? 2u : 0u);
      }
      return;
   }
   // SCATTER.  The tile's output bytes and chunk-end flags are staged in shared memory at the alignment they
   // have in HBM and flushed with 16-byte stores: byte stores straight to HBM cost one sector write each.
   // One output byte of a tile can be "open": the count byte of a run that crosses the tile's end is written
   // by the later tile in which the run (or its 255-byte chunk) ends, so the flush leaves it alone.
   __shared__ __align__(16) u8 s_enc[S1_STAGE];
   __shared__ __align__(16) u8 s_cend[S1_STAGE];
   __shared__ int s_open;
   const bool wr = (p.enc != nullptr);                     // shard scans only need the chunk-end flags
   const u32 tb = p.tile_base[tile];
   const u32 mis = tb & 15u;
   const u32 nst = mis + ttotal;                           // staged bytes [mis, nst) belong to this tile
   for (u32 g = threadIdx.x; g * 16 < nst + 16; g += S1_THREADS) reinterpret_cast<uint4*>(s_cend)[g] = make_uint4(0u, 0u, 0u, 0u);
   if (threadIdx.x == 0) s_open = -1;
   __syncthreads();
   const i64 tile_last = min((i64)(tile + 1) * S1_TILE - (i64)align, (i64)p.W) - 1;
   u32 El = off;                                           // offset inside the tile's output
#pragma unroll
   for (int k = 0; k < 16; k++) {
      if (ph[k] == 0xffff) continue;
      const u32 jj = ph[k];
      const i64 q = pos0 + k;
      const u32 ch = c[k];
      // the next byte continues this run iff its flag says so (an item start never does: the item ends here)
      const u32 nb_ = (k == 15) ? nextb : (((eqmask >> (k + 1)) & 1) ? ch : 256u);
      bool last = (jj == 254);
      if (q == (i64)p.W - 1) last = last || (p.is_final != 0);
      else last = last || (nb_ != ch);
      if (q == tile_last && !last && jj >= 3) {
         const int slot = (jj == 3) ? (int)El + 1 : (int)El - 1;
         if (slot >= 0) s_open = slot;
      }
      if (jj < 3) {
         s_enc[mis + El] = (u8)ch;
         if (last) s_cend[mis + El] = 1;
         El += 1;
      } else if (jj == 3) {
         s_enc[mis + El] = (u8)ch;
         if (last) { s_enc[mis + El + 1] = 0; s_cend[mis + El + 1] = 1; }
         El += 2;
      } else if (last) {
         if (El > 0) { s_enc[mis + El - 1] = (u8)(jj - 3); s_cend[mis + El - 1] = 1; }
         else if (tb > 0) {
            // the count byte lives in an earlier tile's output (that tile left it open).  tb == 0 only in a shard
            // scan that starts inside a run past its fourth byte: the byte belongs to the previous shard's
            // encoding, and no block can start before offset 0 here
            if (wr) p.enc[tb - 1] = (u8)(jj - 3);
            p.cend[tb - 1] = 1;
         }
      }
   }
   __syncthreads();
   {
      const int open = s_open >= 0 ? (int)mis + s_open : -1;
      u8* const gc = p.cend + (tb - mis);
      u8* const ge = wr ? p.enc + (tb - mis) : nullptr;
      for (u32 g = threadIdx.x; g * 16 < nst; g += S1_THREADS) {
         const u32 s0 = g * 16;
         const u32 lo = max(s0, mis), hi = min(s0 + 16, nst);
         const bool full = (lo == s0) && (hi == s0 + 16) && !(open >= (int)s0 && open < (int)s0 + 16);
         if (full) {
            *reinterpret_cast<uint4*>(gc + s0) = *reinterpret_cast<const uint4*>(s_cend + s0);
            if (wr) *reinterpret_cast<uint4*>(ge + s0) = *reinterpret_cast<const uint4*>(s_enc + s0);
         } else {
            for (u32 x = lo; x < hi; x++) {
               if ((int)x == open) continue;
               gc[x] = s_cend[x];
               if (wr) ge[x] = s_enc[x];
            }
         }
      }
   }
}

// Segmented scan of tile aggregates: carry[t] = run length ending just before tile t.
__global__ void __launch_bounds__(1024) k_scan_runs(const u32* tile_len, const u32* tile_ext, u32* carry, u32 ntiles, u32 carry0)
{
   __shared__ RunAgg wsm[32];
   __shared__ RunAgg s_run;
   if (threadIdx.x == 0) { s_run.len = carry0; s_run.ext = 1; }
   __syncthreads();
   const u32 l = lane_id(), w = threadIdx.x >> 5;
   for (u32 base = 0; base < ntiles; base += 1024) {
      u32 t = base + threadIdx.x;
      RunAgg v; v.len = 0; v.ext = 1;
      if (t < ntiles) { v.len = tile_len[t]; v.ext = tile_ext[t]; }
      RunAgg inc = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
         RunAgg q;
         q.len = __shfl_up_sync(FULL, inc.len, d);
         q.ext = __shfl_up_sync(FULL, inc.ext, d);
         if (l >= (u32)d) inc = run_comb(q, inc);
      }
      if (l == 31) wsm[w] = inc;
      __syncthreads();
      RunAgg pre = s_run;
      for (u32 k = 0; k < w; k++) pre = run_comb(pre, wsm[k]);
      RunAgg ex;
      ex.len = __shfl_up_sync(FULL, inc.len, 1);
      ex.ext = __shfl_up_sync(FULL, inc.ext, 1);
      if (l == 0) { ex.len = 0; ex.ext = 1; }
      RunAgg mine = run_comb(pre, ex);            // aggregate of everything before tile t
      if (t < ntiles) carry[t] = mine.len;        // valid as "run ending before t" because position-level len counts the trailing run
      __syncthreads();
      if (threadIdx.x == 1023) s_run = run_comb(pre, inc);
      __syncthreads();
   }
}

// Exclusive scan of a u32 array by one CTA; total -> *total_out.
__global__ void __launch_bounds__(1024) k_scan_u32(const u32* in, u32* out, u32 n, u32* total_out)
{
   __shared__ u32 ssm[34];
   __shared__ u32 s_run;
   if (threadIdx.x == 0) s_run = 0;
   __syncthreads();
   for (u32 base = 0; base < n; base += 1024) {
      u32 t = base + threadIdx.x;
      u32 v = (t < n) ? in[t] : 0;
      u32 tot;
      u32 ex = block_excl_sum<1024>(v, ssm, &tot);
      if (t < n) out[t] = s_run + ex;
      __syncthreads();
      if (threadIdx.x == 0) s_run += tot;
      __syncthreads();
   }
   if (threadIdx.x == 0 && total_out) *total_out = s_run;
}

// Greedy block chain (bzlib.c:227 loop condition + :383): one warp.
// scalars: [0]=nb  [1]=enc_used (X[nb])  [2]=enc_total (in)
__global__ void k_chain(const u8* cend, u32* X, u32* scalars, u32 nmax, u32 is_final, u32 tail_merge, u32 blk_cap)
{
   const u32 l = lane_id();
   const u32 Etot = scalars[2];
   u32 x = 0, nb = 0;
   if (l == 0) X[0] = 0;
   while (x < Etot && nb < blk_cap) {
      u32 target = x + nmax - 1;
      if (target >= Etot) {
         if (is_final) { nb++; if (l == 0) X[nb] = Etot; x = Etot; }
         break;
      }
      u32 e = target + l;
      bool f = (l < 8) && (e < Etot) && (cend[e] != 0);
      u32 m = __ballot_sync(FULL, f);
      if (m == 0) {
         if (is_final) { nb++; if (l == 0) X[nb] = Etot; x = Etot; }
         break;
      }
      u32 nx = target + (u32)(__ffs(m) - 1) + 1;
      if (is_final && tail_merge && Etot - nx == 1) nx = Etot;
      nb++;
      if (l == 0) X[nb] = nx;
      x = nx;
   }
   if (l == 0) { scalars[0] = nb; scalars[1] = x; }
}

// ---- CRC ------------------------------------------------------------------
__device__ __forceinline__ u32 gf_mulmod(u32 a, u32 b)
{
   // (a * b) mod P over GF(2), P = x^32 + 0x04C11DB7; polynomials MSB = highest degree
   u32 r = 0;
#pragma unroll 4
   for (int i = 31; i >= 0; i--) {
      r = (r << 1) ^ ((r & 0x80000000u) ? 0x04C11DB7u : 0u);
      if ((b >> i) & 1) r ^= a;
   }
   return r;
}
// x^(8*m) mod P by square-and-multiply over the precomputed table pw[k] = x^(8*2^k)
__device__ __forceinline__ u32 gf_xpow8(const u32* pw, u64 m)
{
   u32 r = 1;                                    // the polynomial "1"
   bool first = true;
   for (int k = 0; m; k++, m >>= 1) {
      if (m & 1) { r = first ? pw[k] : gf_mulmod(r, pw[k]); first = false; }
   }
   return r;
}

constexpr int CRC_THREADS = 256;
constexpr int CRC_CTAS_PER_BLOCK = 16;

__global__ void __launch_bounds__(CRC_THREADS) k_crc(const u8* in, const u32* P, u32* crc_acc, const u32* nb_dev)
{
   if (blockIdx.y >= *nb_dev) return;                // grid sized by an upper bound of the block count
   __shared__ u32 tab[4][256];       // slicing-by-4: tab[k][b] = crc0 of byte b followed by k zero bytes
   __shared__ u32 pw[40];
   __shared__ u32 red[CRC_THREADS];
   {
      u32 r = threadIdx.x << 24;
#pragma unroll
      for (int k = 0; k < 8; k++) r = (r & 0x80000000u) ? (r << 1) ^ 0x04C11DB7u : (r << 1);
      tab[0][threadIdx.x] = r;
   }
   __syncthreads();
   for (int k = 1; k < 4; k++) {
      const u32 v = tab[k - 1][threadIdx.x];
      tab[k][threadIdx.x] = (v << 8) ^ tab[0][v >> 24];
      __syncthreads();
   }
   if (threadIdx.x == 0) {
      u32 v = 0x100;                              // x^8
      // x^8 as a degree-<32 polynomial is the value 1<<8
      for (int k = 0; k < 40; k++) { pw[k] = v; v = gf_mulmod(v, v); }
   }
   __syncthreads();
   const u32 b = blockIdx.y;
   const u64 lo_b = P[b], hi_b = P[b + 1];
   const u64 L = hi_b - lo_b;
   const u64 per_cta = (L + CRC_CTAS_PER_BLOCK - 1) / CRC_CTAS_PER_BLOCK;
   const u64 lo = lo_b + per_cta * blockIdx.x;
   u64 hi = lo + per_cta; if (hi > hi_b) hi = hi_b;
   if (lo >= hi_b) return;
   // right-aligned pieces of size s
   const u64 len = hi - lo;
   const u64 s = (len + CRC_THREADS - 1) / CRC_THREADS;
   const i64 pe = (i64)hi - (i64)(CRC_THREADS - 1 - threadIdx.x) * (i64)s;   // piece end
   i64 ps = pe - (i64)s;                                                      // piece start
   if (ps < (i64)lo) ps = (i64)lo;
   u32 c = 0;
   i64 q = ps;
   for (; q < pe && ((uintptr_t)(in + q) & 3); q++) c = (c << 8) ^ tab[0][(c >> 24) ^ in[q]];
   for (; q + 4 <= pe; q += 4) {
      const u32 w = *reinterpret_cast<const u32*>(in + q);          // little-endian load: first byte is the low one
      const u32 x = c ^ __byte_perm(w, 0, 0x0123);
      c = tab[3][x >> 24] ^ tab[2][(x >> 16) & 0xff] ^ tab[1][(x >> 8) & 0xff] ^ tab[0][x & 0xff];
   }
   for (; q < pe; q++) c = (c << 8) ^ tab[0][(c >> 24) ^ in[q]];
   red[threadIdx.x] = c;
   __syncthreads();
   // tree combine: v[t] = v[t] * x^(8*s*2^k) ^ v[t + 2^k]
   u32 mult = gf_xpow8(pw, s);
   for (int st = 1; st < CRC_THREADS; st <<= 1) {
      if ((threadIdx.x & (2 * st - 1)) == 0) {
         u32 a = red[threadIdx.x], bb = red[threadIdx.x + st];
         red[threadIdx.x] = gf_mulmod(a, mult) ^ bb;
      }
      mult = gf_mulmod(mult, mult);
      __syncthreads();
   }
   if (threadIdx.x == 0) {
      u32 v = red[0];
      u64 after = hi_b - hi;
      if (after) v = gf_mulmod(v, gf_xpow8(pw, after));
      if (blockIdx.x == 0) v ^= gf_mulmod(0xFFFFFFFFu, gf_xpow8(pw, L));   // the init value shifted through L bytes
      atomicXor(&crc_acc[b], v);
   }
}

__global__ void k_crc_final(u32* crc, const u32* scalars)
{
   const u32 nb = scalars[0];
   u32 b = blockIdx.x * blockDim.x + threadIdx.x;
   if (b < nb) crc[b] = ~crc[b];
}

// input bytes consumed by the window's complete blocks, next to the other scalars the host reads
__global__ void k_s1_consumed(const u32* P, u32* scalars)
{
   const u32 nb = scalars[0];
   scalars[3] = nb ? P[nb] : 0;
}

// ---- fast split of run-free windows ----------------------------------------------------------------
// When several engines work on one stream of data, the next engine can start only when this window's end -- its last
// block boundary -- is known; at eight GPUs that hand-over is the critical path of the whole job (one per 100 MB).
// For a window without any run of four or more equal bytes the RLE1 output IS the input, a chunk ends wherever the
// next byte differs, and the boundary chain of k_chain can be walked on the raw input long before the tiles have been
// scanned, counted and scattered: one streaming test (k_has_run4), one warp (k_chain_raw).  The result is checked
// against the full computation afterwards; windows with longer runs take the normal path.
__global__ void __launch_bounds__(256) k_has_run4(const u8* in, u32 W, u32* flag)
{
   const u64 q0 = ((u64)blockIdx.x * 256 + threadIdx.x) * 16;
   // bytes q0-3 .. q0+15: a run of four ends at q iff in[q-3..q] are equal
   u32 run = 1;
   bool hit = false;
   u32 prev = (q0 >= 3 && q0 - 3 < W) ? in[q0 - 3] : 256u;
   for (int k = -2; k < 16 && q0 < W; k++) {
      const i64 q = (i64)q0 + k;
      if (q < 0 || q >= (i64)W) { prev = 256u; run = 1; continue; }
      const u32 c = in[q];
      run = (c == prev) ? run + 1 : 1;
      prev = c;
      if (run >= 4) hit = true;
   }
   if (__any_sync(FULL, hit) && lane_id() == 0) atomicOr(flag, 1u);
}

// k_chain on the raw input of a NON-FINAL window without runs of four: out[0] = flag, out[1] = consumed, out[2] = blocks
__global__ void k_chain_raw(const u8* in, u32 W, u32 nmax, u32 blk_cap, const u32* flag, u32* out)
{
   const u32 l = lane_id();
   if (*flag) { if (l == 0) { out[0] = 1; out[1] = 0; out[2] = 0; } return; }
   u32 x = 0, nb = 0;
   while (x < W && nb < blk_cap) {
      const u32 target = x + nmax - 1;
      if (target >= W) break;
      const u32 e = target + l;
      const bool f = (l < 8) && (e + 1 < W) && (in[e + 1] != in[e]);      // a chunk ends where the next byte differs
      const u32 m = __ballot_sync(FULL, f);
      if (m == 0) break;
      x = target + (u32)(__ffs(m) - 1) + 1;
      nb++;
   }
   if (l == 0) { out[0] = 0; out[1] = x; out[2] = nb; }
}

int stage1_run(Engine* e, const u8* d_in, u32 W, bool is_final, bool tail_merge,
               u32* nb_out, u32* consumed_out, u32* enc_total_out)
{
   // With several engines on one stream of data (multi.cu) the next engine cannot start its window before this
   // stage has fixed where the window ends, so the stage runs on a high-priority stream when the engine has one:
   // its CTAs are scheduled ahead of the sorts of the other windows in flight on the same GPU.
   cudaStream_t st = e->s1_stream ? e->s1_stream : e->stream;
   if (e->s1_stream) {
      BZ_CUDA(e, cudaEventRecord(e->ev_s1, e->stream));           // after the window's input copy / output clear
      BZ_CUDA(e, cudaStreamWaitEvent(st, e->ev_s1, 0));
   }
   const u32 align = (u32)((uintptr_t)d_in & 15);
   const u32 ntiles = (W + align + S1_TILE - 1) / S1_TILE;
   S1Params p;
   p.in = d_in; p.W = W; p.is_final = is_final ? 1 : 0;
   p.tile_len = e->tile_len; p.tile_ext = e->tile_ext; p.tile_carry = e->tile_carry;
   p.tile_size = e->tile_size; p.tile_base = e->tile_base;
   p.enc = e->enc; p.cend = e->cend; p.X = e->bt.X; p.P = e->bt.P; p.nb_find = 0; p.scalars = e->s1_scalars;
   p.prev_byte = 256; p.carry0 = 0; p.Q = nullptr; p.EQ = nullptr; p.seams = nullptr; p.nseams = 0;

   // One host round trip per window: everything below is sized by upper bounds (RLE1 grows the data by at most 5/4,
   // a block holds at least nmax encoded bytes) and reads the actual counts from device memory.
   const u32 Eub = W + W / 4 + 64;
   u32 nb_ub = Eub / e->nmax + 2;
   if (nb_ub > e->blk_cap) nb_ub = e->blk_cap;
   if (Eub > e->enc_cap) { snprintf(e->err, sizeof e->err, "window %u too large for the engine (capacity %u)", W, e->win_cap); return -3; }
   p.nb_find = 1;
   const bool fast = e->s1_early && !is_final && W > 4u * e->nmax;
   if (fast) {
      BZ_CUDA(e, cudaMemsetAsync(e->s1_scalars + 8, 0, 4 * sizeof(u32), st));
      k_has_run4<<<(W / 16 + 256) / 256, 256, 0, st>>>(d_in, W, e->s1_scalars + 8);        BZ_KCHECK(e);
      k_chain_raw<<<1, 32, 0, st>>>(d_in, W, e->nmax, e->blk_cap, e->s1_scalars + 8, e->s1_scalars + 9); BZ_KCHECK(e);
      BZ_CUDA(e, cudaMemcpyAsync(e->h_scalars + 16, e->s1_scalars + 9, 3 * sizeof(u32), cudaMemcpyDeviceToHost, st));
      BZ_CUDA(e, cudaEventRecord(e->ev_fast, st));
   }
   k_tile<S1_AGG><<<ntiles, S1_THREADS, 0, st>>>(p);                                   BZ_KCHECK(e);
   k_scan_runs<<<1, 1024, 0, st>>>(e->tile_len, e->tile_ext, e->tile_carry, ntiles, 0);   BZ_KCHECK(e);
   k_tile<S1_COUNT><<<ntiles, S1_THREADS, 0, st>>>(p);                                 BZ_KCHECK(e);
   k_scan_u32<<<1, 1024, 0, st>>>(e->tile_size, e->tile_base, ntiles, e->s1_scalars + 2); BZ_KCHECK(e);
   BZ_CUDA(e, cudaMemsetAsync(e->cend, 0, (size_t)Eub + 16, st));
   k_tile<S1_SCATTER><<<ntiles, S1_THREADS, 0, st>>>(p);                               BZ_KCHECK(e);
   k_chain<<<1, 32, 0, st>>>(e->cend, e->bt.X, e->s1_scalars, e->nmax, is_final ? 1 : 0, tail_merge ? 1 : 0, e->blk_cap); BZ_KCHECK(e);
   BZ_CUDA(e, cudaMemsetAsync(e->bt.P, 0, sizeof(u32), st));
   k_tile<S1_FIND><<<nb_ub, S1_THREADS, 0, st>>>(p);                                   BZ_KCHECK(e);
   k_s1_consumed<<<1, 1, 0, st>>>(e->bt.P, e->s1_scalars);                             BZ_KCHECK(e);
   BZ_CUDA(e, cudaMemcpyAsync(e->h_scalars, e->s1_scalars, 4 * sizeof(u32), cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaEventRecord(e->ev_s1, st));
   // the block CRCs are not needed to place the next window: they run behind the round trip
   BZ_CUDA(e, cudaMemsetAsync(e->bt.crc, 0, sizeof(u32) * nb_ub, st));
   k_crc<<<dim3(CRC_CTAS_PER_BLOCK, nb_ub), CRC_THREADS, 0, st>>>(d_in, e->bt.P, e->bt.crc, e->s1_scalars); BZ_KCHECK(e);
   k_crc_final<<<(nb_ub + 255) / 256, 256, 0, st>>>(e->bt.crc, e->s1_scalars);            BZ_KCHECK(e);
   if (e->s1_stream) {
      BZ_CUDA(e, cudaEventRecord(e->ev_s1b, st));                 // the later stages follow on the engine's stream
      BZ_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_s1b, 0));
   }
   u32 fast_cons = 0;
   if (fast) {
      BZ_CUDA(e, cudaEventSynchronize(e->ev_fast));
      if (e->h_scalars[16] == 0 && e->h_scalars[17] != 0) {
         fast_cons = e->h_scalars[17];
         e->s1_early(e, fast_cons);                          // the next engine starts its window now
         e->s1_early_done = true;
      }
   }
   BZ_CUDA(e, cudaEventSynchronize(e->ev_s1));
   if (fast_cons && (e->h_scalars[0] == 0 || e->h_scalars[3] != fast_cons)) {
      snprintf(e->err, sizeof e->err, "fast block split disagrees with the full one (%u vs %u)", fast_cons, e->h_scalars[3]);
      return -6;
   }
   const u32 nb = e->h_scalars[0];
   *nb_out = nb; *enc_total_out = e->h_scalars[1];
   *consumed_out = nb ? e->h_scalars[3] : 0;
   return 0;
}

// ---- batch windows: many independent inputs, each its own stream ---------------------------------
// k_chain's walk, one warp per item, over the item's encoded range [enc[i], enc[i+1]) as a final range (every item is a
// whole stream).  COUNT: the item's block count -> cnt[i] and the largest block -> scalars[5].  WRITE: block ends -> X
// from the item's first block (first[] = exclusive scan of cnt); item 0 also publishes the window's block count.
template <bool WRITE>
__global__ void __launch_bounds__(256) k_chain_items(const u8* cend, const u32* enc, u32 n_items, u32* scalars, u32 nmax,
                                                     u32 tail_merge, u32* cnt, const u32* first, u32* X)
{
   const u32 l = lane_id();
   const u32 i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
   if (i >= n_items) return;
   const u32 Etot = scalars[2];
   const u32 Ee = (i + 1 < n_items) ? enc[i + 1] : Etot;
   u32 x = enc[i], nb = 0, mx = 0;
   const u32 base = WRITE ? first[i] : 0;
   if (WRITE && i == 0 && l == 0) { X[0] = 0; scalars[0] = first[n_items]; scalars[1] = Etot; }
   while (x < Ee) {
      const u32 target = x + nmax - 1;
      u32 nx = Ee;
      if (target < Ee) {
         const u32 e = target + l;
         const bool f = (l < 8) && (e < Ee) && (cend[e] != 0);
         const u32 m = __ballot_sync(FULL, f);
         if (m) {
            nx = target + (u32)(__ffs(m) - 1) + 1;
            if (tail_merge && Ee - nx == 1) nx = Ee;
         }
      }
      nb++;
      if (WRITE && l == 0) X[base + nb] = nx;
      mx = max(mx, nx - x);
      x = nx;
   }
   if (!WRITE && l == 0) { cnt[i] = nb; if (mx) atomicMax(&scalars[5], mx); }
}

// Stage 1 of a batch window: e->it.start[0, n_items) holds the window-relative item starts.  Blocks never cross an item
// start; X, P and crc come out as for a single stream, and it.first[i] is item i's first block.
int stage1_items_run(Engine* e, const u8* d_in, u32 W, u32 n_items, u32 nb_ub, bool tail_merge,
                     u32* nb_out, u32* enc_total_out, u32* max_blk_out)
{
   cudaStream_t st = e->stream;
   const u32 align = (u32)((uintptr_t)d_in & 15);
   const u32 ntiles = (W + align + S1_TILE - 1) / S1_TILE;
   const u32 Eub = W + W / 4 + 64;
   if (Eub > e->enc_cap || nb_ub > e->blk_cap || n_items == 0 || n_items > e->blk_cap) {
      snprintf(e->err, sizeof e->err, "batch window too large for the engine (%u bytes, %u items)", W, n_items);
      return -3;
   }
   S1Params p;
   p.in = d_in; p.W = W; p.is_final = 1;
   p.tile_len = e->tile_len; p.tile_ext = e->tile_ext; p.tile_carry = e->tile_carry;
   p.tile_size = e->tile_size; p.tile_base = e->tile_base;
   p.enc = e->enc; p.cend = e->cend; p.X = e->bt.X; p.P = e->bt.P; p.nb_find = 1; p.scalars = e->s1_scalars;
   p.prev_byte = 256; p.carry0 = 0; p.Q = e->it.start; p.EQ = e->it.enc;
   p.seams = e->it.start; p.nseams = n_items;
   BZ_CUDA(e, cudaMemsetAsync(e->s1_scalars + 5, 0, sizeof(u32), st));
   k_tile<S1_AGG><<<ntiles, S1_THREADS, 0, st>>>(p);                                   BZ_KCHECK(e);
   k_scan_runs<<<1, 1024, 0, st>>>(e->tile_len, e->tile_ext, e->tile_carry, ntiles, 0);   BZ_KCHECK(e);
   k_tile<S1_COUNT><<<ntiles, S1_THREADS, 0, st>>>(p);                                 BZ_KCHECK(e);
   k_scan_u32<<<1, 1024, 0, st>>>(e->tile_size, e->tile_base, ntiles, e->s1_scalars + 2); BZ_KCHECK(e);
   BZ_CUDA(e, cudaMemsetAsync(e->cend, 0, (size_t)Eub + 16, st));
   k_tile<S1_SCATTER><<<ntiles, S1_THREADS, 0, st>>>(p);                               BZ_KCHECK(e);
   k_tile<S1_LOCATE><<<n_items, S1_THREADS, 0, st>>>(p);                               BZ_KCHECK(e);
   const u32 cgrid = (n_items + 7) / 8;
   k_chain_items<false><<<cgrid, 256, 0, st>>>(e->cend, e->it.enc, n_items, e->s1_scalars, e->nmax, tail_merge ? 1 : 0,
                                               e->it.cnt, nullptr, nullptr);        BZ_KCHECK(e);
   k_scan_u32<<<1, 1024, 0, st>>>(e->it.cnt, e->it.first, n_items, e->it.first + n_items); BZ_KCHECK(e);
   k_chain_items<true><<<cgrid, 256, 0, st>>>(e->cend, e->it.enc, n_items, e->s1_scalars, e->nmax, tail_merge ? 1 : 0,
                                              nullptr, e->it.first, e->bt.X);       BZ_KCHECK(e);
   BZ_CUDA(e, cudaMemsetAsync(e->bt.P, 0, sizeof(u32), st));
   k_tile<S1_FIND><<<nb_ub, S1_THREADS, 0, st>>>(p);                                   BZ_KCHECK(e);
   BZ_CUDA(e, cudaMemcpyAsync(e->h_scalars, e->s1_scalars, 6 * sizeof(u32), cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaEventRecord(e->ev_s1, st));
   BZ_CUDA(e, cudaMemsetAsync(e->bt.crc, 0, sizeof(u32) * nb_ub, st));
   k_crc<<<dim3(CRC_CTAS_PER_BLOCK, nb_ub), CRC_THREADS, 0, st>>>(d_in, e->bt.P, e->bt.crc, e->s1_scalars); BZ_KCHECK(e);
   k_crc_final<<<(nb_ub + 255) / 256, 256, 0, st>>>(e->bt.crc, e->s1_scalars);            BZ_KCHECK(e);
   BZ_CUDA(e, cudaEventSynchronize(e->ev_s1));
   *nb_out = e->h_scalars[0]; *enc_total_out = e->h_scalars[1]; *max_blk_out = e->h_scalars[5];
   return 0;
}

// ---- shard scan (multi-GPU sharding of one stream by block, SURVEY 8e) ---------------------------
// The chunk structure of a shard (cend flags, encoded offsets) does not depend on where blocks
// start, so every GPU can build it in parallel; only the greedy walk from the previous GPU's last
// boundary is serial, and that walk is one dependent load per block.
__global__ void k_chain_from(const u8* cend, const u32* scal_in, u32* out, u32 nmax, u32 input_ends, u32 tail_merge)
{
   // scal_in[0] = encoded offset of the start boundary, [1] = encoded offset of the limit, [2] = total
   const u32 l = lane_id();
   const u32 Etot = scal_in[2];
   const u32 xlim = scal_in[1];
   u32 x = scal_in[0];
   u32 nblk = 0;
   while (x < xlim) {
      const u32 target = x + nmax - 1;
      if (target >= Etot) { x = input_ends ? Etot : 0xffffffffu; nblk++; break; }
      const u32 e = target + l;
      const bool f = (l < 8) && (e < Etot) && (cend[e] != 0);
      const u32 m = __ballot_sync(FULL, f);
      if (m == 0) { x = input_ends ? Etot : 0xffffffffu; nblk++; break; }
      u32 nx = target + (u32)(__ffs(m) - 1) + 1;
      if (input_ends && tail_merge && Etot - nx == 1) nx = Etot;
      x = nx; nblk++;
   }
   if (l == 0) { out[0] = x; out[1] = nblk; }
}

int scan_build(ScanState* s, u32 prev_byte, u32 carry0)
{
   cudaStream_t st = s->st;
   const u32 align = (u32)((uintptr_t)s->in & 15);
   s->ntiles = (s->W + align + S1_TILE - 1) / S1_TILE;
   S1Params p;
   memset(&p, 0, sizeof p);
   p.in = s->in; p.W = s->W; p.is_final = s->input_ends;
   p.tile_len = s->tile_len; p.tile_ext = s->tile_ext; p.tile_carry = s->tile_carry;
   p.tile_size = s->tile_size; p.tile_base = s->tile_base;
   p.enc = nullptr; p.cend = s->cend; p.scalars = s->scal;
   p.prev_byte = prev_byte; p.carry0 = carry0;
   const bool dbg = getenv("BZ2_B200_DEBUG_SYNC") != nullptr;
#define SCAN_DBG(name) do { if (dbg) { cudaError_t c_ = cudaStreamSynchronize(st); if (c_ == cudaSuccess) c_ = cudaGetLastError(); \
      if (c_ != cudaSuccess) { fprintf(stderr, "[bz2b200] scan %s: %s\n", name, cudaGetErrorString(c_)); return -1; } } } while (0)
   SCAN_DBG("entry");
   k_tile<S1_AGG><<<s->ntiles, S1_THREADS, 0, st>>>(p);                                           SCAN_DBG("k_tile<AGG>");
   k_scan_runs<<<1, 1024, 0, st>>>(s->tile_len, s->tile_ext, s->tile_carry, s->ntiles, carry0);   SCAN_DBG("k_scan_runs");
   k_tile<S1_COUNT><<<s->ntiles, S1_THREADS, 0, st>>>(p);                                         SCAN_DBG("k_tile<COUNT>");
   k_scan_u32<<<1, 1024, 0, st>>>(s->tile_size, s->tile_base, s->ntiles, s->scal + 2);           SCAN_DBG("k_scan_u32");
   if (cudaMemcpyAsync(s->h_scal, s->scal, 4 * sizeof(u32), cudaMemcpyDeviceToHost, st) != cudaSuccess) return -1;
   if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
   s->enc_total = s->h_scal[2];
   if ((u64)s->enc_total + 16 > s->cend_cap) return -2;
   if (cudaMemsetAsync(s->cend, 0, (size_t)s->enc_total + 16, st) != cudaSuccess) return -1;
   k_tile<S1_SCATTER><<<s->ntiles, S1_THREADS, 0, st>>>(p);                                       SCAN_DBG("k_tile<SCATTER>");
#undef SCAN_DBG
   if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
   return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// first block boundary >= limit when blocks are laid greedily from the boundary `start`
int scan_boundary(ScanState* s, u32 start, u32 limit, u32 tail_merge, u32* boundary, u32* nblocks)
{
   cudaStream_t st = s->st;
   S1Params p;
   memset(&p, 0, sizeof p);
   p.in = s->in; p.W = s->W; p.is_final = s->input_ends;
   p.tile_len = s->tile_len; p.tile_ext = s->tile_ext; p.tile_carry = s->tile_carry;
   p.tile_size = s->tile_size; p.tile_base = s->tile_base;
   p.enc = nullptr; p.cend = s->cend; p.scalars = s->scal;
   p.prev_byte = s->prev_byte; p.carry0 = s->carry0;
   p.Q = s->q; p.EQ = s->scal + 4;            // scal[4] = E(start), scal[5] = E(limit)
   s->h_scal[8] = start; s->h_scal[9] = limit;
   if (cudaMemcpyAsync(s->q, s->h_scal + 8, 2 * sizeof(u32), cudaMemcpyHostToDevice, st) != cudaSuccess) return -1;
   k_tile<S1_LOCATE><<<2, S1_THREADS, 0, st>>>(p);
   // chain input: [0]=E(start) [1]=E(limit) [2]=total  -> reuse scal+4.. as a 3-vector
   if (cudaMemcpyAsync(s->scal + 6, s->scal + 2, sizeof(u32), cudaMemcpyDeviceToDevice, st) != cudaSuccess) return -1;
   k_chain_from<<<1, 32, 0, st>>>(s->cend, s->scal + 4, s->scal + 10, s->nmax, s->input_ends, tail_merge);
   // boundary (encoded) -> input position through the FIND mode: X[1] = scal[10]
   p.X = s->scal + 9; p.P = s->scal + 12;      // X[1] = scal[10]; P[1] = scal[13]
   k_tile<S1_FIND><<<1, S1_THREADS, 0, st>>>(p);
   if (cudaMemcpyAsync(s->h_scal, s->scal, 16 * sizeof(u32), cudaMemcpyDeviceToHost, st) != cudaSuccess) return -1;
   if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
   if (cudaGetLastError() != cudaSuccess) return -1;
   if (s->h_scal[10] == 0xffffffffu) return -3;         // ran off the data before reaching the limit: halo too small
   *boundary = s->h_scal[13];
   *nblocks = s->h_scal[11];
   return 0;
}

} // namespace bz
