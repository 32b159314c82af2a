// stage2_bwt.cu -- S2: Burrows-Wheeler transform of every block of a window.
//
// Replaces BZ2_blockSort and everything under it (reference blocksort.c:1534-1545,
// divsufsort :1503-1514, sort_typeBstar :1314-1437, ss_* :83-664, tr_* / ls_* :669-1309,
// construct_SA :1439-1501).  Same contract: rotations of the block in lexicographic
// order; output byte k is the byte preceding rotation k; origPtr is the rank of
// rotation 0.  The method is not the reference's (induced sorting is serial):
//
//   1. k-gram bucket sort   the first k symbols of every rotation, packed in base-`ninuse` notation, select one
//                           of up to 2^18 buckets per block (text: k = 3, bytes: k = 2, a binary alphabet: k = 18);
//                           one atomic pass keeps each rotation's arrival index, a scan and a placement pass
//                           follow.  The placement pass also writes K[i], the next m symbols of i in <= 51 bits.
//   2. round 0              every bucket ("segment") is sorted by the text key K[i+k]: depth k -> k+m.
//   3. prefix doubling      every unresolved segment is sorted by the rank of the rotation d further on (cyclic),
//                           d = current depth; equal keys stay one segment.  Ranks are tagged two-generation words
//                           updated in place (rk_pack).  Segments are handled by size class, all blocks of the
//                           window in the same launch, the classes of a round on side streams:
//                             2..32       sub-warp bitonic network in registers        (k_refine_small)
//                             33..512     warp / 64-thread CTA, packed-word bitonic    (k_refine_medium)
//                             513..8192   CTA-resident LSD radix sort in shared memory (k_refine_radix)
//                             > 8192      one CTA, LSD radix passes through HBM        (k_refine_large)
//   4. shortcuts            tandem repeats resolved in one step (2d, k_resolve_periodic); long non-tandem repeats
//                           followed to their end by position-indexed scans while refinement stalls (2e, k_rep_*).
//   5. last column          bwt[k] = T[(sa[k]-1) mod n]; origPtr = rank of rotation 0 (k_bwt_out; exact powers: stage2_tie.cu).
//
// A segment that survives to depth >= n holds equal rotations: the block is an exact
// power u^q; q is recorded in power_q[b] (the BWT bytes do not depend on their order).
#include "engine.h"
#include <stdlib.h>

namespace bz {

struct ListsDev {
   u32* small_items[N_SMALL_CLASSES];
   u64* big_items[N_BIG_CLASSES];
   u32* counts;
   u32  small_cap[N_SMALL_CLASSES];
   u32  big_cap[N_BIG_CLASSES];
   u32* overflow;
};

struct S2Params {
   const u8* T;
   const u32* X;
   u32 nb;
   u32 b0;                  // first block of the sub-batch being sorted
   u32* sa;
   u64* rank;               // tagged rank words, see rk_pack()
   u32* keyA; u32* keyB; u32* idxB;
   u32* hist;
   u32 hist_stride;         // bins reserved per block
   u8* code;                // [nb*256] dense symbol codes
   u32* kk;                 // [nb] k of the k-gram bucket sort = initial sorted depth
   u32* hh;                 // [nb] k + m: depth after the text-key round
   u32* kbits;              // [nb] m * bits-per-symbol: significant bits of a text key
   u32* ksym;               // [nb] m | bits-per-symbol << 8
   u64* K;                  // [E] packed codes of the next m symbols of every position
   u64* kscrA; u64* kscrB;  // [E] 64-bit key scratch of the large-segment path
   u32 debug;
   u32 kg_agg_alpha;        // count pass aggregates per tile for alphabets up to this size
   u32* nbins;              // [nb] ninuse^k
   const u32* blockmap;
   u32* power_q;
   u8* inuse; u32* ninuse;
   const u32* jd;           // [E] repeat-chain length of every position (rounds that follow chains), else null
   const u32* jq;           // [E] length of the repeat at the block's dominant offset from every position, else null
   const u32* dstar;        // [g] dominant repeat offset of every block of the sub-batch (0 = none)
};

__device__ __forceinline__ int seg_class(u32 len)
{
   if (len <= 32) return 31 - __clz(len - 1);
   if (len <= 256) return CLS_W256;
   if (len > MED_MAX) return CLS_LARGE;
   return CLS_C512 + (23 - __clz(len - 1));     // 257..512 -> +0, ..1024 -> +1, ..2048 -> +2, ..4096 -> +3, ..8192 -> +4
}

// Rank words carry two generations so that a refinement round can update ranks in place while
// other CTAs still need the values the round started with: [tag:16 | old:24 | new:24].  A word
// written in the current round (tag == round tag) is read through `old`, any other through `new`.
__device__ __forceinline__ u64 rk_pack(u32 tag, u32 oldv, u32 newv) { return ((u64)tag << 48) | ((u64)oldv << 24) | (u64)newv; }
__device__ __forceinline__ u32 rk_read(u64 w, u32 tag) { return ((u32)(w >> 48) == tag) ? ((u32)(w >> 24) & 0xffffffu) : ((u32)w & 0xffffffu); }

// All 32 lanes of the warp must call this together.
__device__ __forceinline__ void push_seg(const ListsDev& L, bool valid, u32 pos, u32 blk, u32 len)
{
   const int cls = valid ? seg_class(len) : -1;
   const u32 m = __match_any_sync(FULL, cls);
   const u32 leader = __ffs(m) - 1;
   u32 base = 0;
   if (valid && lane_id() == leader) base = atomicAdd(&L.counts[cls], __popc(m));
   base = __shfl_sync(FULL, base, leader);
   if (valid) {
      const u32 slot = base + __popc(m & lanemask_lt());
      if (cls < N_SMALL_CLASSES) {
         if (slot < L.small_cap[cls]) L.small_items[cls][slot] = pos | ((len - 1) << 27);
         else atomicOr(L.overflow, 1u);
      } else {
         const int c = cls - N_SMALL_CLASSES;
         if (slot < L.big_cap[c]) L.big_items[c][slot] = ((u64)pos << 32) | ((u64)blk << 20) | (u64)len;
         else atomicOr(L.overflow, 1u);
      }
   }
}

__device__ __forceinline__ u32 block_of(const S2Params& p, u32 pos)
{
   u32 b = p.blockmap[pos >> 12];
   while (b + 1 < p.nb && pos >= p.X[b + 1]) b++;
   return b;
}

__global__ void k_blockmap(const u32* X, u32 nb, u32* blockmap, u32 nchunks)
{
   u32 c = blockIdx.x * blockDim.x + threadIdx.x;
   if (c >= nchunks) return;
   u32 pos = c << 12;
   u32 lo = 0, hi = nb - 1;
   while (lo < hi) { u32 mid = (lo + hi + 1) >> 1; if (X[mid] <= pos) lo = mid; else hi = mid - 1; }
   blockmap[c] = lo;
}

// ---- 1. k-gram bucket sort ------------------------------------------------------------
// The first k symbols of every rotation are packed in base-`ninuse` positional notation
// (k = the largest power that keeps ninuse^k within the per-block bin budget), so text
// with 61 symbols starts at depth 3, a binary alphabet at depth 18, full-byte data at 2.
constexpr int KG_THREADS = 256;
constexpr int KG_ITEMS = 16;
constexpr int KG_TILE = KG_THREADS * KG_ITEMS;
constexpr int KG_MAXK = 24;
constexpr u32 KG_TAB_LOG2 = 13;             // per-tile k-gram table of the count pass: 8192 slots for 4096 positions
constexpr u32 KG_TAB = 1u << KG_TAB_LOG2;
constexpr u32 KG_AGG_MAX_ALPHA = 128;       // aggregate per tile for alphabets up to this size (byte-wide data has few repeats per tile)
constexpr u32 KG_AGG_MAX_BINS = 1u << 19;   // ... and bin counts below this: a slot word holds key + 1 in 19 bits above a 13-bit count

enum { KG_HISTOFF = 3, KG_PLACE = 4 };

__global__ void __launch_bounds__(KG_THREADS) k_inuse(S2Params p)
{
   __shared__ u32 flags[256];
   const u32 b = p.b0 + blockIdx.y;
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   const u32 t0 = blockIdx.x * KG_TILE;
   if (t0 >= n) return;
   flags[threadIdx.x] = 0;
   __syncthreads();
   const u8* T = p.T + xb;
#pragma unroll 4
   for (int k = 0; k < KG_ITEMS; k++) {
      const u32 i = t0 + k * KG_THREADS + threadIdx.x;
      if (i < n) flags[T[i]] = 1;
   }
   __syncthreads();
   if (flags[threadIdx.x]) p.inuse[(size_t)b * 256 + threadIdx.x] = 1;
}

// dense symbol codes, alphabet size, k and bin count of every block
__global__ void __launch_bounds__(256) k_codemap(S2Params p)
{
   __shared__ u32 wcnt[8];
   const u32 b = p.b0 + blockIdx.x, tid = threadIdx.x, w = tid >> 5, l = lane_id();
   const bool used = p.inuse[(size_t)b * 256 + tid] != 0;
   const u32 bal = __ballot_sync(FULL, used);
   if (l == 0) wcnt[w] = __popc(bal);
   __syncthreads();
   u32 base = 0, tot = 0;
   for (u32 k = 0; k < 8; k++) { if (k < w) base += wcnt[k]; tot += wcnt[k]; }
   p.code[(size_t)b * 256 + tid] = (u8)(used ? base + __popc(bal & lanemask_lt()) : 0);
   if (tid == 0) {
      p.ninuse[b] = tot;
      u32 k = 1, bins = tot ? tot : 1;
      while (tot > 1 && k < KG_MAXK && (u64)bins * tot <= (u64)p.hist_stride) { bins *= tot; k++; }
      p.kk[b] = k;
      p.nbins[b] = bins;
      u32 bits = 1;
      while ((1u << bits) < tot) bits++;
      u32 m = 51u / bits;                       // 51 key bits + 13 local-index bits fill a packed 64-bit sort word
      if (m > 48u) m = 48u;
      p.hh[b] = k + m;
      p.kbits[b] = m * bits;
      p.ksym[b] = m | (bits << 8);
   }
}

template <int MODE, bool AGG>
__global__ void __launch_bounds__(KG_THREADS) k_kgram(S2Params p)
{
   __shared__ u8 sc[KG_TILE + 64];
   __shared__ u8 cmap[256];
   __shared__ u32 tab[AGG ? KG_TAB : 1];
   const u32 b = p.b0 + blockIdx.y;
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   const u32 t0 = blockIdx.x * KG_TILE;
   if (t0 >= n) return;
   const u8* T = p.T + xb;
   const u32 k = p.kk[b], base = p.ninuse[b];
   if (AGG) for (u32 h = threadIdx.x; h < KG_TAB; h += KG_THREADS) tab[h] = 0;
   u32* hist = p.hist + (size_t)(b - p.b0) * p.hist_stride;
   cmap[threadIdx.x] = p.code[(size_t)b * 256 + threadIdx.x];
   __syncthreads();
   const u32 msym = p.ksym[b] & 255u, mbits = p.ksym[b] >> 8;
   const u32 halo = (MODE == KG_PLACE) ? max(k, msym) : k;
   u32* const koff = reinterpret_cast<u32*>(p.kscrA);
   const u32 span = min((u32)KG_TILE, n - t0) + halo - 1;
   for (u32 s = threadIdx.x; s < span; s += KG_THREADS) {
      u32 gi = t0 + s;
      if (gi >= n) gi = (gi - n < n) ? gi - n : gi % n;
      sc[s] = cmap[T[gi]];
   }
   __syncthreads();
   if (AGG && base <= p.kg_agg_alpha && p.nbins[b] < KG_AGG_MAX_BINS) {
      // Count pass with per-tile aggregation.  10^8 returning global atomics run at the L2's atomic rate (81 G/s, round 1:
      // 1.25 ms per window) -- but on text only ~22 % of the k-grams of a 4096-position tile are distinct.  The tile first
      // counts its k-grams in a shared-memory hash table (slot word = key+1 << 13 | count; an element's arrival index
      // inside the tile is what its shared-memory atomicAdd returns), then issues ONE global atomicAdd per distinct k-gram
      // for the tile's base inside the bucket.  Order inside a bucket stays irrelevant.
      u32 slot_loc[KG_ITEMS];
#pragma unroll
      for (int it = 0; it < KG_ITEMS; it++) {
         const u32 s = it * KG_THREADS + threadIdx.x;
         slot_loc[it] = 0xffffffffu;
         if (t0 + s < n) {
            u32 key = 0;
            for (u32 j = 0; j < k; j++) key = key * base + sc[s + j];
            const u32 tagw = (key + 1u) << 13;
            u32 h = (key * 2654435761u) >> (32 - KG_TAB_LOG2);
            for (;;) {
               u32 cur = tab[h];
               if (cur == 0) cur = atomicCAS(&tab[h], 0u, tagw);
               if (cur == 0 || (cur >> 13) == key + 1u) { slot_loc[it] = (h << 13) | (atomicAdd(&tab[h], 1u) & 0x1fffu); break; }
               h = (h + 1u) & (KG_TAB - 1u);
            }
         }
      }
      __syncthreads();
      for (u32 h = threadIdx.x; h < KG_TAB; h += KG_THREADS) {
         const u32 w = tab[h];
         if (w) tab[h] = atomicAdd(&hist[(w >> 13) - 1u], w & 0x1fffu);
      }
      __syncthreads();
#pragma unroll
      for (int it = 0; it < KG_ITEMS; it++) {
         const u32 s = it * KG_THREADS + threadIdx.x;
         if (slot_loc[it] != 0xffffffffu) koff[xb + t0 + s] = tab[slot_loc[it] >> 13] + (slot_loc[it] & 0x1fffu);
      }
      return;
   }
#pragma unroll 2
   for (int it = 0; it < KG_ITEMS; it++) {
      const u32 s = it * KG_THREADS + threadIdx.x;
      const u32 i = t0 + s;
      if (i < n) {
         u32 key = 0;
         for (u32 j = 0; j < k; j++) key = key * base + sc[s + j];
         if (MODE == KG_HISTOFF) koff[xb + i] = atomicAdd(&hist[key], 1u);          // arrival order inside the bucket
         else {
            const u32 start = hist[key];
            p.rank[xb + i] = rk_pack(0xffffu, 0, start);
            p.sa[xb + start + koff[xb + i]] = i;
            u64 kw = 0;
            for (u32 j = 0; j < msym; j++) kw = (kw << mbits) | (u64)sc[s + j];
            p.K[xb + i] = kw;
         }
      }
   }
}

// exclusive scan of the bucket counts of one block
__global__ void __launch_bounds__(1024) k_kgram_scan(S2Params p)
{
   __shared__ u32 ssm[34];
   __shared__ u32 s_run;
   const u32 b = p.b0 + blockIdx.x;
   u32* hist = p.hist + (size_t)(b - p.b0) * p.hist_stride;
   const u32 nbins = p.nbins[b];
   if (threadIdx.x == 0) s_run = 0;
   __syncthreads();
   for (u32 base = 0; base < nbins; base += 1024 * 16) {
      const u32 lo = base + threadIdx.x * 16;
      u32 v[16], sum = 0;
      if (lo + 16 <= nbins) {
         const uint4* h4 = reinterpret_cast<const uint4*>(hist + lo);
#pragma unroll
         for (int k = 0; k < 4; k++) { uint4 q = h4[k]; v[4 * k] = q.x; v[4 * k + 1] = q.y; v[4 * k + 2] = q.z; v[4 * k + 3] = q.w; }
      } else {
#pragma unroll
         for (int k = 0; k < 16; k++) v[k] = (lo + k < nbins) ? hist[lo + k] : 0;
      }
#pragma unroll
      for (int k = 0; k < 16; k++) sum += v[k];
      u32 tot;
      u32 ex = block_excl_sum<1024>(sum, ssm, &tot) + s_run;
#pragma unroll
      for (int k = 0; k < 16; k++) { if (lo + k < nbins) hist[lo + k] = ex; ex += v[k]; }
      __syncthreads();
      if (threadIdx.x == 0) s_run += tot;
      __syncthreads();
   }
}

// hist[bin] is the start of bucket `bin` (k_kgram_scan); emit the initial segments
__global__ void __launch_bounds__(256) k_seg_init(S2Params p, ListsDev L)
{
   const u32 b = p.b0 + blockIdx.y;
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   const u32* hist = p.hist + (size_t)(b - p.b0) * p.hist_stride;
   const u32 bin = blockIdx.x * 256 + threadIdx.x;
   const bool vbin = bin < p.nbins[b];
   const u32 end = !vbin ? 0 : (bin + 1 < p.nbins[b] ? hist[bin + 1] : n);
   const u32 start = !vbin ? 0 : hist[bin];
   const u32 len = end - start;
   const bool multi = vbin && len >= 2;
   const bool deep = (p.kk[b] >= n);                  // depth k already covers the whole rotation
   if (multi && deep) atomicMax(&p.power_q[b], len);
   push_seg(L, multi && !deep, xb + start, b, len);
}

// ---- 2. refinement rounds --------------------------------------------------------------
// Round 0 (TEXT) sorts every k-gram bucket by the next m symbols taken from the packed text
// keys K[] (depth k -> k+m).  Later rounds sort by the rank of the rotation `shift` further on
// (classic doubling; depth d -> 2d).  Per block: kk = k, hh = k+m.
template <bool TEXT> struct KeyOf { typedef u32 type; };
template <> struct KeyOf<true> { typedef u64 type; };

__device__ __forceinline__ u32 round_shift(const S2Params& p, u32 b, u32 round, u32* depth_after)
{
   const u32 k = p.kk[b];
   if (round == 0) { *depth_after = p.hh[b]; return k; }
   const u32 sft = p.hh[b] << (round - 1);
   *depth_after = 2u * sft;
   return sft;
}

template <bool TEXT>
__device__ __forceinline__ typename KeyOf<TEXT>::type load_key(const S2Params& p, u32 xb, u32 n, u32 idx, u32 shift, u32 tag, u32 ks)
{
   u32 t = idx + shift; if (t >= n) t -= n;
   if (TEXT) return (typename KeyOf<TEXT>::type)p.K[xb + t];        // (keys rebuilt from a 1-byte code text were measured: 3 % slower)
   if (p.jd) { t += p.jd[xb + idx]; if (t >= n) t -= n; }      // key at the end of the segment's repeat chain (2e)
   return (typename KeyOf<TEXT>::type)rk_read(p.rank[xb + t], tag);
}

// ---- 2a. small segments: sub-warp bitonic network, one element per lane --------------------
template <int LANES, typename KT>
__device__ __forceinline__ void small_sort(KT& key, u32& idx, const u32 sub)
{
#pragma unroll
   for (int k = 2; k <= LANES; k <<= 1) {
#pragma unroll
      for (int j = k >> 1; j > 0; j >>= 1) {
         const KT ok = __shfl_xor_sync(FULL, key, j);
         const u32 oi = __shfl_xor_sync(FULL, idx, j);
         const bool asc = ((sub & k) == 0);
         const bool low = ((sub & j) == 0);
         const bool take = (asc == low) ? (ok < key) : (ok > key);
         if (take) { key = ok; idx = oi; }
      }
   }
}

// group boundaries of the sorted lanes, new ranks, next-round segments
template <int LANES, typename KT>
__device__ __forceinline__ void small_finish(const S2Params& p, const ListsDev& Lout, const KT key, const u32 idx, const u32 sub, const bool active,
                                             const u32 len, const u32 pos, const u32 xb, const u32 b, const u32 n, const u32 depth, const u32 round)
{
   const KT pk = __shfl_up_sync(FULL, key, 1);
   const KT nk = __shfl_down_sync(FULL, key, 1);
   const bool head = active && (sub == 0 || pk != key);
   const u32 bal = __ballot_sync(FULL, head);
   const u32 sh = lane_id() & ~(u32)(LANES - 1);
   const u32 mask = (LANES == 32) ? bal : ((bal >> sh) & ((1u << (LANES & 31)) - 1u));
   const u32 below = mask & ((2u << sub) - 1u);
   const u32 gstart = active ? (31 - __clz(below)) : 0;
   const bool is_end = active && (sub == len - 1 || nk != key);
   const u32 size = sub - gstart + 1;
   if (active) {
      p.sa[pos + sub] = idx;
      p.rank[xb + idx] = rk_pack(round + 1, pos - xb, (pos - xb) + gstart);
   }
   const bool multi = is_end && size >= 2;
   const bool deep = (depth >= n);
   if (multi && deep) atomicMax(&p.power_q[b], size);
   push_seg(Lout, multi && !deep, pos + gstart, b, size);
}

template <int LANES, bool TEXT>
__global__ void __launch_bounds__(256) k_refine_small(S2Params p, ListsDev Lout, const u32* items, u32 count, u32 round)
{
   typedef typename KeyOf<TEXT>::type KT;
   const u32 gid = blockIdx.x * blockDim.x + threadIdx.x;
   const u32 seg = gid / LANES;
   const u32 sub = gid % LANES;
   const bool vseg = seg < count;
   const u32 entry = vseg ? items[seg] : 0;
   const u32 pos = entry & 0x7ffffffu;
   const u32 len = (entry >> 27) + 1;
   u32 b = 0, xb = 0, n = 1, shift = 0, depth = 0;
   if (vseg) { b = block_of(p, pos); xb = p.X[b]; n = p.X[b + 1] - xb; shift = round_shift(p, b, round, &depth); }
   const bool active = vseg && sub < len;
   u32 idx = 0, off0 = 0;
   KT key = ~(KT)0;
   if (active) idx = p.sa[pos + sub];
   if (TEXT) {
      if (active) key = load_key<TEXT>(p, xb, n, idx, shift, round + 1, p.ksym[b]);
   } else {
      const u32 head_lane = lane_id() & ~(u32)(LANES - 1);
      const u32 gm = (LANES == 32) ? FULL : (((1u << (LANES & 31)) - 1u) << head_lane);
      u32 off = shift;
      // (a) the segment's chain: every member sees the same length
      if (p.jd && active) off += p.jd[xb + idx];
      if (p.jq) {
         // (b) members that form a progression with the block's dominant repeat offset agree as far as the
         // shortest of their pairwise repeats reaches, and the rank right behind it separates that pair
         const u32 ds = vseg ? p.dstar[b - p.b0] : 0u;
         const u32 nx = idx + ds;                         // not cyclic: a strictly increasing chain cannot close on itself
         bool has = false;
#pragma unroll
         for (int k = 0; k < LANES; k++) {
            const u32 o = __shfl_sync(FULL, idx, head_lane + k);
            has |= ((u32)k < len && o == nx);
         }
         has = has && active && ds != 0 && nx < n;
         const u32 nhas = __popc(__ballot_sync(FULL, has) & gm);
         u32 jm = has ? p.jq[xb + idx] : 0xffffffffu;
#pragma unroll
         for (int d = LANES >> 1; d > 0; d >>= 1) jm = min(jm, __shfl_xor_sync(FULL, jm, d));
         if (vseg && nhas + 1 == len && jm != 0xffffffffu) off = max(off, jm);
      }
      u32 y = 0;
      if (active) {
         y = idx + off;
         if (y >= n) y -= n;
         if (y >= n) y -= n;
         key = (KT)rk_read(p.rank[xb + y], round + 1);
      }
      off0 = off;
   }
   small_sort<LANES, KT>(key, idx, sub);
   if (!TEXT && LANES >= 4 && LANES <= 8 && p.jq) {
      // More keys in the same visit: a group of equal keys that is again a progression with the dominant offset is
      // decided where the shortest of ITS pairwise repeats ends (a triple a, a+p, a+2p loses a+2p to the first key and
      // is finished by the second).  The group index stands for everything compared so far.
      const u32 head_lane = lane_id() & ~(u32)(LANES - 1);
      const u32 ds = vseg ? p.dstar[b - p.b0] : 0u;
      u64 ck = active ? (u64)key : ~(u64)0;
      u32 offc = off0;                                   // what the lane's group agrees on; the group keeps its lanes through every sort
      for (int it = 0; it < LANES - 2; it++) {
         const u64 pk = __shfl_up_sync(FULL, ck, 1);
         const bool head = active && (sub == 0 || pk != ck);
         const u32 bal = __ballot_sync(FULL, head);
         const u32 mask = (bal >> head_lane) & ((1u << LANES) - 1u);
         const u32 gstart = active ? (31 - __clz(mask & ((2u << sub) - 1u))) : 0xffu;
         const u32 nx = idx + ds;
         bool has = false;
#pragma unroll
         for (int k = 0; k < LANES; k++) {
            const u32 oi = __shfl_sync(FULL, idx, head_lane + k);
            const u32 og = __shfl_sync(FULL, gstart, head_lane + k);
            has |= (og == gstart && oi == nx);
         }
         has = has && active && ds != 0 && nx < n;
         const u32 jv = has ? p.jq[xb + idx] : 0xffffffffu;
         u32 size = 0, nh = 0, jm = 0xffffffffu;
#pragma unroll
         for (int k = 0; k < LANES; k++) {
            const u32 og = __shfl_sync(FULL, gstart, head_lane + k);
            const u32 oh = __shfl_sync(FULL, (u32)has, head_lane + k);
            const u32 oj = __shfl_sync(FULL, jv, head_lane + k);
            if (og == gstart) { size++; nh += oh; jm = min(jm, oj); }
         }
         const bool refine = active && size >= 2 && nh + 1 == size && jm != 0xffffffffu && jm > offc;
         if (!__any_sync(FULL, refine)) break;
         u32 k2 = 0;
         if (refine) {
            u32 y = idx + jm; if (y >= n) y -= n;
            k2 = rk_read(p.rank[xb + y], round + 1);
            offc = jm;
         }
         ck = active ? (((u64)gstart << 32) | k2) : ~(u64)0;
         small_sort<LANES, u64>(ck, idx, sub);
      }
      small_finish<LANES, u64>(p, Lout, ck, idx, sub, active, len, pos, xb, b, n, depth, round);
   } else {
      small_finish<LANES, KT>(p, Lout, key, idx, sub, active, len, pos, xb, b, n, depth, round);
   }
}

// ---- 2b. medium segments: bitonic sort of packed (key, local index) words ----------------
// Every thread owns ITEMS = 8 consecutive elements of the sequence in registers.  Compare
// distances below 8 stay inside the thread, distances below 256 go through shuffles and
// only distances >= 256 (other warps) go through shared memory.  The packed word makes a
// compare-exchange a min/max pair.
constexpr int MS_ITEMS = 8;
constexpr int MS_LBITS = 12;              // local index bits packed under the key

template <int THREADS, typename VT>
__device__ __forceinline__ void bitonic_blocked(VT (&v)[MS_ITEMS], const u32 t, const u32 n2, VT* xch)
{
#pragma unroll
   for (int k = 2; k <= THREADS * MS_ITEMS; k <<= 1) {
      if ((u32)k > n2) break;
#pragma unroll
      for (int j = k >> 1; j > 0; j >>= 1) {
         if (j >= MS_ITEMS * 32) {
            // partner lives in another warp
            const u32 tj = (u32)j / MS_ITEMS;
            const bool keep_min = ((((t * MS_ITEMS) & (u32)k) == 0) == ((t & tj) == 0));
            __syncthreads();
#pragma unroll
            for (int r = 0; r < MS_ITEMS; r++) xch[t * MS_ITEMS + r] = v[r];
            __syncthreads();
#pragma unroll
            for (int r = 0; r < MS_ITEMS; r++) {
               const VT o = xch[(t ^ tj) * MS_ITEMS + r];
               v[r] = keep_min ? min(v[r], o) : max(v[r], o);
            }
         } else if (j >= MS_ITEMS) {
            const u32 lj = (u32)j / MS_ITEMS;
            const bool keep_min = ((((t * MS_ITEMS) & (u32)k) == 0) == ((t & lj) == 0));
#pragma unroll
            for (int r = 0; r < MS_ITEMS; r++) {
               const VT o = __shfl_xor_sync(FULL, v[r], lj);
               v[r] = keep_min ? min(v[r], o) : max(v[r], o);
            }
         } else {
#pragma unroll
            for (int r = 0; r < MS_ITEMS; r++) {
               if ((r & j) == 0) {
                  const bool asc = (((t * MS_ITEMS + r) & (u32)k) == 0);
                  const VT lo = min(v[r], v[r | j]), hi = max(v[r], v[r | j]);
                  v[r] = asc ? lo : hi;
                  v[r | j] = asc ? hi : lo;
               }
            }
         }
      }
   }
}

// One segment per group of THREADS threads (THREADS = 32: a warp, no shared memory;
// THREADS >= 64: a CTA).
template <int THREADS, bool TEXT>
__global__ void __launch_bounds__(THREADS == 32 ? 256 : THREADS)
k_refine_medium(S2Params p, ListsDev Lout, const u64* items, u32 count, u32 round)
{
   typedef typename KeyOf<TEXT>::type VT;            // packed word: key << 12 | local
   constexpr int CAP = THREADS * MS_ITEMS;
   constexpr bool WARP = (THREADS == 32);
   __shared__ __align__(16) VT xch[WARP ? 2 : CAP];
   __shared__ u32 ssm[34];
   const u32 t = WARP ? lane_id() : threadIdx.x;
   const u32 seg = WARP ? (blockIdx.x * 8 + (threadIdx.x >> 5)) : blockIdx.x;
   const bool vseg = seg < count;
   const u64 entry = vseg ? items[seg] : 0;
   const u32 pos = (u32)(entry >> 32);
   const u32 b = (u32)(entry >> 20) & 0xfffu;
   const u32 len = (u32)entry & 0xfffffu;
   if (len == 0 && (WARP || vseg)) return;               // resolved by k_resolve_periodic (warp- resp. CTA-uniform)
   u32 xb = 0, n = 1, shift = 0, depth = 0;
   if (vseg) { xb = p.X[b]; n = p.X[b + 1] - xb; shift = round_shift(p, b, round, &depth); }
   const u32 ks = (TEXT && vseg) ? p.ksym[b] : 0;
   u32 n2 = 64;
   while (n2 < len) n2 <<= 1;
   // blocked load: thread t owns sequence positions t*8 .. t*8+7; the element's local id travels
   // in the low bits of the packed word.  Padding (all ones) sorts to the end of [0, n2).
   VT v[MS_ITEMS];
#pragma unroll
   for (int r = 0; r < MS_ITEMS; r++) {
      const u32 i = t * MS_ITEMS + (u32)r;
      VT w = ~(VT)0;
      if (i < len) {
         const u32 idx = p.sa[pos + i];
         w = (load_key<TEXT>(p, xb, n, idx, shift, round + 1, ks) << MS_LBITS) | (VT)i;
      }
      v[r] = w;
   }
   bitonic_blocked<THREADS, VT>(v, t, n2, xch);
   // sorted position e = t*8 + r.  Heads, group starts (1-based running max), ends.
   VT prevlast = __shfl_up_sync(FULL, v[MS_ITEMS - 1], 1);
   VT nextfirst = __shfl_down_sync(FULL, v[0], 1);
   if (!WARP) {
      // indices are clamped so that a speculated shared-memory load can never leave the array
      const u32 wi = threadIdx.x >> 5;
      const u32 pi = wi ? wi - 1 : 0;
      const u32 ni = (wi + 1 < (u32)(THREADS / 32)) ? wi + 1 : wi;
      __syncthreads();
      if (lane_id() == 31) xch[wi] = v[MS_ITEMS - 1];
      if (lane_id() == 0) xch[32 + wi] = v[0];
      __syncthreads();
      const VT pl = xch[pi], nf = xch[32 + ni];
      if (lane_id() == 0 && wi > 0) prevlast = pl;
      if (lane_id() == 31 && wi + 1 < (u32)(THREADS / 32)) nextfirst = nf;
   }
   const u32 base = t * MS_ITEMS;
   u32 last = 0, gs[MS_ITEMS];
#pragma unroll
   for (int r = 0; r < MS_ITEMS; r++) {
      const u32 e = base + r;
      if (e < len) {
         const VT pv = (r == 0) ? prevlast : v[r - 1];
         if (e == 0 || (pv >> MS_LBITS) != (v[r] >> MS_LBITS)) last = e + 1;
      }
      gs[r] = last;
   }
   u32 incl, prev;
   if (WARP) {
      incl = warp_incl_max(last);
      prev = __shfl_up_sync(FULL, incl, 1);
      if (t == 0) prev = 0;
   } else {
      incl = block_incl_max<THREADS>(last, ssm);
      prev = __shfl_up_sync(FULL, incl, 1);
      if (lane_id() == 0) prev = ssm[threadIdx.x >> 5];
   }
   // fetch the rotation indices before anything is overwritten
   u32 idxs[MS_ITEMS];
#pragma unroll
   for (int r = 0; r < MS_ITEMS; r++) {
      const u32 e = base + r;
      const u32 local = (u32)v[r] & ((1u << MS_LBITS) - 1u);
      idxs[r] = (e < len) ? p.sa[pos + local] : 0;
   }
   if (WARP) __syncwarp(); else __syncthreads();
   const bool deep = (depth >= n);
#pragma unroll
   for (int r = 0; r < MS_ITEMS; r++) {
      const u32 e = base + r;
      const bool in = e < len;
      u32 g = gs[r] ? gs[r] : prev;
      g = g ? g - 1 : 0;
      bool is_end = false;
      if (in) {
         p.sa[pos + e] = idxs[r];
         p.rank[xb + idxs[r]] = rk_pack(round + 1, pos - xb, (pos - xb) + g);
         const VT nx = (r == MS_ITEMS - 1) ? nextfirst : v[r + 1];
         is_end = (e == len - 1) || ((nx >> MS_LBITS) != (v[r] >> MS_LBITS));
      }
      const u32 size = e - g + 1;
      const bool multi = in && is_end && size >= 2;
      if (multi && deep) atomicMax(&p.power_q[b], size);
      push_seg(Lout, multi && !deep, pos + g, b, size);
   }
}

// ---- 2b'. CTA-resident LSD radix sort of the same packed words ---------------------------------
// For segments of 513..4096 elements the bitonic network costs ~1000 instructions per element;
// eight-bit radix passes over a shared-memory copy cost ~30 per element and pass, and digits on
// which every key of the segment agrees are skipped (the rule on periodic data).  A pass ranks each
// element inside its warp with match_any (stable), the per-warp digit counts are scanned over
// warps and bins, and the elements -- held in registers meanwhile -- are written back in place.
template <int THREADS, bool TEXT>
__global__ void __launch_bounds__(THREADS) k_refine_radix(S2Params p, ListsDev Lout, const u64* items, u32 count, u32 round)
{
   constexpr int CAP = THREADS * MS_ITEMS;
   constexpr int LBITS = (CAP > 4096) ? 13 : 12;     // local index bits under the key
   typedef typename KeyOf<(TEXT || CAP > 4096)>::type VT;   // packed word: key << LBITS | local
   constexpr int WARPS = THREADS / 32;
   constexpr int BPT = (256 + THREADS - 1) / THREADS;   // bins per thread in the scan step
   extern __shared__ __align__(16) unsigned char dyn_smem[];
   VT* const buf = reinterpret_cast<VT*>(dyn_smem);   // [CAP]
   __shared__ u16 whist[WARPS][256];            // counts and prefixes stay below CAP <= 4096
   __shared__ u32 binbase[256];
   __shared__ u32 ssm[34];
   __shared__ VT s_red[2][WARPS];
   const u32 t = threadIdx.x, w = t >> 5, l = lane_id();
   const u64 entry = items[blockIdx.x];
   const u32 pos = (u32)(entry >> 32);
   const u32 b = (u32)(entry >> 20) & 0xfffu;
   const u32 len = (u32)entry & 0xfffffu;
   if (len == 0) return;                                  // resolved by k_resolve_periodic
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   u32 depth;
   const u32 shift = round_shift(p, b, round, &depth);
   const u32 ks = TEXT ? p.ksym[b] : 0;

   // striped load: warp w owns positions w*256 .. w*256+255, lane l takes every 32nd of them
   VT v[MS_ITEMS];
   VT vand = ~(VT)0, vor = 0;
#pragma unroll
   for (int k = 0; k < MS_ITEMS; k++) {
      const u32 i = w * (32 * MS_ITEMS) + (u32)k * 32 + l;
      VT word = ~(VT)0;
      if (i < len) {
         const u32 idx = p.sa[pos + i];
         word = ((VT)load_key<TEXT>(p, xb, n, idx, shift, round + 1, ks) << LBITS) | (VT)i;
         vand &= word; vor |= word;
      }
      v[k] = word;
      buf[i] = word;
   }
   // digits on which all keys agree need no pass
#pragma unroll
   for (int d = 16; d > 0; d >>= 1) {
      vand &= __shfl_xor_sync(FULL, vand, d);
      vor |= __shfl_xor_sync(FULL, vor, d);
   }
   if (l == 0) { s_red[0][w] = vand; s_red[1][w] = vor; }
   __syncthreads();
   {
      VT a = ~(VT)0, o = 0;
#pragma unroll
      for (int k = 0; k < WARPS; k++) { a &= s_red[0][k]; o |= s_red[1][k]; }
      vand = a; vor = o;
   }
   const VT diff = (vand ^ vor) >> LBITS;         // key bits that vary inside the segment
   const int npass = TEXT ? (int)((p.kbits[b] + 7) >> 3) : 3;

   for (int pass = 0; pass < npass; pass++) {
      const int sh = LBITS + 8 * pass;
      if (((diff >> (8 * pass)) & 255) == 0) continue;
#pragma unroll
      for (int k = 0; k < 8; k++) whist[w][l * 8 + k] = 0;
      __syncwarp();
      u32 rk[MS_ITEMS];
#pragma unroll
      for (int k = 0; k < MS_ITEMS; k++) {
         const u32 d = (u32)(v[k] >> sh) & 255;
         const u32 m = __match_any_sync(FULL, d);
         const u32 old = whist[w][d];
         __syncwarp();
         if (l == (u32)(__ffs(m) - 1)) whist[w][d] = (u16)(old + __popc(m));
         __syncwarp();
         rk[k] = old + __popc(m & lanemask_lt());
      }
      __syncthreads();
      // per bin: exclusive prefix over the warps, bin total
      u32 tot[BPT];
#pragma unroll
      for (int q = 0; q < BPT; q++) {
         const u32 bin = t + (u32)q * THREADS;
         u32 run = 0;
         if (bin < 256) {
#pragma unroll
            for (int ww = 0; ww < WARPS; ww++) { const u32 c = whist[ww][bin]; whist[ww][bin] = (u16)run; run += c; }
         }
         tot[q] = run;
      }
      // exclusive scan of the 256 bin totals (bins are laid out bin = t + q*THREADS)
      if (THREADS >= 256) {
         u32 dummy;
         const u32 ex = block_excl_sum<THREADS>(t < 256 ? tot[0] : 0u, ssm, &dummy);
         if (t < 256) binbase[t] = ex;
      } else {
         // THREADS = 128 or 64: scan the q-slices one after the other
         u32 carry = 0;
#pragma unroll
         for (int q = 0; q < BPT; q++) {
            u32 total;
            const u32 ex = block_excl_sum<THREADS>(tot[q], ssm, &total);
            binbase[t + (u32)q * THREADS] = carry + ex;
            carry += total;
            __syncthreads();
         }
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < MS_ITEMS; k++) {
         const u32 d = (u32)(v[k] >> sh) & 255;
         buf[binbase[d] + whist[w][d] + rk[k]] = v[k];
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < MS_ITEMS; k++) v[k] = buf[w * (32 * MS_ITEMS) + (u32)k * 32 + l];
   }
   __syncthreads();

   // blocked view of the sorted sequence: thread t owns positions t*8 .. t*8+7
   const u32 base = t * MS_ITEMS;
#pragma unroll
   for (int r = 0; r < MS_ITEMS; r++) v[r] = buf[base + r];
   const VT prevlast = buf[base ? base - 1 : 0];
   const VT nextfirst = buf[(base + MS_ITEMS < (u32)CAP) ? base + MS_ITEMS : (u32)CAP - 1];
   u32 last = 0, gs[MS_ITEMS];
#pragma unroll
   for (int r = 0; r < MS_ITEMS; r++) {
      const u32 e = base + r;
      if (e < len) {
         const VT pv = (r == 0) ? prevlast : v[r - 1];
         if (e == 0 || (pv >> LBITS) != (v[r] >> LBITS)) last = e + 1;
      }
      gs[r] = last;
   }
   const u32 incl = block_incl_max<THREADS>(last, ssm);
   u32 prev = __shfl_up_sync(FULL, incl, 1);
   if (l == 0) prev = ssm[w];
   u32 idxs[MS_ITEMS];
#pragma unroll
   for (int r = 0; r < MS_ITEMS; r++) {
      const u32 e = base + r;
      const u32 local = (u32)v[r] & ((1u << LBITS) - 1u);
      idxs[r] = (e < len) ? p.sa[pos + local] : 0;
   }
   __syncthreads();
   const bool deep = (depth >= n);
#pragma unroll
   for (int r = 0; r < MS_ITEMS; r++) {
      const u32 e = base + r;
      const bool in = e < len;
      u32 g = gs[r] ? gs[r] : prev;
      g = g ? g - 1 : 0;
      bool is_end = false;
      if (in) {
         p.sa[pos + e] = idxs[r];
         p.rank[xb + idxs[r]] = rk_pack(round + 1, pos - xb, (pos - xb) + g);
         const VT nx = (r == MS_ITEMS - 1) ? nextfirst : v[r + 1];
         is_end = (e == len - 1) || ((nx >> LBITS) != (v[r] >> LBITS));
      }
      const u32 size = e - g + 1;
      const bool multi = in && is_end && size >= 2;
      if (multi && deep) atomicMax(&p.power_q[b], size);
      push_seg(Lout, multi && !deep, pos + g, b, size);
   }
}

// ---- 2c. large segments: one CTA, stable LSD radix passes ----------------------------
constexpr int LG_ITEMS = 4;
constexpr int LG_MAXPASS = 7;

// LG_THREADS = 1024: one CTA per SM (64 registers per thread).  512 with two CTAs per SM (one sorts while the other
// waits at a barrier) was measured: no gain (text 50.1 vs 50.9 ms of S2 per 400 MB).
template <bool TEXT, int LG_THREADS>
__global__ void __launch_bounds__(LG_THREADS, 1024 / LG_THREADS) k_refine_large(S2Params p, ListsDev Lout, const u64* items, u32 round)
{
   constexpr int LG_TILE = LG_THREADS * LG_ITEMS;
   constexpr int LG_WARPS = LG_THREADS / 32;
   typedef typename KeyOf<TEXT>::type KT;
   __shared__ u32 whist[LG_WARPS][256];
   __shared__ u32 binbase[TEXT ? LG_MAXPASS : 3][256];
   __shared__ u32 ssm[34];
   __shared__ u32 s_carry;
   __shared__ u32 s_skip;
   const u64 entry = items[blockIdx.x];
   const u32 pos = (u32)(entry >> 32);
   const u32 b = (u32)(entry >> 20) & 0xfffu;
   const u32 len = (u32)entry & 0xfffffu;
   if (len == 0) return;                                  // resolved by k_resolve_periodic
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   u32 depth;
   const u32 shift0 = round_shift(p, b, round, &depth);
   const u32 ks = TEXT ? p.ksym[b] : 0;
   const int npass = TEXT ? (int)((p.kbits[b] + 7) >> 3) : ((n > 65536u) ? 3 : 2);
   KT* const kA = TEXT ? reinterpret_cast<KT*>(p.kscrA) : reinterpret_cast<KT*>(p.keyA);
   KT* const kB = TEXT ? reinterpret_cast<KT*>(p.kscrB) : reinterpret_cast<KT*>(p.keyB);
   const u32 w = threadIdx.x >> 5, l = lane_id();

   for (u32 i = threadIdx.x; i < (u32)npass * 256; i += LG_THREADS) (&binbase[0][0])[i] = 0;
   __syncthreads();
   // phase A: gather keys, digit histograms
   for (u32 i = threadIdx.x; i < len; i += LG_THREADS) {
      const u32 idx = p.sa[pos + i];
      const KT key = load_key<TEXT>(p, xb, n, idx, shift0, round + 1, ks);
      kA[pos + i] = key;
      for (int q = 0; q < npass; q++) atomicAdd(&binbase[q][(u32)(key >> (8 * q)) & 255], 1u);
   }
   __syncthreads();
   if (threadIdx.x == 0) s_skip = 0;
   __syncthreads();
   if (w < (u32)npass) {
      // exclusive scan of 256 bins by one warp: 8 per lane.  A digit on which every key agrees
      // (one bin holds the whole segment -- the rule on periodic data) needs no pass at all.
      u32 v[8], s = 0;
      bool whole = false;
#pragma unroll
      for (int k = 0; k < 8; k++) { v[k] = binbase[w][l * 8 + k]; s += v[k]; whole |= (v[k] == len); }
      if (__any_sync(FULL, whole) && l == 0) atomicOr(&s_skip, 1u << w);
      u32 ex = warp_incl_sum(s) - s;
#pragma unroll
      for (int k = 0; k < 8; k++) { binbase[w][l * 8 + k] = ex; ex += v[k]; }
   }
   __syncthreads();
   const u32 skip = s_skip;

   // phase B: passes
   int done = 0;                                   // passes actually executed (selects the ping-pong side)
   for (int pass = 0; pass < npass; pass++) {
      if ((skip >> pass) & 1u) continue;
      const KT* ksrc = (done & 1) ? kB : kA;
      const u32* isrc = (done & 1) ? p.idxB : p.sa;
      KT* kdst = (done & 1) ? kA : kB;
      u32* idst = (done & 1) ? p.sa : p.idxB;
      const int shift = pass * 8;
      done++;
      for (u32 tb = 0; tb < len; tb += LG_TILE) {
#pragma unroll
         for (int k = 0; k < 8; k++) whist[w][l * 8 + k] = 0;
         __syncwarp();
         KT key[LG_ITEMS];
         u32 idx[LG_ITEMS], rk[LG_ITEMS];
#pragma unroll
         for (int k = 0; k < LG_ITEMS; k++) {
            const u32 i = tb + w * (32 * LG_ITEMS) + k * 32 + l;
            const bool valid = i < len;
            key[k] = valid ? ksrc[pos + i] : 0;
            idx[k] = valid ? isrc[pos + i] : 0;
            const u32 d = (u32)(key[k] >> shift) & 255;
            const u32 m = __match_any_sync(FULL, valid ? d : 0x1000u);
            const u32 old = whist[w][d];
            __syncwarp();
            if (valid && l == (u32)(__ffs(m) - 1)) whist[w][d] = old + __popc(m);
            __syncwarp();
            rk[k] = old + __popc(m & lanemask_lt());
         }
         __syncthreads();
         if (threadIdx.x < 256) {
            u32 run = binbase[pass][threadIdx.x];
#pragma unroll 8
            for (int ww = 0; ww < LG_WARPS; ww++) {
               const u32 c = whist[ww][threadIdx.x];
               whist[ww][threadIdx.x] = run;
               run += c;
            }
            binbase[pass][threadIdx.x] = run;
         }
         __syncthreads();
#pragma unroll
         for (int k = 0; k < LG_ITEMS; k++) {
            const u32 i = tb + w * (32 * LG_ITEMS) + k * 32 + l;
            if (i < len) {
               const u32 d = (u32)(key[k] >> shift) & 255;
               const u32 dst = whist[w][d] + rk[k];
               kdst[pos + dst] = key[k];
               idst[pos + dst] = idx[k];
            }
         }
         __syncthreads();
      }
      __threadfence_block();
   }
   // phase C: group boundaries, new ranks, next-round segments
   const KT* kfin = (done & 1) ? kB : kA;
   const u32* ifin = (done & 1) ? p.idxB : p.sa;
   const bool deep = (depth >= n);
   if (threadIdx.x == 0) s_carry = 0;
   __syncthreads();
   for (u32 tb = 0; tb < len; tb += LG_TILE) {
      const u32 base = tb + threadIdx.x * LG_ITEMS;
      KT kk[LG_ITEMS + 2];
#pragma unroll
      for (int k = 0; k < LG_ITEMS + 2; k++) {
         const i64 i = (i64)base + k - 1;
         kk[k] = (i >= 0 && i < (i64)len) ? kfin[pos + (u32)i] : ~(KT)0;
      }
      u32 last = 0, gs[LG_ITEMS];
#pragma unroll
      for (int k = 0; k < LG_ITEMS; k++) {
         const u32 i = base + k;
         if (i < len) { if (i == 0 || kk[k + 1] != kk[k]) last = i + 1; }
         gs[k] = last;
      }
      const u32 incl = block_incl_max<LG_THREADS>(last, ssm);
      u32 prev = __shfl_up_sync(FULL, incl, 1);
      if (l == 0) prev = ssm[w];
      const u32 carry = s_carry;
      if (prev == 0) prev = carry;
#pragma unroll
      for (int k = 0; k < LG_ITEMS; k++) {
         const u32 i = base + k;
         const bool in = i < len;
         u32 g = gs[k] ? gs[k] : prev;
         g = g ? g - 1 : 0;
         bool is_end = false;
         if (in) {
            const u32 idx = ifin[pos + i];
            if (done & 1) p.sa[pos + i] = idx;
            p.rank[xb + idx] = rk_pack(round + 1, pos - xb, (pos - xb) + g);
            is_end = (i == len - 1) || (kk[k + 2] != kk[k + 1]);
         }
         const u32 size = i - g + 1;
         const bool multi = in && is_end && size >= 2;
         if (multi && deep) atomicMax(&p.power_q[b], size);
         push_seg(Lout, multi && !deep, pos + g, b, size);
      }
      __syncthreads();
      if (threadIdx.x == LG_THREADS - 1) s_carry = incl ? incl : carry;
      __syncthreads();
   }
}

// ---- 2d. tandem repeats ---------------------------------------------------------------------
// A segment sorted to depth d whose members are the positions i, i+p, i+2p, ... (p <= d) needs no more
// doubling: every member is  u . (next member)  with the same p-symbol prefix u, so their order is the order
// of the chain ends.  Only the last member continues outside the segment (at X = max+p); if X ranks below
// the segment the members sort by descending position, if above by ascending position (the tandem-repeat
// rule of suffix sorters; divsufsort's tr_copy plays this role in the reference, blocksort.c:1040-1100).
// Periodic inputs (the reference manual's worst case) otherwise cost log2(n/d) rounds over every element.
// One CTA per listed segment; resolved segments get len = 0 in the worklist and the sort kernels skip them.
constexpr int AP_THREADS = 256;

struct ApLists { u64* items[N_BIG_CLASSES]; u32 start[N_BIG_CLASSES + 1]; };   // the worklists of one round, concatenated

__global__ void __launch_bounds__(AP_THREADS) k_resolve_periodic(S2Params p, ApLists L, u32 round)
{
   __shared__ u32 red_mn[AP_THREADS / 32], red_mx[AP_THREADS / 32];
   __shared__ u32 s_bad;
   int cls = 0;
#pragma unroll
   for (int c = 1; c < N_BIG_CLASSES; c++) if (blockIdx.x >= L.start[c]) cls = c;
   u64* const items = L.items[cls];
   const u32 seg = blockIdx.x - L.start[cls];
   const u64 entry = items[seg];
   const u32 pos = (u32)(entry >> 32);
   const u32 b = (u32)(entry >> 20) & 0xfffu;
   const u32 len = (u32)entry & 0xfffffu;
   if (len < 3) return;
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   u32 depth_after;
   const u32 depth = round_shift(p, b, round, &depth_after);       // the segment's members share their first `depth` symbols
   const u32 tag = round + 1;
   const u32 t = threadIdx.x, w = t >> 5, l = lane_id();
   // 1. min / max position
   u32 mn = 0xffffffffu, mx = 0;
   for (u32 i = t; i < len; i += AP_THREADS) { const u32 v = p.sa[pos + i]; mn = min(mn, v); mx = max(mx, v); }
#pragma unroll
   for (int d = 16; d > 0; d >>= 1) { mn = min(mn, __shfl_xor_sync(FULL, mn, d)); mx = max(mx, __shfl_xor_sync(FULL, mx, d)); }
   if (l == 0) { red_mn[w] = mn; red_mx[w] = mx; }
   if (t == 0) s_bad = 0;
   __syncthreads();
#pragma unroll
   for (int k = 0; k < AP_THREADS / 32; k++) { mn = min(mn, red_mn[k]); mx = max(mx, red_mx[k]); }
   const u32 span = mx - mn;
   const u32 step = span / (len - 1);
   if (p.debug && t == 0 && len > 8192) printf("[ap] round %u blk %u len %u mn %u mx %u step %u depth %u n %u\n", round, b, len, mn, mx, step, depth, n);
   if (step == 0 || step * (len - 1) != span) return;                        // uniform over the CTA
   // step > depth: the members are not yet known to share a whole period -- unless the step is the block's dominant
   // repeat offset and the repeat lengths jq[] (2e) say that every pair of neighbours but the top one agrees on at
   // least `step` symbols.  Then member k is u . member k+1 for all k below the top pair, so all neighbours compare
   // like the top pair does, and that pair is decided by the ranks right behind its repeat.
   const bool relaxed = step > depth;
   if (relaxed && !(p.jq && p.dstar[b - p.b0] == step)) return;
   u32 xpos = mx + step; if (xpos >= n) xpos -= n;
   const u32 gs = pos - xb;
   bool ascending;
   if (relaxed) {
      __shared__ u32 s_jtop;
      for (u32 i = t; i < len; i += AP_THREADS) {
         const u32 v = p.sa[pos + i];
         if ((v - mn) % step) { s_bad = 1; continue; }
         const u32 k = (v - mn) / step;
         if (k + 1 < len) {
            const u32 j = p.jq[xb + v];
            if (k + 2 < len) { if (j < step) s_bad = 1; }
            else s_jtop = j;
         }
      }
      __syncthreads();
      if (s_bad) return;
      const u32 jtop = s_jtop;
      if (jtop < step) {
         u32 ya = mx - step + jtop; if (ya >= n) ya -= n;
         u32 yb = mx + jtop; if (yb >= n) yb -= n;
         const u32 ra = rk_read(p.rank[xb + ya], tag), rb = rk_read(p.rank[xb + yb], tag);
         if (ra == rb) return;
         ascending = ra < rb;
      } else {
         const u32 xr = rk_read(p.rank[xb + xpos], tag);
         if (xr >= gs && xr < gs + len) return;
         ascending = xr >= gs + len;
      }
   } else {
   if (xpos == mn && (u64)step * len == n) {
      // the progression closes on itself: the block is u^len with |u| = step <= depth, these len rotations are
      // equal for good.  Record the multiplicity and retire the segment instead of doubling up to depth n.
      for (u32 i = t; i < len; i += AP_THREADS) { const u32 v = p.sa[pos + i]; if ((v - mn) % step) s_bad = 1; }
      __syncthreads();
      if (!s_bad && t == 0) { atomicMax(&p.power_q[b], len); items[seg] = entry & ~(u64)0xfffffu; }
      return;
   }
   // the continuation of the last member must lie outside the segment
   const u32 xr = rk_read(p.rank[xb + xpos], tag);
   if (xr >= gs && xr < gs + len) return;
   ascending = xr >= gs + len;
   // 2. every member on the progression?  (members are distinct, so len multiples inside [mn, mx] are all of them)
   for (u32 i = t; i < len; i += AP_THREADS) { const u32 v = p.sa[pos + i]; if ((v - mn) % step) s_bad = 1; }
   __syncthreads();
   if (s_bad) return;
   }
   // 3. final order and final ranks
   for (u32 i = t; i < len; i += AP_THREADS) {
      const u32 v = p.sa[pos + i];
      const u32 k = (v - mn) / step;
      const u32 r = ascending ? k : len - 1 - k;
      p.idxB[pos + r] = v;
      p.rank[xb + v] = rk_pack(tag, gs, gs + r);
   }
   __syncthreads();
   for (u32 i = t; i < len; i += AP_THREADS) p.sa[pos + i] = p.idxB[pos + i];
   if (t == 0) items[seg] = entry & ~(u64)0xfffffu;                          // done: nothing left to sort
}

// ---- 2e. repeat chains ---------------------------------------------------------------------------
// Long non-tandem repeats (a file that contains another copy of itself 300 kB further on) leave pairs
// {a, a+p}, {a+1, a+p+1}, ... unresolved over hundreds of thousands of positions, and plain doubling visits
// every one of them in each of log2(repeat length / depth) rounds.  But such a segment S is decided exactly
// where the repeat ends: call S *chained* when the successors {x+1 : x in S} all lie in one unresolved
// segment.  If S, S+1, ..., S+j-1 are chained, the members of S agree on their first j symbols (the members
// of every segment agree on their first symbol) and the members of S+j agree to the current depth d, so
// sorting S by the rank at offset j+d is valid -- the same doubling step, from depth j+d instead of d -- and a
// whole run of chained segments is resolved in the round that resolves its last one.  The chain flag is a
// property of the segment, so all members of S see the same j.  k_rep_small/k_rep_warp mark the members
// of chained segments, k_rep_tiles/k_rep_dist turn the marks into j[x] = distance from x to the next
// unmarked position of the block (cyclic; 0 everywhere if the block has none: an exact power, left to the
// depth test), and load_key adds j[x] to the round's shift.  Rotations that are equal (exact powers) are
// never separated, because their successors are never separated.
template <int LANES>
__global__ void __launch_bounds__(256) k_rep_small(S2Params p, const u32* items, u32 count, u32 round, u8* cflag)
{
   const u32 gid = blockIdx.x * blockDim.x + threadIdx.x;
   const u32 seg = gid / LANES;
   const u32 sub = gid % LANES;
   const bool vseg = seg < count;
   const u32 entry = vseg ? items[seg] : 0;
   const u32 pos = entry & 0x7ffffffu;
   const u32 len = (entry >> 27) + 1;
   u32 xb = 0, n = 1;
   if (vseg) { const u32 b = block_of(p, pos); xb = p.X[b]; n = p.X[b + 1] - xb; }
   const bool active = vseg && sub < len;
   u32 idx = 0, r = 0;
   if (active) {
      idx = p.sa[pos + sub];
      u32 t = idx + 1; if (t >= n) t = 0;
      r = rk_read(p.rank[xb + t], round + 1);
   }
   const u32 r0 = __shfl_sync(FULL, r, lane_id() & ~(u32)(LANES - 1));
   const u32 bal = __ballot_sync(FULL, !active || r == r0);
   const u32 sh = lane_id() & ~(u32)(LANES - 1);
   const u32 gm = (LANES == 32) ? FULL : (((1u << (LANES & 31)) - 1u) << sh);
   if (active && (bal & gm) == gm) cflag[xb + idx] = 1;
}

// one warp per segment of the CTA-sorted classes; gives up at the first successor that falls elsewhere
__global__ void __launch_bounds__(256) k_rep_warp(S2Params p, const u64* items, u32 count, u32 round, u8* cflag)
{
   const u32 seg = blockIdx.x * 8 + (threadIdx.x >> 5);
   if (seg >= count) return;
   const u64 entry = items[seg];
   const u32 pos = (u32)(entry >> 32);
   const u32 b = (u32)(entry >> 20) & 0xfffu;
   const u32 len = (u32)entry & 0xfffffu;
   if (len == 0) return;                                  // retired by k_resolve_periodic
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   const u32 l = lane_id();
   u32 t0 = p.sa[pos] + 1; if (t0 >= n) t0 = 0;
   const u32 r0 = rk_read(p.rank[xb + t0], round + 1);
   for (u32 i = l; i < ((len + 31) & ~31u); i += 32) {
      bool ok = true;
      if (i < len) {
         u32 t = p.sa[pos + i] + 1; if (t >= n) t = 0;
         ok = rk_read(p.rank[xb + t], round + 1) == r0;
      }
      if (!__all_sync(FULL, ok)) return;
   }
   for (u32 i = l; i < len; i += 32) cflag[xb + p.sa[pos + i]] = 1;
}

// Votes for the block's dominant repeat offset: the distance between two members of every small segment,
// counted in a 256-bin hash table per block (warp-aggregated).
constexpr u32 REP_VOTE_STRIDE = 4;
__global__ void __launch_bounds__(256) k_rep_vote(S2Params p, const u32* items, u32 count, u32* vote)
{
   const u32 seg = (blockIdx.x * blockDim.x + threadIdx.x) * REP_VOTE_STRIDE;     // a sample is enough
   const bool v = seg < count;
   u32 slot = 0xffffffffu, dlt = 0;
   if (v) {
      const u32 pos = items[seg] & 0x7ffffffu;
      const u32 b = block_of(p, pos);
      const u32 x0 = p.sa[pos], x1 = p.sa[pos + 1];
      dlt = x0 > x1 ? x0 - x1 : x1 - x0;
      slot = (b - p.b0) * 256u + ((dlt * 2654435761u) >> 24);
   }
   const u32 m = __match_any_sync(FULL, slot);
   if (v && lane_id() == (u32)(__ffs(m) - 1)) {
      atomicAdd(&vote[2 * (size_t)slot], __popc(m));
      vote[2 * (size_t)slot + 1] = dlt;
   }
}

// the same vote from the warp- and CTA-sorted classes: (max - min) / (len - 1), the step if the members are a progression
__global__ void __launch_bounds__(AP_THREADS) k_rep_vote_big(S2Params p, ApLists L, u32* vote)
{
   __shared__ u32 red_mn[AP_THREADS / 32], red_mx[AP_THREADS / 32];
   int cls = 0;
#pragma unroll
   for (int c = 1; c < N_BIG_CLASSES; c++) if (blockIdx.x >= L.start[c]) cls = c;
   const u64 entry = L.items[cls][blockIdx.x - L.start[cls]];
   const u32 pos = (u32)(entry >> 32);
   const u32 b = (u32)(entry >> 20) & 0xfffu;
   const u32 len = (u32)entry & 0xfffffu;
   if (len < 3) return;
   const u32 t = threadIdx.x;
   u32 mn = 0xffffffffu, mx = 0;
   for (u32 i = t; i < len; i += AP_THREADS) { const u32 v = p.sa[pos + i]; mn = min(mn, v); mx = max(mx, v); }
#pragma unroll
   for (int d = 16; d > 0; d >>= 1) { mn = min(mn, __shfl_xor_sync(FULL, mn, d)); mx = max(mx, __shfl_xor_sync(FULL, mx, d)); }
   if (lane_id() == 0) { red_mn[t >> 5] = mn; red_mx[t >> 5] = mx; }
   __syncthreads();
   if (t) return;
#pragma unroll
   for (int k = 0; k < AP_THREADS / 32; k++) { mn = min(mn, red_mn[k]); mx = max(mx, red_mx[k]); }
   const u32 span = mx - mn, step = span / (len - 1);
   if (step == 0 || step * (len - 1) != span) return;
   const u32 slot = (b - p.b0) * 256u + ((step * 2654435761u) >> 24);
   atomicAdd(&vote[2 * (size_t)slot], len);
   vote[2 * (size_t)slot + 1] = step;
}

constexpr u32 CH_MIN_VOTES = 512;       // sampled small segments count 1, progressions their length

// eq[x] = 1 where x and x + d* (cyclic) are in the same segment, d* the block's most voted offset
__global__ void __launch_bounds__(256) k_rep_eq(S2Params p, const u32* vote, u32* dstar, u8* eq, u32 round)
{
   __shared__ u64 red[8];
   const u32 b = p.b0 + blockIdx.y;
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   const u32 t0 = blockIdx.x * 4096u;
   if (t0 >= n) return;
   const u32* v = vote + (size_t)blockIdx.y * 512;
   u64 best = ((u64)v[2 * threadIdx.x] << 32) | v[2 * threadIdx.x + 1];
#pragma unroll
   for (int d = 16; d > 0; d >>= 1) best = max(best, __shfl_xor_sync(FULL, best, d));
   if (lane_id() == 0) red[threadIdx.x >> 5] = best;
   __syncthreads();
#pragma unroll
   for (int k = 0; k < 8; k++) best = max(best, red[k]);
   u32 ds = (u32)best;
   if ((u32)(best >> 32) < CH_MIN_VOTES || ds >= n) ds = 0;
   if (blockIdx.x == 0 && threadIdx.x == 0) dstar[blockIdx.y] = ds;
   if (ds == 0) return;                                    // eq stays all zero
   const u32 tag = round + 1;
#pragma unroll 4
   for (int k = 0; k < 16; k++) {
      const u32 i = t0 + (u32)k * 256u + threadIdx.x;
      if (i < n) {
         u32 y = i + ds; if (y >= n) y -= n;
         eq[xb + i] = rk_read(p.rank[xb + i], tag) == rk_read(p.rank[xb + y], tag);
      }
   }
}

constexpr int CH_THREADS = 256;
constexpr int CH_ITEMS = 16;
constexpr int CH_TILE = CH_THREADS * CH_ITEMS;
constexpr u32 CH_NONE = 0xffffffffu;

// first unmarked position of every 4096-position tile of a block
__global__ void __launch_bounds__(CH_THREADS) k_rep_tiles(S2Params p, const u8* cflag, u32* tilefirst, u32 tpb)
{
   __shared__ u32 red[CH_THREADS / 32];
   const u32 b = p.b0 + blockIdx.y;
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   const u32 t0 = blockIdx.x * CH_TILE;
   if (t0 >= n) return;
   u32 first = CH_NONE;
#pragma unroll 4
   for (int k = CH_ITEMS - 1; k >= 0; k--) {
      const u32 i = t0 + (u32)k * CH_THREADS + threadIdx.x;
      if (i < n && cflag[xb + i] == 0) first = i;
   }
#pragma unroll
   for (int d = 16; d > 0; d >>= 1) first = min(first, __shfl_xor_sync(FULL, first, d));
   if (lane_id() == 0) red[threadIdx.x >> 5] = first;
   __syncthreads();
   if (threadIdx.x == 0) {
#pragma unroll
      for (int k = 1; k < CH_THREADS / 32; k++) first = min(first, red[k]);
      tilefirst[(size_t)blockIdx.y * tpb + blockIdx.x] = first;
   }
}

// j[x] = distance from x to the next unmarked position at or after it, cyclically inside the block
__global__ void __launch_bounds__(CH_THREADS) k_rep_dist(S2Params p, const u8* cflag, const u32* tilefirst, u32 tpb, u32* jd)
{
   __shared__ __align__(16) u8 sf[CH_TILE];
   __shared__ u32 sj[CH_TILE + CH_TILE / 32];                 // index s + s/32: conflict-free for both the blocked and the striped view
   __shared__ u32 wmin[CH_THREADS / 32];
   __shared__ u32 s_carry;
   const u32 b = p.b0 + blockIdx.y;
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   const u32 t0 = blockIdx.x * CH_TILE;
   if (t0 >= n) return;
   const u32 ntiles = (n + CH_TILE - 1) / CH_TILE;
   const u32* tf = tilefirst + (size_t)blockIdx.y * tpb;
   const u32 t = threadIdx.x, w = t >> 5, l = lane_id();
#pragma unroll 4
   for (int k = 0; k < CH_ITEMS; k++) {
      const u32 s = (u32)k * CH_THREADS + t;
      sf[s] = (t0 + s < n) ? cflag[xb + t0 + s] : (u8)1;      // positions past the end are transparent: n-1 is followed by 0
   }
   if (w == 0) {
      // the next unmarked position after this tile: the tiles behind it, then (+n) the tiles from 0 up to this one
      u32 carry = CH_NONE;
      for (u32 base = 1; base <= ntiles; base += 32) {
         const u32 i = base + l;
         u32 tt = blockIdx.x + i;
         const bool wrap = tt >= ntiles;
         if (wrap) tt -= ntiles;
         const u32 v = (i <= ntiles) ? tf[tt] : CH_NONE;
         const u32 found = __ballot_sync(FULL, v != CH_NONE);
         if (found) { const int src = __ffs(found) - 1; carry = __shfl_sync(FULL, v + (wrap ? n : 0u), src); break; }
      }
      if (l == 0) s_carry = carry;
   }
   __syncthreads();
   // thread t owns tile positions t*16 .. t*16+15
   const uint4 f4 = *reinterpret_cast<const uint4*>(&sf[t * CH_ITEMS]);
   const u32 fw[4] = {f4.x, f4.y, f4.z, f4.w};
   u32 mine = CH_NONE;
#pragma unroll
   for (int r = CH_ITEMS - 1; r >= 0; r--) if (((fw[r >> 2] >> (8 * (r & 3))) & 255u) == 0) mine = t0 + t * CH_ITEMS + (u32)r;
   u32 inc = mine;                                            // nearest unmarked position in lanes >= l
#pragma unroll
   for (int d = 1; d < 32; d <<= 1) { const u32 o = __shfl_down_sync(FULL, inc, d); if (l + d < 32) inc = min(inc, o); }
   if (l == 0) wmin[w] = inc;
   __syncthreads();
   u32 after = s_carry;
#pragma unroll
   for (int ww = CH_THREADS / 32 - 1; ww > 0; ww--) if ((u32)ww > w) after = min(after, wmin[ww]);
   u32 cur = __shfl_down_sync(FULL, inc, 1);
   cur = (l == 31) ? after : min(cur, after);
#pragma unroll
   for (int r = CH_ITEMS - 1; r >= 0; r--) {
      const u32 s = t * CH_ITEMS + (u32)r;
      if (((fw[r >> 2] >> (8 * (r & 3))) & 255u) == 0) cur = t0 + s;
      sj[s + (s >> 5)] = (cur == CH_NONE) ? 0u : cur - (t0 + s);
   }
   __syncthreads();
#pragma unroll 4
   for (int k = 0; k < CH_ITEMS; k++) {
      const u32 s = (u32)k * CH_THREADS + t;
      if (t0 + s < n) jd[xb + t0 + s] = sj[s + (s >> 5)];
   }
}

// ---- 3. last column -------------------------------------------------------------------
__global__ void __launch_bounds__(KG_THREADS) k_bwt_out(S2Params p, u8* bwt, u32* origptr)
{
   const u32 b = p.b0 + blockIdx.y;
   const u32 xb = p.X[b], n = p.X[b + 1] - xb;
   const u32 t0 = blockIdx.x * KG_TILE;
   if (t0 >= n) return;
   const u8* T = p.T + xb;
   // rank of rotation 0: its final position, or the start of its tie group for exact powers
   if (blockIdx.x == 0 && threadIdx.x == 0) origptr[b] = (u32)p.rank[xb] & 0xffffffu;
#pragma unroll 4
   for (int k = 0; k < KG_ITEMS; k++) {
      const u32 i = t0 + k * KG_THREADS + threadIdx.x;
      if (i < n) {
         const u32 s = p.sa[xb + i];
         bwt[xb + i] = T[s ? s - 1 : n - 1];
      }
   }
}

// --------------------------------------------------------------------------------------
static ListsDev lists_dev(Engine* e, int which)
{
   ListsDev L;
   for (int c = 0; c < N_SMALL_CLASSES; c++) { L.small_items[c] = e->lists.small_items[which][c]; L.small_cap[c] = e->lists.small_cap[c]; }
   for (int c = 0; c < N_BIG_CLASSES; c++) { L.big_items[c] = e->lists.big_items[which][c]; L.big_cap[c] = e->lists.big_cap[c]; }
   L.counts = e->lists.counts[which];
   L.overflow = e->s1_scalars + 4;
   return L;
}

static bool trace_on()
{
   static int on = -1;
   if (on < 0) { const char* v = getenv("BZ2_B200_TRACE"); on = (v && *v >= '1') ? 1 : 0; }
   return on == 1;
}

// BZ2_B200_DEBUG_SYNC=1: synchronise after every refinement launch and name the kernel that faulted
static bool dbg_sync(Engine* e, const char* what)
{
   static int on = -1;
   if (on < 0) { const char* v = getenv("BZ2_B200_DEBUG_SYNC"); on = (v && *v >= '1') ? 1 : 0; }
   if (!on) return true;
   cudaError_t c = cudaDeviceSynchronize();
   if (c == cudaSuccess) c = cudaGetLastError();
   if (c != cudaSuccess) { fprintf(stderr, "[bz2b200] %s: %s\n", what, cudaGetErrorString(c)); return false; }
   return true;
}

template <int LANES>
static void launch_small(Engine* e, cudaStream_t st, const S2Params& p, const ListsDev& Lout, const u32* items, u32 count, u32 round, bool text)
{
   const u64 threads = (u64)count * LANES;
   const u32 grid = (u32)((threads + 255) / 256);
   if (text) k_refine_small<LANES, true><<<grid, 256, 0, st>>>(p, Lout, items, count, round);
   else      k_refine_small<LANES, false><<<grid, 256, 0, st>>>(p, Lout, items, count, round);
   char nm[64]; snprintf(nm, sizeof nm, "k_refine_small<%d,%d> count=%u round=%u", LANES, (int)text, count, round); dbg_sync(e, nm);
}
template <int THREADS>
static void launch_medium(Engine* e, cudaStream_t st, const S2Params& p, const ListsDev& Lout, const u64* items, u32 count, u32 round, bool text)
{
   const u32 grid = (THREADS == 32) ? (count + 7) / 8 : count;
   const u32 block = (THREADS == 32) ? 256 : THREADS;
   if (text) k_refine_medium<THREADS, true><<<grid, block, 0, st>>>(p, Lout, items, count, round);
   else      k_refine_medium<THREADS, false><<<grid, block, 0, st>>>(p, Lout, items, count, round);
   char nm[64]; snprintf(nm, sizeof nm, "k_refine_medium<%d,%d> count=%u round=%u", THREADS, (int)text, count, round); dbg_sync(e, nm);
}

template <int THREADS>
static void launch_radix(Engine* e, cudaStream_t st, const S2Params& p, const ListsDev& Lout, const u64* items, u32 count, u32 round, bool text)
{
   constexpr size_t CAP = (size_t)THREADS * MS_ITEMS;
   if (text) k_refine_radix<THREADS, true><<<count, THREADS, CAP * sizeof(u64), st>>>(p, Lout, items, count, round);
   else      k_refine_radix<THREADS, false><<<count, THREADS, CAP * (CAP > 4096 ? sizeof(u64) : sizeof(u32)), st>>>(p, Lout, items, count, round);
   char nm[64]; snprintf(nm, sizeof nm, "k_refine_radix<%d,%d> count=%u round=%u", THREADS, (int)text, count, round); dbg_sync(e, nm);
}

static void launch_large(Engine* e, cudaStream_t st, const S2Params& p, const ListsDev& Lout, const u64* items, u32 count, u32 round, bool text)
{
   if (text) k_refine_large<true, 1024><<<count, 1024, 0, st>>>(p, Lout, items, round);
   else      k_refine_large<false, 1024><<<count, 1024, 0, st>>>(p, Lout, items, round);
   dbg_sync(e, "k_refine_large");
}

// the 8192-element radix sort keeps 64 KiB of sort words in dynamic shared memory
int stage2_init()
{
   cudaError_t c = cudaFuncSetAttribute(k_refine_radix<1024, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8192 * (int)sizeof(u64));
   if (c == cudaSuccess) c = cudaFuncSetAttribute(k_refine_radix<1024, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8192 * (int)sizeof(u64));
   return c == cudaSuccess ? 0 : -1;
}

// max_blk = 0: a single-stream window (blocks of up to nmax + 16 bytes, e->hist_stride k-gram bins per block).
// Batch windows pass their largest block: the k-gram budget is the one engine_new picks for an nmax of that size,
// never below 2^16 bins (the tie-order replay uses each slot as its 65,536-entry bucket table, stage2_tie.cu), and
// the per-block grids are sized by that block, so a window of many small blocks does not clear and scan full slots.
u32 s2_batch_stride(const Engine* e, u32 max_blk)
{
   u32 s = 1u << 16;
   while (s < (1u << e->hist_log2) && s < max_blk / 4) s <<= 1;
   if (e->hist_log2 > 18 && s < max_blk * 2u) s = 1u << e->hist_log2;
   return s < e->hist_stride ? s : e->hist_stride;
}

int stage2_run(Engine* e, u32 nb, u32 E, u32 max_blk)
{
   cudaStream_t st = e->stream;
   S2Params p;
   p.T = e->enc; p.X = e->bt.X; p.nb = nb;
   p.sa = e->sa; p.rank = e->rank;
   p.keyA = e->keyA; p.keyB = e->keyB; p.idxB = e->idxB;
   p.hist = e->hist; p.hist_stride = max_blk ? s2_batch_stride(e, max_blk) : e->hist_stride; p.code = e->code; p.kk = e->kk; p.nbins = e->nbins;
   p.hh = e->hh; p.kbits = e->kbits; p.ksym = e->ksym; p.K = e->K; p.kscrA = e->kscrA; p.kscrB = e->kscrB;
   p.debug = trace_on() ? 1 : 0;
   p.kg_agg_alpha = KG_AGG_MAX_ALPHA;
   p.blockmap = e->blockmap;
   p.power_q = e->bt.power_q; p.inuse = e->bt.inuse; p.ninuse = e->bt.ninuse;
   p.jd = nullptr; p.jq = nullptr; p.dstar = nullptr;

   const u32 nchunks = (E >> 12) + 1;
   k_blockmap<<<(nchunks + 255) / 256, 256, 0, st>>>(e->bt.X, nb, e->blockmap, nchunks);     BZ_KCHECK(e);
   BZ_CUDA(e, cudaMemsetAsync(e->bt.inuse, 0, (size_t)nb * 256, st));
   BZ_CUDA(e, cudaMemsetAsync(e->bt.power_q, 0, sizeof(u32) * nb, st));
   BZ_CUDA(e, cudaMemsetAsync(e->s1_scalars + 4, 0, sizeof(u32), st));
   const u32 max_n = (max_blk ? max_blk : e->nmax) + 16;
   // Blocks are sorted in sub-batches small enough for their rank/sa arrays to stay in L2.
   const u32 group = e->s2_group ? e->s2_group : nb;
   for (u32 b0 = 0; b0 < nb; b0 += group) {
      const u32 g = (nb - b0 < group) ? (nb - b0) : group;
      p.b0 = b0;
      BZ_CUDA(e, cudaMemsetAsync(e->hist, 0, (size_t)g * p.hist_stride * sizeof(u32), st));
      BZ_CUDA(e, cudaMemsetAsync(e->lists.counts[0], 0, sizeof(u32) * N_CLASSES, st));
      const dim3 gtiles((max_n + KG_TILE - 1) / KG_TILE, g);
      k_inuse<<<gtiles, KG_THREADS, 0, st>>>(p);                                                BZ_KCHECK(e);
      k_codemap<<<g, 256, 0, st>>>(p);                                                          BZ_KCHECK(e);
      // one atomic pass: the count pass keeps each rotation's arrival index inside its bucket, so the
      // placement pass needs no atomics (bucket start + arrival index)
      k_kgram<KG_HISTOFF, true><<<gtiles, KG_THREADS, 0, st>>>(p);                              BZ_KCHECK(e);
      k_kgram_scan<<<g, 1024, 0, st>>>(p);                                                      BZ_KCHECK(e);
      k_kgram<KG_PLACE, false><<<gtiles, KG_THREADS, 0, st>>>(p);                                      BZ_KCHECK(e);
      k_seg_init<<<dim3((p.hist_stride + 255) / 256, g), 256, 0, st>>>(p, lists_dev(e, 0));    BZ_KCHECK(e);
      dbg_sync(e, "k-gram phase");

      int cur = 0;
      u64 prev_small = 0, prev_big = 0;
      for (u32 round = 0; ; round++) {
         BZ_CUDA(e, cudaMemcpyAsync(e->h_counts, e->lists.counts[cur], sizeof(u32) * (N_CLASSES), cudaMemcpyDeviceToHost, st));
         BZ_CUDA(e, cudaMemcpyAsync(e->h_scalars + 4, e->s1_scalars + 4, sizeof(u32), cudaMemcpyDeviceToHost, st));
         BZ_CUDA(e, cudaStreamSynchronize(st));
         if (e->h_scalars[4]) { snprintf(e->err, sizeof e->err, "segment worklist overflow"); return -4; }
         u32 cnt[N_CLASSES]; u64 total = 0;
         for (int c = 0; c < N_CLASSES; c++) { cnt[c] = e->h_counts[c]; total += cnt[c]; }
         if (total == 0) break;
         if (trace_on()) {
            // BZ2_B200_TRACE=1: segments and elements per size class, every round (debug only: copies the lists)
            fprintf(stderr, "[bz2b200] round %u:", round);
            for (int c = 0; c < N_CLASSES; c++) {
               u64 elems = 0;
               if (cnt[c] && c >= N_SMALL_CLASSES) {
                  u64* h = (u64*)malloc(sizeof(u64) * cnt[c]);
                  cudaMemcpy(h, e->lists.big_items[cur][c - N_SMALL_CLASSES], sizeof(u64) * cnt[c], cudaMemcpyDeviceToHost);
                  for (u32 i = 0; i < cnt[c]; i++) elems += h[i] & 0xfffffu;
                  free(h);
               } else if (cnt[c]) {
                  u32* h = (u32*)malloc(sizeof(u32) * cnt[c]);
                  cudaMemcpy(h, e->lists.small_items[cur][c], sizeof(u32) * cnt[c], cudaMemcpyDeviceToHost);
                  for (u32 i = 0; i < cnt[c]; i++) elems += (h[i] >> 27) + 1;
                  free(h);
               }
               fprintf(stderr, " c%d=%u/%llu", c, cnt[c], (unsigned long long)elems);
            }
            fprintf(stderr, "\n");
         }
         if (round > 22) { snprintf(e->err, sizeof e->err, "prefix doubling did not terminate"); return -5; }
         const int nxt = cur ^ 1;
         BZ_CUDA(e, cudaMemsetAsync(e->lists.counts[nxt], 0, sizeof(u32) * N_CLASSES, st));
         ListsDev Lout = lists_dev(e, nxt);
         u32** si = e->lists.small_items[cur];
         u64** bi = e->lists.big_items[cur];
         const bool text = (round == 0);
         // The size classes of one round touch disjoint segments, so they run side by side: the few
         // long-running CTAs of the large and CTA-sort classes overlap the sub-warp classes' tails.
         // tandem repeats: the large class from round 0 on (few segments), every CTA/warp-sorted class from round 2 on
         // Repeat chains (2e) cost a few passes over the window, so they run only while refinement has stalled: a
         // sizeable part of the window is still unresolved and the last round removed less than 40 % of it.  The segment
         // chains serve the sub-warp and warp classes; the dominant-offset repeats also serve the tandem rule.
         static const u32 minlen[N_CLASSES] = {2, 3, 5, 9, 17, 33, 257, 513, 1025, 2049, 4097, 8193};
         u64 est_small = 0, est_big = 0;
         for (int c = 0; c < 6; c++) est_small += (u64)cnt[c] * minlen[c];
         for (int c = 5; c < N_CLASSES; c++) est_big += (u64)cnt[c] * minlen[c];
         const bool chain_ok = e->chain && !text && round >= 1;
         const bool force = e->chain >= 2;                                      // BZ2_B200_CHAIN=2: always (tests)
         const bool go_small = chain_ok && round >= e->chain_min_round && (force || (est_small >= E / 32 && est_small * 10 >= prev_small * 6));
         const bool go_big = chain_ok && (force || (est_big >= E / 32 && est_big * 10 >= prev_big * 6));
         prev_small = est_small; prev_big = est_big;
         ApLists AL;
         u32 ap_tot = 0;
         for (int c = 0; c < N_BIG_CLASSES; c++) {
            AL.items[c] = bi[c];
            AL.start[c] = ap_tot;
            if (round >= 2 || go_big || c == N_BIG_CLASSES - 1) ap_tot += cnt[N_SMALL_CLASSES + c];
         }
         AL.start[N_BIG_CLASSES] = ap_tot;
         p.jd = nullptr; p.jq = nullptr; p.dstar = nullptr;
         {
            if (go_small || (go_big && ap_tot)) {
               u8* const cflag = reinterpret_cast<u8*>(e->kscrB);      // the 64-bit key scratch is idle after round 0
               u8* const eq = cflag + E;
               u32* const jd = reinterpret_cast<u32*>(e->kscrA);
               u32* const jq = jd + E;
               const u32 tpb = (max_n + CH_TILE - 1) / CH_TILE;
               u32* const tilefirst = e->hist;                          // idle after the k-gram phase
               u32* const tilefirst2 = tilefirst + (size_t)g * tpb;
               u32* const vote = tilefirst2 + (size_t)g * tpb;          // [g][256][2]
               u32* const dstar = vote + (size_t)g * 512;               // [g]
               const dim3 ctiles(tpb, g);
               BZ_CUDA(e, cudaMemsetAsync(cflag, 0, 2 * (size_t)E, st));
               BZ_CUDA(e, cudaMemsetAsync(vote, 0, sizeof(u32) * 513 * (size_t)g, st));
               if (go_big && ap_tot) { k_rep_vote_big<<<ap_tot, AP_THREADS, 0, st>>>(p, AL, vote); BZ_KCHECK(e); }
               if (go_small) {
                  if (cnt[0]) { k_rep_vote<<<(cnt[0] / REP_VOTE_STRIDE + 256) / 256, 256, 0, st>>>(p, si[0], cnt[0], vote); BZ_KCHECK(e); }
                  if (cnt[1]) { k_rep_vote<<<(cnt[1] / REP_VOTE_STRIDE + 256) / 256, 256, 0, st>>>(p, si[1], cnt[1], vote); BZ_KCHECK(e); }
                  if (cnt[0]) { k_rep_small<2><<<(u32)(((u64)cnt[0] * 2 + 255) / 256), 256, 0, st>>>(p, si[0], cnt[0], round, cflag);   BZ_KCHECK(e); }
                  if (cnt[1]) { k_rep_small<4><<<(u32)(((u64)cnt[1] * 4 + 255) / 256), 256, 0, st>>>(p, si[1], cnt[1], round, cflag);   BZ_KCHECK(e); }
                  if (cnt[2]) { k_rep_small<8><<<(u32)(((u64)cnt[2] * 8 + 255) / 256), 256, 0, st>>>(p, si[2], cnt[2], round, cflag);   BZ_KCHECK(e); }
                  if (cnt[3]) { k_rep_small<16><<<(u32)(((u64)cnt[3] * 16 + 255) / 256), 256, 0, st>>>(p, si[3], cnt[3], round, cflag); BZ_KCHECK(e); }
                  if (cnt[4]) { k_rep_small<32><<<(u32)(((u64)cnt[4] * 32 + 255) / 256), 256, 0, st>>>(p, si[4], cnt[4], round, cflag); BZ_KCHECK(e); }
                  if (cnt[5]) { k_rep_warp<<<(cnt[5] + 7) / 8, 256, 0, st>>>(p, bi[0], cnt[5], round, cflag); BZ_KCHECK(e); }
                  k_rep_tiles<<<ctiles, CH_THREADS, 0, st>>>(p, cflag, tilefirst, tpb);       BZ_KCHECK(e);
                  k_rep_dist<<<ctiles, CH_THREADS, 0, st>>>(p, cflag, tilefirst, tpb, jd);    BZ_KCHECK(e);
                  p.jd = jd;
               }
               k_rep_eq<<<ctiles, 256, 0, st>>>(p, vote, dstar, eq, round);                BZ_KCHECK(e);
               k_rep_tiles<<<ctiles, CH_THREADS, 0, st>>>(p, eq, tilefirst2, tpb);         BZ_KCHECK(e);
               k_rep_dist<<<ctiles, CH_THREADS, 0, st>>>(p, eq, tilefirst2, tpb, jq);      BZ_KCHECK(e);
               p.jq = jq; p.dstar = dstar;
               dbg_sync(e, "repeat chains");
            }
         }
         if (ap_tot) {
            k_resolve_periodic<<<ap_tot, AP_THREADS, 0, st>>>(p, AL, round); BZ_KCHECK(e);
            dbg_sync(e, "k_resolve_periodic");
         }
         const bool fork = total > 64;
         cudaStream_t sL = st, sM = st, sW = st;
         if (fork) {
            sL = e->aux[0]; sM = e->aux[1]; sW = e->aux[2];
            BZ_CUDA(e, cudaEventRecord(e->ev_fork, st));
            for (int a = 0; a < 3; a++) BZ_CUDA(e, cudaStreamWaitEvent(e->aux[a], e->ev_fork, 0));
         }
         if (cnt[CLS_LARGE]) {
            launch_large(e, sL, p, Lout, bi[6], cnt[CLS_LARGE], round, text);
            dbg_sync(e, "k_refine_large");
         }
         // 513..8192: shared-memory radix CTAs; 257..512: the packed-word bitonic CTA of 64 (both measured against each other in round 1)
         if (cnt[CLS_C8K])   launch_radix<1024>(e, sL, p, Lout, bi[5], cnt[CLS_C8K], round, text);
         if (cnt[CLS_C4K])   launch_radix<512>(e, sM, p, Lout, bi[4], cnt[CLS_C4K], round, text);
         if (cnt[CLS_C2K])   launch_radix<256>(e, sM, p, Lout, bi[3], cnt[CLS_C2K], round, text);
         if (cnt[CLS_C1K])   launch_radix<128>(e, sW, p, Lout, bi[2], cnt[CLS_C1K], round, text);
         if (cnt[CLS_C512])  launch_medium<64>(e, sW, p, Lout, bi[1], cnt[CLS_C512], round, text);
         if (cnt[CLS_W256])  launch_medium<32>(e, sW, p, Lout, bi[0], cnt[CLS_W256], round, text);
         if (cnt[4]) launch_small<32>(e, st, p, Lout, si[4], cnt[4], round, text);
         if (cnt[3]) launch_small<16>(e, st, p, Lout, si[3], cnt[3], round, text);
         if (cnt[2]) launch_small<8>(e, st, p, Lout, si[2], cnt[2], round, text);
         if (cnt[1]) launch_small<4>(e, st, p, Lout, si[1], cnt[1], round, text);
         if (cnt[0]) launch_small<2>(e, st, p, Lout, si[0], cnt[0], round, text);
         if (fork) {
            for (int a = 0; a < 3; a++) {
               BZ_CUDA(e, cudaEventRecord(e->ev_join[a], e->aux[a]));
               BZ_CUDA(e, cudaStreamWaitEvent(st, e->ev_join[a], 0));
            }
         }
         u32 nl = 0;
         for (int c = 0; c < N_CLASSES; c++) nl += cnt[c] ? 1u : 0u;
         e->launches += nl - 1;
         e->bwt_rounds++;
         BZ_KCHECK(e);
         cur = nxt;
      }
      k_bwt_out<<<gtiles, KG_THREADS, 0, st>>>(p, e->bwt, e->bt.origptr);                       BZ_KCHECK(e);
      { const int rc = stage2_power_origptr(e, b0, g); if (rc) return rc; }                      // exact powers (stage2_tie.cu)
   }
   return 0;
}

} // namespace bz
