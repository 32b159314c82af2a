// stage4_huff.cu -- S4 + S5: Huffman table selection, code construction, bit emission
// and stream assembly.
//
// Replaces sendMTFValues (reference compress.c:250-818), BZ2_hbMakeCodeLengths and
// BZ2_hbAssignCodes (huffman.c:63-148, :152-166), the bit writer (compress.c:37-86) and
// the per-block framing of BZ2_compressBlock (compress.c:822-881).
//
//   k_huff_init     initial partition of the alphabet into nGroups cost tables (:276-319)
//   4 x { k_huff_select   per 50-symbol group: cost under each table, pick the cheapest
//                         (lowest index wins ties), add the group to that table's
//                         frequencies (:324-541)
//         k_huff_lengths  code lengths from frequencies, replaying the reference's heap
//                         exactly, 17-bit limit with halve-and-retry (huffman.c:63-148) }
//   k_huff_finish   canonical codes, selector MTF + unary coding, symbol map and
//                   delta-coded tables -> per-block "preamble" bits; exact coded size
//   k_bit_offsets   scan of block sizes -> absolute bit offset of every block (S5)
//   k_group_bits / k_group_scan   bit offset of every 50-symbol group inside its block
//   k_pack          every group is packed by one thread straight to its final bit
//                   position in the stream (interior words stored, edge words atomicOr)
//   k_pre_copy      preamble bits shifted into place
// Because block sizes are known before packing, blocks are written at their final,
// non-byte-aligned positions and no separate concatenation pass is needed.
#include "engine.h"

namespace bz {

constexpr u32 PRE_STRIDE = 24576;       // bytes reserved per block for preamble bits
constexpr int SEL_THREADS = 128;        // groups per CTA in select/pack kernels

struct S4Params {
   const u16* mtfv;
   const u32* X;
   const u32* nmtf;
   const i32* mtffreq;
   const u8* inuse;
   const u32* ninuse;
   const u32* crc;
   const u32* origptr;
   u8* sel;
   u8* hlen;            // [nb][6][258]
   i32* hfreq;          // [nb][6][258]
   u32* hcode;          // [nb][6][258]  (len << 20 | code)
   u32* grpbits;
   u8* pre;
   u32* prebits;
   u32* ngroups;
   u64* bits;
   u64* bitoff;
};

__device__ __forceinline__ u32 sel_base(u32 xb, u32 b) { return (xb + b) / BZ_G_SIZE + b; }
__device__ __forceinline__ u32 n_groups_for(u32 nmtf)
{
   return nmtf < 200 ? 2 : nmtf < 600 ? 3 : nmtf < 1200 ? 4 : nmtf < 2400 ? 5 : 6;     // compress.c:266-270
}

// ---- initial tables (compress.c:276-319), one thread per block ----------------------------
__global__ void k_huff_init(S4Params p, u32 nb)
{
   const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
   if (b >= nb) return;
   const i32 nmtf = (i32)p.nmtf[b];
   const i32 alpha = (i32)p.ninuse[b] + 2;
   const i32 ng = (i32)n_groups_for((u32)nmtf);
   p.ngroups[b] = (u32)ng;
   u8* len = p.hlen + (size_t)b * 6 * BZ_MAX_ALPHA;
   const i32* freq = p.mtffreq + (size_t)b * BZ_MAX_ALPHA;
   for (i32 t = 0; t < 6; t++) for (i32 v = 0; v < BZ_MAX_ALPHA; v++) len[t * BZ_MAX_ALPHA + v] = (t < ng && v < alpha) ? 15 : 0;
   i32 part = ng, rem = nmtf, gs = 0;
   while (part > 0) {
      const i32 target = rem / part;
      i32 ge = gs - 1, acc = 0;
      while (acc < target && ge < alpha - 1) { ge++; acc += freq[ge]; }
      if (ge > gs && part != ng && part != 1 && ((ng - part) % 2 == 1)) { acc -= freq[ge]; ge--; }
      for (i32 v = gs; v <= ge; v++) len[(part - 1) * BZ_MAX_ALPHA + v] = 0;
      part--; gs = ge + 1; rem -= acc;
   }
}

// ---- one refinement pass: selectors + per-table frequencies --------------------------------
// MODE 0: select (writes sel, accumulates hfreq).  MODE 1: group bit lengths with final tables.
template <int MODE>
__global__ void __launch_bounds__(SEL_THREADS) k_huff_select(S4Params p)
{
   __shared__ u16 ssym[SEL_THREADS * BZ_G_SIZE];
   __shared__ u64 lenpack[BZ_MAX_ALPHA];
   __shared__ u32 hist[6][BZ_MAX_ALPHA];
   const u32 b = blockIdx.y;
   const u32 nmtf = p.nmtf[b];
   const u32 nsel = (nmtf + BZ_G_SIZE - 1) / BZ_G_SIZE;
   const u32 g0 = blockIdx.x * SEL_THREADS;
   if (g0 >= nsel) return;
   const u32 xb = p.X[b];
   const u16* mt = p.mtfv + (size_t)xb + b;
   const u32 ng = p.ngroups[b];
   const u8* len = p.hlen + (size_t)b * 6 * BZ_MAX_ALPHA;
   for (u32 v = threadIdx.x; v < BZ_MAX_ALPHA; v += SEL_THREADS) {
      u64 pk = 0;
      for (u32 t = 0; t < 6; t++) pk |= (u64)len[t * BZ_MAX_ALPHA + v] << (10 * t);
      lenpack[v] = pk;
      if (MODE == 0) for (u32 t = 0; t < 6; t++) hist[t][v] = 0;
   }
   const u32 s0 = g0 * BZ_G_SIZE;
   const u32 s1 = min(nmtf, s0 + SEL_THREADS * BZ_G_SIZE);
   for (u32 i = s0 + threadIdx.x; i < s1; i += SEL_THREADS) ssym[i - s0] = mt[i];
   __syncthreads();
   const u32 g = g0 + threadIdx.x;
   if (g < nsel) {
      const u32 lo = threadIdx.x * BZ_G_SIZE;
      const u32 cnt = min((u32)BZ_G_SIZE, nmtf - g * BZ_G_SIZE);
      u8* selp = p.sel + sel_base(xb, b);
      if (MODE == 0) {
         u64 acc = 0;
         for (u32 i = 0; i < cnt; i++) acc += lenpack[ssym[lo + i]];
         u32 bt = 0, bc = (u32)(acc & 0x3ff);
         for (u32 t = 1; t < ng; t++) {
            const u32 c = (u32)(acc >> (10 * t)) & 0x3ff;
            if (c < bc) { bc = c; bt = t; }
         }
         selp[g] = (u8)bt;
         for (u32 i = 0; i < cnt; i++) atomicAdd(&hist[bt][ssym[lo + i]], 1u);
      } else {
         const u32 t = selp[g];
         u32 bits = 0;
         for (u32 i = 0; i < cnt; i++) bits += (u32)(lenpack[ssym[lo + i]] >> (10 * t)) & 0x3ff;
         p.grpbits[sel_base(xb, b) + g] = bits;
      }
   }
   if (MODE == 0) {
      __syncthreads();
      i32* hf = p.hfreq + (size_t)b * 6 * BZ_MAX_ALPHA;
      for (u32 k = threadIdx.x; k < 6 * BZ_MAX_ALPHA; k += SEL_THREADS) {
         const u32 c = (&hist[0][0])[k];
         if (c) atomicAdd(&hf[k], (i32)c);
      }
   }
}

// ---- code lengths (huffman.c:63-148): one warp per (block, table), heap driven by lane 0 ----
__global__ void __launch_bounds__(192) k_huff_lengths(S4Params p)
{
   // BZ2_hbMakeCodeLengths (huffman.c:63-148) replayed literally -- the merge order under ties is part of the
   // format's de-facto definition.  The heap holds (weight << 32 | node) words so that a sift step is one
   // shared-memory load instead of the reference's weight[heap[y]] double indirection (the whole kernel is
   // one dependent chain per table, so its run time is that chain's latency).
   __shared__ u64 s_hp[6][260];
   __shared__ i32 s_w[6][260];
   __shared__ i32 s_par[6][516];
   const u32 b = blockIdx.x;
   const u32 t = threadIdx.x >> 5, l = lane_id();
   if (t >= p.ngroups[b]) return;
   const i32 alpha = (i32)p.ninuse[b] + 2;
   const i32* freq = p.hfreq + ((size_t)b * 6 + t) * BZ_MAX_ALPHA;
   u8* len = p.hlen + ((size_t)b * 6 + t) * BZ_MAX_ALPHA;
   u64* hp = s_hp[t];
   i32* wt = s_w[t];
   i32* par = s_par[t];
   for (i32 i = l; i < alpha; i += 32) { const i32 f = freq[i]; wt[i + 1] = (f == 0 ? 1 : f) << 8; }
   __syncwarp();
   for (;;) {
      if (l == 0) {
         i32 nnodes = alpha, nheap = 0;
         hp[0] = 0; par[0] = -2;                        // sentinel: weight 0 at the root's parent slot
         for (i32 i = 1; i <= alpha; i++) {
            par[i] = -1;
            nheap++;
            // sift up
            i32 z = nheap; const u32 wtmp = (u32)wt[i];
            for (;;) { const u64 up = hp[z >> 1]; if (!(wtmp < (u32)(up >> 32))) break; hp[z] = up; z >>= 1; }
            hp[z] = ((u64)wtmp << 32) | (u32)i;
         }
         while (nheap > 1) {
            u64 n12[2];
#pragma unroll
            for (int r = 0; r < 2; r++) {
               n12[r] = hp[1];
               const u64 tmp = hp[nheap]; nheap--;
               // sift down from the root
               i32 z = 1; const u32 wtmp = (u32)(tmp >> 32);
               for (;;) {
                  i32 y = z << 1;
                  if (y > nheap) break;
                  u64 e = hp[y];
                  if (y < nheap) { const u64 e1 = hp[y + 1]; if ((u32)(e1 >> 32) < (u32)(e >> 32)) { y++; e = e1; } }
                  if (wtmp < (u32)(e >> 32)) break;
                  hp[z] = e;
                  z = y;
               }
               hp[z] = tmp;
            }
            nnodes++;
            par[(u32)n12[0]] = par[(u32)n12[1]] = nnodes;
            const u32 wa = (u32)(n12[0] >> 32), wb = (u32)(n12[1] >> 32);
            const u32 da = wa & 0xff, db = wb & 0xff;
            const u32 wn = ((wa & 0xffffff00u) + (wb & 0xffffff00u)) | (1u + (da > db ? da : db));
            par[nnodes] = -1;
            nheap++;
            i32 z = nheap;
            for (;;) { const u64 up = hp[z >> 1]; if (!(wn < (u32)(up >> 32))) break; hp[z] = up; z >>= 1; }
            hp[z] = ((u64)wn << 32) | (u32)nnodes;
         }
      }
      __syncwarp();
      bool too_long = false;
      for (i32 i = 1 + (i32)l; i <= alpha; i += 32) {
         i32 d = 0, k = i;
         while (par[k] >= 0) { k = par[k]; d++; }
         len[i - 1] = (u8)d;
         if (d > BZ_MAX_CODELEN) too_long = true;
      }
      if (!__any_sync(FULL, too_long)) break;
      __syncwarp();
      for (i32 i = 1 + (i32)l; i <= alpha; i += 32) wt[i] = (1 + (wt[i] >> 8) / 2) << 8;
      __syncwarp();
   }
}

// ---- serial bit writer into a zeroed byte buffer (MSB first) -----------------------------
struct BitW {
   u8* out; u64 acc; u32 nacc; u32 nbytes;
   __device__ void init(u8* o) { out = o; acc = 0; nacc = 0; nbytes = 0; }
   __device__ void put(u32 nb, u32 v)
   {
      acc |= (u64)v << (64 - nacc - nb);
      nacc += nb;
      while (nacc >= 8) { out[nbytes++] = (u8)(acc >> 56); acc <<= 8; nacc -= 8; }
   }
   __device__ u32 finish() { const u32 bits = nbytes * 8 + nacc; if (nacc) out[nbytes++] = (u8)(acc >> 56); return bits; }
};

__device__ __forceinline__ u32 bswap32(u32 v) { return __byte_perm(v, 0, 0x0123); }

// Bit writer that ORs whole 32-bit words into a zeroed buffer, starting at any bit offset, so
// several writers can fill disjoint bit ranges of the same buffer concurrently.
struct BitWA {
   u32* w; u64 acc; u32 nacc; u32 widx;
   __device__ void init(u32* words, u32 startbit) { w = words; widx = startbit >> 5; nacc = startbit & 31; acc = 0; }
   __device__ void put(u32 nb, u32 v)
   {
      acc |= (u64)v << (64 - nacc - nb);
      nacc += nb;
      if (nacc >= 32) { atomicOr(&w[widx++], bswap32((u32)(acc >> 32))); acc <<= 32; nacc -= 32; }
   }
   __device__ void finish() { if (nacc && (u32)(acc >> 32)) atomicOr(&w[widx], bswap32((u32)(acc >> 32))); }
};

// ---- codes, selectors, tables -> preamble bits; coded size (one CTA per block) ------------
__global__ void __launch_bounds__(192) k_huff_finish(S4Params p)
{
   __shared__ u32 cnt[6][24];
   __shared__ u32 basec[6][24];
   __shared__ u64 s_pay[6];
   __shared__ u32 s_scan[34];
   __shared__ u32 s_misc[4];
   const u32 b = blockIdx.x;
   const u32 t = threadIdx.x >> 5, l = lane_id();
   const u32 ng = p.ngroups[b];
   const u32 alpha = p.ninuse[b] + 2;
   const u32 nmtf = p.nmtf[b];
   const u32 xb = p.X[b];
   const u8* lenb = p.hlen + (size_t)b * 6 * BZ_MAX_ALPHA;
   if (t < ng) {
      // canonical codes (huffman.c:152-166)
      const u8* len = lenb + t * BZ_MAX_ALPHA;
      u32* code = p.hcode + ((size_t)b * 6 + t) * BZ_MAX_ALPHA;
      const i32* freq = p.hfreq + ((size_t)b * 6 + t) * BZ_MAX_ALPHA;
      if (l < 24) cnt[t][l] = 0;
      __syncwarp();
      u64 pay = 0;
      for (u32 v = l; v < alpha; v += 32) { atomicAdd(&cnt[t][len[v]], 1u); pay += (u64)len[v] * (u64)freq[v]; }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) pay += __shfl_xor_sync(FULL, pay, d);
      if (l == 0) s_pay[t] = pay;
      __syncwarp();
      if (l == 0) {
         u32 mn = 32, mx = 0;
         for (u32 L = 1; L <= 20; L++) if (cnt[t][L]) { if (L < mn) mn = L; if (L > mx) mx = L; }
         u32 vec = 0;
         for (u32 L = mn; L <= mx; L++) { basec[t][L] = vec; vec = (vec + cnt[t][L]) << 1; }
      }
      __syncwarp();
      for (u32 v = l; v < alpha; v += 32) {
         const u32 L = len[v];
         u32 r = 0;
         for (u32 u = 0; u < v; u++) r += (len[u] == L) ? 1u : 0u;
         code[v] = (L << 20) | (basec[t][L] + r);
      }
   }
   __syncthreads();
   // ---- preamble bits.  Three writers work on disjoint bit ranges of the zeroed buffer through
   // atomicOr: thread 0 the fixed header + symbol map, all threads the selectors (their MTF
   // positions are computed in parallel from last-occurrence times), thread 32 the tables.
   u32* const prew = reinterpret_cast<u32*>(p.pre + (size_t)b * PRE_STRIDE);
   const u8* iu = p.inuse + (size_t)b * 256;
   const u32 nsel = (nmtf + BZ_G_SIZE - 1) / BZ_G_SIZE;
   const u8* selp = p.sel + sel_base(xb, b);
   // header length: 48 + 32 + 1 + 24 magic/crc/rand/origPtr, 16 + 16 * ranges map, 3 + 15 counts
   if (threadIdx.x < 32) {
      u32 any = 0;
      if (threadIdx.x < 16) for (int j = 0; j < 16; j++) any |= iu[threadIdx.x * 16 + j];
      const u32 bal = __ballot_sync(FULL, any != 0);
      if (threadIdx.x == 0) s_misc[0] = 105u + 16u + 16u * (u32)__popc(bal & 0xffffu) + 18u;
   }
   // selector MTF in parallel (compress.c:573-631): position = number of tables used more recently
   const u32 per = (nsel + 191) / 192;
   const u32 lo = threadIdx.x * per, hi = min(nsel, lo + per);
   u32 lastv[6] = {0, 0, 0, 0, 0, 0};                  // 0 = not seen in my chunk; else index + 8
   for (u32 g = lo; g < hi; g++) lastv[selp[g]] = g + 8;
   u32 startv[6];
#pragma unroll
   for (int v = 0; v < 6; v++) {
      const u32 incl = block_incl_max<192>(lastv[v], s_scan);
      u32 prev = __shfl_up_sync(FULL, incl, 1);
      if (l == 0) prev = s_scan[t];
      startv[v] = max(prev, 7u - (u32)v);             // before the first selector the order is 0,1,2,3,4,5
      __syncthreads();
   }
   u32 mybits = 0;
   {
      u32 cur[6];
#pragma unroll
      for (int v = 0; v < 6; v++) cur[v] = startv[v];
      for (u32 g = lo; g < hi; g++) {
         const u32 sv = selp[g];
         u32 mine = 0, pos = 0;
#pragma unroll
         for (int v = 0; v < 6; v++) if ((u32)v == sv) mine = cur[v];
#pragma unroll
         for (int v = 0; v < 6; v++) pos += (cur[v] > mine) ? 1u : 0u;
         mybits += pos + 1;
#pragma unroll
         for (int v = 0; v < 6; v++) if ((u32)v == sv) cur[v] = g + 8;
      }
   }
   u32 selbits_total;
   const u32 myoff = block_excl_sum<192>(mybits, s_scan, &selbits_total);
   const u32 hdrbits = s_misc[0];
   {
      BitWA w; w.init(prew, hdrbits + myoff);
      u32 cur[6];
#pragma unroll
      for (int v = 0; v < 6; v++) cur[v] = startv[v];
      for (u32 g = lo; g < hi; g++) {
         const u32 sv = selp[g];
         u32 mine = 0, pos = 0;
#pragma unroll
         for (int v = 0; v < 6; v++) if ((u32)v == sv) mine = cur[v];
#pragma unroll
         for (int v = 0; v < 6; v++) pos += (cur[v] > mine) ? 1u : 0u;
         w.put(pos + 1, (1u << (pos + 1)) - 2u);                       // :686-688  pos ones then a zero
#pragma unroll
         for (int v = 0; v < 6; v++) if ((u32)v == sv) cur[v] = g + 8;
      }
      w.finish();
   }
   if (threadIdx.x == 0) {
      BitWA w; w.init(prew, 0);
      const u32 crc = p.crc[b];
      w.put(24, 0x314159); w.put(24, 0x265359);                        // compress.c:849-850
      w.put(16, crc >> 16); w.put(16, crc & 0xffff);                   // :853
      w.put(1, 0);                                                      // :864
      w.put(24, p.origptr[b]);                                          // :866
      u32 used16 = 0;
      for (int i = 0; i < 16; i++) { u32 any = 0; for (int j = 0; j < 16; j++) any |= iu[i * 16 + j]; used16 = (used16 << 1) | (any ? 1u : 0u); }
      w.put(16, used16);                                                // :654-664
      for (int i = 0; i < 16; i++) if (used16 & (0x8000u >> i)) {
         u32 v = 0; for (int j = 0; j < 16; j++) v = (v << 1) | (iu[i * 16 + j] ? 1u : 0u);
         w.put(16, v);                                                  // :666-674
      }
      w.put(3, ng); w.put(15, nsel);                                    // :681-682
      w.finish();
   }
   if (threadIdx.x == 32) {
      BitWA w; w.init(prew, hdrbits + selbits_total);
      u32 tb = 0;
      for (u32 tt = 0; tt < ng; tt++) {                                 // :696-706
         const u8* len = lenb + tt * BZ_MAX_ALPHA;
         u32 cur = len[0];
         w.put(5, cur); tb += 5;
         for (u32 v = 0; v < alpha; v++) {
            while (cur < len[v]) { w.put(2, 2); cur++; tb += 2; }
            while (cur > len[v]) { w.put(2, 3); cur--; tb += 2; }
            w.put(1, 0); tb += 1;
         }
      }
      w.finish();
      const u32 pbits = hdrbits + selbits_total + tb;
      p.prebits[b] = pbits;
      u64 pay = 0;
      for (u32 tt = 0; tt < ng; tt++) pay += s_pay[tt];
      p.bits[b] = (u64)pbits + pay;
   }
}

// exclusive scan of block bit sizes from start_bit (one CTA); bitoff[nb] = end
__global__ void __launch_bounds__(1024) k_bit_offsets(const u64* bits, u64* bitoff, u32 nb, u64 start_bit)
{
   __shared__ u64 wsum[32];
   __shared__ u64 s_run;
   if (threadIdx.x == 0) s_run = start_bit;
   __syncthreads();
   const u32 l = lane_id(), w = threadIdx.x >> 5;
   for (u32 base = 0; base < nb; base += 1024) {
      const u32 i = base + threadIdx.x;
      const u64 v = (i < nb) ? bits[i] : 0;
      u64 inc = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const u64 q = __shfl_up_sync(FULL, inc, d); if (l >= (u32)d) inc += q; }
      if (l == 31) wsum[w] = inc;
      __syncthreads();
      u64 pre = s_run;
      for (u32 k = 0; k < w; k++) pre += wsum[k];
      if (i < nb) bitoff[i] = pre + inc - v;
      __syncthreads();
      if (threadIdx.x == 1023) s_run = pre + inc;
      __syncthreads();
   }
   if (threadIdx.x == 0) bitoff[nb] = s_run;
}

// per-block exclusive scan of group bit lengths (in place)
__global__ void __launch_bounds__(1024) k_group_scan(S4Params p)
{
   __shared__ u32 ssm[34];
   const u32 b = blockIdx.x;
   const u32 nmtf = p.nmtf[b];
   const u32 nsel = (nmtf + BZ_G_SIZE - 1) / BZ_G_SIZE;
   u32* gb = p.grpbits + sel_base(p.X[b], b);
   const u32 per = (nsel + 1023) / 1024;
   const u32 lo = threadIdx.x * per;
   u32 sum = 0;
   for (u32 k = 0; k < per; k++) if (lo + k < nsel) sum += gb[lo + k];
   u32 ex = block_excl_sum<1024>(sum, ssm, nullptr);
   for (u32 k = 0; k < per; k++) if (lo + k < nsel) { const u32 v = gb[lo + k]; gb[lo + k] = ex; ex += v; }
}

// ---- payload: one thread per 50-symbol group, written at its final stream position ----------
__global__ void __launch_bounds__(SEL_THREADS) k_pack(S4Params p, u32* outw, u64 origin_bit)
{
   __shared__ u16 ssym[SEL_THREADS * BZ_G_SIZE];
   __shared__ u32 scode[6 * BZ_MAX_ALPHA];
   const u32 b = blockIdx.y;
   const u32 nmtf = p.nmtf[b];
   const u32 nsel = (nmtf + BZ_G_SIZE - 1) / BZ_G_SIZE;
   const u32 g0 = blockIdx.x * SEL_THREADS;
   if (g0 >= nsel) return;
   const u32 xb = p.X[b];
   const u16* mt = p.mtfv + (size_t)xb + b;
   const u32* code = p.hcode + (size_t)b * 6 * BZ_MAX_ALPHA;
   for (u32 k = threadIdx.x; k < 6 * BZ_MAX_ALPHA; k += SEL_THREADS) scode[k] = code[k];
   const u32 s0 = g0 * BZ_G_SIZE;
   const u32 s1 = min(nmtf, s0 + SEL_THREADS * BZ_G_SIZE);
   for (u32 i = s0 + threadIdx.x; i < s1; i += SEL_THREADS) ssym[i - s0] = mt[i];
   __syncthreads();
   const u32 g = g0 + threadIdx.x;
   if (g >= nsel) return;
   const u32 sb = sel_base(xb, b);
   const u32 t = p.sel[sb + g];
   const u32 cnt = min((u32)BZ_G_SIZE, nmtf - g * BZ_G_SIZE);
   const u64 bitpos = p.bitoff[b] + p.prebits[b] + p.grpbits[sb + g] - origin_bit;
   u64 widx = bitpos >> 5;
   u32 nacc = (u32)(bitpos & 31);          // leading bits owned by whoever precedes us
   u64 acc = 0;
   bool first = true;
   const u32 lo = threadIdx.x * BZ_G_SIZE;
   for (u32 i = 0; i < cnt; i++) {
      const u32 cl = scode[t * BZ_MAX_ALPHA + ssym[lo + i]];
      const u32 L = cl >> 20, c = cl & 0xfffff;
      acc |= (u64)c << (64 - nacc - L);
      nacc += L;
      if (nacc >= 32) {
         const u32 word = bswap32((u32)(acc >> 32));
         if (first) { atomicOr(&outw[widx], word); first = false; }
         else outw[widx] = word;
         widx++;
         acc <<= 32; nacc -= 32;
      }
   }
   if (nacc) atomicOr(&outw[widx], bswap32((u32)(acc >> 32)));
}

// preamble bits -> stream position (one thread per source word)
__global__ void __launch_bounds__(256) k_pre_copy(S4Params p, u32* outw, u64 origin_bit)
{
   const u32 b = blockIdx.y;
   const u32 pbits = p.prebits[b];
   const u32 nwords = (pbits + 31) >> 5;
   const u32 k = blockIdx.x * 256 + threadIdx.x;
   if (k >= nwords) return;
   const u8* src = p.pre + (size_t)b * PRE_STRIDE + (size_t)k * 4;
   u32 v = ((u32)src[0] << 24) | ((u32)src[1] << 16) | ((u32)src[2] << 8) | (u32)src[3];
   const u32 valid = min(32u, pbits - k * 32);
   if (valid < 32) v &= ~((1u << (32 - valid)) - 1u);
   const u64 bitpos = p.bitoff[b] + (u64)k * 32 - origin_bit;
   const u64 widx = bitpos >> 5;
   const u32 sh = (u32)(bitpos & 31);
   atomicOr(&outw[widx], bswap32(v >> sh));
   if (sh && (valid + sh > 32)) atomicOr(&outw[widx + 1], bswap32(v << (32 - sh)));
}

__global__ void k_put_bits(u32* outw, u64 relbit, u64 value, int nbits)
{
   // value occupies the low nbits; MSB first
   for (int done = 0; done < nbits;) {
      const u64 bp = relbit + done;
      const u32 sh = (u32)(bp & 31);
      const int take = min(32 - (int)sh, nbits - done);
      const u32 chunk = (u32)((value >> (nbits - done - take)) & ((take == 32) ? 0xffffffffu : ((1u << take) - 1u)));
      atomicOr(&outw[bp >> 5], bswap32(chunk << (32 - sh - take)));
      done += take;
   }
}

// S5 for shards: OR `nbits` bits of src (from its bit 0) into dst at bit offset dst_bit.
// One thread per source word; each lands in at most two destination words.
__global__ void __launch_bounds__(256) k_concat_bits(u32* dst, u64 dst_bit, const u32* src, u64 nbits)
{
   const u64 k = (u64)blockIdx.x * 256 + threadIdx.x;
   const u64 nwords = (nbits + 31) >> 5;
   if (k >= nwords) return;
   u32 v = bswap32(src[k]);
   const u64 left = nbits - k * 32;
   if (left < 32) v &= ~((1u << (32 - (u32)left)) - 1u);
   const u64 bp = dst_bit + k * 32;
   const u32 sh = (u32)(bp & 31);
   if (v >> sh) atomicOr(&dst[bp >> 5], bswap32(v >> sh));
   if (sh && (v << (32 - sh))) atomicOr(&dst[(bp >> 5) + 1], bswap32(v << (32 - sh)));
}

int concat_bits_device(u8* d_dst, u64 dst_bit, const u8* d_src, u64 nbits)
{
   if (nbits == 0) return 0;
   const u64 nwords = (nbits + 31) >> 5;
   k_concat_bits<<<(unsigned)((nwords + 255) / 256), 256>>>(reinterpret_cast<u32*>(d_dst), dst_bit, reinterpret_cast<const u32*>(d_src), nbits);
   if (cudaGetLastError() != cudaSuccess) return -1;
   return cudaDeviceSynchronize() == cudaSuccess ? 0 : -1;
}

// the same on a given stream, without synchronising (multi.cu: a window's output shifted to its bit position in the stream)
int concat_bits_stream(u8* d_dst, u64 dst_bit, const u8* d_src, u64 nbits, cudaStream_t st)
{
   if (nbits == 0) return 0;
   const u64 nwords = (nbits + 31) >> 5;
   k_concat_bits<<<(unsigned)((nwords + 255) / 256), 256, 0, st>>>(reinterpret_cast<u32*>(d_dst), dst_bit, reinterpret_cast<const u32*>(d_src), nbits);
   return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---- batch windows: every item is its own stream ------------------------------------------------
// Item i's stream is 32 header bits, its blocks in order, 80 trailer bits and padding to a byte (compress.c:841-845,
// :874-879); the streams are laid back to back from bit 0.  One CTA: the byte length of every item, their exclusive scan
// -> ibyte[0..n] (ibyte[n] = bytes of the window), and the bit offset of every block inside its item's stream.
__global__ void __launch_bounds__(1024) k_item_offsets(const u64* bits, u64* bitoff, const u32* first, u32 n, u64* ibyte)
{
   __shared__ u64 wsum[32];
   __shared__ u64 s_run;
   if (threadIdx.x == 0) s_run = 0;
   __syncthreads();
   const u32 l = lane_id(), w = threadIdx.x >> 5;
   for (u32 base = 0; base < n; base += 1024) {
      const u32 i = base + threadIdx.x;
      u64 v = 0;
      if (i < n) {
         u64 nbits = 32 + 80;
         for (u32 b = first[i]; b < first[i + 1]; b++) nbits += bits[b];
         v = (nbits + 7) >> 3;
      }
      u64 inc = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const u64 q = __shfl_up_sync(FULL, inc, d); if (l >= (u32)d) inc += q; }
      if (l == 31) wsum[w] = inc;
      __syncthreads();
      u64 pre = s_run;
      for (u32 k = 0; k < w; k++) pre += wsum[k];
      if (i < n) {
         const u64 off = pre + inc - v;
         ibyte[i] = off;
         u64 bp = off * 8 + 32;
         for (u32 b = first[i]; b < first[i + 1]; b++) { bitoff[b] = bp; bp += bits[b]; }
      }
      __syncthreads();
      if (threadIdx.x == 1023) s_run = pre + inc;
      __syncthreads();
   }
   if (threadIdx.x == 0) { ibyte[n] = s_run; bitoff[first[n]] = s_run * 8; }
}

__device__ void put_bits_or(u32* outw, u64 bitpos, u64 value, int nbits)
{
   for (int done = 0; done < nbits;) {
      const u64 bp = bitpos + done;
      const u32 sh = (u32)(bp & 31);
      const int take = min(32 - (int)sh, nbits - done);
      const u32 chunk = (u32)((value >> (nbits - done - take)) & ((take == 32) ? 0xffffffffu : ((1u << take) - 1u)));
      atomicOr(&outw[bp >> 5], bswap32(chunk << (32 - sh - take)));
      done += take;
   }
}

// One thread per item: the "BZh<level>" header, and the trailer with the combined CRC of the item's blocks
// (compress.c:826-828).  An empty item is header and trailer only.  Runs after k_pack: headers and trailers are ORed
// into words the neighbouring streams share.
__global__ void __launch_bounds__(256) k_item_frames(u32* outw, const u64* ibyte, const u64* bits, const u32* first,
                                                     const u32* crc, u32* icrc, u32 n, u32 level)
{
   const u32 i = blockIdx.x * 256 + threadIdx.x;
   if (i >= n) return;
   const u64 b0 = ibyte[i] * 8;
   put_bits_or(outw, b0, 0x425A6830u + level, 32);
   u32 c = 0;
   u64 end = b0 + 32;
   for (u32 b = first[i]; b < first[i + 1]; b++) { c = ((c << 1) | (c >> 31)) ^ crc[b]; end += bits[b]; }
   put_bits_or(outw, end, 0x177245385090ULL, 48);
   put_bits_or(outw, end + 48, c, 32);
   icrc[i] = c;
}

static int stage4_frames(Engine* e, u32 n_items, u32 nb, u8* d_out)
{
   cudaStream_t st = e->stream;
   k_item_frames<<<(n_items + 255) / 256, 256, 0, st>>>(reinterpret_cast<u32*>(d_out), e->it.byteoff, e->bt.bits,
                                                         e->it.first, e->bt.crc, e->it.crc, n_items, (u32)e->level); BZ_KCHECK(e);
   BZ_CUDA(e, cudaMemcpyAsync(e->h_scalars + 16, e->bt.bitoff + nb, sizeof(u64), cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaStreamSynchronize(st));
   return 0;
}

// a batch window whose items are all empty: headers and trailers only
int stage4_empty_items(Engine* e, u32 n_items, u8* d_out, u64* end_bit_out)
{
   k_item_offsets<<<1, 1024, 0, e->stream>>>(e->bt.bits, e->bt.bitoff, e->it.first, n_items, e->it.byteoff); BZ_KCHECK(e);
   const int rc = stage4_frames(e, n_items, 0, d_out);
   if (rc) return rc;
   *end_bit_out = *reinterpret_cast<u64*>(e->h_scalars + 16);
   return 0;
}

int put_bits_device(Engine* e, u8* d_out, u64 origin_bit, u64 bitpos, u64 value, int nbits)
{
   k_put_bits<<<1, 1, 0, e->stream>>>(reinterpret_cast<u32*>(d_out), bitpos - origin_bit, value, nbits);
   BZ_KCHECK(e);
   return 0;
}

int stage4_run(Engine* e, u32 nb, u32 E, u8* d_out, u64 origin_bit, u64 start_bit, u64* end_bit_out, u32 n_items)
{
   (void)E;
   cudaStream_t st = e->stream;
   S4Params p;
   p.mtfv = e->mtfv; p.X = e->bt.X; p.nmtf = e->bt.nmtf; p.mtffreq = e->bt.mtffreq;
   p.inuse = e->bt.inuse; p.ninuse = e->bt.ninuse; p.crc = e->bt.crc; p.origptr = e->bt.origptr;
   p.sel = e->sel; p.hlen = e->hlen; p.hfreq = e->hfreq; p.hcode = e->hcode;
   p.grpbits = e->grpbits; p.pre = e->pre; p.prebits = e->prebits; p.ngroups = e->ngroups;
   p.bits = e->bt.bits; p.bitoff = e->bt.bitoff;

   const u32 max_nsel = (e->nmax + 16 + 1 + BZ_G_SIZE - 1) / BZ_G_SIZE;
   const dim3 gsel((max_nsel + SEL_THREADS - 1) / SEL_THREADS, nb);
   k_huff_init<<<(nb + 63) / 64, 64, 0, st>>>(p, nb);                                       BZ_KCHECK(e);
   for (int it = 0; it < BZ_N_ITERS; it++) {
      BZ_CUDA(e, cudaMemsetAsync(e->hfreq, 0, sizeof(i32) * 6 * BZ_MAX_ALPHA * nb, st));
      k_huff_select<0><<<gsel, SEL_THREADS, 0, st>>>(p);                                     BZ_KCHECK(e);
      k_huff_lengths<<<nb, 192, 0, st>>>(p);                                                 BZ_KCHECK(e);
   }
   BZ_CUDA(e, cudaMemsetAsync(e->pre, 0, (size_t)PRE_STRIDE * nb, st));
   k_huff_finish<<<nb, 192, 0, st>>>(p);                                                     BZ_KCHECK(e);
   if (n_items) { k_item_offsets<<<1, 1024, 0, st>>>(e->bt.bits, e->bt.bitoff, e->it.first, n_items, e->it.byteoff); BZ_KCHECK(e); }
   else { k_bit_offsets<<<1, 1024, 0, st>>>(e->bt.bits, e->bt.bitoff, nb, start_bit);        BZ_KCHECK(e); }
   k_huff_select<1><<<gsel, SEL_THREADS, 0, st>>>(p);                                        BZ_KCHECK(e);
   k_group_scan<<<nb, 1024, 0, st>>>(p);                                                     BZ_KCHECK(e);
   u32* outw = reinterpret_cast<u32*>(d_out);
   k_pack<<<gsel, SEL_THREADS, 0, st>>>(p, outw, origin_bit);                                BZ_KCHECK(e);
   k_pre_copy<<<dim3((PRE_STRIDE / 4 + 255) / 256, nb), 256, 0, st>>>(p, outw, origin_bit);  BZ_KCHECK(e);
   if (n_items) {
      const int rc = stage4_frames(e, n_items, nb, d_out);
      if (rc) return rc;
      *end_bit_out = *reinterpret_cast<u64*>(e->h_scalars + 16);
      return 0;
   }
   BZ_CUDA(e, cudaMemcpyAsync(e->h_scalars + 16, e->bt.bitoff + nb, sizeof(u64), cudaMemcpyDeviceToHost, st));
   BZ_CUDA(e, cudaStreamSynchronize(st));
   *end_bit_out = *reinterpret_cast<u64*>(e->h_scalars + 16);
   return 0;
}

} // namespace bz
