/*
 * oracle/bz2_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (see bz2_oracle.h).
 *
 * CPU restatement of the reference compression path, written from the format
 * and from the behaviour of the cited reference functions; nothing here is
 * used by libbz2_b200.so.
 */
#include "bz2_oracle.h"
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ CRC -- */
/* CRC-32/BZIP2: polynomial 0x04C11DB7, MSB first, init ~0, final NOT.
 * Follows bzlib_private.h:187-202 (BZ_UPDATE_CRC) with the table of
 * crctable.c:29-99 regenerated arithmetically. */
static uint32_t crc_tab[256];
static int crc_ready = 0;
static void crc_init(void)
{
   for (uint32_t b = 0; b < 256; b++) {
      uint32_t r = b << 24;
      for (int k = 0; k < 8; k++) r = (r & 0x80000000u) ? (r << 1) ^ 0x04C11DB7u : (r << 1);
      crc_tab[b] = r;
   }
   crc_ready = 1;
}
uint32_t orc_crc(const uint8_t* p, uint64_t n)
{
   if (!crc_ready) crc_init();
   uint32_t c = 0xFFFFFFFFu;
   for (uint64_t i = 0; i < n; i++) c = (c << 8) ^ crc_tab[(c >> 24) ^ p[i]];
   return ~c;
}

/* ----------------------------------------------------------------- RLE1 -- */
static inline int chunk_cost(int len) { return len < 4 ? len : 5; }

/* bzlib.c:211-315.  The input is a sequence of "chunks": maximal runs cut at
 * 255.  A chunk is written to the open block at the moment the byte after it
 * is consumed; the block closes once its size reaches nblockMAX (tested before
 * each byte), so blocks are whole numbers of chunks.  If exactly one input byte
 * remains when a block fills and that byte arrived in FINISH mode, it is
 * flushed into the same block (bzlib.c:276-308). */
int64_t orc_rle1_split(const uint8_t* in, uint64_t n, int level, int tail_merge,
                       orc_block* blocks, int64_t max_blocks)
{
   const int32_t nmax = 100000 * level - 19;           /* bzlib.c:190 */
   int64_t nb = 0;
   uint64_t pos = 0, begin = 0;
   int32_t fill = 0;
   while (pos < n) {
      uint8_t ch = in[pos];
      int len = 1;
      while (pos + len < n && len < 255 && in[pos + len] == ch) len++;
      pos += len;
      fill += chunk_cost(len);
      int close = 0;
      if (pos == n) close = 1;
      else if (fill >= nmax) {
         close = 1;
         if (tail_merge && pos + 1 == n) { fill += 1; pos = n; }
      }
      if (close) {
         if (nb < max_blocks) {
            blocks[nb].in_begin = begin; blocks[nb].in_end = pos;
            blocks[nb].nblock = fill;    blocks[nb].crc = orc_crc(in + begin, pos - begin);
         }
         nb++; begin = pos; fill = 0;
      }
   }
   return nb;
}

int32_t orc_rle1_emit(const uint8_t* in, uint64_t begin, uint64_t end,
                      uint8_t* out, uint8_t* in_use)
{
   int32_t o = 0;
   uint64_t pos = begin;
   memset(in_use, 0, 256);
   while (pos < end) {
      uint8_t ch = in[pos];
      int len = 1;
      while (pos + len < end && len < 255 && in[pos + len] == ch) len++;
      pos += len;
      in_use[ch] = 1;
      for (int k = 0; k < (len < 4 ? len : 4); k++) out[o++] = ch;
      if (len >= 4) { out[o++] = (uint8_t)(len - 4); in_use[len - 4] = 1; }
   }
   return o;
}

/* ------------------------------------------------------------------ BWT -- */
/* Contract of BZ2_blockSort (blocksort.c:1520-1545): rotations of the block
 * in lexicographic order; output byte k is the byte preceding rotation k;
 * origPtr is the rank of rotation 0.  Restated with Manber-Myers prefix
 * doubling over cyclic ranks (not the reference's divsufsort); when the block
 * is an exact power the tie among equal rotations is settled as the reference
 * settles it (tie_order.c). */
int32_t orc_bwt(const uint8_t* blk, int32_t n, uint8_t* bwt, int32_t* orig_ptr)
{
   if (n <= 0) return 0;
   int32_t* sa = malloc(sizeof(int32_t) * (size_t)n);
   int32_t* sb = malloc(sizeof(int32_t) * (size_t)n);
   int32_t* rk = malloc(sizeof(int32_t) * (size_t)n);
   int32_t* rn = malloc(sizeof(int32_t) * (size_t)n);
   int32_t* pos = malloc(sizeof(int32_t) * ((size_t)n + 257));
   int32_t cnt[257];
   memset(cnt, 0, sizeof cnt);
   for (int32_t i = 0; i < n; i++) cnt[blk[i] + 1]++;
   for (int c = 0; c < 256; c++) cnt[c + 1] += cnt[c];
   for (int32_t i = 0; i < n; i++) rk[i] = cnt[blk[i]];
   { int32_t fillp[256]; for (int c = 0; c < 256; c++) fillp[c] = cnt[c];
     for (int32_t i = 0; i < n; i++) sa[fillp[blk[i]]++] = i; }
   int32_t groups = 0;
   for (int c = 0; c < 256; c++) if (cnt[c + 1] > cnt[c]) groups++;
   for (int64_t h = 1; groups < n && h < n; h *= 2) {
      /* order by second key: walk sa, shifting each index back by h */
      for (int32_t k = 0; k < n; k++) {
         int64_t i = (int64_t)sa[k] - (h % n); if (i < 0) i += n;
         sb[k] = (int32_t)i;
      }
      /* stable placement by first key; a group's slots start at its rank */
      for (int32_t k = 0; k < n; k++) pos[k] = k;
      for (int32_t k = 0; k < n; k++) { int32_t i = sb[k]; sa[pos[rk[i]]++] = i; }
      groups = 0;
      int32_t cur = 0;
      for (int32_t k = 0; k < n; k++) {
         if (k == 0) { cur = 0; groups = 1; }
         else {
            int32_t a = sa[k - 1], b = sa[k];
            int32_t a2 = (int32_t)(((int64_t)a + h) % n), b2 = (int32_t)(((int64_t)b + h) % n);
            if (rk[a] != rk[b] || rk[a2] != rk[b2]) { cur = k; groups++; }
         }
         rn[sa[k]] = cur;
      }
      int32_t* t = rk; rk = rn; rn = t;
   }
   for (int32_t k = 0; k < n; k++) bwt[k] = blk[sa[k] == 0 ? n - 1 : sa[k] - 1];
   *orig_ptr = rk[0];
   int32_t q = n / groups;
   free(sa); free(sb); free(rk); free(rn); free(pos);
   /* exact power: rk[0] is the start of rotation 0's tie group; the reference's value is that plus
    * the trace of its sorter's tie order (oracle/tie_order.c) */
   if (q > 1) *orig_ptr += orc_tie_offset(blk, n, q);
   return q;
}

/* ------------------------------------------------------------------ MTF -- */
/* compress.c:93-229: move-to-front over the ascending list of in-use bytes,
 * zero runs in bijective base 2 (RUNA=0, RUNB=1), position p>0 -> p+1,
 * EOB = nInUse+1. */
static int32_t put_run(uint16_t* mtfv, int32_t o, int32_t* freq, int64_t run)
{
   int64_t z = run - 1;
   for (;;) {
      int s = (int)(z & 1);
      mtfv[o++] = (uint16_t)s; freq[s]++;
      if (z < 2) break;
      z = (z - 2) >> 1;
   }
   return o;
}
int32_t orc_mtf(const uint8_t* bwt, int32_t n, const uint8_t* in_use,
                uint16_t* mtfv, int32_t* freq, int32_t* n_in_use)
{
   uint8_t list[256];
   int32_t nu = 0, o = 0;
   int64_t run = 0;
   for (int c = 0; c < 256; c++) if (in_use[c]) list[nu++] = (uint8_t)c;
   for (int i = 0; i < 258; i++) freq[i] = 0;
   for (int32_t i = 0; i < n; i++) {
      uint8_t c = bwt[i];
      if (list[0] == c) { run++; continue; }
      if (run) { o = put_run(mtfv, o, freq, run); run = 0; }
      int p = 1;
      uint8_t prev = list[0];
      while (list[p] != c) { uint8_t t = list[p]; list[p] = prev; prev = t; p++; }
      list[p] = prev; list[0] = c;
      mtfv[o++] = (uint16_t)(p + 1); freq[p + 1]++;
   }
   if (run) o = put_run(mtfv, o, freq, run);
   mtfv[o++] = (uint16_t)(nu + 1); freq[nu + 1]++;
   *n_in_use = nu;
   return o;
}

/* -------------------------------------------------------------- Huffman -- */
/* huffman.c:63-148.  Weights are freq<<8 with the subtree depth in the low
 * byte; ties are broken by the exact binary-heap mechanics, which are restated
 * here (1-based heap with a zero-weight sentinel at slot 0). */
typedef struct { int32_t heap[260]; int32_t w[516]; int32_t par[516]; int32_t nheap; } hb_t;

static void hb_up(hb_t* h, int32_t z)
{
   int32_t t = h->heap[z];
   while (h->w[t] < h->w[h->heap[z >> 1]]) { h->heap[z] = h->heap[z >> 1]; z >>= 1; }
   h->heap[z] = t;
}
static void hb_down(hb_t* h, int32_t z)
{
   int32_t t = h->heap[z];
   for (;;) {
      int32_t y = z << 1;
      if (y > h->nheap) break;
      if (y < h->nheap && h->w[h->heap[y + 1]] < h->w[h->heap[y]]) y++;
      if (h->w[t] < h->w[h->heap[y]]) break;
      h->heap[z] = h->heap[y];
      z = y;
   }
   h->heap[z] = t;
}
static int32_t hb_pop(hb_t* h)
{
   int32_t top = h->heap[1];
   h->heap[1] = h->heap[h->nheap--];
   hb_down(h, 1);
   return top;
}
/* returns how many times the weights were halved to meet max_len */
static int32_t make_code_lengths(int32_t* len, const int32_t* freq, int32_t alpha, int32_t max_len)
{
   hb_t h;
   int32_t halvings = 0;
   for (int32_t i = 0; i < alpha; i++) h.w[i + 1] = (freq[i] == 0 ? 1 : freq[i]) << 8;
   for (;;) {
      int32_t nnodes = alpha;
      h.nheap = 0; h.heap[0] = 0; h.w[0] = 0; h.par[0] = -2;
      for (int32_t i = 1; i <= alpha; i++) { h.par[i] = -1; h.heap[++h.nheap] = i; hb_up(&h, h.nheap); }
      while (h.nheap > 1) {
         int32_t a = hb_pop(&h), b = hb_pop(&h);
         nnodes++;
         h.par[a] = h.par[b] = nnodes;
         uint32_t wa = (uint32_t)h.w[a], wb = (uint32_t)h.w[b];
         uint32_t da = wa & 0xff, db = wb & 0xff;
         h.w[nnodes] = (int32_t)(((wa & 0xffffff00u) + (wb & 0xffffff00u)) | (1 + (da > db ? da : db)));
         h.par[nnodes] = -1;
         h.heap[++h.nheap] = nnodes; hb_up(&h, h.nheap);
      }
      int too_long = 0;
      for (int32_t i = 1; i <= alpha; i++) {
         int32_t d = 0, k = i;
         while (h.par[k] >= 0) { k = h.par[k]; d++; }
         len[i - 1] = d;
         if (d > max_len) too_long = 1;
      }
      if (!too_long) break;
      halvings++;
      for (int32_t i = 1; i <= alpha; i++) h.w[i] = (1 + (h.w[i] >> 8) / 2) << 8;
   }
   return halvings;
}
void orc_make_code_lengths(int32_t* len, const int32_t* freq, int32_t alpha, int32_t max_len)
{
   (void)make_code_lengths(len, freq, alpha, max_len);
}
void orc_assign_codes(int32_t* code, const int32_t* len, int32_t min_len, int32_t max_len, int32_t alpha)
{
   int32_t v = 0;
   for (int32_t L = min_len; L <= max_len; L++) {
      for (int32_t i = 0; i < alpha; i++) if (len[i] == L) code[i] = v++;
      v <<= 1;
   }
}

/* ------------------------------------------------------------ bit writer -- */
/* compress.c:37-86: MSB-first.  `out` must be zero beyond *bitpos; out == NULL only counts the bits. */
static void put_bits(uint8_t* out, uint64_t* bitpos, int nb, uint32_t v)
{
   uint64_t p = *bitpos;
   if (!out) { *bitpos = p + (uint64_t)nb; return; }
   for (int k = nb - 1; k >= 0; k--, p++)
      if ((v >> k) & 1) out[p >> 3] |= (uint8_t)(0x80u >> (p & 7));
   *bitpos = p;
}

/* ------------------------------------------------------- sendMTFValues -- */
/* The body of orc_send_mtf and orc_send_mtf_tables: selectors go to sel (nsel entries), the final code lengths
 * to len, the halving count of every (pass, table) to halvings (or nowhere if NULL).  Returns nGroups. */
static int send_mtf(const uint16_t* mtfv, int32_t n_mtf, const uint8_t* in_use, const int32_t* mtf_freq,
                    uint8_t* out, uint64_t* bitpos, uint8_t* sel, int32_t len[6][258], int32_t halvings[4][6])
{
   static const int NG_MAX = 6, GS = 50;
   int32_t code[6][258], fr[6][258];
   int32_t n_in_use = 0;
   for (int c = 0; c < 256; c++) n_in_use += in_use[c] ? 1 : 0;
   const int32_t alpha = n_in_use + 2;
   int ng = n_mtf < 200 ? 2 : n_mtf < 600 ? 3 : n_mtf < 1200 ? 4 : n_mtf < 2400 ? 5 : 6;   /* compress.c:266-270 */
   (void)NG_MAX;
   /* initial partition, compress.c:276-319 */
   for (int t = 0; t < ng; t++) for (int v = 0; v < alpha; v++) len[t][v] = 15;
   {
      int32_t part = ng, rem = n_mtf, gs = 0;
      while (part > 0) {
         int32_t target = rem / part, ge = gs - 1, acc = 0;
         while (acc < target && ge < alpha - 1) { ge++; acc += mtf_freq[ge]; }
         if (ge > gs && part != ng && part != 1 && ((ng - part) % 2 == 1)) { acc -= mtf_freq[ge]; ge--; }
         for (int32_t v = gs; v <= ge; v++) len[part - 1][v] = 0;
         part--; gs = ge + 1; rem -= acc;
      }
   }
   int32_t nsel = (n_mtf + GS - 1) / GS;
   /* refinement passes, compress.c:324-561 */
   for (int it = 0; it < 4; it++) {
      memset(fr, 0, sizeof fr);
      for (int32_t g = 0; g < nsel; g++) {
         int32_t lo = g * GS, hi = lo + GS; if (hi > n_mtf) hi = n_mtf;
         int32_t cost[6] = {0, 0, 0, 0, 0, 0};
         for (int32_t i = lo; i < hi; i++) for (int t = 0; t < ng; t++) cost[t] += len[t][mtfv[i]];
         int bt = 0;
         for (int t = 1; t < ng; t++) if (cost[t] < cost[bt]) bt = t;
         sel[g] = (uint8_t)bt;
         for (int32_t i = lo; i < hi; i++) fr[bt][mtfv[i]]++;
      }
      for (int t = 0; t < ng; t++) {
         const int32_t h = make_code_lengths(len[t], fr[t], alpha, 17);
         if (halvings) halvings[it][t] = h;
      }
   }
   for (int t = 0; t < ng; t++) {
      int32_t mn = 32, mx = 0;
      for (int v = 0; v < alpha; v++) { if (len[t][v] > mx) mx = len[t][v]; if (len[t][v] < mn) mn = len[t][v]; }
      orc_assign_codes(code[t], len[t], mn, mx, alpha);
   }
   /* symbol map, compress.c:654-675 */
   {
      uint32_t used16 = 0;
      for (int i = 0; i < 16; i++) { int any = 0; for (int j = 0; j < 16; j++) any |= in_use[i * 16 + j] ? 1 : 0; used16 = (used16 << 1) | (uint32_t)any; }
      put_bits(out, bitpos, 16, used16);
      for (int i = 0; i < 16; i++) if (used16 & (0x8000u >> i)) {
         uint32_t v = 0; for (int j = 0; j < 16; j++) v = (v << 1) | (in_use[i * 16 + j] ? 1u : 0u);
         put_bits(out, bitpos, 16, v);
      }
   }
   /* selectors, MTF-coded then unary, compress.c:573-631 and :680-689 */
   put_bits(out, bitpos, 3, (uint32_t)ng);
   put_bits(out, bitpos, 15, (uint32_t)nsel);
   {
      uint8_t order[6] = {0, 1, 2, 3, 4, 5};
      for (int32_t g = 0; g < nsel; g++) {
         int p = 0; while (order[p] != sel[g]) p++;
         for (int k = p; k > 0; k--) order[k] = order[k - 1];
         order[0] = sel[g];
         for (int k = 0; k < p; k++) put_bits(out, bitpos, 1, 1);
         put_bits(out, bitpos, 1, 0);
      }
   }
   /* delta-coded code lengths, compress.c:694-706 */
   for (int t = 0; t < ng; t++) {
      int32_t cur = len[t][0];
      put_bits(out, bitpos, 5, (uint32_t)cur);
      for (int v = 0; v < alpha; v++) {
         while (cur < len[t][v]) { put_bits(out, bitpos, 2, 2); cur++; }
         while (cur > len[t][v]) { put_bits(out, bitpos, 2, 3); cur--; }
         put_bits(out, bitpos, 1, 0);
      }
   }
   /* payload, compress.c:713-812 */
   for (int32_t i = 0; i < n_mtf; i++) {
      int t = sel[i / GS];
      put_bits(out, bitpos, len[t][mtfv[i]], (uint32_t)code[t][mtfv[i]]);
   }
   return ng;
}

void orc_send_mtf(const uint16_t* mtfv, int32_t n_mtf, const uint8_t* in_use,
                  const int32_t* mtf_freq, uint8_t* out, uint64_t* bitpos)
{
   int32_t len[6][258];
   uint8_t* sel = malloc((size_t)(n_mtf + 49) / 50 + 1);
   (void)send_mtf(mtfv, n_mtf, in_use, mtf_freq, out, bitpos, sel, len, NULL);
   free(sel);
}

int32_t orc_send_mtf_tables(const uint16_t* mtfv, int32_t n_mtf, const uint8_t* in_use, const int32_t* mtf_freq,
                            uint8_t* sel, int32_t len[6][258], int32_t halvings[4][6], uint64_t* coded_bits)
{
   uint64_t bits = 0;
   memset(len, 0, sizeof(int32_t) * 6 * 258);
   memset(halvings, 0, sizeof(int32_t) * 4 * 6);
   const int ng = send_mtf(mtfv, n_mtf, in_use, mtf_freq, NULL, &bits, sel, len, halvings);
   *coded_bits = bits;
   return ng;
}

/* ---------------------------------------------------------- whole stream -- */
/* flags: 2 = no stream header, 4 = no trailer (segment of a sharded stream).  *bits_out gets the
 * exact bit length, *fold_out the combined-CRC fold of this call's blocks started from 0. */
int64_t orc_compress_ex(const uint8_t* in, uint64_t n, int level, int tail_merge, unsigned flags,
                        const int32_t* force_orig_ptr, uint8_t* out, uint64_t out_cap,
                        uint64_t* bits_out, uint32_t* fold_out, uint32_t* nblocks_out)
{
   int64_t max_blocks = (int64_t)(n / (uint64_t)(100000 * level - 19 - 5)) + 2;
   orc_block* blocks = malloc(sizeof(orc_block) * (size_t)max_blocks);
   int64_t nb = orc_rle1_split(in, n, level, tail_merge, blocks, max_blocks);
   if (nb > max_blocks) { free(blocks); return -1; }
   memset(out, 0, (size_t)out_cap);
   uint64_t bp = 0;
   uint8_t* blk = malloc(900000 + 16);
   uint8_t* bwt = malloc(900000 + 16);
   uint16_t* mtfv = malloc(sizeof(uint16_t) * (900000 + 16));
   uint32_t comb = 0;
   if (!(flags & 2u)) { put_bits(out, &bp, 24, 0x425A68); put_bits(out, &bp, 8, (uint32_t)('0' + level)); }   /* compress.c:841-845 */
   for (int64_t b = 0; b < nb; b++) {
      uint8_t in_use[256];
      int32_t freq[258], nu, op;
      /* worst case for one block: ~ 1.3 * nblock + tables */
      if ((bp >> 3) + (uint64_t)blocks[b].nblock + (uint64_t)blocks[b].nblock / 4 + 40000 > out_cap) { free(blocks); free(blk); free(bwt); free(mtfv); return -2; }
      int32_t nblock = orc_rle1_emit(in, blocks[b].in_begin, blocks[b].in_end, blk, in_use);
      if (nblock != blocks[b].nblock) { free(blocks); free(blk); free(bwt); free(mtfv); return -3; }
      const int32_t q = orc_bwt(blk, nblock, bwt, &op);
      (void)q;
      if (force_orig_ptr && force_orig_ptr[b] >= 0) op = force_orig_ptr[b];
      int32_t nm = orc_mtf(bwt, nblock, in_use, mtfv, freq, &nu);
      comb = ((comb << 1) | (comb >> 31)) ^ blocks[b].crc;                                /* compress.c:826-828 */
      put_bits(out, &bp, 24, 0x314159); put_bits(out, &bp, 24, 0x265359);                /* compress.c:849-850 */
      put_bits(out, &bp, 16, blocks[b].crc >> 16); put_bits(out, &bp, 16, blocks[b].crc & 0xffff);
      put_bits(out, &bp, 1, 0);
      put_bits(out, &bp, 24, (uint32_t)op);
      orc_send_mtf(mtfv, nm, in_use, freq, out, &bp);
   }
   if (!(flags & 4u)) {
      put_bits(out, &bp, 24, 0x177245); put_bits(out, &bp, 24, 0x385090);                /* compress.c:872-880 */
      put_bits(out, &bp, 16, comb >> 16); put_bits(out, &bp, 16, comb & 0xffff);
   }
   if (bits_out) *bits_out = bp;
   if (fold_out) *fold_out = comb;
   if (nblocks_out) *nblocks_out = (uint32_t)nb;
   free(blocks); free(blk); free(bwt); free(mtfv);
   return (int64_t)((bp + 7) >> 3);
}

int64_t orc_compress(const uint8_t* in, uint64_t n, int level, int tail_merge,
                     const int32_t* force_orig_ptr, uint8_t* out, uint64_t out_cap)
{
   return orc_compress_ex(in, n, level, tail_merge, 0, force_orig_ptr, out, out_cap, 0, 0, 0);
}

/* First block boundary >= limit when blocks are laid greedily from the boundary `start`
 * (bzlib.c:227, :383); n_blocks = blocks in [start, boundary).  Returns n if the input ends first
 * (input_ends) or UINT64_MAX if more data is needed. */
uint64_t orc_find_boundary(const uint8_t* in, uint64_t n, uint64_t start, uint64_t limit, int level,
                           int tail_merge, int input_ends, uint32_t* n_blocks)
{
   const int32_t nmax = 100000 * level - 19;
   uint64_t pos = start, bnd = start;
   int32_t fill = 0;
   uint32_t nb = 0;
   while (bnd < limit) {
      if (pos >= n) { if (!input_ends) return UINT64_MAX; if (fill) nb++; bnd = n; break; }
      uint8_t ch = in[pos];
      int len = 1;
      while (pos + len < n && len < 255 && in[pos + len] == ch) len++;
      if (pos + len == n && !input_ends && len < 255) return UINT64_MAX;   /* chunk may continue in unseen data */
      pos += len;
      fill += chunk_cost(len);
      if (fill >= nmax) {
         if (input_ends && tail_merge && pos + 1 == n) pos = n;
         bnd = pos; fill = 0; nb++;
      }
   }
   if (n_blocks) *n_blocks = nb;
   return bnd;
}
