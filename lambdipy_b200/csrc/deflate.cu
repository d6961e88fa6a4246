// deflate.cu -- chunked, deterministic DEFLATE (RFC 1951) of an HBM-resident byte stream, plus CRC-32.
//
// Replaces the zlib level-9 stream `tarfile.open(path, "w:gz")` writes in
// PackageBuild.create_compressed_tarball (/root/reference/lambdipy/package_build.py:165-172).
//
// The input is cut into DEFLATE_CHUNK-byte chunks; one CTA compresses one chunk into its own output slot:
//   1. hash every 3-byte position of the chunk and of the 32 KiB before it (the history, which is also input);
//   2. stable counting sort of the positions by hash (per-warp segments, __match_any_sync ranks): the sorted
//      array holds, for every position, its exact hash chain in position order, so the candidate set is a pure
//      function of the bytes (no atomic list heads);
//   3. every position of the chunk walks at most MAX_CHAIN (32) predecessors of its chain (<= 32 KiB back) and
//      keeps the longest match (nearest on ties);
//   4. one thread parses lazily (zlib deflate_slow rules) over the per-position match lengths in shared memory;
//   5. histogram, length-limited canonical Huffman codes (15 / 7 bits), run-length coded header;
//   6. exact bit counts of the stored, fixed and dynamic encodings pick the block type;
//   7. per-thread bit counts, a CTA scan and atomicOr into a shared-memory bit buffer write the block;
//   8. non-final chunks end with an empty stored block (sync flush) so every slot is a whole number of bytes.
// Per-chunk CRC-32 is computed alongside (per-thread CRCs folded with the GF(2) shift operator).
// Thread 0 of each CTA adds the SM cycles of six phases (hash sort, scatter, match, parse, Huffman + header,
// emit) to DeflateArgs::phase_cycles: the per-phase split lb2_gzip_stats reports.
#include "lb2_common.cuh"

namespace lb2 {

namespace {

constexpr int NT = DEFLATE_THREADS;
constexpr uint32_t CHUNK = DEFLATE_CHUNK;
constexpr uint32_t HIST = DEFLATE_HIST;
constexpr uint32_t WIN = CHUNK + HIST;
constexpr int HBITS = 13, NB = 1 << HBITS, NSEG = 4;
constexpr int PPT = CHUNK / NT;            // chunk positions per thread (contiguous)
constexpr int MAX_CHAIN = 32, NICE = 128, MAX_LAZY = 32, MAXM = 258;
constexpr uint32_t OUTW = DEFLATE_SLOT / 4;
constexpr uint16_t F_START = 0x4000, F_MATCH = 0x8000, LEN_MASK = 0x1ff;

// shared memory: R0 = sort histogram, then per-position match lengths; R1 = bucket starts, then the bit buffer
constexpr uint32_t R0_BYTES = NB * NSEG * 4;       // == CHUNK * 2
constexpr uint32_t R1_BYTES = OUTW * 4;
static_assert(R0_BYTES == CHUNK * 2, "R0 holds either the histogram or the uint16 lengths");
static_assert(R1_BYTES >= NB * 4, "R1 holds the bucket starts");

struct Tree {           // scratch of one serial Huffman build
  uint32_t w[2 * 288];
  uint16_t par[2 * 288];
  uint16_t sym[288];
};
struct Small {
  uint32_t crc_tab[256];
  uint32_t lfreq[288], dfreq[32], cfreq[20];
  uint16_t lcode[288], dcode[32], ccode[20];
  uint8_t llen[288], dlen[32], clen[20];
  uint16_t rle[320];
  uint32_t scan[NT / 32 + 1];
  uint32_t crc[NT], clen_n[NT];
  Tree tr[2];
  uint32_t n_rle, hlit, hdist, hclen, btype, hdr_bits, body_bits;
};
constexpr uint32_t SMEM_BYTES = R0_BYTES + R1_BYTES + sizeof(Small);

__device__ __forceinline__ uint64_t umin64(uint64_t x, uint64_t y) { return x < y ? x : y; }

__device__ __forceinline__ uint32_t ld4(const uint8_t *p) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint32_t *q = reinterpret_cast<const uint32_t *>(a & ~uintptr_t(3));
  const uint32_t sh = (uint32_t)(a & 3) * 8;
  const uint32_t lo = __ldg(q);
  return sh ? __funnelshift_r(lo, __ldg(q + 1), sh) : lo;   // q[1] holds p[3]: inside the buffer
}

__device__ __forceinline__ uint32_t hash3(const uint8_t *p) {
  const uint32_t v = (uint32_t)__ldg(p) | ((uint32_t)__ldg(p + 1) << 8) | ((uint32_t)__ldg(p + 2) << 16);
  return (v * 0x9E3779B1u) >> (32 - HBITS);
}

__device__ __forceinline__ uint32_t match_len(const uint8_t *a, const uint8_t *b, uint32_t maxlen) {
  uint32_t l = 0;
  for (; l + 4 <= maxlen; l += 4) {
    const uint32_t x = ld4(a + l) ^ ld4(b + l);
    if (x) return l + ((__ffs(x) - 1) >> 3);
  }
  while (l < maxlen && __ldg(a + l) == __ldg(b + l)) l++;
  return l;
}

// block-wide exclusive scan; returns the exclusive prefix, *total = sum over the CTA
__device__ uint32_t block_scan(uint32_t v, uint32_t *ws, uint32_t *total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  __syncthreads();
  if (lane == 31) ws[warp] = x;
  __syncthreads();
  if (warp == 0) {
    uint32_t s = lane < NT / 32 ? ws[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += y;
    }
    if (lane < NT / 32) ws[lane] = s;
  }
  __syncthreads();
  const uint32_t before = warp ? ws[warp - 1] : 0;
  const uint32_t t = ws[NT / 32 - 1];
  __syncthreads();
  *total = t;
  return before + x - v;
}

// ---------------------------------------------------------------- length / distance symbols (RFC 1951 3.2.5)
__device__ __forceinline__ void len_sym(uint32_t L, uint32_t &sym, uint32_t &ebits, uint32_t &eval) {
  const uint32_t l = L - 3;
  if (L == 258) { sym = 285; ebits = 0; eval = 0; }
  else if (l < 8) { sym = 257 + l; ebits = 0; eval = 0; }
  else { const uint32_t e = 31 - __clz(l) - 2; sym = 261 + 4 * e + ((l >> e) & 3); ebits = e; eval = l & ((1u << e) - 1); }
}
__device__ __forceinline__ void dist_sym(uint32_t D, uint32_t &sym, uint32_t &ebits, uint32_t &eval) {
  const uint32_t d = D - 1;
  if (d < 4) { sym = d; ebits = 0; eval = 0; }
  else { const uint32_t e = 31 - __clz(d) - 1; sym = 2 * e + 2 + ((d >> e) & 1); ebits = e; eval = d & ((1u << e) - 1); }
}
__device__ __forceinline__ uint32_t len_extra(uint32_t s) { return (s >= 265 && s < 285) ? (s - 261) >> 2 : 0; }
__device__ __forceinline__ uint32_t dist_extra(uint32_t s) { return s < 4 ? 0 : (s >> 1) - 1; }

__device__ __forceinline__ void put_bits(uint32_t *w, uint32_t off, uint32_t v, uint32_t n) {
  if (!n) return;
  const uint64_t x = (uint64_t)v << (off & 31);
  atomicOr(w + (off >> 5), (uint32_t)x);
  if ((off & 31) + n > 32) atomicOr(w + (off >> 5) + 1, (uint32_t)(x >> 32));
}

// Huffman code lengths of freq[0..n) limited to `limit` bits, one thread.  Ties break by symbol index, so the
// result is a function of the frequencies.  At least two symbols get a code (RFC 1951 inflaters want a
// complete code; zlib does the same).  Too-deep trees are rebuilt from halved frequencies.
__device__ void huff_lengths(uint32_t *freq, int n, int limit, uint8_t *len, Tree &t) {
  int used = 0;
  for (int s = 0; s < n; s++) used += freq[s] != 0;
  for (int s = 0; used < 2 && s < n; s++)
    if (!freq[s]) { freq[s] = 1; used++; }
  for (int s = 0; s < n; s++) len[s] = 0;
  for (int shift = 0;; shift++) {
    // leaves sorted by (weight, symbol): insertion sort, n <= 288
    int m = 0;
    for (int s = 0; s < n; s++) {
      if (!freq[s]) continue;
      const uint32_t w = shift ? ((freq[s] >> shift) | 1u) : freq[s];
      int j = m++;
      while (j > 0 && t.w[j - 1] > w) { t.w[j] = t.w[j - 1]; t.sym[j] = t.sym[j - 1]; j--; }
      t.w[j] = w; t.sym[j] = (uint16_t)s;
    }
    // two queues: leaves [0, m), internal nodes [m, 2m-1) created in nondecreasing weight order
    int li = 0, ii = m, nn = m;
    for (int k = 0; k < m - 1; k++) {
      int a, b;
      a = (li < m && (ii >= nn || t.w[li] <= t.w[ii])) ? li++ : ii++;
      b = (li < m && (ii >= nn || t.w[li] <= t.w[ii])) ? li++ : ii++;
      t.w[nn] = t.w[a] + t.w[b];
      t.par[a] = (uint16_t)nn; t.par[b] = (uint16_t)nn;
      nn++;
    }
    // depths: parents have larger indices than children; reuse w[] as depth
    t.w[nn - 1] = 0;
    int maxd = 0;
    for (int k = nn - 2; k >= 0; k--) {
      t.w[k] = t.w[t.par[k]] + 1;
      if (k < m && (int)t.w[k] > maxd) maxd = t.w[k];
    }
    if (maxd <= limit) {
      for (int k = 0; k < m; k++) len[t.sym[k]] = (uint8_t)t.w[k];
      return;
    }
  }
}

// canonical codes (RFC 1951 3.2.2), stored bit-reversed for LSB-first emission
__device__ void canon_codes(const uint8_t *len, int n, uint16_t *code) {
  uint32_t cnt[16] = {0}, next[16];
  for (int s = 0; s < n; s++) cnt[len[s]]++;
  cnt[0] = 0;
  uint32_t c = 0;
  for (int b = 1; b < 16; b++) { c = (c + cnt[b - 1]) << 1; next[b] = c; }
  for (int s = 0; s < n; s++)
    code[s] = len[s] ? (uint16_t)(__brev(next[len[s]]++) >> (32 - len[s])) : 0;
}

__device__ __forceinline__ uint32_t crc_multmodp(uint32_t a, uint32_t b) {   // a * b mod P (reflected)
  uint32_t p = 0;
  for (uint32_t m = 1u << 31; m; m >>= 1) {
    if (a & m) p ^= b;
    b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
  }
  return p;
}
__device__ uint32_t crc_shift_op(uint32_t nbytes) {   // x^(8 nbytes) mod P
  uint32_t p = 1u << 31, sq = 1u << 23;                // x^0, x^8
  for (; nbytes; nbytes >>= 1) {
    if (nbytes & 1) p = crc_multmodp(sq, p);
    sq = crc_multmodp(sq, sq);
  }
  return p;
}

const __device__ uint8_t CL_ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

}  // namespace

__global__ void __launch_bounds__(NT, 1) lb2_deflate_chunk_kernel(DeflateArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint32_t *hist = reinterpret_cast<uint32_t *>(smem);
  uint16_t *lens = reinterpret_cast<uint16_t *>(smem);
  uint32_t *bstart = reinterpret_cast<uint32_t *>(smem + R0_BYTES);
  uint32_t *outw = bstart;
  Small &sm = *reinterpret_cast<Small *>(smem + R0_BYTES + R1_BYTES);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t *S = a.scratch + (size_t)blockIdx.x * (WIN + CHUNK);
  uint32_t *idx = S + WIN;
  uint16_t *dists = a.dists + (size_t)blockIdx.x * CHUNK;

  for (int i = tid; i < 256; i += NT) {
    uint32_t c = i;
    for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
    sm.crc_tab[i] = c;
  }

  for (uint32_t c = blockIdx.x; c < a.n_chunks; c += gridDim.x) {
    const uint64_t base = (uint64_t)c * CHUNK;
    const uint32_t len = (uint32_t)umin64(CHUNK, a.n - base);
    const uint32_t hs = (uint32_t)umin64(HIST, base + a.hist);
    const uint8_t *w = a.in + base - hs;
    const uint32_t nW = hs + len;
    const uint32_t nH = nW >= 3 ? nW - 2 : 0;    // positions with 3 bytes
    const bool final_chunk = a.final_ && c == a.n_chunks - 1;
    long long t_ph = clock64();
#define PHASE(k)                                                                                 \
  if (tid == 0 && a.phase_cycles) {                                                              \
    const long long t_ = clock64();                                                              \
    atomicAdd(a.phase_cycles + (k), (unsigned long long)(t_ - t_ph));                            \
    t_ph = t_;                                                                                   \
  }

    // ---- 1. per-segment hash histogram
    for (int i = tid; i < NB * NSEG; i += NT) hist[i] = 0;
    for (int i = tid; i < 288; i += NT) sm.lfreq[i] = 0;
    for (int i = tid; i < 32; i += NT) sm.dfreq[i] = 0;
    __syncthreads();
    const uint32_t seg_len = (nH + NSEG - 1) / NSEG;
    for (uint32_t i = tid; i < nH; i += NT) atomicAdd(&hist[hash3(w + i) * NSEG + i / seg_len], 1u);
    __syncthreads();
    // ---- 2. exclusive scan in (hash, segment) order -> where each segment's positions of each hash go
    {
      constexpr int E = NB * NSEG / NT;
      uint32_t s = 0;
      for (int k = 0; k < E; k++) s += hist[tid * E + k];
      uint32_t tot;
      uint32_t run = block_scan(s, sm.scan, &tot);
      for (int k = 0; k < E; k++) {
        const uint32_t v = hist[tid * E + k];
        hist[tid * E + k] = run;
        if (((tid * E + k) % NSEG) == 0) bstart[(tid * E + k) / NSEG] = run;
        run += v;
      }
    }
    __syncthreads();
    PHASE(0);
    // ---- 3. stable scatter: warp `seg` walks its segment in position order
    if (warp < NSEG && seg_len) {
      const uint32_t b = warp * seg_len, e = min(nH, b + seg_len);
      for (uint32_t i0 = b; i0 < e; i0 += 32) {
        const uint32_t i = i0 + lane;
        const bool valid = i < e;
        const uint32_t mask = __ballot_sync(0xffffffffu, valid);
        if (valid) {
          const uint32_t h = hash3(w + i);
          const uint32_t grp = __match_any_sync(mask, h);
          const uint32_t rank = __popc(grp & ((1u << lane) - 1));
          const uint32_t slot = hist[h * NSEG + warp] + rank;
          S[slot] = i;
          if (i >= hs) idx[i - hs] = slot;
          __syncwarp(mask);
          if (lane == 31 - __clz(grp)) hist[h * NSEG + warp] += __popc(grp);
        }
        __syncwarp();
      }
    }
    __syncthreads();
    PHASE(1);
    // ---- 4. longest match per chunk position over its hash chain (lens[] overwrites hist[])
    for (uint32_t p = tid; p < len; p += NT) {
      const uint32_t i = hs + p;
      uint32_t best = 0, bd = 0;
      if (i + 3 <= nW) {
        const uint32_t h = hash3(w + i), bs = bstart[h];
        const uint32_t maxlen = min((uint32_t)MAXM, nW - i);
        const uint32_t j = idx[p];
        for (uint32_t k = 0, jj = j; k < MAX_CHAIN && jj > bs; k++) {
          const uint32_t q = S[--jj];
          const uint32_t d = i - q;
          if (d > HIST) break;
          if (best && __ldg(w + q + best) != __ldg(w + i + best)) continue;
          const uint32_t l = match_len(w + q, w + i, maxlen);
          if (l > best) { best = l; bd = d; if (l >= NICE || l == maxlen) break; }
        }
        if (best < 3 || (best == 3 && bd > 4096)) best = 0;   // zlib TOO_FAR
      }
      lens[p] = (uint16_t)best;
      dists[p] = (uint16_t)bd;
    }
    __syncthreads();
    PHASE(2);
    // ---- 5. lazy parse (one thread): a literal is emitted when the next position has a longer match
    if (tid == 0) {
      uint32_t p = 0;
      while (p < len) {
        const uint32_t L = lens[p];
        if (L >= 3) {
          if (L < MAX_LAZY && p + 1 < len && (lens[p + 1] & LEN_MASK) > L) { lens[p] = (uint16_t)(L | F_START); p++; continue; }
          lens[p] = (uint16_t)(L | F_START | F_MATCH);
          p += L;
        } else {
          lens[p] = (uint16_t)(L | F_START);
          p++;
        }
      }
    }
    __syncthreads();
    PHASE(3);
    // ---- 6. histogram of the tokens + CRC of the thread's bytes
    const uint32_t p0 = tid * PPT, p1 = min(len, p0 + (uint32_t)PPT);
    {
      uint32_t crc = 0xFFFFFFFFu;
      for (uint32_t p = p0; p < p1; p++) {
        const uint8_t byte = __ldg(w + hs + p);
        crc = sm.crc_tab[(crc ^ byte) & 0xff] ^ (crc >> 8);
        const uint16_t v = lens[p];
        if (!(v & F_START)) continue;
        if (v & F_MATCH) {
          uint32_t s, e, x;
          len_sym(v & LEN_MASK, s, e, x);
          atomicAdd(&sm.lfreq[s], 1u);
          dist_sym(dists[p], s, e, x);
          atomicAdd(&sm.dfreq[s], 1u);
        } else {
          atomicAdd(&sm.lfreq[byte], 1u);
        }
      }
      sm.crc[tid] = crc ^ 0xFFFFFFFFu;
      sm.clen_n[tid] = p1 > p0 ? p1 - p0 : 0;
    }
    __syncthreads();
    // fold the per-thread CRCs; then threads 0 and 32 build the two Huffman trees
    for (int st = 1; st < NT; st <<= 1) {
      if ((tid & (2 * st - 1)) == 0) {
        const uint32_t n2 = sm.clen_n[tid + st];
        if (n2) sm.crc[tid] = crc_multmodp(crc_shift_op(n2), sm.crc[tid]) ^ sm.crc[tid + st];
        sm.clen_n[tid] += n2;
      }
      __syncthreads();
    }
    if (tid == 0) {
      a.chunk_crc[c] = sm.crc[0];
      sm.lfreq[256] = 1;
      huff_lengths(sm.lfreq, 286, 15, sm.llen, sm.tr[0]);
      sm.llen[286] = sm.llen[287] = 0;
    } else if (tid == 32) {
      huff_lengths(sm.dfreq, 30, 15, sm.dlen, sm.tr[1]);
      sm.dlen[30] = sm.dlen[31] = 0;
    }
    __syncthreads();
    // ---- 7. header run-length coding, code-length code, exact sizes, block type
    if (tid == 0) {
      uint32_t hlit = 286, hdist = 30;
      while (hlit > 257 && !sm.llen[hlit - 1]) hlit--;
      while (hdist > 1 && !sm.dlen[hdist - 1]) hdist--;
      const uint32_t N = hlit + hdist;
      auto L = [&](uint32_t k) -> uint32_t { return k < hlit ? sm.llen[k] : sm.dlen[k - hlit]; };
      for (int s = 0; s < 19; s++) sm.cfreq[s] = 0;
      uint32_t nr = 0;
      for (uint32_t i = 0; i < N;) {
        const uint32_t v = L(i);
        uint32_t run = 1;
        while (i + run < N && L(i + run) == v) run++;
        if (v == 0) {
          while (run >= 11) { const uint32_t r = min(run, 138u); sm.rle[nr++] = (uint16_t)(18 | ((r - 11) << 5)); sm.cfreq[18]++; run -= r; i += r; }
          if (run >= 3) { sm.rle[nr++] = (uint16_t)(17 | ((run - 3) << 5)); sm.cfreq[17]++; i += run; run = 0; }
        } else {
          sm.rle[nr++] = (uint16_t)v; sm.cfreq[v]++; i++; run--;
          while (run >= 3) { const uint32_t r = min(run, 6u); sm.rle[nr++] = (uint16_t)(16 | ((r - 3) << 5)); sm.cfreq[16]++; run -= r; i += r; }
        }
        for (; run; run--, i++) { sm.rle[nr++] = (uint16_t)v; sm.cfreq[v]++; }
      }
      huff_lengths(sm.cfreq, 19, 7, sm.clen, sm.tr[0]);
      uint32_t hclen = 19;
      while (hclen > 4 && !sm.clen[CL_ORDER[hclen - 1]]) hclen--;
      uint64_t dyn = 3 + 5 + 5 + 4 + 3 * hclen;
      for (uint32_t k = 0; k < nr; k++) {
        const uint32_t s = sm.rle[k] & 31;
        dyn += sm.clen[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
      }
      uint64_t dyn_body = 0, fix_body = 0;
      for (int s = 0; s < 286; s++) {
        const uint32_t f = sm.lfreq[s];
        if (!f) continue;
        const uint32_t fl = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
        dyn_body += (uint64_t)f * (sm.llen[s] + len_extra(s));
        fix_body += (uint64_t)f * (fl + len_extra(s));
      }
      for (int s = 0; s < 30; s++) {
        const uint32_t f = sm.dfreq[s];
        if (!f) continue;
        dyn_body += (uint64_t)f * (sm.dlen[s] + dist_extra(s));
        fix_body += (uint64_t)f * (5 + dist_extra(s));
      }
      // lfreq/dfreq hold forced (unused) symbols with weight 1: they cost bits in the estimate only, never in
      // the stream -- the estimate is an upper bound of the bits written, and the choice stays deterministic
      const uint64_t flush = final_chunk ? 0 : 3;                       // empty stored block header, then align
      const uint64_t dyn_bytes = (dyn + dyn_body + flush + 7) / 8 + (final_chunk ? 0 : 4);
      const uint64_t fix_bytes = (3 + fix_body + flush + 7) / 8 + (final_chunk ? 0 : 4);
      const uint32_t nsb = len ? (len + 65534) / 65535 : 1;
      const uint64_t sto_bytes = (uint64_t)len + 5 * nsb + (final_chunk ? 0 : 5);
      uint32_t bt = 2;
      uint64_t best = dyn_bytes;
      if (fix_bytes <= best) { bt = 1; best = fix_bytes; }
      if (sto_bytes <= best) { bt = 0; }
      sm.btype = bt; sm.hlit = hlit; sm.hdist = hdist; sm.hclen = hclen; sm.n_rle = nr;
      if (bt == 1) {
        for (int s = 0; s < 288; s++) sm.llen[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
        for (int s = 0; s < 32; s++) sm.dlen[s] = 5;
      }
    }
    __syncthreads();
    PHASE(4);
    const uint32_t bt = sm.btype;
    uint8_t *slot = a.slots + (size_t)c * DEFLATE_SLOT;
    if (bt == 0) {
      // ---- stored: sub-blocks of <= 65535 bytes, then the sync flush
      const uint32_t nsb = len ? (len + 65534) / 65535 : 1;
      if (tid == 0) {
        for (uint32_t k = 0; k < nsb; k++) {
          const uint32_t b = k * 65535, l = min(65535u, len - b);
          uint8_t *h = slot + b + 5 * k;
          h[0] = (final_chunk && k == nsb - 1) ? 1 : 0;
          h[1] = l & 0xff; h[2] = l >> 8; h[3] = ~l & 0xff; h[4] = (~l >> 8) & 0xff;
        }
        uint32_t o = len + 5 * nsb;
        if (!final_chunk) { slot[o] = 0; slot[o + 1] = 0; slot[o + 2] = 0; slot[o + 3] = 0xff; slot[o + 4] = 0xff; o += 5; }
        a.out_size[c] = o;
      }
      for (uint32_t p = tid; p < len; p += NT) slot[p + 5 * (p / 65535 + 1)] = __ldg(w + hs + p);
      __syncthreads();
      PHASE(5);
      continue;
    }
    // ---- fixed / dynamic: codes, header, body bits, EOB, flush
    if (tid == 0) canon_codes(sm.llen, 288, sm.lcode);
    else if (tid == 32) canon_codes(sm.dlen, 32, sm.dcode);
    else if (tid == 64) canon_codes(sm.clen, 19, sm.ccode);
    for (uint32_t k = tid; k < OUTW; k += NT) outw[k] = 0;
    __syncthreads();
    uint32_t mybits = 0;
    for (uint32_t p = p0; p < p1; p++) {
      const uint16_t v = lens[p];
      if (!(v & F_START)) continue;
      if (v & F_MATCH) {
        uint32_t s, e, x;
        len_sym(v & LEN_MASK, s, e, x);
        mybits += sm.llen[s] + e;
        dist_sym(dists[p], s, e, x);
        mybits += sm.dlen[s] + e;
      } else {
        mybits += sm.llen[__ldg(w + hs + p)];
      }
    }
    if (tid == 0) {
      uint32_t o = 0;
      put_bits(outw, o, final_chunk ? 1 : 0, 1); o += 1;
      put_bits(outw, o, bt, 2); o += 2;
      if (bt == 2) {
        put_bits(outw, o, sm.hlit - 257, 5); o += 5;
        put_bits(outw, o, sm.hdist - 1, 5); o += 5;
        put_bits(outw, o, sm.hclen - 4, 4); o += 4;
        for (uint32_t k = 0; k < sm.hclen; k++) { put_bits(outw, o, sm.clen[CL_ORDER[k]], 3); o += 3; }
        for (uint32_t k = 0; k < sm.n_rle; k++) {
          const uint32_t s = sm.rle[k] & 31, x = sm.rle[k] >> 5;
          put_bits(outw, o, sm.ccode[s], sm.clen[s]); o += sm.clen[s];
          const uint32_t eb = s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0;
          put_bits(outw, o, x, eb); o += eb;
        }
      }
      sm.hdr_bits = o;
    }
    uint32_t total;
    const uint32_t excl = block_scan(mybits, sm.scan, &total);
    uint32_t o = sm.hdr_bits + excl;
    for (uint32_t p = p0; p < p1; p++) {
      const uint16_t v = lens[p];
      if (!(v & F_START)) continue;
      if (v & F_MATCH) {
        uint32_t s, e, x;
        len_sym(v & LEN_MASK, s, e, x);
        put_bits(outw, o, sm.lcode[s] | (x << sm.llen[s]), sm.llen[s] + e); o += sm.llen[s] + e;
        dist_sym(dists[p], s, e, x);
        put_bits(outw, o, sm.dcode[s] | (x << sm.dlen[s]), sm.dlen[s] + e); o += sm.dlen[s] + e;
      } else {
        const uint32_t s = __ldg(w + hs + p);
        put_bits(outw, o, sm.lcode[s], sm.llen[s]); o += sm.llen[s];
      }
    }
    if (tid == 0) {
      uint32_t e = sm.hdr_bits + total;
      put_bits(outw, e, sm.lcode[256], sm.llen[256]); e += sm.llen[256];
      uint32_t bytes;
      if (final_chunk) {
        bytes = (e + 7) / 8;
      } else {
        e += 3;                      // BFINAL=0, BTYPE=00
        bytes = (e + 7) / 8;         // LEN=0000, NLEN=FFFF follow at the byte boundary
        put_bits(outw, bytes * 8 + 16, 0xffffu, 16);
        bytes += 4;
      }
      sm.body_bits = bytes;
      a.out_size[c] = bytes;
    }
    __syncthreads();
    const uint32_t nw = (sm.body_bits + 3) / 4;
    uint32_t *dst = reinterpret_cast<uint32_t *>(slot);
    for (uint32_t k = tid; k < nw; k += NT) dst[k] = outw[k];
    __syncthreads();
    PHASE(5);
  }
}

void deflate_smem_setup() {
  cudaFuncSetAttribute(lb2_deflate_chunk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
}

void launch_deflate(const DeflateArgs &a, int grid, cudaStream_t s) {
  lb2_deflate_chunk_kernel<<<grid, NT, SMEM_BYTES, s>>>(a);
}

}  // namespace lb2
