// rtclj_png_kernels.cuh -- the compressed PNG writer on the device (DESIGN.md section 4.11).
//
// The bytes are fixed by the definition in include/rtclj_b200.h (rtclj_ctx_encode_png); tests/png_model.py
// reproduces them.  Three launches:
//   png_filter_kernel   one CTA per row: the five filters' costs (sum |byte as int8|), a CTA reduction picks the
//                       cheapest (lower type on a tie), the row goes to the filtered stream F
//   png_deflate_kernel  one CTA per 64 KiB segment of F, 64 bytes per thread:
//                         run starts of the thread's bytes as a 64-bit mask; the runs that cross threads by an
//                         exclusive max scan (start before the chunk) and min scan (start after it)
//                         tokens in closed form per byte -> histogram (shared atomics)
//                         package-merge (CTA-wide: rank sort, one merge step per level, leaf positions as bits)
//                         canonical codes, the code-length sequence and its own code
//                         bit count per thread, exclusive scan -> bit offsets; dynamic vs stored decided here
//                         whole words into shared memory, atomicOr only on the words a thread shares
//                         the segment -> its staging slot, {bytes, stored, Adler sums} -> its record
//   png_place_kernel    one CTA per segment (+ one for the rest): offset = sum of the records before it,
//                       chunk header + data + CRC-32 (per-thread CRCs of 128-byte slices, shifted by
//                       multiplication modulo the CRC polynomial and XORed); the last CTA writes signature, IHDR,
//                       the zlib header chunk, the Adler-32 chunk (per-segment sums combined mod 65521), IEND and
//                       the total length
// An animated PNG of a sequence of frames (DESIGN.md section 4.14) takes the same three steps per group of frames:
// png_filter_frames_kernel and png_deflate_frames_kernel (the two above over every frame of the group) and
// png_place_frames_kernel (the chunks with their sequence numbers, each frame's Adler-32 from its own records).
#pragma once
#include <cstddef>
#include <cstdint>

namespace rtclj {

constexpr int kPngFilterThreads = 256;
constexpr int kPngThreads = 1024;
constexpr int kPngSeg = 65536;                      // bytes of F per segment
constexpr int kPngChunk = kPngSeg / kPngThreads;     // 64 bytes per thread
constexpr int kPngSlot = 65552;                     // a dynamic segment is < its stored size (<= 65 546 bytes)
constexpr int kPngCrcSpan = 2 * kPngSeg;             // the place kernel's CRC: 1024 slices of 128 bytes
constexpr int kPngHead = 8 + 25 + 14;                // signature, IHDR, IDAT(78 01)
constexpr int kPngTail = 16 + 12;                    // IDAT(Adler-32), IEND
constexpr uint32_t kCrcPoly = 0xEDB88320u;

struct PngSegRec { unsigned bytes, stored, s1, s2; };  // s1 = sum of bytes, s2 = sum (n - i) * byte, both mod 65521

// The code-length code's order 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15, five bits per entry (the library
// keeps no module-global constant tables)
__device__ __forceinline__ int png_cl_order(int k) {
  constexpr unsigned long long lo = 16ull | 17ull << 5 | 18ull << 10 | 0ull << 15 | 8ull << 20 | 7ull << 25 | 9ull << 30 |
                                    6ull << 35 | 10ull << 40 | 5ull << 45 | 11ull << 50 | 4ull << 55;
  constexpr unsigned long long hi = 12ull | 3ull << 5 | 13ull << 10 | 2ull << 15 | 14ull << 20 | 1ull << 25 | 15ull << 30;
  return (int)((k < 12 ? lo >> (5 * k) : hi >> (5 * (k - 12))) & 31ull);
}
// base length of length symbol 257 + k (RFC 1951 3.2.5)
__device__ __forceinline__ int png_len_base(int k) {
  return k < 8 ? 3 + k : k == 28 ? 258 : ((4 + (k & 3)) << ((k - 4) >> 2)) + 3;
}

// ---- filtering
__device__ __forceinline__ int png_paeth(int a, int b, int c) {
  const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
  return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}
__device__ __forceinline__ unsigned png_filtered(int f, int x, int a, int b, int c) {
  const int pred = f == 0 ? 0 : f == 1 ? a : f == 2 ? b : f == 3 ? ((a + b) >> 1) : png_paeth(a, b, c);
  return (unsigned)(x - pred) & 0xffu;
}

__global__ void __launch_bounds__(kPngFilterThreads) png_filter_kernel(const unsigned char* __restrict__ rgb8,
                                                                       size_t row_bytes, unsigned char* __restrict__ F) {
  __shared__ unsigned long long red[kPngFilterThreads / 32][5];
  __shared__ int pick;
  const size_t y = blockIdx.x;
  const unsigned char* row = rgb8 + y * row_bytes;
  const unsigned char* prev = y ? row - row_bytes : nullptr;
  unsigned long long cost[5] = {0, 0, 0, 0, 0};
  for (size_t x = threadIdx.x; x < row_bytes; x += kPngFilterThreads) {
    const int v = row[x], a = x >= 3 ? row[x - 3] : 0, b = prev ? prev[x] : 0, c = (prev && x >= 3) ? prev[x - 3] : 0;
#pragma unroll
    for (int f = 0; f < 5; ++f) cost[f] += (unsigned)abs((int)(signed char)png_filtered(f, v, a, b, c));
  }
#pragma unroll
  for (int f = 0; f < 5; ++f) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cost[f] += __shfl_xor_sync(0xffffffffu, cost[f], d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][f] = cost[f];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int best = 0;
    unsigned long long bc = ~0ull;
    for (int f = 0; f < 5; ++f) {
      unsigned long long t = 0;
      for (int w = 0; w < kPngFilterThreads / 32; ++w) t += red[w][f];
      if (t < bc) { bc = t; best = f; }
    }
    pick = best;
  }
  __syncthreads();
  const int f = pick;
  unsigned char* dst = F + y * (row_bytes + 1);
  if (threadIdx.x == 0) dst[0] = (unsigned char)f;
  for (size_t x = threadIdx.x; x < row_bytes; x += kPngFilterThreads) {
    const int v = row[x], a = x >= 3 ? row[x - 3] : 0, b = prev ? prev[x] : 0, c = (prev && x >= 3) ? prev[x - 3] : 0;
    dst[1 + x] = (unsigned char)png_filtered(f, v, a, b, c);
  }
}

// ---- deflate: one CTA per segment
struct PngDeflateSmem {
  uint4 in[kPngSeg / 16];
  uint32_t out[kPngSlot / 4];
  uint32_t hist[288];
  uint32_t pm_a[576], pm_b[576], pm_pkg[288], pm_w[288];
  uint32_t pm_bits[15][18];  // per level: which merged positions are leaves (<= 571 positions)
  uint16_t pm_sym[288];
  int pm_c[16];
  uint32_t nxt_code[16];
  uint16_t ll_rev[288], cl_rev[20], lsym[259];  // lsym[len]: symbol - 257 | extra bits << 5 | extra value << 8
  uint8_t ll_len[288], cl_len[20];
  uint32_t cl_hist[20];
  uint8_t cl_sym[292], cl_xv[292];
  unsigned long long red[32];
  int scan_i[32];
  unsigned scan_u[32];
  int ncl, hlit, hclen, header_bits, n_cl_used;
  unsigned total_bits, dyn_bytes, stored;
};

__device__ __forceinline__ uint32_t png_byte(const uint4& v, int p) {  // byte p % 16 of a 16-byte group
  const int k = (p >> 2) & 3;
  const uint32_t x = k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w;
  return (x >> (8 * (p & 3))) & 0xffu;
}

__device__ __forceinline__ unsigned long long png_cta_sum(unsigned long long x, unsigned long long* red) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = x;
  __syncthreads();
  unsigned long long t = 0;
  for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += red[k];
  return t;
}

// Length-limited code lengths of freq[0..nsym) (>= 2 used symbols), CTA-wide.  Items are ordered by (frequency,
// symbol); level `limit` is the leaves, every level above merges the leaves with the pairs of the level below (a
// leaf before a package of equal weight); the first 2n - 2 items of level 1 are selected, and a leaf's length is
// the number of levels whose selected prefix holds it.
__device__ void png_package_merge(PngDeflateSmem& s, const uint32_t* freq, int nsym, int limit, uint8_t* len_out) {
  const int t = threadIdx.x;
  const uint32_t f = t < nsym ? freq[t] : 0u;
  const int n = __syncthreads_count(f != 0u);
  if (f) {
    int r = 0;
    for (int u = 0; u < nsym; ++u) {
      const uint32_t g = freq[u];
      r += (g != 0u) & ((g < f) | ((g == f) & (u < t)));
    }
    s.pm_sym[r] = (uint16_t)t;
    s.pm_w[r] = f;
  }
  for (int i = t; i < 15 * 18; i += blockDim.x) (&s.pm_bits[0][0])[i] = 0u;
  __syncthreads();
  uint32_t* cur = s.pm_a;
  uint32_t* nxt = s.pm_b;
  if (t < n) cur[t] = s.pm_w[t];
  int len = n;
  for (int lev = 1; lev < limit; ++lev) {  // pm_bits[lev]: the level `lev` steps above the leaves
    const int npk = len >> 1;
    __syncthreads();
    if (t < npk) s.pm_pkg[t] = cur[2 * t] + cur[2 * t + 1];
    __syncthreads();
    if (t < n) {
      const uint32_t w = s.pm_w[t];
      int lo = 0, hi = npk;  // packages lighter than w
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (s.pm_pkg[mid] < w) lo = mid + 1; else hi = mid; }
      const int pos = t + lo;
      nxt[pos] = w;
      atomicOr(&s.pm_bits[lev][pos >> 5], 1u << (pos & 31));
    } else if (t < n + npk) {
      const int j = t - n;
      const uint32_t w = s.pm_pkg[j];
      int lo = 0, hi = n;  // leaves no heavier than w
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (s.pm_w[mid] <= w) lo = mid + 1; else hi = mid; }
      nxt[j + lo] = w;
    }
    uint32_t* tmp = cur; cur = nxt; nxt = tmp;
    len = n + npk;
  }
  __syncthreads();
  if (t == 0) {
    int m = 2 * n - 2;
    for (int lev = limit - 1; lev >= 0; --lev) {
      int c = m;
      if (lev > 0) {
        c = 0;
        for (int k = 0; 32 * k < m; ++k) {
          const uint32_t bits = s.pm_bits[lev][k];
          const int left = m - 32 * k;
          c += __popc(left >= 32 ? bits : bits & ((1u << left) - 1u));
        }
      }
      s.pm_c[lev] = c;
      m = 2 * (m - c);
    }
  }
  if (t < nsym) len_out[t] = 0;
  __syncthreads();
  if (t < n) {
    int l = 0;
    for (int lev = 0; lev < limit; ++lev) l += t < s.pm_c[lev];
    len_out[s.pm_sym[t]] = (uint8_t)l;
  }
  __syncthreads();
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for LSB-first packing
__device__ void png_canonical(PngDeflateSmem& s, const uint8_t* len, int nsym, uint16_t* rev) {
  const int t = threadIdx.x;
  if (t < 16) {
    unsigned c = 0;
    for (int u = 0; u < nsym; ++u) c += len[u] == t;
    s.nxt_code[t] = t ? c : 0u;
  }
  __syncthreads();
  if (t == 0) {
    unsigned code = 0, prev = 0;
    for (int b = 1; b < 16; ++b) { code = (code + prev) << 1; prev = s.nxt_code[b]; s.nxt_code[b] = code; }
  }
  __syncthreads();
  if (t < nsym) {
    const int l = len[t];
    if (l) {
      unsigned r = 0;
      for (int u = 0; u < t; ++u) r += len[u] == l;
      rev[t] = (uint16_t)(__brev(s.nxt_code[l] + r) >> (32 - l));
    } else {
      rev[t] = 0;
    }
  }
  __syncthreads();
}

// The tokens whose first byte is in this thread's chunk [c0, c0 + cnt), in order: tok.lit(byte), tok.match(len).
// mask: bit p = a run starts at c0 + p; cin: the start of the run holding c0; cout: the first start after the chunk.
// The chunk's bytes are read from shared memory, 16 at a time (in registers they would spill at 1024 threads).
template <class Tok>
__device__ __forceinline__ void png_walk(const uint4* src, unsigned long long mask, int c0, int cnt, int cin,
                                         int cout, Tok& tok) {
  int s = cin;
  int e = mask ? c0 + __ffsll((long long)mask) - 1 : cout;
  int full = (e - s - 1) / 258, q = (e - s - 1) - 258 * full;
  uint4 v;
#pragma unroll
  for (int p = 0; p < kPngChunk; ++p) {
    if ((p & 15) == 0) v = src[p >> 4];
    if (p < cnt) {
      const int i = c0 + p;
      if ((mask >> p) & 1ull) {
        s = i;
        const unsigned long long rest = p < kPngChunk - 1 ? mask >> (p + 1) : 0ull;
        e = rest ? i + __ffsll((long long)rest) : cout;
        full = (e - s - 1) / 258;
        q = (e - s - 1) - 258 * full;
      }
      const int k = i - s;
      if (k == 0) {
        tok.lit(png_byte(v, p));
      } else {
        const int j = k - 1;
        if (j < 258 * full) {
          if (j % 258 == 0) tok.match(258);
        } else if (q >= 3) {
          if (j == 258 * full) tok.match(q);
        } else {
          tok.lit(png_byte(v, p));
        }
      }
    }
  }
}

struct PngHistTok {
  PngDeflateSmem* s;
  __device__ void lit(uint32_t b) { atomicAdd(&s->hist[b], 1u); }
  __device__ void match(int len) { atomicAdd(&s->hist[257 + (s->lsym[len] & 31)], 1u); }
};
struct PngCountTok {
  const PngDeflateSmem* s;
  unsigned bits;
  __device__ void lit(uint32_t b) { bits += s->ll_len[b]; }
  __device__ void match(int len) {
    const unsigned e = s->lsym[len];
    bits += s->ll_len[257 + (e & 31)] + ((e >> 5) & 7) + 1;  // code, extra bits, distance code 0 (one bit)
  }
};
struct PngBitOut {  // LSB-first; the first and last words of a thread may be shared with its neighbours
  uint32_t* out;
  unsigned widx;
  unsigned long long acc;
  int nacc;
  bool first;
  __device__ void init(uint32_t* o, unsigned bit) { out = o; widx = bit >> 5; nacc = (int)(bit & 31); acc = 0; first = true; }
  __device__ __forceinline__ void put(uint32_t v, int n) {
    acc |= (unsigned long long)v << nacc;
    nacc += n;
    if (nacc >= 32) {
      if (first) { atomicOr(out + widx, (uint32_t)acc); first = false; }
      else out[widx] = (uint32_t)acc;
      ++widx;
      acc >>= 32;
      nacc -= 32;
    }
  }
  __device__ void finish() { if (nacc > 0 && acc) atomicOr(out + widx, (uint32_t)acc); }
};
struct PngEmitTok {
  const PngDeflateSmem* s;
  PngBitOut* o;
  __device__ void lit(uint32_t b) { o->put(s->ll_rev[b], s->ll_len[b]); }
  __device__ void match(int len) {
    const unsigned e = s->lsym[len], sym = 257 + (e & 31), l = s->ll_len[sym];
    o->put(s->ll_rev[sym] | ((e >> 8) << l), (int)(l + ((e >> 5) & 7) + 1));
  }
};

__global__ void __launch_bounds__(kPngThreads, 1) png_deflate_kernel(const unsigned char* __restrict__ F, size_t N,
                                                                     unsigned char* __restrict__ staging,
                                                                     PngSegRec* __restrict__ rec) {
  extern __shared__ __align__(16) unsigned char png_deflate_smem[];
  PngDeflateSmem& s = *reinterpret_cast<PngDeflateSmem*>(png_deflate_smem);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const size_t seg = blockIdx.x;
  const size_t a0 = seg * (size_t)kPngSeg;
  const int n = (int)(N - a0 < (size_t)kPngSeg ? N - a0 : (size_t)kPngSeg);
  const bool last = a0 + (size_t)n == N;

  // load the segment; zero the output words and the histogram; the length table
  {
    const uint4* src = reinterpret_cast<const uint4*>(F + a0);
    for (int i = t; i < kPngSeg / 16; i += kPngThreads) {
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (16 * i + 16 <= n) {
        v = __ldg(src + i);
      } else if (16 * i < n) {
        uint32_t b[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int k = 0; k < 16; ++k)
          if (16 * i + k < n) b[k >> 2] |= (uint32_t)F[a0 + 16 * i + k] << (8 * (k & 3));
        v = make_uint4(b[0], b[1], b[2], b[3]);
      }
      s.in[i] = v;
    }
    for (int i = t; i < kPngSlot / 4; i += kPngThreads) s.out[i] = 0u;
    if (t < 288) s.hist[t] = 0u;
    if (t >= 3 && t <= 258) {
      int k = 0;
      while (k < 28 && png_len_base(k + 1) <= t) ++k;
      if (t == 258) k = 28;
      const int xb = (k >= 8 && k < 28) ? (k - 4) >> 2 : 0;
      s.lsym[t] = (uint16_t)(k | (xb << 5) | ((t - png_len_base(k)) << 8));
    }
  }
  __syncthreads();

  // this thread's 64 bytes, its run starts, its Adler sums
  const int c0 = t * kPngChunk;
  const int cnt = n - c0 < 0 ? 0 : (n - c0 > kPngChunk ? kPngChunk : n - c0);
  const uint4* w = s.in + 4 * t;
  unsigned long long mask = 0;
  unsigned s1 = 0, s2 = 0;
  {
    uint32_t prevb = t ? reinterpret_cast<const unsigned char*>(s.in)[c0 - 1] : 0x100u;
    uint4 v;
#pragma unroll
    for (int p = 0; p < kPngChunk; ++p) {
      if ((p & 15) == 0) v = w[p >> 4];
      const uint32_t b = png_byte(v, p);
      if (p < cnt) {
        if (b != prevb) mask |= 1ull << p;
        s1 += b;
        s2 += (unsigned)(cnt - p) * b;
      }
      prevb = b;
    }
  }
  // the start of the run holding c0 (exclusive max scan) and the first start after the chunk (exclusive min scan)
  int cin, cout;
  {
    const int last_start = mask ? c0 + 63 - __clzll((long long)mask) : -1;
    int inc = last_start;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc = max(inc, y); }
    int ex = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) ex = -1;
    if (lane == 31) s.scan_i[warp] = inc;
    __syncthreads();
    for (int k = 0; k < warp; ++k) ex = max(ex, s.scan_i[k]);
    cin = ex;
    __syncthreads();
    const int first_start = mask ? c0 + __ffsll((long long)mask) - 1 : n;
    int sinc = first_start;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_down_sync(0xffffffffu, sinc, d); if (lane + d < 32) sinc = min(sinc, y); }
    int sex = __shfl_down_sync(0xffffffffu, sinc, 1);
    if (lane == 31) sex = n;
    if (lane == 0) s.scan_i[warp] = sinc;
    __syncthreads();
    for (int k = warp + 1; k < kPngThreads / 32; ++k) sex = min(sex, s.scan_i[k]);
    cout = sex;
  }
  // Adler sums of the segment: s2 weights byte i by n - i
  {
    const unsigned long long a1 = png_cta_sum(s1, s.red);
    const unsigned long long a2 = png_cta_sum((unsigned long long)s2 + (unsigned long long)(n - c0 - cnt) * s1 * (cnt > 0), s.red);
    if (t == 0) { rec[seg].s1 = (unsigned)(a1 % 65521u); rec[seg].s2 = (unsigned)(a2 % 65521u); }
  }

  // histogram of the tokens, end-of-block included
  if (cnt > 0) { PngHistTok h{&s}; png_walk(w, mask, c0, cnt, cin, cout, h); }
  if (t == 0) atomicAdd(&s.hist[256], 1u);
  __syncthreads();
  png_package_merge(s, s.hist, 286, 15, s.ll_len);
  if (t == 0) s.hlit = 257;
  __syncthreads();
  if (t < 286 && s.ll_len[t]) atomicMax(&s.hlit, t + 1);
  png_canonical(s, s.ll_len, 286, s.ll_rev);  // begins and ends with a barrier

  // the code-length sequence (HLIT lit/len lengths, then the distance lengths 1, 1), run-length coded
  if (t == 0) {
    const int hlit = s.hlit, total = hlit + 2;
    for (int k = 0; k < 20; ++k) s.cl_hist[k] = 0u;
    int ncl = 0, i = 0;
    while (i < total) {
      const int v = i < hlit ? s.ll_len[i] : 1;
      int run = 1;
      while (i + run < total && (i + run < hlit ? s.ll_len[i + run] : 1) == v) ++run;
      i += run;
      if (v == 0) {
        while (run >= 11) { const int k = run < 138 ? run : 138; s.cl_sym[ncl] = 18; s.cl_xv[ncl++] = (uint8_t)(k - 11); run -= k; }
        if (run >= 3) { s.cl_sym[ncl] = 17; s.cl_xv[ncl++] = (uint8_t)(run - 3); run = 0; }
        for (; run > 0; --run) { s.cl_sym[ncl] = 0; s.cl_xv[ncl++] = 0; }
      } else {
        s.cl_sym[ncl] = (uint8_t)v; s.cl_xv[ncl++] = 0;
        --run;
        while (run >= 3) { const int k = run < 6 ? run : 6; s.cl_sym[ncl] = 16; s.cl_xv[ncl++] = (uint8_t)(k - 3); run -= k; }
        for (; run > 0; --run) { s.cl_sym[ncl] = (uint8_t)v; s.cl_xv[ncl++] = 0; }
      }
    }
    int used = 0;
    for (int k = 0; k < ncl; ++k) s.cl_hist[s.cl_sym[k]]++;
    for (int k = 0; k < 19; ++k) used += s.cl_hist[k] != 0u;
    s.ncl = ncl;
    s.n_cl_used = used;
  }
  __syncthreads();
  if (s.n_cl_used >= 2) {
    png_package_merge(s, s.cl_hist, 19, 7, s.cl_len);
  } else {
    // One used symbol: a second one of length 1 completes the code.  Defensive: the sequence holds the distance
    // lengths 1, 1 and at least 257 lit/len lengths, of which at least two are non-zero (end-of-block and a literal)
    // and, with HLIT >= 257, either some are zero or all are >= 8, so at least two symbols are always used.  The
    // model's rule for this case is checked on its own (test_png_model.py).
    if (t < 19) s.cl_len[t] = 0;
    __syncthreads();
    if (t == 0) {
      int u = 0;
      while (s.cl_hist[u] == 0u) ++u;
      s.cl_len[u] = 1;
      s.cl_len[u == 0 ? 1 : 0] = 1;
    }
    __syncthreads();
  }
  png_canonical(s, s.cl_len, 19, s.cl_rev);
  if (t == 0) {
    int hclen = 19;
    while (hclen > 4 && s.cl_len[png_cl_order(hclen - 1)] == 0) --hclen;
    int bits = 3 + 5 + 5 + 4 + 3 * hclen;
    for (int k = 0; k < s.ncl; ++k) {
      const int sym = s.cl_sym[k];
      bits += s.cl_len[sym] + (sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0);
    }
    s.hclen = hclen;
    s.header_bits = bits;
  }
  __syncthreads();

  // bit offsets: header (thread 0), tokens, end-of-block (last thread)
  unsigned mybits;
  {
    PngCountTok ct{&s, 0u};
    if (cnt > 0) png_walk(w, mask, c0, cnt, cin, cout, ct);
    mybits = ct.bits + (t == 0 ? (unsigned)s.header_bits : 0u) + (t == kPngThreads - 1 ? (unsigned)s.ll_len[256] : 0u);
  }
  unsigned off;
  {
    unsigned inc = mybits;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
    if (lane == 31) s.scan_u[warp] = inc;
    __syncthreads();
    unsigned before = 0, total = 0;
    for (int k = 0; k < kPngThreads / 32; ++k) { const unsigned v = s.scan_u[k]; if (k < warp) before += v; total += v; }
    off = before + inc - mybits;
    if (t == 0) {
      const unsigned dyn = last ? (total + 7) / 8 : (total + 3 + 7) / 8 + 4;
      const unsigned stored = (unsigned)n + 5u * (((unsigned)n + 65534u) / 65535u);
      s.total_bits = total;
      s.dyn_bytes = dyn;
      s.stored = dyn >= stored;
      rec[seg].bytes = dyn >= stored ? stored : dyn;
      rec[seg].stored = dyn >= stored;
    }
    __syncthreads();
  }
  if (s.stored) return;  // the place kernel copies the segment from F

  {
    PngBitOut o;
    o.init(s.out, off);
    if (t == 0) {
      o.put(last ? 1u : 0u, 1);
      o.put(2u, 2);
      o.put((uint32_t)(s.hlit - 257), 5);
      o.put(1u, 5);
      o.put((uint32_t)(s.hclen - 4), 4);
      for (int k = 0; k < s.hclen; ++k) o.put(s.cl_len[png_cl_order(k)], 3);
      for (int k = 0; k < s.ncl; ++k) {
        const int sym = s.cl_sym[k], l = s.cl_len[sym];
        const int xb = sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0;
        o.put(s.cl_rev[sym] | ((uint32_t)s.cl_xv[k] << l), l + xb);
      }
    }
    PngEmitTok et{&s, &o};
    if (cnt > 0) png_walk(w, mask, c0, cnt, cin, cout, et);
    if (t == kPngThreads - 1) o.put(s.ll_rev[256], s.ll_len[256]);
    o.finish();
  }
  __syncthreads();
  const unsigned bytes = s.dyn_bytes;
  if (!last && t == 0) {  // sync flush: 000, pad, 00 00 FF FF -- only the FF bytes are not zero
    reinterpret_cast<unsigned char*>(s.out)[bytes - 2] = 0xffu;
    reinterpret_cast<unsigned char*>(s.out)[bytes - 1] = 0xffu;
  }
  __syncthreads();
  uint4* dst = reinterpret_cast<uint4*>(staging + seg * (size_t)kPngSlot);
  const uint4* src = reinterpret_cast<const uint4*>(s.out);
  for (unsigned i = t; 16 * i < bytes; i += kPngThreads) dst[i] = src[i];
}

// ---- CRC-32 arithmetic (zlib's multmodp / x2nmodp, reflected bit order)
__device__ __forceinline__ uint32_t png_multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = b & 1 ? (b >> 1) ^ kCrcPoly : b >> 1;
  }
  return p;
}
// x^(8 n) mod P, xpow8[k] = x^(8 * 2^k)
__device__ __forceinline__ uint32_t png_x8n(unsigned long long n, const uint32_t* xpow8) {
  uint32_t p = 1u << 31;
  for (int k = 0; n; ++k, n >>= 1)
    if (n & 1) p = png_multmodp(xpow8[k], p);
  return p;
}
__device__ uint32_t png_crc_bitwise(uint32_t crc, const unsigned char* p, int n) {
  for (int i = 0; i < n; ++i) {
    crc ^= p[i];
    for (int k = 0; k < 8; ++k) crc = crc & 1 ? (crc >> 1) ^ kCrcPoly : crc >> 1;
  }
  return crc;
}

// x^(8 * 2^k) modulo the CRC polynomial, k = 0..16: the shifts of the place kernel's CRCs (all < 2^17 bytes),
// computed on the host once and passed as a kernel parameter
struct PngCrcShifts { uint32_t x8[17]; };
inline uint32_t png_multmodp_host(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = b & 1 ? (b >> 1) ^ kCrcPoly : b >> 1;
  }
  return p;
}
inline PngCrcShifts png_crc_shifts() {
  PngCrcShifts r;
  uint32_t x = 1u << 30;  // x^1
  for (int i = 0; i < 20; ++i) {
    if (i >= 3) r.x8[i - 3] = x;
    x = png_multmodp_host(x, x);
  }
  return r;
}

struct PngPlaceSmem {
  unsigned char data[kPngSlot + 4 + 128];  // "IDAT" + the chunk data, at the CRC slices' alignment
  uint32_t tab[4][256];                    // slicing-by-4
  unsigned long long red[32];
  uint32_t xr[32];
};

__device__ __forceinline__ void png_be32(unsigned char* p, uint32_t v) {
  p[0] = (unsigned char)(v >> 24); p[1] = (unsigned char)(v >> 16); p[2] = (unsigned char)(v >> 8); p[3] = (unsigned char)v;
}

// CTA b < nseg: segment b's IDAT chunk.  CTA nseg: everything else and the total length (state[0]).
__global__ void __launch_bounds__(kPngThreads, 1) png_place_kernel(const unsigned char* __restrict__ F, size_t N,
                                                                   const unsigned char* __restrict__ staging,
                                                                   const PngSegRec* __restrict__ rec, unsigned nseg,
                                                                   unsigned width, unsigned height,
                                                                   unsigned char* __restrict__ out,
                                                                   unsigned long long* __restrict__ state, int count_only,
                                                                   PngCrcShifts shifts) {
  extern __shared__ __align__(16) unsigned char png_place_smem[];
  PngPlaceSmem& s = *reinterpret_cast<PngPlaceSmem*>(png_place_smem);
  const int t = threadIdx.x;
  const unsigned b = blockIdx.x;
  if (b < nseg && count_only) return;
  {  // CRC tables: tab[k][v] = the register after byte v and k zero bytes
    const int k = t >> 8;
    uint32_t c = (uint32_t)(t & 255);
    for (int i = 0; i < 8 * (k + 1); ++i) c = c & 1 ? (c >> 1) ^ kCrcPoly : c >> 1;
    s.tab[k][t & 255] = c;
  }
  if (b == nseg) {  // the total, the Adler-32 of F, and the chunks around the segments
    unsigned long long body = 0, A = 0, B = 0;
    const unsigned long long md = 65521ull;
    for (unsigned j = t; j < nseg; j += kPngThreads) {
      const size_t pj = (size_t)j * kPngSeg;
      const size_t nj = N - pj < (size_t)kPngSeg ? N - pj : (size_t)kPngSeg;
      body += 12ull + rec[j].bytes;
      A += rec[j].s1;
      B = (B + rec[j].s2 + ((N - pj - nj) % md) * rec[j].s1) % md;
    }
    body = png_cta_sum(body, s.red);
    A = png_cta_sum(A, s.red);
    B = png_cta_sum(B, s.red);
    const unsigned long long total = kPngHead + body + kPngTail;
    if (t != 0) return;
    state[0] = total;
    if (count_only) return;
    A = (1 + A) % md;
    B = (N % md + B) % md;
    unsigned char h[64];
    const unsigned char sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    for (int i = 0; i < 8; ++i) h[i] = sig[i];
    png_be32(h + 8, 13); h[12] = 'I'; h[13] = 'H'; h[14] = 'D'; h[15] = 'R';
    png_be32(h + 16, width); png_be32(h + 20, height);
    h[24] = 8; h[25] = 2; h[26] = 0; h[27] = 0; h[28] = 0;
    png_be32(h + 29, png_crc_bitwise(0xffffffffu, h + 12, 17) ^ 0xffffffffu);
    png_be32(h + 33, 2); h[37] = 'I'; h[38] = 'D'; h[39] = 'A'; h[40] = 'T'; h[41] = 0x78; h[42] = 0x01;
    png_be32(h + 43, png_crc_bitwise(0xffffffffu, h + 37, 6) ^ 0xffffffffu);
    for (int i = 0; i < kPngHead; ++i) out[i] = h[i];
    unsigned char* e = out + kPngHead + body;
    png_be32(h, 4); h[4] = 'I'; h[5] = 'D'; h[6] = 'A'; h[7] = 'T';
    png_be32(h + 8, (uint32_t)((B << 16) | A));
    png_be32(h + 12, png_crc_bitwise(0xffffffffu, h + 4, 8) ^ 0xffffffffu);
    png_be32(h + 16, 0); h[20] = 'I'; h[21] = 'E'; h[22] = 'N'; h[23] = 'D';
    png_be32(h + 24, png_crc_bitwise(0xffffffffu, h + 20, 4) ^ 0xffffffffu);
    for (int i = 0; i < kPngTail; ++i) e[i] = h[i];
    return;
  }

  // segment b: where its chunk starts
  unsigned long long before = 0;
  for (unsigned j = t; j < b; j += kPngThreads) before += 12ull + rec[j].bytes;
  const unsigned long long off = kPngHead + png_cta_sum(before, s.red);
  const PngSegRec r = rec[b];
  const size_t a0 = (size_t)b * kPngSeg;
  const int n = (int)(N - a0 < (size_t)kPngSeg ? N - a0 : (size_t)kPngSeg);
  const bool last = b + 1 == nseg;
  // D = "IDAT" + data, m bytes, placed so that the CRC's zero-padded stream of 1024 slices of 128 bytes ends with it
  const int m = 4 + (int)r.bytes;
  const int pad = kPngCrcSpan - m, t0 = pad / 128, lead = pad - 128 * t0;
  unsigned char* o = out + off;
  if (t < lead) s.data[t] = 0;
  for (int j = t; j < m; j += kPngThreads) {
    unsigned char v;
    if (j < 4) {
      v = (unsigned char)(0x54414449u >> (8 * j));  // "IDAT", little-endian
    } else if (!r.stored) {
      v = staging[(size_t)b * kPngSlot + (j - 4)];
    } else {  // stored blocks of <= 65 535 bytes
      const int d = j - 4, blk = d / 65540, x = d - 65540 * blk;
      const int mb = n - 65535 * blk < 65535 ? n - 65535 * blk : 65535;
      if (x == 0) v = (unsigned char)(last && 65535 * blk + mb == n ? 1 : 0);
      else if (x < 5) v = (unsigned char)(((x < 3 ? mb : ~mb) >> (8 * ((x - 1) & 1))) & 0xff);
      else v = F[a0 + 65535 * (size_t)blk + (x - 5)];
    }
    s.data[lead + j] = v;
    o[4 + j] = v;
  }
  if (t == 0) png_be32(o, r.bytes);
  __syncthreads();
  uint32_t crc = 0;
  if (t >= t0) {
    const uint32_t* p = reinterpret_cast<const uint32_t*>(s.data + 128 * (t - t0));
#pragma unroll 4
    for (int k = 0; k < 32; ++k) {
      crc ^= p[k];
      crc = s.tab[3][crc & 0xff] ^ s.tab[2][(crc >> 8) & 0xff] ^ s.tab[1][(crc >> 16) & 0xff] ^ s.tab[0][crc >> 24];
    }
    if (crc) crc = png_multmodp(png_x8n(128ull * (unsigned)(kPngThreads - 1 - t), shifts.x8), crc);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) crc ^= __shfl_xor_sync(0xffffffffu, crc, d);
  if ((t & 31) == 0) s.xr[t >> 5] = crc;
  __syncthreads();
  if (t == 0) {
    uint32_t c = 0;
    for (int k = 0; k < kPngThreads / 32; ++k) c ^= s.xr[k];
    c ^= png_multmodp(png_x8n((unsigned long long)m, shifts.x8), 0xffffffffu) ^ 0xffffffffu;
    png_be32(o + 4 + m, c);
  }
}

// ---- APNG (DESIGN.md section 4.14): the frames of a group in shared launches -- png_filter_frames_kernel,
// png_deflate_frames_kernel, png_place_frames_kernel -- whatever the group's frame count.  Frame f of the group has its
// filtered stream at F + f * nseg * kPngSeg, and its segment s is the group's segment b = f * nseg + s: staging slot b,
// record b.  The file is the signature, IHDR, acTL, then per frame an fcTL and the frame's PNG data chunks (IDAT in
// frame 0; fdAT with a sequence number after it), then IEND.

// The filter twin: one CTA per row of every frame of the group (the frames' rows follow each other in rgb8); frame f's
// filtered stream starts at F + f * fstride.  The body is png_filter_kernel's but for where a row comes from and goes.
__global__ void __launch_bounds__(kPngFilterThreads) png_filter_frames_kernel(const unsigned char* __restrict__ rgb8,
                                                                              size_t row_bytes, unsigned height,
                                                                              size_t fstride,
                                                                              unsigned char* __restrict__ F) {
  __shared__ unsigned long long red[kPngFilterThreads / 32][5];
  __shared__ int pick;
  const size_t frame = blockIdx.x / height, y = blockIdx.x - frame * height;
  const unsigned char* row = rgb8 + (size_t)blockIdx.x * row_bytes;
  const unsigned char* prev = y ? row - row_bytes : nullptr;
  unsigned long long cost[5] = {0, 0, 0, 0, 0};
  for (size_t x = threadIdx.x; x < row_bytes; x += kPngFilterThreads) {
    const int v = row[x], a = x >= 3 ? row[x - 3] : 0, b = prev ? prev[x] : 0, c = (prev && x >= 3) ? prev[x - 3] : 0;
#pragma unroll
    for (int f = 0; f < 5; ++f) cost[f] += (unsigned)abs((int)(signed char)png_filtered(f, v, a, b, c));
  }
#pragma unroll
  for (int f = 0; f < 5; ++f) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cost[f] += __shfl_xor_sync(0xffffffffu, cost[f], d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][f] = cost[f];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int best = 0;
    unsigned long long bc = ~0ull;
    for (int f = 0; f < 5; ++f) {
      unsigned long long t = 0;
      for (int w = 0; w < kPngFilterThreads / 32; ++w) t += red[w][f];
      if (t < bc) { bc = t; best = f; }
    }
    pick = best;
  }
  __syncthreads();
  const int f = pick;
  unsigned char* dst = F + frame * fstride + y * (row_bytes + 1);
  if (threadIdx.x == 0) dst[0] = (unsigned char)f;
  for (size_t x = threadIdx.x; x < row_bytes; x += kPngFilterThreads) {
    const int v = row[x], a = x >= 3 ? row[x - 3] : 0, b = prev ? prev[x] : 0, c = (prev && x >= 3) ? prev[x - 3] : 0;
    dst[1 + x] = (unsigned char)png_filtered(f, v, a, b, c);
  }
}

// The deflate twin: one CTA per segment of every frame of the group.  Frame f's filtered stream (N bytes) starts at
// F + f * nseg * kPngSeg, so CTA b reads F + b * kPngSeg and writes staging slot b and record b as png_deflate_kernel
// does; "last" is the last segment of its frame.  The body is png_deflate_kernel's but for that end.
__global__ void __launch_bounds__(kPngThreads, 1) png_deflate_frames_kernel(const unsigned char* __restrict__ F,
                                                                            size_t N, size_t nseg,
                                                                            unsigned char* __restrict__ staging,
                                                                            PngSegRec* __restrict__ rec) {
  extern __shared__ __align__(16) unsigned char png_deflate_frames_smem[];
  PngDeflateSmem& s = *reinterpret_cast<PngDeflateSmem*>(png_deflate_frames_smem);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const size_t seg = blockIdx.x;
  const size_t a0 = seg * (size_t)kPngSeg;
  const size_t Nf = seg / nseg * nseg * (size_t)kPngSeg + N;  // where the segment's frame ends
  const int n = (int)(Nf - a0 < (size_t)kPngSeg ? Nf - a0 : (size_t)kPngSeg);
  const bool last = a0 + (size_t)n == Nf;

  // load the segment; zero the output words and the histogram; the length table
  {
    const uint4* src = reinterpret_cast<const uint4*>(F + a0);
    for (int i = t; i < kPngSeg / 16; i += kPngThreads) {
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (16 * i + 16 <= n) {
        v = __ldg(src + i);
      } else if (16 * i < n) {
        uint32_t b[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int k = 0; k < 16; ++k)
          if (16 * i + k < n) b[k >> 2] |= (uint32_t)F[a0 + 16 * i + k] << (8 * (k & 3));
        v = make_uint4(b[0], b[1], b[2], b[3]);
      }
      s.in[i] = v;
    }
    for (int i = t; i < kPngSlot / 4; i += kPngThreads) s.out[i] = 0u;
    if (t < 288) s.hist[t] = 0u;
    if (t >= 3 && t <= 258) {
      int k = 0;
      while (k < 28 && png_len_base(k + 1) <= t) ++k;
      if (t == 258) k = 28;
      const int xb = (k >= 8 && k < 28) ? (k - 4) >> 2 : 0;
      s.lsym[t] = (uint16_t)(k | (xb << 5) | ((t - png_len_base(k)) << 8));
    }
  }
  __syncthreads();

  // this thread's 64 bytes, its run starts, its Adler sums
  const int c0 = t * kPngChunk;
  const int cnt = n - c0 < 0 ? 0 : (n - c0 > kPngChunk ? kPngChunk : n - c0);
  const uint4* w = s.in + 4 * t;
  unsigned long long mask = 0;
  unsigned s1 = 0, s2 = 0;
  {
    uint32_t prevb = t ? reinterpret_cast<const unsigned char*>(s.in)[c0 - 1] : 0x100u;
    uint4 v;
#pragma unroll
    for (int p = 0; p < kPngChunk; ++p) {
      if ((p & 15) == 0) v = w[p >> 4];
      const uint32_t b = png_byte(v, p);
      if (p < cnt) {
        if (b != prevb) mask |= 1ull << p;
        s1 += b;
        s2 += (unsigned)(cnt - p) * b;
      }
      prevb = b;
    }
  }
  // the start of the run holding c0 (exclusive max scan) and the first start after the chunk (exclusive min scan)
  int cin, cout;
  {
    const int last_start = mask ? c0 + 63 - __clzll((long long)mask) : -1;
    int inc = last_start;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc = max(inc, y); }
    int ex = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) ex = -1;
    if (lane == 31) s.scan_i[warp] = inc;
    __syncthreads();
    for (int k = 0; k < warp; ++k) ex = max(ex, s.scan_i[k]);
    cin = ex;
    __syncthreads();
    const int first_start = mask ? c0 + __ffsll((long long)mask) - 1 : n;
    int sinc = first_start;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_down_sync(0xffffffffu, sinc, d); if (lane + d < 32) sinc = min(sinc, y); }
    int sex = __shfl_down_sync(0xffffffffu, sinc, 1);
    if (lane == 31) sex = n;
    if (lane == 0) s.scan_i[warp] = sinc;
    __syncthreads();
    for (int k = warp + 1; k < kPngThreads / 32; ++k) sex = min(sex, s.scan_i[k]);
    cout = sex;
  }
  // Adler sums of the segment: s2 weights byte i by n - i
  {
    const unsigned long long a1 = png_cta_sum(s1, s.red);
    const unsigned long long a2 = png_cta_sum((unsigned long long)s2 + (unsigned long long)(n - c0 - cnt) * s1 * (cnt > 0), s.red);
    if (t == 0) { rec[seg].s1 = (unsigned)(a1 % 65521u); rec[seg].s2 = (unsigned)(a2 % 65521u); }
  }

  // histogram of the tokens, end-of-block included
  if (cnt > 0) { PngHistTok h{&s}; png_walk(w, mask, c0, cnt, cin, cout, h); }
  if (t == 0) atomicAdd(&s.hist[256], 1u);
  __syncthreads();
  png_package_merge(s, s.hist, 286, 15, s.ll_len);
  if (t == 0) s.hlit = 257;
  __syncthreads();
  if (t < 286 && s.ll_len[t]) atomicMax(&s.hlit, t + 1);
  png_canonical(s, s.ll_len, 286, s.ll_rev);  // begins and ends with a barrier

  // the code-length sequence (HLIT lit/len lengths, then the distance lengths 1, 1), run-length coded
  if (t == 0) {
    const int hlit = s.hlit, total = hlit + 2;
    for (int k = 0; k < 20; ++k) s.cl_hist[k] = 0u;
    int ncl = 0, i = 0;
    while (i < total) {
      const int v = i < hlit ? s.ll_len[i] : 1;
      int run = 1;
      while (i + run < total && (i + run < hlit ? s.ll_len[i + run] : 1) == v) ++run;
      i += run;
      if (v == 0) {
        while (run >= 11) { const int k = run < 138 ? run : 138; s.cl_sym[ncl] = 18; s.cl_xv[ncl++] = (uint8_t)(k - 11); run -= k; }
        if (run >= 3) { s.cl_sym[ncl] = 17; s.cl_xv[ncl++] = (uint8_t)(run - 3); run = 0; }
        for (; run > 0; --run) { s.cl_sym[ncl] = 0; s.cl_xv[ncl++] = 0; }
      } else {
        s.cl_sym[ncl] = (uint8_t)v; s.cl_xv[ncl++] = 0;
        --run;
        while (run >= 3) { const int k = run < 6 ? run : 6; s.cl_sym[ncl] = 16; s.cl_xv[ncl++] = (uint8_t)(k - 3); run -= k; }
        for (; run > 0; --run) { s.cl_sym[ncl] = (uint8_t)v; s.cl_xv[ncl++] = 0; }
      }
    }
    int used = 0;
    for (int k = 0; k < ncl; ++k) s.cl_hist[s.cl_sym[k]]++;
    for (int k = 0; k < 19; ++k) used += s.cl_hist[k] != 0u;
    s.ncl = ncl;
    s.n_cl_used = used;
  }
  __syncthreads();
  if (s.n_cl_used >= 2) {
    png_package_merge(s, s.cl_hist, 19, 7, s.cl_len);
  } else {
    // One used symbol: a second one of length 1 completes the code.  Defensive: the sequence holds the distance
    // lengths 1, 1 and at least 257 lit/len lengths, of which at least two are non-zero (end-of-block and a literal)
    // and, with HLIT >= 257, either some are zero or all are >= 8, so at least two symbols are always used.  The
    // model's rule for this case is checked on its own (test_png_model.py).
    if (t < 19) s.cl_len[t] = 0;
    __syncthreads();
    if (t == 0) {
      int u = 0;
      while (s.cl_hist[u] == 0u) ++u;
      s.cl_len[u] = 1;
      s.cl_len[u == 0 ? 1 : 0] = 1;
    }
    __syncthreads();
  }
  png_canonical(s, s.cl_len, 19, s.cl_rev);
  if (t == 0) {
    int hclen = 19;
    while (hclen > 4 && s.cl_len[png_cl_order(hclen - 1)] == 0) --hclen;
    int bits = 3 + 5 + 5 + 4 + 3 * hclen;
    for (int k = 0; k < s.ncl; ++k) {
      const int sym = s.cl_sym[k];
      bits += s.cl_len[sym] + (sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0);
    }
    s.hclen = hclen;
    s.header_bits = bits;
  }
  __syncthreads();

  // bit offsets: header (thread 0), tokens, end-of-block (last thread)
  unsigned mybits;
  {
    PngCountTok ct{&s, 0u};
    if (cnt > 0) png_walk(w, mask, c0, cnt, cin, cout, ct);
    mybits = ct.bits + (t == 0 ? (unsigned)s.header_bits : 0u) + (t == kPngThreads - 1 ? (unsigned)s.ll_len[256] : 0u);
  }
  unsigned off;
  {
    unsigned inc = mybits;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
    if (lane == 31) s.scan_u[warp] = inc;
    __syncthreads();
    unsigned before = 0, total = 0;
    for (int k = 0; k < kPngThreads / 32; ++k) { const unsigned v = s.scan_u[k]; if (k < warp) before += v; total += v; }
    off = before + inc - mybits;
    if (t == 0) {
      const unsigned dyn = last ? (total + 7) / 8 : (total + 3 + 7) / 8 + 4;
      const unsigned stored = (unsigned)n + 5u * (((unsigned)n + 65534u) / 65535u);
      s.total_bits = total;
      s.dyn_bytes = dyn;
      s.stored = dyn >= stored;
      rec[seg].bytes = dyn >= stored ? stored : dyn;
      rec[seg].stored = dyn >= stored;
    }
    __syncthreads();
  }
  if (s.stored) return;  // the place kernel copies the segment from F

  {
    PngBitOut o;
    o.init(s.out, off);
    if (t == 0) {
      o.put(last ? 1u : 0u, 1);
      o.put(2u, 2);
      o.put((uint32_t)(s.hlit - 257), 5);
      o.put(1u, 5);
      o.put((uint32_t)(s.hclen - 4), 4);
      for (int k = 0; k < s.hclen; ++k) o.put(s.cl_len[png_cl_order(k)], 3);
      for (int k = 0; k < s.ncl; ++k) {
        const int sym = s.cl_sym[k], l = s.cl_len[sym];
        const int xb = sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0;
        o.put(s.cl_rev[sym] | ((uint32_t)s.cl_xv[k] << l), l + xb);
      }
    }
    PngEmitTok et{&s, &o};
    if (cnt > 0) png_walk(w, mask, c0, cnt, cin, cout, et);
    if (t == kPngThreads - 1) o.put(s.ll_rev[256], s.ll_len[256]);
    o.finish();
  }
  __syncthreads();
  const unsigned bytes = s.dyn_bytes;
  if (!last && t == 0) {  // sync flush: 000, pad, 00 00 FF FF -- only the FF bytes are not zero
    reinterpret_cast<unsigned char*>(s.out)[bytes - 2] = 0xffu;
    reinterpret_cast<unsigned char*>(s.out)[bytes - 1] = 0xffu;
  }
  __syncthreads();
  uint4* dst = reinterpret_cast<uint4*>(staging + seg * (size_t)kPngSlot);
  const uint4* src = reinterpret_cast<const uint4*>(s.out);
  for (unsigned i = t; 16 * i < bytes; i += kPngThreads) dst[i] = src[i];
}

constexpr int kApngHead = 8 + 25 + 20;  // signature, IHDR, acTL
constexpr int kApngFctl = 12 + 26;
constexpr uint32_t kTypeIdat = 0x54414449u, kTypeFdat = 0x54416466u;  // "IDAT", "fdAT", little-endian

struct ApngGroup {
  const unsigned char* F;          // the group's filtered streams
  const unsigned char* staging;    // the group's staging slots
  const PngSegRec* rec;            // the group's segment records
  unsigned char* out;              // the file (nullptr when counting)
  unsigned long long* state;       // [parity]: where the group starts; [parity ^ 1]: where the next starts; [2]: total
  unsigned long long N;            // filtered bytes per frame
  unsigned nseg;                   // segments per frame
  unsigned frames, first, total;   // frames in the group, the first one's index, frames in the file
  unsigned width, height, delay_num, delay_den, plays;
  int parity, count_only;
};

// chunk at o whose n data bytes are written at o + 8: its length, its type and its CRC-32 (one thread)
__device__ void apng_close_chunk(unsigned char* o, uint32_t type, int n) {
  png_be32(o, (uint32_t)n);
  for (int k = 0; k < 4; ++k) o[4 + k] = (unsigned char)(type >> (8 * k));
  png_be32(o + 8 + n, png_crc_bitwise(0xffffffffu, o + 4, 4 + n) ^ 0xffffffffu);
}

// The bytes from the group's start to frame fl's record s: the frames before fl (fcTL, zlib-header chunk, Adler-32
// chunk, segment chunks) and frame fl's segment chunks before s.  A segment chunk is 12 bytes + data in frame 0 of the
// file and 16 bytes + data (the sequence number) in the frames after it.
__device__ unsigned long long apng_before(const ApngGroup& a, unsigned fl, unsigned s, unsigned long long* red) {
  const bool first = a.first == 0;
  const unsigned long long nrec = (unsigned long long)fl * a.nseg + s;
  unsigned long long sum = 0;
  for (unsigned long long j = threadIdx.x; j < nrec; j += kPngThreads)
    sum += (first && j < a.nseg ? 12ull : 16ull) + a.rec[j].bytes;
  const unsigned long long fixed = 76ull * fl - (first && fl > 0 ? 8ull : 0ull);  // 68 in frame 0, 76 after it
  return fixed + png_cta_sum(sum, red);
}

// The sequence number of frame f's fcTL; its fdATs follow: zlib header, segments, Adler-32.
__device__ __forceinline__ uint32_t apng_seq(unsigned f, unsigned nseg) { return f ? 1u + (f - 1u) * (nseg + 3u) : 0u; }

// One chunk of a segment at o: length, type, pre_n (0 or 4) bytes of `pre` big-endian (the sequence number of an
// fdAT), the segment's deflate data (its staging slot, or stored blocks of its filtered bytes seg[0 .. n)), CRC-32.
// png_place_kernel's segment chunk, with the sequence number.
__device__ void apng_place_segment(PngPlaceSmem& s, const unsigned char* __restrict__ seg, int n, bool last,
                                   const unsigned char* __restrict__ slot, PngSegRec r, uint32_t type, int pre_n,
                                   uint32_t pre, unsigned char* __restrict__ o, const PngCrcShifts& shifts) {
  const int t = threadIdx.x;
  // D = type + prefix + data, m bytes, placed so that the CRC's zero-padded stream of 1024 slices of 128 bytes ends
  // with it (m <= 4 + 4 + 65 546: D fits s.data after a lead of < 128 bytes)
  const int m = 4 + pre_n + (int)r.bytes;
  const int pad = kPngCrcSpan - m, t0 = pad / 128, lead = pad - 128 * t0;
  if (t < lead) s.data[t] = 0;
  for (int j = t; j < m; j += kPngThreads) {
    unsigned char v;
    if (j < 4) {
      v = (unsigned char)(type >> (8 * j));
    } else if (j < 4 + pre_n) {
      v = (unsigned char)(pre >> (8 * (7 - j)));
    } else if (!r.stored) {
      v = slot[j - 4 - pre_n];
    } else {  // stored blocks of <= 65 535 bytes
      const int d = j - 4 - pre_n, blk = d / 65540, x = d - 65540 * blk;
      const int mb = n - 65535 * blk < 65535 ? n - 65535 * blk : 65535;
      if (x == 0) v = (unsigned char)(last && 65535 * blk + mb == n ? 1 : 0);
      else if (x < 5) v = (unsigned char)(((x < 3 ? mb : ~mb) >> (8 * ((x - 1) & 1))) & 0xff);
      else v = seg[65535 * (size_t)blk + (x - 5)];
    }
    s.data[lead + j] = v;
    o[4 + j] = v;
  }
  if (t == 0) png_be32(o, (uint32_t)(m - 4));
  __syncthreads();
  uint32_t crc = 0;
  if (t >= t0) {
    const uint32_t* p = reinterpret_cast<const uint32_t*>(s.data + 128 * (t - t0));
#pragma unroll 4
    for (int k = 0; k < 32; ++k) {
      crc ^= p[k];
      crc = s.tab[3][crc & 0xff] ^ s.tab[2][(crc >> 8) & 0xff] ^ s.tab[1][(crc >> 16) & 0xff] ^ s.tab[0][crc >> 24];
    }
    if (crc) crc = png_multmodp(png_x8n(128ull * (unsigned)(kPngThreads - 1 - t), shifts.x8), crc);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) crc ^= __shfl_xor_sync(0xffffffffu, crc, d);
  if ((t & 31) == 0) s.xr[t >> 5] = crc;
  __syncthreads();
  if (t == 0) {
    uint32_t c = 0;
    for (int k = 0; k < kPngThreads / 32; ++k) c ^= s.xr[k];
    c ^= png_multmodp(png_x8n((unsigned long long)m, shifts.x8), 0xffffffffu) ^ 0xffffffffu;
    png_be32(o + 4 + m, c);
  }
}

// CTA b < frames * nseg: segment b's chunk.  CTA frames * nseg + f: frame f's fcTL, zlib-header chunk and Adler-32
// chunk (combined from the frame's own records).  The last CTA: where the next group starts (state[parity ^ 1]); the
// signature, IHDR and acTL in the first group; IEND and the total length (state[2]) in the last.
__global__ void __launch_bounds__(kPngThreads, 1) png_place_frames_kernel(ApngGroup a, PngCrcShifts shifts) {
  extern __shared__ __align__(16) unsigned char png_place_frames_smem[];
  PngPlaceSmem& s = *reinterpret_cast<PngPlaceSmem*>(png_place_frames_smem);
  const int t = threadIdx.x;
  const unsigned b = blockIdx.x, nrec = a.frames * a.nseg;
  if (b < nrec + a.frames && a.count_only) return;
  const unsigned long long base = a.first == 0 ? (unsigned long long)kApngHead : a.state[a.parity];
  if (b == nrec + a.frames) {
    const unsigned long long end = base + apng_before(a, a.frames, 0, s.red);
    if (t != 0) return;
    const bool last_group = a.first + a.frames == a.total;
    a.state[a.parity ^ 1] = end;
    if (last_group) a.state[2] = end + 12;
    if (a.count_only) return;
    if (a.first == 0) {
      unsigned char* o = a.out;
      const unsigned char sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
      for (int i = 0; i < 8; ++i) o[i] = sig[i];
      png_be32(o + 16, a.width); png_be32(o + 20, a.height);
      o[24] = 8; o[25] = 2; o[26] = 0; o[27] = 0; o[28] = 0;
      apng_close_chunk(o + 8, 0x52444849u, 13);  // "IHDR"
      png_be32(o + 41, a.total); png_be32(o + 45, a.plays);
      apng_close_chunk(o + 33, 0x4c546361u, 8);  // "acTL"
    }
    if (last_group) apng_close_chunk(a.out + end, 0x444e4549u, 0);  // "IEND"
    return;
  }
  if (b >= nrec) {
    const unsigned fl = b - nrec, f = a.first + fl;
    const unsigned long long off = base + apng_before(a, fl, 0, s.red);
    const unsigned long long adler_off = base + apng_before(a, fl, a.nseg, s.red) + kApngFctl + (f ? 18 : 14);
    unsigned long long A = 0, B = 0;
    const unsigned long long md = 65521ull, N = a.N;
    for (unsigned j = t; j < a.nseg; j += kPngThreads) {
      const PngSegRec r = a.rec[(size_t)fl * a.nseg + j];
      const unsigned long long pj = (unsigned long long)j * kPngSeg;
      const unsigned long long nj = N - pj < (unsigned long long)kPngSeg ? N - pj : (unsigned long long)kPngSeg;
      A += r.s1;
      B = (B + r.s2 + ((N - pj - nj) % md) * r.s1) % md;
    }
    A = png_cta_sum(A, s.red);
    B = png_cta_sum(B, s.red);
    if (t != 0) return;
    A = (1 + A) % md;
    B = (N % md + B) % md;
    const uint32_t seq = apng_seq(f, a.nseg);
    unsigned char* o = a.out + off;
    png_be32(o + 8, seq); png_be32(o + 12, a.width); png_be32(o + 16, a.height);
    png_be32(o + 20, 0); png_be32(o + 24, 0);
    o[28] = (unsigned char)(a.delay_num >> 8); o[29] = (unsigned char)a.delay_num;
    o[30] = (unsigned char)(a.delay_den >> 8); o[31] = (unsigned char)a.delay_den;
    o[32] = 0; o[33] = 0;  // dispose_op NONE, blend_op SOURCE
    apng_close_chunk(o, 0x4c546366u, 26);  // "fcTL"
    o += kApngFctl;
    unsigned char* e = a.out + adler_off;
    if (f == 0) {
      o[8] = 0x78; o[9] = 0x01;
      apng_close_chunk(o, kTypeIdat, 2);
      png_be32(e + 8, (uint32_t)((B << 16) | A));
      apng_close_chunk(e, kTypeIdat, 4);
    } else {
      png_be32(o + 8, seq + 1); o[12] = 0x78; o[13] = 0x01;
      apng_close_chunk(o, kTypeFdat, 6);
      png_be32(e + 8, seq + 2 + a.nseg); png_be32(e + 12, (uint32_t)((B << 16) | A));
      apng_close_chunk(e, kTypeFdat, 8);
    }
    return;
  }
  {  // CRC tables: tab[k][v] = the register after byte v and k zero bytes
    const int k = t >> 8;
    uint32_t c = (uint32_t)(t & 255);
    for (int i = 0; i < 8 * (k + 1); ++i) c = c & 1 ? (c >> 1) ^ kCrcPoly : c >> 1;
    s.tab[k][t & 255] = c;
  }
  const unsigned fl = b / a.nseg, sg = b - fl * a.nseg, f = a.first + fl;
  const unsigned long long off = base + apng_before(a, fl, sg, s.red) + kApngFctl + (f ? 18 : 14);
  const unsigned long long a0 = (unsigned long long)sg * kPngSeg;
  const int n = (int)(a.N - a0 < (unsigned long long)kPngSeg ? a.N - a0 : (unsigned long long)kPngSeg);
  apng_place_segment(s, a.F + (size_t)b * kPngSeg, n, sg + 1 == a.nseg, a.staging + (size_t)b * kPngSlot, a.rec[b],
                     f ? kTypeFdat : kTypeIdat, f ? 4 : 0, apng_seq(f, a.nseg) + 2 + sg, a.out + off, shifts);
}

}  // namespace rtclj
