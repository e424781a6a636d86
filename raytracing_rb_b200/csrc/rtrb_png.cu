// rtrb_png.cu — PNG encoder on the device (see rtrb_png.h for the pipeline): 8-bit RGB, no interlace, per-row
// filters chosen by the minimum sum of absolute differences (libpng's heuristic), zlib stream cut into
// RTRB_PNG_SEGMENT_BYTES segments that are deflated independently, one CTA each.
//
// Deflate (RFC 1951) per segment:
//   - hash chains over the segment and the 32 KiB before it (matches may reach into earlier segments: the decoder has
//     those bytes as history), built in rounds of one position per thread;
//   - greedy parse: each thread parses its own CHUNK of the segment, a match may run past the chunk end.  An
//     inclusive prefix maximum over the threads' parse ends tells each thread where the bytes it has to cover begin;
//     a token that straddles that point keeps its distance and loses its head, which is still a valid match;
//   - the block is whichever is smallest of stored, fixed Huffman and dynamic Huffman (15-bit limited codes, 7-bit
//     code-length code with the 16/17/18 run-length codes), so a segment never exceeds the stored size;
//   - a non-final segment ends with an empty stored block (sync flush) so the next one starts on a byte boundary.
// Every step is deterministic: the same input gives the same file whatever the scheduling.
#include <cuda_runtime.h>
#include <stdint.h>

#include "rtrb_png.h"

namespace {

constexpr int SEG = RTRB_PNG_SEGMENT_BYTES;
constexpr int WIN = 32768;             // deflate window
constexpr int DT = 512;                // threads of the deflate CTA
// Bytes each parsing thread covers.  Every chunk boundary inside a long match costs about one extra token, so chunks
// are longer than a match: on config 2 at 1080p, 64-byte chunks gave 211 800 bytes (zlib level 1: 147 016), 512-byte
// chunks 127 807 bytes in 1.32 ms of deflate kernel (B200).
constexpr int CHUNK = 256;
constexpr int NPARSE = SEG / CHUNK;    // parsing threads
constexpr int HASH_BITS = 12;
constexpr int MAX_CHAIN = 16;          // candidates tried per position
constexpr int REGION = WIN + SEG;      // history + segment bytes held in shared memory
constexpr int BITBUF_WORDS = (SEG + 64) / 4;
static_assert(SEG % CHUNK == 0 && NPARSE <= DT && SEG <= 65535, "a segment must fit one stored block");
static_assert(BITBUF_WORDS * 4 <= REGION * 2, "the bit buffer reuses the hash-chain links");

constexpr size_t DEFLATE_SMEM = (size_t)REGION + 16 + (size_t)REGION * 2 + (sizeof(int) << HASH_BITS);

__device__ __forceinline__ uint32_t brev_n(uint32_t code, int len) { return __brev(code) >> (32 - len); }

// ---- CRC-32 (ISO-HDLC, as PNG uses it) ----------------------------------------------------------------------
constexpr uint32_t CRC_POLY = 0xedb88320u;

__device__ void crc_table_init(uint32_t* table, uint32_t* x2n) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; ++k) c = c & 1u ? (c >> 1) ^ CRC_POLY : c >> 1;
    table[i] = c;
  }
  if (threadIdx.x == 0) {  // x^(2^k) modulo the polynomial (reflected), for combining CRCs
    uint32_t p = 1u << 30;
    x2n[0] = p;
    for (int n = 1; n < 32; ++n) {
      uint32_t a = p, b = p, m = 1u << 31, r = 0;
      for (;;) {
        if (a & m) { r ^= b; if ((a & (m - 1)) == 0) break; }
        m >>= 1;
        b = b & 1u ? (b >> 1) ^ CRC_POLY : b >> 1;
      }
      x2n[n] = p = r;
    }
  }
}

__device__ uint32_t multmodp(uint32_t a, uint32_t b) {  // a * b modulo the polynomial; a != 0
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
    m >>= 1;
    b = b & 1u ? (b >> 1) ^ CRC_POLY : b >> 1;
  }
  return p;
}

// CRC-32 of A || B from crc(A), crc(B) and |B| (zlib's crc32_combine)
__device__ uint32_t crc_combine(uint32_t crc1, uint32_t crc2, uint32_t len2, const uint32_t* x2n) {
  uint32_t p = 1u << 31;
  for (uint32_t n = len2, k = 3; n; n >>= 1, ++k)
    if (n & 1u) p = multmodp(x2n[k & 31], p);
  return multmodp(p, crc1) ^ crc2;
}

__device__ uint32_t crc_bytes(const uint8_t* p, size_t n, uint32_t crc, const uint32_t* table) {
  crc = ~crc;
  for (size_t i = 0; i < n; ++i) crc = table[(crc ^ p[i]) & 0xffu] ^ (crc >> 8);
  return ~crc;
}

// CRC-32 of "IDAT" || data[0, n), all threads of the block; red needs 2 * (blockDim.x / 32) words
__device__ uint32_t block_chunk_crc(const uint8_t* data, uint32_t n, const uint32_t* table, const uint32_t* x2n,
                                    uint32_t* red) {
  const uint32_t per = (n + blockDim.x - 1) / blockDim.x;
  const uint32_t b = min(n, threadIdx.x * per), e = min(n, b + per);
  uint32_t crc = crc_bytes(data + b, e - b, 0, table), len = e - b;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int off = 1; off < 32; off <<= 1) {
    const uint32_t oc = __shfl_down_sync(0xffffffffu, crc, off), ol = __shfl_down_sync(0xffffffffu, len, off);
    if ((lane & (2 * off - 1)) == 0 && lane + off < 32) { crc = crc_combine(crc, oc, ol, x2n); len += ol; }
  }
  if (lane == 0) { red[2 * warp] = crc; red[2 * warp + 1] = len; }
  __syncthreads();
  uint32_t out = 0;
  if (threadIdx.x == 0) {
    const uint8_t idat[4] = {'I', 'D', 'A', 'T'};
    out = crc_bytes(idat, 4, 0, table);
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) out = crc_combine(out, red[2 * w], red[2 * w + 1], x2n);
  }
  return out;  // valid in thread 0
}

// ---- block-wide scans ------------------------------------------------------------------------------------------
template <bool MAX>
__device__ uint32_t block_scan(uint32_t v, uint32_t* warp_tot, uint32_t& total) {  // inclusive
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int off = 1; off < 32; off <<= 1) {
    const uint32_t o = __shfl_up_sync(0xffffffffu, v, off);
    if (lane >= off) v = MAX ? max(v, o) : v + o;
  }
  if (lane == 31) warp_tot[warp] = v;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < nw ? warp_tot[lane] : 0;
    for (int off = 1; off < 32; off <<= 1) {
      const uint32_t o = __shfl_up_sync(0xffffffffu, w, off);
      if (lane >= off) w = MAX ? max(w, o) : w + o;
    }
    if (lane < nw) warp_tot[lane] = w;
  }
  __syncthreads();
  if (warp > 0) v = MAX ? max(v, warp_tot[warp - 1]) : v + warp_tot[warp - 1];
  total = warp_tot[nw - 1];
  __syncthreads();
  return v;
}

// ---- filters -----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t sabs(uint32_t v) { v &= 0xffu; return v < 128u ? v : 256u - v; }
__device__ __forceinline__ uint32_t paeth(int a, int b, int c) {
  const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
  return (uint32_t)((pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c));
}

__global__ void __launch_bounds__(256) png_filter_kernel(const uint8_t* __restrict__ src, int W, int fmt,
                                                         uint8_t* __restrict__ out) {
  const int y = blockIdx.x, n = 3 * W;
  const int bpp = fmt == RTRB_FMT_RGBA8 ? 4 : 3;
  const size_t stride = fmt == RTRB_FMT_PNG_RGB8 ? (size_t)n + 1 : (size_t)W * bpp;
  const uint8_t* row = src + y * stride + (fmt == RTRB_FMT_PNG_RGB8 ? 1 : 0);
  const uint8_t* up = y > 0 ? row - stride : row;
  auto at = [&](const uint8_t* r, int i) -> int { return r[(i / 3) * bpp + i % 3]; };
  uint32_t s[5] = {0, 0, 0, 0, 0};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int x = at(row, i), a = i >= 3 ? at(row, i - 3) : 0, b = y > 0 ? at(up, i) : 0;
    const int c = (i >= 3 && y > 0) ? at(up, i - 3) : 0;
    s[0] += sabs(x); s[1] += sabs(x - a); s[2] += sabs(x - b); s[3] += sabs(x - ((a + b) >> 1));
    s[4] += sabs(x - paeth(a, b, c));
  }
  __shared__ uint32_t red[8][5];
  __shared__ int choice;
  for (int k = 0; k < 5; ++k)
    for (int off = 16; off; off >>= 1) s[k] += __shfl_down_sync(0xffffffffu, s[k], off);
  if ((threadIdx.x & 31) == 0)
    for (int k = 0; k < 5; ++k) red[threadIdx.x >> 5][k] = s[k];
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t best = 0xffffffffu;
    int f = 0;
    for (int k = 0; k < 5; ++k) {
      uint32_t t = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w][k];
      if (t < best) { best = t; f = k; }  // strict: ties keep the lower filter type
    }
    choice = f;
  }
  __syncthreads();
  const int f = choice;
  uint8_t* o = out + (size_t)y * (n + 1);
  if (threadIdx.x == 0) o[0] = (uint8_t)f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int x = at(row, i), a = i >= 3 ? at(row, i - 3) : 0, b = y > 0 ? at(up, i) : 0;
    const int c = (i >= 3 && y > 0) ? at(up, i - 3) : 0;
    const int pred = f == 0 ? 0 : f == 1 ? a : f == 2 ? b : f == 3 ? ((a + b) >> 1) : (int)paeth(a, b, c);
    o[1 + i] = (uint8_t)(x - pred);
  }
}

// ---- deflate symbols -------------------------------------------------------------------------------------------
// length 3..258 -> symbol 257..285, extra bits, extra value
__device__ __forceinline__ void len_sym(int len, int& sym, int& nb, int& ev) {
  const int l = len - 3;
  if (l == 255) { sym = 285; nb = 0; ev = 0; return; }
  if (l < 8) { sym = 257 + l; nb = 0; ev = 0; return; }
  const int b = 31 - __clz(l);
  sym = 257 + 4 * (b - 1) + ((l >> (b - 2)) & 3);
  nb = b - 2;
  ev = l & ((1 << nb) - 1);
}
// distance 1..32768 -> symbol 0..29, extra bits, extra value
__device__ __forceinline__ void dist_sym(int dist, int& sym, int& nb, int& ev) {
  const int x = dist - 1;
  if (x < 4) { sym = x; nb = 0; ev = 0; return; }
  const int b = 31 - __clz(x);
  sym = 2 * b + ((x >> (b - 1)) & 1);
  nb = b - 1;
  ev = x & ((1 << nb) - 1);
}

// Huffman code lengths limited to `limit` bits (Moffat & Katajainen in-place construction, then the Kraft-sum repair
// miniz uses).  key/sym: the m used symbols sorted by ascending (frequency, symbol); key is overwritten.
__device__ void huff_lengths(uint32_t* key, const uint16_t* sym, int m, int limit, uint8_t* lens, int n) {
  for (int i = 0; i < n; ++i) lens[i] = 0;
  if (m == 0) return;
  if (m == 1) { lens[sym[0]] = 1; return; }
  uint32_t* A = key;
  A[0] += A[1];
  int root = 0, leaf = 2;
  for (int next = 1; next < m - 1; ++next) {
    if (leaf >= m || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = next; }
    else A[next] = A[leaf++];
    if (leaf >= m || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = next; }
    else A[next] += A[leaf++];
  }
  A[m - 2] = 0;
  for (int next = m - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
  int avbl = 1, used = 0, dpth = 0;
  root = m - 2;
  int next = m - 1;
  while (avbl > 0) {
    while (root >= 0 && (int)A[root] == dpth) { ++used; --root; }
    while (avbl > used) { A[next--] = dpth; --avbl; }
    avbl = 2 * used; ++dpth; used = 0;
  }
  int num[33];
  for (int i = 0; i <= 32; ++i) num[i] = 0;
  for (int i = 0; i < m; ++i) num[min(A[i], 32u)]++;
  for (int i = limit + 1; i <= 32; ++i) { num[limit] += num[i]; num[i] = 0; }
  uint32_t total = 0;
  for (int i = limit; i > 0; --i) total += (uint32_t)num[i] << (limit - i);
  while (total != (1u << limit)) {
    num[limit]--;
    for (int i = limit - 1; i > 0; --i)
      if (num[i]) { num[i]--; num[i + 1] += 2; break; }
    total--;
  }
  int j = m;
  for (int i = 1; i <= limit; ++i)
    for (int l = num[i]; l > 0; --l) lens[sym[--j]] = (uint8_t)i;
}

// the used symbols of freq[0, n) in ascending (frequency, symbol) order; one thread per symbol (t < n)
__device__ void rank_symbols(const uint32_t* freq, int n, int t, uint32_t* key, uint16_t* sym) {
  if (t >= n || freq[t] == 0) return;
  const uint32_t f = freq[t];
  int r = 0;
  for (int j = 0; j < n; ++j) {
    const uint32_t g = freq[j];
    r += (g != 0u) & ((g < f) | ((g == f) & (j < t)));
  }
  key[r] = f;
  sym[r] = (uint16_t)t;
}

__device__ int count_used(const uint32_t* freq, int n) {
  int m = 0;
  for (int i = 0; i < n; ++i) m += freq[i] != 0u;
  return m;
}

__device__ void canonical_codes(const uint8_t* lens, int n, uint16_t* codes) {  // bit-reversed for LSB-first output
  int count[16] = {0}, next[16];
  for (int i = 0; i < n; ++i) count[lens[i]]++;
  count[0] = 0;
  int code = 0;
  for (int b = 1; b < 16; ++b) { code = (code + count[b - 1]) << 1; next[b] = code; }
  for (int i = 0; i < n; ++i)
    codes[i] = lens[i] ? (uint16_t)brev_n((uint32_t)next[lens[i]]++, lens[i]) : 0;
}

__device__ __forceinline__ void put_bits(uint32_t* buf, uint32_t pos, uint32_t v, int nb) {  // nb <= 32
  if (nb == 0) return;
  const uint32_t w = pos >> 5, o = pos & 31u;
  atomicOr(&buf[w], v << o);
  if (o + nb > 32) atomicOr(&buf[w + 1], v >> (32 - o));
}

__device__ __forceinline__ uint32_t load32(const uint8_t* d, int i) {  // unaligned little-endian load from smem
  const uint32_t* w = reinterpret_cast<const uint32_t*>(d);
  return __funnelshift_r(w[i >> 2], w[(i >> 2) + 1], (i & 3) * 8);
}

__device__ __forceinline__ int match_len(const uint8_t* d, int a, int b, int maxlen) {
  int l = 0;
  while (l < maxlen) {
    const uint32_t x = load32(d, a + l) ^ load32(d, b + l);
    if (x) return min(maxlen, l + ((__ffs(x) - 1) >> 3));
    l += 4;
  }
  return maxlen;
}

__device__ __forceinline__ uint32_t hash3(const uint8_t* d, int i) {
  const uint32_t v = (uint32_t)d[i] | ((uint32_t)d[i + 1] << 8) | ((uint32_t)d[i + 2] << 16);
  return (v * 2654435761u) >> (32 - HASH_BITS);
}

// Walks thread t's tokens and hands on exactly the ones that cover [from, its parse end): tokens wholly before
// `from` are dropped, one straddling it keeps its distance and tail (or becomes literals when under 3 bytes).
template <typename F>
__device__ __forceinline__ void visit_tokens(const uint32_t* tok, int ntok, int pos, int from, const uint8_t* d,
                                             int r0, F&& f) {
  for (int k = 0; k < ntok; ++k) {
    const uint32_t t = tok[k];
    const int len = (int)(t >> 16), L = len ? len : 1;
    if (pos + L > from) {
      if (pos >= from) {
        if (len) f(len, (int)(t & 0xffffu)); else f(0, (int)(t & 0xffu));
      } else {
        const int rem = pos + L - from;
        if (rem >= 3) f(rem, (int)(t & 0xffffu));
        else for (int i = 0; i < rem; ++i) f(0, (int)d[from + i - r0]);
      }
    }
    pos += L;
  }
}

struct DeflateShared {
  uint32_t freq_ll[288], freq_d[32], freq_c[19];
  uint32_t key[288];
  uint16_t sym[288];
  uint32_t key_d[32];
  uint16_t sym_d[32];
  uint8_t len_ll[288], len_d[32], len_c[19];
  uint16_t code_ll[288], code_d[32], code_c[19];
  uint16_t rle[320];
  uint32_t crc_table[256], x2n[32];
  uint32_t scan[32], red[64], ends[DT];
  unsigned long long adler_a, adler_b;
  uint32_t extra_bits, placeholder_dist;
  int n_rle, hlit, hdist, hclen, btype;
  uint32_t hdr_bits, out_bytes;
};

__global__ void __launch_bounds__(DT, 1) png_deflate_kernel(const uint8_t* __restrict__ in, unsigned long long n_in, int row_bytes,
                                                            uint32_t* __restrict__ tokens, uint8_t* __restrict__ seg_out,
                                                            uint32_t* __restrict__ seg_meta) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint8_t* data = smem;                                                   // [REGION + 16]
  uint16_t* prev = reinterpret_cast<uint16_t*>(smem + REGION + 16);      // [REGION] chain links (distance, 0 = end)
  int* head = reinterpret_cast<int*>(smem + REGION + 16 + REGION * 2);   // [1 << HASH_BITS]
  uint32_t* bitbuf = reinterpret_cast<uint32_t*>(prev);                  // after the parse
  __shared__ DeflateShared sh;

  const int seg = blockIdx.x, tid = threadIdx.x;
  const unsigned long long s0 = (unsigned long long)seg * SEG;
  const int seg_len = (int)min((unsigned long long)SEG, n_in - s0);
  const bool final_seg = s0 + seg_len == n_in;
  // besides the hash chain, the parse tries the byte 3 back (the pixel to the left), 1 back and the row above
  const int fixed_dist[3] = {row_bytes, 3, 1};
  const unsigned long long r0 = s0 > (unsigned long long)WIN ? s0 - WIN : 0ull;
  const int hist = (int)(s0 - r0), rlen = hist + seg_len;  // region [r0, r0 + rlen), segment at [hist, rlen)

  // ---- load the region, clear the tables ----
  for (int i = tid; i < rlen; i += DT) data[i] = in[r0 + i];
  for (int i = rlen + tid; i < rlen + 16; i += DT) data[i] = 0;
  for (int i = tid; i < (1 << HASH_BITS); i += DT) head[i] = -1;
  for (int i = tid; i < 288; i += DT) sh.freq_ll[i] = 0;
  if (tid < 32) sh.freq_d[tid] = 0;
  if (tid < 19) sh.freq_c[tid] = 0;
  if (tid == 0) { sh.adler_a = 0; sh.adler_b = 0; sh.extra_bits = 0; }
  crc_table_init(sh.crc_table, sh.x2n);
  __syncthreads();

  // ---- hash chains, one round of DT positions at a time: a position links to the nearest earlier lane of its warp
  // with the same hash, else to the last such position of the previous rounds ----
  const int lane = tid & 31;
  for (int base = 0; base < rlen; base += DT) {
    const int i = base + tid;
    const bool ok = i + 2 < rlen;
    const uint32_t h = ok ? hash3(data, i) : (0x80000000u | (uint32_t)lane);
    const uint32_t earlier = __match_any_sync(0xffffffffu, h) & ((1u << lane) - 1u);
    if (i < rlen) {
      uint16_t link = 0;
      if (ok && earlier) {
        link = (uint16_t)(lane - (31 - __clz(earlier)));
      } else if (ok) {
        const int q = head[h];
        if (q >= 0 && i - q <= WIN) link = (uint16_t)(i - q);
      }
      prev[i] = link;
    }
    __syncthreads();
    if (ok) atomicMax(&head[h], i);
    __syncthreads();
  }

  // ---- Adler-32 partial of the segment's input ----
  {
    unsigned long long a = 0, b = 0;
    for (int i = tid; i < seg_len; i += DT) {
      const unsigned v = data[hist + i];
      a += v;
      b += (unsigned long long)(seg_len - i) * v;
    }
    for (int off = 16; off; off >>= 1) {
      a += __shfl_down_sync(0xffffffffu, a, off);
      b += __shfl_down_sync(0xffffffffu, b, off);
    }
    if ((tid & 31) == 0) { atomicAdd(&sh.adler_a, a); atomicAdd(&sh.adler_b, b); }
  }

  // ---- greedy parse of this thread's chunk ----
  uint32_t* tok = tokens + (size_t)seg * SEG + (size_t)tid * CHUNK;
  const int c0 = hist + tid * CHUNK, c1 = tid < NPARSE ? min(rlen, c0 + CHUNK) : c0;
  int p = c0, ntok = 0;
  while (p < c1) {
    const int maxl = min(258, rlen - p);
    int best = 0, bdist = 0;
    if (maxl >= 3) {
      int q = p, steps = MAX_CHAIN;
      uint32_t dd = prev[p];
      while (dd && steps-- > 0) {
        q -= (int)dd;
        const int dist = p - q;
        if (dist > WIN) break;
        const int l = match_len(data, q, p, maxl);
        if (l > best) { best = l; bdist = dist; if (l >= maxl) break; }
        dd = prev[q];
      }
      for (int k = 0; k < 3 && best < maxl; ++k) {
        const int dist = fixed_dist[k];
        if (dist > p || dist > WIN) continue;
        const int l = match_len(data, p - dist, p, maxl);
        if (l > best) { best = l; bdist = dist; }
      }
    }
    // a 3-byte match far back costs more bits than three literals (zlib's TOO_FAR)
    if (best == 3 && bdist > 4096) best = 0;
    if (best >= 3) { tok[ntok++] = ((uint32_t)best << 16) | (uint32_t)bdist; p += best; }
    else { tok[ntok++] = data[p]; p += 1; }
  }
  uint32_t unused;
  sh.ends[tid] = block_scan<true>(tid < NPARSE ? (uint32_t)max(p, c0) : 0u, sh.scan, unused);
  __syncthreads();
  // the bytes this thread covers start where the parses of the threads before it stopped
  const int start = tid == 0 ? hist : (int)sh.ends[tid - 1];

  // ---- symbol statistics ----
  uint32_t extra = 0;
  visit_tokens(tok, ntok, c0, start, data, 0, [&](int len, int v) {
    if (len == 0) { atomicAdd(&sh.freq_ll[v], 1u); return; }
    int s, nb, ev;
    len_sym(len, s, nb, ev);
    atomicAdd(&sh.freq_ll[s], 1u);
    extra += nb;
    dist_sym(v, s, nb, ev);
    atomicAdd(&sh.freq_d[s], 1u);
    extra += nb;
  });
  if (extra) atomicAdd(&sh.extra_bits, extra);
  __syncthreads();
  if (tid == 0) {
    sh.freq_ll[256] = 1;  // end of block
    // a dynamic block describes at least one distance code, even when no match uses it
    sh.placeholder_dist = count_used(sh.freq_d, 30) == 0;
    if (sh.placeholder_dist) sh.freq_d[0] = 1;
  }
  __syncthreads();

  // ---- dynamic Huffman tables ----
  rank_symbols(sh.freq_ll, 286, tid, sh.key, sh.sym);
  if (tid >= 320 && tid < 352) rank_symbols(sh.freq_d, 30, tid - 320, sh.key_d, sh.sym_d);
  __syncthreads();
  if (tid == 0) huff_lengths(sh.key, sh.sym, count_used(sh.freq_ll, 286), 15, sh.len_ll, 288);
  if (tid == 32) huff_lengths(sh.key_d, sh.sym_d, count_used(sh.freq_d, 30), 15, sh.len_d, 32);
  __syncthreads();
  if (tid == 0) {
    int hlit = 286, hdist = 30;
    while (hlit > 257 && sh.len_ll[hlit - 1] == 0) --hlit;
    while (hdist > 1 && sh.len_d[hdist - 1] == 0) --hdist;
    const int total = hlit + hdist;
    auto L = [&](int i) -> int { return i < hlit ? sh.len_ll[i] : sh.len_d[i - hlit]; };
    int nr = 0;
    for (int i = 0; i < total;) {
      const int cur = L(i);
      int run = 1;
      while (i + run < total && L(i + run) == cur) ++run;
      int r = run;
      if (cur == 0) {
        while (r >= 11) { const int k = min(r, 138); sh.rle[nr++] = (uint16_t)(18 | ((k - 11) << 5)); r -= k; }
        if (r >= 3) { sh.rle[nr++] = (uint16_t)(17 | ((r - 3) << 5)); r = 0; }
        while (r-- > 0) sh.rle[nr++] = 0;
      } else {
        sh.rle[nr++] = (uint16_t)cur;
        --r;
        while (r >= 3) { const int k = min(r, 6); sh.rle[nr++] = (uint16_t)(16 | ((k - 3) << 5)); r -= k; }
        while (r-- > 0) sh.rle[nr++] = (uint16_t)cur;
      }
      i += run;
    }
    for (int k = 0; k < nr; ++k) sh.freq_c[sh.rle[k] & 31]++;
    sh.n_rle = nr; sh.hlit = hlit; sh.hdist = hdist;
  }
  __syncthreads();
  rank_symbols(sh.freq_c, 19, tid, sh.key_d, sh.sym_d);
  __syncthreads();
  if (tid == 0) {
    huff_lengths(sh.key_d, sh.sym_d, count_used(sh.freq_c, 19), 7, sh.len_c, 19);
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    int hclen = 19;
    while (hclen > 4 && sh.len_c[order[hclen - 1]] == 0) --hclen;
    sh.hclen = hclen;
    // sizes of the three block types (bits, then bytes including the sync flush)
    unsigned long long dyn = 3 + 14 + 3ull * hclen, fix = 3;
    for (int k = 0; k < sh.n_rle; ++k) {
      const int s = sh.rle[k] & 31;
      dyn += sh.len_c[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
    }
    for (int s = 0; s < 286; ++s) {
      const unsigned long long f = sh.freq_ll[s];
      dyn += f * sh.len_ll[s];
      fix += f * (s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8);
    }
    unsigned long long nd = 0;
    for (int s = 0; s < 30; ++s) { dyn += (unsigned long long)sh.freq_d[s] * sh.len_d[s]; nd += sh.freq_d[s]; }
    fix += 5 * nd;
    if (sh.placeholder_dist) { dyn -= sh.len_d[0]; fix -= 5; }  // described, never emitted
    dyn += sh.extra_bits; fix += sh.extra_bits;
    auto bytes = [&](unsigned long long bits) -> unsigned long long {
      return final_seg ? (bits + 7) / 8 : (bits + 3 + 7) / 8 + 4;
    };
    const unsigned long long stored = (unsigned long long)seg_len + (final_seg ? 5 : 10);
    const unsigned long long bf = bytes(fix), bd = bytes(dyn);
    int bt = 0;
    unsigned long long best = stored;
    if (bf < best) { best = bf; bt = 1; }
    if (bd < best) { best = bd; bt = 2; }
    sh.btype = bt;
    sh.out_bytes = (uint32_t)best;
    if (bt == 1) {
      for (int s = 0; s < 288; ++s) sh.len_ll[s] = (uint8_t)(s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8);
      for (int s = 0; s < 32; ++s) sh.len_d[s] = 5;
    }
    if (bt != 0) {
      canonical_codes(sh.len_ll, 288, sh.code_ll);
      canonical_codes(sh.len_d, 32, sh.code_d);
      canonical_codes(sh.len_c, 19, sh.code_c);
    }
  }
  __syncthreads();
  const int bt = sh.btype;
  const uint32_t out_bytes = sh.out_bytes;
  uint8_t* out = seg_out + (size_t)seg * RTRB_PNG_SEGMENT_WORST(SEG);

  if (bt == 0) {  // stored
    for (int i = tid; i < seg_len; i += DT) out[5 + i] = data[hist + i];
    if (tid == 0) {
      out[0] = final_seg ? 1 : 0;
      out[1] = (uint8_t)seg_len; out[2] = (uint8_t)(seg_len >> 8);
      out[3] = (uint8_t)~seg_len; out[4] = (uint8_t)(~seg_len >> 8);
      if (!final_seg) { uint8_t* f = out + 5 + seg_len; f[0] = 0; f[1] = 0; f[2] = 0; f[3] = 0xff; f[4] = 0xff; }
    }
  } else {
    for (int i = tid; i < BITBUF_WORDS; i += DT) bitbuf[i] = 0;
    // bits of this thread's tokens
    uint32_t nbits = 0;
    visit_tokens(tok, ntok, c0, start, data, 0, [&](int len, int v) {
      if (len == 0) { nbits += sh.len_ll[v]; return; }
      int s, nb, ev;
      len_sym(len, s, nb, ev);
      nbits += sh.len_ll[s] + nb;
      dist_sym(v, s, nb, ev);
      nbits += sh.len_d[s] + nb;
    });
    uint32_t token_bits;
    const uint32_t incl = block_scan<false>(nbits, sh.scan, token_bits);
    __syncthreads();
    if (tid == 0) {  // block header (+ code tables)
      uint32_t pos = 0;
      put_bits(bitbuf, pos, (final_seg ? 1u : 0u) | ((uint32_t)bt << 1), 3); pos += 3;
      if (bt == 2) {
        put_bits(bitbuf, pos, sh.hlit - 257, 5); pos += 5;
        put_bits(bitbuf, pos, sh.hdist - 1, 5); pos += 5;
        put_bits(bitbuf, pos, sh.hclen - 4, 4); pos += 4;
        const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        for (int k = 0; k < sh.hclen; ++k) { put_bits(bitbuf, pos, sh.len_c[order[k]], 3); pos += 3; }
        for (int k = 0; k < sh.n_rle; ++k) {
          const int s = sh.rle[k] & 31, x = sh.rle[k] >> 5;
          put_bits(bitbuf, pos, sh.code_c[s], sh.len_c[s]); pos += sh.len_c[s];
          const int xb = s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0;
          put_bits(bitbuf, pos, (uint32_t)x, xb); pos += xb;
        }
      }
      sh.hdr_bits = pos;
    }
    __syncthreads();
    uint32_t pos = sh.hdr_bits + incl - nbits;
    visit_tokens(tok, ntok, c0, start, data, 0, [&](int len, int v) {
      if (len == 0) { put_bits(bitbuf, pos, sh.code_ll[v], sh.len_ll[v]); pos += sh.len_ll[v]; return; }
      int s, nb, ev;
      len_sym(len, s, nb, ev);
      put_bits(bitbuf, pos, sh.code_ll[s] | ((uint32_t)ev << sh.len_ll[s]), sh.len_ll[s] + nb);
      pos += sh.len_ll[s] + nb;
      dist_sym(v, s, nb, ev);
      put_bits(bitbuf, pos, sh.code_d[s] | ((uint32_t)ev << sh.len_d[s]), sh.len_d[s] + nb);
      pos += sh.len_d[s] + nb;
    });
    if (tid == 0) {
      const uint32_t eob = sh.hdr_bits + token_bits;
      put_bits(bitbuf, eob, sh.code_ll[256], sh.len_ll[256]);
    }
    __syncthreads();
    uint8_t* bytes = reinterpret_cast<uint8_t*>(bitbuf);
    if (tid == 0 && !final_seg) { bytes[out_bytes - 2] = 0xff; bytes[out_bytes - 1] = 0xff; }  // 00 00 ff ff
    __syncthreads();
    for (int i = tid; i < (int)out_bytes; i += DT) out[i] = bytes[i];
  }
  __syncthreads();
  const uint32_t crc = block_chunk_crc(out, out_bytes, sh.crc_table, sh.x2n, sh.red);
  if (tid == 0) {
    const uint32_t a = (uint32_t)((1ull + sh.adler_a) % 65521ull);
    const uint32_t b = (uint32_t)(((unsigned long long)seg_len + sh.adler_b) % 65521ull);
    seg_meta[3 * seg] = out_bytes;
    seg_meta[3 * seg + 1] = crc;
    seg_meta[3 * seg + 2] = (b << 16) | a;
  }
}

__device__ __forceinline__ void put_be32(uint8_t* p, uint32_t v) {
  p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}

__device__ uint32_t adler_combine(uint32_t a1, uint32_t a2, unsigned long long len2) {  // zlib's adler32_combine
  const uint32_t BASE = 65521u;
  const uint32_t rem = (uint32_t)(len2 % BASE);
  uint32_t sum1 = a1 & 0xffffu;
  uint32_t sum2 = (uint32_t)(((unsigned long long)rem * sum1) % BASE);
  sum1 += (a2 & 0xffffu) + BASE - 1;
  sum2 += ((a1 >> 16) & 0xffffu) + ((a2 >> 16) & 0xffffu) + BASE - rem;
  if (sum1 >= BASE) sum1 -= BASE;
  if (sum1 >= BASE) sum1 -= BASE;
  if (sum2 >= (BASE << 1)) sum2 -= (BASE << 1);
  if (sum2 >= BASE) sum2 -= BASE;
  return sum1 | (sum2 << 16);
}

// one CTA: segment offsets, the framing chunks, the Adler-32 trailer, the file size
__global__ void __launch_bounds__(1024) png_assemble_kernel(const uint32_t* __restrict__ seg_meta, int nseg,
                                                            unsigned long long n_in, int W, int H,
                                                            unsigned long long* __restrict__ seg_off,
                                                            uint8_t* __restrict__ file,
                                                            unsigned long long* __restrict__ total) {
  __shared__ uint32_t crc_table[256], x2n[32], scan[32];
  __shared__ unsigned long long carry;
  crc_table_init(crc_table, x2n);
  if (threadIdx.x == 0) carry = RTRB_PNG_FIXED_BYTES - 16 - 12;  // after the signature, IHDR and the zlib header
  __syncthreads();
  for (int base = 0; base < nseg; base += blockDim.x) {
    const int s = base + threadIdx.x;
    const uint32_t sz = s < nseg ? seg_meta[3 * s] + RTRB_PNG_CHUNK_BYTES : 0;
    uint32_t tot;
    const uint32_t incl = block_scan<false>(sz, scan, tot);
    if (s < nseg) seg_off[s] = carry + incl - sz;
    __syncthreads();
    if (threadIdx.x == 0) carry += tot;
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  uint8_t* p = file;
  const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
  for (int i = 0; i < 8; ++i) p[i] = sig[i];
  p += 8;
  put_be32(p, 13); p[4] = 'I'; p[5] = 'H'; p[6] = 'D'; p[7] = 'R';
  put_be32(p + 8, (uint32_t)W); put_be32(p + 12, (uint32_t)H);
  p[16] = 8; p[17] = 2; p[18] = 0; p[19] = 0; p[20] = 0;  // 8-bit RGB, deflate, adaptive filters, no interlace
  put_be32(p + 21, crc_bytes(p + 4, 17, 0, crc_table));
  p += 25;
  put_be32(p, 2); p[4] = 'I'; p[5] = 'D'; p[6] = 'A'; p[7] = 'T';
  p[8] = 0x78; p[9] = 0x01;  // zlib: deflate, 32 KiB window
  put_be32(p + 10, crc_bytes(p + 4, 6, 0, crc_table));
  uint32_t adler = 1;
  for (int s = 0; s < nseg; ++s) {
    const unsigned long long len = min((unsigned long long)SEG, n_in - (unsigned long long)s * SEG);
    adler = adler_combine(adler, seg_meta[3 * s + 2], len);
  }
  p = file + carry;
  put_be32(p, 4); p[4] = 'I'; p[5] = 'D'; p[6] = 'A'; p[7] = 'T';
  put_be32(p + 8, adler);
  put_be32(p + 12, crc_bytes(p + 4, 8, 0, crc_table));
  p += 16;
  const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xae, 0x42, 0x60, 0x82};
  for (int i = 0; i < 12; ++i) p[i] = iend[i];
  *total = carry + 16 + 12;
}

// one CTA per segment: its IDAT chunk at its offset
__global__ void __launch_bounds__(256) png_place_kernel(const uint8_t* __restrict__ seg_out,
                                                        const uint32_t* __restrict__ seg_meta,
                                                        const unsigned long long* __restrict__ seg_off,
                                                        uint8_t* __restrict__ file) {
  const int s = blockIdx.x;
  const uint32_t n = seg_meta[3 * s];
  uint8_t* p = file + seg_off[s];
  const uint8_t* q = seg_out + (size_t)s * RTRB_PNG_SEGMENT_WORST(SEG);
  if (threadIdx.x == 0) {
    put_be32(p, n); p[4] = 'I'; p[5] = 'D'; p[6] = 'A'; p[7] = 'T';
    put_be32(p + 8 + n, seg_meta[3 * s + 1]);
  }
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) p[8 + i] = q[i];
}

// the finished file into mapped host memory: 16-byte stores where the destination allows, then the byte count
__global__ void __launch_bounds__(256) png_publish_kernel(const uint8_t* __restrict__ file,
                                                          const unsigned long long* __restrict__ total,
                                                          uint8_t* host, unsigned long long* count) {
  const unsigned long long n = *total;
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  const unsigned long long head = (16u - ((uintptr_t)host & 15u)) & 15u;
  const unsigned long long h = min(head, n);
  // the device buffer is 256-byte aligned; read it byte-wise at the host's alignment
  for (size_t i = tid; i < h; i += nth) host[i] = file[i];
  const unsigned long long nv = (n - h) / 16;
  uint4* dst = reinterpret_cast<uint4*>(host + h);
  for (size_t v = tid; v < nv; v += nth) {
    const uint8_t* s = file + h + v * 16;
    uint32_t w[4];
    for (int k = 0; k < 4; ++k)
      w[k] = (uint32_t)s[4 * k] | ((uint32_t)s[4 * k + 1] << 8) | ((uint32_t)s[4 * k + 2] << 16) | ((uint32_t)s[4 * k + 3] << 24);
    dst[v] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  for (size_t i = h + nv * 16 + tid; i < n; i += nth) host[i] = file[i];
  __threadfence_system();
  if (tid == 0) *count = n;
}

}  // namespace

cudaError_t rtrb_png_encode(RtrbPngScratch& s, const uint8_t* src, int width, int height, int pixel_format,
                            cudaStream_t stream, uint8_t* host_mapped, unsigned long long* count_mapped,
                            unsigned long long* launches) {
  const size_t n = rtrb_png_filtered_bytes(width, height), nseg = rtrb_png_segments(width, height);
  cudaError_t e;
  if ((e = s.filtered.ensure(n)) != cudaSuccess || (e = s.tokens.ensure(nseg * SEG)) != cudaSuccess ||
      (e = s.seg_out.ensure(nseg * RTRB_PNG_SEGMENT_WORST(SEG))) != cudaSuccess ||
      (e = s.seg_meta.ensure(nseg * 3)) != cudaSuccess || (e = s.seg_off.ensure(nseg)) != cudaSuccess ||
      (e = s.file.ensure(rtrb_png_bound(width, height))) != cudaSuccess || (e = s.total.ensure(1)) != cudaSuccess)
    return e;
  if ((e = cudaFuncSetAttribute(png_deflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DEFLATE_SMEM)) != cudaSuccess)
    return e;
  png_filter_kernel<<<height, 256, 0, stream>>>(src, width, pixel_format, s.filtered.p);
  png_deflate_kernel<<<(unsigned)nseg, DT, DEFLATE_SMEM, stream>>>(s.filtered.p, n, 3 * width + 1, s.tokens.p, s.seg_out.p,
                                                                   s.seg_meta.p);
  png_assemble_kernel<<<1, 1024, 0, stream>>>(s.seg_meta.p, (int)nseg, n, width, height, s.seg_off.p, s.file.p, s.total.p);
  png_place_kernel<<<(unsigned)nseg, 256, 0, stream>>>(s.seg_out.p, s.seg_meta.p, s.seg_off.p, s.file.p);
  *launches += 4;
  if (host_mapped) {
    png_publish_kernel<<<64, 256, 0, stream>>>(s.file.p, s.total.p, host_mapped, count_mapped);
    *launches += 1;
  }
  return cudaGetLastError();
}
