// JPEG decode on the GPU, byte-equal to cv2.imdecode (libjpeg-turbo's default decode plus OpenCV's EXIF orientation).
//
// The host plans a batch (dvd_jpeg_plan): it parses the headers of every file (never the entropy-coded bytes), validates them and
// writes one table with the geometry, quantisation tables in natural order and Huffman lookup tables of each document.  The decode
// is a fixed sequence of persistent launches over that table, so one captured graph serves every batch planned into it:
//
//   k_jpeg_count    per 4 KB tile of a scan: bytes kept after destuffing (0xFF00 -> 0xFF, markers dropped), RSTn markers
//   k_jpeg_offsets  per document: exclusive scan of the tile counts, destuffed length, segment table defaults
//   k_jpeg_compact  per tile: the destuffed bytes at their scanned offsets; the destuffed offset of every RSTn
//   k_jpeg_sync     per chunk of 128 windows of 128 destuffed bytes: Huffman decode by self-synchronisation (Weissenberger &
//                   Schmidt, ICPP 2018).  A window's entry state is (bit position, block within the MCU, coefficient index).  A
//                   thread decodes its window from its entry state to the first symbol boundary past the window's end and hands
//                   the state it reaches to the next window; the chunk iterates until no entry changes.  Window 0 of a chunk
//                   starts from a guess unless it is the scan's first.
//   k_jpeg_resync   per chunk: a chunk whose entry differs from its predecessor's exit iterates again from that exit (a guessed
//                   chain merges with the true one after some windows, so the exits are already right: this pass is parallel)
//   k_jpeg_fix      per document: chains the chunks in order (a chunk whose entry still differs from its predecessor's exit is
//                   iterated again), then scans the blocks and the DC differences per window (segmented at restarts)
//   k_jpeg_write    per chunk: decodes each window again from its final entry state and writes the int16 coefficients of the
//                   blocks that start in it (natural order, DC predicted)
//   k_jpeg_idct     per 32 blocks: dequantise + jpeg_idct_islow + range limit into component planes
//   k_jpeg_color    per 32x8 output tile: fancy upsampling, ycc_rgb_convert and the EXIF orientation, uint8 HWC RGB out
//
// Correctness never depends on how fast windows synchronise: after n iterations of a chunk its first n entries are exact, so the
// worst case is a sequential decode of the chunk.  A state is compared whole, so the fixed point is the sequential decode.
//
// Restart segments: a segment ends after its last MCU, padded with 1 bits to the byte boundary.  A decoder that completes an MCU ends
// the segment when fewer than 8 bits remain before the next segment's first byte and all of them are 1s: no block starts with an
// all-ones code (the planner rejects tables that would contain one, as libjpeg does), so this happens exactly after the last MCU.
// The restatement is oracle/jpeg_decode.py.
#include "common.cuh"

#include <math.h>
#include <string.h>

#include <algorithm>

namespace dvd {
namespace jpeg {

static constexpr int kTile = 4096;              // raw scan bytes per destuff tile
static constexpr int kTileThreads = 256;        // 16 bytes a thread
static constexpr int kWin = 128;                // destuffed bytes per window
static constexpr int kChunk = 128;              // windows per chunk (= threads of the decode kernels)
static constexpr int kIdctBlocks = 32;          // blocks per k_jpeg_idct task (8 threads each)
static constexpr int kPixW = 32, kPixH = 8;     // output pixels per k_jpeg_color task
static constexpr int kMaxDocs = 1 << 16;
static constexpr long long kMaxScan = 1ll << 28;                 // bit positions stay below 2^31
static constexpr uint32_t kInf = 0xFFFFFFFFu;                    // position of the state past the scan's last MCU

struct alignas(16) Huff {                 // one Huffman table in the decoder's form (jdhuff.c d_derived_tbl)
  uint16_t lut[512];          // 9-bit window -> (length << 8) | symbol; 0: a code longer than 9 bits
  int32_t maxcode[18];        // largest code of length l (10..16), -1 if none
  int32_t valoff[18];         // symbol index of code c of length l: c + valoff[l]
  uint8_t val[256];
};
struct alignas(16) Header {
  int32_t n_docs, pad;
  long long tiles, chunks, idct_tasks, pix_tasks;   // totals of the batch
};
struct alignas(16) Doc {
  const uint8_t* scan;        // device: first entropy-coded byte
  uint8_t* out;               // device: [Ho,Wo,3]
  long long ws;               // workspace offset of this document's regions
  long long tile_base, chunk_base, idct_base, pix_base;       // first global task of each kind
  int32_t stream_off, tiles_off, seg_off, win_off, exit_off, coef_off, plane_off[3];     // offsets from ws
  int32_t scan_len, ntiles, nwin, nchunks, nblocks, nseg, restart;
  int32_t H, W, Ho, Wo, orient, ncomp, mcux, mcuy, bpm;
  int32_t fh, fv;             // chroma upsampling factors (1 or 2)
  int32_t pw[3], dw[3], dh[3];                // plane row pitch, real (downsampled) width and height per component
  int8_t bcomp[8], bdx[8], bdy[8];            // component and offset of each block of an MCU
  int32_t h[3], v[3];
  int32_t pad2;
  uint16_t quant[3][64];      // natural order, per component
  Huff dc[3], ac[3];          // per component
};
static_assert(sizeof(Huff) % 16 == 0 && sizeof(Doc) % 16 == 0 && sizeof(Header) == 48, "jpeg table layout");

struct Win {                  // per window, 32 bytes
  unsigned long long entry;   // entry state: pos << 16 | block << 8 | coefficient
  int32_t nblk;               // blocks started in the window; after k_jpeg_fix: index of the first of them
  int32_t reset;              // the window crossed a restart boundary
  int32_t dc[3];              // DC differences after the last restart in the window; after k_jpeg_fix: predictor at entry
  int32_t pad;
};

static_assert(sizeof(Win) == 32, "window record");

__constant__ uint8_t c_natural[80] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13,
                                      6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                                      39, 46, 53, 60, 61, 54, 47, 55, 62, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63};

static __device__ __forceinline__ unsigned long long pack(uint32_t pos, int b, int z) {
  return ((unsigned long long)pos << 16) | ((unsigned)b << 8) | (unsigned)z;
}

// the document of global task t: the last d with base(d) <= t (bases ascend)
template <typename F>
static __device__ __forceinline__ int doc_of(long long t, int n, F base) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (base(mid) <= t) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// ---- destuffing ----
// keep: a byte other than 0xFF unless it follows 0xFF (stuffed 0x00, marker code), 0xFF only when 0x00 follows; an RSTn is the code
// byte D0..D7 after 0xFF
static __device__ __forceinline__ void tile_load(const Doc& d, long long t0, int n, uint8_t* sm, int& prev, int& next) {
  for (int i = threadIdx.x; i < n; i += kTileThreads) sm[i] = __ldg(d.scan + t0 + i);
  prev = t0 > 0 ? __ldg(d.scan + t0 - 1) : 0;
  next = t0 + n < d.scan_len ? __ldg(d.scan + t0 + n) : 0xFF;
}
static __device__ __forceinline__ void byte_flags(const uint8_t* sm, int n, int i, int prev, int next, bool& keep, bool& rst) {
  const int b = sm[i], p = i > 0 ? sm[i - 1] : prev, nx = i + 1 < n ? sm[i + 1] : next;
  keep = b == 0xFF ? nx == 0 : p != 0xFF;
  rst = p == 0xFF && b >= 0xD0 && b <= 0xD7;
}

template <int N>
static __device__ __forceinline__ int block_excl_scan(int v, int* sm_warp, int& total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sm_warp[wid] = x;
  __syncthreads();
  if (wid == 0) {
    int s = lane < N / 32 ? sm_warp[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += y;
    }
    if (lane < N / 32) sm_warp[lane] = s;
  }
  __syncthreads();
  total = sm_warp[N / 32 - 1];
  const int r = x - v + (wid ? sm_warp[wid - 1] : 0);
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(kTileThreads) k_jpeg_count(const Header* __restrict__ hdr, const Doc* __restrict__ docs,
                                                             uint8_t* __restrict__ ws) {
  __shared__ uint8_t sm[kTile];
  __shared__ int red[kTileThreads / 32];
  const int n_docs = hdr->n_docs;
  for (long long t = blockIdx.x; t < hdr->tiles; t += gridDim.x) {
    const int di = doc_of(t, n_docs, [&](int i) { return docs[i].tile_base; });
    const Doc& d = docs[di];
    const long long tile = t - d.tile_base, t0 = tile * kTile;
    const int n = (int)min((long long)kTile, d.scan_len - t0);
    int prev, next;
    tile_load(d, t0, n, sm, prev, next);
    __syncthreads();
    int keep = 0, rst = 0;
    for (int i = threadIdx.x * 16; i < min(n, threadIdx.x * 16 + 16); ++i) {
      bool k, r;
      byte_flags(sm, n, i, prev, next, k, r);
      keep += k;
      rst += r;
    }
    int tk, tr;
    block_excl_scan<kTileThreads>(keep, red, tk);
    block_excl_scan<kTileThreads>(rst, red, tr);
    if (threadIdx.x == 0) {
      int* cnt = reinterpret_cast<int*>(ws + d.ws + d.tiles_off) + 2 * tile;
      cnt[0] = tk;
      cnt[1] = tr;
    }
  }
}

// one CTA per document: tile counts -> offsets, destuffed length into seg[nseg], zero padding after the stream, segment starts past
// the markers found default to the end (a corrupt scan with too few markers decodes its missing segments as empty)
__global__ void __launch_bounds__(1024) k_jpeg_offsets(const Header* __restrict__ hdr, const Doc* __restrict__ docs,
                                                       uint8_t* __restrict__ ws) {
  __shared__ int red[32];
  for (int di = blockIdx.x; di < hdr->n_docs; di += gridDim.x) {
    const Doc& d = docs[di];
    int* cnt = reinterpret_cast<int*>(ws + d.ws + d.tiles_off);
    int ck = 0, cr = 0;
    for (int t0 = 0; t0 < d.ntiles; t0 += 1024) {
      const int t = t0 + threadIdx.x;
      const int k = t < d.ntiles ? cnt[2 * t] : 0, r = t < d.ntiles ? cnt[2 * t + 1] : 0;
      int tk, tr;
      const int ek = block_excl_scan<1024>(k, red, tk), er = block_excl_scan<1024>(r, red, tr);
      if (t < d.ntiles) {
        cnt[2 * t] = ck + ek;
        cnt[2 * t + 1] = cr + er;
      }
      ck += tk;
      cr += tr;
    }
    uint32_t* seg = reinterpret_cast<uint32_t*>(ws + d.ws + d.seg_off);
    if (threadIdx.x == 0) seg[0] = 0;
    for (int k = min(cr, d.nseg - 1) + 1 + threadIdx.x; k <= d.nseg; k += 1024) seg[k] = ck;
    if (threadIdx.x < 8) ws[d.ws + d.stream_off + ck + threadIdx.x] = 0;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kTileThreads) k_jpeg_compact(const Header* __restrict__ hdr, const Doc* __restrict__ docs,
                                                               uint8_t* __restrict__ ws) {
  __shared__ uint8_t sm[kTile];
  __shared__ int red[kTileThreads / 32];
  const int n_docs = hdr->n_docs;
  for (long long t = blockIdx.x; t < hdr->tiles; t += gridDim.x) {
    const int di = doc_of(t, n_docs, [&](int i) { return docs[i].tile_base; });
    const Doc& d = docs[di];
    const long long tile = t - d.tile_base, t0 = tile * kTile;
    const int n = (int)min((long long)kTile, d.scan_len - t0);
    int prev, next;
    tile_load(d, t0, n, sm, prev, next);
    __syncthreads();
    const int i0 = threadIdx.x * 16, i1 = min(n, i0 + 16);
    int keep = 0, rst = 0;
    for (int i = i0; i < i1; ++i) {
      bool k, r;
      byte_flags(sm, n, i, prev, next, k, r);
      keep += k;
      rst += r;
    }
    int tk, tr;
    const int* cnt = reinterpret_cast<const int*>(ws + d.ws + d.tiles_off) + 2 * tile;
    int o = cnt[0] + block_excl_scan<kTileThreads>(keep, red, tk);
    int m = cnt[1] + block_excl_scan<kTileThreads>(rst, red, tr);
    uint8_t* out = ws + d.ws + d.stream_off;
    uint32_t* seg = reinterpret_cast<uint32_t*>(ws + d.ws + d.seg_off);
    for (int i = i0; i < i1; ++i) {
      bool k, r;
      byte_flags(sm, n, i, prev, next, k, r);
      if (k) out[o++] = sm[i];
      if (r) {
        if (m < d.nseg - 1) seg[m + 1] = o;
        ++m;
      }
    }
    __syncthreads();
  }
}

// ---- entropy decode ----
struct Dec {
  const uint32_t* words;      // destuffed stream, 16-byte aligned, zero-padded for 8 bytes past len
  const uint32_t* seg;        // segment starts in bytes, seg[nseg] = len
  const Huff* huff;           // shared: dc[0..2], ac[0..2]
  const int8_t* bcomp;        // shared
  uint32_t len;
  int nseg, bpm;
};

static __device__ __forceinline__ uint32_t word_be(const Dec& d, uint32_t wi) {
  return 4ull * wi < (unsigned long long)d.len + 8 ? __byte_perm(d.words[wi], 0, 0x0123) : 0u;
}
// 32 bits starting at bit pos (zeros past the stream)
static __device__ __forceinline__ uint32_t peek32(const Dec& d, uint32_t pos) {
  const uint32_t wi = pos >> 5, sh = pos & 31;
  const uint32_t hi = word_be(d, wi);
  return sh ? (hi << sh) | (word_be(d, wi + 1) >> (32 - sh)) : hi;
}
// (length, symbol) of the code at the top of w; a bad code decodes as symbol 0 and consumes 16 bits
static __device__ __forceinline__ void huff_decode(const Huff& h, uint32_t w, int& len, int& sym) {
  const int e = h.lut[w >> 23];
  if (e) {
    len = e >> 8;
    sym = e & 255;
    return;
  }
  len = 16;
  sym = 0;
#pragma unroll 1
  for (int l = 10; l <= 16; ++l) {
    const int code = (int)(w >> (32 - l));
    if (code <= h.maxcode[l]) {
      len = l;
      sym = h.val[(code + h.valoff[l]) & 255];
      break;
    }
  }
}
static __device__ __forceinline__ int extend(int r, int s) { return s && r < (1 << (s - 1)) ? r - (1 << s) + 1 : r; }

static __device__ __forceinline__ int segment_of(const Dec& d, uint32_t pos) {
  int lo = 0, hi = d.nseg - 1;
  const uint32_t byte = pos >> 3;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (d.seg[mid] <= byte) lo = mid; else hi = mid - 1;
  }
  return lo;
}

struct Acc {                  // what the sync pass records about a window
  int nblk, reset, dc[3];
};
struct Out {                  // where the write pass puts the coefficients of a window
  int16_t* coef;
  int blk, nblocks, pred[3];
};

// Decodes from state st.  Sync pass (WRITE = false): up to the first symbol boundary at or past bit `end`, accumulating into acc.
// Write pass: the blocks whose DC starts before `end`, in full, into out.  Returns the state reached.
template <bool WRITE>
static __device__ __forceinline__ unsigned long long run(const Dec& d, unsigned long long st, uint32_t end, Acc& acc, Out& out) {
  uint32_t pos = (uint32_t)(st >> 16);
  int b = (int)(st >> 8) & 255, z = (int)st & 255;
  int k = pos == kInf ? 0 : segment_of(d, pos);
  bool writing = false;
  int16_t* blk = nullptr;
  while (true) {
    if (WRITE) {
      if (z == 0) {
        if (pos >= end) break;
        ++out.blk;
        writing = out.blk < out.nblocks;
        blk = out.coef + 64ll * out.blk;
        if (writing) {
          int4* p = reinterpret_cast<int4*>(blk);
#pragma unroll
          for (int i = 0; i < 8; ++i) p[i] = make_int4(0, 0, 0, 0);
        }
      } else if (!writing && pos >= end) {
        break;
      }
    } else if (pos >= end) {
      break;
    }
    const int c = d.bcomp[b];
    const uint32_t w = peek32(d, pos);
    int len, sym;
    if (z == 0) {
      huff_decode(d.huff[c], w, len, sym);
      const int s = min(sym, 16);
      const int r = s ? (int)((w << len) >> (32 - s)) : 0;
      pos += len + s;
      const int diff = extend(r, s);
      if (WRITE) {                                   // component indices select registers (no local-memory array)
        const int p = (c == 0 ? out.pred[0] : c == 1 ? out.pred[1] : out.pred[2]) + diff;
        out.pred[0] = c == 0 ? p : out.pred[0];
        out.pred[1] = c == 1 ? p : out.pred[1];
        out.pred[2] = c == 2 ? p : out.pred[2];
        if (writing) blk[0] = (int16_t)p;
      } else {
        ++acc.nblk;
        acc.dc[0] += c == 0 ? diff : 0;
        acc.dc[1] += c == 1 ? diff : 0;
        acc.dc[2] += c == 2 ? diff : 0;
      }
      z = 1;
    } else {
      huff_decode(d.huff[3 + c], w, len, sym);
      const int r = sym >> 4, s = sym & 15;
      if (s) {
        const int v = (int)((w << len) >> (32 - s));
        z += r;
        if (WRITE && writing) blk[c_natural[z]] = (int16_t)extend(v, s);
        z += 1;
      } else {
        z = r == 15 ? z + 16 : 64;
      }
      pos += len + s;
    }
    if (z >= 64) {
      z = 0;
      b = b + 1 == d.bpm ? 0 : b + 1;
      if (WRITE) writing = false;
      // an MCU is complete: at the end of the segment, go to the next one right away, so that a state handed to the next window is
      // never "end of segment k" (which would share its position with "start of segment k + 1" when there is no padding)
      while (b == 0) {
        const uint32_t q = 8u * d.seg[k + 1], left = q - pos;
        if (!(pos >= q || (left < 8 && (peek32(d, pos) >> (32 - left)) == (1u << left) - 1))) break;
        if (k + 1 >= d.nseg) {
          pos = kInf;
          break;
        }
        ++k;
        pos = max(pos, q);
        if (WRITE) {
          out.pred[0] = out.pred[1] = out.pred[2] = 0;
        } else {
          acc.reset = 1;
          acc.dc[0] = acc.dc[1] = acc.dc[2] = 0;
        }
      }
      if (pos == kInf) break;
    }
  }
  return pack(pos, b, z);
}

// exit states of the chunks: 0 as k_jpeg_sync leaves them, 1 after k_jpeg_resync (and k_jpeg_fix)
static __device__ __forceinline__ unsigned long long* exits_of(const Doc& d, uint8_t* ws, int which) {
  return reinterpret_cast<unsigned long long*>(ws + d.ws + d.exit_off) + (long long)which * d.nchunks;
}

// The decode kernels run a CTA of kChunk threads per chunk; the document's tables go to shared memory.
struct Shared {
  Huff huff[6];
  int8_t bcomp[8];
  unsigned long long entry[kChunk];
  int any;
};

static __device__ Dec load_doc(const Doc& d, uint8_t* ws, Shared& sh) {
  __syncthreads();                                  // the previous task of this CTA is done with the tables
  const int4* src = reinterpret_cast<const int4*>(d.dc);
  int4* dst = reinterpret_cast<int4*>(sh.huff);
  for (int i = threadIdx.x; i < (int)(6 * sizeof(Huff) / 16); i += blockDim.x) dst[i] = src[i];
  if (threadIdx.x < 8) sh.bcomp[threadIdx.x] = d.bcomp[threadIdx.x];
  __syncthreads();
  Dec dec;
  dec.words = reinterpret_cast<const uint32_t*>(ws + d.ws + d.stream_off);
  dec.seg = reinterpret_cast<const uint32_t*>(ws + d.ws + d.seg_off);
  dec.len = dec.seg[d.nseg];
  dec.huff = sh.huff;
  dec.bcomp = sh.bcomp;
  dec.nseg = d.nseg;
  dec.bpm = d.bpm;
  return dec;
}

// The fixed point of one chunk: entries start from `guess` (the stored ones, or each window's first bit with block 0, coefficient
// 0); entry 0 is `entry0`.  Writes the final entries and what each window's decode recorded, and the chunk's exit state.
static __device__ __forceinline__ void fixpoint(const Doc& d, const Dec& dec, uint8_t* ws, Shared& sh, int chunk, unsigned long long entry0,
                                                bool stored, unsigned long long* exits) {
  Win* win = reinterpret_cast<Win*>(ws + d.ws + d.win_off);
  const int t = threadIdx.x, w = chunk * kChunk + t;
  const bool valid = w < d.nwin;
  const uint32_t end = (uint32_t)min((unsigned long long)(w + 1) * kWin * 8, 0xFFFFFFFEull);
  unsigned long long e = t == 0 ? entry0 : valid ? (stored ? win[w].entry : pack((uint32_t)w * kWin * 8, 0, 0)) : 0;
  sh.entry[t] = e;
  Acc acc{};
  Out none{};
  unsigned long long x = e;
  bool dirty = true;
  __syncthreads();
  while (true) {
    if (dirty && valid) {
      acc = Acc{};
      x = run<false>(dec, e, end, acc, none);
    }
    const bool ch = valid && t + 1 < kChunk && w + 1 < d.nwin && sh.entry[t + 1] != x;
    __syncthreads();
    if (ch) sh.entry[t + 1] = x;
    if (!__syncthreads_or(ch)) break;
    dirty = sh.entry[t] != e;
    e = sh.entry[t];
  }
  if (valid) {
    Win r;
    r.entry = e;
    r.nblk = acc.nblk;
    r.reset = acc.reset;
    r.dc[0] = acc.dc[0];
    r.dc[1] = acc.dc[1];
    r.dc[2] = acc.dc[2];
    r.pad = 0;
    win[w] = r;
    if (t == kChunk - 1 || w == d.nwin - 1) exits[chunk] = x;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kChunk, 8) k_jpeg_sync(const Header* __restrict__ hdr, const Doc* __restrict__ docs, uint8_t* ws) {
  __shared__ Shared sh;
  const int n_docs = hdr->n_docs;
  for (long long t = blockIdx.x; t < hdr->chunks; t += gridDim.x) {
    const int di = doc_of(t, n_docs, [&](int i) { return docs[i].chunk_base; });
    const Doc& d = docs[di];
    const int chunk = (int)(t - d.chunk_base);
    const Dec dec = load_doc(d, ws, sh);
    fixpoint(d, dec, ws, sh, chunk, pack((uint32_t)chunk * kChunk * kWin * 8, 0, 0), false, exits_of(d, ws, 0));
  }
}

// All chunks at once: a chunk whose guessed entry is not its predecessor's exit after k_jpeg_sync iterates again from that exit.
// A chunk's guessed chain usually merges with the true one well inside the chunk, so its exit is already right and one such pass
// leaves k_jpeg_fix nothing but checks.  Exits go to a second array so that every chunk reads its predecessor's k_jpeg_sync exit.
__global__ void __launch_bounds__(kChunk, 8) k_jpeg_resync(const Header* __restrict__ hdr, const Doc* __restrict__ docs, uint8_t* ws) {
  __shared__ Shared sh;
  const int n_docs = hdr->n_docs;
  for (long long t = blockIdx.x; t < hdr->chunks; t += gridDim.x) {
    const int di = doc_of(t, n_docs, [&](int i) { return docs[i].chunk_base; });
    const Doc& d = docs[di];
    const int chunk = (int)(t - d.chunk_base);
    const unsigned long long* prev = exits_of(d, ws, 0);
    unsigned long long* next = exits_of(d, ws, 1);
    const unsigned long long entry = chunk ? prev[chunk - 1] : 0;
    if (chunk == 0 || reinterpret_cast<const Win*>(ws + d.ws + d.win_off)[chunk * kChunk].entry == entry) {
      if (threadIdx.x == 0) next[chunk] = prev[chunk];
      continue;
    }
    const Dec dec = load_doc(d, ws, sh);
    fixpoint(d, dec, ws, sh, chunk, entry, true, next);
  }
}

// one CTA per document
__global__ void __launch_bounds__(kChunk) k_jpeg_fix(const Header* __restrict__ hdr, const Doc* __restrict__ docs, uint8_t* ws) {
  __shared__ Shared sh;
  __shared__ int first;
  __shared__ int agg[kChunk][5];
  __shared__ int carry[5];
  for (int di = blockIdx.x; di < hdr->n_docs; di += gridDim.x) {
    const Doc& d = docs[di];
    const Dec dec = load_doc(d, ws, sh);
    Win* win = reinterpret_cast<Win*>(ws + d.ws + d.win_off);
    unsigned long long* exits = exits_of(d, ws, 1);
    // chain the chunks: find the first chunk whose entry is not its predecessor's exit, iterate it again, go on after it
    for (int c = 1; c < d.nchunks;) {
      if (threadIdx.x == 0) first = d.nchunks;
      __syncthreads();
      const int i = c + threadIdx.x;
      if (i < d.nchunks && *(volatile const unsigned long long*)&exits[i - 1] != *(volatile const unsigned long long*)&win[i * kChunk].entry)
        atomicMin(&first, i);
      __syncthreads();
      const int f = first;
      __syncthreads();
      if (f >= d.nchunks) {
        c += kChunk;
        continue;
      }
      fixpoint(d, dec, ws, sh, f, *(volatile const unsigned long long*)&exits[f - 1], true, exits);
      __threadfence_block();
      c = f + 1;
    }
    // scan the windows: blocks (a sum) and DC differences (per component, restarted where a window crossed a restart boundary).
    // A thread aggregates kPer consecutive windows, thread 0 scans the aggregates, each thread writes its windows.
    constexpr int kPer = 8;
    if (threadIdx.x == 0) carry[0] = carry[1] = carry[2] = carry[3] = carry[4] = 0;
    for (int w0 = 0; w0 < d.nwin; w0 += kChunk * kPer) {
      const int a = w0 + threadIdx.x * kPer, e = min(a + kPer, d.nwin);
      int g[5] = {0, 0, 0, 0, 0};                           // blocks, reset, dc[3]
      for (int w = a; w < e; ++w) {
        const Win& r = win[w];
        g[0] += r.nblk;
        if (r.reset) g[1] = 1, g[2] = g[3] = g[4] = 0;
        g[2] += r.dc[0];
        g[3] += r.dc[1];
        g[4] += r.dc[2];
      }
      for (int k = 0; k < 5; ++k) agg[threadIdx.x][k] = g[k];
      __syncthreads();
      if (threadIdx.x == 0) {
        int p[5] = {carry[0], 0, carry[2], carry[3], carry[4]};
        for (int j = 0; j < kChunk; ++j) {
          int x[5];
          for (int k = 0; k < 5; ++k) x[k] = agg[j][k], agg[j][k] = p[k];
          p[0] += x[0];
          for (int k = 2; k < 5; ++k) p[k] = x[1] ? x[k] : p[k] + x[k];
        }
        for (int k = 0; k < 5; ++k) carry[k] = p[k];
      }
      __syncthreads();
      int base = agg[threadIdx.x][0], p[3] = {agg[threadIdx.x][2], agg[threadIdx.x][3], agg[threadIdx.x][4]};
      for (int w = a; w < e; ++w) {
        Win r = win[w];
        const int n = r.nblk, d0 = r.dc[0], d1 = r.dc[1], d2 = r.dc[2];
        r.nblk = base;
        r.dc[0] = p[0];
        r.dc[1] = p[1];
        r.dc[2] = p[2];
        win[w] = r;
        base += n;
        if (r.reset) p[0] = p[1] = p[2] = 0;
        p[0] += d0;
        p[1] += d1;
        p[2] += d2;
      }
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(kChunk) k_jpeg_write(const Header* __restrict__ hdr, const Doc* __restrict__ docs, uint8_t* ws) {
  __shared__ Shared sh;
  const int n_docs = hdr->n_docs;
  for (long long t = blockIdx.x; t < hdr->chunks; t += gridDim.x) {
    const int di = doc_of(t, n_docs, [&](int i) { return docs[i].chunk_base; });
    const Doc& d = docs[di];
    const Dec dec = load_doc(d, ws, sh);
    const int w = (int)(t - d.chunk_base) * kChunk + threadIdx.x;
    if (w >= d.nwin) continue;
    const Win r = reinterpret_cast<const Win*>(ws + d.ws + d.win_off)[w];
    Acc acc{};
    Out out;
    out.coef = reinterpret_cast<int16_t*>(ws + d.ws + d.coef_off);
    out.blk = r.nblk - 1;
    out.nblocks = d.nblocks;
    out.pred[0] = r.dc[0];
    out.pred[1] = r.dc[1];
    out.pred[2] = r.dc[2];
    run<true>(dec, r.entry, (uint32_t)min((unsigned long long)(w + 1) * kWin * 8, 0xFFFFFFFEull), acc, out);
  }
}

// ---- pixels ----
// jidctint.c jpeg_idct_islow, CONST_BITS 13, PASS1_BITS 2
#define FIX_0_298631336 2446
#define FIX_0_390180644 3196
#define FIX_0_541196100 4433
#define FIX_0_765366865 6270
#define FIX_0_899976223 7373
#define FIX_1_175875602 9633
#define FIX_1_501321110 12299
#define FIX_1_847759065 15137
#define FIX_1_961570560 16069
#define FIX_2_053119869 16819
#define FIX_2_562915447 20995
#define FIX_3_072711026 25172

static __device__ __forceinline__ void idct8(const int* in, int* out, int shift) {
  int z2 = in[2], z3 = in[6];
  int z1 = (z2 + z3) * FIX_0_541196100;
  const int tmp2 = z1 + z3 * -FIX_1_847759065;
  const int tmp3 = z1 + z2 * FIX_0_765366865;
  const int tmp0 = (in[0] + in[4]) * (1 << 13);
  const int tmp1 = (in[0] - in[4]) * (1 << 13);
  const int t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
  int o0 = in[7], o1 = in[5], o2 = in[3], o3 = in[1];
  z1 = o0 + o3;
  z2 = o1 + o2;
  z3 = o0 + o2;
  int z4 = o1 + o3;
  const int z5 = (z3 + z4) * FIX_1_175875602;
  o0 *= FIX_0_298631336;
  o1 *= FIX_2_053119869;
  o2 *= FIX_3_072711026;
  o3 *= FIX_1_501321110;
  z1 *= -FIX_0_899976223;
  z2 *= -FIX_2_562915447;
  z3 = z3 * -FIX_1_961570560 + z5;
  z4 = z4 * -FIX_0_390180644 + z5;
  o0 += z1 + z3;
  o1 += z2 + z4;
  o2 += z2 + z3;
  o3 += z1 + z4;
  const int rnd = 1 << (shift - 1);
  out[0] = (t10 + o3 + rnd) >> shift;
  out[7] = (t10 - o3 + rnd) >> shift;
  out[1] = (t11 + o2 + rnd) >> shift;
  out[6] = (t11 - o2 + rnd) >> shift;
  out[2] = (t12 + o1 + rnd) >> shift;
  out[5] = (t12 - o1 + rnd) >> shift;
  out[3] = (t13 + o0 + rnd) >> shift;
  out[4] = (t13 - o0 + rnd) >> shift;
}
// jdmaster.c post-IDCT range limit indexed with & RANGE_MASK
static __device__ __forceinline__ uint32_t range_limit(int v) {
  v &= 1023;
  return (uint32_t)min(max((v < 512 ? v : v - 1024) + 128, 0), 255);
}

__global__ void __launch_bounds__(8 * kIdctBlocks) k_jpeg_idct(const Header* __restrict__ hdr, const Doc* __restrict__ docs,
                                                               uint8_t* __restrict__ ws) {
  __shared__ int16_t coef[kIdctBlocks][64];
  __shared__ int mid[kIdctBlocks][8][9];
  const int n_docs = hdr->n_docs, g = threadIdx.x >> 3, j = threadIdx.x & 7;
  for (long long t = blockIdx.x; t < hdr->idct_tasks; t += gridDim.x) {
    const int di = doc_of(t, n_docs, [&](int i) { return docs[i].idct_base; });
    const Doc& d = docs[di];
    const int b0 = (int)(t - d.idct_base) * kIdctBlocks, nb = min(kIdctBlocks, d.nblocks - b0);
    const int4* src = reinterpret_cast<const int4*>(ws + d.ws + d.coef_off) + (long long)b0 * 8;
    __syncthreads();
    if (threadIdx.x < nb * 8) reinterpret_cast<int4*>(coef)[threadIdx.x] = src[threadIdx.x];
    __syncthreads();
    const int k = b0 + g;
    const int mcu = k / d.bpm, jb = k - mcu * d.bpm, c = d.bcomp[jb];
    if (g < nb) {                                   // pass 1: column j
      int in[8], out[8];
      const bool ac0 = coef[g][8 + j] == 0 && coef[g][16 + j] == 0 && coef[g][24 + j] == 0 && coef[g][32 + j] == 0 &&
                       coef[g][40 + j] == 0 && coef[g][48 + j] == 0 && coef[g][56 + j] == 0;
#pragma unroll
      for (int r = 0; r < 8; ++r) in[r] = (int)coef[g][8 * r + j] * (int)d.quant[c][8 * r + j];
      if (ac0) {
#pragma unroll
        for (int r = 0; r < 8; ++r) out[r] = in[0] * 4;
      } else {
        idct8(in, out, 13 - 2);
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) mid[g][r][j] = out[r];
    }
    __syncthreads();
    if (g < nb) {                                   // pass 2: row j
      int in[8], out[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) in[i] = mid[g][j][i];
      idct8(in, out, 13 + 2 + 3);
      const int mx = mcu % d.mcux, my = mcu / d.mcux;
      const int bx = mx * d.h[c] + d.bdx[jb], by = my * d.v[c] + d.bdy[jb];
      uint8_t* dst = ws + d.ws + d.plane_off[c] + (long long)(by * 8 + j) * d.pw[c] + bx * 8;
      uint2 v;
      v.x = range_limit(out[0]) | range_limit(out[1]) << 8 | range_limit(out[2]) << 16 | range_limit(out[3]) << 24;
      v.y = range_limit(out[4]) | range_limit(out[5]) << 8 | range_limit(out[6]) << 16 | range_limit(out[7]) << 24;
      *reinterpret_cast<uint2*>(dst) = v;
    }
  }
}

// jdsample.c: chroma sample at full-resolution (y, x) of a component downsampled by (fh, fv)
static __device__ __forceinline__ int chroma(const uint8_t* __restrict__ p, int pitch, int dw, int dh, int fh, int fv, int y, int x) {
  if (fh == 1) return __ldg(p + (long long)y * pitch + x);
  if (dw <= 2) return __ldg(p + (long long)(y / fv) * pitch + (x >> 1));       // jinit_upsampler: plain replication
  const int j = x >> 1, jn = x & 1 ? min(j + 1, dw - 1) : max(j - 1, 0);
  if (fv == 1) {
    const uint8_t* row = p + (long long)y * pitch;
    return (3 * __ldg(row + j) + __ldg(row + jn) + 1 + (x & 1)) >> 2;
  }
  const int i = y >> 1, fi = y & 1 ? min(i + 1, dh - 1) : max(i - 1, 0);
  const uint8_t* near = p + (long long)i * pitch;
  const uint8_t* far = p + (long long)fi * pitch;
  const int cs = 3 * __ldg(near + j) + __ldg(far + j), csn = 3 * __ldg(near + jn) + __ldg(far + jn);
  return (3 * cs + csn + 8 - (x & 1)) >> 4;
}

__global__ void __launch_bounds__(kPixW * kPixH) k_jpeg_color(const Header* __restrict__ hdr, const Doc* __restrict__ docs,
                                                              const uint8_t* __restrict__ ws) {
  const int n_docs = hdr->n_docs;
  for (long long t = blockIdx.x; t < hdr->pix_tasks; t += gridDim.x) {
    const int di = doc_of(t, n_docs, [&](int i) { return docs[i].pix_base; });
    const Doc& d = docs[di];
    const int tile = (int)(t - d.pix_base), tx = (d.Wo + kPixW - 1) / kPixW;
    const int r = tile / tx * kPixH + (threadIdx.x >> 5), c = tile % tx * kPixW + (threadIdx.x & 31);
    if (r >= d.Ho || c >= d.Wo) continue;
    int y, x;                                        // OpenCV's EXIF transform: the source pixel of output (r, c)
    switch (d.orient) {
      case 2: y = r; x = d.W - 1 - c; break;
      case 3: y = d.H - 1 - r; x = d.W - 1 - c; break;
      case 4: y = d.H - 1 - r; x = c; break;
      case 5: y = c; x = r; break;
      case 6: y = d.H - 1 - c; x = r; break;
      case 7: y = d.H - 1 - c; x = d.W - 1 - r; break;
      case 8: y = c; x = d.W - 1 - r; break;
      default: y = r; x = c; break;
    }
    const uint8_t* base = ws + d.ws;
    const int Y = __ldg(base + d.plane_off[0] + (long long)y * d.pw[0] + x);
    int R = Y, G = Y, B = Y;
    if (d.ncomp == 3) {
      const int cb = chroma(base + d.plane_off[1], d.pw[1], d.dw[1], d.dh[1], d.fh, d.fv, y, x) - 128;
      const int cr = chroma(base + d.plane_off[2], d.pw[2], d.dw[2], d.dh[2], d.fh, d.fv, y, x) - 128;
      // jdcolor.c build_ycc_rgb_table, SCALEBITS 16
      R = min(max(Y + ((91881 * cr + 32768) >> 16), 0), 255);
      G = min(max(Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16), 0), 255);
      B = min(max(Y + ((116130 * cb + 32768) >> 16), 0), 255);
    }
    uint8_t* o = d.out + ((long long)r * d.Wo + c) * 3;
    o[0] = (uint8_t)R;
    o[1] = (uint8_t)G;
    o[2] = (uint8_t)B;
  }
}

// ---- host: header parsing and planning ----
struct Parsed {
  int H, W, ncomp, hmax, vmax, restart, orient, scan_start, scan_len;
  int h[3], v[3], tq[3], td[3], ta[3];
  uint16_t quant[4][64];
  bool qdef[4];
  int hbits[2][4][17];        // [class][id][length]
  uint8_t hval[2][4][256];
  bool hdef[2][4];
};

static const int kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

static int be16(const uint8_t* p) { return p[0] << 8 | p[1]; }

// orientation 1..8 of an APP1 Exif payload (1 when malformed)
static int exif_orientation(const uint8_t* s, int n) {
  if (n < 14 || memcmp(s, "Exif\0\0", 6) != 0) return 1;
  const uint8_t* t = s + 6;
  const int tn = n - 6;
  bool le;
  if (t[0] == 'I' && t[1] == 'I') le = true;
  else if (t[0] == 'M' && t[1] == 'M') le = false;
  else return 1;
  auto u16 = [&](int o) { return le ? t[o] | t[o + 1] << 8 : t[o] << 8 | t[o + 1]; };
  auto u32 = [&](int o) {
    return le ? (uint32_t)t[o] | (uint32_t)t[o + 1] << 8 | (uint32_t)t[o + 2] << 16 | (uint32_t)t[o + 3] << 24
              : (uint32_t)t[o] << 24 | (uint32_t)t[o + 1] << 16 | (uint32_t)t[o + 2] << 8 | (uint32_t)t[o + 3];
  };
  const uint32_t ifd = u32(4);
  if (ifd + 2ull > (uint32_t)tn) return 1;
  const int ne = u16(ifd);
  for (int e = 0; e < ne; ++e) {
    const uint64_t p = ifd + 2ull + 12ull * e;
    if (p + 12 > (uint64_t)tn) return 1;
    if (u16((int)p) == 0x0112) {
      const int v = u16((int)p + 8);
      return v >= 1 && v <= 8 ? v : 1;
    }
  }
  return 1;
}

#define JREQ(cond, fmt, ...) DVD_REQUIRE(cond, "jpeg_plan: document %d: " fmt, di, ##__VA_ARGS__)

static int parse(int di, const uint8_t* b, long long n, Parsed& P) {
  memset(&P, 0, sizeof(P));
  P.orient = 1;
  JREQ(n >= 4 && b[0] == 0xFF && b[1] == 0xD8, "not a JPEG file (no SOI marker)");
  JREQ(b[n - 2] == 0xFF && b[n - 1] == 0xD9, "missing EOI marker at the end of the file (truncated file?)");
  JREQ(n < kMaxScan, "file of %lld bytes is too large (limit %lld)", n, kMaxScan);
  bool sof = false, jfif = false, adobe = false, exif_seen = false;
  int transform = -1, ids[3] = {0, 0, 0};
  long long i = 2;
  while (true) {
    JREQ(i + 4 <= n - 2 && b[i] == 0xFF, "corrupt header: no marker at byte %lld", i);
    while (b[i + 1] == 0xFF && i + 5 <= n - 2) ++i;             // fill bytes
    const int m = b[i + 1];
    JREQ(!(m >= 0xD0 && m <= 0xD9) && m != 0x01 && m != 0x00, "unexpected marker 0x%02X in the header", m);
    const int ln = be16(b + i + 2);
    JREQ(ln >= 2 && i + 2 + ln <= n - 2, "truncated header segment (marker 0x%02X)", m);
    const uint8_t* s = b + i + 4;
    const int sl = ln - 2;
    if (m == 0xC2 || m == 0xC6) {
      JREQ(false, "progressive JPEG is not supported");
    } else if (m == 0xC9 || m == 0xCA || m == 0xCB || m == 0xCC || m == 0xCD || m == 0xCE || m == 0xCF) {
      JREQ(false, "arithmetic coding is not supported");
    } else if (m == 0xC3 || m == 0xC7) {
      JREQ(false, "lossless JPEG is not supported");
    } else if (m == 0xC5) {
      JREQ(false, "hierarchical (differential) JPEG is not supported");
    } else if (m == 0xC0 || m == 0xC1) {
      JREQ(!sof, "more than one frame header");
      JREQ(sl >= 6, "truncated frame header");
      JREQ(s[0] == 8, "%d-bit samples are not supported (8-bit only)", s[0]);
      P.H = be16(s + 1);
      P.W = be16(s + 3);
      P.ncomp = s[5];
      JREQ(P.H > 0, "height 0 (DNL) is not supported");
      JREQ(P.W > 0, "width 0");
      JREQ(P.ncomp == 1 || P.ncomp == 3, "%d components (CMYK / 4 components) are not supported (1 or 3 only)", P.ncomp);
      JREQ(sl >= 6 + 3 * P.ncomp, "truncated frame header");
      for (int c = 0; c < P.ncomp; ++c) {
        ids[c] = s[6 + 3 * c];
        P.h[c] = s[7 + 3 * c] >> 4;
        P.v[c] = s[7 + 3 * c] & 15;
        P.tq[c] = s[8 + 3 * c];
        JREQ(P.tq[c] < 4, "component %d uses quantization table %d", c, P.tq[c]);
        JREQ(P.h[c] >= 1 && P.h[c] <= 4 && P.v[c] >= 1 && P.v[c] <= 4, "bad sampling factors");
      }
      if (P.ncomp == 1) {
        P.h[0] = P.v[0] = 1;                     // one component: a non-interleaved scan of 8x8 blocks
      } else {
        const bool luma_ok = (P.h[0] == 1 && P.v[0] == 1) || (P.h[0] == 2 && P.v[0] == 1) || (P.h[0] == 2 && P.v[0] == 2);
        JREQ(luma_ok && P.h[1] == 1 && P.v[1] == 1 && P.h[2] == 1 && P.v[2] == 1,
             "sampling %dx%d,%dx%d,%dx%d is not supported (4:4:4, 4:2:2 and 4:2:0 only)", P.h[0], P.v[0], P.h[1], P.v[1], P.h[2],
             P.v[2]);
      }
      P.hmax = P.h[0];
      P.vmax = P.v[0];
      sof = true;
    } else if (m == 0xDB) {
      for (int p = 0; p < sl;) {
        const int pq = s[p] >> 4, tq = s[p] & 15, nb = pq ? 128 : 64;
        JREQ(pq <= 1 && tq < 4 && p + 1 + nb <= sl, "bad quantization table");
        for (int k = 0; k < 64; ++k) P.quant[tq][kZigzag[k]] = pq ? be16(s + p + 1 + 2 * k) : s[p + 1 + k];
        P.qdef[tq] = true;
        p += 1 + nb;
      }
    } else if (m == 0xC4) {
      for (int p = 0; p < sl;) {
        JREQ(p + 17 <= sl, "truncated Huffman table");
        const int tc = s[p] >> 4, th = s[p] & 15;
        JREQ(tc <= 1 && th < 4, "bad Huffman table class %d / id %d", tc, th);
        int count = 0;
        P.hbits[tc][th][0] = 0;
        for (int l = 1; l <= 16; ++l) count += (P.hbits[tc][th][l] = s[p + l]);
        JREQ(count <= 256 && p + 17 + count <= sl, "bad Huffman table");
        memset(P.hval[tc][th], 0, 256);
        memcpy(P.hval[tc][th], s + p + 17, count);
        P.hdef[tc][th] = true;
        p += 17 + count;
      }
    } else if (m == 0xDD) {
      JREQ(sl >= 2, "truncated restart interval");
      P.restart = be16(s);
    } else if (m == 0xDC) {
      JREQ(false, "height 0 (DNL) is not supported");
    } else if (m == 0xE0) {
      if (sl >= 5 && memcmp(s, "JFIF\0", 5) == 0) jfif = true;
    } else if (m == 0xE1) {
      if (!exif_seen && sl >= 6 && memcmp(s, "Exif\0\0", 6) == 0) {
        P.orient = exif_orientation(s, sl);
        exif_seen = true;
      }
    } else if (m == 0xEE) {
      if (sl >= 12 && memcmp(s, "Adobe", 5) == 0) {
        adobe = true;
        transform = s[11];
      }
    } else if (m == 0xDA) {
      JREQ(sof, "scan before the frame header");
      JREQ(sl >= 1 && sl >= 1 + 2 * s[0] + 3, "truncated scan header");
      JREQ(s[0] == P.ncomp, "more than one scan (the first has %d of %d components)", s[0], P.ncomp);
      for (int c = 0; c < P.ncomp; ++c) {
        JREQ(s[1 + 2 * c] == ids[c], "scan component order differs from the frame");
        P.td[c] = s[2 + 2 * c] >> 4;
        P.ta[c] = s[2 + 2 * c] & 15;
        JREQ(P.td[c] < 4 && P.hdef[0][P.td[c]] && P.ta[c] < 4 && P.hdef[1][P.ta[c]],
             "scan references an undefined Huffman table");
        JREQ(P.qdef[P.tq[c]], "component references an undefined quantization table");
      }
      P.scan_start = (int)(i + 2 + ln);
      P.scan_len = (int)(n - 2 - P.scan_start);
      break;
    }
    i += 2 + ln;
  }
  if (P.ncomp == 3) {
    // jdapimin.c default_decompress_parms: a JFIF marker means YCbCr, else an Adobe marker's transform decides, else the ids
    JREQ(jfif || !(adobe && transform == 0), "Adobe transform 0 (RGB-coded) is not supported");
    JREQ(jfif || adobe || !(ids[0] == 'R' && ids[1] == 'G' && ids[2] == 'B'), "RGB-coded components are not supported");
  }
  JREQ((long long)P.H * P.W * 3 < (1ll << 31), "%dx%d is too large (H*W*3 must stay below 2^31)", P.H, P.W);
  return 0;
}

// jdhuff.c jpeg_make_d_derived_tbl, with its checks
static int derive(int di, const int* bits, const uint8_t* val, bool is_dc, Huff& h) {
  memset(&h, 0, sizeof(h));
  int code = 0, p = 0;
  int huffcode[257], huffsize[257];
  for (int l = 1; l <= 16; ++l)
    for (int i = 0; i < bits[l]; ++i) huffsize[p++] = l;
  huffsize[p] = 0;
  const int count = p;
  p = 0;
  int si = huffsize[0];
  while (huffsize[p]) {
    while (huffsize[p] == si) huffcode[p++] = code++;
    JREQ(code < (1 << si), "over-subscribed Huffman table");
    code <<= 1;
    ++si;
  }
  p = 0;
  for (int l = 1; l <= 16; ++l) {
    h.maxcode[l] = -1;
    if (bits[l]) {
      h.valoff[l] = p - huffcode[p];
      p += bits[l];
      h.maxcode[l] = huffcode[p - 1];
    }
  }
  for (int i = 0; i < count; ++i) {
    if (is_dc) JREQ(val[i] <= 15, "DC Huffman table with a symbol > 15");
    h.val[i] = val[i];
    if (huffsize[i] <= 9) {
      const int lo = huffcode[i] << (9 - huffsize[i]);
      for (int k = 0; k < (1 << (9 - huffsize[i])); ++k) h.lut[lo + k] = (uint16_t)(huffsize[i] << 8 | val[i]);
    }
  }
  return 0;
}

static long long a256(long long x) { return (x + 255) & ~255ll; }

struct Layout {               // a document's workspace regions
  long long stream, tiles, seg, win, exits, coef, planes, total;
};
static Layout layout(long long scan_len, long long nblocks, long long nseg, long long plane_bytes) {
  Layout L;
  const long long ntiles = (scan_len + kTile - 1) / kTile, nwin = std::max(1ll, (scan_len + kWin - 1) / kWin);
  L.stream = 0;
  L.tiles = L.stream + a256(scan_len + 16);
  L.seg = L.tiles + a256(8 * ntiles);
  L.win = L.seg + a256(4 * (nseg + 1));
  L.exits = L.win + a256((long long)sizeof(Win) * nwin);
  L.coef = L.exits + a256(2 * 8 * ((nwin + kChunk - 1) / kChunk));
  L.planes = L.coef + a256(128 * nblocks);
  L.total = L.planes + a256(plane_bytes) + 3 * 256;
  return L;
}

// An upper bound of the layouts of up to max_docs documents whose pixels and bytes sum to at most max_pixels and max_jpeg_bytes: a
// region of layout() takes at most its size plus 255 bytes, a document at most 3 (H + 15) (W + 15) / 64 blocks, and
// 15 (H + W) + 225 <= 40 sqrt(H W) + 256 for sides within about 1:5 (summed over documents, sqrt(max_docs * max_pixels) bounds it).
static size_t workspace_bytes(int max_docs, long long max_pixels, long long max_jpeg_bytes) {
  if (max_docs < 0 || max_pixels < 0 || max_jpeg_bytes < 0) return 0;
  const long long n = max_docs, J = max_jpeg_bytes;
  const long long area = max_pixels + 40 * (long long)ceil(sqrt((double)n * (double)max_pixels)) + 256 * n;
  const long long blocks = 3 * area / 64 + 3 * n;
  const long long per_doc = 16 + 8 + 4 * 2 + 32 + 16 * 2 + 10 * 255 + 3 * 256 + 64;
  return (size_t)(J + 8 * (J / kTile) + 32 * (J / kWin) + 16 * (J / (kWin * kChunk)) + (4 + 128 + 64) * blocks + n * per_doc);
}

static size_t table_bytes(int max_docs) {
  return max_docs < 0 || max_docs > kMaxDocs ? 0 : sizeof(Header) + (size_t)max_docs * sizeof(Doc);
}

static int plan(const dvd_jpeg_doc_t* in, int n, void* table_host, size_t tbytes, size_t wbytes, int32_t* out_hw) {
  DVD_REQUIRE(n >= 0 && n <= kMaxDocs && (n == 0 || in), "jpeg_plan: n_docs=%d, docs %p", n, (const void*)in);
  DVD_REQUIRE(!table_host || tbytes >= table_bytes(n), "jpeg_plan: table of %zu bytes is too small for %d documents (%zu needed)",
              tbytes, n, table_bytes(n));
  Header* hdr = static_cast<Header*>(table_host);
  Doc* docs = hdr ? reinterpret_cast<Doc*>(hdr + 1) : nullptr;
  long long ws = 0, tiles = 0, chunks = 0, idct = 0, pix = 0;
  Parsed P;
  for (int di = 0; di < n; ++di) {
    JREQ(in[di].file_host && in[di].bytes > 0, "null file pointer or empty file");
    if (parse(di, in[di].file_host, in[di].bytes, P)) return DVD_E_BADARG;
    Huff dc[3], ac[3];
    for (int c = 0; c < P.ncomp; ++c)
      if (derive(di, P.hbits[0][P.td[c]], P.hval[0][P.td[c]], true, dc[c]) || derive(di, P.hbits[1][P.ta[c]], P.hval[1][P.ta[c]], false, ac[c]))
        return DVD_E_BADARG;
    const bool swap = P.orient >= 5;
    if (out_hw) {
      out_hw[2 * di] = swap ? P.W : P.H;
      out_hw[2 * di + 1] = swap ? P.H : P.W;
    }
    if (!docs) continue;
    JREQ(in[di].file && in[di].out, "null device pointer (file %p, out %p)", (const void*)in[di].file, (void*)in[di].out);
    Doc& d = docs[di];
    memset(&d, 0, sizeof(d));
    d.scan = in[di].file + P.scan_start;
    d.out = in[di].out;
    d.scan_len = P.scan_len;
    d.H = P.H;
    d.W = P.W;
    d.Ho = swap ? P.W : P.H;
    d.Wo = swap ? P.H : P.W;
    d.orient = P.orient;
    d.ncomp = P.ncomp;
    d.mcux = cdiv(P.W, 8 * P.hmax);
    d.mcuy = cdiv(P.H, 8 * P.vmax);
    d.fh = P.hmax;
    d.fv = P.vmax;
    int bpm = 0;
    long long plane_bytes = 0;
    long long plane_off[3];
    for (int c = 0; c < P.ncomp; ++c) {
      d.h[c] = P.h[c];
      d.v[c] = P.v[c];
      for (int y = 0; y < P.v[c]; ++y)
        for (int x = 0; x < P.h[c]; ++x) {
          d.bcomp[bpm] = (int8_t)c;
          d.bdx[bpm] = (int8_t)x;
          d.bdy[bpm] = (int8_t)y;
          ++bpm;
        }
      d.pw[c] = d.mcux * P.h[c] * 8;
      d.dw[c] = cdiv((long long)P.W * P.h[c], P.hmax);
      d.dh[c] = cdiv((long long)P.H * P.v[c], P.vmax);
      plane_off[c] = plane_bytes;
      plane_bytes += a256((long long)d.pw[c] * d.mcuy * P.v[c] * 8);
      for (int k = 0; k < 64; ++k) d.quant[c][k] = P.quant[P.tq[c]][k];
      d.dc[c] = dc[c];
      d.ac[c] = ac[c];
    }
    d.bpm = bpm;
    const long long mcus = (long long)d.mcux * d.mcuy, nblocks = mcus * bpm;
    JREQ(nblocks < (1ll << 31) / 64, "too many blocks");
    d.nblocks = (int)nblocks;
    d.restart = P.restart;
    d.nseg = P.restart ? cdiv(mcus, P.restart) : 1;
    d.ntiles = cdiv(P.scan_len, kTile);
    d.nwin = std::max(1, cdiv(P.scan_len, kWin));
    d.nchunks = cdiv(d.nwin, kChunk);
    const Layout L = layout(P.scan_len, nblocks, d.nseg, plane_bytes);
    d.ws = ws;
    d.stream_off = (int32_t)L.stream;
    d.tiles_off = (int32_t)L.tiles;
    d.seg_off = (int32_t)L.seg;
    d.win_off = (int32_t)L.win;
    d.exit_off = (int32_t)L.exits;
    JREQ(L.total < (1ll << 31), "workspace of one document exceeds 2 GB");
    d.coef_off = (int32_t)L.coef;
    for (int c = 0; c < P.ncomp; ++c) d.plane_off[c] = (int32_t)(L.planes + plane_off[c]);
    d.tile_base = tiles;
    d.chunk_base = chunks;
    d.idct_base = idct;
    d.pix_base = pix;
    tiles += d.ntiles;
    chunks += d.nchunks;
    idct += cdiv(nblocks, kIdctBlocks);
    pix += (long long)cdiv(d.Wo, kPixW) * cdiv(d.Ho, kPixH);
    ws += L.total;
    DVD_REQUIRE((size_t)ws <= wbytes, "jpeg_plan: the batch needs more than the workspace's %zu bytes (documents 0..%d need %lld)",
                wbytes, di, ws);
  }
  if (hdr) {
    hdr->n_docs = n;
    hdr->pad = 0;
    hdr->tiles = tiles;
    hdr->chunks = chunks;
    hdr->idct_tasks = idct;
    hdr->pix_tasks = pix;
  }
  return 0;
}

template <typename K>
static int grid_of(K kernel, int threads, int& grid) {
  int dev = 0, n_sm = 0, per = 0;
  DVD_CUDA(cudaGetDevice(&dev));
  DVD_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  DVD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kernel, threads, 0));
  DVD_REQUIRE(per >= 1, "jpeg_decode: kernel does not fit an SM");
  grid = n_sm * per;
  return 0;
}

static int decode(const void* table, void* workspace, cudaStream_t st) {
  DVD_REQUIRE(table && workspace, "jpeg_decode: null pointer (table %p, workspace %p)", table, workspace);
  DVD_REQUIRE(((uintptr_t)workspace & 255) == 0, "jpeg_decode: workspace must be 256-byte aligned");
  const Header* hdr = static_cast<const Header*>(table);
  const Doc* docs = reinterpret_cast<const Doc*>(hdr + 1);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  static int g[9] = {};                     // grid of each kernel (the device's SM count times its occupancy)
  static int g_dev = -1;
  int dev = 0;
  DVD_CUDA(cudaGetDevice(&dev));
  if (g_dev != dev) {
    int rc;
    if ((rc = grid_of(k_jpeg_count, kTileThreads, g[0])) || (rc = grid_of(k_jpeg_compact, kTileThreads, g[2])) ||
        (rc = grid_of(k_jpeg_sync, kChunk, g[3])) || (rc = grid_of(k_jpeg_write, kChunk, g[5])) ||
        (rc = grid_of(k_jpeg_resync, kChunk, g[8])) ||
        (rc = grid_of(k_jpeg_idct, 8 * kIdctBlocks, g[6])) || (rc = grid_of(k_jpeg_color, kPixW * kPixH, g[7])))
      return rc;
    int n_sm = 0;
    DVD_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    g[1] = g[4] = n_sm;                     // one CTA per document
    g_dev = dev;
  }
  k_jpeg_count<<<g[0], kTileThreads, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_count");
  k_jpeg_offsets<<<g[1], 1024, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_offsets");
  k_jpeg_compact<<<g[2], kTileThreads, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_compact");
  k_jpeg_sync<<<g[3], kChunk, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_sync");
  k_jpeg_resync<<<g[8], kChunk, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_resync");
  k_jpeg_fix<<<g[4], kChunk, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_fix");
  k_jpeg_write<<<g[5], kChunk, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_write");
  k_jpeg_idct<<<g[6], 8 * kIdctBlocks, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_idct");
  k_jpeg_color<<<g[7], kPixW * kPixH, 0, st>>>(hdr, docs, ws);
  DVD_LAUNCH_CHECK("k_jpeg_color");
  return 0;
}

}  // namespace jpeg
}  // namespace dvd

extern "C" size_t dvd_jpeg_table_bytes(int max_docs) { return dvd::jpeg::table_bytes(max_docs); }
extern "C" size_t dvd_jpeg_workspace_bytes(int max_docs, long long max_pixels, long long max_jpeg_bytes) {
  return dvd::jpeg::workspace_bytes(max_docs, max_pixels, max_jpeg_bytes);
}
extern "C" int dvd_jpeg_plan(const dvd_jpeg_doc_t* docs_host, int n_docs, void* table_host, size_t table_bytes, size_t workspace_bytes,
                             int32_t* out_hw) {
  return dvd::jpeg::plan(docs_host, n_docs, table_host, table_bytes, workspace_bytes, out_hw);
}
extern "C" int dvd_jpeg_decode(const void* table, void* workspace, void* stream) {
  return dvd::jpeg::decode(table, workspace, (cudaStream_t)stream);
}
