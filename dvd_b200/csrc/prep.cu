// Input preparation: the denoiser's 512x512 conditioning image y512 from the uint8 photo, on the GPU.
//
// The reference loader computes y512 = cv2.resize(photo, (512, 512), INTER_LINEAR) / 255 on the host.  k_y512_u8 computes the same
// bytes with OpenCV's fixed-point arithmetic (11-bit coefficients, an int32 horizontal pass, the SIMD form of the vertical pass) and
// writes fp32 NCHW, so the caller uploads only the photo.  The restatement is oracle/resize512.py.
//
// One persistent launch serves a batch of photos of any sizes: the host plans a small table (dvd_y512_u8_plan), the caller uploads it,
// and the grid depends only on the device, so a CUDA graph captured once serves every batch planned into the same device table.
#include "common.cuh"

namespace dvd {

static constexpr int kOut = 512;                 // output side
static constexpr int kThreads = 256;             // a thread owns output columns tid and tid + 256 of every row of its tasks
static constexpr int kBand = 2;                  // output rows per task: 256 tasks per document
static constexpr int kTasksPerDoc = kOut / kBand;
static constexpr int kMaxDocs = 1 << 22;         // task indices stay inside int32

struct PrepHeader {
  int32_t n_docs, pad[3];
};
struct PrepDoc {                          // 32 bytes
  const uint8_t* photo;                   // [H,W,3] uint8
  double scale_x, scale_y;                // 1.0 / (512.0 / W), 1.0 / (512.0 / H): OpenCV's form, computed on the host
  int32_t H, W;
};
static_assert(sizeof(PrepHeader) == 16 && sizeof(PrepDoc) == 32, "y512 table layout");

// OpenCV's source index and fractional offset of output index i: f = float((i + 0.5) * scale - 0.5), s = floor(f), f -= s.  The
// product and the sum are exact for a 512-long target (scale = n / 512), so the explicit roundings only keep the compiler from
// contracting them into an FMA of another rounding.
static __device__ __forceinline__ int src_index(int i, double scale, float& f) {
  f = __double2float_rn(__dadd_rn(__dmul_rn((double)i + 0.5, scale), -0.5));
  const float s = floorf(f);
  f -= s;
  return (int)s;
}
// 11-bit fixed-point weights: saturate_cast<short>(w * 2048) rounds half to even
static __device__ __forceinline__ int coef(float w) { return __float2int_rn(w * 2048.f); }

__global__ void __launch_bounds__(kThreads) k_y512_u8(const PrepHeader* __restrict__ hdr, const PrepDoc* __restrict__ docs,
                                                      float* __restrict__ y512) {
  const int total = __ldg(&hdr->n_docs) * kTasksPerDoc;
  for (int t = blockIdx.x; t < total; t += gridDim.x) {
    const int d = t / kTasksPerDoc, dy0 = (t - d * kTasksPerDoc) * kBand;
    const uint8_t* __restrict__ photo = (const uint8_t*)__ldg((const unsigned long long*)&docs[d].photo);
    const int H = __ldg(&docs[d].H), W = __ldg(&docs[d].W);
    const double sx_scale = __ldg(&docs[d].scale_x), sy_scale = __ldg(&docs[d].scale_y);

    // x taps of this thread's two columns: the column index is clamped together with its weight (OpenCV's xmin / xmax ranges)
    int xo0[2], xo1[2], a0[2], a1[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      float fx;
      int sx = src_index(threadIdx.x + k * kThreads, sx_scale, fx);
      if (sx < 0) { sx = 0; fx = 0.f; }
      if (sx >= W - 1) { sx = W - 1; fx = 0.f; }
      xo0[k] = sx * 3;
      xo1[k] = min(sx + 1, W - 1) * 3;
      a0[k] = coef(1.f - fx);
      a1[k] = coef(fx);
    }
    // y taps: the weight keeps its fraction, only the two row indices are clamped
    const uint8_t* r0[kBand];
    const uint8_t* r1[kBand];
    int b0[kBand], b1[kBand];
#pragma unroll
    for (int j = 0; j < kBand; ++j) {
      float fy;
      const int sy = src_index(dy0 + j, sy_scale, fy);
      r0[j] = photo + (size_t)min(max(sy, 0), H - 1) * W * 3;
      r1[j] = photo + (size_t)min(max(sy + 1, 0), H - 1) * W * 3;
      b0[j] = coef(1.f - fy);
      b1[j] = coef(fy);
    }
    // all 48 byte loads of the task are independent; issue them before any arithmetic
    int p[kBand][2][2][2][3];             // [row][column][tap row][tap column][channel]
#pragma unroll
    for (int j = 0; j < kBand; ++j)
#pragma unroll
      for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          p[j][k][0][0][c] = __ldg(r0[j] + xo0[k] + c);
          p[j][k][0][1][c] = __ldg(r0[j] + xo1[k] + c);
          p[j][k][1][0][c] = __ldg(r1[j] + xo0[k] + c);
          p[j][k][1][1][c] = __ldg(r1[j] + xo1[k] + c);
        }
    float* __restrict__ out = y512 + (size_t)d * 3 * kOut * kOut;
#pragma unroll
    for (int j = 0; j < kBand; ++j)
#pragma unroll
      for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int h0 = p[j][k][0][0][c] * a0[k] + p[j][k][0][1][c] * a1[k];
          const int h1 = p[j][k][1][0][c] * a0[k] + p[j][k][1][1][c] * a1[k];
          // VResizeLinearVec_32s8u: 16-bit high products of (h >> 4) with the row weights, +2, >> 2
          const int v = min(max((((b0[j] * (h0 >> 4)) >> 16) + ((b1[j] * (h1 >> 4)) >> 16) + 2) >> 2, 0), 255);
          out[((size_t)c * kOut + dy0 + j) * kOut + threadIdx.x + k * kThreads] = __fdiv_rn((float)v, 255.f);
        }
  }
}

static size_t table_bytes(int max_docs) { return max_docs < 0 ? 0 : sizeof(PrepHeader) + (size_t)max_docs * sizeof(PrepDoc); }

static int plan(const dvd_y512_doc_t* docs_host, int n_docs, void* table_host, size_t bytes) {
  DVD_REQUIRE(n_docs >= 0 && n_docs <= kMaxDocs && (n_docs == 0 || docs_host) && table_host,
              "y512_u8_plan: n_docs=%d, docs %p, table %p", n_docs, (const void*)docs_host, table_host);
  DVD_REQUIRE(bytes >= table_bytes(n_docs), "y512_u8_plan: table of %zu bytes is too small for %d documents (%zu needed)", bytes,
              n_docs, table_bytes(n_docs));
  PrepHeader* hdr = static_cast<PrepHeader*>(table_host);
  PrepDoc* recs = reinterpret_cast<PrepDoc*>(hdr + 1);
  for (int d = 0; d < n_docs; ++d) {
    const dvd_y512_doc_t& in = docs_host[d];
    DVD_REQUIRE(in.H >= 1 && in.W >= 1, "y512_u8_plan: document %d has size %dx%d (at least 1x1)", d, in.H, in.W);
    DVD_REQUIRE((long long)in.H * in.W * 3 < (1ll << 31), "y512_u8_plan: document %d (%dx%dx3) is too large for 32-bit offsets", d,
                in.H, in.W);
    DVD_REQUIRE(in.photo, "y512_u8_plan: document %d has a null photo pointer", d);
    recs[d] = PrepDoc{in.photo, 1.0 / ((double)kOut / in.W), 1.0 / ((double)kOut / in.H), in.H, in.W};
  }
  *hdr = PrepHeader{n_docs, {0, 0, 0}};
  return 0;
}

static int launch(const void* table, float* y512, cudaStream_t st) {
  DVD_REQUIRE(table && y512, "y512_u8: null pointer");
  const PrepHeader* hdr = static_cast<const PrepHeader*>(table);
  int dev = 0, n_sm = 0;
  DVD_CUDA(cudaGetDevice(&dev));
  DVD_REQUIRE(dev < 64, "y512_u8: device %d", dev);
  DVD_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  static int per_sm[64] = {};             // per device: occupancy of the kernel
  if (!per_sm[dev]) {
    DVD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[dev], k_y512_u8, kThreads, 0));
    DVD_REQUIRE(per_sm[dev] >= 1, "y512_u8: kernel does not fit an SM");
  }
  k_y512_u8<<<n_sm * per_sm[dev], kThreads, 0, st>>>(hdr, reinterpret_cast<const PrepDoc*>(hdr + 1), y512);
  DVD_LAUNCH_CHECK("k_y512_u8");
  return 0;
}

}  // namespace dvd

extern "C" size_t dvd_y512_table_bytes(int max_docs) { return dvd::table_bytes(max_docs); }
extern "C" int dvd_y512_u8_plan(const dvd_y512_doc_t* docs_host, int n_docs, void* table_host, size_t table_bytes) {
  return dvd::plan(docs_host, n_docs, table_host, table_bytes);
}
extern "C" int dvd_y512_u8(const void* table, float* y512, void* stream) { return dvd::launch(table, y512, (cudaStream_t)stream); }
