// same_ingest.cu — interleaved multi-channel PCM -> the engine's planar input rows (include/same_engine.h,
// same_engine_submit_interleaved).
//
// One launch per submit.  A block takes a tile of tf frames x tc columns (tc a power of two <= 32, tf = kTile / tc) and
// moves it in three steps:
//   1. the tile's raw bytes -> shared memory, in the widest unit (16, 8, 4, 2 or 1 bytes) that the source address,
//      the frame pitch and the tile's row length allow: coalesced along frames, 16-byte loads for aligned input, and
//      still correct for any misaligned device pointer;
//   2. decode (`sa as f32` of the reference, receiver.rs:119-130: s24 and f32 exactly, s32 rounded to nearest even;
//      s16 stays int16) and transpose into per-column runs of shared memory, each run padded by 16 bytes so that the
//      16-byte stores of consecutive columns fall on distinct banks;
//   3. each mapped column's run -> its output row with 16-byte stores, coalesced along the row.
// Output rows start 16-byte aligned (the engine's pitch is a multiple of 8 samples), so a store never needs a narrower
// path; the samples from the end of the data up to the next multiple of 8 are written as 0.
//
// The receiver kernels are not changed: they read these rows exactly as they read a planar submit.  Reading the
// interleaved frames in place would be the lane-major layout DESIGN.md §5 rejected (each lane gathers its own column).
#include <cuda_runtime.h>
#include <stdint.h>

#include "same_internal.h"

namespace same_dev {

constexpr uint32_t kThreads = 256;
constexpr uint32_t kTile = 4096;      // samples per tile
constexpr uint32_t kMaxCols = 32;     // columns per tile

template <int Fmt> struct Fmt_;
template <> struct Fmt_<SAME_FMT_S16> {
  static constexpr uint32_t kIn = 2;
  using Out = int16_t;
  __device__ static Out decode(const uint8_t* p) { return *reinterpret_cast<const int16_t*>(p); }
};
template <> struct Fmt_<SAME_FMT_S24> {
  static constexpr uint32_t kIn = 3;
  using Out = float;
  __device__ static Out decode(const uint8_t* p) {
    const int v = (int)p[0] | ((int)p[1] << 8) | ((int)(int8_t)p[2] << 16);
    return __int2float_rn(v);   // |v| < 2^24: exact
  }
};
template <> struct Fmt_<SAME_FMT_S32> {
  static constexpr uint32_t kIn = 4;
  using Out = float;
  __device__ static Out decode(const uint8_t* p) { return __int2float_rn(*reinterpret_cast<const int*>(p)); }
};
template <> struct Fmt_<SAME_FMT_F32> {
  static constexpr uint32_t kIn = 4;
  using Out = float;
  __device__ static Out decode(const uint8_t* p) { return *reinterpret_cast<const float*>(p); }
};

struct IngestArgs {
  const uint8_t* src;        // column 0 of frame 0
  unsigned long long pitch;  // bytes from one frame to the next
  uint32_t n_cols, n_frames;
  uint32_t tc, tf;           // tile shape: tc columns (power of two <= kMaxCols) x tf = kTile / tc frames
  const int32_t* row;        // output row of each column, -1 = not mapped
  void* dst;
  unsigned long long dpitch; // samples from one output row to the next (a multiple of 8)
};

// `rows` rows of `len` bytes, `pitch` apart in global memory -> packed in shared memory, in units of V
template <class V>
__device__ __forceinline__ void load_units(uint8_t* raw, const uint8_t* __restrict__ src, unsigned long long pitch,
                                           uint32_t rows, uint32_t len) {
  const uint32_t per = len / (uint32_t)sizeof(V), n = rows * per;
#pragma unroll 4
  for (uint32_t i = threadIdx.x; i < n; i += kThreads) {
    const uint32_t r = i / per, j = i - r * per;
    reinterpret_cast<V*>(raw + r * len)[j] = reinterpret_cast<const V*>(src + r * pitch)[j];
  }
}

template <int Fmt>
__global__ void __launch_bounds__(kThreads) same_ingest_kernel(IngestArgs a) {
  using F = Fmt_<Fmt>;
  using Out = typename F::Out;
  constexpr uint32_t G = 16u / (uint32_t)sizeof(Out);   // samples per 16-byte store
  __shared__ __align__(16) uint8_t raw[kTile * 4];
  __shared__ __align__(16) uint8_t tr[kTile * 4 + kMaxCols * 16];
  const uint32_t tc = a.tc, tf = a.tf;
  const uint64_t f0 = (uint64_t)blockIdx.x * tf;
  const uint32_t nf = (uint32_t)min((uint64_t)tf, (uint64_t)a.n_frames - f0);
  const uint32_t groups = (nf + G - 1u) / G;
  const uint32_t n_ct = (a.n_cols + tc - 1u) / tc;
  for (uint32_t ct = blockIdx.y; ct < n_ct; ct += gridDim.y) {
    const uint32_t c0 = ct * tc, nc = min(tc, a.n_cols - c0);
    const uint32_t rowbytes = nc * F::kIn;
    const uint8_t* base = a.src + f0 * a.pitch + (uint64_t)c0 * F::kIn;
    __syncthreads();   // the previous column tile's shared memory is no longer read
    {
      // whole frames are one contiguous run of bytes
      uint32_t rows = nf, len = rowbytes;
      unsigned long long pitch = a.pitch;
      if (pitch == rowbytes) { rows = 1; len = nf * rowbytes; }
      const unsigned long long align = (unsigned long long)(uintptr_t)base | (rows > 1 ? pitch : 0ull) | len;
      if ((align & 15u) == 0) load_units<uint4>(raw, base, pitch, rows, len);
      else if ((align & 7u) == 0) load_units<uint2>(raw, base, pitch, rows, len);
      else if ((align & 3u) == 0) load_units<uint32_t>(raw, base, pitch, rows, len);
      else if ((align & 1u) == 0) load_units<uint16_t>(raw, base, pitch, rows, len);
      else load_units<uint8_t>(raw, base, pitch, rows, len);
    }
    __syncthreads();
    // decode and transpose: column c's run starts at c * (tf + G) samples, 16-byte aligned
    for (uint32_t i = threadIdx.x; i < tc * groups; i += kThreads) {
      const uint32_t c = i & (tc - 1u), g = i / tc;
      if (c >= nc) continue;
      union { uint4 u; Out v[G]; } pk;
#pragma unroll
      for (uint32_t k = 0; k < G; ++k) {
        const uint32_t f = g * G + k;
        pk.v[k] = f < nf ? F::decode(raw + f * rowbytes + c * F::kIn) : Out(0);
      }
      *reinterpret_cast<uint4*>(tr + (c * (tf + G) + g * G) * sizeof(Out)) = pk.u;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < nc * groups; i += kThreads) {
      const uint32_t c = i / groups, g = i - c * groups;
      const int32_t r = __ldg(a.row + c0 + c);
      if (r < 0) continue;
      const uint4 v = *reinterpret_cast<const uint4*>(tr + (c * (tf + G) + g * G) * sizeof(Out));
      *reinterpret_cast<uint4*>(static_cast<Out*>(a.dst) + (uint64_t)r * a.dpitch + f0 + g * G) = v;
    }
  }
}

}  // namespace same_dev

extern "C" cudaError_t same_launch_ingest(uint32_t format, const void* src, uint64_t frame_pitch_bytes, uint32_t n_cols,
                                          uint32_t n_frames, const int32_t* d_row, void* dst, uint64_t dpitch,
                                          cudaStream_t stream) {
  if (n_cols == 0 || n_frames == 0) return cudaSuccess;
  using namespace same_dev;
  IngestArgs a;
  a.src = static_cast<const uint8_t*>(src); a.pitch = frame_pitch_bytes;
  a.n_cols = n_cols; a.n_frames = n_frames;
  a.tc = 1;
  while (a.tc < n_cols && a.tc < kMaxCols) a.tc <<= 1;
  a.tf = kTile / a.tc;
  a.row = d_row; a.dst = dst; a.dpitch = dpitch;
  const uint32_t col_tiles = (n_cols + a.tc - 1u) / a.tc;
  const dim3 grid((n_frames + a.tf - 1u) / a.tf, col_tiles < 65535u ? col_tiles : 65535u);
  switch (format) {
    case SAME_FMT_S16: same_ingest_kernel<SAME_FMT_S16><<<grid, kThreads, 0, stream>>>(a); break;
    case SAME_FMT_S24: same_ingest_kernel<SAME_FMT_S24><<<grid, kThreads, 0, stream>>>(a); break;
    case SAME_FMT_S32: same_ingest_kernel<SAME_FMT_S32><<<grid, kThreads, 0, stream>>>(a); break;
    case SAME_FMT_F32: same_ingest_kernel<SAME_FMT_F32><<<grid, kThreads, 0, stream>>>(a); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}
