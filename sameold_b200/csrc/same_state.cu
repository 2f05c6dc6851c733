// same_state.cu — device side of the portable stream-state records (include/same_engine.h, "Portable stream state").
//
// A record is one stream's complete receiver state: the n_words state words (word order, independent of n_pad) and
// the raw StreamBlob, framed by the source stream id, a flags word and a CRC-32 (zlib polynomial).  Three kernels:
//   gather    state32 (structure of arrays) + blobs -> records in a device staging buffer, CRC included
//   validate  CRC + range check of every field the receiver kernels use as an index or a length
//   scatter   records -> state32 + blobs (launched only after every record of the batch passed validation)
// Word rows are moved through shared memory 32 streams x 32 words at a time: for a contiguous id run each row of a
// tile is one 128-byte line of state32; for an arbitrary id list the same code gathers stream by stream.
#include <cuda_runtime.h>

#include "same_params.h"

namespace same_state {

constexpr uint32_t kCrcPoly = 0xEDB88320u;   // zlib, reflected

// Record geometry (bytes): id, flags, words, zero pad to 16 | blob, zero pad | CRC in the last 4 bytes
struct RecGeom {
  uint32_t words_off, blob_off, crc_off, bytes;
};

__host__ __device__ inline RecGeom rec_geom(uint32_t n_words) {
  RecGeom g;
  g.words_off = 8u;
  g.blob_off = (8u + 4u * n_words + 15u) & ~15u;
  g.crc_off = g.blob_off + (((uint32_t)sizeof(StreamBlob) + 4u + 15u) & ~15u) - 4u;
  g.bytes = g.crc_off + 4u;
  return g;
}

// a * b modulo the CRC polynomial, reflected representation (as zlib's multmodp)
__host__ __device__ inline uint32_t multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1u)) == 0) break;
    }
    m >>= 1;
    b = (b & 1u) ? (b >> 1) ^ kCrcPoly : b >> 1;
  }
  return p;
}

// x^(8 * nbytes) modulo the polynomial: the operator that runs a CRC register through nbytes zero bytes
inline uint32_t x8nmodp(uint64_t nbytes) {
  uint32_t p = 1u << 31;          // x^0
  uint32_t sq = 1u << 30;         // x^1, squared below to x^(2^k)
  uint64_t n = nbytes * 8u;
  while (n) {
    if (n & 1u) p = multmodp(sq, p);
    sq = multmodp(sq, sq);
    n >>= 1;
  }
  return p;
}

// The warp-parallel CRC of one record: lane i runs a zero-initialised register over words [i*k, min((i+1)*k, w)) of
// the record; shifting each lane's register past the bytes after its slice and XOR-ing gives the register of the
// whole record, to which the zlib initial value 0xFFFFFFFF (shifted past all bytes) is added.
struct CrcPlan {
  uint32_t k, w;        // words per lane, words covered (crc_off / 4)
  uint32_t op[32];      // per lane: x^(8 * bytes after the lane's slice)
  uint32_t init;        // multmodp(x^(8 * crc_off), 0xFFFFFFFF)
};

CrcPlan make_plan(uint32_t n_words) {
  const RecGeom g = rec_geom(n_words);
  CrcPlan c;
  c.w = g.crc_off / 4u;
  c.k = (c.w + 31u) / 32u;
  for (uint32_t i = 0; i < 32; ++i) {
    const uint32_t end = min((i + 1u) * c.k, c.w);
    c.op[i] = x8nmodp((uint64_t)4u * (c.w - end));
  }
  c.init = multmodp(x8nmodp(g.crc_off), 0xFFFFFFFFu);
  return c;
}

// slicing-by-4 tables, built per block into shared memory
__device__ inline void build_tables(uint32_t (*t)[256]) {
  for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ kCrcPoly : c >> 1;
    t[0][i] = c;
  }
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) {
    uint32_t c = t[0][i];
    c = (c >> 8) ^ t[0][c & 0xffu]; t[1][i] = c;
    c = (c >> 8) ^ t[0][c & 0xffu]; t[2][i] = c;
    c = (c >> 8) ^ t[0][c & 0xffu]; t[3][i] = c;
  }
  __syncthreads();
}

// CRC-32 of rec[0 .. crc_off), computed by the whole warp; every lane returns it
__device__ inline uint32_t warp_crc(const uint8_t* rec, const CrcPlan& c, const uint32_t (*t)[256]) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(rec);
  const uint32_t b = min(lane * c.k, c.w), e = min(b + c.k, c.w);
  uint32_t r = 0;
  for (uint32_t i = b; i < e; ++i) {
    r ^= w[i];
    r = t[3][r & 0xffu] ^ t[2][(r >> 8) & 0xffu] ^ t[1][(r >> 16) & 0xffu] ^ t[0][r >> 24];
  }
  uint32_t v = (b < e) ? multmodp(c.op[lane], r) : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v ^= __shfl_xor_sync(0xffffffffu, v, o);
  return ~(v ^ c.init);
}

// Blob copy by one warp: 16-byte vectors when both sides are 16-byte aligned, else 8-byte vectors (a StreamBlob is
// 8 mod 16 bytes long, so every other blob in the engine's array starts 8 bytes off a 16-byte boundary)
__device__ inline void warp_copy_blob(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src) {
  const uint32_t lane = threadIdx.x & 31u;
  constexpr uint32_t kBytes = (uint32_t)sizeof(StreamBlob);
  static_assert(kBytes % 8u == 0u, "StreamBlob is a whole number of 8-byte words");
  if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15u) == 0u) {
    constexpr uint32_t n16 = kBytes / 16u;
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    for (uint32_t i = lane; i < n16; i += 32u) d[i] = s[i];
    if (kBytes % 16u && lane == 0)
      *reinterpret_cast<uint2*>(dst + 16u * n16) = *reinterpret_cast<const uint2*>(src + 16u * n16);
  } else {
    const uint2* s = reinterpret_cast<const uint2*>(src);
    uint2* d = reinterpret_cast<uint2*>(dst);
    for (uint32_t i = lane; i < kBytes / 8u; i += 32u) d[i] = s[i];
  }
}

constexpr uint32_t kTileWords = 32;
constexpr uint32_t kThreads = 256;   // 8 warps per 32-stream tile

__device__ inline uint32_t stream_of(const uint32_t* ids, uint32_t first, uint32_t r) { return ids ? ids[r] : first + r; }

__global__ void __launch_bounds__(kThreads) gather_kernel(const __grid_constant__ SameParams p, const uint32_t* __restrict__ ids,
                                                          uint32_t first, uint32_t n, uint32_t id_base, uint32_t rec_flags,
                                                          uint8_t* __restrict__ out, const __grid_constant__ CrcPlan plan) {
  __shared__ uint32_t tile[kTileWords][33];
  __shared__ uint32_t tbl[4][256];
  build_tables(tbl);
  const SameLayout& L = p.layout;
  const RecGeom g = rec_geom(L.n_words);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t r0 = blockIdx.x * 32u;
  const uint32_t nr = min(32u, n - r0);
  const uint32_t my_s = lane < nr ? stream_of(ids, first, r0 + lane) : 0u;
  for (uint32_t w0 = 0; w0 < L.n_words; w0 += kTileWords) {
    // rows: word w0+wi of the tile's 32 streams (one 128-byte line for a contiguous run)
    for (uint32_t wi = warp; wi < kTileWords; wi += kThreads / 32u)
      if (w0 + wi < L.n_words && lane < nr) tile[wi][lane] = p.state32[(size_t)(w0 + wi) * L.n_pad + my_s];
    __syncthreads();
    // columns: 32 consecutive words of one record
    for (uint32_t r = warp; r < nr; r += kThreads / 32u)
      if (w0 + lane < L.n_words)
        reinterpret_cast<uint32_t*>(out + (size_t)(r0 + r) * g.bytes + g.words_off)[w0 + lane] = tile[lane][r];
    __syncthreads();
  }
  for (uint32_t r = warp; r < nr; r += kThreads / 32u) {
    uint8_t* rec = out + (size_t)(r0 + r) * g.bytes;
    const uint32_t s = stream_of(ids, first, r0 + r);
    if (lane == 0) {
      reinterpret_cast<uint32_t*>(rec)[0] = s + id_base;
      reinterpret_cast<uint32_t*>(rec)[1] = rec_flags;
    }
    for (uint32_t o = g.words_off + 4u * L.n_words + 4u * lane; o < g.blob_off; o += 128u) *reinterpret_cast<uint32_t*>(rec + o) = 0u;
    for (uint32_t o = g.blob_off + (uint32_t)sizeof(StreamBlob) + 4u * lane; o < g.crc_off; o += 128u) *reinterpret_cast<uint32_t*>(rec + o) = 0u;
    warp_copy_blob(rec + g.blob_off, reinterpret_cast<const uint8_t*>(p.blobs + s));
  }
  __syncthreads();   // the block's record bytes are visible to all of its warps
  for (uint32_t r = warp; r < nr; r += kThreads / 32u) {
    uint8_t* rec = out + (size_t)(r0 + r) * g.bytes;
    const uint32_t crc = warp_crc(rec, plan, tbl);
    if (lane == 0) *reinterpret_cast<uint32_t*>(rec + g.crc_off) = crc;
  }
}

// Failure codes of validate (0 = valid); the host names them (same_engine.cu: state_check_name)
enum Check : uint32_t {
  CK_OK = 0, CK_CRC, CK_REC_FLAGS, CK_FLAGS, CK_FRAMER, CK_TRANSPORT, CK_CLOCK, CK_TEDCNT, CK_BYTECLK, CK_SQ_HEAD,
  CK_HIST_N, CK_HIST_LEN, CK_PENDING_LEN, CK_PENDING_KIND, CK_PENDING_ERR, CK_PENDING_OFFSET, CK_PREV_LEN
};

// Every field a receiver kernel uses as an index, a length or a loop bound (same_lane.cuh, same_transport.cuh,
// same_kernels.cu), checked against the range the kernels can produce themselves
__device__ inline uint32_t check_record(const uint8_t* rec, const RecGeom& g) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(rec + g.words_off);
  const StreamBlob* b = reinterpret_cast<const StreamBlob*>(rec + g.blob_off);
  if (reinterpret_cast<const uint32_t*>(rec)[1] & ~1u) return CK_REC_FLAGS;
  const uint32_t flags = w[F_FLAGS];
  const uint32_t known = FLAG_AGC_LOCKED | FLAG_SQ_LOCK | FLAG_BW_LOCKED | FLAG_EQ_TRAINING | FLAG_FORCE_EOM |
                         FLAG_PENDING | FLAG_HAVE_PREV | (3u << FLAG_FR_SHIFT) | (3u << FLAG_LINK_SHIFT) | (3u << FLAG_TR_SHIFT);
  if (flags & ~known) return CK_FLAGS;
  if (((flags >> FLAG_FR_SHIFT) & 3u) > 2u) return CK_FRAMER;                     // Framer state: Idle/PrefixSearch/DataRead
  if (((flags >> FLAG_TR_SHIFT) & 3u) > 2u) return CK_TRANSPORT;                  // Idle/Assembling/Message
  if (w[F_CLOCK] > (1u << 22)) return CK_CLOCK;                                    // fire_clock: next = clock + 1 must not overflow
  if (w[F_TEDCNT] > 1u) return CK_TEDCNT;
  if ((int)w[F_SQ_BYTECLK] < -1 || (int)w[F_SQ_BYTECLK] > 7) return CK_BYTECLK;
  if (w[F_SQ_HEAD] >= SAME_SQ_HIST) return CK_SQ_HEAD;                             // ring slot of sqh
  if (w[F_HIST_N] > 3u) return CK_HIST_N;                                          // b->hist[hist_n] after pruning
  for (int k = 0; k < 3; ++k)
    if (b->hist[k].len > SAME_MAX_MESSAGE_LENGTH) return CK_HIST_LEN;              // copy_words / combine bounds
  if (b->pending_len > SAME_MAX_MESSAGE_LENGTH) return CK_PENDING_LEN;             // pending_text -> event payload, prev_text
  if (b->pending_kind > 2u) return CK_PENDING_KIND;
  if (b->pending_err > 3u) return CK_PENDING_ERR;
  if (b->pending_offset > b->pending_len) return CK_PENDING_OFFSET;
  if (b->prev_len > SAME_MAX_MESSAGE_LENGTH) return CK_PREV_LEN;
  return CK_OK;
}

// result[0] (u64): min over failing records of (index << 32 | code), ~0 if none; result[1] low word: OR of record flags
__global__ void __launch_bounds__(kThreads) validate_kernel(const uint8_t* __restrict__ in, uint32_t n, uint32_t n_words,
                                                            unsigned long long* __restrict__ result,
                                                            const __grid_constant__ CrcPlan plan) {
  __shared__ uint32_t tbl[4][256];
  build_tables(tbl);
  const RecGeom g = rec_geom(n_words);
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t r = blockIdx.x * (kThreads / 32u) + (threadIdx.x >> 5);
  if (r >= n) return;
  const uint8_t* rec = in + (size_t)r * g.bytes;
  const uint32_t crc = warp_crc(rec, plan, tbl);
  if (lane != 0) return;
  uint32_t code = crc != *reinterpret_cast<const uint32_t*>(rec + g.crc_off) ? (uint32_t)CK_CRC : check_record(rec, g);
  if (code != CK_OK) atomicMin(&result[0], ((unsigned long long)r << 32) | code);
  const uint32_t rf = reinterpret_cast<const uint32_t*>(rec)[1];
  if (rf) atomicOr(&result[1], (unsigned long long)rf);
}

__global__ void __launch_bounds__(kThreads) scatter_kernel(const __grid_constant__ SameParams p, const uint32_t* __restrict__ ids,
                                                           uint32_t first, uint32_t n, const uint8_t* __restrict__ in) {
  __shared__ uint32_t tile[kTileWords][33];
  const SameLayout& L = p.layout;
  const RecGeom g = rec_geom(L.n_words);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t r0 = blockIdx.x * 32u;
  const uint32_t nr = min(32u, n - r0);
  const uint32_t my_s = lane < nr ? stream_of(ids, first, r0 + lane) : 0u;
  for (uint32_t w0 = 0; w0 < L.n_words; w0 += kTileWords) {
    for (uint32_t r = warp; r < nr; r += kThreads / 32u)
      if (w0 + lane < L.n_words)
        tile[lane][r] = reinterpret_cast<const uint32_t*>(in + (size_t)(r0 + r) * g.bytes + g.words_off)[w0 + lane];
    __syncthreads();
    for (uint32_t wi = warp; wi < kTileWords; wi += kThreads / 32u) {
      const uint32_t w = w0 + wi;
      if (w < L.n_words && lane < nr) p.state32[(size_t)w * L.n_pad + my_s] = (w == F_TRACE_N) ? 0u : tile[wi][lane];
    }
    __syncthreads();
  }
  for (uint32_t r = warp; r < nr; r += kThreads / 32u)
    warp_copy_blob(reinterpret_cast<uint8_t*>(p.blobs + stream_of(ids, first, r0 + r)), in + (size_t)(r0 + r) * g.bytes + g.blob_off);
}

// host CRC-32 (zlib) for the export header
uint32_t crc32_host(const uint8_t* d, size_t n) {
  static uint32_t t[256];
  static bool init = false;
  if (!init) {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ kCrcPoly : c >> 1;
      t[i] = c;
    }
    init = true;
  }
  uint32_t c = 0xFFFFFFFFu;
  for (size_t i = 0; i < n; ++i) c = t[(c ^ d[i]) & 0xffu] ^ (c >> 8);
  return ~c;
}

}  // namespace same_state

extern "C" uint32_t same_state_record_bytes(uint32_t n_words) { return same_state::rec_geom(n_words).bytes; }

extern "C" uint32_t same_state_crc32(const void* data, size_t n) {
  return same_state::crc32_host(static_cast<const uint8_t*>(data), n);
}

// ids == nullptr: the contiguous run first .. first+n-1
extern "C" cudaError_t same_state_launch_gather(const SameParams* p, const uint32_t* d_ids, uint32_t first, uint32_t n,
                                                uint32_t id_base, uint32_t rec_flags, uint8_t* d_out, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const same_state::CrcPlan plan = same_state::make_plan(p->layout.n_words);
  same_state::gather_kernel<<<(n + 31u) / 32u, same_state::kThreads, 0, stream>>>(*p, d_ids, first, n, id_base, rec_flags, d_out, plan);
  return cudaGetLastError();
}

extern "C" cudaError_t same_state_launch_validate(const uint8_t* d_in, uint32_t n, uint32_t n_words, unsigned long long* d_result,
                                                  cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const same_state::CrcPlan plan = same_state::make_plan(n_words);
  const uint32_t per = same_state::kThreads / 32u;
  same_state::validate_kernel<<<(n + per - 1u) / per, same_state::kThreads, 0, stream>>>(d_in, n, n_words, d_result, plan);
  return cudaGetLastError();
}

extern "C" cudaError_t same_state_launch_scatter(const SameParams* p, const uint32_t* d_ids, uint32_t first, uint32_t n,
                                                 const uint8_t* d_in, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  same_state::scatter_kernel<<<(n + 31u) / 32u, same_state::kThreads, 0, stream>>>(*p, d_ids, first, n, d_in);
  return cudaGetLastError();
}
