// same_state.cu — device side of the portable stream-state records (include/same_engine.h, "Portable stream state").
//
// A record is one stream's complete receiver state: the n_words state words (word order, independent of n_pad) and
// the raw StreamBlob, framed by the source stream id, a flags word and a CRC-32 (zlib polynomial).  Three kernels:
//   gather    state32 (structure of arrays) + blobs -> records in a device staging buffer, CRC included
//   validate  CRC + range check of every field the receiver kernels use as an index or a length
//   scatter   records -> state32 + blobs (launched only after every record of the batch passed validation)
// Word rows are moved through shared memory 32 streams x 32 words at a time: for a contiguous id run each row of a
// tile is one 128-byte line of state32; for an arbitrary id list the same code gathers stream by stream.
// The host half of the format, the header that names the configuration a state was produced under, is here too.
#include <cuda_runtime.h>

#include <cstring>
#include <string>

#include "same_internal.h"

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

// Failure codes of validate (0 = valid), and their text in the same order
enum Check : uint32_t {
  CK_OK = 0, CK_CRC, CK_REC_FLAGS, CK_FLAGS, CK_FRAMER, CK_TRANSPORT, CK_CLOCK, CK_TEDCNT, CK_BYTECLK, CK_SQ_HEAD,
  CK_HIST_N, CK_HIST_LEN, CK_PENDING_LEN, CK_PENDING_KIND, CK_PENDING_ERR, CK_PENDING_OFFSET, CK_PREV_LEN, CK_COUNT
};
const char* const kCheckNames[] = {
    "valid", "CRC mismatch", "record flags (only bit 0 is defined)", "F_FLAGS (undefined bits)", "framer state > 2",
    "transport state > 2", "F_CLOCK > 2^22", "F_TEDCNT not in {0, 1}", "F_SQ_BYTECLK not in -1..7", "F_SQ_HEAD >= 64",
    "F_HIST_N > 3", "burst history length > 268", "pending length > 268", "pending kind > 2", "pending error > 3",
    "pending_offset beyond the pending text", "previous-message length > 268"};
static_assert(sizeof kCheckNames / sizeof kCheckNames[0] == CK_COUNT, "one text per Check code");

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

// ---- header (host) ----

struct CrcTable { uint32_t t[256]; };

CrcTable make_crc_table() {
  CrcTable tbl;
  for (uint32_t i = 0; i < 256; ++i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ kCrcPoly : c >> 1;
    tbl.t[i] = c;
  }
  return tbl;
}

// host CRC-32 (zlib) for the header
uint32_t crc32_host(const uint8_t* d, size_t n) {
  static const CrcTable tbl = make_crc_table();   // initialised once, thread-safe
  uint32_t c = 0xFFFFFFFFu;
  for (size_t i = 0; i < n; ++i) c = tbl.t[(c ^ d[i]) & 0xffu] ^ (c >> 8);
  return ~c;
}

constexpr uint32_t kStMagic = 0x54534D53u;   // "SMST"
constexpr uint32_t kStVersion = 1u;
constexpr uint32_t kStBom = 0x01020304u;
// Offsets of the sections after the derived constants follow the tap entries per section T = tap_slots(ntaps):
// mark taps at 164, space taps at 164 + 8 T, 8 zero bytes, CRC at 164 + 16 T + 8 (2220 for T = 128)
constexpr size_t kStOffConfig = 40, kStOffDerived = 116, kStOffMark = 164;
constexpr size_t off_crc(uint32_t slots) { return kStOffMark + 16 * (size_t)slots + 8; }
static_assert(sizeof(same_config) == 19 * 4 && sizeof(same_derived) == 12 * 4, "4-byte fields only");
static_assert(kStOffDerived == kStOffConfig + sizeof(same_config) && kStOffMark == kStOffDerived + sizeof(same_derived) &&
              off_crc(kMinTapSlots) + 4 == kHeaderBytes, "header layout");

void put32(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }
uint32_t get32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
// a struct of 4-byte fields <-> little-endian words
void put_words(uint8_t* p, const void* src, size_t bytes) {
  for (size_t i = 0; i < bytes; i += 4) { uint32_t v; memcpy(&v, static_cast<const uint8_t*>(src) + i, 4); put32(p + i, v); }
}
void get_words(void* dst, const uint8_t* p, size_t bytes) {
  for (size_t i = 0; i < bytes; i += 4) { const uint32_t v = get32(p + i); memcpy(static_cast<uint8_t*>(dst) + i, &v, 4); }
}

const char* const kConfigFields[19] = {
    "input_rate", "dc_blocker_len", "agc_bandwidth", "agc_gain_min", "agc_gain_max", "timing_bw_unlocked",
    "timing_bw_locked", "timing_max_deviation", "squelch_power_open", "squelch_power_close", "squelch_bandwidth",
    "preamble_max_errors", "eq_enabled", "eq_nff", "eq_nfb", "eq_relaxation", "eq_regularization",
    "frame_prefix_max_errors", "frame_max_invalid_bytes"};
const char* const kDerivedFields[12] = {"sps", "agc_bw", "agc_gain0", "samples_per_ted", "period_min", "period_max",
                                        "alpha_unlocked", "beta_unlocked", "alpha_locked", "beta_locked", "dc_len", "ntaps"};

Header make_header(const same_config& cfg, const same_derived& derived, const SameTapsWide& taps, uint32_t ntaps,
                   uint32_t n_words, uint32_t n_records) {
  Header s;
  memset(&s, 0, sizeof s);
  s.cfg = cfg; s.derived = derived;
  s.slots = tap_slots(ntaps);
  s.n_records = n_records; s.n_words = n_words; s.record_bytes = same_state_record_bytes(n_words);
  for (uint32_t i = 0; i < ntaps; ++i) {
    const float v[4] = {taps.t[i].x, taps.t[i].y, taps.t[i].z, taps.t[i].w};
    put_words(s.taps + 8 * i, v, 8);
    put_words(s.taps + 8 * s.slots + 8 * i, v + 2, 8);
  }
  return s;
}

void write_header(const Header& s, uint8_t* h) {
  const size_t bytes = header_bytes(s.slots);
  memset(h, 0, bytes);
  put32(h + 0, kStMagic); put32(h + 4, kStVersion); put32(h + 8, kStBom); put32(h + 12, (uint32_t)bytes);
  put32(h + 16, s.n_records); put32(h + 20, s.n_words); put32(h + 24, (uint32_t)sizeof(StreamBlob));
  put32(h + 28, SAME_BURST_CAP); put32(h + 32, s.record_bytes);
  put_words(h + kStOffConfig, &s.cfg, sizeof(same_config));
  put_words(h + kStOffDerived, &s.derived, sizeof(same_derived));
  memcpy(h + kStOffMark, s.taps, 16 * (size_t)s.slots);
  put32(h + off_crc(s.slots), crc32_host(h, off_crc(s.slots)));
}

int parse_header(const void* buf, size_t len, Header* out, std::string* why) {
  const uint8_t* h = static_cast<const uint8_t*>(buf);
  auto bad = [&](const std::string& m) { *why = "state buffer: " + m; return (int)SAME_ERR_INVALID_ARG; };
  if (!h) return bad("null pointer");
  if (len < 16) return bad("truncated header");
  if (get32(h) != kStMagic) return bad("bad magic");
  if (get32(h + 8) != kStBom) return bad("wrong byte order");
  if (get32(h + 4) != kStVersion) return bad("format version " + std::to_string(get32(h + 4)) + ", this library reads version " + std::to_string(kStVersion));
  // the header size says how many tap entries each section holds; checked against the configuration below
  const uint32_t hbytes = get32(h + 12);
  if (hbytes < kHeaderBytes || hbytes > header_bytes(SAME_MAX_TAPS) || (hbytes - kHeaderBytes) % 16u != 0)
    return bad("bad header size");
  const uint32_t slots = (uint32_t)((hbytes - kFixedHeaderBytes) / 16u);
  if (len < hbytes) return bad("truncated header");
  if (get32(h + off_crc(slots)) != crc32_host(h, off_crc(slots))) return bad("header CRC mismatch");
  Header s;
  memset(&s, 0, sizeof s);
  s.slots = slots;
  get_words(&s.cfg, h + kStOffConfig, sizeof(same_config));
  const size_t ntaps = same_ntaps(s.cfg.input_rate);
  if (ntaps > SAME_MAX_TAPS || hbytes != header_bytes(ntaps))
    return bad("header size " + std::to_string(hbytes) + " does not match the " + std::to_string(ntaps) + "-tap filters of input_rate " +
               std::to_string(s.cfg.input_rate) + " Hz (" + std::to_string(header_bytes(ntaps)) + " bytes)");
  s.n_records = get32(h + 16); s.n_words = get32(h + 20); s.record_bytes = get32(h + 32);
  if (get32(h + 24) != sizeof(StreamBlob) || get32(h + 28) != SAME_BURST_CAP) return bad("stream blob layout differs from this library's");
  if (s.n_words < F_NUM_SCALARS || s.n_words > (1u << 16) || s.record_bytes != same_state_record_bytes(s.n_words))
    return bad("inconsistent record size");
  const size_t need = hbytes + (size_t)s.n_records * s.record_bytes;
  if (len < need) return bad("truncated: " + std::to_string(len) + " bytes, the header announces " + std::to_string(need));
  if (len > need) return bad("trailing bytes after the last record");
  get_words(&s.derived, h + kStOffDerived, sizeof(same_derived));
  memcpy(s.taps, h + kStOffMark, 16 * (size_t)slots);
  *out = s;
  return SAME_OK;
}

// derived values and taps are compared bit for bit: they are libm results of the exporting host
int compare_header(const Header& mine, const Header& s, std::string* why) {
  uint32_t a[19], b[19];
  memcpy(a, &mine.cfg, sizeof a); memcpy(b, &s.cfg, sizeof b);
  for (int i = 0; i < 19; ++i)
    if (a[i] != b[i]) { *why = std::string("state was produced under another configuration: ") + kConfigFields[i] + " differs"; return SAME_ERR_INVALID_CONFIG; }
  uint32_t c[12], d[12];
  memcpy(c, &mine.derived, sizeof c); memcpy(d, &s.derived, sizeof d);
  for (int i = 0; i < 12; ++i)
    if (c[i] != d[i]) { *why = std::string("derived constant ") + kDerivedFields[i] + " differs from this engine's (another host's libm?)"; return SAME_ERR_INVALID_CONFIG; }
  // equal input rates (checked above) mean equal tap entries per section
  const size_t sec = 8 * (size_t)mine.slots;
  if (memcmp(mine.taps, s.taps, sec) != 0) { *why = "mark filter taps differ from this engine's"; return SAME_ERR_INVALID_CONFIG; }
  if (memcmp(mine.taps + sec, s.taps + sec, sec) != 0) {
    *why = "space filter taps differ from this engine's"; return SAME_ERR_INVALID_CONFIG;
  }
  if (s.n_words != mine.n_words) { *why = "state words per stream differ from this engine's"; return SAME_ERR_INVALID_CONFIG; }
  return SAME_OK;
}

const char* check_name(uint32_t code) { return code < CK_COUNT ? kCheckNames[code] : "invalid"; }

}  // namespace same_state

extern "C" uint32_t same_state_record_bytes(uint32_t n_words) { return same_state::rec_geom(n_words).bytes; }

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
