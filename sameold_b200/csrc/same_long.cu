// same_long.cu — the long-stream path: ONE stream (BASELINE config 5: a single 24 h stream with sparse bursts), where
// there is no second stream to fill a warp and the receiver's dependent chain per TED round (~1500 cycles) is all there
// is.  What the north star asks for here — "time-parallel FIR/correlator tiles, per-stream loop kernels" — is possible
// bit-exactly as long as the AGC is unlocked, i.e. everywhere except inside bursts (0.5 % of such a stream):
//
//   A  same_long_dc_kernel    s16 -> exact DC-blocked f32, time-parallel (the integer recursion has 31 samples of memory)
//   B  same_long_agc_kernel   the AGC recurrence (agc.rs:72-77) in blocks of 2048 samples, one thread per block.  Block 0
//                             starts from the stream's true gain; every other block warms up on the 1024 samples before
//                             it from a guessed gain.  The unlocked AGC map contracts (|1 - |d| bw| per sample), so
//                             the trajectories coalesce BITWISE on loud noise (corpus level: within ~400 samples) and
//                             when a gain limit pins them (quiet input at gmax) -- but NOT in between: with samedec
//                             limits, noise of sigma ~300-1000 LSB (-40 to -30 dBFS) fails nearly every hand-over
//                             (DESIGN.md §4).  So whether a block's start gain equals its predecessor's end gain is
//                             CHECKED, bit for bit:
//      same_long_verify_kernel   first block whose hand-over fails -> end of the range that may be consumed.
//   C  same_long_mf_kernel    the mark/space matched filters (demod.rs:156-164) at EVERY sample position of that AGC
//                             output, time-parallel: 21x the arithmetic of the sequential receiver, in parallel.
//   D  same_long_seq_kernel   the timing loop (A5) strictly sequential on one lane, picking its soft symbols out of C's
//                             output (staged through shared memory), and the squelch, equalizer, framer and transport
//                             (A6-A9) on a second warp, one ring of symbol records behind: ~250 cycles per TED round
//                             instead of ~1500.  It stops when the symbol stages lock the AGC (sync found: a burst
//                             begins) or reset the timing loop, at the end of the verified range, or at the end.
//   bursts                    the ordinary tile-fed single-warp kernel (same_rx_fast_kernel<true>) on A's output, until
//                             the AGC is unlocked again; then B-D restart from the true state.
//   unverified spans          after a pass that stopped at its verified end: the ordinary pipelined kernel on the raw
//                             samples (DC state brought to the span start by A), in spans that grow while the stops
//                             repeat; the host also bounds each pass's range (same_long_run, at the end of this file).
// The speculation in B never decides anything: a block is used only after its hand-over gain was verified, and D's
// arithmetic is the sequential receiver's (same_lane.cuh), so the events are those of the reference, bit for bit
// (tests: the full 24 h stream, the 16-minute stream in chunks, every single-stream test above the length threshold).
// All state stays in the ordinary resident layout between kernels; the DC-blocker state is committed at the end.
//
// Every other geometry (1..512 taps, DC length 1..512: 11 025, 44 100, 48 000, 88 200-192 000 Hz, 22 050 Hz with another
// DC length), s16 input only:
//   A  the general DC front ("A, general" below): the literal f32 recursion of the generic / wide kernels split into an
//      exact integer feed-forward sum, time-parallel, and the rounded feedback sum as one sequential scan; ma0 and
//      fbsum are kept for the whole chunk, so that same_long_commit_dcg_kernel can write the state at any position
//   B, D  the same kernels instantiated for p.ntaps (template argument 0)
//   C  same_long_mf_wide_kernel: the taps of SameTapsWide, the packed exact FFMA2 pair
//   bursts and unverified spans   the ordinary generic (or wide) kernel on the raw samples, after a DC commit at the
//      span's start: the tile-fed and pipelined kernels exist for the 22050 Hz class only.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstddef>

#include "same_fast.cuh"
#include "same_internal.h"
#include "same_lane.cuh"

namespace same_dev {

#define LS_RUN 256        // samples per thread in A
#define LS_BLOCK 2048     // samples per thread in B
#define LS_WARM 1024      // warm-up samples of a speculative block
#define LS_TILE 4096      // soft symbols staged per shared-memory tile in D

// ---------------------------------------------------------------------------------------------------------------- A
__global__ void same_long_dc_kernel(const __grid_constant__ SameParams p, const int16_t* __restrict__ src, const uint32_t len,
                                    float* __restrict__ d, uint32_t* __restrict__ dc_next) {
  const SameLayout& L = p.layout;
  const uint32_t run = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t r0 = run * LS_RUN;
  if (r0 >= len) return;
  const uint32_t r1 = min(r0 + (uint32_t)LS_RUN, len);
  const uint32_t* st = p.state32;   // stream 0
  DcInt dc;
  RawFeed feed;
  uint32_t cur[FAST_CHUNK / 2];
  if (run == 0) {
    dc_load(dc, st, L);
    feed.init(src, 0u, len);
  } else {
    dc_zero(dc);
    feed.init(src, r0 - FAST_CHUNK, len);
    feed.take_full(cur, r0 - FAST_CHUNK, len);
    dc_chunk<FAST_CHUNK>(dc, cur, [](int, float) {});      // warm-up: exact from the 32nd sample on
  }
  uint32_t c = r0;
  for (; c + FAST_CHUNK <= r1; c += FAST_CHUNK) {
    feed.take_full(cur, c, len);
    float* dst = d + c;
    dc_chunk<FAST_CHUNK>(dc, cur, [&](int i, float v) { dst[i] = v; });
  }
  const auto to_next = [&](uint32_t w, uint32_t bits) { dc_next[(size_t)w * L.n_pad] = bits; };
  if (c < r1) {
    const uint32_t nnew = r1 - c;
    feed.take_partial(cur, c, nnew);
    float* dst = d + c;
    dc_chunk_partial<FAST_CHUNK>(dc, cur, (int)nnew, [&](int i, float v) { dst[i] = v; });
    dc_store_after_partial<FAST_CHUNK>(dc, cur, nnew, to_next);
  } else if (r1 == len) {
    dc_store(dc, to_next);
  }
}

// commit A's DC-blocker state (end of the submit)
__global__ void same_long_commit_dc_kernel(const __grid_constant__ SameParams p, const uint32_t* __restrict__ dc_next) {
  const SameLayout& L = p.layout;
  if (threadIdx.x < DCW_WORDS) DcToState{p.state32, L}(threadIdx.x, dc_next[(size_t)threadIdx.x * L.n_pad]);
}

// -------------------------------------------------------------------------------------------------------- A, general
// Any other geometry (DC length L = 1..512, s16 samples): the literal f32 recursion of dcblock.rs:45-49,104-108 (as in
// same_rx_generic_kernel / same_rx_wide_kernel) split into what is exact and what is not.
//   ffsum[n] = ffsum[n-1] + (x[n] - x[n-L])   every operand an integer, |ffsum| <= 512 * 32768 = 2^24: exact, so it is
//                                             the integer D + (x[n-L+1] + ... + x[n]) (D = ffsum - window sum of the
//                                             state, 0 unless the state came from elsewhere), time-parallel
//   ma0[n]   = ffsum[n] * inv_len             time-parallel
//   fbsum[n] = fbsum[n-1] + (ma0[n] - ma0[n-L])   rounded (inv_len is not dyadic, or |fbsum| > 2^19 at L = 32): a
//                                             sequential scan of one thread, tiles staged by the rest of the warp
//   d[n]     = x[n-L+1] - gate * (fbsum[n] * inv_len)   time-parallel
// x[m] and ma0[m] for m < 0 are the windows the chunk started with: dc0, a copy of the state's DC words taken before
// the first launch, because ordinary-kernel spans overwrite the resident words.  Every zero is +0 here as in the
// recursion (integer input, x - x = +0).  ma0 and fbsum are kept for the whole chunk, so that the state can be
// committed at any position (same_long_commit_dcg_kernel).
// dc0 words: [0, L) ff window, [L, 2L) fb window (oldest first), 2L ffsum, 2L+1 fbsum, 2L+2 D (int).
#define LG_RUN 1024       // samples per thread in the feed-forward kernel

// x[m] of the chunk as an integer, m >= -L
__device__ __forceinline__ int lg_x(const int16_t* src, const uint32_t* dc0, int L, int m) {
  return m >= 0 ? (int)src[m] : __float2int_rn(__uint_as_float(dc0[m + L]));
}

__global__ void __launch_bounds__(512) same_long_dc_save_kernel(const __grid_constant__ SameParams p, uint32_t* __restrict__ dc0) {
  __shared__ int wsum;
  const SameLayout& L = p.layout;
  const uint32_t* st = p.state32;   // stream 0
  const int dcl = (int)p.dc_len;
  if (threadIdx.x == 0) wsum = 0;
  __syncthreads();
  int part = 0;
  for (int i = threadIdx.x; i < dcl; i += blockDim.x) {
    const uint32_t ff = LANE_ST(st, L, L.dc_ff + i);
    dc0[i] = ff;
    dc0[dcl + i] = LANE_ST(st, L, L.dc_fb + i);
    part += __float2int_rn(__uint_as_float(ff));
  }
  atomicAdd(&wsum, part);
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t ffsum = LANE_ST(st, L, F_DC_FFSUM);
    dc0[2 * dcl] = ffsum;
    dc0[2 * dcl + 1] = LANE_ST(st, L, F_DC_FBSUM);
    dc0[2 * dcl + 2] = (uint32_t)(__float2int_rn(__uint_as_float(ffsum)) - wsum);
  }
}

// ma0[n], n in [0, len): one run of LG_RUN samples per thread, the window sum slid along it
__global__ void same_long_ma0_kernel(const __grid_constant__ SameParams p, const int16_t* __restrict__ src, const uint32_t len,
                                     const uint32_t* __restrict__ dc0, float* __restrict__ ma0) {
  const uint32_t r0 = (blockIdx.x * blockDim.x + threadIdx.x) * LG_RUN;
  if (r0 >= len) return;
  const uint32_t r1 = min(r0 + (uint32_t)LG_RUN, len);
  const int dcl = (int)p.dc_len;
  const float inv_len = p.dc_inv_len;
  int s = (int)dc0[2 * dcl + 2];                                    // D + the window x[r0-L .. r0-1]
  for (int m = (int)r0 - dcl; m < (int)r0; ++m) s += lg_x(src, dc0, dcl, m);
  for (uint32_t n = r0; n < r1; ++n) {
    s += (int)src[n] - lg_x(src, dc0, dcl, (int)n - dcl);           // = ffsum[n], exact
    ma0[n] = FMUL(__int2float_rn(s), inv_len);
  }
}

// fbs[n] = ma0[n] - ma0[n - L]: the increments the scan adds
__global__ void same_long_dfb_kernel(const __grid_constant__ SameParams p, const uint32_t len, const uint32_t* __restrict__ dc0,
                                     const float* __restrict__ ma0, float* __restrict__ fbs) {
  const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= len) return;
  const uint32_t dcl = p.dc_len;
  const float aged = n >= dcl ? ma0[n - dcl] : __uint_as_float(dc0[dcl + n]);   // fb window: ma0[m] at dc0[2L + m]
  fbs[n] = FSUB(ma0[n], aged);
}

// In place: fbs[n] = fbsum[n] = fbsum[n-1] + fbs[n], from the state's fbsum.  One warp: lane 0 adds (one shared load
// per 4 samples, 4 dependent FADDs, one shared store); all lanes stage the next tile with 16-byte asynchronous copies
// and write the finished one back.  `fbs` is padded by two tiles.
__global__ void __launch_bounds__(32) same_long_fbscan_kernel(const __grid_constant__ SameParams p, const uint32_t len,
                                                              const uint32_t* __restrict__ dc0, float* __restrict__ fbs) {
  __shared__ __align__(16) float tile[2][LS_TILE];
  const uint32_t lane = threadIdx.x;
  const auto stage = [&](uint32_t tbase, int buf) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&tile[buf][0]);
#pragma unroll 4
    for (uint32_t j = lane * 4u; j < LS_TILE; j += 128u)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + j * 4u), "l"(fbs + tbase + j) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  float f = __uint_as_float(dc0[2 * p.dc_len + 1]);
  stage(0u, 0);
  int buf = 0;
  for (uint32_t tbase = 0; tbase < len; tbase += LS_TILE, buf ^= 1) {
    stage(tbase + LS_TILE, buf ^ 1);
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncwarp();
    float4* t4 = reinterpret_cast<float4*>(&tile[buf][0]);
    const uint32_t n4 = (min((uint32_t)LS_TILE, len - tbase) + 3u) / 4u;
    if (lane == 0) {
#pragma unroll 8
      for (uint32_t j = 0; j < n4; ++j) {
        float4 v = t4[j];
        f = FADD(f, v.x); v.x = f;
        f = FADD(f, v.y); v.y = f;
        f = FADD(f, v.z); v.z = f;
        f = FADD(f, v.w); v.w = f;
        t4[j] = v;
      }
    }
    __syncwarp();
    float4* g4 = reinterpret_cast<float4*>(fbs + tbase);
    for (uint32_t j = lane; j < n4; j += 32u) g4[j] = t4[j];
    __syncwarp();
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// d[n] = x[n-L+1] - gate * (fbsum[n] * inv_len)
__global__ void same_long_dcout_kernel(const __grid_constant__ SameParams p, const int16_t* __restrict__ src, const uint32_t len,
                                       const uint32_t* __restrict__ dc0, const float* __restrict__ fbs, float* __restrict__ d) {
  const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= len) return;
  const int dcl = (int)p.dc_len;
  const int m = (int)n - dcl + 1;
  const float sig = m >= 0 ? (float)src[m] : __uint_as_float(dc0[m + dcl]);
  d[n] = FSUB(sig, FMUL(p.dc_gate, FMUL(fbs[n], p.dc_inv_len)));
}

// The generic-layout DC state after sample pos - 1 of the chunk (1 <= pos <= len): windows x[pos-L .. pos-1] and
// ma0[pos-L .. pos-1], ffsum = D + their sum, fbsum[pos - 1]
__global__ void __launch_bounds__(512) same_long_commit_dcg_kernel(const __grid_constant__ SameParams p, const int16_t* __restrict__ src,
                                                                   const uint32_t pos, const uint32_t* __restrict__ dc0,
                                                                   const float* __restrict__ ma0, const float* __restrict__ fbs) {
  __shared__ int wsum;
  const SameLayout& L = p.layout;
  uint32_t* st = p.state32;   // stream 0
  const int dcl = (int)p.dc_len;
  if (threadIdx.x == 0) wsum = 0;
  __syncthreads();
  int part = 0;
  for (int i = threadIdx.x; i < dcl; i += blockDim.x) {
    const int m = (int)pos - dcl + i;
    const int x = lg_x(src, dc0, dcl, m);
    part += x;
    LANE_ST(st, L, L.dc_ff + i) = m >= 0 ? __float_as_uint((float)x) : dc0[m + dcl];
    LANE_ST(st, L, L.dc_fb + i) = m >= 0 ? __float_as_uint(ma0[m]) : dc0[2 * dcl + m];
  }
  atomicAdd(&wsum, part);
  __syncthreads();
  if (threadIdx.x == 0) {
    LANE_ST(st, L, F_DC_FFSUM) = __float_as_uint(__int2float_rn((int)dc0[2 * dcl + 2] + wsum));
    LANE_ST(st, L, F_DC_FBSUM) = __float_as_uint(fbs[pos - 1u]);
  }
}

// ---------------------------------------------------------------------------------------------------------------- B
// d: DC-blocked samples of the submit; the range is [pos0, end).  yfull[ntaps + (n - pos0)] = AGC output of sample n,
// yfull[0..ntaps) = the demod window before pos0 (copied from the state); gspec[n - pos0] = gain AFTER sample n;
// g_in[k] = the gain block k > 0 started with after its warm-up.  NT = ntaps, or 0: p.ntaps (general geometry).  The
// AGC itself has no geometry: its bandwidth per sample is agc_bandwidth / 520.83 at every rate (receiver.rs:511).
template <int NT>
__global__ void same_long_agc_kernel(const __grid_constant__ SameParams p, const float* __restrict__ d, const uint32_t pos0,
                                     const uint32_t end, float* __restrict__ yfull, float* __restrict__ gspec,
                                     float* __restrict__ g_in) {
  const int ntaps = NT ? NT : (int)p.ntaps;
  const SameLayout& L = p.layout;
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long sk64 = (unsigned long long)pos0 + (unsigned long long)k * LS_BLOCK;
  if (sk64 >= end) return;
  const uint32_t sk = (uint32_t)sk64;
  const float bw = p.agc_bw, gmin = p.agc_min, gmax = p.agc_max;
  const float g_true = __uint_as_float(LANE_ST(p.state32, L, F_AGC_GAIN));   // gain at pos0
  float g = g_true;
  if (k == 0) {
    for (int i = 0; i < ntaps; ++i) yfull[i] = __uint_as_float(LANE_ST(p.state32, L, L.win + i));
  } else {
    for (uint32_t n = sk - LS_WARM; n < sk; ++n) (void)agc_step(g, d[n], bw, gmin, gmax);   // LS_BLOCK >= LS_WARM: n >= pos0
    g_in[k] = g;
  }
  const uint32_t e = min(sk + (uint32_t)LS_BLOCK, end);
  float* yo = yfull + ntaps - pos0;
  float* go = gspec - pos0;
  for (uint32_t n = sk; n < e; ++n) {
    yo[n] = agc_step(g, d[n], bw, gmin, gmax);
    go[n] = g;
  }
}

// ctrl[0] = end of the verified range: the start of the first block whose warm-started gain differs (bitwise) from its
// predecessor's end gain, or `end`.  (ctrl[0] is preset to `end` by the host.)
__global__ void same_long_verify_kernel(const float* __restrict__ gspec, const float* __restrict__ g_in, const uint32_t pos0,
                                        const uint32_t end, uint32_t* __restrict__ ctrl) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x + 1u;
  const unsigned long long sk64 = (unsigned long long)pos0 + (unsigned long long)k * LS_BLOCK;
  if (sk64 >= end) return;
  const uint32_t sk = (uint32_t)sk64;
  if (__float_as_uint(g_in[k]) != __float_as_uint(gspec[sk - 1u - pos0])) atomicMin(&ctrl[0], sk);
}

// ---------------------------------------------------------------------------------------------------------------- C
// soft[i] = demodulated sample at the position pos0 + i (window = samples pos0 + i - 42 .. pos0 + i - 1 = yfull[i .. i+41]),
// i = 1 .. n_out: one rounded multiply and one rounded add per component and tap, newest sample first
// (filter.rs:363-377), |mark| - |space| clamped (demod.rs:163).
__global__ void __launch_bounds__(256) same_long_mf_kernel(const __grid_constant__ SameTaps2 taps, const float* __restrict__ yfull,
                                                           const uint32_t n_out, float* __restrict__ soft) {
  __shared__ float tile[256 + FAST_NTAPS];
  const uint32_t i0 = blockIdx.x * 256u + 1u;
  for (uint32_t j = threadIdx.x; j < 256u + FAST_NTAPS - 1u; j += 256u) {
    const uint32_t idx = i0 + j;                       // yfull index; valid up to n_out + 41
    tile[j] = (idx <= n_out + FAST_NTAPS - 1u) ? yfull[idx] : 0.0f;
  }
  __syncthreads();
  const uint32_t i = i0 + threadIdx.x;
  if (i > n_out) return;
  float mr = 0.0f, mi = 0.0f, sr = 0.0f, si = 0.0f;
#pragma unroll
  for (int j = 0; j < FAST_NTAPS; ++j) {
    const float v = tile[threadIdx.x + (FAST_NTAPS - 1) - j];
    mr = FADD(mr, FMUL(v, taps.mark[j].x));
    mi = FADD(mi, FMUL(v, taps.mark[j].y));
    sr = FADD(sr, FMUL(v, taps.space[j].x));
    si = FADD(si, FMUL(v, taps.space[j].y));
  }
  soft[i] = rclamp(FSUB(hypot_fixed(mr, mi), hypot_fixed(sr, si)), -1.0f, 1.0f);
}

// The same at any geometry (1..512 taps, SameTapsWide): a shared tile of 256 + ntaps - 1 samples, one output per
// thread, newest sample first with the exact packed FFMA2 pair of same_rx_wide_kernel.
__global__ void __launch_bounds__(256) same_long_mf_wide_kernel(const __grid_constant__ SameParams p,
                                                                const __grid_constant__ SameTapsWide taps,
                                                                const float* __restrict__ yfull, const uint32_t n_out,
                                                                float* __restrict__ soft) {
  __shared__ float wtile[256 + SAME_MAX_TAPS - 1];
  const uint32_t ntaps = p.ntaps;
  const uint32_t i0 = blockIdx.x * 256u + 1u;
  for (uint32_t j = threadIdx.x; j < 256u + ntaps - 1u; j += 256u) {
    const uint32_t idx = i0 + j;                       // yfull index; valid up to n_out + ntaps - 1
    wtile[j] = (idx <= n_out + ntaps - 1u) ? yfull[idx] : 0.0f;
  }
  __syncthreads();
  const uint32_t i = i0 + threadIdx.x;
  if (i > n_out) return;
  const float2 one2 = make_float2(p.f_one, p.f_one), negz2 = make_float2(p.f_negzero, p.f_negzero);
  float2 am = make_float2(0.0f, 0.0f), as = make_float2(0.0f, 0.0f);
  const float* yp = wtile + threadIdx.x + ntaps - 1u;   // newest sample of this output's window
#pragma unroll 4
  for (uint32_t j = 0; j < ntaps; ++j) {
    const float v = yp[-(int)j];
    const float4 t = taps.t[j];
    const float2 vv = make_float2(v, v);
    am = __ffma2_rn(am, one2, __ffma2_rn(vv, make_float2(t.x, t.y), negz2));
    as = __ffma2_rn(as, one2, __ffma2_rn(vv, make_float2(t.z, t.w), negz2));
  }
  soft[i] = rclamp(FSUB(hypot_fixed(am.x, am.y), hypot_fixed(as.x, as.y)), -1.0f, 1.0f);
}

// ---------------------------------------------------------------------------------------------------------------- D
// Two warps, one lane each doing sequential work, pipelined:
//   warp T  the timing loop (A5): picks its soft symbol out of the staged tile (the warp's other lanes stage tiles one
//           ahead with 16-byte asynchronous copies), TED, PI loop, next fire clock; every emitted symbol goes into a ring
//           of records together with the loop state it left behind.
//   warp S  the symbol stages (A6-A9) on those records: squelch, equalizer, framer, events, transport.
// Until the squelch finds sync nothing the symbol stages do feeds back into the timing loop (receiver.rs:423-438,
// 479-490 all hang off sync / carrier-drop / burst-end), so T may run ahead of S by the ring.  When S's symbol locks the
// AGC (sync found: a burst begins) or resets the timing loop (end()), the record's state IS the receiver's state at that
// symbol: S stops the kernel there and whatever T did beyond it is dropped (T touches no global state).
// ctrl[0] in: end of the verified range (absolute position in the submit).  Out: ctrl[1] = position reached,
// ctrl[2] = why it stopped (0 range end, 1 AGC locked by the symbol stages, 2 timing loop reset by them).
#define LS_RING 64
struct LsRec { uint32_t pos; float zero, sym, until, pavg, pinst, ted0; uint32_t pad; };

// The counters are published in batches (the release store's MEMBAR is what costs): T every LS_HEAD_BATCH records and
// when it finishes, S every LS_TAIL_BATCH records and whenever it has drained the ring.
#ifndef LS_HEAD_BATCH
#define LS_HEAD_BATCH 4u
#endif
#define LS_TAIL_BATCH 8u

// NT = ntaps, or 0: p.ntaps (general geometry).  Only the demod window stored at the end depends on it: the timing loop
// runs the same number of TED rounds per second of audio at every rate.
template <int NT>
__global__ void __launch_bounds__(64) same_long_seq_kernel(const __grid_constant__ SameParams p, const float* __restrict__ soft,
                                                           const float* __restrict__ yfull, const float* __restrict__ gspec,
                                                           const uint32_t pos0, uint32_t* __restrict__ ctrl) {
  __shared__ __align__(16) float tile[2][LS_TILE];
  __shared__ LsRec ring[LS_RING];
  __shared__ volatile uint32_t sh_head, sh_tail, sh_stop, sh_tdone;
  __shared__ float t_final[8];          // T's loop state at the end of the range: until, pavg, pinst, ted0, ted1, ted2, tedcnt, clock
  __shared__ uint32_t t_pos;
  const SameLayout& L = p.layout;
  const int lane = threadIdx.x & 31;
  const int role = threadIdx.x >> 5;   // 0 = T, 1 = S
  uint32_t* st = p.state32;            // stream 0
  StreamBlob* blob = p.blobs;
  const uint32_t range = ctrl[0] - pos0;   // samples that may be consumed
  if (threadIdx.x == 0) { sh_head = 0u; sh_tail = 0u; sh_stop = 0u; sh_tdone = 0u; }
  __syncthreads();

  Lane a;
  lane_load(a, p, st, 0u);
  uint32_t why = 0, stop_pos = 0;

  if (role == 0) {
    // ================================================ T: timing loop ================================================
    uint32_t pos = 0;                    // relative to pos0
    int cfire = fire_clock(a.until, a.clock);
    uint32_t done = 0, head = 0, tail_seen = 0;
    const auto stage = [&](uint32_t tbase, int buf) {   // `soft` is padded by two tiles: reading past `range` is harmless
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&tile[buf][0]);
#pragma unroll 4
      for (uint32_t j = (uint32_t)lane * 4u; j < LS_TILE; j += 128u)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + j * 4u), "l"(soft + tbase + j) : "memory");
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    stage(0u, 0);
    int buf = 0;
    for (uint32_t tbase = 0; !done; tbase += LS_TILE, buf ^= 1) {
      stage(tbase + LS_TILE, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        const float* tl = &tile[buf][0];
        if (sh_stop) done = 1;                                           // checked per tile and while the ring is full
        while (!done) {
          const uint32_t next = pos + (uint32_t)(cfire - a.clock);      // position of the next TED instant
          if (next > range) {                                            // not inside the range: consume what is left
            a.clock += (int)(range - pos);
            pos = range;
            done = 1;
            break;
          }
          if (next >= tbase + LS_TILE) break;                            // in the next tile
          a.clock = cfire;
          pos = next;
          const float s_in = tl[pos - tbase];
          const float rem = FSUB(a.until, (float)a.clock);               // receiver.rs:352
          a.clock = 0;
          const bool have_sym = ted_step(a, p, s_in, rem);
          cfire = fire_clock(a.until, 0);
          if (have_sym) {
            if (head - tail_seen >= (uint32_t)LS_RING) {                   // ring full as far as T knows: look again, wait for S
              while (head - (tail_seen = ls_observe(&sh_tail)) >= (uint32_t)LS_RING) { if (sh_stop) { done = 1; break; } }
              if (done) break;
            }
            // the record, then the head counter that publishes it (ls_publish)
            volatile float* q = reinterpret_cast<volatile float*>(&ring[head & (LS_RING - 1)]);
            q[1] = a.ted1; q[2] = a.ted2; q[3] = a.until; q[4] = a.pavg; q[5] = a.pinst; q[6] = a.ted0;
            reinterpret_cast<volatile uint32_t*>(q)[0] = pos;
            head += 1u;
            if ((head & (LS_HEAD_BATCH - 1u)) == 0u) ls_publish(&sh_head, head);   // S may lag: it feeds back only by stopping
          }
        }
        if (done) {
          t_final[0] = a.until; t_final[1] = a.pavg; t_final[2] = a.pinst; t_final[3] = a.ted0; t_final[4] = a.ted1;
          t_final[5] = a.ted2; t_final[6] = __uint_as_float(a.tedcnt); t_final[7] = __int_as_float(a.clock);
          t_pos = pos;
          ls_publish(&sh_head, head);          // whatever the batching held back
          ls_publish(&sh_tdone, 1u);
        }
      }
      done = __shfl_sync(0xffffffffu, done, 0);
      __syncwarp();
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (lane == 0) {
    // ================================================ S: symbol stages ================================================
    uint32_t tail = 0, tail_pub = 0;
    while (true) {
      uint32_t head = ls_observe(&sh_head);
      if (tail == head) {
        if (tail_pub != tail) { ls_publish(&sh_tail, tail); tail_pub = tail; }   // ring drained: T may be waiting for room
        if (ls_observe(&sh_tdone)) { head = ls_observe(&sh_head); if (tail == head) break; }
        else continue;
      }
      LsRec r;
      {
        const volatile float* q = reinterpret_cast<const volatile float*>(&ring[tail & (LS_RING - 1)]);
        r.pos = reinterpret_cast<const volatile uint32_t*>(q)[0];
        r.zero = q[1]; r.sym = q[2]; r.until = q[3]; r.pavg = q[4]; r.pinst = q[5]; r.ted0 = q[6];
      }
      // The quiet symbol (nearly all of a long stream): no carrier, framer idle, nothing pending in the transport layer
      // and this symbol does not complete the sync word.  Then symbol_squelch + symbol_finish reduce to the squelch's
      // own bookkeeping (same expressions as same_lane.cuh:symbol_squelch, codesquelch.rs:228-304,421-428,483-488) --
      // written out here because a single lane pays for every instruction of the select-based general form.
      bool quiet = false;
      if (p.trace == nullptr && a.byteclk < 0 && a.fr.st == 0u && a.link_last == 0u) {
        const uint32_t nd = (a.sq_data >> 1) | ((r.sym >= 0.0f) ? 0x80000000u : 0u);
        const uint32_t cerr = __popc(nd ^ p.sq_sync_word);
        const float pw = fmaxf(FADD(a.sq_power, FMUL(FSUB(FMUL(r.sym, r.sym), a.sq_power), p.sq_bw)), 0.0f);
        const unsigned long long sc = a.symcount + 1ull;
        const unsigned long long n = a.n0 + r.pos;
        const bool acquire = sc >= 32ull && !(a.flags & FLAG_SQ_LOCK) && cerr <= p.sq_max_err && pw >= p.sq_open;
        const bool transport_due = (a.tr.have_eom && n > a.tr.eom_at) || sc >= a.tr.next_deadline ||
                                   ((a.tr.hist_n ? 1u : 0u) != a.tr.tr_state);
        if (!acquire && !transport_due) {
          LANE_ST(st, L, L.sqh + (a.sq_head & 63u)) = __float_as_uint(r.zero);
          LANE_ST(st, L, L.sqh + ((a.sq_head + 1u) & 63u)) = __float_as_uint(r.sym);
          a.sq_head = (a.sq_head + 2u) & 63u;
          a.sq_data = nd;
          a.sq_power = pw;
          a.sq_pflags = (a.sq_pflags >> 1) | ((pw >= p.sq_close) ? 0x80000000u : 0u);
          a.symcount = sc;
          quiet = true;
        }
      }
      if (quiet) {
        tail += 1u;
        if ((tail & (LS_TAIL_BATCH - 1u)) == 0u) { ls_publish(&sh_tail, tail); tail_pub = tail; }
        continue;
      }
      a.until = r.until; a.pavg = r.pavg; a.pinst = r.pinst;
      a.ted0 = r.ted0; a.ted1 = r.zero; a.ted2 = r.sym; a.tedcnt = 1u; a.clock = 0;
      symbol_step(a, p, 0u, st, blob, r.zero, r.sym, a.n0 + r.pos);
      tail += 1u;
      ls_publish(&sh_tail, tail);
      tail_pub = tail;
      if ((a.flags & FLAG_AGC_LOCKED) || a.tedcnt != 1u) {       // sync found (AGC locked) or end() reset the timing loop
        why = (a.flags & FLAG_AGC_LOCKED) ? 1u : 2u;
        stop_pos = r.pos;
        __threadfence_block();
        sh_stop = 1u;
        break;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x != 32) return;
  // ---- state out (S's lane): the symbol stages' state + the timing loop's state at the stop symbol / at the range end ----
  uint32_t pos = stop_pos;
  if (why == 0u) {
    a.until = t_final[0]; a.pavg = t_final[1]; a.pinst = t_final[2]; a.ted0 = t_final[3]; a.ted1 = t_final[4];
    a.ted2 = t_final[5]; a.tedcnt = __float_as_uint(t_final[6]); a.clock = __float_as_int(t_final[7]);
    pos = t_pos;
  }
  if (pos > 0u) a.g = gspec[pos - 1u];
  lane_store(a, p, st, a.n0 + pos);
  const int ntaps = NT ? NT : (int)p.ntaps;
  for (int i = 0; i < ntaps; ++i) LANE_ST(st, L, L.win + i) = __float_as_uint(yfull[pos + i]);
  ctrl[1] = pos0 + pos;
  ctrl[2] = why;
}

}  // namespace same_dev

// ---------------------------------------------------------------- host: the driver (same_long_run) and its operations
namespace {

constexpr uint32_t kLongChunk = 1u << 24;       // samples per internal pass (bounds the scratch buffers: 16 B per sample)
constexpr uint32_t kLongSpan = 8192;            // samples per ordinary span while the AGC is locked (inside a burst)
constexpr uint32_t kLongSpanMax = 1u << 20;     // longest ordinary span after verification stops in a row
constexpr uint32_t kLongMinPass = 1u << 16;     // shortest range of a speculative pass
// The three above are samples of the 22050 Hz class; any other tap count scales them by ntaps / 42 to cover the same
// audio time (an ordinary span then costs the same share of a stream, a pass the same number of TED rounds).  The
// speculative AGC's block and warm-up stay in samples: its bandwidth per sample is the same at every rate.

#define LS_CU(call) do { const cudaError_t _err = (call); if (_err != cudaSuccess) return _err; } while (0)

// One call of the driver: the engine's receiver, the chunk in hand, and the operations on it.  Each operation that
// differs between the 22050 Hz class and any other geometry tests `general` itself; the driver's loop does not.
struct Run {
  LongPath& lp;
  const SameParams& p;
  const SameTaps& taps; const SameTaps2& taps2; const SameTapsWide& taps_wide;
  uint32_t lanes_per_warp;
  cudaStream_t st;
  bool general;          // any geometry but the 22050 Hz class's (42 taps, DC length 16)
  const int16_t* src;    // the chunk's samples
  uint32_t n, dc_at;     // their number; the position the resident DC-blocker state belongs to
  // The pinned block lp.host carries the control words.  A read-back lands in it and is waited for.  An upload leaves
  // it when the stream gets there: the host may write it again only after a synchronisation that follows the copy.
  // The driver reads a word back before every span, so that holds; upload_span() synchronises first should it not.
  cudaError_t read_back(void* to, const void* from, size_t bytes) {
    LS_CU(cudaMemcpyAsync(to, from, bytes, cudaMemcpyDeviceToHost, st));
    lp.uploading = false;
    return cudaStreamSynchronize(st);
  }
  // an ordinary span's length -> ctrl[3] and, unless off is null, its offset in the chunk -> off
  cudaError_t upload_span(uint32_t span, const uint32_t* off) {
    LongPath::Host& h = *lp.host;
    if (lp.uploading) LS_CU(cudaStreamSynchronize(st));
    lp.uploading = true;
    h.span = span;
    LS_CU(cudaMemcpyAsync(lp.ctrl + 3, &h.span, sizeof h.span, cudaMemcpyHostToDevice, st));
    if (!off) return cudaSuccess;
    h.off = *off;
    return cudaMemcpyAsync(lp.off, &h.off, sizeof h.off, cudaMemcpyHostToDevice, st);
  }
  // A on the 22050 Hz class: len samples from `from` on -> d, the DC-blocker state after the last of them -> dc_next
  cudaError_t launch_dc(uint32_t from, uint32_t len, float* d, uint32_t* dc_next) {
    same_dev::same_long_dc_kernel<<<((len + LS_RUN - 1u) / LS_RUN + 127u) / 128u, 128, 0, st>>>(p, src + from, len, d, dc_next);
    lp.launches += 1;
    return cudaGetLastError();
  }
  // the 22050 Hz class's DC-blocker state words <- `words` (A's, 34 per stream, word-major)
  cudaError_t commit_dc(const uint32_t* words) {
    same_dev::same_long_commit_dc_kernel<<<1, 64, 0, st>>>(p, words);
    lp.launches += 1;
    return cudaGetLastError();
  }
  // The chunk's scratch, and A over the chunk: d, and what the DC-blocker state is later taken from (general: dc0, ma0
  // and fbsum; else dc_next)
  cudaError_t dc_front() {
    const uint32_t runs = (n + LG_RUN - 1u) / LG_RUN;
    LS_CU(lp.d.grow((size_t)n + 64));
    LS_CU(lp.y.grow((size_t)n + 128 + p.ntaps));        // + the demod window before the range
    LS_CU(lp.g.grow((size_t)n + 64));
    LS_CU(lp.soft.grow((size_t)n + 2 * LS_TILE + 64));    // + two tiles: D stages ahead
    LS_CU(lp.g_in.grow(n / LS_BLOCK + 8));
    LS_CU(lp.dc_next.grow((size_t)DCW_WORDS * p.layout.n_pad));
    LS_CU(lp.dc_at.grow((size_t)DCW_WORDS * p.layout.n_pad));
    LS_CU(lp.ctrl.grow(4));
    LS_CU(lp.off.grow(1));
    LS_CU(lp.host.grow(1));
    if (!general) return launch_dc(0, n, lp.d, lp.dc_next);
    LS_CU(lp.ma0.grow((size_t)n + 64));
    LS_CU(lp.fbsum.grow((size_t)n + 2 * LS_TILE + 64));   // + two tiles: the scan stages ahead
    LS_CU(lp.dc0.grow(2 * (size_t)p.dc_len + 3));
    same_dev::same_long_dc_save_kernel<<<1, 512, 0, st>>>(p, lp.dc0);
    same_dev::same_long_ma0_kernel<<<(runs + 127u) / 128u, 128, 0, st>>>(p, src, n, lp.dc0, lp.ma0);
    same_dev::same_long_dfb_kernel<<<(n + 255u) / 256u, 256, 0, st>>>(p, n, lp.dc0, lp.ma0, lp.fbsum);
    same_dev::same_long_fbscan_kernel<<<1, 32, 0, st>>>(p, n, lp.dc0, lp.fbsum);
    same_dev::same_long_dcout_kernel<<<(n + 255u) / 256u, 256, 0, st>>>(p, src, n, lp.dc0, lp.fbsum, lp.d);
    lp.launches += 5;
    return cudaGetLastError();
  }
  // The resident DC-blocker state brought to pos: general, written from dc0, ma0 and fbsum; else A run again from where
  // the state is (its samples go to y, unused between passes) and its end state committed
  cudaError_t dc_to(uint32_t pos) {
    const uint32_t from = dc_at;
    if (from >= pos) return cudaSuccess;
    dc_at = pos;
    if (!general) {
      LS_CU(launch_dc(from, pos - from, lp.y, lp.dc_at));
      return commit_dc(lp.dc_at);
    }
    same_dev::same_long_commit_dcg_kernel<<<1, 512, 0, st>>>(p, src, pos, lp.dc0, lp.ma0, lp.fbsum);
    lp.launches += 1;
    return cudaGetLastError();
  }
  // Up to `span` samples from pos on by an ordinary kernel ("bursts" and "unverified spans" at the top of this file; at
  // any other geometry both go to the generic or wide kernel); pos advances past them
  cudaError_t ordinary_span(uint32_t& pos, uint32_t span, bool locked) {
    const uint32_t at = pos;
    span = std::min(span, n - at);
    pos += span;
    lp.launches += 1; lp.fallback_spans += 1;
    if (locked && !general) {   // tile-fed on A's output: the DC-blocker state words stay as they are (commit_dc 0)
      LS_CU(upload_span(span, nullptr));
      const SameTiles t{lp.d + at, lp.dc_next, span, 1u, 0u};
      return same_launch_rx_tilefed(&p, &taps2, lp.ctrl + 3, &t, st);
    }
    LS_CU(dc_to(at));
    LS_CU(upload_span(span, &at));
    dc_at = pos;
    return same_launch_rx(&p, &taps, &taps2, &taps_wide, general ? GENERIC : PIPE, lanes_per_warp, src, 0, lp.off, lp.ctrl + 3, nullptr, st);
  }
  // The DC-blocker state words at the chunk's end: general, written there unless an ordinary span ended the chunk; else
  // A's end state
  cudaError_t commit() { return general ? dc_to(n) : commit_dc(lp.dc_next); }
  // B + verify + C + D over [pos0, end) of the chunk, their result in ctrl[0..2].  42 taps: the kernels of the 22050 Hz
  // class (taps2); any other tap count: the general instantiations and the wide matched filter (taps_wide).
  cudaError_t pass(uint32_t pos0, uint32_t end) {
    const uint32_t len = end - pos0, blocks = (len + LS_BLOCK - 1u) / LS_BLOCK;
    const bool fast = p.ntaps == FAST_NTAPS;
    LS_CU(cudaMemcpyAsync(lp.ctrl, &end, sizeof(uint32_t), cudaMemcpyHostToDevice, st));   // pageable source: staged
    if (fast)
      same_dev::same_long_agc_kernel<FAST_NTAPS><<<(blocks + 63u) / 64u, 64, 0, st>>>(p, lp.d, pos0, end, lp.y, lp.g, lp.g_in);
    else
      same_dev::same_long_agc_kernel<0><<<(blocks + 63u) / 64u, 64, 0, st>>>(p, lp.d, pos0, end, lp.y, lp.g, lp.g_in);
    if (blocks > 1u)
      same_dev::same_long_verify_kernel<<<(blocks - 1u + 127u) / 128u, 128, 0, st>>>(lp.g, lp.g_in, pos0, end, lp.ctrl);
    if (fast) {
      same_dev::same_long_mf_kernel<<<(len + 255u) / 256u, 256, 0, st>>>(taps2, lp.y, len, lp.soft);
      same_dev::same_long_seq_kernel<FAST_NTAPS><<<1, 64, 0, st>>>(p, lp.soft, lp.y, lp.g, pos0, lp.ctrl);
    } else {
      same_dev::same_long_mf_wide_kernel<<<(len + 255u) / 256u, 256, 0, st>>>(p, taps_wide, lp.y, len, lp.soft);
      same_dev::same_long_seq_kernel<0><<<1, 64, 0, st>>>(p, lp.soft, lp.y, lp.g, pos0, lp.ctrl);
    }
    lp.launches += 4; lp.passes += 1;
    return cudaGetLastError();
  }
};
static_assert(offsetof(LongPath::Host, why) == 2 * sizeof(uint32_t), "ctrl[0..2] are read back in one copy");

}  // namespace

// The driver.  A pass covers [pos, pos + window) of a chunk: the window doubles after every pass that verified all of
// it (a burst-free chunk at a level where hand-overs verify takes one pass) and halves after every verification stop,
// whose unverified span doubles with every stop in a row.  So no pass costs more than a constant times what it
// consumes plus what the pass before it consumed, and input that never verifies runs at the ordinary kernel's speed.
#define LS_CK(call) \
  do { const cudaError_t _err = (call); if (_err != cudaSuccess) return fail(std::string(#call) + ": " + cudaGetErrorString(_err)); } while (0)

int same_long_run(LongPath* lp, const SameParams* p, const SameTaps* taps, const SameTaps2* taps2, const SameTapsWide* taps_wide,
                  uint32_t lanes_per_warp, const int16_t* d_src, uint32_t len, cudaStream_t stream, std::string* error) {
  const auto fail = [error](const std::string& msg) { *error = msg; return SAME_ERR_CUDA; };
  Run r{*lp, *p, *taps, *taps2, *taps_wide, lanes_per_warp, stream, p->ntaps != FAST_NTAPS || p->dc_len != 16, nullptr, 0, 0};
  const auto scaled = [p](uint32_t v) { return (uint32_t)std::max<uint64_t>(1u, (uint64_t)v * p->ntaps / FAST_NTAPS); };
  const uint32_t span_locked = scaled(kLongSpan), span_max = scaled(kLongSpanMax), min_pass = scaled(kLongMinPass);
  for (uint32_t base = 0; base < len; base += kLongChunk) {
    const uint32_t n = std::min(kLongChunk, len - base);
    r.src = d_src + base; r.n = n; r.dc_at = 0;
    LS_CK(r.dc_front());
    LongPath::Host& h = *lp->host;
    uint32_t pos = 0, window = n, stops = 0;
    while (pos < n) {
      LS_CK(r.read_back(&h.flags, p->state32 + (size_t)F_FLAGS * p->layout.n_pad, sizeof(uint32_t)));   // stream 0
      if (h.flags & FLAG_AGC_LOCKED) {   // inside a burst: the samples are the ordinary kernel's, span by span
        LS_CK(r.ordinary_span(pos, span_locked, true));
        continue;
      }
      const uint32_t end = pos + std::min(window, n - pos);
      LS_CK(r.pass(pos, end));
      LS_CK(r.read_back(&h.verified_end, lp->ctrl, 3 * sizeof(uint32_t)));
      if (h.reached < pos || h.reached > end) return fail("long-stream pass reported an impossible position");
      if (h.reached == pos && h.why == 0u) return fail("long-stream pass made no progress");
      pos = h.reached;
      if (h.why != 0u) continue;   // the symbol stages locked the AGC or reset the timing loop: the next round decides
      if (pos == end) {            // all of the range verified
        window = (uint32_t)std::min<uint64_t>(2ull * window, n);
        stops = 0;
        continue;
      }
      // verification stop: the hand-over at pos did not match, and the span after it goes to an ordinary kernel
      window = std::max(min_pass, window / 2u);
      LS_CK(r.ordinary_span(pos, std::min(span_max, span_locked << std::min(stops, 7u)), false));
      stops += 1;
    }
    LS_CK(r.commit());
  }
  return SAME_OK;
}
