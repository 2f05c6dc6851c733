// same_kernels.cu — the receiver kernels: one SAME receiver per lane, 32 independent streams per warp.
//
// Path (SURVEY.md §8a, reference crates/sameold/src/receiver.rs:233-490):
//   A0 s16 -> f32                      samedec app.rs:112
//   A1 DC blocker                      dcblock.rs:45-49,104-108
//   A2 AGC                             agc.rs:72-77
//   A3 demod window                    demod.rs:177-179
//   A4 mark/space matched filter       demod.rs:156-164, filter.rs:363-377
//   A5 TED scheduler + timing loop     receiver.rs:347-360, symsync.rs:198-244,278-322      (same_lane.cuh)
//   A6 code + power squelch            codesquelch.rs:228-304                               (same_lane.cuh)
//   A7 NLMS DFE                        equalize.rs:173-186,249-386                          (same_lane.cuh)
//   A8 framer + link glue              framing.rs:109-197, receiver.rs:407-490              (same_lane.cuh)
//   A9 link/transport events           receiver.rs:245-265,291-333                          (same_lane.cuh, same_transport.cuh)
//
// The chain is numerically chaotic (SURVEY.md §7 H0): results are bit-identical to the oracle or they are different,
// there is no tolerance.  Every f32 operation is therefore one IEEE round-to-nearest operation in the reference's
// order, never contracted, subnormals kept.
//
// Loop structure (all receiver kernels): a warp advances in "rounds".  In each round every lane consumes its own samples
// up to its next timing-error-detector (TED) instant (19..24 samples), then all lanes evaluate the matched filter +
// timing loop together (converged), then the lanes whose TED emitted a symbol run the squelch, and the few lanes that
// completed a byte run the equalizer/framer.  Lane sample cursors drift apart; nothing is shared between lanes.
//
//   same_rx_generic_kernel  any rate / DC length, s16 or f32 samples: literal f32 recursion (needed where the DC blocker
//                           is not exact in integers).
//   22050 Hz class (42 taps, DC length 16, s16 samples) -- shared helpers DcInt / RawFeedT / agc_step / agc_segment /
//   mf_soft, exact integer DC blocker, 16-byte loads, per-lane shared-memory rings [slot][lane], packed FFMA2 filters:
//   same_rx_fast_kernel     one warp per 32 streams (also in tile-fed form behind same_frontend_kernel)
//   same_rx_la_kernel       one warp, DC + AGC in static chunks ahead of the timing loop: 16 resident warps per SM
//   same_rx_ws_kernel       three warps: producer, look-ahead AGC, consumer
//   same_rx_pipe_kernel     five warps: producer, free-running AGC, space filter, timing loop, symbol stages
//   same_frontend_kernel    time-parallel feed-forward stages (A0 + A1) into lane-major f32 tiles, HBM-bound
// The engine (same_engine.cu) picks one from the batch size; every kernel reads and writes the same resident state.
#include <cuda_runtime.h>

#include "same_fast.cuh"
#include "same_internal.h"
#include "same_lane.cuh"

namespace same_dev {

// ----------------------------------------------------------------------------------------------------------------
// Generic kernel.  RW = demod window ring slots (power of two >= ntaps); RD = DC ring slots (power of two >= dc_len)
// ----------------------------------------------------------------------------------------------------------------
// T = sample type at the boundary: int16_t (`sa as f32`, samedec app.rs:112) or float (the reference's own
// iter_events item type, receiver.rs:119-130).
template <int RW, int RD, typename T>
__global__ void __launch_bounds__(32) same_rx_generic_kernel(const __grid_constant__ SameParams p,
                                                             const __grid_constant__ SameTaps taps,
                                                             const T* __restrict__ samples,
                                                             const unsigned long long* __restrict__ offsets,
                                                             const uint32_t* __restrict__ lengths) {
  extern __shared__ float smem[];
  float* win = smem;             // [RW][32]  AGC output window   (A3)
  float* dcf = win + RW * 32;    // [RD][32]  DC feed-forward window (A1)
  float* dcb = dcf + RD * 32;    // [RD][32]  DC feedback window

  const SameLayout& L = p.layout;
  const int lane = threadIdx.x;
  const uint32_t s = blockIdx.x * 32u + lane;
  const bool valid = s < p.n_streams;
  const uint32_t sidx = valid ? s : 0u;  // padded lanes read stream 0's words but never write
  uint32_t* st = p.state32 + sidx;
  StreamBlob* blob = p.blobs + sidx;

  const uint32_t len = valid ? lengths[s] : 0u;
  if (__all_sync(0xffffffffu, len == 0u)) return;
  const T* src = (samples != nullptr && valid) ? samples + offsets[s] : nullptr;

  Lane a;
  lane_load(a, p, st, s);
  float ffsum = __uint_as_float(LANE_ST(st, L, F_DC_FFSUM)), fbsum = __uint_as_float(LANE_ST(st, L, F_DC_FBSUM));
  const int dcl = (int)p.dc_len, ntaps = (int)p.ntaps;
  for (int i = 0; i < dcl; ++i) {
    dcf[i * 32 + lane] = __uint_as_float(LANE_ST(st, L, L.dc_ff + i));
    dcb[i * 32 + lane] = __uint_as_float(LANE_ST(st, L, L.dc_fb + i));
  }
  for (int i = 0; i < ntaps; ++i) win[i * 32 + lane] = __uint_as_float(LANE_ST(st, L, L.win + i));
  int dch = dcl;    // next DC write slot (ring index grows monotonically, masked on use)
  int wh = ntaps;   // next window write slot
  __syncwarp();

  const float inv_len = p.dc_inv_len, gate = p.dc_gate;
  const float bw = p.agc_bw, gmin = p.agc_min, gmax = p.agc_max;

  uint32_t pos = 0;
  int cfire = fire_clock(a.until, a.clock);

  while (__any_sync(0xffffffffu, pos < len)) {
    // ---------------- segment: this lane's samples up to its next TED instant (A0-A3) ----------------
    int nseg = 0;
    if (pos < len) nseg = min(cfire - a.clock, (int)min(len - pos, 1u << 20));
    const int maxseg = __reduce_max_sync(0xffffffffu, nseg);
    for (int k = 0; k < maxseg; ++k) {
      if (k < nseg) {
        float x = src ? (float)src[pos + k] : 0.0f;
        // DC blocker  dcblock.rs:45-49,104-108
        const int ia = ((dch - dcl) & (RD - 1)) * 32 + lane;
        const int iw = (dch & (RD - 1)) * 32 + lane;
        const int ifr = ((dch - dcl + 1) & (RD - 1)) * 32 + lane;
        float aged = dcf[ia];
        dcf[iw] = x;
        ffsum = FADD(ffsum, FSUB(x, aged));
        float ma0 = FMUL(ffsum, inv_len);
        float sig = dcf[ifr];
        float aged2 = dcb[ia];
        dcb[iw] = ma0;
        fbsum = FADD(fbsum, FSUB(ma0, aged2));
        float ma1 = FMUL(fbsum, inv_len);
        dch += 1;
        float d = FSUB(sig, FMUL(gate, ma1));
        // AGC  agc.rs:72-77
        float y = FMUL(d, a.g);
        float u = (a.flags & FLAG_AGC_LOCKED) ? 0.0f : 1.0f;
        a.g = FADD(a.g, FMUL(FMUL(u, FSUB(1.0f, fabsf(y))), bw));
        a.g = rclamp(a.g, gmin, gmax);
        // demod window  demod.rs:177-179
        win[(wh & (RW - 1)) * 32 + lane] = y;
        wh += 1;
      }
    }
    pos += (uint32_t)nseg;
    a.clock += nseg;
    const bool fire = (nseg > 0) && (a.clock == cfire);
    if (!__any_sync(0xffffffffu, fire)) continue;

    // ---------------- TED instant (A4, A5) ----------------
    float soft;
    {
      float mr = 0.0f, mi = 0.0f, sr = 0.0f, si = 0.0f;
      for (int i = 0; i < ntaps; ++i) {  // newest sample pairs with tap 0, sequential accumulation  filter.rs:363-377
        float v = win[((wh - 1 - i) & (RW - 1)) * 32 + lane];
        mr = FADD(mr, FMUL(v, taps.mark_re[i]));
        mi = FADD(mi, FMUL(v, taps.mark_im[i]));
        sr = FADD(sr, FMUL(v, taps.space_re[i]));
        si = FADD(si, FMUL(v, taps.space_im[i]));
      }
      soft = rclamp(FSUB(hypot_fixed(mr, mi), hypot_fixed(sr, si)), -1.0f, 1.0f);  // demod.rs:163
    }
    bool have_sym = false;
    if (fire) {
      const float rem = FSUB(a.until, (float)a.clock);  // receiver.rs:352
      a.clock = 0;
      have_sym = ted_step(a, p, soft, rem);
      cfire = fire_clock(a.until, 0);
    }
    if (!__any_sync(0xffffffffu, have_sym)) continue;

    // ---------------- symbol (A6-A9) ----------------
    if (have_sym) symbol_step(a, p, s, st, blob, a.ted1, a.ted2, a.n0 + pos);
  }

  if (!valid || len == 0u) return;

  // ---- store state ----
  lane_store(a, p, st, a.n0 + len);
  LANE_ST(st, L, F_DC_FFSUM) = __float_as_uint(ffsum);
  LANE_ST(st, L, F_DC_FBSUM) = __float_as_uint(fbsum);
  for (int i = 0; i < dcl; ++i) {  // canonical order: oldest first
    LANE_ST(st, L, L.dc_ff + i) = __float_as_uint(dcf[((dch - dcl + i) & (RD - 1)) * 32 + lane]);
    LANE_ST(st, L, L.dc_fb + i) = __float_as_uint(dcb[((dch - dcl + i) & (RD - 1)) * 32 + lane]);
  }
  for (int i = 0; i < ntaps; ++i) LANE_ST(st, L, L.win + i) = __float_as_uint(win[((wh - ntaps + i) & (RW - 1)) * 32 + lane]);
}

// ----------------------------------------------------------------------------------------------------------------
// Fast kernel: ntaps == 42, dc_len == 16 (22050 Hz).
//
// Shared memory per warp (static, so every access is [register + constant]): d ring [64][32] f32 (DC-blocked samples
// waiting for the AGC) + y ring [128][32] f32 (AGC output; slot j and its mirror j+64 hold the same sample so that the
// 42 newest samples are always readable at descending addresses without a wrap) + the 42 taps as float4.
// Sample j of this chunk lives at slot j & 63 in both rings; [slot][lane] layout: bank == lane, conflict-free for any
// per-lane slot.
//
// `lanes` (1,2,4,...,32) = streams per warp.  Small batches use lane-sparse warps: the per-stream chain is latency
// bound, so spreading few streams over more warps costs nothing and removes most of the divergence (equalizer bytes,
// refill alignment, trip-count spread) from each warp.
// ----------------------------------------------------------------------------------------------------------------

// AGC over one lane's segment of the d ring into the y ring (A2, A3), shared by the single-warp and three-warp kernels.
// Every lane runs the warp's longest trip count.  Samples k0 .. nmin-1 (nmin = warp minimum) need no predicate; in the
// short tail, samples beyond a lane's own segment use bandwidth 0 (g + t*0 == g exactly; the stale d they read is
// finite) and store nothing.  The d loads of a group are issued together so that their latency is paid once per group.
// od / oy: byte offsets ((slot * 128) | lane * 4) of sample k0 in the d ring (mask DMASK) and the y ring (64 slots,
// each y stored at slot j and at its mirror j + 64).
template <uint32_t DMASK>
__device__ __forceinline__ float agc_segment(float g, const float bw_eff, const float gmin, const float gmax,
                                             const uint32_t d_base, const uint32_t y_base, uint32_t od, uint32_t oy, int k,
                                             const int nmin, const int maxseg, const int nseg) {
  constexpr bool ONE = (DMASK == 0x1fffu);   // d ring and y ring of the same size: one running offset serves both
  for (; k + 4 <= nmin; k += 4) {
    float dv[4]; uint32_t oo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      oo[j] = oy; dv[j] = lds_f32(d_base + (ONE ? oy : od));
      if (!ONE) od = (od + 128u) & DMASK;
      oy = (oy + 128u) & 0x1fffu;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float y = agc_step(g, dv[j], bw_eff, gmin, gmax);
      sts_f32_mirrored(y_base + oo[j], y);                                              // demod.rs:177-179
    }
  }
  for (; k < maxseg; k += 2) {
    float dv[2]; uint32_t oo[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      oo[j] = oy; dv[j] = lds_f32(d_base + (ONE ? oy : od));
      if (!ONE) od = (od + 128u) & DMASK;
      oy = (oy + 128u) & 0x1fffu;
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const bool act = (k + j) < nseg;
      const float y = agc_step(g, dv[j], act ? bw_eff : 0.0f, gmin, gmax);
      if (act) sts_f32_mirrored(y_base + oo[j], y);
    }
  }
  return g;
}

// Matched filters (A4) at the sample that ends at ring position `end` (exclusive), packed exact f32 ops:
// fma(v, h, -0) == RN(v*h) and fma(acc, 1, prod) == RN(acc + prod): two separately rounded operations per tap and
// accumulator, as filter.rs:363-377 requires.  The -0 and 1 operands are run-time values (SameParams) so that ptxas
// cannot fold the pair back into one fused multiply-add.  The window is read at descending static offsets from its
// newest slot in the mirrored ring (never wraps).
__device__ __forceinline__ float mf_soft(const float* yring, const float4* tapsm, const int lane, const uint32_t end,
                                         const float2 one2, const float2 negz2) {
  float2 am = make_float2(0.0f, 0.0f), as = make_float2(0.0f, 0.0f);
  int nslot = (int)((end - 1u) & (FAST_RING - 1));
  if (nslot < FAST_NTAPS - 1) nslot += FAST_RING;
  const float* yp = yring + nslot * 32 + lane;
#pragma unroll
  for (int i = 0; i < FAST_NTAPS; ++i) {
    const float v = yp[-i * 32];
    const float4 t = tapsm[i];
    const float2 vv = make_float2(v, v);
    am = __ffma2_rn(am, one2, __ffma2_rn(vv, make_float2(t.x, t.y), negz2));
    as = __ffma2_rn(as, one2, __ffma2_rn(vv, make_float2(t.z, t.w), negz2));
  }
  return rclamp(FSUB(hypot_fixed(am.x, am.y), hypot_fixed(as.x, as.y)), -1.0f, 1.0f);  // demod.rs:163
}

// TILE_FED: the DC-blocked samples come from same_frontend_kernel's lane-major f32 tiles instead of the fused integer
// recursion (measured A/B of DESIGN.md §5; the kernel then only commits the front end's DC state).
template <bool TILE_FED>
__global__ void __launch_bounds__(32, 8) same_rx_fast_kernel(const __grid_constant__ SameParams p,
                                                          const __grid_constant__ SameTaps2 taps,
                                                          const int16_t* __restrict__ samples,
                                                          const unsigned long long* __restrict__ offsets,
                                                          const uint32_t* __restrict__ lengths, const uint32_t lanes,
                                                          const SameTiles tiles) {
  __shared__ float dring[FAST_RING * 32];
  __shared__ float yring[2 * FAST_RING * 32];
  __shared__ float4 tapsm[FAST_NTAPS];

  const SameLayout& L = p.layout;
  const int lane = threadIdx.x;
  const uint32_t s = blockIdx.x * lanes + lane;
  const bool valid = (uint32_t)lane < lanes && s < p.n_streams;
  const uint32_t sidx = valid ? s : 0u;
  uint32_t* st = p.state32 + sidx;
  StreamBlob* blob = p.blobs + sidx;

  const uint32_t len = valid ? lengths[s] : 0u;
  if (__all_sync(0xffffffffu, len == 0u)) return;
  const int16_t* src = (!TILE_FED && samples != nullptr && valid) ? samples + offsets[s] : nullptr;
  // tile-fed: sample n of this lane is tiles.d[(tile * n_max + n) * stride + lane] (lanes == 32 only; stride 32 =
  // lane-major tiles, stride 1 = one dense stream)
  const uint32_t tstride = TILE_FED ? tiles.stride : 0u;
  const float* tsrc = TILE_FED ? tiles.d + (size_t)blockIdx.x * tiles.n_max * tstride + (uint32_t)lane : nullptr;

  Lane a;
  lane_load(a, p, st, s);

  DcInt dc;
  RawFeed feed;
  if (!TILE_FED) {
    dc_load(dc, st, L);
    feed.init(src, 0u, len);
  }
  // demod window -> y ring slots of samples -42..-1 (and mirrors); d ring starts finite (stale slots are read, never used)
  for (int i = 0; i < FAST_RING; ++i) dring[i * 32 + lane] = 0.0f;
  for (int i = 0; i < FAST_NTAPS; ++i) {
    const float v = __uint_as_float(LANE_ST(st, L, L.win + i));
    const int slot = (i - FAST_NTAPS) & (FAST_RING - 1);
    yring[slot * 32 + lane] = v;
    yring[(slot + FAST_RING) * 32 + lane] = v;
  }
  for (int i = lane; i < FAST_NTAPS; i += 32)
    tapsm[i] = make_float4(taps.mark[i].x, taps.mark[i].y, taps.space[i].x, taps.space[i].y);
  __syncwarp();

  const float bw = p.agc_bw, gmin = p.agc_min, gmax = p.agc_max;
  const float2 one2 = make_float2(p.f_one, p.f_one), negz2 = make_float2(p.f_negzero, p.f_negzero);
  const uint32_t d_base = smem_u32(dring), y_base = smem_u32(yring);

  uint32_t pos = 0;   // samples consumed by the AGC/TED side
  uint32_t rp = 0;    // samples produced into the d ring (multiple of 32 except after the final partial chunk)
  bool dc_windows_stored = false;
  int cfire = fire_clock(a.until, a.clock);
  // Byte-phase alignment: a lane whose squelch hands out a byte parks (consumes nothing) until the next round whose
  // index is a multiple of 16, where all parked lanes run the equalizer/framer together.  Bytes are 16 TED instants
  // apart, so after its first wait a lane's bytes keep falling on those rounds: the warp pays for the byte path once
  // per 16 rounds instead of once per in-burst lane.
  // TED-phase alignment: the timing loop emits a symbol at every second TED instant (symsync.rs:280).  A lane whose
  // instant counter is out of step with the round counter sits out one round, after which all lanes of the warp emit
  // their symbols on the even rounds: the symbol-rate stages (loop filter, squelch, link bookkeeping) then run every
  // second round for the whole warp instead of every round for half of its lanes.  Byte rounds are even rounds, so
  // byte parking (an even number of rounds) keeps the phase.  Neither kind of parking changes what a lane computes.
  uint32_t pend = 0;       // SYM_BYTE_READY | SYM_ADJUSTED while parked
  uint32_t round_ctr = 0;

  while (__any_sync(0xffffffffu, pos < len || pend != 0u)) {
    round_ctr += 1;
    const bool byte_round = (round_ctr & 15u) == 0u;
    // ---------------- refill: raw s16 -> exact DC-blocked f32 into the d ring (A0, A1) ----------------
    // One uniform decision per warp keeps the lanes' refills aligned (a lane-private decision would make nearly every
    // round pay for a refill executed by a few lanes).
    while (__any_sync(0xffffffffu, (rp - pos) < 24u && rp < len && pend == 0u)) {
      const bool take = (rp < len) && (rp - pos) <= (uint32_t)(FAST_RING - FAST_CHUNK);
      const uint32_t nnew = take ? min((uint32_t)FAST_CHUNK, len - rp) : 0u;
      float* dst = dring + (rp & (FAST_RING - 1)) * 32 + lane;  // rp % 32 == 0: the chunk never wraps
      if (TILE_FED) {
        if (nnew) {
          const float* q = tsrc + (size_t)rp * tstride;
          float v[FAST_CHUNK];
#pragma unroll
          for (int i = 0; i < FAST_CHUNK; ++i) v[i] = (i < (int)nnew) ? __ldg(q + (size_t)i * tstride) : 0.0f;
#pragma unroll
          for (int i = 0; i < FAST_CHUNK; ++i) dst[i * 32] = v[i];
          rp += nnew;
        }
      } else if (nnew == FAST_CHUNK) {
        // ---- full chunk: everything static, no per-sample predicates ----
        uint32_t cur[FAST_CHUNK / 2];
        feed.take_full(cur, rp, len);
        dc_chunk<FAST_CHUNK>(dc, cur, [&](int i, float d) { dst[i * 32] = d; });
        rp += FAST_CHUNK;
      } else if (nnew) {
        // ---- final partial chunk of this submit (rp reaches len): scalar loads, per-sample predicates; the DC
        // windows are final now and are stored right here, rotated back into canonical order ----
        uint32_t cur[FAST_CHUNK / 2];
        feed.take_partial(cur, rp, nnew);
        dc_chunk_partial<FAST_CHUNK>(dc, cur, (int)nnew, [&](int i, float d) { dst[i * 32] = d; });
        dc_store_after_partial<FAST_CHUNK>(dc, cur, nnew, DcToState{st, L});
        dc_windows_stored = true;
        rp += nnew;
      }
      __syncwarp();
    }

    // ---------------- segment: AGC over this lane's samples up to its next TED instant (A2, A3) ----------------
    int nseg = 0;
    if (pos < len && pend == 0u) nseg = min(cfire - a.clock, (int)(rp - pos));
    if (((a.tedcnt ^ round_ctr) & 1u) != 0u) nseg = 0;   // TED-phase alignment, see above
    const int maxseg = __reduce_max_sync(0xffffffffu, nseg);
    const int nmin = __reduce_min_sync(0xffffffffu, nseg);
    const float bw_eff = (a.flags & FLAG_AGC_LOCKED) ? 0.0f : bw;   // (!locked as f32) * (1-|y|) * bw   agc.rs:74
    const uint32_t o = ((pos << 7) & 0x1f80u) | ((uint32_t)lane << 2);
    a.g = agc_segment<0x1fffu>(a.g, bw_eff, gmin, gmax, d_base, y_base, o, o, 0, nmin, maxseg, nseg);
    pos += (uint32_t)nseg;
    a.clock += nseg;
    const bool fire = (nseg > 0) && (a.clock == cfire);
    bool have_sym = false;
    if (__any_sync(0xffffffffu, fire)) {
      // ---------------- TED instant: matched filters (A4), timing loop (A5) ----------------
      const float soft = mf_soft(yring, tapsm, lane, pos, one2, negz2);
      if (fire) {
        const float rem = FSUB(a.until, (float)a.clock);  // receiver.rs:352
        a.clock = 0;
        have_sym = ted_step(a, p, soft, rem);
        cfire = fire_clock(a.until, 0);
      }
    }

    // ---------------- symbol: squelch now (A6), byte path (A7-A9) on the aligned rounds ----------------
    if (have_sym) pend = symbol_squelch(a, p, s, st, blob, a.ted1, a.ted2, a.n0 + pos);
    if (byte_round && __any_sync(0xffffffffu, pend != 0u)) {
      if (pend != 0u) {
        symbol_byte(a, p, s, st, blob, (pend & SYM_ADJUSTED) != 0u, a.n0 + pos);
        pend = 0u;
      }
    }
  }

  if (!valid || len == 0u) return;

  // ---- store state (same f32 layout as the generic kernel) ----
  lane_store(a, p, st, a.n0 + len);
  if (TILE_FED) {
    // commit the DC-blocker state the front-end kernel left for this stream (it could not write the state words
    // itself: its first run of each stream was still reading them)
    if (tiles.commit_dc)
      for (int w = 0; w < DCW_WORDS; ++w) DcToState{st, L}((uint32_t)w, tiles.dc_next[(size_t)w * L.n_pad + s]);
  } else if (!dc_windows_stored) {
    dc_store(dc, DcToState{st, L});
  }
  for (int i = 0; i < FAST_NTAPS; ++i)
    LANE_ST(st, L, L.win + i) = __float_as_uint(yring[((int)(len + i - FAST_NTAPS) & (FAST_RING - 1)) * 32 + lane]);
}

// ----------------------------------------------------------------------------------------------------------------
// Look-ahead kernel: the single-warp receiver for the THROUGHPUT regime (many more warps than schedulers).
//
// What the profiles of same_rx_fast_kernel say (profiles/ncu_r02_fast_65536x5.*): 57.7 warp-instructions per sample, but
// only 0.49 issue slots used, because each SM sub-partition holds two warps (254 registers, 25 KB of shared memory per
// warp) and one warp on its own issues 0.3 instructions per cycle (dependent AGC and accumulator chains).  Residency
// comes in steps of four warps per SM (the register file is split over the four sub-partitions): 16 resident warps need
// <= 128 registers and <= 13.2 KB per warp.  This kernel gets there by dropping the d ring and the mirror slots:
//   * The AGC no longer waits for the timing loop.  It depends on the rest of the receiver only through the lock flag
//     (agc.rs:74), so DC blocker and AGC run together in static 8-sample chunks (one 16-byte load), straight from
//     registers into the y ring, until they have passed the lane's next TED instant — at most 7 samples of look-ahead.
//     The look-ahead is exact speculation: if the symbol stages at that instant flip the lock flag, the tail of the last
//     chunk is recomputed from its saved inputs (8 d values in registers, starting gain, per-sample flag mask).  No d
//     ring, no per-sample loop of run-time length, and the independent DC arithmetic of later samples fills the issue
//     slots under the gain chain.  Each lane streams along its own row, so the 128-byte line two ahead is pulled into
//     L2 with a prefetch (without it the first load of every line is the kernel's top stall).
//   * DC-blocker history: the last 16 raw samples stay in registers (packed pairs), the last 16 values of S1 live in a
//     2 KB shared-memory ring (static offsets from a per-chunk base).
//   * y ring: 64 slots, no mirror (8 KB): the matched filter wraps every tap address into the ring.
// Same arithmetic, same rounds, same parking rules and same resident state as the other fast kernels.
// Measured (profiles/README.md, round 2): 65 536 x 20 s 97 ms against 116 ms; 49 152: 83 / 109; 131 072 x 10 s: 88 / 101;
// below 8 blocks per SM the fast kernel's fewer instructions win (32 768: 58 / 81).  Tried and dropped: cold lane
// state through the state words around each symbol stage (131 ms), redo inputs in shared memory (108), byte path as a
// real call (115), 168 registers / 12 warps per SM (142: the 13.8 warps per SM of 65 536 streams then leave a tail wave).
// ----------------------------------------------------------------------------------------------------------------
#define LA_CHUNK 8
#define LA_MAXREG 128
constexpr int LA_MF_UNROLL_N = 14;   // matched-filter unroll: 3 x 14 taps (the full unroll costs registers the loop cannot spare)

__global__ void __maxnreg__(LA_MAXREG) same_rx_la_kernel(const __grid_constant__ SameParams p,
                                                         const __grid_constant__ SameTaps2 taps,
                                                         const int16_t* __restrict__ samples,
                                                         const unsigned long long* __restrict__ offsets,
                                                         const uint32_t* __restrict__ lengths, const uint32_t lanes) {
  __shared__ float yring[FAST_RING * 32];
  __shared__ int s1ring[FAST_DCL * 32];
  __shared__ float4 tapsm[FAST_NTAPS];

  const SameLayout& L = p.layout;
  const int lane = threadIdx.x;
  const uint32_t s = blockIdx.x * lanes + lane;
  const bool valid = (uint32_t)lane < lanes && s < p.n_streams;
  const uint32_t sidx = valid ? s : 0u;
  uint32_t* st = p.state32 + sidx;
  StreamBlob* blob = p.blobs + sidx;

  const uint32_t len = valid ? lengths[s] : 0u;
  if (__all_sync(0xffffffffu, len == 0u)) return;
  const int16_t* src = (samples != nullptr && valid) ? samples + offsets[s] : nullptr;
  const bool aligned = (reinterpret_cast<uintptr_t>(src) & 15u) == 0;

  Lane a;
  lane_load(a, p, st, s);

  // ---- DC blocker state as integers (see DcInt): sums and raw history in registers, S1 history in shared memory ----
  int S1 = __float2int_rn(__uint_as_float(LANE_ST(st, L, F_DC_FFSUM)));
  int S2 = __float2int_rn(__uint_as_float(LANE_ST(st, L, F_DC_FBSUM)) * 16.0f);
  uint32_t rawh[FAST_DCL / 2];
#pragma unroll
  for (int i = 0; i < FAST_DCL / 2; ++i) {
    const int lo = __float2int_rn(__uint_as_float(LANE_ST(st, L, L.dc_ff + 2 * i)));
    const int hi = __float2int_rn(__uint_as_float(LANE_ST(st, L, L.dc_ff + 2 * i + 1)));
    rawh[i] = ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16);
  }
  for (int i = 0; i < FAST_DCL; ++i)     // the S1 of sample n lives in slot n & 15: samples -16..-1 -> slots 0..15
    s1ring[i * 32 + lane] = __float2int_rn(__uint_as_float(LANE_ST(st, L, L.dc_fb + i)) * 16.0f);
  for (int i = 0; i < FAST_RING; ++i) yring[i * 32 + lane] = 0.0f;
  for (int i = 0; i < FAST_NTAPS; ++i)   // demod window -> y ring slots of samples -42..-1
    yring[((i - FAST_NTAPS) & (FAST_RING - 1)) * 32 + lane] = __uint_as_float(LANE_ST(st, L, L.win + i));
  for (int i = lane; i < FAST_NTAPS; i += 32)
    tapsm[i] = make_float4(taps.mark[i].x, taps.mark[i].y, taps.space[i].x, taps.space[i].y);
  __syncwarp();

  const float bw = p.agc_bw, gmin = p.agc_min, gmax = p.agc_max;
  const float2 one2 = make_float2(p.f_one, p.f_one), negz2 = make_float2(p.f_negzero, p.f_negzero);
  const uint32_t y_lane = smem_u32(yring) + ((uint32_t)lane << 2);
  const uint32_t s1_lane = smem_u32(s1ring) + ((uint32_t)lane << 2);

  uint32_t pos = 0;        // samples consumed by the timing loop
  uint32_t rp = 0;         // samples through DC blocker + AGC (pos <= rp <= pos + 7 between rounds)
  float g = a.g;           // AGC gain after sample rp - 1
  // the last chunk, kept for the exact redo after a lock flip: inputs, gain before it, per-sample lock flags, length
  float dlast[LA_CHUNK];
#pragma unroll
  for (int i = 0; i < LA_CHUNK; ++i) dlast[i] = 0.0f;
  float g0 = g;
  uint32_t lockmask = 0, nlast = 0;
  bool dc_windows_stored = false;
  int4 nx = make_int4(0, 0, 0, 0);
  bool pf_ok = src != nullptr && aligned && len >= (uint32_t)LA_CHUNK;
  if (pf_ok) nx = __ldg(reinterpret_cast<const int4*>(src));

  int cfire = fire_clock(a.until, a.clock);
  uint32_t pend = 0;       // byte-phase / TED-phase alignment: see same_rx_fast_kernel
  uint32_t round_ctr = 0;

  while (__any_sync(0xffffffffu, pos < len || pend != 0u)) {
    round_ctr += 1;
    const bool byte_round = (round_ctr & 15u) == 0u;
    int nseg = 0;
    if (pos < len && pend == 0u) nseg = min(cfire - a.clock, (int)(len - pos));
    if (((a.tedcnt ^ round_ctr) & 1u) != 0u) nseg = 0;   // TED-phase alignment
    const uint32_t target = pos + (uint32_t)nseg;

    // ---------------- DC blocker + AGC in 8-sample chunks until this lane's target is covered (A0-A3) ----------------
    while (__any_sync(0xffffffffu, rp < target)) {
      if (rp < target) {
        const uint32_t nnew = min((uint32_t)LA_CHUNK, len - rp);
        const bool locked = (a.flags & FLAG_AGC_LOCKED) != 0u;
        const float bw_eff = locked ? 0.0f : bw;           // (!locked as f32) * (1-|y|) * bw   agc.rs:74
        const uint32_t ys = y_lane + ((rp & (FAST_RING - 1)) << 7);   // rp % 8 == 0: a chunk never wraps in either ring
        const uint32_t ss = s1_lane + ((rp & (FAST_DCL - 1)) << 7);
        uint32_t cur[LA_CHUNK / 2];
        g0 = g; lockmask = locked ? 0xffu : 0u; nlast = nnew;
        if (nnew == LA_CHUNK) {
          if (pf_ok) { cur[0] = nx.x; cur[1] = nx.y; cur[2] = nx.z; cur[3] = nx.w; }
          else {
#pragma unroll
            for (int i = 0; i < LA_CHUNK / 2; ++i) {
              const uint32_t lo = src ? (uint32_t)(uint16_t)src[rp + 2 * i] : 0u;
              const uint32_t hi = src ? (uint32_t)(uint16_t)src[rp + 2 * i + 1] : 0u;
              cur[i] = lo | (hi << 16);
            }
          }
          pf_ok = src != nullptr && aligned && (len - rp) >= 2u * LA_CHUNK;
          if (pf_ok) nx = __ldg(reinterpret_cast<const int4*>(src + rp + LA_CHUNK));
          // each lane streams along its own row: pull the 128-byte line two ahead (64 samples each) into L2 early
          if (pf_ok && (rp & 63u) == 0u && (len - rp) > 192u) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + rp + 128));
#pragma unroll
          for (int i = 0; i < LA_CHUNK; ++i) {
            const int x = s16_at(cur, i), x16 = s16_at(rawh, i), x15 = s16_at(rawh, i + 1);
            S1 += x - x16;                                         // dcblock.rs:106 (ff)
            int s1old;
            asm volatile("ld.shared.s32 %0, [%1];" : "=r"(s1old) : "r"(ss + (uint32_t)(i << 7)));
            S2 += S1 - s1old;                                      // dcblock.rs:106 (fb)
            asm volatile("st.shared.s32 [%0], %1;" ::"r"(ss + (uint32_t)(i << 7)), "r"(S1) : "memory");
            const float d = (float)((x15 << 8) - S2) * 0.00390625f;  // dcblock.rs:48
            dlast[i] = d;
            sts_f32(ys + (uint32_t)(i << 7), agc_step(g, d, bw_eff, gmin, gmax));   // agc.rs:72-77, demod.rs:177-179
          }
#pragma unroll
          for (int i = 0; i < FAST_DCL / 4; ++i) { rawh[i] = rawh[i + FAST_DCL / 4]; rawh[i + FAST_DCL / 4] = cur[i]; }
          rp += LA_CHUNK;
        } else {
          // ---- the final, partial chunk of this submit: scalar loads, per-sample predicates; the DC windows are final
          // and go to the state words right here, rotated back into canonical order (oldest first) ----
#pragma unroll
          for (int i = 0; i < LA_CHUNK / 2; ++i) cur[i] = 0u;
#pragma unroll
          for (int i = 0; i < LA_CHUNK; ++i) {
            const uint32_t v = (src && i < (int)nnew) ? (uint32_t)(uint16_t)src[rp + i] : 0u;
            cur[i >> 1] |= (i & 1) ? (v << 16) : v;
          }
#pragma unroll
          for (int i = 0; i < LA_CHUNK; ++i) {
            if (i < (int)nnew) {
              const int x = s16_at(cur, i), x16 = s16_at(rawh, i), x15 = s16_at(rawh, i + 1);
              S1 += x - x16;
              const int s1old = s1ring[((rp + i) & (FAST_DCL - 1)) * 32 + lane];
              S2 += S1 - s1old;
              s1ring[((rp + i) & (FAST_DCL - 1)) * 32 + lane] = S1;
              const float d = (float)((x15 << 8) - S2) * 0.00390625f;
              dlast[i] = d;
              sts_f32(ys + (uint32_t)(i << 7), agc_step(g, d, bw_eff, gmin, gmax));
            }
          }
          // ff window = the last 16 of (rawh ++ cur[0..nnew)); static register indices, run-time word numbers
#pragma unroll
          for (int i = 0; i < FAST_DCL; ++i)
            if (i >= (int)nnew) LANE_ST(st, L, L.dc_ff + ((uint32_t)i - nnew)) = __float_as_uint((float)s16_at(rawh, i));
#pragma unroll
          for (int i = 0; i < LA_CHUNK; ++i)
            if (i < (int)nnew) LANE_ST(st, L, L.dc_ff + ((uint32_t)(FAST_DCL + i) - nnew)) = __float_as_uint((float)s16_at(cur, i));
          dc_windows_stored = true;
          rp += nnew;
        }
      }
      __syncwarp();
    }

    // ---------------- the timing loop's side: advance to the target, TED instant (A4, A5) ----------------
    pos = target;
    a.clock += nseg;
    const bool fire = (nseg > 0) && (a.clock == cfire);
    const uint32_t lock_before = a.flags & FLAG_AGC_LOCKED;
    bool have_sym = false;
    if (__any_sync(0xffffffffu, fire)) {
      float2 am = make_float2(0.0f, 0.0f), as = make_float2(0.0f, 0.0f);
      uint32_t e = (pos - 1u) << 7;             // running byte offset of the tap's sample, wrapped into the ring per tap
#pragma unroll LA_MF_UNROLL_N
      for (int i = 0; i < FAST_NTAPS; ++i) {    // filter.rs:363-377 with packed exact f32 ops, see mf_soft
        const float v = lds_f32(y_lane + (e & 0x1f80u));
        e -= 128u;
        const float4 t = tapsm[i];
        const float2 vv = make_float2(v, v);
        am = __ffma2_rn(am, one2, __ffma2_rn(vv, make_float2(t.x, t.y), negz2));
        as = __ffma2_rn(as, one2, __ffma2_rn(vv, make_float2(t.z, t.w), negz2));
      }
      const float soft = rclamp(FSUB(hypot_fixed(am.x, am.y), hypot_fixed(as.x, as.y)), -1.0f, 1.0f);  // demod.rs:163
      if (fire) {
        const float rem = FSUB(a.until, (float)a.clock);  // receiver.rs:352
        a.clock = 0;
        have_sym = ted_step(a, p, soft, rem);
        cfire = fire_clock(a.until, 0);
      }
    }
    // ---------------- symbol: squelch now (A6), byte path (A7-A9) on the aligned rounds ----------------
    if (have_sym) {
      pend = symbol_squelch(a, p, s, st, blob, a.ted1, a.ted2, a.n0 + pos);
    }
    if (byte_round && __any_sync(0xffffffffu, pend != 0u)) {
      if (pend != 0u) {
        symbol_byte(a, p, s, st, blob, (pend & SYM_ADJUSTED) != 0u, a.n0 + pos);
        pend = 0u;
      }
    }
    // ---------------- the lock flag flipped: the look-ahead samples pos .. rp-1 were speculated with the old flag ----------------
    const bool flipped = (a.flags & FLAG_AGC_LOCKED) != lock_before;
    if (__any_sync(0xffffffffu, flipped)) {
      if (flipped) {
        const uint32_t base = rp - nlast;                  // first sample of the last chunk
        const uint32_t idx = pos - base;                   // samples of it that are final (pos >= base: look-ahead < 8)
        const uint32_t newbits = (a.flags & FLAG_AGC_LOCKED) ? 0xffu : 0u;
        lockmask = (lockmask & ((1u << idx) - 1u)) | (newbits & ~((1u << idx) - 1u));
        const uint32_t ys = y_lane + ((base & (FAST_RING - 1)) << 7);
        float gr = g0;
#pragma unroll
        for (int i = 0; i < LA_CHUNK; ++i) {
          if (i < (int)nlast) {
            const float din = dlast[i];
            const float y = agc_step(gr, din, ((lockmask >> i) & 1u) ? 0.0f : bw, gmin, gmax);
            if (i >= (int)idx) sts_f32(ys + (uint32_t)(i << 7), y);
          }
        }
        g = gr;
      }
      __syncwarp();
    }
  }

  if (!valid || len == 0u) return;

  // ---- store state (same f32 layout as the generic kernel); pos == rp == len: g is the gain at the sample counter ----
  a.g = g;
  lane_store(a, p, st, a.n0 + len);
  LANE_ST(st, L, F_DC_FFSUM) = __float_as_uint((float)S1);
  LANE_ST(st, L, F_DC_FBSUM) = __float_as_uint((float)S2 * 0.0625f);
  if (!dc_windows_stored) {
#pragma unroll
    for (int i = 0; i < FAST_DCL; ++i) LANE_ST(st, L, L.dc_ff + i) = __float_as_uint((float)s16_at(rawh, i));
  }
  for (int i = 0; i < FAST_DCL; ++i)
    LANE_ST(st, L, L.dc_fb + i) = __float_as_uint((float)s1ring[((len + i) & (FAST_DCL - 1)) * 32 + lane] * 0.0625f);
  for (int i = 0; i < FAST_NTAPS; ++i)
    LANE_ST(st, L, L.win + i) = __float_as_uint(yring[((int)(len + i - FAST_NTAPS) & (FAST_RING - 1)) * 32 + lane]);
}

// ----------------------------------------------------------------------------------------------------------------
// Front-end kernel (feed-forward stages A0 + A1, time-parallel): s16 stream-major -> exact DC-blocked f32 in lane-major
// tiles  d[(tile * n_max + n) * 32 + lane],  tile = 32 consecutive streams — one 128-byte line per (tile, sample), the
// layout a warp of the loop kernel reads with one coalesced request.  HBM-bound: 2 B read + 4 B written per sample.
//
// One warp = one tile x one run of FE_RUN (2048) samples; lane = stream.  The DC blocker has finite memory (31 samples), so a
// run that does not start the chunk warms up on the 32 samples before it (integer recursion from zero is exact after
// 31 samples) and is independent of every other run; the first run of a stream starts from the resident state.  Reads:
// each lane streams along its own row with 16-byte loads (L1 keeps the 128-byte lines between a lane's consecutive
// loads); writes: 32 lanes x 4 B = one full line per sample.  The run that ends a stream's chunk writes the new DC
// state to tiles.dc_next (committed to the state words by the tile-fed loop kernel).
// ----------------------------------------------------------------------------------------------------------------
#define FE_RUN 2048      // samples per run: 32 of warm-up per run = 1.6 % extra reads (512: 83.9 %, 2048: 87.4 % of HBM peak)
#define FE_WARPS 4
__global__ void __launch_bounds__(FE_WARPS * 32) same_frontend_kernel(const __grid_constant__ SameParams p,
                                                                      const int16_t* __restrict__ samples,
                                                                      const unsigned long long* __restrict__ offsets,
                                                                      const uint32_t* __restrict__ lengths,
                                                                      const SameTiles tiles) {
  const SameLayout& L = p.layout;
  const int lane = threadIdx.x & 31;
  const uint32_t run_blocks = (tiles.n_max + FE_RUN * FE_WARPS - 1u) / (FE_RUN * FE_WARPS);   // 1-D grid: tile-major
  const uint32_t tile = blockIdx.x / run_blocks;
  const uint32_t run = (blockIdx.x - tile * run_blocks) * FE_WARPS + (threadIdx.x >> 5);
  const uint32_t s = tile * 32u + (uint32_t)lane;
  const bool valid = s < p.n_streams;
  const uint32_t len = valid ? lengths[s] : 0u;
  const uint32_t r0 = run * FE_RUN;
  if (r0 >= len) return;
  const uint32_t r1 = min(r0 + (uint32_t)FE_RUN, len);
  const int16_t* src = samples + offsets[s];
  uint32_t* st = p.state32 + s;

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
    dc_chunk<FAST_CHUNK>(dc, cur, [](int, float) {});          // warm-up: exact from the 32nd sample on
  }
  float* dst = tiles.d + ((size_t)tile * tiles.n_max + r0) * 32u + (uint32_t)lane;
  uint32_t c = r0;
  for (; c + FAST_CHUNK <= r1; c += FAST_CHUNK, dst += FAST_CHUNK * 32) {
    feed.take_full(cur, c, len);
    dc_chunk<FAST_CHUNK>(dc, cur, [&](int i, float d) { __stcs(dst + i * 32, d); });
  }
  const auto to_next = [&](uint32_t w, uint32_t bits) { tiles.dc_next[(size_t)w * L.n_pad + s] = bits; };
  if (c < r1) {                                      // r1 == len: the partial tail of the chunk
    const uint32_t nnew = r1 - c;
    feed.take_partial(cur, c, nnew);
    dc_chunk_partial<FAST_CHUNK>(dc, cur, (int)nnew, [&](int i, float d) { __stcs(dst + i * 32, d); });
    dc_store_after_partial<FAST_CHUNK>(dc, cur, nnew, to_next);
  } else if (r1 == len) {
    dc_store(dc, to_next);
  }
}

// ----------------------------------------------------------------------------------------------------------------
// Three-warp kernel: the same algorithm as same_rx_fast_kernel, split over three warps per 32 streams.
//
//   warp 1 (producer)    raw s16 -> exact DC-blocked f32 into the d ring (A0, A1): vector loads with one chunk of
//                        prefetch, integer recursion in registers.  Runs ahead of the consumer by up to the ring size.
//   warp 2 (look-ahead)  while the consumer is busy with round r, the AGC recurrence of the next WS_SPEC samples
//                        (the segment of round r+1) into the y ring, the gain after every sample into a gain ring
//                        (A2, A3).  Exact speculation: see the comment at its loop.
//   warp 0 (consumer)    picks up the look-ahead (or runs the recurrence itself when it does not apply), matched
//                        filters, timing loop, squelch, byte path, events (A4-A9).
//
// The warps sit on different schedulers of the SM, so the refill (global-load latency + ~11 instructions per sample)
// and the AGC chain leave the consumer's critical path.  Hand-off: per-lane counters in shared memory and three named
// barriers used in strict alternation — no polling, no sleeping:
//     consumer:    bar.sync B_DATA, B_LA -> segment -> publish pos, gain, flag -> bar.arrive B_POS -> filters/TED/symbol
//     producer:    bar.sync B_POS -> refill lanes that have room -> publish rp -> bar.arrive B_DATA
//     look-ahead:  bar.sync B_POS -> recurrence over WS_SPEC samples              -> bar.arrive B_LA
// so the refill and the look-ahead for round r+1 overlap the matched-filter half of round r, and after every refill
// each lane holds at least one full segment (>= 32 samples) of data.
// ----------------------------------------------------------------------------------------------------------------
#define WS_DRING 128       // d ring slots of the warp-specialised kernel
#define WS_SPEC 22         // look-ahead samples: 42 taps + 22 new samples just fit the 64-slot y ring; covers most whole segments
#define WS_BAR_DATA 1      // producer -> consumer            (64 threads)
#define WS_BAR_POS 2       // consumer -> producer, look-ahead (96 threads)
#define WS_BAR_LA 3        // look-ahead -> consumer          (64 threads)
#define WS_THREADS 96
__device__ __forceinline__ void ws_bar_sync(int id, int n = 64) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void ws_bar_arrive(int id, int n = 64) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// Producer warp of the warp-specialised kernels: raw s16 -> exact DC-blocked f32 into the d ring (A0, A1).  Each round:
// wait for the position the consumer may still need samples from (bar_pos), refill every lane that has room for a whole
// 32-sample chunk, publish rp, arrive on bar_data.  Stores the DC-blocker state of the lane when the consumer signals the end.
template <uint32_t DRING>   // d ring slots (power of two)
__device__ __forceinline__ void ws_producer(const SameParams& p, uint32_t* st, const int16_t* src, const uint32_t len,
                                            const int lane, const bool valid, float* dring, volatile uint32_t* sh_rp,
                                            volatile uint32_t* sh_pos, volatile uint32_t* sh_done, const int bar_pos,
                                            const int bar_pos_n, const int bar_data, const int bar_data_n) {
  const SameLayout& L = p.layout;
  DcInt dc;
  RawFeed feed;
  dc_load(dc, st, L);
  feed.init(src, 0u, len);
  uint32_t rp = 0;
  bool dc_windows_stored = false;
  bool first = true;
  while (true) {
    if (!first) {
      ws_bar_sync(bar_pos, bar_pos_n);   // the consumer finished a segment and published pos
      if (*sh_done) break;
    }
    first = false;
    const uint32_t cpos = sh_pos[lane];
    // every lane with room for a whole chunk takes one: afterwards it holds >= 32 samples, more than any segment
    const bool take = (rp < len) && (rp - cpos) <= DRING - FAST_CHUNK;
    const uint32_t nnew = take ? min((uint32_t)FAST_CHUNK, len - rp) : 0u;
    float* dst = dring + (rp & (DRING - 1)) * 32 + lane;  // rp % 32 == 0: the chunk never wraps
    if (nnew == FAST_CHUNK) {
      uint32_t cur[FAST_CHUNK / 2];
      feed.take_full(cur, rp, len);
      dc_chunk<FAST_CHUNK>(dc, cur, [&](int i, float d) { dst[i * 32] = d; });
      rp += FAST_CHUNK;
    } else if (nnew) {
      uint32_t cur[FAST_CHUNK / 2];
      feed.take_partial(cur, rp, nnew);
      dc_chunk_partial<FAST_CHUNK>(dc, cur, (int)nnew, [&](int i, float d) { dst[i * 32] = d; });
      dc_store_after_partial<FAST_CHUNK>(dc, cur, nnew, DcToState{st, L});   // final DC windows, back in canonical order
      dc_windows_stored = true;
      rp += nnew;
    }
    sh_rp[lane] = rp;
    __threadfence_block();             // d values and rp visible before the consumer is released
    ws_bar_arrive(bar_data, bar_data_n);
  }
  if (valid && len != 0u && !dc_windows_stored) dc_store(dc, DcToState{st, L});
}

// up to four blocks per SM (engine policy): 12 warps = three per sub-partition -> at most 168 registers
__global__ void __launch_bounds__(WS_THREADS, 4) same_rx_ws_kernel(const __grid_constant__ SameParams p,
                                                        const __grid_constant__ SameTaps2 taps,
                                                        const int16_t* __restrict__ samples,
                                                        const unsigned long long* __restrict__ offsets,
                                                        const uint32_t* __restrict__ lengths, const uint32_t lanes) {
  __shared__ float dring[WS_DRING * 32];   // 128 slots: room for a whole segment of look-ahead (speculative AGC)
  __shared__ float yring[2 * FAST_RING * 32];
  __shared__ float4 tapsm[FAST_NTAPS];
  __shared__ float gring[WS_SPEC * 32];      // look-ahead AGC gain after each look-ahead sample
  __shared__ volatile uint32_t sh_rp[32];    // samples produced per lane (written by the producer warp)
  __shared__ volatile uint32_t sh_pos[32];   // samples consumed per lane (written by the consumer warp)
  __shared__ volatile uint32_t sh_done;      // consumer -> producer: no more rounds
  __shared__ volatile float sh_la_g[32];     // consumer -> look-ahead: AGC gain at pos
  __shared__ volatile uint32_t sh_la_rq[32]; // consumer -> look-ahead: bit 0 look-ahead wanted, bit 1 AGC locked

  const SameLayout& L = p.layout;
  const int lane = threadIdx.x & 31;
  const int role = threadIdx.x >> 5;         // 0 consumer, 1 producer, 2 look-ahead
  const uint32_t s = blockIdx.x * lanes + lane;
  const bool valid = (uint32_t)lane < lanes && s < p.n_streams;
  const uint32_t sidx = valid ? s : 0u;
  uint32_t* st = p.state32 + sidx;
  StreamBlob* blob = p.blobs + sidx;

  const uint32_t len = valid ? lengths[s] : 0u;
  if (__syncthreads_and(len == 0u)) return;   // block-uniform
  const int16_t* src = (samples != nullptr && valid) ? samples + offsets[s] : nullptr;

  // ---- shared set-up (both warps) ----
  for (int i = role; i < WS_DRING; i += 3) dring[i * 32 + lane] = 0.0f;   // stale slots are read, never used: keep them finite
  if (role == 2) {
    sh_la_rq[lane] = 0u;
  } else if (role == 0) {
    for (int i = 0; i < FAST_NTAPS; ++i) {   // demod window -> y ring slots of samples -42..-1 (and mirrors)
      const float v = __uint_as_float(LANE_ST(st, L, L.win + i));
      const int slot = (i - FAST_NTAPS) & (FAST_RING - 1);
      yring[slot * 32 + lane] = v;
      yring[(slot + FAST_RING) * 32 + lane] = v;
    }
    sh_pos[lane] = 0u;
    if (lane == 0) sh_done = 0u;
  } else {
    for (int i = lane; i < FAST_NTAPS; i += 32)
      tapsm[i] = make_float4(taps.mark[i].x, taps.mark[i].y, taps.space[i].x, taps.space[i].y);
    sh_rp[lane] = 0u;
  }
  __syncthreads();

  if (role == 1) {
    ws_producer<WS_DRING>(p, st, src, len, lane, valid, dring, sh_rp, sh_pos, &sh_done, WS_BAR_POS, WS_THREADS, WS_BAR_DATA, 64);
    return;
  }

  const float bw = p.agc_bw, gmin = p.agc_min, gmax = p.agc_max;
  const uint32_t d_base = smem_u32(dring), y_base = smem_u32(yring);
  const uint32_t g_base = smem_u32(gring) + ((uint32_t)lane << 2);

  if (role == 2) {
    // ============================================== look-ahead ==============================================
    // While the consumer runs the matched filters, timing loop and symbol stages of round r, this warp evaluates the
    // AGC recurrence of the next WS_SPEC samples — normally the whole segment of round r+1 — into the y ring, keeping
    // the gain after every sample (gring).  The AGC does not depend on the timing loop, only on the lock flag, so the
    // look-ahead is exact unless the symbol processing of round r flips that flag (a few times per burst) or parks
    // the lane; the consumer then throws it away and runs the recurrence itself.
    ws_bar_arrive(WS_BAR_LA);                // nothing to wait for in the first round
    while (true) {
      ws_bar_sync(WS_BAR_POS, WS_THREADS);
      if (sh_done) break;
      const uint32_t rq = sh_la_rq[lane];
      if (__any_sync(0xffffffffu, (rq & 1u) != 0u)) {
        // lanes that did not ask run along and store too: their slots pos .. pos+21 hold samples nobody has produced
        // yet (they alias samples pos-64 .. pos-43, older than the 42-tap window) and are rewritten before use
        const float bw_eff = (rq & 2u) ? 0.0f : bw;
        float gs = sh_la_g[lane];
        const uint32_t lpos = sh_pos[lane];
        uint32_t sd = ((lpos << 7) & 0x3f80u) | ((uint32_t)lane << 2);
        uint32_t sy = ((lpos << 7) & 0x1f80u) | ((uint32_t)lane << 2);
        float dsp[WS_SPEC];
#pragma unroll
        for (int j = 0; j < WS_SPEC; ++j) { dsp[j] = lds_f32(d_base + sd); sd = (sd + 128u) & 0x3fffu; }
#pragma unroll
        for (int j = 0; j < WS_SPEC; ++j) {
          const float y = agc_step(gs, dsp[j], bw_eff, gmin, gmax);                         // agc.rs:72-77
          sts_f32_mirrored(y_base + sy, y);
          sts_f32(g_base + (uint32_t)(j * 128), gs);
          sy = (sy + 128u) & 0x1fffu;
        }
      }
      __threadfence_block();
      ws_bar_arrive(WS_BAR_LA);
    }
    return;
  }

  // ================================================= consumer =================================================
  Lane a;
  lane_load(a, p, st, s);
  const float2 one2 = make_float2(p.f_one, p.f_one), negz2 = make_float2(p.f_negzero, p.f_negzero);

  uint32_t pos = 0;
  int cfire = fire_clock(a.until, a.clock);
  uint32_t pend = 0;       // SYM_BYTE_READY | SYM_ADJUSTED while parked (byte-phase alignment, see same_rx_fast_kernel)
  uint32_t round_ctr = 0;
  bool pre_ok = false;     // gring / the y ring already hold samples pos .. pos+WS_SPEC-1 (look-ahead warp)

  while (true) {
    ws_bar_sync(WS_BAR_DATA);              // the producer's refill for this round is complete and visible
    ws_bar_sync(WS_BAR_LA);                // ... and so is the look-ahead
    if (!__any_sync(0xffffffffu, pos < len || pend != 0u)) {
      if (lane == 0) sh_done = 1u;
      __threadfence_block();
      ws_bar_arrive(WS_BAR_POS, WS_THREADS);
      break;
    }
    // ---------------- segment: AGC over this lane's samples up to its next TED instant (A2, A3) ----------------
    const uint32_t rp = sh_rp[lane];
    int nseg = 0;
    round_ctr += 1;
    const bool byte_round = (round_ctr & 15u) == 0u;
    if (pos < len && pend == 0u) nseg = min(cfire - a.clock, (int)(rp - pos));
    if (((a.tedcnt ^ round_ctr) & 1u) != 0u) nseg = 0;   // TED-phase alignment (see same_rx_fast_kernel)
    const int maxseg = __reduce_max_sync(0xffffffffu, nseg);
    const int nmin = __reduce_min_sync(0xffffffffu, nseg);
    const float bw_eff = (a.flags & FLAG_AGC_LOCKED) ? 0.0f : bw;   // (!locked as f32) * (1-|y|) * bw   agc.rs:74
    // use the look-ahead only if every lane that works this round has one (uniform start index keeps the loop simple)
    const bool use_pre = __all_sync(0xffffffffu, nseg == 0 || pre_ok);
    float g = a.g;
    if (use_pre && nseg > 0) g = lds_f32(g_base + (uint32_t)((min(nseg, WS_SPEC) - 1) << 7));
    const int k0 = use_pre ? WS_SPEC : 0;
    const uint32_t od = (((pos + (uint32_t)k0) << 7) & 0x3f80u) | ((uint32_t)lane << 2);   // d ring: 128 slots
    const uint32_t oy = (((pos + (uint32_t)k0) << 7) & 0x1f80u) | ((uint32_t)lane << 2);   // y ring: 64 slots + mirror
    g = agc_segment<0x3fffu>(g, bw_eff, gmin, gmax, d_base, y_base, od, oy, k0, nmin, maxseg, nseg);
    if (nseg > 0) a.g = g;
    pre_ok = false;
    pos += (uint32_t)nseg;
    a.clock += nseg;
    const bool fire = (nseg > 0) && (a.clock == cfire);
    const uint32_t lock_before = a.flags & FLAG_AGC_LOCKED;
    // ask for the look-ahead of the next segment when this lane is at a TED instant and has the samples for it
    const bool spec = fire && (rp - pos) >= (uint32_t)WS_SPEC && (len - pos) >= (uint32_t)WS_SPEC;
    sh_pos[lane] = pos;      // lets the producer reuse the ring slots behind pos
    sh_la_g[lane] = a.g;
    sh_la_rq[lane] = (spec ? 1u : 0u) | (lock_before ? 2u : 0u);
    __threadfence_block();
    ws_bar_arrive(WS_BAR_POS, WS_THREADS);
    bool have_sym = false;
    if (__any_sync(0xffffffffu, fire)) {
      // ---------------- TED instant: matched filters (A4, packed exact f32 ops), timing loop (A5) ----------------
      const float soft = mf_soft(yring, tapsm, lane, pos, one2, negz2);
      if (fire) {
        const float rem = FSUB(a.until, (float)a.clock);  // receiver.rs:352
        a.clock = 0;
        have_sym = ted_step(a, p, soft, rem);
        cfire = fire_clock(a.until, 0);
      }
    }
    // ---------------- symbol: squelch now (A6), byte path (A7-A9) on the aligned rounds ----------------
    if (have_sym) pend = symbol_squelch(a, p, s, st, blob, a.ted1, a.ted2, a.n0 + pos);
    if (byte_round && __any_sync(0xffffffffu, pend != 0u)) {
      if (pend != 0u) {
        symbol_byte(a, p, s, st, blob, (pend & SYM_ADJUSTED) != 0u, a.n0 + pos);
        pend = 0u;
      }
    }
    // the look-ahead stands if this lane is not parked and its AGC lock flag is what the look-ahead assumed
    if (spec && pend == 0u && (a.flags & FLAG_AGC_LOCKED) == lock_before) pre_ok = true;
  }

  if (!valid || len == 0u) return;
  lane_store(a, p, st, a.n0 + pos);
  for (int i = 0; i < FAST_NTAPS; ++i)
    LANE_ST(st, L, L.win + i) = __float_as_uint(yring[((int)(pos + i - FAST_NTAPS) & (FAST_RING - 1)) * 32 + lane]);
}

// ----------------------------------------------------------------------------------------------------------------
// Pipelined kernel: the receiver of 32 streams spread over five warps, so that the per-round critical path is
// "segment bookkeeping -> one matched filter -> timing loop" and the symbol stages run beside it.
//
//   warp P   producer   raw s16 -> exact DC-blocked f32 (d ring), refilled up to PK_RING samples past the oldest
//                       position the timing warp may still roll back to                                    A0, A1
//   warp A   AGC        free-running gain recurrence, up to PK_LEAD samples ahead of the timing warp:
//                       y ring + gain ring (gain after every sample)                                       A2, A3
//   warp X   space      the space matched filter and its magnitude at the timing warp's TED instant        A4
//   warp T   timing     picks the gain that belongs to its position, mark matched filter and magnitude,
//                       timing loop; every symbol goes into a per-lane ring of records                     A4, A5
//   warp Y   symbols    consumes each lane's records in order: squelch, equalizer, framer, transport       A6-A9
//
// The AGC depends on the timing warp only through the lock flag (agc.rs:74), so it runs ahead speculatively and exactly:
// whenever T's flag flips, or the AGC warp has not got far enough, T runs the recurrence itself with the same
// arithmetic (fallback below) and tells the AGC warp to restart from its position and gain.
// Lockstep rounds of P, A, X and T on four named barriers:
//   T: sync DONE -> roll-back -> segment -> publish pos -> arrive POS -> publish (gain, flag, restart) -> arrive AGC
//      -> mark -> sync SPACE -> TED, record
//   X: sync POS -> space filter at pos -> arrive SPACE     P: sync POS -> refill -> arrive DONE
//   A: sync AGC -> recurrence -> arrive DONE
//
// The symbol stages feed back into the timing loop only through SameReceiver::end() (TED state reset, locks cleared) and
// an adjusted squelch acquire (AGC and bandwidth locked), receiver.rs:423-438, 479-490: a dozen symbols per stream-minute.
// So T runs ahead of Y without waiting, each record carrying T's state right after that symbol's TED step.  Y never
// speculates: its lane state is the sequential receiver's, and so is every global write it makes.  When Y's symbol k
// changes what T uses, Y posts that state (a roll-back) and waits for that lane; T resumes the lane from symbol k with
// it and drops the records it wrote after k.  Records carry no epoch: T publishes its head count together with the
// number of roll-backs it applied, and Y reads a lane's records only once that number matches its own.
// T waits for Y only when a lane's ring is full (PK_REC records) or the lane is PK_TLEAD samples past its oldest
// unconfirmed symbol: the rings keep everything a roll-back needs (d from that symbol on, y from 42 samples before it).
// ----------------------------------------------------------------------------------------------------------------
#define PK_THREADS 160
#define PK_RING 512        // d, gain and y ring slots (one running offset serves all three)
#define PK_OMASK ((PK_RING - 1) * 128u)   // ring byte offset ((slot * 32 + lane) * 4) mask for the slot part
#define PK_YMIRROR (FAST_NTAPS - 1)       // y slots 0..40 are mirrored at PK_RING + slot: a 42-tap window never wraps
#ifndef PK_REC
#define PK_REC 8           // records per lane: T's maximum lead over Y in symbols (power of two)
#endif
#define PK_TLEAD (PK_RING - 128)   // T's maximum lead in samples over its oldest unconfirmed symbol (see the AGC stores)
#define PK_RECW 8          // words per record: pos, zero, sym, until, pavg, pinst, ted0, g
#define PK_PARK 4          // Y rounds a squelched byte may wait for more lanes' bytes (the byte path runs once per warp)
#define PK_DYN_SMEM ((3 * PK_RING + PK_YMIRROR) * 32 * 4 + PK_RECW * PK_REC * 32 * 4)   // gain | y + mirror | d | records
#define PK_LEAD 48         // the AGC warp stays at most this far ahead of the timing warp
#define PK_ADV 32          // ... and advances at most this much per round
#define PK_BAR_POS 1       // T -> X, P        (96 threads)   position published
#define PK_BAR_DONE 2      // A, P -> T        (96 threads)
#define PK_BAR_SPACE 3     // X -> T           (64 threads)
#define PK_BAR_AGC 4       // T -> A           (64 threads)   gain / flag / restart published
#define PK_LOCKS (FLAG_AGC_LOCKED | FLAG_BW_LOCKED)

// |matched filter output| over the 42 samples that end at sample index `end` (exclusive); taps from the constant bank.
// One rounded multiply and one rounded add per component and tap, newest sample first (demod.rs:156-163).
__device__ __forceinline__ float pk_mag(const float* yring, const float2* __restrict__ h, const int lane,
                                        const uint32_t end, const float f_one, const float f_negzero) {
  int nslot = (int)((end - 1u) & (PK_RING - 1));
  if (nslot < PK_YMIRROR) nslot += PK_RING;
  const float* yp = yring + nslot * 32 + lane;
  // packed exact f32 ops (see mf_soft): 3 instructions per tap instead of 5; measured 60.9 against 62.3 ms on config 3
  // although the dependent FFMA2 chain is slower per step than FADD (6 against 4 cycles) -- the warp was issue-bound
  const float2 one2 = make_float2(f_one, f_one), negz2 = make_float2(f_negzero, f_negzero);
  float2 acc = make_float2(0.0f, 0.0f);
#pragma unroll
  for (int i = 0; i < FAST_NTAPS; ++i) {
    const float v = yp[-i * 32];
    acc = __ffma2_rn(acc, one2, __ffma2_rn(make_float2(v, v), h[i], negz2));
  }
  return hypot_fixed(acc.x, acc.y);
}

// y of ring byte offset o (slot * 128 + lane * 4) into the y ring, and into its mirror for slots 0..40
__device__ __forceinline__ void pk_store_y(const uint32_t y_lane, const uint32_t o, const float y) {
  asm volatile("{\n\t.reg .pred m;\n\tsetp.lt.u32 m, %1, %3;\n\tst.shared.f32 [%0], %2;\n\t@m st.shared.f32 [%0+%4], %2;\n\t}"
               ::"r"(y_lane + o), "r"(o), "f"(y), "n"(PK_YMIRROR * 128), "n"(PK_RING * 128) : "memory");
}

// one block per SM at most (engine policy): every register the role code wants.  Warp i runs on scheduler i mod 4:
// T has one to itself, Y shares one with the producer, which waits most of the time.
__global__ void __launch_bounds__(PK_THREADS, 1) same_rx_pipe_kernel(const __grid_constant__ SameParams p,
                                                                  const __grid_constant__ SameTaps2 taps,
                                                                  const int16_t* __restrict__ samples,
                                                                  const unsigned long long* __restrict__ offsets,
                                                                  const uint32_t* __restrict__ lengths,
                                                                  const uint32_t lanes) {
  // gring[PK_RING][32] | yring[PK_RING + PK_YMIRROR][32] | dring[PK_RING][32] | rec[PK_RECW][PK_REC][32]
  extern __shared__ float pk_dyn[];
  float* const gring = pk_dyn;
  float* const yring = gring + PK_RING * 32;
  float* const dring = yring + (PK_RING + PK_YMIRROR) * 32;
  float* const rec = dring + PK_RING * 32;
  __shared__ volatile float sh_space[32];    // |space filter| at pos                                (X)
  __shared__ volatile uint32_t sh_rp[32];    // samples produced per lane                            (P)
  __shared__ volatile uint32_t sh_apos[32];  // samples AGC'd per lane                               (A)
  __shared__ volatile uint32_t sh_pos[32];   // samples consumed per lane                            (T)
  __shared__ volatile uint32_t sh_low[32];   // oldest position T may roll back to: P refills from it (T)
  __shared__ volatile float sh_g[32];        // AGC gain at pos                                      (T)
  __shared__ volatile uint32_t sh_rq[32];    // bit 0 restart the AGC at pos, bit 1 AGC locked       (T)
  __shared__ volatile uint32_t sh_frp[32];   // rp as T saw it at the top of the round               (T)
  __shared__ volatile uint32_t sh_head[32];  // records written (low 16 bits) | roll-backs applied << 16   (T)
  __shared__ volatile uint32_t sh_tail[32];  // records confirmed (low 16 bits)                      (Y)
  __shared__ volatile uint32_t sh_rbreq[32]; // roll-backs requested (low 16 bits)                   (Y)
  __shared__ volatile uint32_t sh_rb[10][32];   // roll-back: pos, g, until, pavg, pinst, ted0..2, tedcnt | locks, head (Y)
  __shared__ volatile uint32_t sh_fin[10][32];  // T's state at the end: pos, g, clock, until, pavg, pinst, ted0..2, tedcnt
  __shared__ volatile uint32_t sh_done;

  const SameLayout& L = p.layout;
  const int lane = threadIdx.x & 31;
  enum { R_Y = 0, R_T = 1, R_X = 2, R_A = 3, R_P = 4 };
  const int role = threadIdx.x >> 5;
  const uint32_t s = blockIdx.x * lanes + lane;
  const bool valid = (uint32_t)lane < lanes && s < p.n_streams;
  const uint32_t sidx = valid ? s : 0u;
  uint32_t* st = p.state32 + sidx;
  StreamBlob* blob = p.blobs + sidx;

  const uint32_t len = valid ? lengths[s] : 0u;
  if (__syncthreads_and(len == 0u)) return;   // block-uniform
  const int16_t* src = (samples != nullptr && valid) ? samples + offsets[s] : nullptr;

  // ---- shared set-up ----
  for (int i = role; i < PK_RING; i += 5) dring[i * 32 + lane] = 0.0f;   // stale slots are read, never used: keep them finite
  if (role == R_T) {
    for (int i = 0; i < FAST_NTAPS; ++i) {   // demod window -> y ring slots of samples -42..-1 (470..511: no mirror)
      const float v = __uint_as_float(LANE_ST(st, L, L.win + i));
      yring[((i - FAST_NTAPS) & (PK_RING - 1)) * 32 + lane] = v;
    }
    sh_pos[lane] = 0u;
    sh_low[lane] = 0u;
    sh_head[lane] = 0u;
    if (lane == 0) sh_done = 0u;
  } else if (role == R_A) {
    sh_apos[lane] = 0u;
    for (int i = 0; i < PK_RING - FAST_NTAPS; ++i) yring[i * 32 + lane] = 0.0f;   // keep never-written slots finite
  } else if (role == R_X) {
    for (int i = 0; i < PK_YMIRROR; ++i) yring[(PK_RING + i) * 32 + lane] = 0.0f;
    sh_space[lane] = 0.0f;
  } else if (role == R_Y) {
    sh_tail[lane] = 0u;
    sh_rbreq[lane] = 0u;
  } else {
    sh_rp[lane] = 0u;
  }
  __syncthreads();

  if (role == R_P) {
    ws_producer<PK_RING>(p, st, src, len, lane, valid, dring, sh_rp, sh_low, &sh_done, PK_BAR_POS, 96, PK_BAR_DONE, 96);
    return;
  }

  const float bw = p.agc_bw, gmin = p.agc_min, gmax = p.agc_max;
  const uint32_t d_lane = smem_u32(dring) + ((uint32_t)lane << 2);
  const uint32_t g_lane = smem_u32(gring) + ((uint32_t)lane << 2);
  const uint32_t y_lane = smem_u32(yring) + ((uint32_t)lane << 2);

  if (role == R_A) {
    // ================================================= AGC =================================================
    uint32_t apos = 0;
    float ag = 0.0f;
    ws_bar_arrive(PK_BAR_DONE, 96);
    while (true) {
      ws_bar_sync(PK_BAR_AGC, 64);
      if (sh_done) break;
      const uint32_t rq = sh_rq[lane];
      const uint32_t fpos = sh_pos[lane];
      const uint32_t rp = sh_frp[lane];  // as of the previous round: the refill running now only adds to it
      if (rq & 1u) { apos = fpos; ag = sh_g[lane]; }
      const float bw_eff = (rq & 2u) ? 0.0f : bw;    // (!locked as f32) * (1-|y|) * bw   agc.rs:74
      int n = min((int)PK_ADV, min((int)(rp - apos), (int)(fpos + PK_LEAD - apos)));
      n = max(n, 0);
      const int nmax = __reduce_max_sync(0xffffffffu, n);
      float g = ag;
      // 8 samples per step, the d values of the next step prefetched.  One running byte offset (ring slot * 128 +
      // lane * 4) addresses all three rings.  Every lane stores all nmax (rounded up to 8) samples: what lies beyond
      // its own n is overwritten with the right values before anything reads it, and lands at most 79 samples ahead
      // of T.  T stays within PK_TLEAD = PK_RING - 128 samples of its oldest unconfirmed symbol, so these stores never
      // reach the 42 samples before that symbol, which a roll-back needs.
      // Software pipeline, distance 2: the d value of sample j+2 is loaded right after the stores of sample j-1.
      // The explicit shared-memory accesses keep their program order, so the stores have to issue in the shadow of
      // the gain chain (one dependent op every 4-5 cycles) instead of in a bunch after it.
      uint32_t o0 = (apos & (PK_RING - 1)) << 7, o1 = (o0 + 128u) & PK_OMASK;
      float d0 = lds_f32(d_lane + o0), d1 = lds_f32(d_lane + o1);
      for (int k = 0; k < nmax; k += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t o2 = (o1 + 128u) & PK_OMASK;
          const float d2 = lds_f32(d_lane + o2);
          const float y = agc_step(g, d0, bw_eff, gmin, gmax);                            // agc.rs:72-77
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(g_lane + o0), "f"(g) : "memory");
          pk_store_y(y_lane, o0, y);
          o0 = o1; o1 = o2; d0 = d1; d1 = d2;
        }
      }
      if (n > 0) {
        apos += (uint32_t)n;
        ag = gring[((apos - 1u) & (PK_RING - 1)) * 32 + lane];          // the gain after this lane's last sample
      }
      sh_apos[lane] = apos;
      __threadfence_block();
      ws_bar_arrive(PK_BAR_DONE, 96);
    }
    return;
  }

  if (role == R_X) {
    // ============================================== space filter ==============================================
    while (true) {
      ws_bar_sync(PK_BAR_POS, 96);
      if (sh_done) break;
      sh_space[lane] = pk_mag(yring, taps.space, lane, sh_pos[lane], p.f_one, p.f_negzero);
      __threadfence_block();
      ws_bar_arrive(PK_BAR_SPACE, 64);
    }
    return;
  }

  if (role == R_Y) {
    // ============================================== symbol stages ==============================================
    Lane a;
    lane_load(a, p, st, s);
    uint32_t tail = 0, ep = 0;   // records confirmed; roll-backs requested
    bool wait_ack = false;       // a roll-back is posted and T has not applied it yet: consume nothing of this lane
    uint32_t park = 0;           // SYM_BYTE_READY | SYM_ADJUSTED of a symbol whose byte path waits (see PK_PARK)
    uint32_t r_pos = 0, r_lock = 0;
    float r_g = 0.0f;
    int age = 0;
    while (true) {
      const uint32_t hw = sh_head[lane];
      if (wait_ack && (hw >> 16) == (ep & 0xffffu)) {      // T resumed from the roll-back's symbol: it is confirmed
        wait_ack = false;
        tail += 1u;
        ls_publish(&sh_tail[lane], tail & 0xffffu);
      }
      const bool have = !wait_ack && park == 0u && (hw >> 16) == (ep & 0xffffu) && ((hw - tail) & 0xffffu) != 0u;
      const bool any_have = __any_sync(0xffffffffu, have);
      const bool any_park = __any_sync(0xffffffffu, park != 0u);
      if (!any_have && !any_park) {
        if (sh_done) break;   // T finishes only when every record is confirmed
        continue;
      }
      bool sym_done = false;
      if (any_have) {
        __threadfence_block();   // with T's fence before the head word: the records are complete
        if (have) {
          const float* q = rec + (tail & (PK_REC - 1)) * 32 + lane;
          r_pos = __float_as_uint(q[0]);
          const float zero = q[1 * PK_REC * 32], sym = q[2 * PK_REC * 32];
          a.until = q[3 * PK_REC * 32]; a.pavg = q[4 * PK_REC * 32]; a.pinst = q[5 * PK_REC * 32];
          a.ted0 = q[6 * PK_REC * 32]; a.ted1 = zero; a.ted2 = sym; a.tedcnt = 1u;
          r_g = q[7 * PK_REC * 32];
          r_lock = a.flags & PK_LOCKS;
          park = symbol_squelch(a, p, s, st, blob, zero, sym, a.n0 + r_pos);
          sym_done = park == 0u;
        }
      }
      // the byte path of parked lanes: when no lane has a new record, or after PK_PARK rounds
      if (__any_sync(0xffffffffu, park != 0u) && (!any_have || ++age >= PK_PARK)) {
        age = 0;
        if (park != 0u) {
          symbol_byte(a, p, s, st, blob, (park & SYM_ADJUSTED) != 0u, a.n0 + r_pos);
          park = 0u;
          sym_done = true;
        }
      }
      if (sym_done) {
        if ((a.flags & PK_LOCKS) != r_lock || a.tedcnt != 1u) {
          // end() or an adjusted acquire changed the timing loop's state: T resumes from this symbol with it
          sh_rb[0][lane] = r_pos; sh_rb[1][lane] = __float_as_uint(r_g); sh_rb[2][lane] = __float_as_uint(a.until);
          sh_rb[3][lane] = __float_as_uint(a.pavg); sh_rb[4][lane] = __float_as_uint(a.pinst);
          sh_rb[5][lane] = __float_as_uint(a.ted0); sh_rb[6][lane] = __float_as_uint(a.ted1);
          sh_rb[7][lane] = __float_as_uint(a.ted2); sh_rb[8][lane] = a.tedcnt | (a.flags & PK_LOCKS) << 16;
          sh_rb[9][lane] = (tail + 1u) & 0xffffu;
          ep += 1u;
          ls_publish(&sh_rbreq[lane], ep & 0xffffu);
          wait_ack = true;
          atomicAdd(&p.counters[3], 1u);
        } else {
          tail += 1u;
          ls_publish(&sh_tail[lane], tail & 0xffffu);
        }
      }
    }
    if (!valid || len == 0u) return;
    __threadfence_block();
    const uint32_t pos = sh_fin[0][lane];
    a.g = __uint_as_float(sh_fin[1][lane]); a.clock = (int)sh_fin[2][lane];
    a.until = __uint_as_float(sh_fin[3][lane]); a.pavg = __uint_as_float(sh_fin[4][lane]);
    a.pinst = __uint_as_float(sh_fin[5][lane]); a.ted0 = __uint_as_float(sh_fin[6][lane]);
    a.ted1 = __uint_as_float(sh_fin[7][lane]); a.ted2 = __uint_as_float(sh_fin[8][lane]); a.tedcnt = sh_fin[9][lane];
    lane_store(a, p, st, a.n0 + pos);
    for (int i = 0; i < FAST_NTAPS; ++i)
      LANE_ST(st, L, L.win + i) = __float_as_uint(yring[((int)(pos + i - FAST_NTAPS) & (PK_RING - 1)) * 32 + lane]);
    return;
  }

  // ================================================= timing =================================================
  Lane a;
  lane_load(a, p, st, s);
  uint32_t pos = 0;
  int cfire = fire_clock(a.until, a.clock);
  uint32_t round_ctr = 0;
  uint32_t head = 0, ep = 0;   // records written; roll-backs applied
  bool la_valid = false;       // the AGC warp's chain continues this lane's exact state under the current lock flag

  while (true) {
    ws_bar_sync(PK_BAR_DONE, 96);           // refill and AGC of the previous round are complete and visible
    // ---------------- roll-back: resume from the symbol Y names, with the state its symbol stages left ----------------
    const uint32_t rq_ep = sh_rbreq[lane];
    const bool rb = rq_ep != ep;
    if (__any_sync(0xffffffffu, rb)) {
      __threadfence_block();
      if (rb) {
        pos = sh_rb[0][lane]; a.g = __uint_as_float(sh_rb[1][lane]); a.until = __uint_as_float(sh_rb[2][lane]);
        a.pavg = __uint_as_float(sh_rb[3][lane]); a.pinst = __uint_as_float(sh_rb[4][lane]);
        a.ted0 = __uint_as_float(sh_rb[5][lane]); a.ted1 = __uint_as_float(sh_rb[6][lane]);
        a.ted2 = __uint_as_float(sh_rb[7][lane]);
        const uint32_t w = sh_rb[8][lane];
        a.tedcnt = w & 0xffffu;
        a.flags = (a.flags & ~PK_LOCKS) | (w >> 16);
        head = sh_rb[9][lane];
        a.clock = 0;                         // the symbol's TED instant, where cfire was computed (before end())
        cfire = fire_clock(a.until, 0);
        la_valid = false;
        ep = rq_ep;
      }
    }
    const uint32_t tail = sh_tail[lane];
    const uint32_t inflight = (head - tail) & 0xffffu;
    if (!__any_sync(0xffffffffu, pos < len || inflight != 0u)) break;
    const uint32_t low = inflight ? __float_as_uint(rec[(tail & (PK_REC - 1)) * 32 + lane]) : pos;
    // ---------------- segment: this lane's samples up to its next TED instant (A2, A3) ----------------
    const uint32_t rp = sh_rp[lane];
    const uint32_t apos = sh_apos[lane];
    int nseg = 0;
    round_ctr += 1;
    if (pos < len && inflight < (uint32_t)PK_REC)
      nseg = min(min(cfire - a.clock, (int)(rp - pos)), (int)(low + PK_TLEAD - pos));
    if (((a.tedcnt ^ round_ctr) & 1u) != 0u) nseg = 0;   // TED-phase alignment: Y gets the lanes' records together
    const uint32_t lock_now = a.flags & FLAG_AGC_LOCKED;
    const bool use_la = la_valid && (int)(apos - pos) >= nseg;
    const bool need_fb = nseg > 0 && !use_la;
    if (__any_sync(0xffffffffu, need_fb)) {
      // fallback: run the recurrence here (start of a chunk, after a roll-back, AGC warp not far enough)
      const int nfb = __reduce_max_sync(0xffffffffu, need_fb ? nseg : 0);
      const float bw_eff = lock_now ? 0.0f : bw;
      float g = a.g;
      for (int k = 0; k < nfb; ++k) {
        const bool act = need_fb && k < nseg;
        const uint32_t o = ((pos + (uint32_t)k) & (PK_RING - 1)) << 7;
        const float dv = lds_f32(d_lane + o);
        float gn = g;
        const float y = agc_step(gn, dv, bw_eff, gmin, gmax);
        if (act) {
          g = gn;
          pk_store_y(y_lane, o, y);
        }
      }
      if (need_fb) a.g = g;
    }
    // the position first: it is all the space-filter and producer warps wait for
    sh_pos[lane] = pos + (uint32_t)nseg;
    sh_low[lane] = low;
    __threadfence_block();
    sh_head[lane] = (head & 0xffffu) | (ep << 16);   // the records of earlier rounds, behind the fence above
    ws_bar_arrive(PK_BAR_POS, 96);
    if (use_la && nseg > 0) a.g = lds_f32(g_lane + (((pos + (uint32_t)nseg - 1u) & (PK_RING - 1)) << 7));
    pos += (uint32_t)nseg;
    a.clock += nseg;
    const bool fire = (nseg > 0) && (a.clock == cfire);
    const bool restart = !la_valid || need_fb;
    la_valid = true;
    sh_g[lane] = a.g;
    sh_frp[lane] = rp;
    sh_rq[lane] = (restart ? 1u : 0u) | (lock_now ? 2u : 0u);
    __threadfence_block();
    ws_bar_arrive(PK_BAR_AGC, 64);

    // ---------------- TED instant (A4, A5): mark here, space from warp X ----------------
    // what the timing loop needs besides the soft symbol is computed first, off the critical path
    const float rem = FSUB(a.until, (float)a.clock);                         // receiver.rs:352
    const float off = rclamp(rem, -0.5f, 0.5f);                              // symsync.rs:220
    const float offq = __fdiv_rn(off, p.spt);                                // symsync.rs:225
    asm volatile("" ::"f"(offq));
    const float mag_m = pk_mag(yring, taps.mark, lane, pos, p.f_one, p.f_negzero);
    asm volatile("" ::"f"(mag_m));          // keep the mark magnitude ahead of the wait for the space magnitude
    ws_bar_sync(PK_BAR_SPACE, 64);
    if (fire) {
      const float soft = rclamp(FSUB(mag_m, sh_space[lane]), -1.0f, 1.0f);   // demod.rs:163
      a.clock = 0;
      if (ted_step(a, p, soft, off, offq)) {
        float* q = rec + (head & (PK_REC - 1)) * 32 + lane;                   // published with the next round's head
        q[0] = __uint_as_float(pos); q[1 * PK_REC * 32] = a.ted1; q[2 * PK_REC * 32] = a.ted2;
        q[3 * PK_REC * 32] = a.until; q[4 * PK_REC * 32] = a.pavg; q[5 * PK_REC * 32] = a.pinst;
        q[6 * PK_REC * 32] = a.ted0; q[7 * PK_REC * 32] = a.g;
        head += 1u;
      }
      cfire = fire_clock(a.until, 0);
    }
  }

  // every record is confirmed and no roll-back is pending: hand the timing state to Y, which stores the lane
  sh_fin[0][lane] = pos; sh_fin[1][lane] = __float_as_uint(a.g); sh_fin[2][lane] = (uint32_t)a.clock;
  sh_fin[3][lane] = __float_as_uint(a.until); sh_fin[4][lane] = __float_as_uint(a.pavg);
  sh_fin[5][lane] = __float_as_uint(a.pinst); sh_fin[6][lane] = __float_as_uint(a.ted0);
  sh_fin[7][lane] = __float_as_uint(a.ted1); sh_fin[8][lane] = __float_as_uint(a.ted2); sh_fin[9][lane] = a.tedcnt;
  __threadfence_block();
  if (lane == 0) sh_done = 1u;
  __threadfence_block();
  ws_bar_arrive(PK_BAR_POS, 96);
  ws_bar_arrive(PK_BAR_AGC, 64);
}

// Constructor state (receiver.rs:502-560) or SameReceiver::reset (receiver.rs:182-198) for the selected streams.
// `ids` == nullptr: all streams.  `after_reset`: AGC gain 1.0 (agc.rs:61) instead of min(1, min_gain) (agc.rs:55).
__global__ void same_init_kernel(const __grid_constant__ SameParams p, const uint32_t* __restrict__ ids, uint32_t n,
                                 int after_reset) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = ids ? ids[i] : i;
  if (s >= p.n_streams) return;
  const SameLayout& L = p.layout;
  uint32_t* st = p.state32 + s;
  for (uint32_t w = 0; w < L.n_words; ++w) st[(size_t)w * L.n_pad] = 0u;
  st[(size_t)F_AGC_GAIN * L.n_pad] = __float_as_uint(after_reset ? 1.0f : p.agc_gain0);
  st[(size_t)F_UNTIL * L.n_pad] = __float_as_uint(p.spt);
  st[(size_t)F_PAVG * L.n_pad] = __float_as_uint(p.spt);
  st[(size_t)F_PINST * L.n_pad] = __float_as_uint(p.spt);
  st[(size_t)F_SQ_BYTECLK * L.n_pad] = (uint32_t)(-1);
  st[(size_t)F_TRNEXT_LO * L.n_pad] = 0xffffffffu;
  st[(size_t)F_TRNEXT_HI * L.n_pad] = 0xffffffffu;
  st[(size_t)L.eq_ffc * L.n_pad] = __float_as_uint(1.0f);  // identity taps  equalize.rs:131-132
  st[(size_t)L.eq_fbc * L.n_pad] = __float_as_uint(1.0f);
}

// ----------------------------------------------------------------------------------------------------------------
// Event read-back order: the host API hands events out per stream in order of occurrence (receiver.rs:238-240).  The
// arena holds them in atomicAdd order, so they are counting-sorted by stream here before the device->host copy; within
// a stream the position is seq - (first seq of this batch), sequence numbers being consecutive.
// ----------------------------------------------------------------------------------------------------------------
__global__ void same_evsort_hist(const same_event* __restrict__ ev, uint32_t n, uint32_t n_streams,
                                 uint32_t* __restrict__ cnt, uint32_t* __restrict__ minseq, uint32_t* __restrict__ bad) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = ev[i].stream;
  if (s >= n_streams) { *bad = 1u; return; }
  atomicAdd(&cnt[s], 1u);
  atomicMin(&minseq[s], ev[i].seq);
}
// exclusive scan of cnt[0..n) into start[0..n], one block
__global__ void __launch_bounds__(1024) same_evsort_scan(const uint32_t* __restrict__ cnt, uint32_t* __restrict__ start,
                                                         uint32_t n) {
  __shared__ uint32_t part[1024];
  const uint32_t t = threadIdx.x, per = (n + 1023u) / 1024u;
  const uint32_t lo = min(t * per, n), hi = min(lo + per, n);
  uint32_t sum = 0;
  for (uint32_t i = lo; i < hi; ++i) sum += cnt[i];
  part[t] = sum;
  __syncthreads();
  for (uint32_t d = 1; d < 1024u; d <<= 1) {
    const uint32_t v = t >= d ? part[t - d] : 0u;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  uint32_t run = part[t] - sum;   // exclusive prefix of this thread's range
  for (uint32_t i = lo; i < hi; ++i) { start[i] = run; run += cnt[i]; }
  if (t == 1023u) start[n] = part[1023];
}
__global__ void same_evsort_scatter(const same_event* __restrict__ ev, uint32_t n, uint32_t n_streams,
                                    const uint32_t* __restrict__ start, const uint32_t* __restrict__ minseq,
                                    same_event* __restrict__ out, uint32_t* __restrict__ bad) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const same_event e = ev[i];
  if (e.stream >= n_streams) return;
  const uint32_t k = e.seq - minseq[e.stream];
  const uint32_t dst = start[e.stream] + k;
  if (k >= start[e.stream + 1] - start[e.stream]) { *bad = 1u; return; }   // gap in the sequence numbers: host sorts
  out[dst] = e;
}

}  // namespace same_dev

// ----------------------------------------------------------------------------------------------------------------
// Launchers (called from same_engine.cu)
// ----------------------------------------------------------------------------------------------------------------
extern "C" cudaError_t same_launch_rx(const SameParams* p, const SameTaps* taps, const SameTaps2* taps2, Kernel kernel,
                                      uint32_t lanes_per_warp, const void* d_samples_v, int sample_fmt,
                                      const unsigned long long* d_offsets, const uint32_t* d_lengths,
                                      const SameTiles* tiles, cudaStream_t stream) {
  const uint32_t blocks = (p->n_streams + 31u) / 32u;
  const int16_t* d_samples = static_cast<const int16_t*>(d_samples_v);
  const uint32_t lanes = (kernel == SPLIT) ? 32u : (lanes_per_warp ? lanes_per_warp : 32u);
  const uint32_t fblocks = (p->n_streams + lanes - 1u) / lanes;
  const SameTiles no_tiles{nullptr, nullptr, 0u, 32u, 1u};
  switch (kernel) {
    case SPLIT: {
      if (!tiles || !tiles->d || !d_samples) return cudaErrorInvalidValue;
      const SameTiles t = *tiles;
      const unsigned long long grid = (unsigned long long)((t.n_max + FE_RUN * FE_WARPS - 1u) / (FE_RUN * FE_WARPS)) * blocks;
      if (grid == 0ull || grid > 0x7fffffffull) return cudaErrorInvalidValue;
      same_dev::same_frontend_kernel<<<(unsigned)grid, FE_WARPS * 32, 0, stream>>>(*p, d_samples, d_offsets, d_lengths, t);
      same_dev::same_rx_fast_kernel<true><<<fblocks, 32, 0, stream>>>(*p, *taps2, d_samples, d_offsets, d_lengths, lanes, t);
      break;
    }
    case LOOKAHEAD:
      same_dev::same_rx_la_kernel<<<fblocks, 32, 0, stream>>>(*p, *taps2, d_samples, d_offsets, d_lengths, lanes);
      break;
    case SINGLE:
      same_dev::same_rx_fast_kernel<false><<<fblocks, 32, 0, stream>>>(*p, *taps2, d_samples, d_offsets, d_lengths, lanes, no_tiles);
      break;
    case PIPE: {
      // per device, cheap: set on every launch rather than tracking which devices have seen it
      cudaError_t e = cudaFuncSetAttribute(same_dev::same_rx_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           PK_DYN_SMEM);
      if (e != cudaSuccess) return e;
      same_dev::same_rx_pipe_kernel<<<fblocks, PK_THREADS, PK_DYN_SMEM, stream>>>(*p, *taps2, d_samples, d_offsets,
                                                                                   d_lengths, lanes);
      break;
    }
    case THREE:
      same_dev::same_rx_ws_kernel<<<fblocks, WS_THREADS, 0, stream>>>(*p, *taps2, d_samples, d_offsets, d_lengths, lanes);
      break;
    case GENERIC: {
      const bool small = p->ntaps <= 64 && p->dc_len <= 16;
      const size_t smem = small ? (size_t)(64 + 2 * 16) * 32 * sizeof(float) : (size_t)(128 + 2 * 64) * 32 * sizeof(float);
      if (sample_fmt == 1) {
        const float* f = static_cast<const float*>(d_samples_v);
        if (small) same_dev::same_rx_generic_kernel<64, 16, float><<<blocks, 32, smem, stream>>>(*p, *taps, f, d_offsets, d_lengths);
        else same_dev::same_rx_generic_kernel<128, 64, float><<<blocks, 32, smem, stream>>>(*p, *taps, f, d_offsets, d_lengths);
      } else {
        if (small) same_dev::same_rx_generic_kernel<64, 16, int16_t><<<blocks, 32, smem, stream>>>(*p, *taps, d_samples, d_offsets, d_lengths);
        else same_dev::same_rx_generic_kernel<128, 64, int16_t><<<blocks, 32, smem, stream>>>(*p, *taps, d_samples, d_offsets, d_lengths);
      }
      break;
    }
    default:
      return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// The tile-fed single-warp kernel on its own, on DC-blocked samples some front end already produced (the long-stream path
// of same_long.cu feeds it one dense stream: tiles->stride == 1).
extern "C" cudaError_t same_launch_rx_tilefed(const SameParams* p, const SameTaps2* taps2, const uint32_t* d_lengths,
                                              const SameTiles* tiles, cudaStream_t stream) {
  const uint32_t blocks = (p->n_streams + 31u) / 32u;
  same_dev::same_rx_fast_kernel<true><<<blocks, 32, 0, stream>>>(*p, *taps2, nullptr, nullptr, d_lengths, 32u, *tiles);
  return cudaGetLastError();
}

// The front-end kernel alone (measurement of the HBM-bound feed-forward stage; the resident state is not touched).
extern "C" cudaError_t same_launch_frontend(const SameParams* p, const int16_t* d_samples, const unsigned long long* d_offsets,
                                            const uint32_t* d_lengths, const SameTiles* tiles, cudaStream_t stream) {
  const uint32_t blocks = (p->n_streams + 31u) / 32u;
  const unsigned long long grid = (unsigned long long)((tiles->n_max + FE_RUN * FE_WARPS - 1u) / (FE_RUN * FE_WARPS)) * blocks;
  if (grid == 0ull || grid > 0x7fffffffull) return cudaErrorInvalidValue;
  same_dev::same_frontend_kernel<<<(unsigned)grid, FE_WARPS * 32, 0, stream>>>(*p, d_samples, d_offsets, d_lengths, *tiles);
  return cudaGetLastError();
}

// Counting sort of `n` arena events by (stream, seq) into `d_sorted`; *d_bad != 0 afterwards means "not sorted, use
// the arena order and sort on the host".  d_cnt / d_start: n_streams + 1 words, d_minseq: n_streams words.
extern "C" cudaError_t same_launch_evsort(const same_event* d_events, uint32_t n, uint32_t n_streams, uint32_t* d_cnt,
                                          uint32_t* d_minseq, uint32_t* d_start, same_event* d_sorted, uint32_t* d_bad,
                                          cudaStream_t stream) {
  cudaError_t err;
  if ((err = cudaMemsetAsync(d_cnt, 0, ((size_t)n_streams + 1) * 4, stream)) != cudaSuccess) return err;
  if ((err = cudaMemsetAsync(d_minseq, 0xff, (size_t)n_streams * 4, stream)) != cudaSuccess) return err;
  if ((err = cudaMemsetAsync(d_bad, 0, 4, stream)) != cudaSuccess) return err;
  const uint32_t blocks = (n + 255u) / 256u;
  same_dev::same_evsort_hist<<<blocks, 256, 0, stream>>>(d_events, n, n_streams, d_cnt, d_minseq, d_bad);
  same_dev::same_evsort_scan<<<1, 1024, 0, stream>>>(d_cnt, d_start, n_streams);
  same_dev::same_evsort_scatter<<<blocks, 256, 0, stream>>>(d_events, n, n_streams, d_start, d_minseq, d_sorted, d_bad);
  return cudaGetLastError();
}

extern "C" cudaError_t same_launch_init(const SameParams* p, const uint32_t* d_ids, uint32_t n, int after_reset,
                                        cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  same_dev::same_init_kernel<<<(n + 127u) / 128u, 128, 0, stream>>>(*p, d_ids, n, after_reset);
  return cudaGetLastError();
}
