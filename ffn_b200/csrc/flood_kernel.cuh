// flood_kernel.cuh — the persistent flood-fill kernel.
//
// ONE cooperative launch runs whole objects (or a whole canvas): per FoV step it stages the
// (image, seed) tile from the HBM-resident canvas, evaluates the residual conv stack with the
// field of view spread over all CTAs (tcgen05 implicit GEMM, or fp32 FMA in the parity mode),
// fuses bias / ReLU / residual / conv_lom / seed-add as epilogues, applies the disco merge,
// pastes into the seed canvas, evaluates the face-max movement policy and pops the next position
// from the device-side queue — without returning to the host.
//
// Up to kMaxChains flood fills ("chains": independent objects of one canvas, or independent patches of a
// batched predict) are TIME-MULTIPLEXED over all SMs: the kernel works in rounds, a round runs one FoV step
// of every active chain, and inside a round the layers of the chains are interleaved — (layer 0: chain A, B,
// C), (layer 1: A, B, C), ... — through one TMA -> UMMA -> epilogue pipeline per CTA.  The dependency
// "layer l of chain A needs layer l-1 of chain A from EVERY CTA" is a split-phase barrier per chain: the
// epilogue warps arrive (red.release) and move on to the next chain's tile, only the TMA producer waits
// (ld.acquire) just before it loads that chain's operands.  The barrier / L2 latency of one chain is thereby
// hidden behind the tensor-core work of the others, and a layer's weights are loaded once for all chains.
//
// Reference semantics restated here (file:line in the reference checkout):
//   stage        ffn/inference/inference.py:348-354 (_get_image), :399-407 (seed copy, NaN -> pad),
//                ffn/inference/runner.py:383-385 (normalisation)
//   network      ffn/training/models/convstack_3d.py:26-56, :83-95; ffn/training/model.py:168-183
//   tail         ffn/inference/inference.py:416-439 (disco merge, paste)
//   policy       ffn/inference/movement.py:42-100, :166-222
//   validity     ffn/inference/inference.py:312-346
//   object loop  ffn/inference/inference.py:460-533
//   canvas loop  ffn/inference/inference.py:538-683; ffn/inference/storage.py:137-143
//   batching     ffn/inference/executor.py:266-340 (one session.run over a [B, ...] feed)
// Included TWICE by engine.cu: namespace FFN_KNS = plain (FFN_PROFILE 0, the product kernel) and
// = profiled (FFN_PROFILE 1: device cycle counters, ffn_engine_profile), so that the timing code costs
// the product kernel nothing.

#include <math_constants.h>

#include "device_types.cuh"
#include "sm100.cuh"

namespace ffn {
namespace FFN_KNS {

// ------------------------------------------------------------------------------------------
// Per-CTA context
// ------------------------------------------------------------------------------------------
struct Ctx {
  const KParams* p;
  int tid, warp, lane, cta, G;
  int t_begin, t_end;          // tiles owned by this CTA
  unsigned bar_target;         // whole-grid barrier
  unsigned ev0, ev1, ev2, ev3, ev4;   // split-phase barrier events completed so far (this launch), per chain
  unsigned round;              // rounds completed in this launch (parity of seed_raw / count buffers)
  unsigned long long t_start;  // globaltimer at kernel entry (watchdog)
  unsigned char* smem;
  float* s_bias;               // [(nconv)*32] biases, then w_lom[32], b_lom
  uint64_t* mb_w;              // [2]
  uint64_t* mb_full;           // [kActStages] TMA -> UMMA: a tile's operands have landed
  uint64_t* mb_empty;          // [kActStages] UMMA -> TMA: the stage may be overwritten
  uint64_t* mb_tfull;          // [kAccSlots]  UMMA -> epilogue: accumulators complete
  uint64_t* mb_tempty;         // [kAccSlots]  epilogue -> UMMA: accumulators drained (8 arrivals)
  uint64_t* mb_sig;            // [kMaxChains] epilogue -> signal warp: a chain's layer is stored (8 arrivals)
  unsigned load_cnt, mma_cnt, epi_cnt;   // per-role running tile counters (ring index + phase parity)
  uint32_t* s_tmem;            // TMEM base address
  int* s_misc;                 // per-chain step-count accumulators, abort copy, disco flags, leader scratch (device_types.cuh: kOffMisc)
  int* s_round;                // [k][8] this round: action, z, y, x, buffer ; [kMaxChains + k][8] previous step: flags, z, y, x, buffer
  float* s_xchg;               // [2 tile parities][2 halves][4 warps][2][16] partial sums crossing warp boundaries
  float* s_dot;                // [2][128] conv_lom partial dot products of the upper channel half
  CanvasState* s_state;        // CTA 0: shared-memory working copies of the chain states (512-byte slots)
  Sched* s_sched;              // CTA 0: working copy of the scheduler state
  long long* prof;             // profiling slots of this CTA in SHARED memory (null unless CTA 0 / G-1);
                               // flushed to global once, at kernel end, so timing does not stall the timed code
#if FFN_PROFILE
  long long* trace;            // per-tile event times of CTA kTraceCta (global, [kTraceEvents][kTraceTiles]); else null
  unsigned sig_cnt;            // signaller: releases so far
#endif
  // mbarrier phase parities and pending-prefetch flags as ONE bit field: dynamically indexed arrays
  // would push this whole struct into local memory (behind the L1 every grid barrier invalidates).
  uint32_t bits;   // bit b: weights[b] parity; 8+b: weights[b] in flight
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t bit_get(const Ctx& c, int k) { return (c.bits >> k) & 1u; }
__device__ __forceinline__ void bit_flip(Ctx& c, int k) { c.bits ^= 1u << k; }
__device__ __forceinline__ void bit_set(Ctx& c, int k, bool v) { c.bits = (c.bits & ~(1u << k)) | ((v ? 1u : 0u) << k); }

__device__ __forceinline__ unsigned ev_get(const Ctx& c, int k) {
  return k == 0 ? c.ev0 : (k == 1 ? c.ev1 : (k == 2 ? c.ev2 : (k == 3 ? c.ev3 : c.ev4)));
}
__device__ __forceinline__ void ev_add(Ctx& c, int k, unsigned n) {
  if (k == 0) c.ev0 += n;
  else if (k == 1) c.ev1 += n;
  else if (k == 2) c.ev2 += n;
  else if (k == 3) c.ev3 += n;
  else c.ev4 += n;
}
__device__ __forceinline__ CanvasState* chain_state(const Ctx& c, int k) {
  return reinterpret_cast<CanvasState*>(reinterpret_cast<unsigned char*>(c.s_state) + k * kStateSlot);
}

__device__ __forceinline__ bool aborted(const Ctx& c) {
  return sm100::ld_volatile_s32(c.p->ws.abort_flag) != 0;
}

// Profiling is opt-in (ffn_engine_profile_enable): reading the clock is not free, and CTA G-1 —
// one of the two profiled CTAs — is on the critical path of every layer.
#if FFN_PROFILE
__device__ __forceinline__ long long prof_now(const Ctx& c) { return c.prof ? clock64() : 0ll; }
__device__ __forceinline__ void prof_add(const Ctx& c, int slot, long long dt) {
  if (c.prof) c.prof[slot] += dt;
}
// Tile timeline of one CTA (ffn_engine_trace): event e of the role's idx-th tile since kernel start.
//   0 producer saw the chain barrier   1 tile's copies issued   2 UMMA issuer saw the operands   3 ... got a TMEM slot
//   4 UMMAs issued   5 epilogue saw the accumulators   6 epilogue done   7 signaller released (idx = signal number)
__device__ __forceinline__ void trace_ev(const Ctx& c, int ev, unsigned idx) {
  if (c.trace && idx < (unsigned)kTraceTiles) c.trace[ev * kTraceTiles + idx] = clock64();
}
#else
__device__ __forceinline__ long long prof_now(const Ctx&) { return 0ll; }
__device__ __forceinline__ void prof_add(const Ctx&, int, long long) {}
__device__ __forceinline__ void trace_ev(const Ctx&, int, unsigned) {}
#endif

// Bounded spin on an mbarrier phase; a timeout raises the abort flag instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(const Ctx& c, uint64_t* bar, uint32_t parity) {
  unsigned spins = 0;
  long long t0 = 0;
  while (!sm100::mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3FF) == 0) {
      if (aborted(c)) return;
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      if (now - t0 > (1ll << 32)) {   // ~2 s
        atomicExch(c.p->ws.abort_flag, 2);
        return;
      }
    }
  }
}

// Bounded spin until *ctr (monotonic, wrap-around safe) reaches target; `code` is the abort reason.
__device__ __forceinline__ void spin_until(const Ctx& c, const unsigned* ctr, unsigned target, int code) {
  long long tw = 0;
  unsigned spins = 0;
  while ((int)(sm100::ld_acquire_u32(ctr) - target) < 0) {
    if ((++spins & 0xFF) == 0) {
      if (aborted(c)) break;
      const long long now = clock64();
      if (tw == 0) tw = now;
      if (now - tw > (1ll << 32)) {
        atomicExch(c.p->ws.abort_flag, code);
        break;
      }
    }
  }
}

// Grid-wide barrier (all CTAs are co-resident: cooperative launch, one CTA per SM): once per round.
// One red.release per CTA counts the arrival; one thread polls with acquire loads and releases the
// others through a named barrier.
__device__ __forceinline__ void grid_barrier(Ctx& c) {
  sm100::tc_fence_before();
  __syncthreads();
  c.bar_target += c.G;
  if (c.warp == kLoadWarp) {
    if (c.lane == 0) {
      const long long t0 = prof_now(c);
      // release: everything this CTA wrote (ordered before by bar.sync) becomes visible gpu-wide
      // before the arrival is counted
      sm100::red_release_add(c.p->ws.bar, 1u);
      spin_until(c, c.p->ws.bar, c.bar_target, 1);
      // the acquire load that observed the full count orders every later read of this CTA (after
      // the named barrier below) behind the other CTAs' writes; TMA readers add their proxy fence
      prof_add(c, 0, prof_now(c) - t0);
    }
    __syncwarp();
    // named barriers count whole warps: the polling WARP arrives (without waiting), the nine others sync
    asm volatile("bar.arrive 4, %0;" ::"n"(kThreads) : "memory");
  } else {
    asm volatile("bar.sync 4, %0;" ::"n"(kThreads) : "memory");
  }
  sm100::tc_fence_after();
}

// Split-phase barrier of one chain.  ARRIVE: each of the eight epilogue warps, after its global stores of one
// layer of chain k, arrives at the chain's shared-memory mbarrier and goes on with the next tile; the signal
// warp waits for the eight arrivals and does the gpu-scope red.release (a release waits for the CTA's earlier
// stores to be performed: ~1 k cycles that would otherwise sit on the epilogue's critical path three times per
// layer).  WAIT (the TMA producer warp, before it loads chain k's operands of the next layer): acquire-poll
// until `events` arrivals of every CTA have been counted since the start of this chain's round.
__device__ __forceinline__ void chain_arrive_epi(Ctx& c, int k) {
  sm100::tc_fence_before();
  __syncwarp();
  if (c.lane == 0) sm100::mbar_arrive(&c.mb_sig[k]);   // release.cta: this warp's stores -> the signal warp
}
__device__ __forceinline__ void chain_signal(Ctx& c, int k, uint32_t parity) {   // signal warp
  mbar_wait(c, &c.mb_sig[k], parity);                     // acquire.cta: the eight epilogue warps' stores
  if (c.lane == 0) sm100::red_release_add(c.p->ch[k].bar, 1u);   // cumulative: they become visible gpu-wide first
  __syncwarp();
}
__device__ __forceinline__ void chain_wait(Ctx& c, int k, unsigned events) {
  if (c.lane == 0) {
    const long long t0 = prof_now(c);
    spin_until(c, c.p->ch[k].bar, (unsigned)c.G * (ev_get(c, k) + events), 3);
    prof_add(c, 14, prof_now(c) - t0);
  }
  __syncwarp();
}

// row -> (z, y, x); false for the zero pad column / pad line / rows past the FoV.
__device__ __forceinline__ bool row_to_zyx(const Geom& g, int r, int& z, int& y, int& x) {
  if (r >= g.nr) return false;
  z = (int)(((float)r + 0.5f) * g.inv_pp);          // exact for every row (verified in ffn_engine_create)
  const int rem = r - z * g.pp;
  y = (int)(((float)rem + 0.5f) * g.inv_xp);
  x = rem - y * g.xp;
  return y < g.fy && x < g.fx;
}

__device__ __forceinline__ bool disco_active(const KParams& p, int k, unsigned parity) {
  // inference.py:416-424: np.mean(logits >= move_threshold) > disco_seed_threshold (float64 compare)
  if (!(p.cv.opt.disco_seed_threshold >= 0.f)) return false;
  const unsigned cnt = __ldcg(p.ch[k].count + 2 * parity);
  return (double)cnt / (double)p.g.V > (double)p.cv.opt.disco_seed_threshold;
}

// Merged logit of FoV row r of chain k's step staged with `parity` (what Canvas.update_at writes back and returns).
__device__ __forceinline__ float merged_row(const KParams& p, int k, unsigned parity, int r, bool disco) {
  float l = __ldcg(p.ch[k].logits + r);
  if (disco) {
    const float o = __ldcg(p.ch[k].seed_raw[parity] + r);
    if (o < 0.f && l > o) l = o;   // NaN old value: both compares false (inference.py:427-433)
  }
  return l;
}

// ------------------------------------------------------------------------------------------
// Stage: canvas (or host-provided patch) -> layer-0 operands + raw seed copy
// ------------------------------------------------------------------------------------------
// The previous step of the same chain may still be pasting into the canvas in other CTAs (paste and
// stage of consecutive steps are separated by no grid barrier), so seed values inside the previous
// FoV are taken from that step's merged logits in the workspace — exactly what the paste writes.
__device__ __forceinline__ void stage_fov(Ctx& c, int k, int b, int pz, int py, int px, int batch_idx) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const ChainDev& ch = p.ch[k];
  const bool predict = p.job.mode == MODE_PREDICT;
  const unsigned par = c.round & 1u;
  const int* prev = c.s_round + 8 * (kMaxChains + k);
  const bool have_prev = !predict && prev[0] != 0 && prev[4] == b;
  const bool prev_disco = have_prev && (prev[0] & 2) != 0;
  const int qz = prev[1] - g.mz, qy = prev[2] - g.my, qx = prev[3] - g.mx;   // previous FoV corner
  float* raw_out = ch.seed_raw[par];
  for (int r = c.t_begin * kTileOut + c.tid; r < c.t_end * kTileOut; r += kThreads) {
    int z, y, x;
    if (!row_to_zyx(g, r, z, y, x)) continue;
    float img, s, fed;
    if (predict) {
      const size_t i = (size_t)batch_idx * g.V + ((size_t)z * g.fy + y) * g.fx + x;
      img = __ldg(p.job.in_image + i);
      s = __ldg(p.job.in_seed + i);
      fed = s;
    } else {
      const int gz = pz - g.mz + z, gy = py - g.my + y, gx = px - g.mx + x;
      const size_t i = ((size_t)gz * p.cv.sy + gy) * p.cv.sx + gx;
      if (p.cv.image_is_u8) {
        const float raw = (float)__ldg(reinterpret_cast<const uint8_t*>(p.cv.image) + i);
        img = __fdiv_rn(__fsub_rn(raw, p.cv.mean), p.cv.stddev);
      } else {
        img = __ldg(reinterpret_cast<const float*>(p.cv.image) + i);
      }
      const int fz = gz - qz, fy = gy - qy, fx = gx - qx;
      if (have_prev && fz >= 0 && fz < g.fz && fy >= 0 && fy < g.fy && fx >= 0 && fx < g.fx) {
        s = merged_row(p, k, par ^ 1u, fz * g.pp + fy * g.xp + fx, prev_disco);
      } else {
        s = __ldcg(p.ob[b].seed + i);
      }
      fed = isnan(s) ? p.cv.opt.pad_value : s;
    }
    raw_out[r] = predict ? fed : s;
    if (p.compute_mode != FFN_COMPUTE_FP32) {
      const __half2 h01 = __floats2half2_rn(img, fed);
      uint4 v;
      v.x = *reinterpret_cast<const uint32_t*>(&h01);
      v.y = v.z = v.w = 0u;
      *reinterpret_cast<uint4*>(ch.act0_h + ((size_t)g.guard + r) * 8) = v;
      if (p.compute_mode == FFN_COMPUTE_FP16X2_TC) {   // lo parts: x - fp16(x), exact in fp32
        const float2 hf = __half22float2(h01);
        const __half2 l01 = __floats2half2_rn(img - hf.x, fed - hf.y);
        v.x = *reinterpret_cast<const uint32_t*>(&l01);
        *reinterpret_cast<uint4*>(p.ws.act0_l + ((size_t)g.guard + r) * 8) = v;
      }
    } else {
      p.ws.act0_f[(size_t)g.guard + r] = make_float4(img, fed, 0.f, 0.f);
    }
  }
  if (c.cta == 0 && c.tid == 0) {
    ch.count[2 * par] = 0u;       // voxels >= move threshold
    ch.count[2 * par + 1] = 0u;   // Canvas.history_deleted of this step
  }
  if (c.tid == 0) c.s_misc[k] = 0;
}

// ------------------------------------------------------------------------------------------
// Epilogue shared by both compute modes: v[32] = conv accumulators of one FoV row.
//   even layers ("_a"): out = relu(v + b)                         (convstack_3d.py:38,45)
//   odd  layers ("_b"): net = v + b (+ residual); out = relu(net) (convstack_3d.py:39,46-49)
//   last layer        : logits = seed + b_lom + <relu(net), w_lom> (convstack_3d.py:51-54,
//                       model.py:176-177)
// `out` feeds the next convolution: the pre-activation ReLU of the next residual module and the
// ReLU before conv_lom are applied here, once, when the value is produced.
// ------------------------------------------------------------------------------------------
// Per-row contribution to the two per-step counters, packed (low 16 bits: voxels with logit >= move
// threshold, inference.py:423; high bits: Canvas.history_deleted, inference.py:420-422 — old seed >= logit(0.8)
// turned into logit < logit(0.5), counted only while the event trace records history).
__device__ __forceinline__ int step_counts(const KParams& p, float raw, float logit) {
  int v = (logit >= p.cv.opt.move_threshold) ? 1 : 0;
  if (p.cv.trace && p.cv.opt.disco_seed_threshold >= 0.f && (double)raw >= 1.3862943611198908 && logit < 0.f)
    v += 1 << 16;
  return v;
}

// fp32 parity mode only (one chain: chain 0).
__device__ __forceinline__ void epilogue_row(const Ctx& c, int layer, int r, float (&v)[32], int& hit) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const float* b = c.s_bias + layer * 32;
#pragma unroll
  for (int k = 0; k < 32; ++k) v[k] += b[k];
  const bool is_b = (layer & 1) != 0;
  const bool last = layer == g.nconv - 1;
  const size_t ra = (size_t)g.guard + r;
  if (is_b) {
    if (layer > 1) {
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 o = __ldcg(p.ws.res + (size_t)q * g.rows_alloc + ra);
        v[4 * q + 0] += o.x;
        v[4 * q + 1] += o.y;
        v[4 * q + 2] += o.z;
        v[4 * q + 3] += o.w;
      }
    }
    if (!last) {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        p.ws.res[(size_t)q * g.rows_alloc + ra] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    }
  }
#pragma unroll
  for (int k = 0; k < 32; ++k) v[k] = fmaxf(v[k], 0.f);
  if (last) {
    const float* wl = c.s_bias + g.nconv * 32;
    float upd = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) upd = fmaf(v[k], wl[k], upd);
    upd += wl[32];
    const float raw = p.ch[0].seed_raw[c.round & 1u][r];
    const float fed = isnan(raw) ? p.cv.opt.pad_value : raw;
    const float logit = fed + upd;
    p.ch[0].logits[r] = logit;
    hit += step_counts(p, raw, logit);
    return;
  }
  float4* dst = p.ws.act_f[layer & 1];
#pragma unroll
  for (int q = 0; q < 8; ++q)
    dst[(size_t)q * g.rows_alloc + ra] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

// ------------------------------------------------------------------------------------------
// Tensor-core layer: implicit GEMM, M = 128 FoV rows, N = 32 features, K = 27 taps x Cin.
// A = activation rows (K-major, no swizzle: [k-chunk][row] 16-byte units, so a tap is a shifted
// start address), B = packed weights, D = fp32 accumulators in TMEM (32 columns per tile).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_issue_weight_load(Ctx& c, int layer) {
  const KParams& p = *c.p;
  const int buf = layer & 1;
  const uint32_t bytes = (layer == 0 ? 27 * 2 : 27 * 4) * 512;
  sm100::mbar_expect_tx(&c.mb_w[buf], bytes);
  sm100::bulk_g2s(c.smem + buf * (27 * 4 * 512), p.w.w16 + w16_layer_offset_halfs(layer), bytes, &c.mb_w[buf]);
}

// Issues the 9 * NCH/2 UMMAs (128 x 96 x 16) of one tile: one per (dz, dy) tap-row and k-pair; the
// three dx taps ride along N.  Fully unrolled: every A start-address offset is
// (const * seg_rows + const * xp), so the loop body is two adds and the UMMA.
template <int NCH>
__device__ __forceinline__ void tc_issue_tile(uint32_t d, uint32_t a_lo, uint32_t b_lo, int seg_rows, int xp) {
  const uint32_t idesc = sm100::umma_idesc_f16(kTileM, kStackN);
  const uint64_t hi = (uint64_t)((128u >> 4) | (1u << 14)) << 32;   // SBO = 128 B, descriptor version 1
  // one (dz, dy) tap-row per iteration: fully unrolled, the 36 descriptors overflow the uniform register
  // file into ordinary registers
#pragma unroll 1
  for (int row = 0; row < 9; ++row) {
    const int tz = row / 3, ty = row % 3;
#pragma unroll
    for (int j = 0; j < NCH / 2; ++j) {
      const uint32_t aoff = (uint32_t)((2 * j * 3 + tz) * seg_rows + ty * xp);   // stage layout [k-chunk][dz][row]
      const uint32_t boff = (uint32_t)((row * NCH + 2 * j) * (12 * 128 / 16));
      sm100::umma_f16(d, hi | (uint64_t)(a_lo + aoff), hi | (uint64_t)(b_lo + boff), idesc,
                      (row | j) != 0 ? 1u : 0u);
    }
  }
}

__device__ __forceinline__ void quad_sync(int quad) {   // the four epilogue warps of one channel half
  asm volatile("bar.sync %0, 128;" ::"r"(quad + 1) : "memory");
}

// Epilogue of the tensor-core layer (warps 0-7; 2 channel halves x 4 TMEM lane quarters), specialised
// by layer kind so that the residual / conv_lom paths cost nothing where they do not apply:
//   EPI_A        "_a" convolutions   : out = relu(v + b)                          (convstack_3d.py:38,45)
//   EPI_B_FIRST  conv0_b             : net = v + b            ; out = relu(net)   (:39) starts the residual stream
//   EPI_B        conv{i}_b, i >= 1   : net = v + b + residual ; out = relu(net)   (:46-49)
//   EPI_LAST     the final "_b"      : as EPI_B, then logits = seed + b_lom + <relu(net), w_lom> (:51-54, model.py:176-177)
//   EPI_LAST0    conv0_b at depth 1  : net = v + b, then the logits of EPI_LAST (no residual module: there is no
//                                      residual stream to read)
// The fp32 residual stream lives in this thread's TMEM lane, columns behind the accumulator ring
// (32 columns per tile and chain).
// Accumulator row m of a tile holds, for the FoV row u = tile_row0 - 1 + m,
//   D[u][dx*32 + co] = sum_{dz,dy,ci} act[u + dz*pp + dy*xp][ci] * W[dz,dy,dx][ci][co]
// and the convolution output is out[v] = D[v-1][dx=-1] + D[v][dx=0] + D[v+1][dx=+1]: one lane up /
// down, done with warp shuffles (+ a 2 KB shared-memory exchange at the three warp boundaries).
enum EpiKind : int { EPI_A = 0, EPI_B_FIRST = 1, EPI_B = 2, EPI_LAST = 3, EPI_LAST0 = 4 };

template <int KIND, bool X2 = false>
__device__ __forceinline__ int tc_epilogue(Ctx& c, int k, int layer, int ntiles) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const ChainDev& ch = p.ch[k];
  constexpr float kUnscale = 1.0f / (float)(1 << kSplitShift);   // X2: accumulators carry w * 2^kSplitShift
  constexpr bool kReadRes = KIND == EPI_B || KIND == EPI_LAST;
  constexpr bool kWriteRes = KIND == EPI_B_FIRST || KIND == EPI_B;
  constexpr bool kLast = KIND == EPI_LAST || KIND == EPI_LAST0;
  const int half = c.warp >> 2, wq = c.warp & 3;
  const float4* bias4 = reinterpret_cast<const float4*>(c.s_bias + layer * 32 + half * 16);   // re-read per tile: 16 registers less
  const size_t chunk_stride = (size_t)g.rows_alloc * 8;
  __half* out_base = ch.act_h[layer & 1] + (size_t)(half * 2) * chunk_stride + (size_t)g.guard * 8;
  __half* out_lo_base = X2 ? p.ws.act_l[layer & 1] + (size_t)(half * 2) * chunk_stride + (size_t)g.guard * 8 : nullptr;
  const float* raw_in = ch.seed_raw[c.round & 1u];
  int hit = 0;
  for (int j = 0; j < ntiles; ++j) {
    const int slot = c.epi_cnt % kAccSlots;
    float* xch = c.s_xchg + ((c.epi_cnt & 1) * 2 + half) * (4 * 2 * 16);   // double-buffered by tile parity
    const int m = wq * 32 + c.lane;                                 // accumulator row of this thread
    const int r = (c.t_begin + j) * kTileOut - 1 + m;               // FoV row it holds partial sums for
    int z = 0, y = 0, x = 1;
    const bool valid = m >= 1 && m <= kTileOut && r >= 0 && row_to_zyx(g, r, z, y, x);
    long long t0 = prof_now(c);
    mbar_wait(c, &c.mb_tfull[slot], (c.epi_cnt / kAccSlots) & 1u);
    if (c.tid == 0) prof_add(c, 4, prof_now(c) - t0);
    if (c.tid == 0) trace_ev(c, 5, c.epi_cnt);
    t0 = prof_now(c);
    sm100::tc_fence_after();
    const uint32_t tbase = c.tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(slot * kStackN + half * 16);
    const uint32_t tres = c.tmem_base + ((uint32_t)(wq * 32) << 16) +
                          (uint32_t)(kAccSlots * kStackN + (k * ntiles + j) * kFeat + half * 16);
    uint32_t a[16], b[16], d2[16], rr[16];
    sm100::tmem_ld16(tbase, a);          // dx = -1 block: consumed by the lane above (m + 1)
    sm100::tmem_ld16(tbase + 32, b);     // dx =  0 block
    sm100::tmem_ld16(tbase + 64, d2);    // dx = +1 block: consumed by the lane below (m - 1)
    if (kReadRes) sm100::tmem_ld16(tres, rr);
    sm100::tmem_ld_wait();
    // the accumulators are in registers: hand the TMEM slot back to the UMMA issuer
    sm100::tc_fence_before();
    __syncwarp();
    if (c.lane == 0) sm100::mbar_arrive(&c.mb_tempty[slot]);
    if (c.lane == 31) {
      float4* q = reinterpret_cast<float4*>(xch + (wq * 2 + 0) * 16);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        q[i] = make_float4(__uint_as_float(a[4 * i]), __uint_as_float(a[4 * i + 1]), __uint_as_float(a[4 * i + 2]),
                           __uint_as_float(a[4 * i + 3]));
    }
    if (c.lane == 0) {
      float4* q = reinterpret_cast<float4*>(xch + (wq * 2 + 1) * 16);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        q[i] = make_float4(__uint_as_float(d2[4 * i]), __uint_as_float(d2[4 * i + 1]), __uint_as_float(d2[4 * i + 2]),
                           __uint_as_float(d2[4 * i + 3]));
    }
    quad_sync(half);
    // out[v] = D[v-1][dx=-1] + D[v][dx=0] + D[v+1][dx=+1]
    float up[16], dn[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      up[i] = __shfl_up_sync(0xffffffffu, __uint_as_float(a[i]), 1);      // from lane - 1
      dn[i] = __shfl_down_sync(0xffffffffu, __uint_as_float(d2[i]), 1);   // from lane + 1
    }
    if (c.lane == 0 && wq > 0) {     // row m - 1 lives in the previous warp
      const float4* q = reinterpret_cast<const float4*>(xch + ((wq - 1) * 2 + 0) * 16);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 t = q[i];
        up[4 * i] = t.x; up[4 * i + 1] = t.y; up[4 * i + 2] = t.z; up[4 * i + 3] = t.w;
      }
    }
    if (c.lane == 31 && wq < 3) {    // row m + 1 lives in the next warp
      const float4* q = reinterpret_cast<const float4*>(xch + ((wq + 1) * 2 + 1) * 16);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 t = q[i];
        dn[4 * i] = t.x; dn[4 * i + 1] = t.y; dn[4 * i + 2] = t.z; dn[4 * i + 3] = t.w;
      }
    }
    // SAME padding in x: at x = 0 / x = fx-1 row v-1 / v+1 belongs to the neighbouring line (mask 0);
    // all partial sums are finite (pad rows multiply zero activations), so 0 * value is exact
    const float m_up = x == 0 ? 0.f : 1.f, m_dn = x == g.fx - 1 ? 0.f : 1.f;
    float v[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 bi = bias4[i];
      const float bias[4] = {bi.x, bi.y, bi.z, bi.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int q = 4 * i + e;
        const float acc = fmaf(up[q], m_up, fmaf(dn[q], m_dn, __uint_as_float(b[q])));
        v[q] = X2 ? fmaf(acc, kUnscale, bias[e]) : acc + bias[e];
        if (kReadRes) v[q] += __uint_as_float(rr[q]);
      }
    }
    if (kWriteRes) {
      // rows outside the FoV carry values nobody reads; storing them unconditionally keeps the warp converged
#pragma unroll
      for (int q = 0; q < 16; ++q) rr[q] = __float_as_uint(v[q]);
      sm100::tmem_st16(tres, rr);
    }
    if (!kLast) {
      if (valid) {
        // out = relu(.) as fp16: the ReLU rides on the conversion (cvt.rn.relu.f16x2.f32)
        __half* dst = out_base + (size_t)r * 8;   // [k-chunk][row][8 halfs]; this half owns chunks 2*half, 2*half+1
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          uint4 o;
          o.x = sm100::cvt_relu_f16x2(v[8 * q + 0], v[8 * q + 1]);
          o.y = sm100::cvt_relu_f16x2(v[8 * q + 2], v[8 * q + 3]);
          o.z = sm100::cvt_relu_f16x2(v[8 * q + 4], v[8 * q + 5]);
          o.w = sm100::cvt_relu_f16x2(v[8 * q + 6], v[8 * q + 7]);
          *reinterpret_cast<uint4*>(dst + q * chunk_stride) = o;
          if (X2) {   // lo parts of relu(v): relu(v) - fp16(relu(v)) is exact in fp32
            const uint32_t hi[4] = {o.x, o.y, o.z, o.w};
            uint32_t lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi[e]));
              const __half2 l = __floats2half2_rn(fmaxf(v[8 * q + 2 * e], 0.f) - hf.x, fmaxf(v[8 * q + 2 * e + 1], 0.f) - hf.y);
              lo[e] = *reinterpret_cast<const uint32_t*>(&l);
            }
            *reinterpret_cast<uint4*>(out_lo_base + (size_t)r * 8 + q * chunk_stride) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
      }
    } else {
      // conv_lom: this half's share of <relu(net), w_lom>; combine the halves, then logits = seed + update
      const float* wl = c.s_bias + g.nconv * 32;
      float part = 0.f;
#pragma unroll
      for (int q = 0; q < 16; ++q) part = fmaf(fmaxf(v[q], 0.f), wl[half * 16 + q], part);
      float* dot = c.s_dot + (c.epi_cnt & 1) * kTileM;
      if (half == 1) dot[m] = part;
      asm volatile("bar.sync 3, 256;" ::: "memory");
      if (half == 0 && valid) {
        const float upd = part + dot[m] + wl[32];
        const float raw = raw_in[r];
        const float fed = isnan(raw) ? p.cv.opt.pad_value : raw;
        const float logit = fed + upd;
        ch.logits[r] = logit;
        hit += step_counts(p, raw, logit);
      }
    }
    if (kWriteRes) sm100::tmem_st_wait();
    if (c.tid == 0) prof_add(c, 5, prof_now(c) - t0);
    if (c.tid == 0) trace_ev(c, 6, c.epi_cnt);
    ++c.epi_cnt;
  }
  return hit;
}

// Adds the per-row counts of the last layer (this warp's `hit`) to the chain's step counters.
__device__ __forceinline__ void publish_counts(Ctx& c, int k, int hit) {
  hit = __reduce_add_sync(0xffffffffu, hit);
  if (c.lane == 0 && hit) atomicAdd(&c.s_misc[k], hit);
  asm volatile("bar.sync 5, 256;" ::: "memory");
  if (c.tid == 0 && c.s_misc[k]) {   // packed per-CTA sums (step_counts): <= 882 rows per CTA, so no carry
    const unsigned packed = (unsigned)c.s_misc[k];
    unsigned* cnt = c.p->ch[k].count + 2 * (c.round & 1u);
    if (packed & 0xffffu) atomicAdd(cnt, packed & 0xffffu);
    if (packed >> 16) atomicAdd(cnt + 1, packed >> 16);
  }
}

// One round of the conv stacks of the chains in `mask`, as ONE warp-specialised pipeline over the work
// items (layer, chain, tile) in that order:
//   warp 8  TMA producer : waits for the chain's split-phase barrier (previous layer complete in every
//                          CTA), then per tile twelve 1-D bulk copies (3 z-planes x 4 k-chunks of 126 + 2*halo
//                          rows; or ONE tiled TMA through the buffer's tensor map, FFN_B200_TMAP=1) into a
//                          kActStages-stage shared-memory ring            full[stage]  <-  empty[stage]
//   warp 9  UMMA issuer  : 18 UMMAs 128x96x16 per tile into a kAccSlots-slot TMEM ring; one commit frees the
//                          smem stage, one publishes the slot           tfull[slot]  <-  tempty[slot]
//   warps 0-7 epilogue   : every tile by all eight warps (2 channel halves x 4 TMEM lane quarters); after a
//                          chain's tiles of a layer they ARRIVE at that chain's barrier and go on
// A layer's weights are shared by all chains (double-buffered, the next layer prefetched once every UMMA of
// the layer before has completed).
__device__ __forceinline__ void layers_pipelined(Ctx& c, unsigned mask) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  unsigned char* act_smem = c.smem + 2 * 27 * 4 * 512;
  const int seg_rows = kTileOut + 2 * g.halo;                 // k-chunk plane pitch of a stage (rows)
  const int stage_bytes = 3 * 4 * seg_rows * 16;
  const int ntiles = c.t_end - c.t_begin;
  const int nconv = g.nconv;
  const long long t_layers = prof_now(c);

  // The two single-issuer roles run with the WHOLE warp converged (c.warp is warp-uniform by
  // construction, see the kernel entry) and elect one lane only for the instructions with side effects:
  // addresses and descriptors then live in uniform registers, instead of being broadcast from one
  // lane's registers (ELECT / R2UR loop) in front of every bulk copy and every UMMA.
  if (c.warp == kLoadWarp) {
    // ------------------------------------------------------------------ TMA producer
    for (int layer = 0; layer < nconv; ++layer) {
      const int nch = layer == 0 ? 2 : 4;
      // The next layer's weights (next round's layer 0 after the last layer) are prefetched into the other
      // buffer during this layer.  That buffer's previous user — layer - 1 — must have completed every UMMA,
      // i.e. the tile issued just before this layer's first one (n0 - 1; commits are in order), and that is
      // exactly what the `empty` wait of this layer's kActStages-th tile waits for (same stage).  A layer with
      // fewer tiles waits for that phase explicitly at its end (it cannot have been overtaken: the stage's next
      // user has not been loaded).
      const unsigned n0 = c.load_cnt;   // first tile of this layer
      bool weights_pending = true;
      for (int k = 0; k < kMaxChains; ++k) {
        if (!((mask >> k) & 1u)) continue;
        const ChainDev& ch = p.ch[k];
        const __half* in = layer == 0 ? ch.act0_h : ch.act_h[(layer - 1) & 1];
        chain_wait(c, k, (unsigned)layer + 1u);   // event 1 = staged, event l + 1 = layer l - 1 complete everywhere
        if (c.lane == 0) trace_ev(c, 0, c.load_cnt);
#ifndef FFN_EXP_NO_READER_FENCE
        sm100::fence_proxy_async_global();
#endif        // other CTAs' generic-proxy stores (ordered by the acquire) -> async proxy
        for (int j = 0; j < ntiles; ++j) {
          const int s = c.load_cnt % kActStages;
          mbar_wait(c, &c.mb_empty[s], ((c.load_cnt / kActStages) & 1u) ^ 1u);
          if (weights_pending && c.load_cnt - n0 == (unsigned)(kActStages - 1)) {
            weights_pending = false;
            if (sm100::elect_one()) tc_issue_weight_load(c, (layer + 1 == nconv) ? 0 : layer + 1);
            __syncwarp();
          }
          const int r0 = (c.t_begin + j) * kTileOut;
          unsigned char* dst = act_smem + (size_t)s * stage_bytes;
          if (sm100::elect_one()) {
            sm100::mbar_expect_tx(&c.mb_full[s], (uint32_t)(3 * nch * seg_rows * 16));
            if (p.use_tmap) {
              // one tiled TMA: box (8 halfs, seg_rows rows, 3 z-planes, nch k-chunks) -> stage layout [k-chunk][dz][row]
              sm100::tma_load_4d(dst, &p.tmap[k][layer == 0 ? 0 : 1 + ((layer - 1) & 1)], 0, g.guard + r0 - g.halo - g.pp, 0, 0,
                                 &c.mb_full[s]);
            } else {
              for (int cc = 0; cc < nch; ++cc)
                for (int dzi = 0; dzi < 3; ++dzi)
                  sm100::bulk_g2s(dst + (size_t)(cc * 3 + dzi) * seg_rows * 16,
                                  in + ((size_t)cc * g.rows_alloc + g.guard + r0 + (dzi - 1) * g.pp - g.halo) * 8,
                                  (uint32_t)seg_rows * 16, &c.mb_full[s]);
            }
          }
          __syncwarp();
          if (c.lane == 0) trace_ev(c, 1, c.load_cnt);
          ++c.load_cnt;
        }
      }
      if (weights_pending) {
        if (n0 > 0) mbar_wait(c, &c.mb_empty[(n0 - 1u) % kActStages], ((n0 - 1u) / kActStages) & 1u);
        if (sm100::elect_one()) tc_issue_weight_load(c, (layer + 1 == nconv) ? 0 : layer + 1);
        __syncwarp();
      }
    }
  } else if (c.warp == kMmaWarp) {
    // ------------------------------------------------------------------ UMMA issuer
    for (int layer = 0; layer < nconv; ++layer) {
      const int buf = layer & 1;
      long long t0 = prof_now(c);
      mbar_wait(c, &c.mb_w[buf], (c.bits >> buf) & 1u);
      c.bits ^= 1u << buf;
      if (c.lane == 0) prof_add(c, 2, prof_now(c) - t0);
      const uint32_t b_lo = ((sm100::smem_u32(c.smem + buf * (27 * 4 * 512)) >> 4) & 0x3FFFu) | ((12u * 128u >> 4) << 16);
      for (int k = 0; k < kMaxChains; ++k) {
        if (!((mask >> k) & 1u)) continue;
        for (int j = 0; j < ntiles; ++j) {
          const int s = c.mma_cnt % kActStages, slot = c.mma_cnt % kAccSlots;
#ifdef FFN_EXP_TEMPTY_FIRST
          mbar_wait(c, &c.mb_tempty[slot], ((c.mma_cnt / kAccSlots) & 1u) ^ 1u);
#endif
          t0 = prof_now(c);
          mbar_wait(c, &c.mb_full[s], (c.mma_cnt / kActStages) & 1u);
          if (c.lane == 0) prof_add(c, 1, prof_now(c) - t0);
          if (c.lane == 0) trace_ev(c, 2, c.mma_cnt);
#ifndef FFN_EXP_TEMPTY_FIRST
          mbar_wait(c, &c.mb_tempty[slot], ((c.mma_cnt / kAccSlots) & 1u) ^ 1u);
#endif
          sm100::tc_fence_after();
          if (c.lane == 0) trace_ev(c, 3, c.mma_cnt);
          t0 = prof_now(c);
          const uint32_t a_lo = ((sm100::smem_u32(act_smem + (size_t)s * stage_bytes) >> 4) & 0x3FFFu) | ((uint32_t)(3 * seg_rows) << 16);
          const uint32_t d = c.tmem_base + (uint32_t)(slot * kStackN);
          if (sm100::elect_one()) {
            if (layer == 0) {
              tc_issue_tile<2>(d, a_lo, b_lo, seg_rows, g.xp);
            } else {
              tc_issue_tile<4>(d, a_lo, b_lo, seg_rows, g.xp);
            }
            sm100::umma_commit(&c.mb_tfull[slot]);   // accumulators of this tile complete
            sm100::umma_commit(&c.mb_empty[s]);      // ... and its shared-memory stage is free again
          }
          __syncwarp();
          if (c.lane == 0) prof_add(c, 3, prof_now(c) - t0);
          if (c.lane == 0) trace_ev(c, 4, c.mma_cnt);
          ++c.mma_cnt;
        }
      }
    }
  } else if (c.warp == kSigWarp) {
    // ------------------------------------------------------------------ barrier signaller
    for (int layer = 0; layer + 1 < nconv; ++layer)
      for (int k = 0; k < kMaxChains; ++k) {
        if (!((mask >> k) & 1u)) continue;
        // phase of the chain's mbarrier: nconv - 1 (odd) arrivals per round the chain was active in
        chain_signal(c, k, ((ev_get(c, k) / (unsigned)nconv) + (unsigned)layer) & 1u);
#if FFN_PROFILE
        if (c.lane == 0) trace_ev(c, 7, c.sig_cnt);
        ++c.sig_cnt;
#endif
      }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 0-7)
    for (int layer = 0; layer < nconv; ++layer) {
      const bool last = layer == nconv - 1;
      for (int k = 0; k < kMaxChains; ++k) {
        if (!((mask >> k) & 1u)) continue;
        if (last) {
          const int hit = layer == 1 ? tc_epilogue<EPI_LAST0>(c, k, layer, ntiles) : tc_epilogue<EPI_LAST>(c, k, layer, ntiles);
          publish_counts(c, k, hit);          // the round ends with a grid barrier: no chain arrival needed
        } else {
          if (!(layer & 1)) {
            tc_epilogue<EPI_A>(c, k, layer, ntiles);
          } else if (layer == 1) {
            tc_epilogue<EPI_B_FIRST>(c, k, layer, ntiles);
          } else {
            tc_epilogue<EPI_B>(c, k, layer, ntiles);
          }
          chain_arrive_epi(c, k);
        }
      }
    }
  }
  // role-independent bookkeeping, identical in every thread (the weight-barrier parities, bits 0 / 1, are
  // tracked by the UMMA issuer warp alone: nobody else waits on those barriers)
  bit_set(c, 8, true);   // the last layer prefetched layer 0's weights of the next round into buffer 0
#pragma unroll
  for (int k = 0; k < kMaxChains; ++k)
    if ((mask >> k) & 1u) ev_add(c, k, (unsigned)nconv);   // staged + layers 0 .. nconv-2
  if (c.tid == 0) prof_add(c, 11, prof_now(c) - t_layers);
}

// Near-fp32 tensor-core layer (FFN_COMPUTE_FP16X2_TC): activations and weights are both split into fp16
// hi + lo parts and every (tap-row, k-pair) becomes THREE UMMAs into the same fp32 accumulator,
//   a * w  ~=  a_hi * w_hi + a_lo * w_hi + a_hi * w_lo        (the dropped a_lo * w_lo term is ~2^-22 relative),
// which gives ~22 significant bits per product.  One chain (chain 0), whole-grid barriers between layers;
// shared memory is used differently from the fp16 path: activation stage 0 holds the hi parts and stage 1
// the lo parts of ONE tile, weight buffer 0 holds w_hi and buffer 1 w_lo of THIS layer (so there is no
// cross-layer weight prefetch and no tile double-buffering: this is the label-exact parity mode, not the
// throughput mode).
__device__ __forceinline__ void tc_layer_x2(Ctx& c, int layer) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const int nch = layer == 0 ? 2 : 4;
  const __half* in_hi = layer == 0 ? p.ch[0].act0_h : p.ch[0].act_h[(layer - 1) & 1];
  const __half* in_lo = layer == 0 ? p.ws.act0_l : p.ws.act_l[(layer - 1) & 1];
  unsigned char* act_smem = c.smem + 2 * 27 * 4 * 512;
  const int seg_rows = kTileOut + 2 * g.halo;
  const int stage_bytes = 3 * 4 * seg_rows * 16;
  const int ntiles = c.t_end - c.t_begin;
  const bool last = layer == g.nconv - 1;
  int hit = 0;
  bit_set(c, 8, true);
  if (c.warp == kLoadWarp) {
    sm100::fence_proxy_async_global();
    if (sm100::elect_one()) {
      // both halves of this layer's weights; every UMMA of the previous layer has completed (its
      // epilogue waited for the accumulators), so the buffers are free
      const uint32_t wbytes = (uint32_t)(27 * nch * 512);
      const __half* src = p.w.w16x2 + 2 * w16_layer_offset_halfs(layer);
      sm100::mbar_expect_tx(&c.mb_w[0], 2 * wbytes);
      sm100::bulk_g2s(c.smem, src, wbytes, &c.mb_w[0]);
      sm100::bulk_g2s(c.smem + 27 * 4 * 512, src + wbytes / 2, wbytes, &c.mb_w[0]);
    }
    __syncwarp();
    for (int j = 0; j < ntiles; ++j) {
      if (j > 0) mbar_wait(c, &c.mb_empty[0], (c.load_cnt & 1u) ^ 1u);
      const int r0 = (c.t_begin + j) * kTileOut;
      if (sm100::elect_one()) {
        sm100::mbar_expect_tx(&c.mb_full[0], (uint32_t)(2 * 3 * nch * seg_rows * 16));
        for (int part = 0; part < 2; ++part) {
          const __half* in = part ? in_lo : in_hi;
          unsigned char* dst = act_smem + (size_t)part * stage_bytes;
          for (int dzi = 0; dzi < 3; ++dzi)
            for (int cc = 0; cc < nch; ++cc)
              sm100::bulk_g2s(dst + (size_t)(dzi * nch + cc) * seg_rows * 16,
                              in + ((size_t)cc * g.rows_alloc + g.guard + r0 + (dzi - 1) * g.pp - g.halo) * 8,
                              (uint32_t)seg_rows * 16, &c.mb_full[0]);
        }
      }
      __syncwarp();
      ++c.load_cnt;
    }
  } else if (c.warp == kMmaWarp) {
    mbar_wait(c, &c.mb_w[0], bit_get(c, 0));
    const uint32_t idesc = sm100::umma_idesc_f16(kTileM, kStackN);
    const uint64_t hi = (uint64_t)((128u >> 4) | (1u << 14)) << 32;
    const uint32_t bw_hi = ((sm100::smem_u32(c.smem) >> 4) & 0x3FFFu) | ((12u * 128u >> 4) << 16);
    const uint32_t bw_lo = ((sm100::smem_u32(c.smem + 27 * 4 * 512) >> 4) & 0x3FFFu) | ((12u * 128u >> 4) << 16);
    const uint32_t aa_hi = ((sm100::smem_u32(act_smem) >> 4) & 0x3FFFu) | ((uint32_t)seg_rows << 16);
    const uint32_t aa_lo = ((sm100::smem_u32(act_smem + stage_bytes) >> 4) & 0x3FFFu) | ((uint32_t)seg_rows << 16);
    for (int j = 0; j < ntiles; ++j) {
      const int slot = c.mma_cnt % kAccSlots;
      mbar_wait(c, &c.mb_full[0], c.mma_cnt & 1u);
      mbar_wait(c, &c.mb_tempty[slot], ((c.mma_cnt / kAccSlots) & 1u) ^ 1u);
      sm100::tc_fence_after();
      const uint32_t d = c.tmem_base + (uint32_t)(slot * kStackN);
      if (sm100::elect_one()) {
        // The tensor core truncates when it aligns an MMA's sum to the accumulator, so the error of every
        // accumulation scales with the accumulator's magnitude: the small cross terms (a_lo*w_hi, a_hi*w_lo,
        // ~2^-11 of the result) go in FIRST, while the accumulator is small, the 9*nch/2 main MMAs last.
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
#pragma unroll 1
          for (int row = 0; row < 9; ++row) {
            const int tz = row / 3, ty = row % 3;
            for (int jj = 0; jj < nch / 2; ++jj) {
              const uint32_t aoff = (uint32_t)((tz * nch + 2 * jj) * seg_rows + ty * g.xp);
              const uint32_t boff = (uint32_t)((row * nch + 2 * jj) * (12 * 128 / 16));
              if (pass == 0) {
                sm100::umma_f16(d, hi | (uint64_t)(aa_lo + aoff), hi | (uint64_t)(bw_hi + boff), idesc, (row | jj) != 0 ? 1u : 0u);
                sm100::umma_f16(d, hi | (uint64_t)(aa_hi + aoff), hi | (uint64_t)(bw_lo + boff), idesc, 1u);
              } else {
                sm100::umma_f16(d, hi | (uint64_t)(aa_hi + aoff), hi | (uint64_t)(bw_hi + boff), idesc, 1u);
              }
            }
          }
        }
        sm100::umma_commit(&c.mb_tfull[slot]);
        sm100::umma_commit(&c.mb_empty[0]);
      }
      __syncwarp();
      ++c.mma_cnt;
    }
  } else if (c.warp < 8) {
    if (last) {
      hit = layer == 1 ? tc_epilogue<EPI_LAST0, true>(c, 0, layer, ntiles) : tc_epilogue<EPI_LAST, true>(c, 0, layer, ntiles);
    } else if (!(layer & 1)) {
      tc_epilogue<EPI_A, true>(c, 0, layer, ntiles);
    } else if (layer == 1) {
      tc_epilogue<EPI_B_FIRST, true>(c, 0, layer, ntiles);
    } else {
      tc_epilogue<EPI_B, true>(c, 0, layer, ntiles);
    }
    if (last) publish_counts(c, 0, hit);
  }
  bit_flip(c, 0);
  bit_set(c, 8, false);
}

// ------------------------------------------------------------------------------------------
// fp32 layer ("precise" parity mode): one thread per FoV row, 32 accumulators, weights
// broadcast from shared memory, activations through L1.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void f32_layer(Ctx& c, int layer) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const int ngrp = layer == 0 ? 1 : 8;           // input groups of 4 channels
  const int cin = ngrp * 4;
  const float4* in = layer == 0 ? p.ws.act0_f : p.ws.act_f[(layer - 1) & 1];
  float* wsm = reinterpret_cast<float*>(c.smem);
  {
    const float4* src = reinterpret_cast<const float4*>(p.w.w32 + w32_layer_offset_floats(layer));
    float4* dst = reinterpret_cast<float4*>(wsm);
    const int n4 = 27 * cin * 32 / 4;
    for (int i = c.tid; i < n4; i += kThreads) dst[i] = __ldg(src + i);
  }
  __syncthreads();
  int hit = 0;
  for (int r = c.t_begin * kTileOut + c.tid; r < c.t_end * kTileOut; r += kThreads) {
    int z, y, x;
    if (!row_to_zyx(g, r, z, y, x)) continue;
    float v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = 0.f;
    for (int tap = 0; tap < 27; ++tap) {
      const int tx = tap % 3;
      if ((tx == 0 && x == 0) || (tx == 2 && x == g.fx - 1)) continue;   // SAME padding in x
      const int off = (tap / 9 - 1) * g.pp + ((tap / 3) % 3 - 1) * g.xp + (tx - 1);
      const float4* a = in + (size_t)g.guard + r + off;
      const float* wt = wsm + (size_t)tap * cin * 32;
      for (int q = 0; q < ngrp; ++q) {
        const float4 av = a[(size_t)q * g.rows_alloc];
        const float ain[4] = {av.x, av.y, av.z, av.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float4* w4 = reinterpret_cast<const float4*>(wt + (q * 4 + e) * 32);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float4 w = w4[k];
            v[4 * k + 0] = fmaf(ain[e], w.x, v[4 * k + 0]);
            v[4 * k + 1] = fmaf(ain[e], w.y, v[4 * k + 1]);
            v[4 * k + 2] = fmaf(ain[e], w.z, v[4 * k + 2]);
            v[4 * k + 3] = fmaf(ain[e], w.w, v[4 * k + 3]);
          }
        }
      }
    }
    epilogue_row(c, layer, r, v, hit);
  }
  if (layer == g.nconv - 1) {
    hit = __reduce_add_sync(0xffffffffu, hit);
    if (c.lane == 0 && hit) atomicAdd(&c.s_misc[0], hit);
    __syncthreads();
    if (c.tid == 0 && c.s_misc[0]) {
      const unsigned packed = (unsigned)c.s_misc[0];
      unsigned* cnt = p.ch[0].count + 2 * (c.round & 1u);
      if (packed & 0xffffu) atomicAdd(cnt, packed & 0xffffu);
      if (packed >> 16) atomicAdd(cnt + 1, packed >> 16);
    }
  }
  __syncthreads();
}

// Parity modes (fp32 FMA / split fp16): the conv stack of chain 0 with a whole-grid barrier after every
// layer.  On return the caller's end-of-round grid barrier makes logits and counts visible.
__device__ __forceinline__ void layers_blocking(Ctx& c) {
  const KParams& p = *c.p;
  grid_barrier(c);   // staged operands visible
  for (int layer = 0; layer < p.g.nconv; ++layer) {
    if (p.compute_mode == FFN_COMPUTE_FP16X2_TC) {
      tc_layer_x2(c, layer);
    } else {
      f32_layer(c, layer);
    }
    if (layer + 1 < p.g.nconv) grid_barrier(c);
  }
}

// Paste this CTA's rows of chain k's last step into the seed canvas (inference.py:439) / the prediction
// output.  `par` = round parity the step was staged with.
__device__ __forceinline__ void tail_paste(Ctx& c, int k, int b, unsigned par, int pz, int py, int px, int batch_idx, bool disco) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const ChainDev& ch = p.ch[k];
  const bool predict = p.job.mode == MODE_PREDICT;
  for (int r = c.t_begin * kTileOut + c.tid; r < c.t_end * kTileOut; r += kThreads) {
    int z, y, x;
    if (!row_to_zyx(g, r, z, y, x)) continue;
    const size_t fi = ((size_t)z * g.fy + y) * g.fx + x;
    if (predict) {
      p.job.out_logits[(size_t)batch_idx * g.V + fi] = __ldcg(ch.logits + r);
      continue;
    }
    const float m = merged_row(p, k, par, r, disco);
    const size_t i = ((size_t)(pz - g.mz + z) * p.cv.sy + (py - g.my + y)) * p.cv.sx + (px - g.mx + x);
    p.ob[b].seed[i] = m;
    if (p.job.mode == MODE_UPDATE_AT && p.job.pred_out) p.job.pred_out[fi] = m;
  }
}

// ------------------------------------------------------------------------------------------
// Leader logic (CTA 0): movement policy, validity, object / canvas loops, the scheduler
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ size_t cv_index(const CanvasDev& cv, int z, int y, int x) {
  return ((size_t)z * cv.sy + y) * cv.sx + x;
}

__device__ __forceinline__ int floordiv(int a, int b) {
  int q = a / b;
  if ((a % b != 0) && ((a < 0) != (b < 0))) --q;
  return q;
}

// movement.py:200-208 quantize_pos -> index into the epoch-stamped lattice.
__device__ __forceinline__ size_t lattice_index(const KParams& p, const CanvasState* st, int z, int y, int x) {
  const Geom& g = p.g;
  const int qz = floordiv(z - st->start[0] + g.dz / 2, max(g.dz, 1)) + p.cv.lat_off[0];
  const int qy = floordiv(y - st->start[1] + g.dy / 2, max(g.dy, 1)) + p.cv.lat_off[1];
  const int qx = floordiv(x - st->start[2] + g.dx / 2, max(g.dx, 1)) + p.cv.lat_off[2];
  return ((size_t)qz * p.cv.lat_dim[1] + qy) * p.cv.lat_dim[2] + qx;
}

// Leader-side view of one chain: k, its state copy, the parity its last step was staged with, its disco flag.
struct LChain {
  int k;                 // chain (workspace of the step)
  int b;                 // object buffer (seed array, queue, done set, trajectory)
  CanvasState* st;
  unsigned par;
  bool disco;
};

// Current value of chain.seed[z,y,x] as the reference would see it after the paste of the step
// at `cur` (which other CTAs may still be writing): inside that FoV use the merged logits.
__device__ __forceinline__ float seed_value(const KParams& p, const LChain& L, int z, int y, int x) {
  const Geom& g = p.g;
  const CanvasState* st = L.st;
  if (st->have_cur) {
    const int fz = z - (st->cur[0] - g.mz), fy = y - (st->cur[1] - g.my), fx = x - (st->cur[2] - g.mx);
    if (fz >= 0 && fz < g.fz && fy >= 0 && fy < g.fy && fx >= 0 && fx < g.fx)
      return merged_row(p, L.k, L.par, fz * g.pp + fy * g.xp + fx, L.disco);
  }
  return __ldcg(p.ob[L.b].seed + cv_index(p.cv, z, y, x));
}

// Optional event log for debugging / history export (one chain only; lane 0 of the leader warp).
enum TraceEvent : int { EV_PUSH = 1, EV_POP_VALID = 2, EV_POP_INVALID = 3, EV_POP_THRESHOLD = 4, EV_POP_DONE = 5,
                        EV_STEP = 6, EV_SEED_INVALID = 7, EV_SEED_START = 8, EV_DELETED = 9 };
__device__ __forceinline__ void trace_event(const KParams& p, CanvasState* st, int type, int z, int y, int x) {
  if (!p.cv.trace) return;
  const int i = st->n_trace++;
  if (i < p.cv.trace_cap) {
    p.cv.trace[4 * i] = type;
    p.cv.trace[4 * i + 1] = z;
    p.cv.trace[4 * i + 2] = y;
    p.cv.trace[4 * i + 3] = x;
  }
}

__device__ __forceinline__ void push_move(const KParams& p, const LChain& L, float score, int z, int y, int x) {
  CanvasState* st = L.st;
  if (st->q_tail >= p.cv.q_cap) {
    st->overflow |= 1;
    return;
  }
  const int t = st->q_tail++;
  trace_event(p, st, EV_PUSH, z, y, x);
  p.ob[L.b].q_score[t] = score;
  p.ob[L.b].q_pos[3 * t + 0] = z;
  p.ob[L.b].q_pos[3 * t + 1] = y;
  p.ob[L.b].q_pos[3 * t + 2] = x;
}

// Policy scratch of chain k in shared memory: score[6] floats, rel[6][3], ok[6].
__device__ __forceinline__ int* policy_scratch(const Ctx& c, int k) { return c.s_misc + kMiscScratch + 32 * k; }

// movement.get_scored_move_offsets (movement.py:42-100) for ONE face of the step just executed at
// st->cur: arg-max of the merged logits over the face (first index, C order); one warp, every load of
// the face in flight at once.
__device__ __forceinline__ void face_argmax(const Ctx& c, const LChain& L, int face) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const ChainDev& ch = p.ch[L.k];
  int* scr = policy_scratch(c, L.k);
  float* s_score = reinterpret_cast<float*>(scr);
  int* s_rel = scr + 8;     // [6][3]
  int* s_ok = scr + 26;     // [6]
  const int cz = g.fz / 2, cy = g.fy / 2, cx = g.fx / 2;
  const int axis = face >> 1;
  const int dax = axis == 0 ? g.dz : (axis == 1 ? g.dy : g.dx);
  const int off = (face & 1) ? dax : -dax;
  // the two in-face axes in their original (C) order: (y,x) for z faces, (z,x) for y, (z,y) for x
  const int d0 = axis == 0 ? g.dy : g.dz;
  const int d1 = axis == 2 ? g.dy : g.dx;
  const int n0 = 2 * d0 + 1, n1 = 2 * d1 + 1;
  const float* lgp = ch.logits;
  const float* odp = ch.seed_raw[L.par];
  int ok = 0;
  if (dax != 0) {
    float best = -CUDART_INF_F;
    int best_i = 0x7fffffff;
    constexpr int kPerLane = 10;   // 320 >= 17 x 17 face elements: one L2 round trip for a whole face
    for (int base = c.lane; base < n0 * n1; base += 32 * kPerLane) {
      float lg[kPerLane], od[kPerLane];
#pragma unroll
      for (int u = 0; u < kPerLane; ++u) {
        const int e = base + 32 * u;
        lg[u] = 0.f;
        od[u] = 0.f;
        if (e < n0 * n1) {
          const int i0 = e / n1, i1 = e - i0 * n1;
          const int z = axis == 0 ? cz + off : cz - g.dz + i0;
          const int y = axis == 0 ? cy - g.dy + i0 : (axis == 1 ? cy + off : cy - g.dy + i1);
          const int x = axis == 2 ? cx + off : cx - g.dx + i1;
          const int row = z * g.pp + y * g.xp + x;
          lg[u] = __ldcg(lgp + row);
          if (L.disco) od[u] = __ldcg(odp + row);
        }
      }
#pragma unroll
      for (int u = 0; u < kPerLane; ++u) {
        const int e = base + 32 * u;
        if (e < n0 * n1) {
          float v = lg[u];
          if (L.disco && od[u] < 0.f && v > od[u]) v = od[u];
          if (v > best || best_i == 0x7fffffff) {
            best = v;
            best_i = e;
          }
        }
      }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, s);
      const int oi = __shfl_xor_sync(0xffffffffu, best_i, s);
      if (oi != 0x7fffffff && (best_i == 0x7fffffff || ov > best || (ov == best && oi < best_i))) {
        best = ov;
        best_i = oi;
      }
    }
    if (c.lane == 0) {
      // movement.py:84-86: skip when score < threshold (float64 compare == f32 compare against
      // the smallest float32 >= threshold)
      ok = (best >= p.cv.policy_th_f32) ? 1 : 0;
      const int i0 = best_i / n1, i1 = best_i - i0 * n1;
      const int r0 = i0 - n0 / 2, r1 = i1 - n1 / 2;
      s_score[face] = best;
      s_rel[3 * face + 0] = axis == 0 ? off : r0;
      s_rel[3 * face + 1] = axis == 0 ? r0 : (axis == 1 ? off : r1);
      s_rel[3 * face + 2] = axis == 2 ? off : r1;
    }
  }
  if (c.lane == 0) s_ok[face] = ok;
}

// FaceMaxMovementPolicy.update (movement.py:210-222) once the six faces are reduced: lanes 0-5 of ONE warp
// each own one face's move and work out, with shuffles, whether it is a duplicate and its rank in the
// descending (score, (dz, dy, dx)) order — the position it is written to in the queue.  (No dynamically
// indexed local arrays here: local memory lives behind the L1 that every acquire invalidates.)
__device__ __forceinline__ void policy_finish(const Ctx& c, const LChain& L) {
  const KParams& p = *c.p;
  const ObjDev& ob = p.ob[L.b];
  CanvasState* st = L.st;
  int* scr = policy_scratch(c, L.k);
  const float* s_score = reinterpret_cast<const float*>(scr);
  const int* s_rel = scr + 8;
  const int* s_ok = scr + 26;
  const unsigned full = 0xffffffffu;
  const int f = c.lane;
  const bool mine = f < 6 && s_ok[f] != 0;
  const float sc = f < 6 ? s_score[f] : 0.f;
  const int rz = f < 6 ? s_rel[3 * f] : 0, ry = f < 6 ? s_rel[3 * f + 1] : 0, rx = f < 6 ? s_rel[3 * f + 2] : 0;
  // movement.py:95-99: identical (score, offset) tuples are yielded once — two faces share an
  // edge, and the same edge voxel can be the arg-max of both: the later face's copy is dropped
  bool dropped = false;
#pragma unroll
  for (int h = 0; h < 5; ++h) {
    const bool oh = __shfl_sync(full, (int)mine, h) != 0;
    const float sh = __shfl_sync(full, sc, h);
    const int zh = __shfl_sync(full, rz, h), yh = __shfl_sync(full, ry, h), xh = __shfl_sync(full, rx, h);
    if (h < f && oh && sh == sc && zh == rz && yh == ry && xh == rx) dropped = true;
  }
  const bool keep = mine && !dropped;
  // sorted(..., reverse=True) on (score, (dz, dy, dx)) tuples (movement.py:218): rank = kept moves ahead of mine
  int rank = 0;
#pragma unroll
  for (int h = 0; h < 6; ++h) {
    const bool kh = __shfl_sync(full, (int)keep, h) != 0;
    const float sh = __shfl_sync(full, sc, h);
    const int zh = __shfl_sync(full, rz, h), yh = __shfl_sync(full, ry, h), xh = __shfl_sync(full, rx, h);
    bool ahead = sh > sc;
    if (sh == sc) ahead = zh != rz ? zh > rz : (yh != ry ? yh > ry : xh > rx);
    if (kh && h != f && ahead) ++rank;
  }
  const int n = __popc(__ballot_sync(full, keep));
  const int tail = st->q_tail;
  const int room = max(p.cv.q_cap - tail, 0);
  if (keep && rank < room) {
    const int t = tail + rank;
    ob.q_score[t] = sc;
    ob.q_pos[3 * t + 0] = st->cur[0] + rz;
    ob.q_pos[3 * t + 1] = st->cur[1] + ry;
    ob.q_pos[3 * t + 2] = st->cur[2] + rx;
  }
  __syncwarp();
  if (c.lane == 0) {
    ob.lattice[lattice_index(p, st, st->cur[0], st->cur[1], st->cur[2])] = st->epoch;
    if (n > room) st->overflow |= 1;
    const int wrote = min(n, room);
    if (p.cv.trace) {
      for (int i = 0; i < wrote; ++i)
        trace_event(p, st, EV_PUSH, __ldcg(ob.q_pos + 3 * (tail + i)), __ldcg(ob.q_pos + 3 * (tail + i) + 1),
                    __ldcg(ob.q_pos + 3 * (tail + i) + 2));
    }
    st->q_tail = tail + wrote;
  }
  __syncwarp();
}

// FaceMaxMovementPolicy.__next__ (movement.py:186-198) + Canvas.is_valid_pos (inference.py:312-346)
// for queue entries; lane 0 only (used while the event trace records: per-candidate events in order).
__device__ __forceinline__ bool pop_next(const KParams& p, const LChain& L, int& z, int& y, int& x) {
  const Geom& g = p.g;
  const ObjDev& ob = p.ob[L.b];
  CanvasState* st = L.st;
  while (st->q_head < st->q_tail) {
    const int h = st->q_head++;
    z = __ldcg(ob.q_pos + 3 * h);
    y = __ldcg(ob.q_pos + 3 * h + 1);
    x = __ldcg(ob.q_pos + 3 * h + 2);
    const unsigned stamp = __ldcg(ob.lattice + lattice_index(p, st, z, y, x));
    const bool inside = z >= 0 && y >= 0 && x >= 0 && z < p.cv.sz && y < p.cv.sy && x < p.cv.sx;
    float v = 0.f;
    int sg = 0;
    if (inside) {
      sg = __ldcg(p.cv.seg + cv_index(p.cv, z, y, x));
      v = seed_value(p, L, z, y, x);
    }
    if (stamp == st->epoch) {
      trace_event(p, st, EV_POP_DONE, z, y, x);
      continue;
    }
    if (inside && v < p.cv.opt.move_threshold) {
      st->ctr.skip_threshold++;
      trace_event(p, st, EV_POP_THRESHOLD, z, y, x);
      continue;
    }
    if (z - g.mz < 0 || y - g.my < 0 || x - g.mx < 0 || z + g.mz >= p.cv.sz || y + g.my >= p.cv.sy ||
        x + g.mx >= p.cv.sx || sg > 0) {
      st->ctr.skip_invalid_pos++;
      trace_event(p, st, EV_POP_INVALID, z, y, x);
      continue;
    }
    trace_event(p, st, EV_POP_VALID, z, y, x);
    return true;
  }
  return false;
}

// quantize_probability(expit(v)) (storage.py:137-143, inference.py:655-657).
__device__ __forceinline__ uint8_t quantize_prob(float logit) {
  const float pf = 1.0f / (1.0f + expf(-logit));
  const double pd = (double)pf;
  int k = (int)(pd * 254.0);
  if (k > 254) k = 254;
  if (k < 0) k = 0;
  const double step = 1.0 / 254.0;
  // bins[j] = j * step for j < 254, bins[254] = 1.0 ; result = #bins <= p
  while (k < 254 && ((k + 1 == 254) ? 1.0 : (double)(k + 1) * step) <= pd) ++k;
  while (k > 0 && ((k == 254) ? 1.0 : (double)k * step) > pd) --k;
  return (uint8_t)(k + 1);
}

// FaceMaxMovementPolicy.__next__ + Canvas.is_valid_pos + the per-step checks of segment_at
// (inference.py:503-509) as a WARP-collective: lane i examines queue entry head + i, so a run of
// rejected candidates costs two L2 round trips instead of two per candidate.  Exactly equivalent to the
// sequential loop: a candidate's verdict depends only on state that pops do not modify (the done
// lattice, the seed / label canvases, the masks), and the counters of the rejected candidates in
// front of the first accepted one are added up from the ballot masks.
// Returns true (all lanes) with the next position in z / y / x.
__device__ __forceinline__ bool warp_pop(const KParams& p, const LChain& L, int lane, int& z, int& y, int& x) {
  const Geom& g = p.g;
  const CanvasDev& cv = p.cv;
  const ChainDev& ch = p.ch[L.k];
  const ObjDev& ob = p.ob[L.b];
  CanvasState* st = L.st;
  // inference.py:503-505: value of the object's start voxel — the same for every candidate of this call
  const bool weak = seed_value(p, L, st->start[0], st->start[1], st->start[2]) < cv.opt.move_threshold;
  for (;;) {
    const int head = st->q_head, n = st->q_tail - head;
    __syncwarp();   // every lane has read the queue bounds before lane 0 advances them
    if (n <= 0) return false;
    const bool act = lane < n;
    int cz = 0, cy = 0, cx = 0, cls = 0;   // 0 done, 1 below threshold, 2 invalid, 3 valid
    bool restricted = false;
    if (act) {
      const int h = head + lane;
      cz = __ldcg(ob.q_pos + 3 * h);
      cy = __ldcg(ob.q_pos + 3 * h + 1);
      cx = __ldcg(ob.q_pos + 3 * h + 2);
      const unsigned stamp = __ldcg(ob.lattice + lattice_index(p, st, cz, cy, cx));
      const bool inside = cz >= 0 && cy >= 0 && cx >= 0 && cz < cv.sz && cy < cv.sy && cx < cv.sx;
      float v = 0.f, old = 0.f;
      int sg = 0;
      bool in_fov = false;
      if (inside) {
        const size_t i = cv_index(cv, cz, cy, cx);
        sg = __ldcg(cv.seg + i);
        if (cv.mask) restricted = __ldg(cv.mask + i) != 0;
        if (st->have_cur) {
          const int fz = cz - (st->cur[0] - g.mz), fy = cy - (st->cur[1] - g.my), fx = cx - (st->cur[2] - g.mx);
          in_fov = fz >= 0 && fz < g.fz && fy >= 0 && fy < g.fy && fx >= 0 && fx < g.fx;
          if (in_fov) {
            const int row = fz * g.pp + fy * g.xp + fx;
            v = __ldcg(ch.logits + row);
            old = __ldcg(ch.seed_raw[L.par] + row);
          }
        }
        if (!in_fov) v = __ldcg(ob.seed + i);
      }
      if (in_fov && L.disco && old < 0.f && v > old) v = old;
      const bool border = cz - g.mz < 0 || cy - g.my < 0 || cx - g.mx < 0 || cz + g.mz >= cv.sz ||
                          cy + g.my >= cv.sy || cx + g.mx >= cv.sx;
      if (stamp == st->epoch) {
        cls = 0;
      } else if (inside && v < cv.opt.move_threshold) {
        cls = 1;
      } else if (border || sg > 0) {
        cls = 2;
      } else {
        cls = 3;
      }
    }
    const unsigned full = 0xffffffffu;
    const unsigned m_act = __ballot_sync(full, act);
    const unsigned m_thr = __ballot_sync(full, act && cls == 1);
    const unsigned m_inv = __ballot_sync(full, act && cls == 2);
    const unsigned m_res = __ballot_sync(full, act && cls == 3 && !weak && restricted);
    const unsigned m_stop = __ballot_sync(full, act && cls == 3 && (weak || !restricted));
    const int f = m_stop ? __ffs(m_stop) - 1 : -1;
    const unsigned before = f >= 0 ? ((1u << f) - 1u) : m_act;
    if (st->seg_all) {
      // Candidates that passed Canvas.is_valid_pos without being stepped on — skipped by the restrictor
      // (inference.py:507-509), or the one in hand when the loop ends with 'seed_got_too_weak' (:503-505) — relied on
      // `segmentation <= 0` like a FoV step does: an object run ahead of its turn is only the reference's run if they
      // are still unlabelled when its turn comes (run_conflicts), so they go into the trajectory log, from its end.
      const unsigned m_log = (m_res & before) | ((f >= 0 && weak) ? (1u << f) : 0u);
      if (m_log) {
        const int slot = st->n_unstepped + __popc(m_log & ((1u << lane) - 1u));
        if ((m_log >> lane) & 1u) {
          if (st->iters + slot + 1 < (long long)p.cv.traj_cap) {
            int* t = ob.traj + 3 * ((long long)p.cv.traj_cap - 1 - slot);
            t[0] = cz;
            t[1] = cy;
            t[2] = cx;
          }
        }
        __syncwarp();   // every lane has read n_unstepped
        if (lane == 0) {
          if (st->iters + st->n_unstepped + __popc(m_log) + 1 >= (long long)p.cv.traj_cap) st->overflow |= 8;
          st->n_unstepped += __popc(m_log);
        }
      }
    }
    if (lane == 0) {
      st->ctr.skip_threshold += __popc(m_thr & before);
      st->ctr.skip_invalid_pos += __popc(m_inv & before);
      st->ctr.skip_restricted_pos += __popc(m_res & before);
      st->q_head = head + (f >= 0 ? f + 1 : __popc(m_act));
      if (f >= 0 && weak) {
        st->ctr.seed_got_too_weak++;
        st->weak = 1;
      }
    }
    __syncwarp();
    if (f >= 0) {
      z = __shfl_sync(full, cz, f);
      y = __shfl_sync(full, cy, f);
      x = __shfl_sync(full, cx, f);
      return !weak;
    }
  }
}

// The serial reference of warp_pop (lane 0 only): used when the event trace is recording, which
// needs the per-candidate events in order.
__device__ __forceinline__ bool serial_pop(const KParams& p, const LChain& L, int& z, int& y, int& x) {
  const CanvasDev& cv = p.cv;
  CanvasState* st = L.st;
  for (;;) {
    if (!pop_next(p, L, z, y, x)) return false;
    // inference.py:503-505
    if (seed_value(p, L, st->start[0], st->start[1], st->start[2]) < cv.opt.move_threshold) {
      st->ctr.seed_got_too_weak++;
      st->weak = 1;
      return false;
    }
    // inference.py:507-509
    if (cv.mask && cv.mask[cv_index(cv, z, y, x)]) {
      st->ctr.skip_restricted_pos++;
      continue;
    }
    return true;
  }
}

// Pops the chain's queue (warp-collective) and parks the outcome in the state: the decision is then the
// same whether this round goes on or the launch pauses (step budget) and a later launch resumes.
__device__ __forceinline__ void chain_pop(const Ctx& c, const LChain& L) {
  const KParams& p = *c.p;
  CanvasState* st = L.st;
  const long long t_pop = prof_now(c);
  int z = 0, y = 0, x = 0;
  bool run;
  if (p.cv.trace) {
    run = false;
    if (c.lane == 0) run = serial_pop(p, L, z, y, x);
    run = __shfl_sync(0xffffffffu, (int)run, 0) != 0;
    z = __shfl_sync(0xffffffffu, z, 0);
    y = __shfl_sync(0xffffffffu, y, 0);
    x = __shfl_sync(0xffffffffu, x, 0);
  } else {
    run = warp_pop(p, L, c.lane, z, y, x);
  }
  if (c.lane == 0) {
    st->popped = 1;
    st->pop_run = run ? 1 : 0;
    st->pop_pos[0] = z;
    st->pop_pos[1] = y;
    st->pop_pos[2] = x;
    prof_add(c, 13, prof_now(c) - t_pop);
  }
  __syncwarp();
}

// What follows a FoV step of chain L.k (one warp): policy update, bookkeeping of segment_at
// (inference.py:511-521), then the pop that decides the next step.
__device__ __forceinline__ void after_step(const Ctx& c, const LChain& L) {
  const KParams& p = *c.p;
  CanvasState* st = L.st;
  if (p.job.mode == MODE_UPDATE_AT) return;       // Canvas.update_at driven from the host: no policy
  policy_finish(c, L);                             // movement.py:210-222
  if (c.lane == 0) {
    if (p.cv.trace && p.cv.opt.disco_seed_threshold >= 0.f)
      trace_event(p, st, EV_DELETED, (int)__ldcg(p.ch[L.k].count + 2 * L.par + 1), 0, 0);   // inference.py:420-422
    for (int q = 0; q < 3; ++q) {
      st->min_pos[q] = min(st->min_pos[q], st->cur[q]);
      st->max_pos[q] = max(st->max_pos[q], st->cur[q]);
    }
    if (st->seg_all) {   // trajectory: the positions whose `segmentation <= 0` test this object relied on
      if (st->iters + st->n_unstepped < (long long)p.cv.traj_cap) {
        int* t = p.ob[L.b].traj + 3 * st->iters;
        t[0] = st->cur[0];
        t[1] = st->cur[1];
        t[2] = st->cur[2];
      } else {
        st->overflow |= 8;
      }
    }
    st->iters++;
    st->ctr.inference_calls++;
    st->phase = PH_POP;
    st->popped = 0;
  }
  __syncwarp();
  chain_pop(c, L);
}

// ---- seed gating (inference.py:562-581 + the border filter of seed.py:81-88), warp-collective ----------
// final = true : the in-order gating of the reference, with its side effects (counters, -1 markers);
// final = false: a side-effect-free preview used to pick seeds that are worth starting ahead of their turn.
// Returns 1 = accept, 0 = reject.
__device__ __forceinline__ int gate_seed(const Ctx& c, Sched* sc, long long idx, bool final, int& sz, int& sy, int& sx) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const CanvasDev& cv = p.cv;
  sz = __ldg(p.job.seeds + 3 * idx);
  sy = __ldg(p.job.seeds + 3 * idx + 1);
  sx = __ldg(p.job.seeds + 3 * idx + 2);
  // seed.py:81-88 border filter (BaseSeedPolicy.__next__)
  if (sz - g.mz < 0 || sy - g.my < 0 || sx - g.mx < 0 || sz + g.mz >= cv.sz || sy + g.my >= cv.sy || sx + g.mx >= cv.sx)
    return 0;
  const size_t i = cv_index(cv, sz, sy, sx);
  const int* mbd = cv.opt.min_boundary_dist_zyx;
  const int z0 = max(sz - mbd[0], 0), z1 = min(sz + mbd[0] + 1, cv.sz);
  const int y0 = max(sy - mbd[1], 0), y1 = min(sy + mbd[1] + 1, cv.sy);
  const int x0 = max(sx - mbd[2], 0), x1 = min(sx + mbd[2] + 1, cv.sx);
  const int ny = y1 - y0, nx = x1 - x0, total = (z1 - z0) * ny * nx;
  // everything the verdict depends on, issued together
  const int sg = __ldcg(cv.seg + i);
  const bool masked = (cv.mask && __ldg(cv.mask + i)) || (cv.seed_mask && __ldg(cv.seed_mask + i));
  bool close = false;   // inference.py:573-581 (numpy slice semantics clamp at the canvas border)
  for (int e = c.lane; e < total; e += 32) {
    const int zz = z0 + e / (ny * nx), rem = e % (ny * nx);
    if (__ldcg(cv.seg + cv_index(cv, zz, y0 + rem / nx, x0 + rem % nx)) > 0) close = true;
  }
  close = __any_sync(0xffffffffu, close);
  if (final && c.lane == 0) sc->ctr.seeds_examined++;
  if (sg > 0) {                                  // Canvas.is_valid_pos(pos, ignore_move_threshold=True), inference.py:562-568
    if (final && c.lane == 0) {
      sc->ctr.skip_invalid_pos++;
      trace_event(p, chain_state(c, 0), EV_SEED_INVALID, sz, sy, sx);
    }
    return 0;
  }
  if (masked) return 0;
  if (close) {
    if (final && c.lane == 0) cv.seg[i] = -1;
    return 0;
  }
  return 1;
}

// Did any FoV position of the (early) run get a label since it was tested?  Warp-collective.
__device__ __forceinline__ bool run_conflicts(const Ctx& c, int b, const CanvasState* st) {
  const KParams& p = *c.p;
  bool bad = false;
  const long long n = min(st->iters, (long long)p.cv.traj_cap);
  for (long long i = c.lane; i < n; i += 32) {
    const int* t = p.ob[b].traj + 3 * i;
    if (__ldcg(p.cv.seg + cv_index(p.cv, __ldcg(t), __ldcg(t + 1), __ldcg(t + 2))) > 0) bad = true;
  }
  // ... or any position it popped as valid without stepping on it (see warp_pop)
  for (long long i = c.lane; i < min((long long)st->n_unstepped, (long long)p.cv.traj_cap - n); i += 32) {
    const int* t = p.ob[b].traj + 3 * ((long long)p.cv.traj_cap - 1 - i);
    if (__ldcg(p.cv.seg + cv_index(p.cv, __ldcg(t), __ldcg(t + 1), __ldcg(t + 2))) > 0) bad = true;
  }
  return __any_sync(0xffffffffu, bad);
}

__device__ __forceinline__ void start_object(CanvasState* st, const Sched* sc, long long idx, int spec, int sz, int sy, int sx) {
  st->seed_index = idx;
  st->start_max_id = sc->max_id;
  st->spec = spec;
  st->start[0] = sz;
  st->start[1] = sy;
  st->start[2] = sx;
  st->reset_seed = 1;
  st->phase = PH_START_SEGMENT;
}

// The seed at the head of the line has been dealt with.
__device__ __forceinline__ void finalize_seed(Sched* sc, CanvasState* st) {
  if (st->seed_index >= 0) sc->commit_idx = st->seed_index + 1;
  sc->owner = -1;
  st->seed_index = -1;
  st->spec = 0;
  st->phase = PH_FREE;
}

// The head of the line (warp-collective; lane 0 mutates): while nobody holds the seed at commit_idx, gate it in
// order (the reference's loop, inference.py:552-581) and run the first accepted one HERE, in turn, in the free
// buffer L.b of chain k.  Stops when an object in flight (running, parked or suspended, in any buffer) holds the
// seed: that buffer becomes the owner.
__device__ __forceinline__ void advance_pointer(const Ctx& c, const LChain& L, Sched* sc) {
  const KParams& p = *c.p;
  CanvasState* st = L.st;
  while (sc->owner < 0 && sc->commit_idx < p.job.n_seeds) {
    const long long i = sc->commit_idx;
    __syncwarp();   // reads of this iteration before lane 0's writes
    if (__ldcg(p.job.seed_status + i) != 0) {      // an early run holds it: its buffer is now at the head of the line
      int who = -1;
      for (int q = 0; q < p.nchains; ++q)
        if (chain_state(c, q)->seed_index == i && chain_state(c, q)->phase != PH_FREE) who = sc->active[q];
      for (int b = 0; b < p.nchains * kBufsPerChain; ++b)
        if ((sc->bkind[b] == 1 || sc->bkind[b] == 2) && sc->bseed[b] == i) who = b;
      if (c.lane == 0) sc->owner = who;
      __syncwarp();
      if (who < 0) {   // cannot happen; do not spin on it
        if (c.lane == 0) sc->commit_idx = i + 1;
        __syncwarp();
        continue;
      }
      break;
    }
    int sz, sy, sx;
    const int ok = gate_seed(c, sc, i, true, sz, sy, sx);
    if (c.lane == 0) {
      if (ok) {
        p.job.seed_status[i] = 1;
        sc->owner = L.b;
        start_object(st, sc, i, 0, sz, sy, sx);
      } else {
        sc->commit_idx = i + 1;
      }
    }
    __syncwarp();
    if (ok) return;
  }
}

// Look ahead for a seed worth starting early in the free buffer L.b: not taken, would pass the gating as things
// stand, and not next to an object a chain is growing right now (warp-collective; lane 0 mutates).
__device__ __forceinline__ void lookahead(const Ctx& c, const LChain& L, Sched* sc) {
  const KParams& p = *c.p;
  const int k = L.k;
  CanvasState* st = L.st;
  const unsigned full = 0xffffffffu;
  if (sc->owner == L.b || p.nchains == 1 || (p.job.debug & 2)) return;
  constexpr int kWindow = 256;
  const long long base = sc->commit_idx + 1;
  for (int w = 0; w < kWindow; w += 32) {
    const long long j = base + w + c.lane;
    bool ok = j < p.job.n_seeds && __ldcg(p.job.seed_status + (j < p.job.n_seeds ? j : 0)) == 0;
    int sz = 0, sy = 0, sx = 0;
    if (ok) {
      const Geom& g = p.g;
      const CanvasDev& cv = p.cv;
      sz = __ldg(p.job.seeds + 3 * j);
      sy = __ldg(p.job.seeds + 3 * j + 1);
      sx = __ldg(p.job.seeds + 3 * j + 2);
      ok = !(sz - g.mz < 0 || sy - g.my < 0 || sx - g.mx < 0 || sz + g.mz >= cv.sz || sy + g.my >= cv.sy || sx + g.mx >= cv.sx);
      if (ok) {
        const size_t i = cv_index(cv, sz, sy, sx);
        ok = __ldcg(cv.seg + i) <= 0 && !(cv.mask && __ldg(cv.mask + i)) && !(cv.seed_mask && __ldg(cv.seed_mask + i));
        const int* mbd = cv.opt.min_boundary_dist_zyx;
        for (int zz = max(sz - mbd[0], 0); zz < min(sz + mbd[0] + 1, cv.sz); ++zz)
          for (int yy = max(sy - mbd[1], 0); yy < min(sy + mbd[1] + 1, cv.sy); ++yy)
            for (int xx = max(sx - mbd[2], 0); xx < min(sx + mbd[2] + 1, cv.sx); ++xx)
              if (__ldcg(cv.seg + cv_index(cv, zz, yy, xx)) > 0) ok = false;
        // keep clear of the objects being grown: inside (their touched box + half a FoV) the run would most likely be wasted
        for (int q = 0; q < p.nchains; ++q) {
          const CanvasState* o = chain_state(c, q);
          if (q == k || o->phase == PH_FREE) continue;
          // (measured on the 250^3 bench canvas: half a FoV of clearance beats a whole one for 3, 4 and 5 chains — fewer
          // chain-rounds spent waiting; scheduler experiments: FFN_B200_DEBUG bit 256 = a whole FoV, bit 512 = two)
          const int ms = (p.job.debug & 256) ? 2 : ((p.job.debug & 512) ? 4 : 1);
          const int ez = g.fz * ms / 2, ey = g.fy * ms / 2, ex = g.fx * ms / 2;
          const bool has_box = o->dirty_hi[0] > o->dirty_lo[0];
          const int lo0 = (has_box ? min(o->dirty_lo[0], o->start[0]) : o->start[0]) - ez,
                    hi0 = (has_box ? max(o->dirty_hi[0], o->start[0] + 1) : o->start[0] + 1) + ez;
          const int lo1 = (has_box ? min(o->dirty_lo[1], o->start[1]) : o->start[1]) - ey,
                    hi1 = (has_box ? max(o->dirty_hi[1], o->start[1] + 1) : o->start[1] + 1) + ey;
          const int lo2 = (has_box ? min(o->dirty_lo[2], o->start[2]) : o->start[2]) - ex,
                    hi2 = (has_box ? max(o->dirty_hi[2], o->start[2] + 1) : o->start[2] + 1) + ex;
          if (sz >= lo0 && sz < hi0 && sy >= lo1 && sy < hi1 && sx >= lo2 && sx < hi2) ok = false;
        }
        // ... and of the finished objects that wait for their turn (parked) or were suspended: one that comes EARLIER in
        // the seed order writes its labels before this seed's turn, and a seed inside it is then rejected by the
        // in-order gating (inference.py:562-568) — its run would be thrown away.  The object's own seed array says
        // which voxels it will label (>= segment_threshold, inference.py:635; NaN compares false).
        if (!(p.job.debug & 32))
          for (int b = 0; ok && b < p.nchains * kBufsPerChain; ++b)
            if ((sc->bkind[b] == 1 || sc->bkind[b] == 2) && sc->bseed[b] >= 0 && sc->bseed[b] < j &&
                __ldcg(p.ob[b].seed + i) >= cv.opt.segment_threshold)
              ok = false;
      }
    }
    const unsigned m = __ballot_sync(full, ok);
    if (m) {
      const int f = __ffs(m) - 1;
      const long long j0 = base + w + f;
      sz = __shfl_sync(full, sz, f);
      sy = __shfl_sync(full, sy, f);
      sx = __shfl_sync(full, sx, f);
      if (c.lane == 0) {
        p.job.seed_status[j0] = 1;
        sc->spec_runs++;
        start_object(st, sc, j0, 1, sz, sy, sx);
      }
      __syncwarp();
      return;
    }
    if (base + w + 32 >= p.job.n_seeds) break;
  }
}

// A chain turns to another of its object buffers (warp-collective): the object it leaves is written back to its
// buffer's state block (empty, parked = finished and waiting for its turn, or suspended = a run that goes on
// later) and the target buffer's state is loaded.  A suspended run must not go on before the round after: its
// last paste lands during this one.
__device__ __forceinline__ void swap_buffers(const Ctx& c, LChain& L, Sched* sc, int nb) {
  const KParams& p = *c.p;
  CanvasState* st = L.st;
  constexpr int kStateWords = (int)(sizeof(CanvasState) / 8);
  const int kind = st->phase == PH_FREE ? 0 : (st->phase == PH_FINISHED ? 1 : 2);
  const long long left_seed = st->seed_index;
  if (c.lane == 0 && kind == 2) st->have_cur = 0;
  __syncwarp();
  for (int w = c.lane; w < kStateWords; w += 32)
    reinterpret_cast<unsigned long long*>(p.ob[L.b].st)[w] = reinterpret_cast<const unsigned long long*>(st)[w];
  __syncwarp();
  for (int w = c.lane; w < kStateWords; w += 32)
    reinterpret_cast<unsigned long long*>(st)[w] = __ldcg(reinterpret_cast<const unsigned long long*>(p.ob[nb].st) + w);
  if (c.lane == 0) {
    sc->bkind[L.b] = kind;
    sc->bseed[L.b] = kind ? left_seed : -1;
    sc->bround[L.b] = (int)sc->round;
    sc->bkind[nb] = 3;
    sc->active[L.k] = nb;
  }
  L.b = nb;
  __syncwarp();
}

// Buffers of chain k other than the active one: a parked object whose turn has come (sets the owner) / an empty
// buffer / a suspended run that may go on (suspended before this round).  -1: none.  Uniform over the warp.
__device__ __forceinline__ int find_turn_buf(const Sched* sc, int k) {
  for (int b = k * kBufsPerChain; b < (k + 1) * kBufsPerChain; ++b)
    if (sc->bkind[b] == 1 && (sc->owner == b || (sc->owner < 0 && sc->bseed[b] == sc->commit_idx))) return b;
  return -1;
}
__device__ __forceinline__ int find_empty_buf(const Sched* sc, int k) {
  for (int b = k * kBufsPerChain; b < (k + 1) * kBufsPerChain; ++b)
    if (sc->bkind[b] == 0) return b;
  return -1;
}
__device__ __forceinline__ int find_suspended_buf(const Sched* sc, int k, bool& too_early) {
  too_early = false;
  for (int b = k * kBufsPerChain; b < (k + 1) * kBufsPerChain; ++b)
    if (sc->bkind[b] == 2) {
      if ((int)sc->round > sc->bround[b]) return b;
      too_early = true;
    }
  return -1;
}

// One chain's state machine up to its next collective action (the leader warp; serial transitions on
// lane 0, queue pops / gating / scans as warp collectives).  Returns the action of this round.
__device__ __forceinline__ int chain_advance(const Ctx& c, LChain L, Sched* sc, bool pause) {
  const KParams& p = *c.p;
  const Geom& g = p.g;
  const CanvasDev& cv = p.cv;
  CanvasState* st = L.st;
  const unsigned full = 0xffffffffu;
  for (int guard = 0; guard < (1 << 20); ++guard) {
    const int phase = st->phase;
    __syncwarp();   // every lane has read the state of this iteration before lane 0 changes it
    // ------------------------------------------------------------- terminal / idle phases
    if (phase == PH_IDLE || phase == PH_SEGMENT_DONE || phase == PH_ALL_DONE) return ACT_EXIT;
    if (pause) {
      // step budget reached: stop at this round boundary; everything needed to go on is in the state
      if (c.lane == 0) st->have_cur = 0;   // by the next launch every paste has landed in the canvas
      __syncwarp();
      return ACT_EXIT;
    }
    // A finished object parked in one of this chain's buffers is at the head of the line: the chain turns to it
    // now (whatever it is growing is suspended and goes on after the commit).
    if (st->seg_all && (phase == PH_FREE || phase == PH_POP || phase == PH_AFTER_CLEAR || phase == PH_FINISHED)) {
      const int tb = find_turn_buf(sc, L.k);
      if (tb >= 0) {
        if (c.lane == 0) sc->owner = tb;
        __syncwarp();
        swap_buffers(c, L, sc, tb);
        continue;
      }
    }
    if (phase == PH_FORCE_STEP) {          // Canvas.update_at driven from the host: one step at st->cur
      if (c.lane == 0) {
        st->have_cur = 1;
        for (int q = 0; q < 3; ++q) {
          const int m = q == 0 ? g.mz : q == 1 ? g.my : g.mx;
          st->dirty_lo[q] = min(st->dirty_lo[q], st->cur[q] - m);
          st->dirty_hi[q] = max(st->dirty_hi[q], st->cur[q] + m + 1);
        }
        st->phase = PH_AFTER_STEP;
      }
      __syncwarp();
      return ACT_STEP;
    }
    if (phase == PH_AFTER_STEP) {          // only reached in MODE_UPDATE_AT (after_step handles the others)
      if (c.lane == 0) {
        st->ctr.inference_calls++;
        st->have_cur = 0;
        st->phase = PH_SEGMENT_DONE;
      }
      __syncwarp();
      return ACT_EXIT;
    }
    if (phase == PH_START_SEGMENT) {
      if (c.lane == 0) {
        trace_event(p, st, EV_SEED_START, st->start[0], st->start[1], st->start[2]);
        st->ctr.segment_at_calls++;
        st->seg_t0 = sm100::globaltimer_ns();
        st->phase = PH_AFTER_CLEAR;
        st->popped = 0;
      }
      __syncwarp();
      if (st->reset_seed) {
        // an object started ahead of its turn may be discarded: if this chain's seed array still holds the last
        // in-turn object (what Canvas.seed shows after segment_all), move that box to the snapshot array instead
        // of just clearing it
        int act = ACT_CLEAR;
        if (st->seg_all && st->spec && sc->last_chain == L.b && !sc->last_in_snap && p.snap && !(p.job.debug & 8)) {
          act = ACT_CLEAR_MOVE;
          if (c.lane == 0) {
            for (int q = 0; q < 3; ++q) {
              sc->snap_old_lo[q] = sc->snap_lo[q];
              sc->snap_old_hi[q] = sc->snap_hi[q];
              sc->snap_lo[q] = max(st->dirty_lo[q], 0);
              sc->snap_hi[q] = min(st->dirty_hi[q], q == 0 ? cv.sz : q == 1 ? cv.sy : cv.sx);
            }
            sc->last_in_snap = 1;
          }
          __syncwarp();
        }
        return act;
      }
      continue;
    }
    if (phase == PH_AFTER_CLEAR) {
      // init_seed (inference.py:443-450) + reset_state (:291-310) + first queue item (:492-496)
      if (c.lane == 0) {
        if (st->reset_seed) {   // Canvas.reset_seed_per_segment (inference.py:486-490): seed and extents start over
          p.ob[L.b].seed[cv_index(cv, st->start[0], st->start[1], st->start[2])] = cv.opt.init_activation;
          for (int q = 0; q < 3; ++q) {
            st->dirty_lo[q] = st->start[q];
            st->dirty_hi[q] = st->start[q] + 1;
            st->min_pos[q] = st->max_pos[q] = st->start[q];
          }
        }
        st->epoch++;
        st->q_head = st->q_tail = 0;
        st->iters = 0;
        st->n_unstepped = 0;
        st->have_cur = 0;
        st->weak = 0;
        push_move(p, L, (float)(cv.opt.policy_score_threshold * 2.0), st->start[0], st->start[1], st->start[2]);
        st->phase = PH_POP;
        st->popped = 0;
      }
      __syncwarp();
      // the init_seed store above is read back (through L2) by the pop below
      __threadfence();
      continue;
    }
    if (phase == PH_POP) {
      if (!st->popped) chain_pop(c, L);
      const bool run = st->pop_run != 0;
      __syncwarp();
      if (run) {
        if (c.lane == 0) {
          st->popped = 0;
          for (int q = 0; q < 3; ++q) st->cur[q] = st->pop_pos[q];
          st->have_cur = 1;
          trace_event(p, st, EV_STEP, st->cur[0], st->cur[1], st->cur[2]);
          for (int q = 0; q < 3; ++q) {
            const int m = q == 0 ? g.mz : q == 1 ? g.my : g.mx;
            st->dirty_lo[q] = min(st->dirty_lo[q], st->cur[q] - m);
            st->dirty_hi[q] = max(st->dirty_hi[q], st->cur[q] + m + 1);
          }
          st->phase = PH_AFTER_STEP;
        }
        __syncwarp();
        return ACT_STEP;
      }
      // object finished
      if (c.lane == 0) {
        st->popped = 0;
        if (!st->seg_all) {
          st->phase = PH_SEGMENT_DONE;
        } else {
          st->phase = PH_FINISHED;
          st->fin_round = (int)sc->round;
        }
      }
      __syncwarp();
      if (!st->seg_all) return ACT_EXIT;
      continue;
    }
    if (phase == PH_FINISHED) {
      // The last step's paste lands during the round the object finished in; and labels are committed in
      // seed order, so an object that ran ahead waits until it is at the head of the line.
      if (st->have_cur && st->fin_round == (int)sc->round) {
        // nothing can be decided about this object before the next round; if it is not at the head of the line
        // the chain need not wait with it: park it at once and go on in another buffer
        const bool at_head = sc->owner == L.b || (sc->owner < 0 && st->seed_index >= 0 && st->seed_index == sc->commit_idx);
        if (!at_head) {
          bool too_early;
          int nb = find_suspended_buf(sc, L.k, too_early);
          if (nb < 0 && !too_early) nb = find_empty_buf(sc, L.k);
          if (nb >= 0) {
            swap_buffers(c, L, sc, nb);
            continue;
          }
        }
        return ACT_IDLE;
      }
      __syncwarp();
      if (c.lane == 0) st->have_cur = 0;
      __syncwarp();
      if (sc->owner != L.b) {
        if (sc->owner < 0 && st->seed_index >= 0 && st->seed_index == sc->commit_idx) {
          if (c.lane == 0) sc->owner = L.b;
          __syncwarp();
        } else {
          // not its turn yet: park it and use the chain for another buffer (the suspended run, or a new object)
          bool too_early;
          int nb = find_suspended_buf(sc, L.k, too_early);
          if (nb < 0 && !too_early) nb = find_empty_buf(sc, L.k);
          if (nb < 0) return ACT_IDLE;
          swap_buffers(c, L, sc, nb);
          continue;
        }
      }
      if (st->spec) {
        int sz, sy, sx;
        const int ok = gate_seed(c, sc, st->seed_index, true, sz, sy, sx);   // the reference's gating, now, in order
        const bool conflict = ok && (run_conflicts(c, L.b, st) || (p.job.debug & 1) ||
                                     ((p.job.debug & 4) && sc->max_id != st->start_max_id));
        if (!ok || conflict) {
          if (c.lane == 0) {
            sc->spec_discarded++;
            sc->spec_steps_discarded += st->ctr.inference_calls;
            FfnCounters zero{};
            st->ctr = zero;
            if (!ok) {
              finalize_seed(sc, st);                                  // rejected before it would have started
            } else {
              start_object(st, sc, st->seed_index, 0, sz, sy, sx);    // redo it in turn
            }
          }
          __syncwarp();
          continue;
        }
        if (c.lane == 0) st->spec = 0;
        __syncwarp();
      }
      // from here on this is the reference's code after segment_at returned (inference.py:593-620)
      if (c.lane == 0) {
        sc->ctr.inference_calls += st->ctr.inference_calls;
        sc->ctr.segment_at_calls += st->ctr.segment_at_calls;
        sc->ctr.skip_threshold += st->ctr.skip_threshold;
        sc->ctr.skip_invalid_pos += st->ctr.skip_invalid_pos;
        sc->ctr.skip_restricted_pos += st->ctr.skip_restricted_pos;
        sc->ctr.seed_got_too_weak += st->ctr.seed_got_too_weak;
        FfnCounters zero{};
        st->ctr = zero;
        if (st->overflow) sc->overflow |= st->overflow;
        sc->last_chain = L.b;        // Canvas.seed now shows this object (buffer index)
        sc->last_in_snap = 0;
      }
      __syncwarp();
      const size_t si = cv_index(cv, st->start[0], st->start[1], st->start[2]);
      if (st->iters <= 0) {
        if (c.lane == 0) {
          sc->ctr.invalid_other++;
          finalize_seed(sc, st);
        }
        __syncwarp();
        continue;
      }
      if (__ldcg(p.ob[L.b].seed + si) < cv.opt.move_threshold) {
        if (c.lane == 0) {
          if (__ldcg(cv.seg + si) == 0) cv.seg[si] = -1;
          sc->ctr.invalid_weak++;
          finalize_seed(sc, st);
        }
        __syncwarp();
        continue;
      }
      if (c.lane == 0) {
        const int half[3] = {g.fz / 2, g.fy / 2, g.fx / 2};
        const int shp[3] = {cv.sz, cv.sy, cv.sx};
        for (int q = 0; q < 3; ++q) {
          st->box_lo[q] = max(st->min_pos[q] - half[q], 0);
          st->box_hi[q] = min(st->max_pos[q] + half[q] + 1, shp[q]);
        }
        st->cnt_raw = st->cnt_actual = 0ull;
        st->n_touched = 0;
        st->phase = PH_AFTER_COUNT;
      }
      __syncwarp();
      return ACT_COUNT;
    }
    if (phase == PH_AFTER_COUNT) {
      int ret = -1;
      if (c.lane == 0) {
        const size_t si = cv_index(cv, st->start[0], st->start[1], st->start[2]);
        const long long raw = (long long)st->cnt_raw, actual = (long long)st->cnt_actual;
        if (actual < (long long)cv.opt.min_segment_size) {   // inference.py:639-646
          if (__ldcg(cv.seg + si) == 0) cv.seg[si] = -1;
          sc->ctr.invalid_small++;
          for (int i = 0; i < st->n_touched; ++i) p.job.ovl_count[p.job.ovl_touched[i]] = 0;
          st->n_touched = 0;
          finalize_seed(sc, st);
        } else {
          sc->ctr.voxels_segmented += actual;
          sc->ctr.voxels_overlapping += raw - actual;
          sc->max_id++;
          st->cur_sid = sc->max_id;
          sc->ctr.max_id = sc->max_id;
          sc->ctr.segments++;
          for (int i = 0; i < st->n_touched; ++i) {       // Canvas.overlaps (inference.py:668)
            const int id = p.job.ovl_touched[i];
            if (sc->n_overlaps < p.job.overlaps_cap) {
              FfnOverlap o;
              o.id = st->cur_sid;
              o.other_id = id;
              o.count = p.job.ovl_count[id];
              p.job.overlaps[sc->n_overlaps] = o;
            } else {
              sc->overflow |= 2;
            }
            sc->n_overlaps++;
            p.job.ovl_count[id] = 0;
          }
          st->n_touched = 0;
          if (sc->n_origins < p.job.origins_cap) {        // Canvas.origins (inference.py:671)
            FfnOrigin o;
            o.id = st->cur_sid;
            o.start_zyx[0] = st->start[0];
            o.start_zyx[1] = st->start[1];
            o.start_zyx[2] = st->start[2];
            o.iters = st->iters;
            o.walltime_sec = (double)(sm100::globaltimer_ns() - st->seg_t0) * 1e-9;
            if (p.job.debug & 16) o.walltime_sec = L.k * 1e5 + st->start_max_id;   // experiments
            p.job.origins[sc->n_origins] = o;
          } else {
            sc->overflow |= 4;
          }
          sc->n_origins++;
          st->phase = PH_AFTER_WRITE;
          ret = ACT_WRITE;
        }
      }
      ret = __shfl_sync(full, ret, 0);
      if (ret >= 0) return ret;
      continue;
    }
    if (phase == PH_AFTER_WRITE) {
      if (c.lane == 0) finalize_seed(sc, st);
      __syncwarp();
      continue;
    }
    if (phase == PH_FREE) {
      advance_pointer(c, L, sc);                     // the head of the line first: an object whose turn it is runs here
      if (st->phase != PH_FREE) continue;
      {                                              // then a run this chain suspended
        bool too_early;
        const int nb = find_suspended_buf(sc, L.k, too_early);
        if (nb >= 0) {
          swap_buffers(c, L, sc, nb);
          continue;
        }
        if (too_early) return ACT_IDLE;
      }
      lookahead(c, L, sc);                           // then an object ahead of its turn
      if (st->phase == PH_FREE) return ACT_IDLE;     // nothing to start right now
      continue;
    }
    return ACT_EXIT;   // unknown phase
  }
  return ACT_EXIT;
}

// The round boundary on CTA 0 (all threads): policy + pops of the chains that just stepped in parallel
// (faces spread over all warps, then one warp per chain), then the scheduler transitions of every chain,
// serially and in chain order on warp 0 (deterministic), then the actions of the new round are published.
// `stepped`: chains that ran a FoV step in the round just finished (staged with parity round-1).
__device__ __forceinline__ void leader_round(Ctx& c, unsigned stepped) {
  const KParams& p = *c.p;
  const int K = p.nchains;
  Sched* sc = c.s_sched;
  constexpr int kStateWords = (int)(sizeof(CanvasState) / 8);
  constexpr int kSchedWords = (int)(sizeof(Sched) / 8);
  static_assert(sizeof(CanvasState) <= kStateSlot && sizeof(CanvasState) % 8 == 0, "state copy area");
  static_assert(sizeof(Sched) % 8 == 0 && kMaxChains * kStateSlot + sizeof(Sched) <= kXchgBytes,
                "the leader's working copies alias the epilogue exchange area");
  const unsigned par = (c.round & 1u) ^ 1u;   // parity the finished round was staged with
  const long long t_all = prof_now(c);
  // Watchdog: one launch covers at most 2^15 FoV steps (a few seconds).  A launch that is still going after
  // 60 s (FFN_B200_WATCHDOG_S; sanitizer runs need more) has stalled; raise the abort flag so that every CTA leaves
  // at this round boundary and the host reports it.
  if (c.tid == 0 && sm100::globaltimer_ns() - c.t_start > (unsigned long long)p.job.watchdog_ns) atomicExch(p.ws.abort_flag, 5);
  // Work on shared-memory copies: the serial code is full of read-after-write on these fields, and in
  // global memory every one of those is an L2 round trip.
  for (int i = c.tid; i < K * kStateWords; i += 256) {
    if (c.tid >= 256) break;
    const int k = i / kStateWords, w = i - k * kStateWords;
    const int b = __ldcg(&p.sched->active[k]);   // the object buffer chain k works on
    reinterpret_cast<unsigned long long*>(chain_state(c, k))[w] =
        __ldcg(reinterpret_cast<const unsigned long long*>(p.ob[b].st) + w);
  }
  if (c.tid >= 256)
    for (int i = c.tid - 256; i < kSchedWords; i += kThreads - 256)
      reinterpret_cast<unsigned long long*>(sc)[i] = __ldcg(reinterpret_cast<const unsigned long long*>(p.sched) + i);
  if (c.tid >= kThreads - kMaxChains) {
    const int k = c.tid - (kThreads - kMaxChains);
    if (k < K) c.s_misc[kMiscDisco + k] = (((stepped >> k) & 1u) && disco_active(p, k, par)) ? 1 : 0;
  }
  __syncthreads();
  // ---- phase A.1: the six faces of every chain that stepped, one warp per (chain, face)
  const long long t_pol = prof_now(c);
  if (p.job.mode != MODE_UPDATE_AT) {
    for (int t = c.warp; t < K * 6; t += kThreads / 32) {
      const int k = t / 6, f = t - 6 * k;
      if (!((stepped >> k) & 1u)) continue;
      LChain L{k, sc->active[k], chain_state(c, k), par, c.s_misc[kMiscDisco + k] != 0};
      face_argmax(c, L, f);
    }
  }
  __syncthreads();
  // ---- phase A.2: one warp per chain: queue pushes, bookkeeping, the pop that decides the next step
  if (c.warp < K && ((stepped >> c.warp) & 1u)) {
    LChain L{c.warp, sc->active[c.warp], chain_state(c, c.warp), par, c.s_misc[kMiscDisco + c.warp] != 0};
    if (L.st->phase == PH_AFTER_STEP) after_step(c, L);
  }
  if (c.tid == 0) prof_add(c, 12, prof_now(c) - t_pol);
  __syncthreads();
  // ---- phase B: warp 0, chains in order
  if (c.warp == 0) {
    if (c.lane == 0) {
      sc->steps_executed += __popc(stepped);
    }
    __syncwarp();
    bool pause = false;
    if (p.job.step_budget > 0 && p.job.mode == MODE_SEGMENT) {
      const CanvasState* s0 = chain_state(c, 0);
      pause = s0->seg_all ? sc->steps_executed >= p.job.step_budget : s0->ctr.inference_calls >= p.job.step_budget;
    }
    int acts[kMaxChains];
    bool any = false;
#pragma unroll
    for (int k = 0; k < kMaxChains; ++k) {
      acts[k] = ACT_EXIT;
      if (k < K) {
        LChain L{k, sc->active[k], chain_state(c, k), par, ((stepped >> k) & 1u) && c.s_misc[kMiscDisco + k] != 0};
        acts[k] = chain_advance(c, L, sc, pause);
        if (acts[k] != ACT_EXIT && acts[k] != ACT_IDLE) any = true;
        if (acts[k] == ACT_IDLE && c.lane == 0) {
          if (L.st->phase == PH_FREE) sc->idle_free++;
          else sc->idle_wait++;
        }
      }
    }
    // segment_all: done when the line is empty and no chain holds an object; otherwise idle chains keep the
    // kernel going as long as somebody works (an all-idle round cannot happen: the head of the line is
    // always runnable by a free chain)
    const CanvasState* s0 = chain_state(c, 0);
    if (p.job.mode == MODE_SEGMENT && s0->seg_all && !pause) {
      bool all_free = true;
      for (int k = 0; k < K; ++k) all_free = all_free && chain_state(c, k)->phase == PH_FREE;
      for (int b = 0; b < K * kBufsPerChain; ++b) all_free = all_free && sc->bkind[b] != 1 && sc->bkind[b] != 2;
      __syncwarp();   // every lane has read the phases before lane 0 changes them
      if (all_free && sc->commit_idx >= p.job.n_seeds && sc->owner < 0) {
        if (c.lane == 0) {
          sc->all_done = 1;
          for (int k = 0; k < K; ++k) chain_state(c, k)->phase = PH_ALL_DONE;
        }
        any = false;
      } else if (!any) {
        // nobody has a collective action: keep going only if someone is waiting for a paste to land — for
        // one round; a second one means the scheduler has stalled (reported by the host, never spun on)
        bool waiting = false;
        for (int k = 0; k < K; ++k)
          waiting = waiting || (chain_state(c, k)->phase == PH_FINISHED && chain_state(c, k)->fin_round + 1 >= (int)sc->round);
        for (int b = 0; b < K * kBufsPerChain; ++b)   // an object parked / a run suspended this round goes on next round
          waiting = waiting || ((sc->bkind[b] == 1 || sc->bkind[b] == 2) && sc->bround[b] + 1 >= (int)sc->round);
        // the head of the line was handed to an object of a chain that had already been looked at this round
        // (chains are processed in order): it acts next round
        any = waiting || sc->owner >= 0;
      }
    }
    // watchdog: a launch that runs far more rounds than its step budget and seed count allow is reported, not spun on
    if (p.job.mode == MODE_SEGMENT && s0->seg_all && c.round > (unsigned)p.job.round_cap) {
      if (c.lane == 0) sc->overflow |= 16;
      any = false;
    }
    if (c.lane == 0) {
      sc->round++;
#pragma unroll
      for (int k = 0; k < kMaxChains; ++k) {
        int a = acts[k];
        if (!any) a = ACT_EXIT;
        else if (a == ACT_EXIT && k < K) a = ACT_IDLE;   // a paused / finished chain idles while others go on
        p.ctl->action[k] = k < K ? a : ACT_EXIT;
        if (k < K) {
          const CanvasState* s = chain_state(c, k);
          p.ctl->pos[k][0] = s->cur[0];
          p.ctl->pos[k][1] = s->cur[1];
          p.ctl->pos[k][2] = s->cur[2];
          p.ctl->buf[k] = sc->active[k];
        }
      }
    }
    __syncwarp();
  }
  __syncthreads();
  for (int i = c.tid; i < K * kStateWords; i += 256) {
    if (c.tid >= 256) break;
    const int k = i / kStateWords, w = i - k * kStateWords;
    reinterpret_cast<unsigned long long*>(p.ob[sc->active[k]].st)[w] = reinterpret_cast<const unsigned long long*>(chain_state(c, k))[w];
  }
  if (c.tid >= 256)
    for (int i = c.tid - 256; i < kSchedWords; i += kThreads - 256)
      reinterpret_cast<unsigned long long*>(p.sched)[i] = reinterpret_cast<const unsigned long long*>(sc)[i];
  __syncthreads();
  // everything above (ordered by bar.sync) becomes visible before the round is announced
  if (c.tid == 0) {
    sm100::red_release_add(p.round_flag, 1u);
    prof_add(c, 8, prof_now(c) - t_all);
  }
}

// ------------------------------------------------------------------------------------------
// Collective helpers over a canvas box (all CTAs)
// ------------------------------------------------------------------------------------------
// What the leader published this round (boxes, ids) is read through L2, like every other cross-CTA datum.
__device__ __forceinline__ void load3(const int* src, int (&dst)[3]) {
  dst[0] = __ldcg(src);
  dst[1] = __ldcg(src + 1);
  dst[2] = __ldcg(src + 2);
}

__device__ __forceinline__ void clear_dirty(Ctx& c, int b) {   // NumpyArray.clear restricted to the touched box
  const KParams& p = *c.p;
  const CanvasState* st = p.ob[b].st;
  int dlo[3], dhi[3];
  load3(st->dirty_lo, dlo);
  load3(st->dirty_hi, dhi);
  const int lo[3] = {max(dlo[0], 0), max(dlo[1], 0), max(dlo[2], 0)};
  const int hi[3] = {min(dhi[0], p.cv.sz), min(dhi[1], p.cv.sy), min(dhi[2], p.cv.sx)};
  const int nz = hi[0] - lo[0], ny = hi[1] - lo[1], nx = hi[2] - lo[2];
  if (nz <= 0 || ny <= 0 || nx <= 0) return;
  const long long lines = (long long)nz * ny;
  const float nanv = CUDART_NAN_F;
  for (long long l = (long long)c.cta * (kThreads / 32) + c.warp; l < lines; l += (long long)c.G * (kThreads / 32)) {
    const int z = lo[0] + (int)(l / ny), y = lo[1] + (int)(l % ny);
    float* row = p.ob[b].seed + cv_index(p.cv, z, y, lo[2]);
    for (int x = c.lane; x < nx; x += 32) row[x] = nanv;
  }
}

// Moves chain k's touched box into the snapshot array (and clears it), after clearing what the snapshot held
// before.  The two passes write disjoint voxels of the snapshot array, so no barrier is needed between them.
__device__ __forceinline__ void clear_move(Ctx& c, int b) {
  const KParams& p = *c.p;
  const Sched* sc = p.sched;
  const CanvasState* st = p.ob[b].st;
  int olo[3], ohi[3], dlo[3], dhi[3];
  load3(sc->snap_old_lo, olo);
  load3(sc->snap_old_hi, ohi);
  // the box to move is the chain's touched box, read exactly like clear_dirty does (the leader recorded the same
  // numbers as the new snapshot box for the host)
  load3(st->dirty_lo, dlo);
  load3(st->dirty_hi, dhi);
  const int lo[3] = {max(dlo[0], 0), max(dlo[1], 0), max(dlo[2], 0)};
  const int hi[3] = {min(dhi[0], p.cv.sz), min(dhi[1], p.cv.sy), min(dhi[2], p.cv.sx)};
  const float nanv = CUDART_NAN_F;
  {
    const int nz = ohi[0] - olo[0], ny = ohi[1] - olo[1], nx = ohi[2] - olo[2];
    if (nz > 0 && ny > 0 && nx > 0) {
      const long long lines = (long long)nz * ny;
      for (long long l = (long long)c.cta * (kThreads / 32) + c.warp; l < lines; l += (long long)c.G * (kThreads / 32)) {
        const int z = olo[0] + (int)(l / ny), y = olo[1] + (int)(l % ny);
        const bool in_new_zy = z >= lo[0] && z < hi[0] && y >= lo[1] && y < hi[1];
        float* row = p.snap + cv_index(p.cv, z, y, olo[2]);
        for (int x = c.lane; x < nx; x += 32)
          if (!(in_new_zy && olo[2] + x >= lo[2] && olo[2] + x < hi[2])) row[x] = nanv;
      }
    }
  }
  {
    const int nz = hi[0] - lo[0], ny = hi[1] - lo[1], nx = hi[2] - lo[2];
    if (nz > 0 && ny > 0 && nx > 0) {
      const long long lines = (long long)nz * ny;
      for (long long l = (long long)c.cta * (kThreads / 32) + c.warp; l < lines; l += (long long)c.G * (kThreads / 32)) {
        const int z = lo[0] + (int)(l / ny), y = lo[1] + (int)(l % ny);
        const size_t base = cv_index(p.cv, z, y, lo[2]);
        for (int x = c.lane; x < nx; x += 32) {
          p.snap[base + x] = __ldcg(p.ob[b].seed + base + x);
          p.ob[b].seed[base + x] = nanv;
        }
      }
    }
  }
}

__device__ __forceinline__ void commit_count(Ctx& c, int b) {   // inference.py:624-636
  const KParams& p = *c.p;
  CanvasState* st = p.ob[b].st;
  int lo[3], hi[3];
  load3(st->box_lo, lo);
  load3(st->box_hi, hi);
  const int nz = hi[0] - lo[0], ny = hi[1] - lo[1], nx = hi[2] - lo[2];
  const long long lines = (long long)nz * ny;
  unsigned raw = 0, actual = 0;
  for (long long l = (long long)c.cta * (kThreads / 32) + c.warp; l < lines; l += (long long)c.G * (kThreads / 32)) {
    const int z = lo[0] + (int)(l / ny), y = lo[1] + (int)(l % ny);
    const size_t base = cv_index(p.cv, z, y, lo[2]);
    for (int x = c.lane; x < nx; x += 32) {
      const float s = __ldcg(p.ob[b].seed + base + x);
      if (!(s >= p.cv.opt.segment_threshold)) continue;
      ++raw;
      const int sg = __ldcg(p.cv.seg + base + x);
      if (sg > 0) {
        if (sg < p.job.ovl_ids) {
          if (atomicAdd(p.job.ovl_count + sg, 1) == 0) {
            const int t = atomicAdd(&st->n_touched, 1);
            if (t < p.job.ovl_ids) p.job.ovl_touched[t] = sg;
          }
        }
      } else {
        ++actual;
      }
    }
  }
  raw = __reduce_add_sync(0xffffffffu, raw);
  actual = __reduce_add_sync(0xffffffffu, actual);
  if (c.lane == 0 && raw) {
    atomicAdd(&st->cnt_raw, (unsigned long long)raw);
    atomicAdd(&st->cnt_actual, (unsigned long long)actual);
  }
}

__device__ __forceinline__ void commit_write(Ctx& c, int b) {   // inference.py:653-658
  const KParams& p = *c.p;
  const CanvasState* st = p.ob[b].st;
  int lo[3], hi[3];
  load3(st->box_lo, lo);
  load3(st->box_hi, hi);
  const int nz = hi[0] - lo[0], ny = hi[1] - lo[1], nx = hi[2] - lo[2];
  const long long lines = (long long)nz * ny;
  const int sid = __ldcg(&st->cur_sid);
  for (long long l = (long long)c.cta * (kThreads / 32) + c.warp; l < lines; l += (long long)c.G * (kThreads / 32)) {
    const int z = lo[0] + (int)(l / ny), y = lo[1] + (int)(l % ny);
    const size_t base = cv_index(p.cv, z, y, lo[2]);
    for (int x = c.lane; x < nx; x += 32) {
      const float s = __ldcg(p.ob[b].seed + base + x);
      if (!(s >= p.cv.opt.segment_threshold)) continue;
      if (__ldcg(p.cv.seg + base + x) > 0) continue;
      p.cv.seg[base + x] = sid;
      if (p.cv.qprob) p.cv.qprob[base + x] = quantize_prob(s);
    }
  }
}

// ------------------------------------------------------------------------------------------
// The kernel
// ------------------------------------------------------------------------------------------
// One round = one FoV step of every chain in `mask` (staged by the caller with the current parity).
__device__ __forceinline__ void run_layers(Ctx& c, unsigned mask) {
  const KParams& p = *c.p;
  if (p.compute_mode == FFN_COMPUTE_FP16_TC) {
    // the staged operands: every thread's stores, then one arrival per chain (event 1 of the round)
    sm100::tc_fence_before();
    __syncthreads();
    if (c.tid == 0) {
#pragma unroll
      for (int k = 0; k < kMaxChains; ++k)
        if ((mask >> k) & 1u) sm100::red_release_add(p.ch[k].bar, 1u);
    }
    sm100::tc_fence_after();
    layers_pipelined(c, mask);
  } else {
    layers_blocking(c);
  }
}

__global__ void __launch_bounds__(kThreads, 1) ffn_flood_kernel(const __grid_constant__ KParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  Ctx c;
  c.p = &p;
  c.tid = threadIdx.x;
  // warp-uniform BY CONSTRUCTION (a shuffle from lane 0): role branches on it are uniform branches
  c.warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  c.lane = threadIdx.x & 31;
  c.cta = blockIdx.x;
  c.G = gridDim.x;
  c.t_begin = (int)(((long long)c.cta * p.g.nt) / c.G);
  c.t_end = (int)(((long long)(c.cta + 1) * p.g.nt) / c.G);
  c.bar_target = 0;
  c.ev0 = c.ev1 = c.ev2 = c.ev3 = c.ev4 = 0;
  c.round = 0;
  c.t_start = sm100::globaltimer_ns();
  c.smem = smem_raw;
  const SmemLayout L = smem_layout(p.g);
  c.s_bias = reinterpret_cast<float*>(smem_raw + L.bias);
  c.mb_w = reinterpret_cast<uint64_t*>(smem_raw + L.bars);
  c.mb_full = c.mb_w + 2;
  c.mb_empty = c.mb_full + kActStages;
  c.mb_tfull = c.mb_empty + kActStages;
  c.mb_tempty = c.mb_tfull + kAccSlots;
  c.mb_sig = c.mb_tempty + kAccSlots;
  c.s_tmem = reinterpret_cast<uint32_t*>(c.mb_sig + kMaxChains);
  c.load_cnt = c.mma_cnt = c.epi_cnt = 0;
  c.s_misc = reinterpret_cast<int*>(smem_raw + L.bars + kOffMisc);
  c.s_round = reinterpret_cast<int*>(smem_raw + L.bars + kOffRound);   // 2 * kMaxChains * 8 ints
  c.s_xchg = reinterpret_cast<float*>(smem_raw + L.bars + kOffXchg);
  c.s_dot = c.s_xchg + 2 * 2 * 4 * 2 * 16;
  // CTA 0's working copies of the chain states and the scheduler block live in the epilogue's exchange area: they are
  // only used inside leader_round, between the grid barrier and the round's first tile
  c.s_state = reinterpret_cast<CanvasState*>(smem_raw + L.bars + kOffXchg);
  c.s_sched = reinterpret_cast<Sched*>(smem_raw + L.bars + kOffXchg + kMaxChains * kStateSlot);
  static_assert((2 + 2 * kActStages + 2 * kAccSlots + kMaxChains) * 8 + 8 <= kOffMisc, "mbarrier area");
  c.prof = nullptr;
  if (FFN_PROFILE && p.ws.prof && (c.cta == 0 || c.cta == c.G - 1)) {
    c.prof = reinterpret_cast<long long*>(smem_raw + L.bars + kOffProf);
    if (c.tid < 16) c.prof[c.tid] = 0;
  }
#if FFN_PROFILE
  c.trace = (p.ws.prof && c.cta == kTraceCta) ? p.ws.prof + 32 : nullptr;
  c.sig_cnt = 0;
#endif
  const long long t_kernel = prof_now(c);
  c.bits = 0;
  c.tmem_base = 0;
  const bool tc = p.compute_mode != FFN_COMPUTE_FP32;
  const int K = p.nchains;

  for (int i = c.tid; i < p.g.nconv * 32; i += kThreads) c.s_bias[i] = p.w.bias[i];
  if (c.tid < 32) c.s_bias[p.g.nconv * 32 + c.tid] = p.w.w_lom[c.tid];
  if (c.tid == 0) c.s_bias[p.g.nconv * 32 + 32] = p.w.b_lom;
  if (c.tid < 2 * kMaxChains * 8) c.s_round[c.tid] = 0;
  if (tc) {
    if (c.tid == 0) {
      sm100::mbar_init(&c.mb_w[0], 1);
      sm100::mbar_init(&c.mb_w[1], 1);
      for (int i = 0; i < kActStages; ++i) {
        sm100::mbar_init(&c.mb_full[i], 1);
        sm100::mbar_init(&c.mb_empty[i], 1);
      }
      for (int i = 0; i < kAccSlots; ++i) {
        sm100::mbar_init(&c.mb_tfull[i], 1);
        sm100::mbar_init(&c.mb_tempty[i], 8);   // one arrival per epilogue warp
      }
      for (int i = 0; i < kMaxChains; ++i) sm100::mbar_init(&c.mb_sig[i], 8);
      sm100::fence_mbar_init();
    }
    __syncwarp();
    if (c.warp == 0) sm100::tmem_alloc<kTmemCols>(c.s_tmem);
    sm100::tc_fence_before();
    __syncthreads();
    sm100::tc_fence_after();
    c.tmem_base = __shfl_sync(0xffffffffu, *c.s_tmem, 0);
    if (p.compute_mode == FFN_COMPUTE_FP16_TC) {   // the split mode loads both weight halves per layer
      if (c.warp == kLoadWarp && c.lane == 0) {
        tc_issue_weight_load(c, 0);
        if (p.use_tmap)
          for (int k = 0; k < p.nchains; ++k)
            for (int i = 0; i < 3; ++i) sm100::tma_prefetch_desc(&p.tmap[k][i]);
      }
      bit_set(c, 8, true);
    }
  }
  __syncthreads();

  if (p.job.mode == MODE_PREDICT) {
    // Batched ExecutorClient.predict (executor.py:266-340): the patches of a batch are independent, so K
    // of them run per round as K chains of the same pipeline.
    for (int b0 = 0; b0 < p.job.batch; b0 += K) {
      unsigned mask = 0;
      for (int k = 0; k < K; ++k)
        if (b0 + k < p.job.batch) {
          stage_fov(c, k, 0, 0, 0, 0, b0 + k);
          mask |= 1u << k;
        }
      run_layers(c, mask);
      grid_barrier(c);
      for (int k = 0; k < K; ++k)
        if ((mask >> k) & 1u) tail_paste(c, k, 0, c.round & 1u, 0, 0, 0, b0 + k, false);
      ++c.round;
      if (c.tid == 0) c.s_misc[kMiscAbort] = sm100::ld_volatile_s32(p.ws.abort_flag);   // one reader: no divergent exit
      __syncthreads();
      if (c.s_misc[kMiscAbort] != 0) break;
    }
  } else {
    unsigned stepped = 0;   // chains that ran a FoV step in the round just finished
    for (;;) {
      // ---- round boundary: everything of the previous round is complete and visible
      grid_barrier(c);
      if (c.cta == 0) leader_round(c, stepped);
      // paste the previous steps (their logits / counts are final; the positions are still in s_round)
      const long long t_paste = prof_now(c);
      const unsigned ppar = (c.round & 1u) ^ 1u;
      for (int k = 0; k < K; ++k) {
        int* prev = c.s_round + 8 * (kMaxChains + k);   // read by the next stage of this chain (two CTA barriers from here)
        if ((stepped >> k) & 1u) {
          const int* cur = c.s_round + 8 * k;
          const bool disco = disco_active(p, k, ppar);
          tail_paste(c, k, cur[4], ppar, cur[1], cur[2], cur[3], 0, disco);
          if (c.tid == 0) {
            prev[0] = 1 | (disco ? 2 : 0);
            prev[1] = cur[1];
            prev[2] = cur[2];
            prev[3] = cur[3];
            prev[4] = cur[4];
          }
        } else if (c.tid == 0) {
          prev[0] = 0;
        }
      }
      if (c.tid == 0) prof_add(c, 7, prof_now(c) - t_paste);
      // ---- the leader's decisions for this round
      if (c.tid == 0) {
        spin_until(c, p.round_flag, c.round + 1u, 4);
        c.s_misc[kMiscAbort] = sm100::ld_volatile_s32(p.ws.abort_flag);   // one reader: the whole CTA must take the same branch
      }
      __syncthreads();
      const int abort_now = c.s_misc[kMiscAbort];
      if (c.tid < K) {
        int* cur = c.s_round + 8 * c.tid;
        cur[0] = sm100::ld_volatile_s32(&p.ctl->action[c.tid]);
        cur[1] = sm100::ld_volatile_s32(&p.ctl->pos[c.tid][0]);
        cur[2] = sm100::ld_volatile_s32(&p.ctl->pos[c.tid][1]);
        cur[3] = sm100::ld_volatile_s32(&p.ctl->pos[c.tid][2]);
        cur[4] = sm100::ld_volatile_s32(&p.ctl->buf[c.tid]);
      }
      __syncthreads();
      if (abort_now != 0) break;
      bool all_exit = true;
      for (int k = 0; k < K; ++k) all_exit = all_exit && c.s_round[8 * k] == ACT_EXIT;
      if (all_exit) break;
      // ---- collectives of this round, then the FoV steps
      long long t0 = prof_now(c);
      unsigned mask = 0;
      for (int k = 0; k < K; ++k) {
        const int* cur = c.s_round + 8 * k;
        const int action = cur[0], b = cur[4];
        if (action == ACT_STEP) {
          stage_fov(c, k, b, cur[1], cur[2], cur[3], 0);
          mask |= 1u << k;
        } else if (action == ACT_CLEAR) {
          clear_dirty(c, b);
        } else if (action == ACT_CLEAR_MOVE) {
          clear_move(c, b);
        } else if (action == ACT_COUNT) {
          commit_count(c, b);
        } else if (action == ACT_WRITE) {
          commit_write(c, b);
        }
      }
      if (c.tid == 0) prof_add(c, 6, prof_now(c) - t0);
      if (mask) {
        run_layers(c, mask);
        if (c.tid == 0) prof_add(c, 9, __popc(mask));
      }
      stepped = mask;
      ++c.round;
    }
  }

  if (c.tid == 0) prof_add(c, 10, prof_now(c) - t_kernel);
  __syncthreads();
  if (c.prof && c.tid < 16) p.ws.prof[(c.cta == 0 ? 0 : 16) + c.tid] += c.prof[c.tid];
  // Teardown: no bulk copy may be in flight into this CTA's shared memory at exit (the fp16 path always
  // has the next round's layer-0 weights in flight; only the UMMA issuer warp knows that barrier's parity).
  if (tc) {
    if (c.warp == kMmaWarp && bit_get(c, 8)) mbar_wait(c, &c.mb_w[0], bit_get(c, 0));
    sm100::tc_fence_before();
    __syncthreads();
    if (c.warp == 0) sm100::tmem_dealloc<kTmemCols>(c.tmem_base);
  }
}

}  // namespace FFN_KNS

#ifndef FFN_MISC_KERNELS_DEFINED
#define FFN_MISC_KERNELS_DEFINED
// Adds `offset` to every label > 0 (multi-GPU merge, SURVEY.md 8e). HBM-bound, grid-stride.
__global__ void relabel_offset_kernel(int* seg, size_t n, int offset) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int v = seg[i];
    if (v > 0) seg[i] = v + offset;
  }
}

// u8 -> normalised float32 (runner.py:383-385), for ffn_canvas_read(FFN_ARRAY_IMAGE).
__global__ void normalize_u8_kernel(const uint8_t* src, float* dst, size_t n, float mean, float stddev) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = __fdiv_rn(__fsub_rn((float)src[i], mean), stddev);
}

__global__ void fill_f32_kernel(float* dst, size_t n, float v) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = v;
}

// NaN-fill of a box (lo, size) of a float canvas: Canvas.init_seed's clear restricted to the touched box.
__global__ void fill_box_f32_kernel(float* dst, int sy, int sx, int lz, int ly, int lx, int nz, int ny, int nx, float v) {
  const size_t n = (size_t)nz * ny * nx;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int x = (int)(i % nx), y = (int)((i / nx) % ny), z = (int)(i / ((size_t)nx * ny));
    dst[((size_t)(lz + z) * sy + (ly + y)) * sx + (lx + x)] = v;
  }
}

// dst box <- src box (same canvas geometry): moves the last object's seed values into the canvas's own array.
__global__ void copy_box_f32_kernel(float* dst, const float* src, int sy, int sx, int lz, int ly, int lx, int nz, int ny,
                                    int nx) {
  const size_t n = (size_t)nz * ny * nx;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int x = (int)(i % nx), y = (int)((i / nx) % ny), z = (int)(i / ((size_t)nx * ny));
    const size_t a = ((size_t)(lz + z) * sy + (ly + y)) * sx + (lx + x);
    dst[a] = src[a];
  }
}

#endif  // FFN_MISC_KERNELS_DEFINED

}  // namespace ffn
