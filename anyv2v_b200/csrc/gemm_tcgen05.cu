// tcgen05 GEMM core of the I2VGen-XL UNet hot path (sm_100a only).
//
//   out[slot][m, n] = sum_k A[m, k] * Wt[n, k] + bias[n] + rowbias[m / rpr, n] + residual[slot][m, n]
//
// One persistent CTA per SM, warp-specialised:
//   warp 0  : TMA producer  (A tile 128 x 64 and W tile BN x 64, both K-major, SWIZZLE_128B, mbarrier ring)
//   warp 1  : MMA issuer    (one lane issues tcgen05.mma 128 x BN x 16, fp32 accumulators in TMEM, double-buffered)
//   warp 2  : TMEM allocator
//   warps 4-11: epilogue    (two warpgroups on alternate 32-column chunks: tcgen05.ld -> +bias/+rowbias/+residual -> fp16 ->
//                            swizzled smem -> bulk TMA store, 1..n_slots copies; a conv tile that is a block of pixels goes
//                            through a 5-D (c, x, y, frame, slot) map that clips it at the image edges; direct 16 B stores for
//                            temporal-conv tiles whose rows are not contiguous in the output).  The epilogue is a template parameter: three lean straight-line flavours
//                            (plain / +residual / GEGLU, one slot) and the generic one — for short K the epilogue warps' instruction
//                            stream, not the tensor pipe, sets the tile time (profiles/r02_gemm_k320_epilogue.txt)
//
// The A operand is never materialised as an im2col buffer: for 3x3 convolutions the producer issues one 4-D TMA
// box per filter tap with the (dy, dx) shift folded into the coordinates (out-of-bounds = zero padding; the box is the tile's
// block of box_h x box_w output pixels, or whole frames — av2v_conv3x3_plan); for the
// (3,1,1) temporal convolution a 3-D box shifted by +-HW rows within the clip.
//
// Replaces (reference = library calls inside PyTorch): cuBLAS Linear at pnp_utils.py:178-186,216; cuDNN conv at
// pnp_utils.py:78,107,117-122; and, as "next" rows, every other Linear/Conv of the UNet.
#include <cstdlib>
#include <cstring>

#include "host_util.cuh"
#include "ptx.cuh"

namespace av2v {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kThreads = 384;
constexpr int kEpiBufBytes = 128 * 64;   // one 128-row x 32-column fp16 staging tile (SWIZZLE_64B)
constexpr int kEpiGroups = 2;            // epilogue warpgroups (alternate chunks)
constexpr int kNumOutBufs = 3;           // per group: output staging ring (TMA store sources)
// residual staging buffers per epilogue group (TMA load destinations): ONE residual load in flight per group.  Measured on B200
// (profiles/r02_probe.txt): four buffers (three loads in flight) gain 5 % at K = 320 and lose 7 % at K >= 1280 (they cost a
// pipeline stage) — not kept.  A W-stationary schedule for K <= 320 was also measured and is slower (-5 ... -13 %): not kept.
constexpr int kRes = 2;

// epilogue flavours (template parameter): the generic one covers every combination (slots, row bias, up-sampling store, GEGLU,
// residual, direct stores); the lean ones are straight-line code for the three shapes the short-K projections use.  E_BLOCK (a flag
// on E_PLAIN / E_RES): the conv tiles are pixel blocks stored through the 5-D block map — a separate instantiation, so that the
// row-contiguous lean kernels the projections run carry none of the block bookkeeping
enum { E_GENERIC = 0, E_PLAIN = 1, E_RES = 2, E_GEGLU = 3, E_BLOCK = 4 };

template <int BN, bool kPair, int kEpi>
struct GemmCfg {
  // ... and two output staging buffers per group are enough for the lean flavours (the store of chunk n - 1 has one chunk time to
  // read its source): +1 pipeline stage for most tile shapes (measured: 196608x960x320 147.7 -> 131.7 us, GEGLU 12288x10240x1280 213.8 -> 202.7)
  static constexpr int kOutBufs = ((kEpi & 3) != E_GENERIC) ? 2 : kNumOutBufs;
  // the plain and GEGLU flavours never stage a residual: their two buffers per group become (part of) one more pipeline stage
  static constexpr int kResBufs = ((kEpi & 3) == E_PLAIN || (kEpi & 3) == E_GEGLU) ? 0 : kRes;
  static constexpr int kEpiBytes = kEpiGroups * (kOutBufs + kResBufs) * kEpiBufBytes;
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = (kPair ? BN / 2 : BN) * BK * 2;  // pair mode: each CTA stages only its half of the W tile
  static constexpr int kSmemBudget = 232448 - 1024 - 512 - 1024 - kEpiBytes;  // 227 KB minus slack, barriers, fp32 bias, staging
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStagesRaw = kSmemBudget / kStageBytes;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  static constexpr int kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  static constexpr int kOperandBytes = kStages * kStageBytes;  // A + B ring
  static constexpr int kSmemBytes = kOperandBytes + kEpiBytes + 1024 + 512 + 1024;
  static_assert(2 * BN <= 512, "double-buffered accumulator must fit TMEM");
  static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "UMMA N constraint for M=128");
  static_assert(kBBytes % 1024 == 0, "SWIZZLE_128B tiles need 1024 B aligned bases");
};

struct GemmKParams {
  int M, N;
  int num_kb, kb_per_tap;
  int mode;
  int m_tiles, n_tiles;
  // conv3x3 geometry: a tile is a block of box_h rows x box_w columns of one frame (x_tiles = ceil(W / box_w) blocks per row of
  // blocks), or frames_per_tile > 1 whole frames; tile order (frame, row block, column block) — av2v_conv3x3_plan
  int H, W, HW, NF, box_w, box_h, tiles_per_frame, frames_per_tile;
  int x_tiles;
  int block_store;  // conv3x3: the tile's rows are not 128 consecutive output rows -> stores / residual loads through the 5-D
                    // block map (c, x, y, frame, slot), which clips the block at the image's right and bottom edges
  uint32_t o_box_bytes;  // bytes of one 32-column staging chunk as the store / residual map moves it (64 B per tile row)
  int stride;   // conv3x3: 1 or 2 (H, W above are the OUTPUT geometry; the taps address input pixel stride * out + tap - 1)
  int taps_w;   // 3: 3 x 3 taps at offsets -1 .. +1; 2: the 2 x 2 taps of one output phase of "nearest-up x 2 then conv 3 x 3"
  int tap_oy, tap_ox;  // taps_w = 2: phase (py, px): tap (a, b) reads input pixel (i + a - 1 + py, j + b - 1 + px)
  int up2;      // 1: the tile's pixels (i, j) are stored to output pixels (2 i + py, 2 j + px) through a 5-D tensor map
                //    (px * N + c, j, py, i, frame)
  int kb_split; // linear: k-blocks [0, kb_split) come from tmap_a, the rest from tmap_a2 (two-source K loop); = num_kb otherwise
  // tconv geometry
  int tiles_per_clip, rows_per_clip;
  uint32_t a_box_bytes;
  // epilogue
  const __half* bias;
  const __half* rowbias;
  int rows_per_rowbias;
  const __half* residual;
  __half* out;
  int ldo;
  int n_slots;
  long long slot_stride;
  int fast_epi;  // 1: tile rows are contiguous in the output -> smem-staged TMA-store epilogue
  int geglu;     // 1: column chunks come in (h, gate) pairs; store h * gelu_erf(gate) -> N/2 output columns
  int debug;     // bring-up only (AV2V_GEMM_DEBUG): bit3 role timers
  int mc2;       // 2: CTA pair with cta_group::2 MMA (UMMA M = 256): clusters of 2 CTAs on M-adjacent tiles of the same N
                 //    tile; each CTA holds its 128 rows of A and HALF of the W tile; the leader CTA issues the MMAs for both
                 //    tensor cores (halves the L2 -> smem traffic of B).  0: independent CTAs.  (A plain W-tile multicast
                 //    between independent MMAs — "1" in round 1 — was measured neutral and is gone.)
};

// Static persistent tile schedule shared by all warp roles.  Unit u = tile (plain) or pair of M-adjacent tiles (mc2).
struct TileSched {
  int first, stride, n_tiles, num_units, rank, mc2;
  __device__ __forceinline__ bool get(int i, int& m_tile, int& n_tile) const {
    const int u = first + i * stride;
    if (u >= num_units) return false;
    int mu = u / n_tiles;
    n_tile = u - mu * n_tiles;
    m_tile = mc2 ? 2 * mu + rank : mu;
    return true;
  }
};

// conv3x3: first output pixel (frame n0, row y0, column x0) of tile m_tile; tile row r of the accumulator is pixel
// (n0 + r / (box_w * box_h), y0 + (r / box_w) % box_h, x0 + r % box_w) — the order of the A box in shared memory
__device__ __forceinline__ void conv_tile_origin(const GemmKParams& p, int m_tile, int& n0, int& y0, int& x0) {
  if (p.frames_per_tile == 1) {
    n0 = m_tile / p.tiles_per_frame;
    const int rem = m_tile - n0 * p.tiles_per_frame;
    const int yb = rem / p.x_tiles;
    y0 = yb * p.box_h;
    x0 = (rem - yb * p.x_tiles) * p.box_w;
  } else {
    n0 = m_tile * p.frames_per_tile;
    y0 = 0;
    x0 = 0;
  }
}

// Exact-erf GELU, branch-free: gelu(g) = g/2 + |g|/2 * erf(|g|/sqrt 2) with erf from Abramowitz & Stegun 7.1.25
// (3-term, |abs err| < 2.5e-5 — two orders below fp16 resolution) on MUFU rcp / ex2: ~14 instructions per element.
// The GEGLU epilogue is issue-bound for K = 320 (128 x 128 activations per 2560 tensor-pipe cycles), so every
// instruction counts; libdevice erff costs about twice as much and diverges.
__device__ __forceinline__ float gelu_erf_fast(float g) {
  const float u = fabsf(g) * 0.70710678118654752f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.47047f, u, 1.0f)));
  float poly = fmaf(t, 0.7478556f, -0.0958798f);
  poly = fmaf(poly, t, 0.3480242f);
  poly *= t;
  const float e = ex2_approx(u * u * -1.4426950408889634f);
  const float erf_abs = fmaf(-poly, e, 1.0f);
  const float hg = 0.5f * g;
  return fmaf(fabsf(hg), erf_abs, hg);
}

// gelu_erf_fast on two elements with packed fp32x2 arithmetic (FFMA2 / FMUL2): the SAME operations per element in the same
// order (IEEE fma / mul per lane), so the result is bit-identical to gelu_erf_fast; ~8.5 issue slots per element instead of
// ~14.  The GEGLU epilogue at K = 320 is instruction-issue bound: +2 ... +7 % on the fused GEGLU GEMMs (profiles/r02_probe.txt).
__device__ __forceinline__ float2 gelu_erf_fast2(float2 g) {
  const float2 u = make_float2(fabsf(g.x) * 0.70710678118654752f, fabsf(g.y) * 0.70710678118654752f);
  const float2 d = ffma2(make_float2(0.47047f, 0.47047f), u, make_float2(1.0f, 1.0f));
  float2 t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.x) : "f"(d.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.y) : "f"(d.y));
  float2 poly = ffma2(t, make_float2(0.7478556f, 0.7478556f), make_float2(-0.0958798f, -0.0958798f));
  poly = ffma2(poly, t, make_float2(0.3480242f, 0.3480242f));
  poly = fmul2(poly, t);
  const float2 a = fmul2(fmul2(u, u), make_float2(-1.4426950408889634f, -1.4426950408889634f));
  const float2 e = make_float2(ex2_approx(a.x), ex2_approx(a.y));
  const float2 erf_abs = ffma2(make_float2(-poly.x, -poly.y), e, make_float2(1.0f, 1.0f));
  const float2 hg = fmul2(make_float2(0.5f, 0.5f), g);
  return make_float2(fmaf(fabsf(hg.x), erf_abs.x, hg.x), fmaf(fabsf(hg.y), erf_abs.y, hg.y));
}

// bring-up instrumentation (AV2V_GEMM_DEBUG bit3): cycles CTA 0 spends waiting, per role
__device__ unsigned long long g_gemm_timers[16];
#ifdef AV2V_GEMM_BRINGUP
#define AV2V_DBG(bit) ((p.debug & (bit)) != 0)
#else
#define AV2V_DBG(bit) false
#endif
#define AV2V_T0() const long long t0__ = AV2V_DBG(8) ? clock64() : 0
#define AV2V_T1(acc) do { if (AV2V_DBG(8)) (acc) += clock64() - t0__; } while (0)

template <int BN, bool kPair, int kEpi>  // kPair: cta_group::2 build (ptxas marks such kernels cluster-only -> separate instantiation)
__global__ void __launch_bounds__(kThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                    const __grid_constant__ CUtensorMap tmap_o, const __grid_constant__ CUtensorMap tmap_r,
                    const __grid_constant__ CUtensorMap tmap_bh, const __grid_constant__ CUtensorMap tmap_a2, const GemmKParams p) {
  using Cfg = GemmCfg<BN, kPair, kEpi>;
  constexpr int S = Cfg::kStages;
  constexpr int kNumResBufs = kRes;
  constexpr int kEpiBytes = Cfg::kEpiBytes;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + S * Cfg::kABytes;
  uint8_t* smem_epi_out = smem + Cfg::kOperandBytes;
  uint8_t* smem_epi_res = smem_epi_out + kEpiGroups * Cfg::kOutBufs * kEpiBufBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kOperandBytes + kEpiBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + S;
  uint64_t* tfull = bars + 2 * S;
  uint64_t* tempty = bars + 2 * S + 2;
  uint64_t* res_full = bars + 2 * S + 4;  // kEpiGroups * kNumResBufs
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 4 + kEpiGroups * kNumResBufs);
  float* bias_stage = reinterpret_cast<float*>(smem + Cfg::kOperandBytes + kEpiBytes + 512);  // kEpiGroups x 128 floats

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    if (p.kb_split < p.num_kb) tma_prefetch_desc(&tmap_a2);
    if (p.fast_epi) {
      tma_prefetch_desc(&tmap_o);
      if (p.residual != nullptr) tma_prefetch_desc(&tmap_r);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < S; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kPair ? 16 : (p.fast_epi ? 8 : 4));  // pair mode: both CTAs' epilogues free the leader
    }
    for (int i = 0; i < kEpiGroups * kNumResBufs; ++i) mbar_init(&res_full[i], 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    if constexpr (kPair) tmem_alloc_cg2<Cfg::kTmemCols>(tmem_slot);
    else tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  if (p.mc2) cluster_sync();  // peer barriers must be initialised before any multicast lands / remote arrive
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);  // provably warp-uniform -> uniform registers

  TileSched sched;
  sched.mc2 = p.mc2;
  sched.rank = p.mc2 ? static_cast<int>(blockIdx.x & 1u) : 0;
  sched.first = p.mc2 ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  sched.stride = p.mc2 ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  sched.n_tiles = p.n_tiles;
  sched.num_units = p.mc2 ? ((p.m_tiles + 1) / 2) * p.n_tiles : p.m_tiles * p.n_tiles;

  if (warp == 0) {
    // ===================================================================== TMA producer
    // The whole warp runs the loop convergently with warp-uniform operands (-> uniform registers); `lead` issues.  Under
    // a divergent `if (lane == 0)` every UTMALDG / UTCHMMA is wrapped in an ELECT + R2UR + BRA.U.ANY loop (~90 cycles).
    {
      const uint32_t lead = elect_one() ? 1u : 0u;
      int stage = 0;
      uint32_t phase = 0;
      long long tm_prod_wait = 0;
      const long long tm_start = clock64();
      int m_tile, n_tile;
      for (int ti = 0; sched.get(ti, m_tile, n_tile); ++ti) {
        int c_n = 0, c_y = 0, c_r = 0, c_x = 0;
        if (p.mode == AV2V_A_CONV3X3) {
          conv_tile_origin(p, m_tile, c_n, c_y, c_x);
        } else if (p.mode == AV2V_A_TCONV3) {
          c_n = m_tile / p.tiles_per_clip;
          c_r = (m_tile - c_n * p.tiles_per_clip) * BM;
        }
        for (int kb = 0; kb < p.num_kb; ++kb) {
          {
            AV2V_T0();
            mbar_wait(&empty[stage], phase ^ 1u);
            AV2V_T1(tm_prod_wait);
          }
          void* da = smem_a + stage * Cfg::kABytes;
          void* db = smem_b + stage * Cfg::kBBytes;
          const int tap = p.mode == AV2V_A_LINEAR ? 0 : kb / p.kb_per_tap;
          const int cb = p.mode == AV2V_A_LINEAR ? kb : kb - tap * p.kb_per_tap;
          // linear: which source holds this k-block (skip-concat as a two-source K loop)
          const CUtensorMap* ta_lin = kb < p.kb_split ? &tmap_a : &tmap_a2;
          const int kcol = (kb < p.kb_split ? kb : kb - p.kb_split) * BK;
          if constexpr (kPair) {
            // CTA pair: this CTA's A rows + its half of the W tile go to its own smem; the bytes of BOTH CTAs complete
            // on the leader's barrier, which the leader's producer arms for the pair
            const uint32_t lead_full = mapa_u32(smem_u32(&full[stage]), 0);
            if (sched.rank == 0) mbar_arrive_expect_tx_w(lead, &full[stage], 2 * (p.a_box_bytes + Cfg::kBBytes));
            if (p.mode == AV2V_A_LINEAR) {
              tma_load_2d_cg2_w(lead, da, ta_lin, lead_full, kcol, m_tile * BM);
            } else if (p.mode == AV2V_A_CONV3X3) {
              const int dy = tap / p.taps_w - 1 + p.tap_oy, dx = tap - (tap / p.taps_w) * p.taps_w - 1 + p.tap_ox;
              tma_load_4d_cg2_w(lead, da, &tmap_a, lead_full, cb * BK, c_x * p.stride + dx, c_y * p.stride + dy, c_n);
            } else {
              tma_load_3d_cg2_w(lead, da, &tmap_a, lead_full, cb * BK, c_r + (tap - 1) * p.HW, c_n);
            }
            tma_load_2d_cg2_w(lead, db, &tmap_bh, lead_full, kb * BK, n_tile * BN + sched.rank * (BN / 2));
          } else {
            const bool skip_b = AV2V_DBG(32) && !(ti == 0 && kb < S);  // bring-up: bit5 = W tiles loaded once per stage only
            const bool skip_a = AV2V_DBG(1024) && !(ti == 0 && kb < S);  // bring-up: bit10 = A tiles loaded once per stage only
            mbar_arrive_expect_tx_w(lead, &full[stage], (skip_a ? 0 : p.a_box_bytes) + (skip_b ? 0 : Cfg::kBBytes));
            if (p.mode == AV2V_A_LINEAR) {
              if (!skip_a) tma_load_2d_w(lead, da, ta_lin, &full[stage], kcol, m_tile * BM);
            } else if (p.mode == AV2V_A_CONV3X3) {
              const int dy = tap / p.taps_w - 1 + p.tap_oy, dx = tap - (tap / p.taps_w) * p.taps_w - 1 + p.tap_ox;
              tma_load_4d_w(lead, da, &tmap_a, &full[stage], cb * BK, c_x * p.stride + dx, c_y * p.stride + dy, c_n);
            } else {
              tma_load_3d_w(lead, da, &tmap_a, &full[stage], cb * BK, c_r + (tap - 1) * p.HW, c_n);
            }
            if (!skip_b) tma_load_2d_w(lead, db, &tmap_b, &full[stage], kb * BK, n_tile * BN);
          }
          if (++stage == S) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
      if (AV2V_DBG(8) && blockIdx.x == 0 && lead) {
        g_gemm_timers[0] = tm_prod_wait;
        g_gemm_timers[1] = clock64() - tm_start;
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    if (!(kPair && sched.rank != 0)) {  // CTA pair: the leader CTA issues for both tensor cores; warp-convergent issue
      const uint32_t lead = elect_one() ? 1u : 0u;
      constexpr uint32_t idesc = make_idesc_f16(BM, BN, 0, 0);
      constexpr uint32_t idesc_pair = make_idesc_f16(2 * BM, BN, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t it = 0;
      long long tm_mma_tempty = 0, tm_mma_full = 0;
      const long long tm_start = clock64();
      int m_tile, n_tile;
      for (int ti = 0; sched.get(ti, m_tile, n_tile); ++ti, ++it) {
        const uint32_t acc = it & 1u;
        const uint32_t acc_phase = (it >> 1) & 1u;
        {
          AV2V_T0();
          mbar_wait(&tempty[acc], acc_phase ^ 1u);
          AV2V_T1(tm_mma_tempty);
        }
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          {
            AV2V_T0();
            mbar_wait(&full[stage], phase);
            AV2V_T1(tm_mma_full);
          }
          tc_fence_after();
          const uint64_t adesc = make_sdesc(smem_u32(smem_a + stage * Cfg::kABytes), 16, 1024);
          const uint64_t bdesc = make_sdesc(smem_u32(smem_b + stage * Cfg::kBBytes), 16, 1024);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // +32 B along K inside the 128 B swizzle row = +2 in the (addr >> 4) field
            if constexpr (kPair) umma_ss_cg2_w(lead, d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc_pair, (kb | k) != 0 ? 1u : 0u);
            else umma_ss_w(lead, d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          if constexpr (kPair) umma_commit_cg2_mc_w(lead, &empty[stage], 0x3);  // release the stage in BOTH CTAs of the pair
          else umma_commit_w(lead, &empty[stage]);
          if (++stage == S) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if constexpr (kPair) umma_commit_cg2_mc_w(lead, &tfull[acc], 0x3);  // both CTAs' epilogues drain their half of the tile
        else umma_commit_w(lead, &tfull[acc]);
      }
      if (AV2V_DBG(8) && blockIdx.x == 0 && lead) {
        g_gemm_timers[2] = tm_mma_tempty;
        g_gemm_timers[3] = tm_mma_full;
        g_gemm_timers[4] = clock64() - tm_start;
      }
    }
  } else if (warp >= 4) {
    // ===================================================================== epilogue
    const int q = warp & 3;
    const int r = q * 32 + lane;
    uint32_t it = 0;
    if constexpr ((kEpi & 3) != E_GENERIC) {
      // ---- lean staged epilogue (one output slot, no up-sampling store): the flavour is a template parameter, so
      // the per-chunk code is one straight line.  Why: for K = 320 the tile time is set by the epilogue warps, two per
      // scheduler, whose time is their instruction count times the exposed latency (and an instruction-fetch stall after every
      // taken branch over the generic path's cold code) — profiles/r02_gemm_k320_epilogue.txt.  Tile coordinates advance
      // incrementally (no divisions), ring indices are counters, the bias is fp32 in shared memory (packed fp32x2 adds).
      constexpr bool kWithRes = ((kEpi & 3) == E_RES), kGeglu = ((kEpi & 3) == E_GEGLU), kBlock = (kEpi & E_BLOCK) != 0;
      constexpr int kStep = kGeglu ? 4 : 2, kLog = kGeglu ? 2 : 1;
      const int eg = (warp - 4) >> 2;                         // epilogue group 0 / 1
      const uint32_t el = elect_one() ? 1u : 0u;              // this warp's issuing lane, when it is the warp's turn
      const int swz = (r >> 1) & 3;                           // SWIZZLE_64B: 16-byte chunk index ^= address bits [7:8]
      constexpr int kOB = Cfg::kOutBufs;                      // output staging ring of this group
      const uint32_t u_out = smem_u32(smem_epi_out + eg * kOB * kEpiBufBytes);
      const uint32_t u_res = smem_u32(smem_epi_res + eg * kNumResBufs * kEpiBufBytes);
      const uint32_t u_bias = smem_u32(bias_stage + eg * 128);
      const uint32_t u_resbar = smem_u32(res_full + eg * kNumResBufs);
      uint32_t soff[4];
#pragma unroll
      for (int j4 = 0; j4 < 4; ++j4) soff[j4] = r * 64 + ((j4 ^ swz) << 4);
      // block-shaped conv tiles: this thread's row is pixel (bz, by, bx) of the block (fixed); the block's origin is derived from
      // m_tile once per tile (divisions by runtime constants — only on this path)
      int bx = 0, by = 0, bz = 0;
      if constexpr (kBlock) {
        const int bwh = p.box_w * p.box_h;
        bz = r / bwh;
        by = (r - bz * bwh) / p.box_w;
        bx = r - bz * bwh - by * p.box_w;
      }
      // tile iterator: unit u = first + i * stride -> (mu, n_tile), advanced without divisions
      const int nt = sched.n_tiles;
      const int dm = sched.stride / nt, dn = sched.stride - dm * nt;
      const int mu_count = sched.num_units / nt;
      int mu = sched.first / nt, n_tile = sched.first - mu * nt;
      const int full_chunks = BN / 32;
      auto chunks_of = [&](int n) {
        const int nc = (p.N - n * BN + 31) >> 5;
        return nc < full_chunks ? nc : full_chunks;
      };
      // residual prefetch cursor: one load in flight ahead of the chunk being staged; all four warps advance it, the warp whose
      // turn it is issues
      int pf_mu = mu, pf_n = n_tile, pf_c = kGeglu ? 2 * eg : eg, pf_par = 0;
      uint32_t pf_buf = 0;
      auto prefetch_one = [&](uint32_t issue) {
        while (pf_mu < mu_count && pf_c >= chunks_of(pf_n)) {
          pf_n += dn;
          pf_mu += dm;
          if (pf_n >= nt) {
            pf_n -= nt;
            ++pf_mu;
          }
          pf_par ^= 1;
          pf_c = kGeglu ? 2 * eg : (eg ^ pf_par);
        }
        if (pf_mu >= mu_count) return;
        const uint32_t bar = u_resbar + pf_buf * 8, dst = u_res + pf_buf * kEpiBufBytes;
        const int pf_m = sched.mc2 ? 2 * pf_mu + sched.rank : pf_mu;
        mbar_arrive_expect_tx_w(issue, bar, kBlock ? p.o_box_bytes : static_cast<uint32_t>(kEpiBufBytes));
        if constexpr (kBlock) {
          int n0, y0, x0;
          conv_tile_origin(p, pf_m, n0, y0, x0);
          tma_load_5d_w(issue, dst, &tmap_r, bar, pf_n * BN + pf_c * 32, x0, y0, n0, 0);
        } else {
          tma_load_3d_w(issue, dst, &tmap_r, bar, pf_n * BN + pf_c * 32, pf_m * BM, 0);
        }
        pf_buf ^= 1u;
        pf_c += kStep;
      };
      static_assert(kRes == 2, "the lean epilogue toggles between two residual buffers");
      if constexpr (kWithRes) {  // both buffers in flight from the start; afterwards chunk n + 2 is fetched once chunk n is staged
        prefetch_one(q == 0 ? el : 0u);
        prefetch_one(q == 0 ? el : 0u);
      }
      uint32_t ob = 0;       // output staging ring position (kOB)
      uint32_t rb = 0, rph = 0;  // residual ring position / phase
      uint32_t turn = 0;     // warp of the group that issues this chunk's store
      int par = 0;
      for (; mu < mu_count; ++it, par ^= 1) {
        const int m_tile = sched.mc2 ? 2 * mu + sched.rank : mu;
        const uint32_t acc = it & 1u;
        const uint32_t acc_phase = (it >> 1) & 1u;
        const int nchunks = AV2V_DBG(16) ? 0 : chunks_of(n_tile);
        long long grow = static_cast<long long>(m_tile) * BM + r;  // contiguous tiles: 128 consecutive output rows
        bool valid = grow < p.M;
        int o_x = 0, o_y = m_tile * BM, o_n = 0;  // store / residual coordinates of the tile (contiguous: row, -)
        if constexpr (kBlock) {
          conv_tile_origin(p, m_tile, o_n, o_y, o_x);
          const int xx = o_x + bx, yy = o_y + by, nn = o_n + bz;
          valid = bz < p.frames_per_tile && xx < p.W && yy < p.H && nn < p.NF;
          grow = static_cast<long long>(nn) * p.HW + static_cast<long long>(yy) * p.W + xx;
        }
        const int rb_row = (p.rowbias != nullptr && valid) ? static_cast<int>(grow / p.rows_per_rowbias) : 0;
        const int first = kGeglu ? 2 * eg : (eg ^ par);
        const int n_own = nchunks > first ? (nchunks - first + kStep - 1) >> kLog : 0;
        const int last_c = n_own > 0 ? first + (n_own - 1) * kStep + (kGeglu ? 1 : 0) : -1;
        {
          // warp q stages the fp32 bias of the group's q-th chunk of this tile (GEGLU: value / gate chunks of its pairs), lane =
          // column; the previous tile's reads all precede its last chunk barrier, so the buffer is free here
          const int c_k = kGeglu ? first + (q >> 1) * kStep + (q & 1) : first + q * kStep;
          const int col = n_tile * BN + c_k * 32 + lane;
          float bv = 0.0f;
          if (p.bias != nullptr && c_k < nchunks && col < p.N) bv = __half2float(__ldg(p.bias + col));
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(u_bias + (q * 32 + lane) * 4), "f"(bv) : "memory");
          asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
        }
        mbar_wait(&tfull[acc], acc_phase);
        tc_fence_after();
        const uint32_t t_row = tmem_base + acc * BN + (static_cast<uint32_t>(q * 32) << 16);
        auto release_acc = [&]() {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (kPair) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[acc]), 0));  // the leader's MMA warp waits
            else mbar_arrive(&tempty[acc]);
          }
        };
        if (last_c < 0) release_acc();
        auto load_acc_biased = [&](int c, int k, float (&f)[32]) {  // accumulator chunk c + the k-th staged bias chunk
          uint32_t v[32];
          tmem_ld32(t_row + c * 32, v);
          float4 b[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b[j].x), "=f"(b[j].y), "=f"(b[j].z), "=f"(b[j].w) : "r"(u_bias + k * 128 + j * 16));
          tmem_ld_wait();
          if (c == last_c) release_acc();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float2 lo = fadd2(make_float2(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1])), make_float2(b[j].x, b[j].y));
            const float2 hi = fadd2(make_float2(__uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])), make_float2(b[j].z, b[j].w));
            f[4 * j] = lo.x;
            f[4 * j + 1] = lo.y;
            f[4 * j + 2] = hi.x;
            f[4 * j + 3] = hi.y;
          }
        };
        int k = 0;
#pragma unroll 1
        for (int c = first; c < nchunks; c += kStep, ++k) {
          float f[32];
          int col0;
          if constexpr (kGeglu) {
            float gate[32];
            load_acc_biased(c, 2 * k, f);
            load_acc_biased(c + 1, 2 * k + 1, gate);
#pragma unroll
            for (int j = 0; j < 32; j += 2) {  // packed fp32x2 arithmetic; one rounding (to fp16) at the store
              const float2 r2 = fmul2(make_float2(f[j], f[j + 1]), gelu_erf_fast2(make_float2(gate[j], gate[j + 1])));
              f[j] = r2.x;
              f[j + 1] = r2.y;
            }
            col0 = n_tile * (BN / 2) + (c >> 1) * 32;
          } else {
            load_acc_biased(c, k, f);
            col0 = n_tile * BN + c * 32;
            if (p.rowbias != nullptr && valid) {  // per-row-block bias (time embedding of conv1): fp16 [rows / rpr][N]
              const uint4* b4 = reinterpret_cast<const uint4*>(p.rowbias + static_cast<long long>(rb_row) * p.N + col0);
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4) {
                if (col0 + j4 * 8 < p.N) {
                  const uint4 bv = __ldg(b4 + j4);
                  const __half2* h2 = reinterpret_cast<const __half2*>(&bv);
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float2 s2 = fadd2(make_float2(f[j4 * 8 + 2 * e], f[j4 * 8 + 2 * e + 1]), __half22float2(h2[e]));
                    f[j4 * 8 + 2 * e] = s2.x;
                    f[j4 * 8 + 2 * e + 1] = s2.y;
                  }
                }
              }
            }
          }
          const uint32_t obuf = u_out + ob * kEpiBufBytes;
          if constexpr (kWithRes) {
            mbar_wait(&res_full[eg * kNumResBufs + rb], rph);
            const uint32_t rbuf = u_res + rb * kEpiBufBytes;
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              uint4 rv;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rv.x), "=r"(rv.y), "=r"(rv.z), "=r"(rv.w) : "r"(rbuf + soff[j4]));
              const __half2* h2 = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 s2 = fadd2(make_float2(f[j4 * 8 + 2 * e], f[j4 * 8 + 2 * e + 1]), __half22float2(h2[e]));
                f[j4 * 8 + 2 * e] = s2.x;
                f[j4 * 8 + 2 * e + 1] = s2.y;
              }
            }
            rph ^= rb;  // phase flips after buffer 1
            rb ^= 1u;
          }
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4)
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(obuf + soff[j4]), "r"(pack_half2(f[j4 * 8], f[j4 * 8 + 1])),
                         "r"(pack_half2(f[j4 * 8 + 2], f[j4 * 8 + 3])), "r"(pack_half2(f[j4 * 8 + 4], f[j4 * 8 + 5])),
                         "r"(pack_half2(f[j4 * 8 + 6], f[j4 * 8 + 7]))
                         : "memory");
          // the buffer staged NEXT was the source of the store issued kOB - 1 chunks ago by the warp whose turn it was then: that
          // warp confirms the store has read its source before this chunk's barrier (bulk groups are per thread)
          if (q == static_cast<int>((turn + 5u - kOB) & 3u)) {
            if (el) tma_store_wait_read<0>();
            __syncwarp();
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
          const uint32_t issue = (q == static_cast<int>(turn)) ? el : 0u;
          if (q == static_cast<int>(turn) && !AV2V_DBG(64)) {
            if constexpr (kBlock)
              tma_store_5d_w(issue, &tmap_o, __shfl_sync(0xffffffffu, obuf, 0), __shfl_sync(0xffffffffu, col0, 0),
                             __shfl_sync(0xffffffffu, o_x, 0), __shfl_sync(0xffffffffu, o_y, 0), __shfl_sync(0xffffffffu, o_n, 0), 0);
            else
              tma_store_3d_w(issue, &tmap_o, __shfl_sync(0xffffffffu, obuf, 0), __shfl_sync(0xffffffffu, col0, 0),
                             __shfl_sync(0xffffffffu, o_y, 0), 0);
            if (issue) tma_store_commit();
            __syncwarp();
          }
          if constexpr (kWithRes) prefetch_one(issue);
          ob = (ob == kOB - 1) ? 0u : ob + 1u;
          turn = (turn + 1u) & 3u;
        }
        n_tile += dn;
        mu += dm;
        if (n_tile >= nt) {
          n_tile -= nt;
          ++mu;
        }
      }
      if (el) tma_store_wait0();
    } else
    if (p.fast_epi) {
      // (generic flavour: 3-slot injection stores and the up-sampling store in the product; its GEGLU / single-slot branches only run
      // when the bring-up build forces this flavour for an A/B against the lean ones)
      // ---- staged epilogue: TMEM -> registers -> (+bias, +rowbias, +TMA-prefetched residual) -> swizzled smem tile
      //      -> one bulk TMA store per 128 x 32 sub-tile and slot.  All global traffic is asynchronous bulk copies.
      // Two epilogue warpgroups take alternate 32-column chunks of every tile so that one group's latency chain
      // (TMEM load -> bias -> convert -> staging -> fence/barrier -> TMA issue) overlaps the other's.  For short K the
      // epilogue, not the tensor pipe, bounds the tile time (profiles/r02_gemm_k320_epilogue.txt), hence:
      //  * the group that owns the odd chunk alternates from tile to tile (BN = 160 has five chunks),
      //  * the issuing role (TMA store, residual prefetch) rotates over the group's four warps per staged chunk, so no
      //    single warp carries that work while the other three wait for it at the next barrier,
      //  * the bias is converted to fp32 ONCE per tile into shared memory and added with packed fp32x2 adds.
      const int eg = (warp - 4) >> 2;                         // epilogue group 0 / 1
      const uint32_t el = elect_one() ? 1u : 0u;              // this warp's issuing lane, when it is the warp's turn
      const bool has_res = p.residual != nullptr;
      const int swz = (r >> 1) & 3;  // SWIZZLE_64B: 16-byte chunk index ^= address bits [7:8]
      const uint32_t u_out = smem_u32(smem_epi_out + eg * kNumOutBufs * kEpiBufBytes);
      const uint32_t u_res = smem_u32(smem_epi_res + eg * kNumResBufs * kEpiBufBytes);
      uint32_t soff[4];              // this thread's four 16-byte pieces of its staging row
#pragma unroll
      for (int j4 = 0; j4 < 4; ++j4) soff[j4] = r * 64 + ((j4 ^ swz) << 4);
      uint64_t* my_res_full = res_full + eg * kNumResBufs;
      float* my_bias = bias_stage + eg * 128;                  // fp32 bias of the (up to four) chunks this group owns in a tile
      int bx = 0, by = 0, bz = 0;                              // block-shaped conv tiles: this thread's pixel within the block
      if (p.block_store) {
        const int bwh = p.box_w * p.box_h;
        bz = r / bwh;
        by = (r - bz * bwh) / p.box_w;
        bx = r - bz * bwh - by * p.box_w;
      }
      const int step = p.geglu ? 4 : 2;                        // chunk stride between this group's work units
      auto first_of = [&](int ti) { return p.geglu ? 2 * eg : (eg ^ (ti & 1)); };  // first chunk of this group in tile ti
      auto chunks_of = [&](int n_tile) {
        const int rem = p.N - n_tile * BN;
        const int nc = (rem + 31) / 32;
        return nc < BN / 32 ? nc : BN / 32;
      };
      // cursor of the residual prefetcher: this group's iteration -> (tile, chunk, slot).  All four warps advance it; the warp
      // whose turn it is issues the load.
      int pf_ti = 0, pf_c = first_of(0), pf_s = 0, pf_m = 0, pf_n = 0;
      uint32_t pf_iter = 0;
      bool pf_live = sched.get(0, pf_m, pf_n);
      auto pf_normalise = [&]() {  // skip tiles in which this group owns no chunk
        while (pf_live && pf_c >= chunks_of(pf_n)) {
          pf_live = sched.get(++pf_ti, pf_m, pf_n);
          pf_c = first_of(pf_ti);
        }
      };
      auto prefetch_one = [&](uint32_t issue) {
        pf_normalise();
        if (!pf_live) return;
        const uint32_t b = pf_iter % kNumResBufs;
        const uint32_t u_bar = __shfl_sync(0xffffffffu, smem_u32(&my_res_full[b]), 0);
        const uint32_t u_dst = __shfl_sync(0xffffffffu, u_res + b * kEpiBufBytes, 0);
        mbar_arrive_expect_tx_w(issue, u_bar, p.o_box_bytes);
        if (p.block_store) {
          int n0, y0, x0;
          conv_tile_origin(p, pf_m, n0, y0, x0);
          tma_load_5d_w(issue, u_dst, &tmap_r, u_bar, __shfl_sync(0xffffffffu, pf_n * BN + pf_c * 32, 0), __shfl_sync(0xffffffffu, x0, 0),
                        __shfl_sync(0xffffffffu, y0, 0), __shfl_sync(0xffffffffu, n0, 0), __shfl_sync(0xffffffffu, pf_s, 0));
        } else {
          tma_load_3d_w(issue, u_dst, &tmap_r, u_bar, __shfl_sync(0xffffffffu, pf_n * BN + pf_c * 32, 0),
                        __shfl_sync(0xffffffffu, pf_m * BM, 0), __shfl_sync(0xffffffffu, pf_s, 0));
        }
        ++pf_iter;
        if (++pf_s == p.n_slots) {
          pf_s = 0;
          pf_c += step;
        }
      };
      if (has_res) {
        for (int i = 0; i < kNumResBufs - 1; ++i) prefetch_one(q == 0 ? el : 0u);
      }
      uint32_t ei = 0;
      int m_tile, n_tile;
      for (int ti = 0; sched.get(ti, m_tile, n_tile); ++ti, ++it) {
        const uint32_t acc = it & 1u;
        const uint32_t acc_phase = (it >> 1) & 1u;
        long long grow = static_cast<long long>(m_tile) * BM + r;
        bool valid = grow < p.M;
        int o_n = 0, o_y = 0, o_x = 0;  // block stores / up2: the tile's first output pixel
        if (p.block_store || p.up2) conv_tile_origin(p, m_tile, o_n, o_y, o_x);
        if (p.block_store) {
          const int xx = o_x + bx, yy = o_y + by, nn = o_n + bz;
          valid = bz < p.frames_per_tile && xx < p.W && yy < p.H && nn < p.NF;
          grow = static_cast<long long>(nn) * p.HW + static_cast<long long>(yy) * p.W + xx;
        }
        const long long rb_row = (p.rowbias != nullptr && valid) ? grow / p.rows_per_rowbias : 0;
        const int nchunks = AV2V_DBG(16) ? 0 : chunks_of(n_tile);  // bring-up: bit4 = epilogue only frees the accumulator
        const int first = first_of(ti);
        // last chunk this group reads from the accumulator (after it, the TMEM buffer can go back to the MMA warp)
        const int n_own = nchunks > first ? (nchunks - first + step - 1) / step : 0;
        const int last_c = n_own > 0 ? first + (n_own - 1) * step + (p.geglu ? 1 : 0) : -1;
        if (p.bias != nullptr) {
          // warp q stages the bias of the group's q-th chunk of this tile (GEGLU: value / gate chunks of the pairs), lane =
          // column.  The previous tile's reads all precede its last chunk barrier, so the buffer is free here.
          const int c_k = p.geglu ? first + (q >> 1) * step + (q & 1) : first + q * step;
          const int col = n_tile * BN + c_k * 32 + lane;
          my_bias[q * 32 + lane] = (c_k < nchunks && col < p.N) ? __half2float(p.bias[col]) : 0.0f;
          asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
        }
        auto add_bias = [&](int k, float (&f)[32]) {  // k: ordinal of the chunk in my_bias
          if (p.bias == nullptr) return;
          const float4* b4 = reinterpret_cast<const float4*>(my_bias + k * 32);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b = b4[j];
            const float2 lo = fadd2(make_float2(f[4 * j], f[4 * j + 1]), make_float2(b.x, b.y));
            const float2 hi = fadd2(make_float2(f[4 * j + 2], f[4 * j + 3]), make_float2(b.z, b.w));
            f[4 * j] = lo.x;
            f[4 * j + 1] = lo.y;
            f[4 * j + 2] = hi.x;
            f[4 * j + 3] = hi.y;
          }
        };
        mbar_wait(&tfull[acc], acc_phase);
        tc_fence_after();
        const uint32_t t_row = tmem_base + acc * BN + (static_cast<uint32_t>(q * 32) << 16);
        auto release_acc = [&]() {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (kPair) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[acc]), 0));  // the leader's MMA warp waits
            else mbar_arrive(&tempty[acc]);
          }
        };
        if (last_c < 0) release_acc();  // this group owns nothing in a narrow last tile: release immediately
        auto load_acc = [&](int c, float (&f)[32]) {
          uint32_t v[32];
          tmem_ld32(t_row + c * 32, v);
          tmem_ld_wait();
          if (c == last_c) release_acc();
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
        };
        auto add_rowbias = [&](int c, float (&f)[32]) {
          if (p.rowbias == nullptr || !valid) return;
          const int col0 = n_tile * BN + c * 32;
          const uint4* b4 = reinterpret_cast<const uint4*>(p.rowbias + rb_row * p.N + col0);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            if (col0 + j4 * 8 < p.N) {
              const uint4 bv = __ldg(b4 + j4);
              const __half2* h2 = reinterpret_cast<const __half2*>(&bv);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 t = __half22float2(h2[e]);
                f[j4 * 8 + 2 * e] += t.x;
                f[j4 * 8 + 2 * e + 1] += t.y;
              }
            }
          }
        };
        int k = 0;
#pragma unroll 1
        for (int c = first; c < nchunks; c += step, ++k) {
          float f[32];
          int col0;
          if (p.geglu) {
            float gate[32];
            load_acc(c, f);
            add_bias(2 * k, f);
            load_acc(c + 1, gate);
            add_bias(2 * k + 1, gate);
#pragma unroll
            for (int j = 0; j < 32; j += 2) {  // packed fp32x2 arithmetic; one rounding (to fp16) at the store
              const float2 r2 = fmul2(make_float2(f[j], f[j + 1]), gelu_erf_fast2(make_float2(gate[j], gate[j + 1])));
              f[j] = r2.x;
              f[j + 1] = r2.y;
            }
            col0 = n_tile * (BN / 2) + (c >> 1) * 32;
          } else {
            load_acc(c, f);
            add_bias(k, f);
            add_rowbias(c, f);
            col0 = n_tile * BN + c * 32;
          }
#pragma unroll 1
          for (int s = 0; s < p.n_slots; ++s, ++ei) {
            const uint32_t obuf = u_out + (ei % kNumOutBufs) * kEpiBufBytes;
            const uint32_t rbuf = u_res + (ei % kNumResBufs) * kEpiBufBytes;
            if (has_res) mbar_wait(&my_res_full[ei % kNumResBufs], (ei / kNumResBufs) & 1u);
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              float g[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) g[e] = f[j4 * 8 + e];
              if (has_res) {
                uint4 rv;
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rv.x), "=r"(rv.y), "=r"(rv.z), "=r"(rv.w) : "r"(rbuf + soff[j4]));
                const __half2* h2 = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 t = __half22float2(h2[e]);
                  g[2 * e] += t.x;
                  g[2 * e + 1] += t.y;
                }
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(obuf + soff[j4]), "r"(pack_half2(g[0], g[1])),
                           "r"(pack_half2(g[2], g[3])), "r"(pack_half2(g[4], g[5])), "r"(pack_half2(g[6], g[7]))
                           : "memory");
            }
            // the buffer staged NEXT iteration was the source of the store issued two iterations ago, by the warp whose turn it
            // was then: that warp confirms the store has read its source before this iteration's barrier (bulk groups are per thread)
            if (q == static_cast<int>((ei + 2) & 3u)) {
              if (el) tma_store_wait_read<0>();
              __syncwarp();
            }
            fence_proxy_async_smem();
            asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
            const uint32_t issue = (q == static_cast<int>(ei & 3u)) ? el : 0u;
            if (q == static_cast<int>(ei & 3u) && !AV2V_DBG(64)) {  // bring-up: bit6 = no TMA stores
              // operands made provably warp-uniform (shfl) so that the store is issued from uniform registers
              const uint32_t u_src = __shfl_sync(0xffffffffu, obuf, 0);
              const int u_c0 = __shfl_sync(0xffffffffu, col0, 0), u_c1 = __shfl_sync(0xffffffffu, m_tile * BM, 0);
              const int u_x = __shfl_sync(0xffffffffu, o_x, 0), u_y = __shfl_sync(0xffffffffu, o_y, 0), u_n = __shfl_sync(0xffffffffu, o_n, 0);
              if (p.up2)  // tile pixel (n, i, j) -> output pixel (n, 2 i + py, 2 j + px)
                tma_store_5d_w(issue, &tmap_o, u_src, u_c0 + p.tap_ox * p.N, u_x, p.tap_oy, u_y, u_n);
              else if (p.block_store)
                tma_store_5d_w(issue, &tmap_o, u_src, u_c0, u_x, u_y, u_n, __shfl_sync(0xffffffffu, s, 0));
              else
                tma_store_3d_w(issue, &tmap_o, u_src, u_c0, u_c1, __shfl_sync(0xffffffffu, s, 0));
              if (issue) tma_store_commit();
              __syncwarp();
            }
            if (has_res) prefetch_one(issue);
          }
        }
      }
      if (el) tma_store_wait0();
    } else if (warp < 8)
    for (int ti = 0, m_tile = 0, n_tile = 0; sched.get(ti, m_tile, n_tile); ++ti, ++it) {
      const uint32_t acc = it & 1u;
      const uint32_t acc_phase = (it >> 1) & 1u;

      long long grow;
      bool valid;
      if (p.mode == AV2V_A_TCONV3) {  // (conv3x3 tiles always take the staged epilogue through the block map)
        const int b = m_tile / p.tiles_per_clip;
        const int r0 = (m_tile - b * p.tiles_per_clip) * BM;
        valid = (r0 + r) < p.rows_per_clip;
        grow = static_cast<long long>(b) * p.rows_per_clip + r0 + r;
      } else {
        grow = static_cast<long long>(m_tile) * BM + r;
        valid = grow < p.M;
      }
      const long long rb_row = (p.rowbias != nullptr && valid) ? grow / p.rows_per_rowbias : 0;

      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + acc * BN + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        const int col0 = n_tile * BN + c * 32;
        if (col0 >= p.N) break;  // warp-uniform
        uint32_t v[32];
        tmem_ld32(t_row + c * 32, v);
        tmem_ld_wait();
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
        if (p.bias != nullptr) {
          const uint4* b4 = reinterpret_cast<const uint4*>(p.bias + col0);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            if (col0 + j4 * 8 < p.N) {
              const uint4 bv = __ldg(b4 + j4);
              const __half2* h2 = reinterpret_cast<const __half2*>(&bv);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 t = __half22float2(h2[e]);
                f[j4 * 8 + 2 * e] += t.x;
                f[j4 * 8 + 2 * e + 1] += t.y;
              }
            }
          }
        }
        if (p.rowbias != nullptr && valid) {
          const uint4* b4 = reinterpret_cast<const uint4*>(p.rowbias + rb_row * p.N + col0);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            if (col0 + j4 * 8 < p.N) {
              const uint4 bv = __ldg(b4 + j4);
              const __half2* h2 = reinterpret_cast<const __half2*>(&bv);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 t = __half22float2(h2[e]);
                f[j4 * 8 + 2 * e] += t.x;
                f[j4 * 8 + 2 * e + 1] += t.y;
              }
            }
          }
        }
        if (valid) {
          for (int s = 0; s < p.n_slots; ++s) {
            const long long off = s * p.slot_stride + grow * p.ldo + col0;
            uint4* o4 = reinterpret_cast<uint4*>(p.out + off);
            const uint4* r4 = p.residual ? reinterpret_cast<const uint4*>(p.residual + off) : nullptr;
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              if (col0 + j4 * 8 < p.N) {
                float g[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) g[e] = f[j4 * 8 + e];
                if (r4 != nullptr) {
                  const uint4 rv = r4[j4];
                  const __half2* h2 = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float2 t = __half22float2(h2[e]);
                    g[2 * e] += t.x;
                    g[2 * e + 1] += t.y;
                  }
                }
                uint4 ov;
                ov.x = pack_half2(g[0], g[1]);
                ov.y = pack_half2(g[2], g[3]);
                ov.z = pack_half2(g[4], g[5]);
                ov.w = pack_half2(g[6], g[7]);
                o4[j4] = ov;
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (p.mc2) cluster_sync();  // no CTA may exit while its peer can still multicast into it / arrive on its barriers
  if (warp == 2) {
    tc_fence_after();
    if constexpr (kPair) tmem_dealloc_cg2<Cfg::kTmemCols>(tmem_base);
    else tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

template <int BN, bool kPair, int kEpi>
int launch_gemm_impl(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, const CUtensorMap& tr,
                     const CUtensorMap& tbh, const CUtensorMap& ta2, const GemmKParams& p, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, kPair, kEpi>;
  static bool attr_set = false;
  if (!attr_set) {
    AV2V_CHECK_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<BN, kPair, kEpi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg::kSmemBytes));
    attr_set = true;
  }
  const int sms = sm_count_cached();
  if constexpr (!kPair) {
    const int tiles = p.m_tiles * p.n_tiles;
    const int grid = tiles < sms ? tiles : sms;
    gemm_tcgen05_kernel<BN, false, kEpi><<<grid, kThreads, Cfg::kSmemBytes, stream>>>(ta, tb, to, tr, tbh, ta2, p);
  } else {
    const int pairs = ((p.m_tiles + 1) / 2) * p.n_tiles;
    const int clusters = pairs < sms / 2 ? pairs : sms / 2;
    AV2V_CHECK_CUDA(launch_ex(gemm_tcgen05_kernel<BN, true, kEpi>, dim3(2 * clusters), dim3(kThreads), Cfg::kSmemBytes, stream, 2,
                              ta, tb, to, tr, tbh, ta2, p));
  }
  AV2V_CHECK_CUDA(cudaGetLastError());
  return AV2V_OK;
}

template <int BN>
int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, const CUtensorMap& tr,
                const CUtensorMap& tbh, const CUtensorMap& ta2, const GemmKParams& p, cudaStream_t stream) {
  // lean epilogue flavours: staged stores, one output slot, no up-sampling store
#ifdef AV2V_GEMM_BRINGUP
  const bool lean = p.fast_epi && p.n_slots == 1 && !p.up2 && !(p.debug & 512);
#else
  const bool lean = p.fast_epi && p.n_slots == 1 && !p.up2;
#endif
  const int epi = !lean ? E_GENERIC : p.geglu ? E_GEGLU : (p.residual != nullptr ? E_RES : E_PLAIN) | (p.block_store ? E_BLOCK : 0);
#define AV2V_LAUNCH(E)                                                                              \
  return p.mc2 == 2 ? launch_gemm_impl<BN, true, E>(ta, tb, to, tr, tbh, ta2, p, stream)           \
                    : launch_gemm_impl<BN, false, E>(ta, tb, to, tr, tbh, ta2, p, stream)
  switch (epi) {
    case E_PLAIN: AV2V_LAUNCH(E_PLAIN);
    case E_RES: AV2V_LAUNCH(E_RES);
    case E_GEGLU: AV2V_LAUNCH(E_GEGLU);
    case E_PLAIN | E_BLOCK: AV2V_LAUNCH(E_PLAIN | E_BLOCK);
    case E_RES | E_BLOCK: AV2V_LAUNCH(E_RES | E_BLOCK);
    default: AV2V_LAUNCH(E_GENERIC);
  }
#undef AV2V_LAUNCH
}

}  // namespace
}  // namespace av2v

using namespace av2v;

extern "C" int av2v_gemm_debug_timers(unsigned long long* out16) {
  AV2V_CHECK_CUDA(cudaMemcpyFromSymbol(out16, av2v::g_gemm_timers, sizeof(unsigned long long) * 16));
  return AV2V_OK;
}

// Validation and tile plan of a CONV3X3 call (host only).  Frames of at most 64 pixels: several whole frames per tile.  Widths
// that divide 128: whole image rows.  Any other width: the block of box_w x box_h pixels (box_w in {128, 64, 32, 16, 8, W_out},
// box_h = 128 / box_w) with the fewest tiles per frame, the wider block on a tie — 128-pixel row segments for widths that are
// multiples of 128, e.g. 32 x 4 at 160 x 88 and 8 x 16 at 88 x 160 (both fill every tile).
extern "C" int av2v_conv3x3_plan(const av2v_gemm_args* a, av2v_conv_plan* out) {
  AV2V_REQUIRE(a != nullptr && out != nullptr, AV2V_EINVAL, "conv3x3 plan: null args");
  AV2V_REQUIRE(a->mode == AV2V_A_CONV3X3, AV2V_EINVAL, "conv3x3 plan: mode must be AV2V_A_CONV3X3 (got %d)", a->mode);
  AV2V_REQUIRE(a->NF > 0 && a->H > 0 && a->W > 0 && a->Cin > 0, AV2V_EINVAL, "gemm/conv3x3: bad geometry");
  AV2V_REQUIRE(a->Cin % BK == 0, AV2V_ENOSUP, "gemm/conv3x3: Cin must be a multiple of 64 (got %d)", a->Cin);
  const int up = a->up2_phase;  // 0: plain conv; 1..4: phase (py, px) = ((up-1) >> 1, (up-1) & 1) of nearest-up x 2 + conv 3 x 3
  AV2V_REQUIRE(up >= 0 && up <= 4, AV2V_EINVAL, "gemm/conv3x3: up2_phase must be 0..4 (got %d)", up);
  AV2V_REQUIRE(a->K == (up ? 4 : 9) * a->Cin, AV2V_EINVAL, "gemm/conv3x3: K must equal 9*Cin (4*Cin for an up2 phase)");
  AV2V_REQUIRE(!up || (a->stride <= 1 && !a->rowbias && !a->residual && a->n_slots == 1), AV2V_EINVAL,
               "gemm/conv3x3: an up2 phase takes bias only (no stride, rowbias, residual, slots)");
  // the up2 store map merges (px, channel) into one dimension of 2 N contiguous channels; 32-column chunks must not straddle px
  AV2V_REQUIRE(!up || (a->ldo == a->N && a->N % 32 == 0), AV2V_ENOSUP,
               "gemm/conv3x3 up2: needs a contiguous output (ldo == N) and N a multiple of 32 (N = %d, ldo = %d)", a->N, a->ldo);
  const int stride = a->stride == 0 ? 1 : a->stride;
  AV2V_REQUIRE(stride == 1 || stride == 2, AV2V_ENOSUP, "gemm/conv3x3: stride must be 1 or 2 (got %d)", a->stride);
  AV2V_REQUIRE(a->H % stride == 0 && a->W % stride == 0, AV2V_ENOSUP, "gemm/conv3x3: H, W must be multiples of the stride");
  const int chan = a->a_channels == 0 ? a->Cin : a->a_channels;
  AV2V_REQUIRE(chan > 0 && chan <= a->Cin && chan % 8 == 0, AV2V_EINVAL, "gemm/conv3x3: a_channels must be a multiple of 8 in (0, Cin]");
  const int Ho = a->H / stride, Wo = a->W / stride;  // output geometry: the plan tiles the OUTPUT pixels
  AV2V_REQUIRE(static_cast<long long>(a->NF) * Ho * Wo == a->M, AV2V_EINVAL, "gemm/conv3x3: M != NF*(H/stride)*(W/stride)");
  const long long HW = static_cast<long long>(Ho) * Wo;
  av2v_conv_plan pl{};
  if (2 * HW <= BM) {  // several whole frames per tile
    pl.box_w = Wo;
    pl.box_h = Ho;
    pl.frames_per_tile = static_cast<int>(BM / HW);
    pl.tiles_per_frame = 1;
    pl.m_tiles = (a->NF + pl.frames_per_tile - 1) / pl.frames_per_tile;
  } else {
    pl.frames_per_tile = 1;
    if (Wo <= BM && BM % Wo == 0) {  // whole image rows
      pl.box_w = Wo;
      pl.box_h = BM / Wo < Ho ? BM / Wo : Ho;
    } else {
      const int cands[6] = {BM, 64, 32, 16, 8, Wo < BM ? Wo : 0};
      long long best = -1;
      for (int i = 0; i < 6; ++i) {
        const int bw = cands[i];
        if (bw == 0) continue;
        const int bh = BM / bw < Ho ? BM / bw : Ho;
        const long long tiles = static_cast<long long>((Wo + bw - 1) / bw) * ((Ho + bh - 1) / bh);
        if (best < 0 || tiles < best || (tiles == best && bw > pl.box_w)) {  // fewest tiles, then the wider block
          best = tiles;
          pl.box_w = bw;
          pl.box_h = bh;
        }
      }
    }
    pl.tiles_per_frame = ((Wo + pl.box_w - 1) / pl.box_w) * ((Ho + pl.box_h - 1) / pl.box_h);
    pl.m_tiles = a->NF * pl.tiles_per_frame;
  }
  *out = pl;
  return AV2V_OK;
}

extern "C" int av2v_gemm_f16(const av2v_gemm_args* a, av2v_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  AV2V_REQUIRE(a != nullptr, AV2V_EINVAL, "gemm: null args");
  AV2V_REQUIRE(a->a && a->w && a->out, AV2V_EINVAL, "gemm: null a/w/out pointer");
  AV2V_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0, AV2V_EINVAL, "gemm: M,N,K must be positive (%d,%d,%d)", a->M, a->N,
               a->K);
  AV2V_REQUIRE(a->N % 8 == 0 && a->K % 8 == 0, AV2V_EINVAL, "gemm: N and K must be multiples of 8 (%d,%d)", a->N,
               a->K);
  AV2V_REQUIRE((a->geglu || a->ldo >= a->N) && a->ldo % 8 == 0, AV2V_EINVAL,
               "gemm: ldo must be >= N and a multiple of 8");
  AV2V_REQUIRE(a->n_slots >= 1, AV2V_EINVAL, "gemm: n_slots must be >= 1");
  AV2V_REQUIRE(a->n_slots == 1 || a->slot_stride % 8 == 0, AV2V_EALIGN, "gemm: slot_stride must be a multiple of 8");
  AV2V_REQUIRE(aligned16(a->a) && aligned16(a->w) && aligned16(a->out), AV2V_EALIGN,
               "gemm: a/w/out must be 16-byte aligned");
  AV2V_REQUIRE(!a->bias || aligned16(a->bias), AV2V_EALIGN, "gemm: bias must be 16-byte aligned");
  AV2V_REQUIRE(!a->rowbias || (aligned16(a->rowbias) && a->rows_per_rowbias > 0), AV2V_EALIGN,
               "gemm: rowbias must be 16-byte aligned with rows_per_rowbias > 0");
  AV2V_REQUIRE(!a->residual || aligned16(a->residual), AV2V_EALIGN, "gemm: residual must be 16-byte aligned");

  GemmKParams p{};
  p.x_tiles = 1;
  p.M = a->M;
  p.N = a->N;
  p.mode = a->mode;
  p.bias = static_cast<const __half*>(a->bias);
  p.rowbias = static_cast<const __half*>(a->rowbias);
  p.rows_per_rowbias = a->rows_per_rowbias;
  p.residual = static_cast<const __half*>(a->residual);
  p.out = static_cast<__half*>(a->out);
  p.ldo = a->ldo;
  p.n_slots = a->n_slots;
  p.slot_stride = a->slot_stride;
  p.geglu = a->geglu ? 1 : 0;
  {
#ifdef AV2V_GEMM_BRINGUP  // tools/build_dbg.sh only: the shipped library reads no environment
    const char* e = getenv("AV2V_GEMM_DEBUG");
    p.debug = e ? atoi(e) : 0;
#else
    p.debug = 0;
#endif
  }
  if (a->geglu) {
    AV2V_REQUIRE(a->mode == AV2V_A_LINEAR, AV2V_EINVAL, "gemm/geglu: LINEAR mode only");
    AV2V_REQUIRE(a->N % 64 == 0, AV2V_EINVAL, "gemm/geglu: N must be a multiple of 64 (got %d)", a->N);
    AV2V_REQUIRE(!a->residual && !a->rowbias && a->n_slots == 1, AV2V_EINVAL, "gemm/geglu: no residual / rowbias / slots");
    AV2V_REQUIRE(a->ldo >= a->N / 2, AV2V_EINVAL, "gemm/geglu: ldo must be >= N/2");
  }

  CUtensorMap ta, tb, ta2;
  memset(&ta2, 0, sizeof(ta2));
  int rc;
  p.stride = 1;
  p.taps_w = 3;
  if (a->mode == AV2V_A_LINEAR) {
    AV2V_REQUIRE((a->a2 != nullptr || a->lda >= a->K) && a->lda % 8 == 0, AV2V_EINVAL, "gemm: lda must be >= K and a multiple of 8");
    const uint64_t dims[2] = {static_cast<uint64_t>(a->K), static_cast<uint64_t>(a->M)};
    const uint64_t str[1] = {static_cast<uint64_t>(a->lda) * 2};
    const uint32_t box[2] = {BK, BM};
    if (a->a2 == nullptr && (rc = make_tmap_f16(&ta, a->a, 2, dims, str, box)) != AV2V_OK) return rc;
    p.num_kb = (a->K + BK - 1) / BK;
    p.kb_per_tap = p.num_kb;
    p.kb_split = p.num_kb;
    p.m_tiles = (a->M + BM - 1) / BM;
    p.a_box_bytes = BM * BK * 2;
    if (a->a2 != nullptr) {  // two-source K loop: A = [a | a2]
      AV2V_REQUIRE(a->k_split > 0 && a->k_split < a->K && a->k_split % BK == 0, AV2V_EINVAL,
                   "gemm: k_split must be a multiple of 64 inside (0, K) (got %d, K = %d)", a->k_split, a->K);
      AV2V_REQUIRE(a->lda >= a->k_split && a->lda2 >= a->K - a->k_split && a->lda2 % 8 == 0 && aligned16(a->a2), AV2V_EINVAL,
                   "gemm: a / a2 row strides must cover their column ranges (multiples of 8), a2 16-byte aligned");
      const uint64_t dims1[2] = {static_cast<uint64_t>(a->k_split), static_cast<uint64_t>(a->M)};
      if ((rc = make_tmap_f16(&ta, a->a, 2, dims1, str, box)) != AV2V_OK) return rc;  // clip the first source at k_split
      const uint64_t dims2[2] = {static_cast<uint64_t>(a->K - a->k_split), static_cast<uint64_t>(a->M)};
      const uint64_t str2[1] = {static_cast<uint64_t>(a->lda2) * 2};
      if ((rc = make_tmap_f16(&ta2, a->a2, 2, dims2, str2, box)) != AV2V_OK) return rc;
      p.kb_split = a->k_split / BK;
    }
  } else if (a->mode == AV2V_A_CONV3X3) {
    av2v_conv_plan pl;
    if ((rc = av2v_conv3x3_plan(a, &pl)) != AV2V_OK) return rc;
    const int up = a->up2_phase;
    if (up) {
      p.taps_w = 2;
      p.tap_oy = (up - 1) >> 1;
      p.tap_ox = (up - 1) & 1;
      p.up2 = 1;
    }
    const int stride = a->stride == 0 ? 1 : a->stride;
    const int chan = a->a_channels == 0 ? a->Cin : a->a_channels;  // channels really present (the rest of the K block reads zeros)
    const int Ho = a->H / stride, Wo = a->W / stride;
    p.stride = stride;
    p.H = Ho;
    p.W = Wo;
    p.HW = Ho * Wo;
    p.NF = a->NF;
    p.box_w = pl.box_w;
    p.box_h = pl.box_h;
    p.frames_per_tile = pl.frames_per_tile;
    p.tiles_per_frame = pl.tiles_per_frame;
    p.x_tiles = (Wo + pl.box_w - 1) / pl.box_w;
    p.m_tiles = pl.m_tiles;
    // the tensor map describes the INPUT image; with stride 2 the box spans 2x the output pixels and TMA picks every second one
    const uint64_t dims[4] = {static_cast<uint64_t>(chan), static_cast<uint64_t>(a->W),
                              static_cast<uint64_t>(a->H), static_cast<uint64_t>(a->NF)};
    const uint64_t str[3] = {static_cast<uint64_t>(chan) * 2, static_cast<uint64_t>(chan) * 2 * a->W,
                             static_cast<uint64_t>(chan) * 2 * a->W * a->H};
    const uint32_t box[4] = {BK, static_cast<uint32_t>(pl.box_w * stride), static_cast<uint32_t>(pl.box_h * stride),
                             static_cast<uint32_t>(pl.frames_per_tile)};
    const uint32_t estr[4] = {1, static_cast<uint32_t>(stride), static_cast<uint32_t>(stride), 1};
    if ((rc = make_tmap_f16(&ta, a->a, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, estr)) != AV2V_OK) return rc;
    p.kb_per_tap = a->Cin / BK;
    p.num_kb = (up ? 4 : 9) * p.kb_per_tap;
    p.kb_split = p.num_kb;
    p.a_box_bytes = static_cast<uint32_t>(BK * 2 * pl.box_w * pl.box_h * pl.frames_per_tile);  // < 128 rows: the rest is never stored
  } else if (a->mode == AV2V_A_TCONV3) {
    AV2V_REQUIRE(a->B > 0 && a->rows_per_clip > 0 && a->HW > 0 && a->Cin > 0, AV2V_EINVAL, "gemm/tconv3: bad geometry");
    AV2V_REQUIRE(a->Cin % BK == 0, AV2V_ENOSUP, "gemm/tconv3: Cin must be a multiple of 64 (got %d)", a->Cin);
    AV2V_REQUIRE(a->K == 3 * a->Cin, AV2V_EINVAL, "gemm/tconv3: K must equal 3*Cin");
    AV2V_REQUIRE(a->rows_per_clip % a->HW == 0, AV2V_EINVAL, "gemm/tconv3: rows_per_clip must be F*HW");
    AV2V_REQUIRE(static_cast<long long>(a->B) * a->rows_per_clip == a->M, AV2V_EINVAL, "gemm/tconv3: M != B*F*HW");
    p.HW = a->HW;
    p.rows_per_clip = a->rows_per_clip;
    p.tiles_per_clip = (a->rows_per_clip + BM - 1) / BM;  // a ragged last tile is zero-filled by TMA and masked on store
    p.m_tiles = a->B * p.tiles_per_clip;
    const uint64_t dims[3] = {static_cast<uint64_t>(a->Cin), static_cast<uint64_t>(a->rows_per_clip),
                              static_cast<uint64_t>(a->B)};
    const uint64_t str[2] = {static_cast<uint64_t>(a->Cin) * 2,
                             static_cast<uint64_t>(a->Cin) * 2 * static_cast<uint64_t>(a->rows_per_clip)};
    const uint32_t box[3] = {BK, BM, 1};
    if ((rc = make_tmap_f16(&ta, a->a, 3, dims, str, box)) != AV2V_OK) return rc;
    p.kb_per_tap = a->Cin / BK;
    p.num_kb = 3 * p.kb_per_tap;
    p.kb_split = p.num_kb;
    p.a_box_bytes = BM * BK * 2;
  } else {
    return fail(AV2V_EINVAL, "gemm: unknown A mode %d", a->mode);
  }

  // tile-N choice: every channel width of I2VGen-XL is a multiple of 320 = 2*160, the FF widths of 256.  Among the
  // widths that divide N pick the one with the least (waves x per-tile cost) on this many SMs.
  int bn = 0;
  {
    const int cands[4] = {256, 160, 128, 64};
    const int sms = sm_count_cached();
    long long best = -1;
    for (int i = 0; i < 4; ++i) {
      const int c = cands[i];
      if (a->N % c != 0) continue;
      if (a->geglu && (c / 32) % 2 != 0) continue;  // (h, gate) chunk pairs must not straddle tiles
      const long long tiles = static_cast<long long>(p.m_tiles) * (a->N / c);
      const long long waves = (tiles + sms - 1) / sms;
      // per-tile time ~ max(tensor pipe: c, L2->smem operand traffic: 0.8 * (128 + c)) + fixed overhead
      const long long l2 = (128 + c) * 4 / 5;
      const long long cost = waves * ((c > l2 ? c : l2) + 32);
      if (best < 0 || cost < best) {
        best = cost;
        bn = c;
      }
    }
    if (bn == 0) bn = (a->N > 256) ? 128 : 64;  // ragged N: partial last tile, masked by the epilogue / TMA clipping
  }
  p.n_tiles = (a->N + bn - 1) / bn;
  {
    const uint64_t dims[2] = {static_cast<uint64_t>(a->K), static_cast<uint64_t>(a->N)};
    const uint64_t str[1] = {static_cast<uint64_t>(a->K) * 2};
    const uint32_t box[2] = {BK, static_cast<uint32_t>(bn)};
    if ((rc = make_tmap_f16(&tb, a->w, 2, dims, str, box)) != AV2V_OK) return rc;
  }
  // staged TMA-store epilogue whenever a tile's 128 rows are contiguous rows of the output
  CUtensorMap to, tr;
  memset(&to, 0, sizeof(to));
  memset(&tr, 0, sizeof(tr));
  bool contig = true;
  if (a->mode == AV2V_A_CONV3X3) {  // p.W / p.H = output geometry
    // whole row segments / rows / frames that fill the tile and tile the image exactly: output rows m_tile*128 ... (3-D map)
    if (p.frames_per_tile > 1) contig = (p.frames_per_tile * p.HW == BM);
    else if (p.box_w * p.box_h != BM) contig = false;
    else if (p.box_w == p.W) contig = (p.H % p.box_h == 0);
    else contig = (p.box_h == 1 && p.W % p.box_w == 0);
    p.block_store = (contig || p.up2) ? 0 : 1;
  } else if (a->mode == AV2V_A_TCONV3) {
    contig = (a->rows_per_clip % BM == 0);
  }
  p.fast_epi = (contig || a->mode == AV2V_A_CONV3X3) ? 1 : 0;
  p.o_box_bytes = p.block_store ? static_cast<uint32_t>(64 * p.box_w * p.box_h * p.frames_per_tile) : static_cast<uint32_t>(kEpiBufBytes);
  if (p.up2) {
    // output = [NF][2H][2W][N] (ldo == N); tile pixel (n, i, j) goes to (n, 2i + py, 2j + px): dims (px*N + c, j, py, i, n), so that
    // the store box {32, box_w, 1, box_h, frames} is clipped at the right / bottom edge of the frame
    const uint64_t ld = static_cast<uint64_t>(a->ldo) * 2;
    const uint64_t dims[5] = {2 * static_cast<uint64_t>(a->N), static_cast<uint64_t>(p.W), 2, static_cast<uint64_t>(p.H),
                              static_cast<uint64_t>(p.NF)};
    const uint64_t str[4] = {2 * ld, 2 * static_cast<uint64_t>(p.W) * ld, 4 * static_cast<uint64_t>(p.W) * ld,
                             4 * static_cast<uint64_t>(p.HW) * ld};
    const uint32_t box[5] = {32, static_cast<uint32_t>(p.box_w), 1, static_cast<uint32_t>(p.box_h), static_cast<uint32_t>(p.frames_per_tile)};
    if ((rc = make_tmap_f16(&to, a->out, 5, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B)) != AV2V_OK) return rc;
  } else if (p.block_store) {
    // [n_slots][NF][H][W][ldo] with box {32, box_w, box_h, frames, 1}: the out-of-image part of an edge block is not written
    // (stores) or reads as zeros (residual loads)
    const uint64_t ld = static_cast<uint64_t>(a->ldo) * 2;
    const uint64_t slot_b = (a->n_slots > 1) ? static_cast<uint64_t>(a->slot_stride) * 2 : ld * static_cast<uint64_t>(a->M);
    const uint64_t dims[5] = {static_cast<uint64_t>(a->N), static_cast<uint64_t>(p.W), static_cast<uint64_t>(p.H),
                              static_cast<uint64_t>(p.NF), static_cast<uint64_t>(a->n_slots)};
    const uint64_t str[4] = {ld, ld * p.W, ld * static_cast<uint64_t>(p.HW), slot_b};
    const uint32_t box[5] = {32, static_cast<uint32_t>(p.box_w), static_cast<uint32_t>(p.box_h), static_cast<uint32_t>(p.frames_per_tile), 1};
    if ((rc = make_tmap_f16(&to, a->out, 5, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B)) != AV2V_OK) return rc;
    if (a->residual && (rc = make_tmap_f16(&tr, a->residual, 5, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B)) != AV2V_OK)
      return rc;
  } else if (p.fast_epi) {
    const uint64_t slot_b = (a->n_slots > 1) ? static_cast<uint64_t>(a->slot_stride) * 2
                                             : static_cast<uint64_t>(a->ldo) * 2 * static_cast<uint64_t>(a->M);
    const uint64_t dims[3] = {static_cast<uint64_t>(a->geglu ? a->N / 2 : a->N), static_cast<uint64_t>(a->M),
                              static_cast<uint64_t>(a->n_slots)};
    const uint64_t str[2] = {static_cast<uint64_t>(a->ldo) * 2, slot_b};
    const uint32_t box[3] = {32, BM, 1};
    if ((rc = make_tmap_f16(&to, a->out, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B)) != AV2V_OK) return rc;
    if (a->residual && (rc = make_tmap_f16(&tr, a->residual, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B)) != AV2V_OK)
      return rc;
  }
  // pair mode: clusters of 2 CTAs on M-adjacent tiles share each W tile through TMA multicast
  CUtensorMap tbh;
  memset(&tbh, 0, sizeof(tbh));
  {
    // the cta_group::2 pair wins once the K loop is long enough to hide the pair's coupled accumulator hand-over (measured
    // on B200, profiles/r01_gemm_pair_mode.txt: +4 % at K = 640 ... +15 % at K >= 1280, -22 % at K = 320)
    p.mc2 = (p.num_kb >= 10 && p.fast_epi && p.m_tiles >= 2 && a->N % bn == 0) ? 2 : 0;
#ifdef AV2V_GEMM_BRINGUP
    if ((p.debug & 128) && p.fast_epi && p.m_tiles >= 2 && a->N % bn == 0) p.mc2 = 2;
    if (p.debug & 256) p.mc2 = 0;
#endif
  }
  if (p.mc2) {
    const uint64_t dims[2] = {static_cast<uint64_t>(a->K), static_cast<uint64_t>(a->N)};
    const uint64_t str[1] = {static_cast<uint64_t>(a->K) * 2};
    const uint32_t box[2] = {BK, static_cast<uint32_t>(bn / 2)};
    if ((rc = make_tmap_f16(&tbh, a->w, 2, dims, str, box)) != AV2V_OK) return rc;
  }
  switch (bn) {
    case 256: return launch_gemm<256>(ta, tb, to, tr, tbh, ta2, p, stream);
    case 160: return launch_gemm<160>(ta, tb, to, tr, tbh, ta2, p, stream);
    case 128: return launch_gemm<128>(ta, tb, to, tr, tbh, ta2, p, stream);
    default: return launch_gemm<64>(ta, tb, to, tr, tbh, ta2, p, stream);
  }
}
