// drsim_actor.cuh -- MA-PPO actor on the observation rows, fused with the categorical draw
// (SURVEY 8f-2; reference: agents/trainables/network.py:14-35 `Actor`, mappo.py:83-97 `select_actions`).
//
// The reference runs N batch-1 forwards of a [D -> h1 -> h2 -> 2] ReLU MLP per step on the CPU.  Here a
// persistent CTA takes 128 observation rows at a time (row t = TMEM lane t, UMMA M = 128); the hidden layers are
// tcgen05 GEMMs issued by one thread per CTA (cta_group::1) into fp32 accumulators in tensor memory, and the
// softmax and the Philox draw keyed (replica, house, step) -> action byte + probability of the draw follow in
// the same kernel.  Three precisions:
//   0 "tf32"    k_actor2: one TF32 pass per layer, the output layer a third GEMM;
//   1 "tf32x3"  k_actor3<SplitTf32x3>: three TF32 passes per product on hi / lo halves (the default);
//   2 "f16x3"   k_actor3<SplitF16x3>: three fp16 passes per product with per-neuron power-of-two weight scales.
// A small pack kernel before each launch (k_actor_pack, k_actor_pack3x, k_actor_pack3h) converts the weights
// once into the shared-memory image the actor kernel fetches; only the observation rows move per tile.
// Operands sit in shared memory in the canonical no-swizzle K-major layout of the UMMA shared-memory
// descriptor: 8-row x 16-byte core matrices, SBO = 128 B between 8-row groups, LBO = (rows / 8) * 128 B
// between 16-byte K chunks.
#pragma once

#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "drsim_device.cuh"

namespace drsim {

constexpr int kActRows = 128;       // rows per tile == UMMA M == TMEM lanes
constexpr uint32_t PURPOSE_POLICY = 6;

struct ActorArgs {
  const void *obs;         // [rows][D] float, or __nv_bfloat16 (k_actor3<S, PRE, __nv_bfloat16>)
  const unsigned char *image;   // packed weight operands (k_actor_pack, k_actor_pack3x, k_actor_pack3h)
  const float *w1, *b1;    // [h1][D], [h1]
  const float *w2, *b2;    // [h2][h1], [h2]
  const float *w3, *b3;    // [2][h2], [2]
  uint8_t *actions;        // [rows]      1 = turn the HVAC on
  float *prob;             // [rows] or NULL: probability of the action that was drawn
  float *prob_on;          // [rows] or NULL: probability of action 1
  long long rows;          // R * Ns (padding slots included; they get action 0)
  int Ns, N, D, h1, h2;
  int K1, N1, K2, N2, K3;  // padded: K multiple of UMMA_K (8 for tf32, 16 for f16), N multiple of 16 (K3: k_actor2's output layer)
  int off_w1, off_w2, off_a1, off_a2, off_vec, off_bar, smem_bytes;   // off_a2, off_vec: k_actor2
  unsigned long long *dbg; // DRSIM_ACTOR_DBG: clock64 stamps [tile < 8][role][16] of CTA 0 (k_actor3)
  int off_w3, w_bytes;     // k_actor3: the fp32 output layer in the image; size of one (hi, d or lo) weight block
  unsigned long long seed;
  long long step, rep_offset;
  int off_sc;              // k_actor3<SplitF16x3>: 2^-s of each layer-1 output column [N1] in the image
  int *range_err;          // k_actor3<SplitF16x3>: mapped host flag, set when a live row's operand overflows fp16
};

// byte offset of element (row, k) of a K-major fp32 operand with `rows` rows in the canonical layout
DRSIM_HD int umma_kmajor_off(int rows, int row, int k) {
  return (k >> 2) * (rows >> 3) * 128 + (row >> 3) * 128 + (row & 7) * 16 + (k & 3) * 4;
}

#if defined(__CUDACC__)
DRSIM_D uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  // cute::UMMA::SmemDescriptor: start >> 4 [0,14), LBO >> 4 [16,30), SBO >> 4 [32,46), version = 1 [46,48),
  // base_offset = 0, lbo_mode = 0, layout_type = SWIZZLE_NONE (0) [61,64)
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fffu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
DRSIM_D uint32_t umma_instr_desc_tf32(int M, int N) {
  // cute::UMMA::InstrDescriptor: c_format F32 = 1 [4,6), a/b_format TF32 = 2 [7,10) [10,13), K-major A and B,
  // n_dim = N >> 3 [17,23), m_dim = M >> 4 [24,29)
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
DRSIM_D void umma_tf32_ss(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}
DRSIM_D void umma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(bar))
               : "memory");
}
// round-to-nearest (ties away from zero) TF32: the tensor core would otherwise truncate the 13 low mantissa bits.
// Two integer instructions on the sign-magnitude bit pattern; `cvt.rna.tf32.f32` gives the same value for every
// finite input but compiles to a six-instruction sequence with Inf / NaN handling on sm_100a, which made the
// operand split of k_actor3<SplitTf32x3> ALU-bound (activations and weights are finite).
DRSIM_D float to_tf32(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
DRSIM_D void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
DRSIM_D void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// bounded wait on an mbarrier phase: a wedged tensor pipe must fail the launch, not hang the GPU
DRSIM_D void mbar_wait_bounded(uint64_t *bar, uint32_t parity) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  for (long long spin = 0; spin < 400000000ll; ++spin) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
    if (ok) return;
  }
  asm volatile("trap;");
}

// ------------------------------------------------------------------------------------------------
// k_actor2: the single-pass "tf32" precision:
//   * two tiles in flight per CTA: 512 threads = two groups of 8 warps; group g owns tile slot g (its own
//     observation buffers, TMEM columns, mbarrier and named barrier), so one slot runs its epilogue on the
//     CUDA cores while the other's GEMM occupies the tensor core; the weights are shared;
//   * all THREE layers are tcgen05 GEMMs and the activations never leave tensor memory: each epilogue
//     reads its accumulator row with tcgen05.ld, applies ReLU + TF32 rounding and writes it back IN PLACE
//     with tcgen05.st; the next layer takes its A operand from TMEM (tcgen05.mma [d], [a_tmem], b_desc);
//   * the biases ride in the GEMMs: operand A carries a constant-one column (index D resp. h1, h2: a
//     padding column), the weight matrix the bias in that column, plus one extra output row that
//     regenerates the one for the next layer -- the epilogues are max(x, 0) only;
//   * the 128 observation rows of the slot's NEXT tile (one contiguous run) arrive by a single TMA bulk
//     copy in a raw staging buffer while the current tile computes, and are re-tiled into the canonical
//     operand layout by the slot's threads;
//   * two threads per row: warps w and w + 4 of a slot address the same TMEM lane quadrant and split the
//     row's columns, halving every latency-bound epilogue pass.
// ------------------------------------------------------------------------------------------------
constexpr int kAct2Threads = 512;   // two tile slots x (128 rows x 2 column halves)
constexpr int kAct2TmemCols = 512;
constexpr int kActN3 = 16;   // the 2-wide output layer, padded to the smallest UMMA N for M = 128

DRSIM_D void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}
DRSIM_D void tmem_ld16_issue(uint32_t taddr, uint32_t r[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
DRSIM_D void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
DRSIM_D void tmem_st16(uint32_t taddr, const uint32_t r[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
DRSIM_D void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
DRSIM_D void slot_barrier(int slot) { asm volatile("bar.sync %0, 256;" ::"r"(slot + 1) : "memory"); }

// ReLU + TF32 rounding of the accumulator columns [c_begin, cols) of this thread's TMEM lane, in place,
// 32 columns per load / store round trip (64 per round trip spills at 128 registers and is slower)
DRSIM_D void tmem_relu_inplace(uint32_t lane_addr, int c_begin, int cols) {
  for (int c0 = c_begin; c0 < cols; c0 += 32) {
    uint32_t r[2][16];
    const bool two = c0 + 16 < cols;
    tmem_ld16_issue(lane_addr + (uint32_t)c0, r[0]);
    if (two) tmem_ld16_issue(lane_addr + (uint32_t)(c0 + 16), r[1]);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < 16; ++j) r[0][j] = __float_as_uint(to_tf32(fmaxf(__uint_as_float(r[0][j]), 0.f)));
    tmem_st16(lane_addr + (uint32_t)c0, r[0]);
    if (two) {
#pragma unroll
      for (int j = 0; j < 16; ++j) r[1][j] = __float_as_uint(to_tf32(fmaxf(__uint_as_float(r[1][j]), 0.f)));
      tmem_st16(lane_addr + (uint32_t)(c0 + 16), r[1]);
    }
  }
  tmem_wait_st();
}

// weight matrix [n_out][n_in] (+ bias) -> canonical K-major operand with the bias in column n_in and the
// "one regenerating" row n_out (0 ... 0 1 0 ...), everything else zero; `gen_one` = 0 for the last layer.
// Thread `tid` of `nthreads` (a whole grid in k_actor_pack).
DRSIM_D void pack_weights(unsigned char *dst, const float *w, const float *b, int n_out, int n_in, int Np, int Kp,
                          bool gen_one, int tid, int nthreads) {
  for (int e = tid; e < Np * Kp; e += nthreads) {
    const int n = e / Kp, k = e - n * Kp;
    float v = 0.f;
    if (n < n_out) v = k < n_in ? __ldg(w + (size_t)n * n_in + k) : (k == n_in ? __ldg(b + n) : 0.f);
    else if (n == n_out && gen_one && k == n_in) v = 1.f;
    *reinterpret_cast<float *>(dst + umma_kmajor_off(Np, n, k)) = to_tf32(v);
  }
}

// The three weight operands in their shared-memory image (offsets off_w1 / off_w2 / off_vec of ActorArgs),
// packed ONCE per launch by a small grid instead of once per CTA: k_actor2 then fetches the whole image
// with a single TMA bulk copy (the per-CTA packing cost ~20k scattered loads = 10-15 us of every launch).
__global__ void k_actor_pack(ActorArgs a, unsigned char *image) {
  pdl_trigger();   // k_actor2 may set itself up (TMEM, barriers, constant columns) while this grid runs
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  pack_weights(image + a.off_w1, a.w1, a.b1, a.h1, a.D, a.N1, a.K1, true, tid, nt);
  pack_weights(image + a.off_w2, a.w2, a.b2, a.h2, a.h1, a.N2, a.K2, true, tid, nt);
  pack_weights(image + a.off_vec, a.w3, a.b3, 2, a.h2, kActN3, a.K3, false, tid, nt);
}

__global__ void __launch_bounds__(kAct2Threads, 1) k_actor2(ActorArgs a) {
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char *s_w1 = smem + a.off_w1, *s_w2 = smem + a.off_w2, *s_w3 = smem + a.off_vec;
  uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem + a.off_bar);   // per slot: GEMM1 [0,2), bulk copy [2,4), GEMM2 [4,6), GEMM3 [6,8)
  uint32_t *s_tmem = reinterpret_cast<uint32_t *>(s_bar + 9);
  // slot = tile slot; t = row of the tile (= TMEM lane); part = which half of the row's columns this thread
  // handles (warps w and w + 4 of a slot address the same TMEM lane quadrant)
  const int tid = threadIdx.x, warp = tid >> 5, slot = tid >> 8, t = tid & 127, part = (tid >> 7) & 1;
  const int n_tiles = (int)((a.rows + kActRows - 1) / kActRows);
  const int a1_bytes = kActRows * a.K1 * 4;
  const int k3 = a.K3;
  unsigned char *s_a1 = smem + a.off_a1 + slot * a1_bytes;             // this slot's observation operand (canonical layout)
  const int stage_bytes = (kActRows * a.D * 4 + 127) / 128 * 128;
  float *s_stage = reinterpret_cast<float *>(smem + a.off_a2 + slot * stage_bytes);   // this slot's raw row-major tile
  uint64_t *ldbar = s_bar + 2 + slot;                                  // completion of the slot's bulk copy

  // observation buffers: the constant-one column at k = D, the other padding columns zero
  for (int i = tid; i < 2 * kActRows; i += kAct2Threads) {
    const int b = i / kActRows, row = i - b * kActRows;
    for (int k = a.D; k < a.K1; ++k)
      *reinterpret_cast<float *>(smem + a.off_a1 + b * a1_bytes + umma_kmajor_off(kActRows, row, k)) = k == a.D ? 1.f : 0.f;
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(s_bar)));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(s_bar + 1)));
    for (int i = 2; i < 9; ++i)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(s_bar + i)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(s_tmem)),
                 "r"((uint32_t)kAct2TmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // everything above overlapped the tail of k_actor_pack (programmatic dependent launch); its image and the
  // observation rows of the env step before it are read only from here on
  pdl_wait();
  uint64_t *wbar = s_bar + 8;
  if (tid == 0) {       // the packed weight image: one TMA bulk copy per CTA
    mbar_expect_tx(wbar, (uint32_t)a.off_a1);
    bulk_load_g2s(smem, a.image, (uint32_t)a.off_a1, wbar);
  }
  // this slot's 256 TMEM columns: D1 -> A2 at [0, N1), D2 -> A3 at [N1, N1 + N2), D3 at [N1 + N2, +16)
  const uint32_t tmem = *s_tmem + (uint32_t)(slot * 256);
  const uint32_t idesc1 = umma_instr_desc_tf32(kActRows, a.N1), idesc2 = umma_instr_desc_tf32(kActRows, a.N2),
                 idesc3 = umma_instr_desc_tf32(kActRows, kActN3);
  const uint32_t w1_addr = (uint32_t)__cvta_generic_to_shared(s_w1), w2_addr = (uint32_t)__cvta_generic_to_shared(s_w2),
                 w3_addr = (uint32_t)__cvta_generic_to_shared(s_w3);
  const uint32_t lbo_a = (kActRows / 8) * 128, lbo_w1 = (a.N1 / 8) * 128, lbo_w2 = (a.N2 / 8) * 128, lbo_w3 = (kActN3 / 8) * 128;
  const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);   // this warp's TMEM lane quadrant
  uint64_t *bar = s_bar + slot;

  // The 128 observation rows of a tile are one contiguous run of global memory: a single TMA bulk copy
  // (cp.async.bulk, completion on the slot's mbarrier) brings it into a raw row-major staging buffer one
  // tile ahead; the threads then re-tile it (row t by thread t: 8-byte shared loads, TF32 rounding,
  // conflict-free stores) into the canonical operand layout.  (cp.async pieces straight into the operand
  // layout cost 2.8k cycles per tile: 32 sectors per warp instruction on the global side, or 16-way bank
  // conflicts on the shared side; a tiled TMA cannot address rows of 200 bytes -- pitch not 16-byte aligned.)
  auto fetch = [&](int tile) {
    if (t == 0 && part == 0) {
      const long long row0 = (long long)tile * kActRows;
      const int n_valid = (int)min((long long)kActRows, a.rows - row0);
      const uint32_t bytes = (uint32_t)(n_valid * a.D * 4);     // rows % 4 == 0: a multiple of 16
      mbar_expect_tx(ldbar, bytes);
      bulk_load_g2s(s_stage, static_cast<const float *>(a.obs) + (size_t)row0 * a.D, bytes, ldbar);
    }
  };
  uint32_t ld_phase = 0;
  const int stride = 2 * gridDim.x;
  const uint32_t a1_addr = (uint32_t)__cvta_generic_to_shared(s_a1);
  const uint32_t r1 = tmem, r2 = tmem + (uint32_t)a.N1, r3 = tmem + (uint32_t)(a.N1 + a.N2);   // D1/A2, D2/A3, D3
  uint64_t *bar1 = bar, *bar2 = s_bar + 4 + slot, *bar3 = s_bar + 6 + slot;
  uint32_t ph1 = 0, ph2 = 0, ph3 = 0;
  const bool issuer = t == 0 && part == 0;

  // Software pipeline over the slot's tiles, two tiles in different stages at any time.  The tensor pipe
  // executes the GEMMs of a slot in issue order, which is what makes the TMEM regions safe to recycle:
  //   S1(b): re-tile b, issue GEMM1(b) -> R1          (R1's last reader, GEMM2(a), was issued earlier)
  //   S2(a): wait GEMM2(a), ReLU R2 in place, issue GEMM3(a): R2 -> R3
  //   S3(b): wait GEMM1(b), ReLU R1 in place, issue GEMM2(b): R1 -> R2   (after GEMM3(a), which reads R2)
  //   S4(a): wait GEMM3(a), softmax + draw from R3
  // so every GEMM round trip is covered by the other tile's epilogue work.
  int tile_b = 2 * blockIdx.x + slot, tile_a = -1;
  if (tile_b < n_tiles) fetch(tile_b);
  if (issuer) mbar_wait_bounded(wbar, 0);   // the weight image has landed (async proxy -> tensor core: no proxy fence)
  while (tile_b < n_tiles || tile_a >= 0) {
    const bool has_b = tile_b < n_tiles, has_a = tile_a >= 0;
    if (has_b) {   // ---- S1(b)
      const long long row0 = (long long)tile_b * kActRows;
      const int n_valid = (int)min((long long)kActRows, a.rows - row0);
      mbar_wait_bounded(ldbar, ld_phase);
      ld_phase ^= 1u;
      unsigned char *d = s_a1 + umma_kmajor_off(kActRows, t, 0);
      const float *g = s_stage + (size_t)t * a.D;
      const bool live = t < n_valid;
      const int k_mid = ((a.D / 2) + 1) & ~1, k_lo = part ? k_mid : 0, k_hi = part ? a.D : k_mid;   // this thread's half of the row
      if ((a.D & 1) == 0) {
#pragma unroll 4
        for (int k = k_lo; k < k_hi; k += 2) {
          const float2 v = live ? *reinterpret_cast<const float2 *>(g + k) : make_float2(0.f, 0.f);
          *reinterpret_cast<float2 *>(d + (k >> 2) * (int)((kActRows / 8) * 128) + (k & 3) * 4) = make_float2(to_tf32(v.x), to_tf32(v.y));
        }
      } else {
#pragma unroll 4
        for (int k = k_lo; k < k_hi; ++k)
          *reinterpret_cast<float *>(d + (k >> 2) * (int)((kActRows / 8) * 128) + (k & 3) * 4) = live ? to_tf32(g[k]) : 0.f;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      slot_barrier(slot);   // operand complete, staging buffer drained
      if (tile_b + stride < n_tiles) fetch(tile_b + stride);   // flies during the next stages
      if (issuer) {         // layer 1: D1[128 x N1] = [obs | 1] . [W1 | b1]^T
        tc_fence_after();
        for (int ks = 0; ks < a.K1 / 8; ++ks)
          umma_tf32_ss(r1, umma_smem_desc(a1_addr + ks * 2 * lbo_a, lbo_a, 128),
                       umma_smem_desc(w1_addr + ks * 2 * lbo_w1, lbo_w1, 128), idesc1, ks > 0);
        umma_commit(bar1);
      }
    }
    if (has_a) {   // ---- S2(a)
      mbar_wait_bounded(bar2, ph2);
      ph2 ^= 1u;
      tc_fence_after();
      const int mid = (k3 / 2 + 15) & ~15;                    // A3 = relu(D2) (column h2 = 1)
      tmem_relu_inplace(lane_addr + (uint32_t)a.N1, part ? mid : 0, part ? k3 : mid);
      tc_fence_before();
      slot_barrier(slot);
      if (issuer) {         // layer 3: D3[128 x 16] = A3 . [W3 | b3]^T (two real output columns)
        tc_fence_after();
        for (int ks = 0; ks < k3 / 8; ++ks)
          umma_tf32_ts(r3, r2 + (uint32_t)(ks * 8), umma_smem_desc(w3_addr + ks * 2 * lbo_w3, lbo_w3, 128), idesc3, ks > 0);
        umma_commit(bar3);
      }
    }
    if (has_b) {   // ---- S3(b)
      mbar_wait_bounded(bar1, ph1);
      ph1 ^= 1u;
      tc_fence_after();
      const int mid = (a.K2 / 2 + 15) & ~15;                  // A2 = relu(D1) (column h1 = 1), half the columns per thread
      tmem_relu_inplace(lane_addr, part ? mid : 0, part ? a.K2 : mid);
      tc_fence_before();
      slot_barrier(slot);
      if (issuer) {         // layer 2: D2[128 x N2] = A2 (tensor memory) . [W2 | b2]^T
        tc_fence_after();
        for (int ks = 0; ks < a.K2 / 8; ++ks)
          umma_tf32_ts(r2, r1 + (uint32_t)(ks * 8), umma_smem_desc(w2_addr + ks * 2 * lbo_w2, lbo_w2, 128), idesc2, ks > 0);
        umma_commit(bar2);
      }
    }
    if (has_a) {   // ---- S4(a): softmax + categorical draw
      mbar_wait_bounded(bar3, ph3);
      ph3 ^= 1u;
      tc_fence_after();
      uint32_t lg[16];
      tmem_ld16_issue(lane_addr + (uint32_t)(a.N1 + a.N2), lg);
      tmem_wait_ld();
      const float l0 = __uint_as_float(lg[0]), l1 = __uint_as_float(lg[1]);
      const long long row = (long long)tile_a * kActRows + t;
      if (row < a.rows && part == 0) {
        const long long rr = row / a.Ns;
        const int n = (int)(row - rr * a.Ns);
        uint8_t act = 0;
        float p_draw = 0.f, p1 = 0.f;
        if (n < a.N) {
          const float m = fmaxf(l0, l1);                      // F.softmax(dim=1), network.py:34
          const float e0 = __expf(l0 - m), e1 = __expf(l1 - m);
          const float p0 = e0 / (e0 + e1);
          p1 = 1.f - p0;
          const U4 u = philox4x32_10(a.seed, (uint32_t)(a.rep_offset + rr), (uint32_t)n, (uint32_t)a.step, PURPOSE_POLICY);
          const float uf = (float)(u.x >> 8) * 5.9604644775390625e-8f;   // 24 random bits: [0, 1) exactly
          act = uf < p0 ? 0 : 1;
          p_draw = act ? p1 : p0;
        }
        a.actions[row] = act;
        if (a.prob) a.prob[row] = p_draw;
        if (a.prob_on) a.prob_on[row] = p1;
      }
    }
    tile_a = has_b ? tile_b : -1;
    tile_b += stride;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*s_tmem), "r"((uint32_t)kAct2TmemCols) : "memory");
}

// ------------------------------------------------------------------------------------------------
// k_actor3<S, PRE, O>: the same network at fp32-grade accuracy on the same tensor cores, every product as three passes on
// split operands.  S is the split: SplitTf32x3 ("3xTF32", precision 1, the default) or SplitF16x3 ("f16x3", precision 2,
// below); the roles, the pipeline and the consumers are one code.
//
// 3xTF32: a TF32 operand keeps 10 mantissa bits; splitting every operand into hi = tf32(x) and lo = tf32(x - hi) and
// accumulating  A_hi W_hi + A_lo W_hi + A_hi W_lo  in the fp32 accumulator recovers ~21 bits per product (the
// dropped A_lo W_lo term is 2^-22 relative): probabilities agree with a plain fp32 forward to ~1e-6 instead of
// the 5e-3 of the single-pass kernel.
//
// Structure: ONE CTA per SM, three warp-specialised roles decoupled by mbarriers (no CTA barrier in the loop):
//   * producers (warps 0-7, two threads per row): the observation rows of the NEXT tile wait in registers; they
//     are split into the hi / lo operands of layer 1 in shared memory (16-byte stores, canonical K-major layout),
//     and after GEMM1 the accumulator R1 is turned into the layer-2 operand IN tensor memory: ReLU, hi in place,
//     lo into a second column range L1 (3xTF32).  This pass is pipelined with GEMM2 by 32-column chunks: a chunk's K steps
//     are issued as soon as all rows have published it, so the tensor pipe idles for the first chunk only;
//   * the MMA warp (warp 12, one thread): GEMM1 (shared x shared) and GEMM2 (A from tensor memory), three passes
//     per K step, completion by tcgen05.commit on mbarriers;
//   * consumers (warps 8-11, one thread per row): the layer-2 accumulator R2 is DOUBLE-buffered in tensor memory, so tile i's
//     epilogue overlaps tile i+1's GEMMs: ReLU + the 2-wide output layer in plain fp32 FMAs straight from the
//     tcgen05.ld registers (no third GEMM, no split, no write-back), softmax, Philox draw.
// 3xTF32 tensor memory: R1 | L1 | R2[0] | R2[1] = 2 N1 + 2 N2 <= 512 columns.  Weight image (k_actor_pack3x):
// [w1_hi | w2_hi | w1_lo | w2_lo | w3 fp32 [2][N2] zero-padded, b3[2]], one TMA bulk copy per CTA.
// The kernel is instantiated for the observation widths of S::kPre, so that the unrolled row handling carries no
// predicated-off work.
// ------------------------------------------------------------------------------------------------
constexpr int kAct3Threads = 416;    // 8 producer warps + 4 consumer warps + the MMA warp (13 warps: 128 registers each)
constexpr int kAct3MaxChunks = 5;    // 32-column chunks of the layer-2 operand (N1 <= 144)

DRSIM_D void pack_weights_split(unsigned char *dst_hi, unsigned char *dst_lo, const float *w, const float *b, int n_out, int n_in,
                                int Np, int Kp, bool gen_one, int tid, int nthreads) {
  for (int e = tid; e < Np * Kp; e += nthreads) {
    const int n = e / Kp, k = e - n * Kp;
    float v = 0.f;
    if (n < n_out) v = k < n_in ? __ldg(w + (size_t)n * n_in + k) : (k == n_in ? __ldg(b + n) : 0.f);
    else if (n == n_out && gen_one && k == n_in) v = 1.f;
    const float hi = to_tf32(v);
    const int off = umma_kmajor_off(Np, n, k);
    *reinterpret_cast<float *>(dst_hi + off) = hi;
    *reinterpret_cast<float *>(dst_lo + off) = to_tf32(v - hi);
  }
}

__global__ void k_actor_pack3x(ActorArgs a, unsigned char *image) {
  pdl_trigger();
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  unsigned char *lo = image + a.w_bytes;
  pack_weights_split(image + a.off_w1, lo + a.off_w1, a.w1, a.b1, a.h1, a.D, a.N1, a.K1, true, tid, nt);
  pack_weights_split(image + a.off_w2, lo + a.off_w2, a.w2, a.b2, a.h2, a.h1, a.N2, a.K2, false, tid, nt);
  float *w3 = reinterpret_cast<float *>(image + a.off_w3);     // output layer in plain fp32: [2][N2], then b3
  for (int e = tid; e < 2 * a.N2 + 2; e += nt) {
    const int n = e / a.N2, k = e - n * a.N2;
    w3[e] = e >= 2 * a.N2 ? __ldg(a.b3 + (e - 2 * a.N2)) : (k < a.h2 ? __ldg(a.w3 + (size_t)n * a.h2 + k) : 0.f);
  }
}

// one lane of a converged warp (elect.sync): the form the compiler recognises as a single-thread region
DRSIM_D bool elect_one_lane() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}\n" : "=r"(pred));
  return pred != 0;
}
DRSIM_D void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}
// tcgen05.wait::ld that also DEFINES the registers of the load it completes: nothing computed from them can be
// scheduled above it
DRSIM_D void tmem_wait_ld_dep(uint32_t r[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// phase stamps of CTA 0 (first 8 tiles; producer warp 0, consumer warp 8, MMA warp), read back by drsim_debug_actor_times
#define ACT3_STAMP(slot)                                                                          \
  do {                                                                                            \
    if (a.dbg && blockIdx.x == 0 && it < 8 && (tid & 31) == 0 && (warp == 0 || warp == 8 || warp == 12)) \
      a.dbg[(it * 3 + role) * 16 + (slot)] = (unsigned long long)clock64();                       \
  } while (0)

// ------------------------------------------------------------------------------------------------
// SplitF16x3: the "f16x3" precision -- k_actor3's roles, pipeline and consumers, with all three passes of a product on fp16
// halves (kind::f16, K = 16 per instruction instead of 8: C4's 100 x 100 actor issues 24 MMAs per tile instead of 45).
//
// Split, into ONE fp32 accumulator.  An fp16 value has 11 significant bits like TF32, so hi + lo carries 22 bits:
//   A_hi = fp16(x),  A_lo = fp16((x - A_hi) 2^11);   W' = W 2^s  (s per output neuron: the row's largest |w| in [2^13, 2^14)),
//   W_hi = fp16(W'), W_d = fp16(W_hi 2^-11), W_lo = fp16(W' - W_hi);     A_hi W_hi + A_lo W_d + A_hi W_lo  ~  x W'.
// The per-neuron scale keeps W_hi, W_d and W_lo normal fp16 numbers however small or large the weights are.  It is a power of
// two, so it commutes with ReLU and is undone exactly: by the producers for layer 1 (2^-s per column, from the image), through the
// output-layer weights for layer 2 (the image holds w3 2^-s: relu(acc) (w3 2^-s) is the same fp32 product as relu(acc 2^-s) w3).
// Range: an A value of a live row -- an observation element, or a hidden activation once its scale is undone -- with
// |x| >= 65520 has no fp16 hi half.  The producers detect it and set the mapped host flag a.range_err; the host reports it
// (drsim_actor_status, and the next drsim_policy_step / drsim_rollout_transition fails).  Padding slots (house >= N) and rows past
// the end enter as zero rows, so whatever they hold never sets it.
// Layouts: layer-1 A and all weights in the canonical no-swizzle K-major layout for 16-bit elements (8 per 16-byte core-matrix
// row; LBO / SBO as for fp32).  Layer-2 A lives in tensor memory IN PLACE of R1: the 16 fp32 columns of granule g (K values
// 16 g ... 16 g + 15) become 8 columns of packed hi pairs, [16 g, 16 g + 8), and 8 of packed lo pairs, [16 g + 8, 16 g + 16),
// written by the one thread that read the granule.  Tensor memory: R1 | R2[0] | R2[1] = N1 + 2 N2 <= 400 columns.
// Image (k_actor_pack3h): [w1_hi | w2_hi | w1_d | w2_d | w1_lo | w2_lo | 2^-s of layer 1 [N1] | w3 2^-s [2][N2] zero-padded, b3[2]].
// ------------------------------------------------------------------------------------------------
constexpr float kF16Overflow = 65520.f;   // the smallest |x| that fp16 round-to-nearest-even turns into infinity

// byte offset of element (row, k) of a K-major 16-bit operand with `rows` rows in the canonical layout
DRSIM_D int umma_kmajor_off16(int rows, int row, int k) {
  return (k >> 3) * (rows >> 3) * 128 + (row >> 3) * 128 + (row & 7) * 16 + (k & 7) * 2;
}
DRSIM_D uint32_t umma_instr_desc_f16(int M, int N) {
  // c_format F32 = 1 [4,6), a/b_format F16 = 0, K-major A and B, n_dim = N >> 3 [17,23), m_dim = M >> 4 [24,29)
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
DRSIM_D void umma_f16_ss(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}
DRSIM_D void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}
// the hi and the 2^11-scaled lo fp16 halves of two values, packed in pairs (the first value in the low 16 bits)
DRSIM_D void split_f16x2(float x0, float x1, uint32_t &hi, uint32_t &lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  const float2 f = __half22float2(h);
  const __half2 l = __floats2half2_rn((x0 - f.x) * 2048.f, (x1 - f.y) * 2048.f);
  hi = *reinterpret_cast<const uint32_t *>(&h);
  lo = *reinterpret_cast<const uint32_t *>(&l);
}

// Row n of the augmented operand [W | b] (+ the one-regenerating row n_out when `gen_one`) as W_hi / W_d / W_lo at img + off,
// + w_bytes, + 2 w_bytes, scaled by the row's 2^s; returns 2^-s.  One warp per row.  s <= 126 keeps 2^s and 2^-s normal
// (weights below 2^-112 then lose fp16 precision instead); s >= -114 holds for every finite weight.
DRSIM_D float pack_row_f16x3(unsigned char *img, int w_bytes, int off, const float *w, const float *b, int n, int n_out, int n_in,
                             int Np, int Kp, bool gen_one, int lane) {
  auto val = [&](int k) -> float {
    if (n < n_out) return k < n_in ? __ldg(w + (size_t)n * n_in + k) : (k == n_in ? __ldg(b + n) : 0.f);
    return (n == n_out && gen_one && k == n_in) ? 1.f : 0.f;
  };
  float m = 0.f;
  for (int k = lane; k < Kp; k += 32) m = fmaxf(m, fabsf(val(k)));
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  int e = 0;
  if (m > 0.f) frexpf(m, &e);                                     // m = f 2^e, f in [0.5, 1)
  const int s = m > 0.f ? min(14 - e, 126) : 0;
  const float up = __int_as_float((127 + s) << 23), down = __int_as_float((127 - s) << 23);
  for (int k = lane; k < Kp; k += 32) {
    const float v = val(k) * up;
    const __half hi = __float2half_rn(v);
    const float hf = __half2float(hi);
    const int o = off + umma_kmajor_off16(Np, n, k);
    *reinterpret_cast<__half *>(img + o) = hi;
    *reinterpret_cast<__half *>(img + w_bytes + o) = __float2half_rn(hf * 0.00048828125f);   // W_hi 2^-11
    *reinterpret_cast<__half *>(img + 2 * w_bytes + o) = __float2half_rn(v - hf);
  }
  return down;
}

// the image of k_actor3<SplitF16x3>, once per launch: one warp per output neuron of layers 1 and 2
__global__ void k_actor_pack3h(ActorArgs a, unsigned char *image) {
  pdl_trigger();
  const int lane = threadIdx.x & 31, wid = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), nw = (int)(gridDim.x * blockDim.x >> 5);
  float *sc1 = reinterpret_cast<float *>(image + a.off_sc), *w3 = reinterpret_cast<float *>(image + a.off_w3);
  for (int r = wid; r < a.N1 + a.N2; r += nw) {
    if (r < a.N1) {
      const float down = pack_row_f16x3(image, a.w_bytes, a.off_w1, a.w1, a.b1, r, a.h1, a.D, a.N1, a.K1, true, lane);
      if (lane == 0) sc1[r] = down;
    } else {
      const int n = r - a.N1;
      const float down = pack_row_f16x3(image, a.w_bytes, a.off_w2, a.w2, a.b2, n, a.h2, a.h1, a.N2, a.K2, false, lane);
      if (lane < 2) w3[lane * a.N2 + n] = n < a.h2 ? __ldg(a.w3 + (size_t)lane * a.h2 + n) * down : 0.f;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x < 2) w3[2 * a.N2 + threadIdx.x] = __ldg(a.b3 + threadIdx.x);
}

// ------------------------------------------------------------------------------------------------
// The operand split of k_actor3: everything in which precision 1 ("tf32x3") and precision 2 ("f16x3") differ.
//   kEl          bytes of an operand element (a 16-byte chunk holds 16 / kEl values)
//   kK           K of one MMA instruction
//   kWBlocks     weight blocks in the image, w_bytes each: a K step multiplies A_hi by block 0, A_lo by block kWLo and
//                A_hi by block kWHi
//   kR1Sets      N1-wide column ranges in front of R2 in tensor memory
//   kRangeCheck  fp16 range: padding slots enter as zero rows, layer 1's 2^-s sit in the image at off_sc, and the
//                producers set a.range_err
//   kPre         the PRE instantiations (16-byte K chunks of the observation operand per producer thread)
// split_a1 writes 16 / kEl layer-1 values as one 16-byte chunk of A_hi and one of A_lo; split_a2 turns granule g of R1
// (its 16 accumulator columns r, read from tensor-memory address col) into layer-2 A; mx collects the largest |A value|.
// ------------------------------------------------------------------------------------------------
struct SplitTf32x3 {   // fp32 as TF32 hi / lo; layer-2 A_lo in L1
  static constexpr int kEl = 4, kK = 8, kWBlocks = 2, kWLo = 0, kWHi = 1, kR1Sets = 2;
  static constexpr bool kRangeCheck = false;
  static constexpr int kPre[4] = {2, 4, 7, 9};
  static DRSIM_D uint32_t idesc(int N) { return umma_instr_desc_tf32(kActRows, N); }
  static DRSIM_D void mma_ss(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) { umma_tf32_ss(d, da, db, idesc, acc); }
  static DRSIM_D void mma_ts(uint32_t d, uint32_t ta, uint64_t db, uint32_t idesc, uint32_t acc) { umma_tf32_ts(d, ta, db, idesc, acc); }
  static DRSIM_D uint32_t a2_lo(int N1) { return (uint32_t)N1; }   // layer-2 A_lo, in columns from A_hi
  static DRSIM_D void split_a1(const float (&v)[4], unsigned char *dh, unsigned char *dl, float &) {
    float h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      h[i] = to_tf32(v[i]);
      l[i] = to_tf32(v[i] - h[i]);
    }
    *reinterpret_cast<float4 *>(dh) = make_float4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<float4 *>(dl) = make_float4(l[0], l[1], l[2], l[3]);
  }
  // ReLU, hi in place, lo to L1
  static DRSIM_D void split_a2(uint32_t (&r)[16], uint32_t col, int N1, const float *, float &) {
    uint32_t l[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float x = fmaxf(__uint_as_float(r[j]), 0.f);
      const float hi = to_tf32(x);
      r[j] = __float_as_uint(hi);
      l[j] = __float_as_uint(to_tf32(x - hi));
    }
    tmem_st16(col, r);
    tmem_st16(col + (uint32_t)N1, l);
  }
};

struct SplitF16x3 {    // fp16 hi / d / lo with per-neuron 2^s; layer-2 A as packed hi | lo pairs in place of R1
  static constexpr int kEl = 2, kK = 16, kWBlocks = 3, kWLo = 1, kWHi = 2, kR1Sets = 1;
  static constexpr bool kRangeCheck = true;
  static constexpr int kPre[4] = {1, 2, 4, 5};
  static DRSIM_D uint32_t idesc(int N) { return umma_instr_desc_f16(kActRows, N); }
  static DRSIM_D void mma_ss(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) { umma_f16_ss(d, da, db, idesc, acc); }
  static DRSIM_D void mma_ts(uint32_t d, uint32_t ta, uint64_t db, uint32_t idesc, uint32_t acc) { umma_f16_ts(d, ta, db, idesc, acc); }
  static DRSIM_D uint32_t a2_lo(int) { return 8u; }
  static DRSIM_D void split_a1(const float (&v)[8], unsigned char *dh, unsigned char *dl, float &mx) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      mx = fmaxf(mx, fmaxf(fabsf(v[2 * i]), fabsf(v[2 * i + 1])));
      split_f16x2(v[2 * i], v[2 * i + 1], h[i], l[i]);
    }
    *reinterpret_cast<uint4 *>(dh) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4 *>(dl) = make_uint4(l[0], l[1], l[2], l[3]);
  }
  // ReLU(x 2^-s), s of each column from sc; packed hi pairs to [col, col + 8), lo pairs to [col + 8, col + 16)
  static DRSIM_D void split_a2(uint32_t (&r)[16], uint32_t col, int, const float *sc, float &mx) {
    const float4 *sc4 = reinterpret_cast<const float4 *>(sc);
    uint32_t o[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 u = sc4[q];
      const float x0 = fmaxf(__uint_as_float(r[4 * q]) * u.x, 0.f), x1 = fmaxf(__uint_as_float(r[4 * q + 1]) * u.y, 0.f),
                  x2 = fmaxf(__uint_as_float(r[4 * q + 2]) * u.z, 0.f), x3 = fmaxf(__uint_as_float(r[4 * q + 3]) * u.w, 0.f);
      mx = fmaxf(mx, fmaxf(fmaxf(x0, x1), fmaxf(x2, x3)));
      split_f16x2(x0, x1, o[2 * q], o[8 + 2 * q]);
      split_f16x2(x2, x3, o[2 * q + 1], o[9 + 2 * q]);
    }
    tmem_st16(col, o);
  }
};

// S: the split (SplitTf32x3, SplitF16x3).  PRE: 16-byte K chunks of the observation operand per producer thread, one of
// S::kPre (>= K1 / S::kK).  O = element type of the observation rows.  bf16 rows are widened in the producers' load: a bf16
// value is exact in TF32, so its hi half is the value itself, its lo half zero, and the products equal those on the widened
// fp32 rows.
template <class S, int PRE, typename O>
__global__ void __launch_bounds__(kAct3Threads, 1) k_actor3(ActorArgs a) {
  constexpr int kVec = 16 / S::kEl;   // operand values per 16-byte chunk
  extern __shared__ __align__(1024) unsigned char smem[];
  // mbarriers: 0 a1_ready (256) | 1 GEMM1 done | 2..6 a2_ready[chunk] (256) | 7, 8 GEMM2 done [slot] |
  //            9, 10 R2 slot drained (128) | 11 weight image
  uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem + a.off_bar);
  uint64_t *a1_ready = s_bar, *bar1 = s_bar + 1, *a2_ready = s_bar + 2, *bar2 = s_bar + 7, *r2_free = s_bar + 9, *wbar = s_bar + 11;
  uint32_t *s_tmem = reinterpret_cast<uint32_t *>(s_bar + 12);
  // the warp index through a shuffle: provably warp-uniform, so the role branches and the MMA warp's descriptor arithmetic
  // stay on the uniform datapath (a divergent single-lane issuer costs ~100 cycles per tcgen05.mma: R2UR + an elect loop
  // around every instruction, twice the 56 cycles the tensor pipe needs for it)
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), role = warp < 8 ? 0 : (warp < 12 ? 1 : 2);   // producer, consumer, MMA warp
  const int t = tid & 127, part = (tid >> 7) & 1;                   // row of the tile (= TMEM lane), column half
  const int n_tiles = (int)((a.rows + kActRows - 1) / kActRows);
  const int n_my = blockIdx.x < n_tiles ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  unsigned char *s_a1h = smem + a.off_a1, *s_a1l = s_a1h + kActRows * a.K1 * S::kEl;   // observation operand, hi and lo

  if (tid == 0) {
    mbar_init(a1_ready, 256);
    mbar_init(bar1, 1);
    for (int k = 0; k < kAct3MaxChunks; ++k) mbar_init(a2_ready + k, 256);
    mbar_init(bar2, 1);
    mbar_init(bar2 + 1, 1);
    mbar_init(r2_free, 128);
    mbar_init(r2_free + 1, 128);
    mbar_init(wbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(s_tmem)),
                 "r"((uint32_t)kAct2TmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_trigger();   // the env step behind us may become resident (it waits for our completion before it reads actions)
  pdl_wait();      // the packed image, the observation rows; the action plane may still be read by the step before us
  if (tid == 0) {  // the packed weight image (weight blocks + output layer): one TMA bulk copy per CTA
    mbar_expect_tx(wbar, (uint32_t)a.off_a1);
    bulk_load_g2s(smem, a.image, (uint32_t)a.off_a1, wbar);
  }
  const uint32_t tmem = *s_tmem;
  const uint32_t R1 = tmem, R2 = tmem + (uint32_t)(S::kR1Sets * a.N1);   // R2 slot s at R2 + s * N2
  const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;   // this warp's TMEM lane quadrant
  const int ng = (a.K2 + 15) >> 4, nchunk = (ng + 1) >> 1;       // 16-column granules / 32-column chunks of R1

  if (role == 0) {
    // ---------------------------------------------------------------- producers
    const int nch = (a.K1 * S::kEl) >> 4, c_lo = part ? nch / 2 : 0, c_hi = part ? nch : nch / 2;   // this thread's 16-byte K chunks
    const float *sc1 = reinterpret_cast<const float *>(smem + a.off_sc);
    float pre[PRE * kVec];
    bool pre_live = false, bad = false;
    auto fetch = [&](int tile) {
      const long long row = (long long)tile * kActRows + t;
      bool live = row < a.rows;
      if constexpr (S::kRangeCheck) {
        if (live) {
          const long long rr = a.rows < (1ll << 31) ? (long long)((uint32_t)row / (uint32_t)a.Ns) : row / a.Ns;
          live = row - rr * a.Ns < a.N;
        }
        pre_live = live;
      }
      const O *g = static_cast<const O *>(a.obs) + (size_t)(live ? row : 0) * a.D;
      if ((a.D & 1) == 0) {
#pragma unroll
        for (int j = 0; j < PRE * kVec / 2; ++j) {
          const int k = c_lo * kVec + 2 * j;
          float2 v = make_float2(0.f, 0.f);
          if (live && k < c_hi * kVec && k < a.D) {
            if constexpr (sizeof(O) == 2) v = __bfloat1622float2(__ldg(reinterpret_cast<const __nv_bfloat162 *>(g + k)));
            else v = __ldg(reinterpret_cast<const float2 *>(g + k));
          }
          pre[2 * j] = v.x;
          pre[2 * j + 1] = v.y;
        }
      } else {
#pragma unroll
        for (int j = 0; j < PRE * kVec; ++j) {
          const int k = c_lo * kVec + j;
          pre[j] = (live && k < c_hi * kVec && k < a.D) ? (float)__ldg(g + k) : 0.f;
        }
      }
    };
    if (n_my > 0) fetch((int)blockIdx.x);
    for (int it = 0; it < n_my; ++it) {
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const bool live = pre_live;
      float mx = 0.f;   // largest |A value| of this row in this thread's columns
      ACT3_STAMP(0);
      // layer-1 operand: [obs | 1 | 0 ...] as hi + lo, one 16-byte store per K chunk (consecutive rows are contiguous:
      // conflict-free).  The previous tile's GEMM1 has completed (bar1 was waited for below).
#pragma unroll
      for (int j = 0; j < PRE; ++j) {
        const int c = c_lo + j;
        if (c < c_hi) {
          float v[kVec];
#pragma unroll
          for (int i = 0; i < kVec; ++i) v[i] = (kVec * c + i == a.D) ? 1.f : pre[kVec * j + i];
          const int off = c * (kActRows * 16) + t * 16;   // row t, 16-byte K chunk c of the canonical layout
          S::split_a1(v, s_a1h + off, s_a1l + off, mx);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(a1_ready);
      ACT3_STAMP(1);
      if (it + 1 < n_my) fetch(tile + (int)gridDim.x);   // in flight during the rest of the round
      ACT3_STAMP(2);
      // layer-2 operand from R1, published chunk by chunk.  bar1 also covers GEMM2 of the previous tile (commit tracks
      // everything issued before it), the last reader of the layer-2 operand.
      mbar_wait_bounded(bar1, (uint32_t)(it & 1));
      tc_fence_after();
      ACT3_STAMP(3);
      uint32_t r[2][16];
      const uint32_t src = R1 + lane_off;
      if (part < ng) tmem_ld16_issue(src + (uint32_t)(16 * part), r[0]);
#pragma unroll
      for (int k = 0; k < kAct3MaxChunks; ++k) {
        if (k < nchunk) {
          const int g = 2 * k + part;                    // granule g of chunk k belongs to column half g & 1
          if (g < ng) {
            tmem_wait_ld_dep(r[k & 1]);
            if (k + 1 < nchunk && g + 2 < ng)            // the next granule flies under this one
              tmem_ld16_issue(src + (uint32_t)(16 * (g + 2)), r[(k + 1) & 1]);
            S::split_a2(r[k & 1], src + (uint32_t)(16 * g), a.N1, sc1 + 16 * g, mx);
            tmem_wait_st();
          }
          tc_fence_before();
          mbar_arrive(a2_ready + k);
          ACT3_STAMP(4 + k);
        }
      }
      if constexpr (S::kRangeCheck) bad |= live && mx >= kF16Overflow;
    }
    if (bad) *reinterpret_cast<volatile int *>(a.range_err) = 1;
  } else if (role == 2) {
    // ---------------------------------------------------------------- MMA warp: one thread issues everything
    if (n_my > 0 && elect_one_lane()) {
      const uint32_t idesc1 = S::idesc(a.N1), idesc2 = S::idesc(a.N2);
      const uint32_t w1 = (uint32_t)__cvta_generic_to_shared(smem + a.off_w1), w2 = (uint32_t)__cvta_generic_to_shared(smem + a.off_w2);
      const uint32_t wlo = (uint32_t)(S::kWLo * a.w_bytes), whi = (uint32_t)(S::kWHi * a.w_bytes);   // weight blocks of passes 2, 3
      const uint32_t a1h = (uint32_t)__cvta_generic_to_shared(s_a1h), a1l = (uint32_t)__cvta_generic_to_shared(s_a1l);
      const uint32_t a2l = S::a2_lo(a.N1);
      const uint32_t lbo_a = (kActRows / 8) * 128, lbo_w1 = (a.N1 / 8) * 128, lbo_w2 = (a.N2 / 8) * 128;
      const int ks1 = a.K1 / S::kK, ks2 = a.K2 / S::kK, kpc = 32 / S::kK;   // K steps of layer 1, of layer 2, per chunk
      mbar_wait_bounded(wbar, 0);   // the weight image has landed (async proxy -> tensor core: no proxy fence)
      for (int it = 0; it < n_my; ++it) {
        const int s = it & 1;
        const uint32_t d2 = R2 + (uint32_t)(s * a.N2);
        mbar_wait_bounded(a1_ready, (uint32_t)(it & 1));
        tc_fence_after();
        ACT3_STAMP(0);
        for (int ks = 0; ks < ks1; ++ks) {      // layer 1: D1[128 x N1] = [obs | 1] . [W1 | b1]^T
          const uint64_t dah = umma_smem_desc(a1h + ks * 2 * lbo_a, lbo_a, 128), dal = umma_smem_desc(a1l + ks * 2 * lbo_a, lbo_a, 128);
          const uint32_t wk = w1 + ks * 2 * lbo_w1;
          S::mma_ss(R1, dah, umma_smem_desc(wk, lbo_w1, 128), idesc1, ks > 0);
          S::mma_ss(R1, dal, umma_smem_desc(wk + wlo, lbo_w1, 128), idesc1, 1);
          S::mma_ss(R1, dah, umma_smem_desc(wk + whi, lbo_w1, 128), idesc1, 1);
        }
        umma_commit(bar1);
        ACT3_STAMP(1);
        for (int k = 0; k < nchunk; ++k) {      // layer 2: D2[128 x N2] = A2 (tensor memory) . [W2 | b2]^T, chunk by chunk
          mbar_wait_bounded(a2_ready + k, (uint32_t)(it & 1));
          if (k == 0 && it >= 2) mbar_wait_bounded(r2_free + s, (uint32_t)(((it >> 1) & 1) ^ 1));   // tile it - 2 has left the slot
          tc_fence_after();
          ACT3_STAMP(2 + k);
          const int ke = min(kpc * k + kpc, ks2);
          for (int ks = kpc * k; ks < ke; ++ks) {
            const uint32_t wk = w2 + ks * 2 * lbo_w2, ah = R1 + (uint32_t)(ks * S::kK);
            S::mma_ts(d2, ah, umma_smem_desc(wk, lbo_w2, 128), idesc2, ks > 0);
            S::mma_ts(d2, ah + a2l, umma_smem_desc(wk + wlo, lbo_w2, 128), idesc2, 1);
            S::mma_ts(d2, ah, umma_smem_desc(wk + whi, lbo_w2, 128), idesc2, 1);
          }
        }
        umma_commit(bar2 + s);
        ACT3_STAMP(7);
      }
    }
  } else {
    // ---------------------------------------------------------------- consumers
    // one thread per row: ReLU + the 2-wide output layer in plain fp32 FMAs straight from the tcgen05.ld registers of the R2
    // slot, softmax, Philox draw
    const float *w3 = reinterpret_cast<const float *>(smem + a.off_w3);   // [2][N2] zero-padded, then b3[2]
    const int ng2 = (a.h2 + 15) >> 4;
    if (n_my > 0) mbar_wait_bounded(wbar, 0);
    for (int it = 0; it < n_my; ++it) {
      const int s = it & 1;
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const uint32_t src = R2 + (uint32_t)(s * a.N2) + lane_off;
      float acc0 = w3[2 * a.N2], acc1 = w3[2 * a.N2 + 1];
      ACT3_STAMP(0);
      mbar_wait_bounded(bar2 + s, (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      ACT3_STAMP(1);
      // rounds of two 16-column granules; the next round's loads fly under this round's arithmetic, two accumulators
      // per logit keep the FMA chains short
      float acc2 = 0.f, acc3 = 0.f;
      uint32_t r[2][2][16];
      const int nrounds = (ng2 + 1) >> 1;
      tmem_ld16_issue(src, r[0][0]);
      if (1 < ng2) tmem_ld16_issue(src + 16u, r[0][1]);
#pragma unroll
      for (int rd = 0; rd < (kAct3MaxChunks + 1); ++rd) {
        if (rd < nrounds) {
          const int g = 2 * rd;
          const bool two = g + 1 < ng2;
          tmem_wait_ld_dep(r[rd & 1][0]);
          if (two) tmem_wait_ld_dep(r[rd & 1][1]);
          if (rd + 1 < nrounds) {
            tmem_ld16_issue(src + (uint32_t)(16 * g + 32), r[(rd + 1) & 1][0]);
            if (g + 3 < ng2) tmem_ld16_issue(src + (uint32_t)(16 * g + 48), r[(rd + 1) & 1][1]);
          } else {                   // the slot's last loads have completed: GEMM2 of tile it + 2 may overwrite it
            tc_fence_before();
            mbar_arrive(r2_free + s);
            ACT3_STAMP(2);
          }
          const float4 *wa = reinterpret_cast<const float4 *>(w3 + 16 * g), *wb = reinterpret_cast<const float4 *>(w3 + a.N2 + 16 * g);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 u = wa[q], v = wb[q];
            const float x0 = fmaxf(__uint_as_float(r[rd & 1][0][4 * q]), 0.f), x1 = fmaxf(__uint_as_float(r[rd & 1][0][4 * q + 1]), 0.f),
                        x2 = fmaxf(__uint_as_float(r[rd & 1][0][4 * q + 2]), 0.f), x3 = fmaxf(__uint_as_float(r[rd & 1][0][4 * q + 3]), 0.f);
            acc0 = fmaf(x0, u.x, acc0); acc2 = fmaf(x1, u.y, acc2); acc0 = fmaf(x2, u.z, acc0); acc2 = fmaf(x3, u.w, acc2);
            acc1 = fmaf(x0, v.x, acc1); acc3 = fmaf(x1, v.y, acc3); acc1 = fmaf(x2, v.z, acc1); acc3 = fmaf(x3, v.w, acc3);
          }
          if (two) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 u = wa[4 + q], v = wb[4 + q];
              const float x0 = fmaxf(__uint_as_float(r[rd & 1][1][4 * q]), 0.f), x1 = fmaxf(__uint_as_float(r[rd & 1][1][4 * q + 1]), 0.f),
                          x2 = fmaxf(__uint_as_float(r[rd & 1][1][4 * q + 2]), 0.f), x3 = fmaxf(__uint_as_float(r[rd & 1][1][4 * q + 3]), 0.f);
              acc0 = fmaf(x0, u.x, acc0); acc2 = fmaf(x1, u.y, acc2); acc0 = fmaf(x2, u.z, acc0); acc2 = fmaf(x3, u.w, acc2);
              acc1 = fmaf(x0, v.x, acc1); acc3 = fmaf(x1, v.y, acc3); acc1 = fmaf(x2, v.z, acc1); acc3 = fmaf(x3, v.w, acc3);
            }
          }
        }
      }
      {
        const float l0 = acc0 + acc2, l1 = acc1 + acc3;
        const long long row = (long long)tile * kActRows + t;
        if (row < a.rows) {
          // replica / house of the row: 32-bit division whenever the row index allows it (the 64-bit one is ~100 instructions)
          const long long rr = a.rows < (1ll << 31) ? (long long)((uint32_t)row / (uint32_t)a.Ns) : row / a.Ns;
          const int n = (int)(row - rr * a.Ns);
          uint8_t act = 0;
          float p_draw = 0.f, p1 = 0.f;
          if (n < a.N) {
            const float m = fmaxf(l0, l1);                      // F.softmax(dim=1), network.py:34
            const float e0 = expf(l0 - m), e1 = expf(l1 - m);
            const float p0 = e0 / (e0 + e1);
            p1 = e1 / (e0 + e1);
            const U4 u = philox4x32_10(a.seed, (uint32_t)(a.rep_offset + rr), (uint32_t)n, (uint32_t)a.step, PURPOSE_POLICY);
            const float uf = (float)(u.x >> 8) * 5.9604644775390625e-8f;   // 24 random bits: [0, 1) exactly
            act = uf < p0 ? 0 : 1;
            p_draw = act ? p1 : p0;
          }
          a.actions[row] = act;
          if (a.prob) a.prob[row] = p_draw;
          if (a.prob_on) a.prob_on[row] = p1;
        }
      }
      ACT3_STAMP(3);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*s_tmem), "r"((uint32_t)kAct2TmemCols) : "memory");
}
#undef ACT3_STAMP
#endif  // __CUDACC__

}  // namespace drsim
