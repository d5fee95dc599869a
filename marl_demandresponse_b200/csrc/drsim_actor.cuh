// drsim_actor.cuh -- MA-PPO actor on the observation rows, fused with the categorical draw
// (SURVEY 8f-2; reference: agents/trainables/network.py:14-35 `Actor`, mappo.py:83-97 `select_actions`).
//
// The reference runs N batch-1 forwards of a [D -> h1 -> h2 -> 2] ReLU MLP per step on the CPU.  Here
// one persistent CTA per SM takes 128 observation rows at a time:
//
//   A1 [128 x D]  (fp32 words, read as TF32)  x  W1^T  --tcgen05.mma-->  TMEM cols [0, N1)
//   epilogue 1 (thread t owns row t = TMEM lane t): tcgen05.ld, + b1, ReLU  ->  A2 in shared memory
//   A2 [128 x h1]                               x  W2^T  --tcgen05.mma-->  TMEM cols [N1, N1 + N2)
//   epilogue 2: tcgen05.ld, + b2, ReLU, the 2-wide output layer on the CUDA cores, softmax,
//               Philox uniform keyed (replica, house, step) -> action byte + probability of the draw
//
// Both GEMMs are issued by ONE thread per CTA (kind::tf32, cta_group::1, M = 128), accumulate in tensor
// memory and signal completion through tcgen05.commit on an mbarrier.  Operands sit in shared memory in
// the canonical no-swizzle K-major layout of the UMMA shared-memory descriptor: 8-row x 16-byte core
// matrices, SBO = 128 B between 8-row groups, LBO = (rows / 8) * 128 B between 16-byte K chunks.  The
// weights are converted once per CTA; only the 128 x D observation tile moves per iteration.
#pragma once

#include <cuda_runtime.h>

#include "drsim_device.cuh"

namespace drsim {

constexpr int kActRows = 128;       // rows per tile == UMMA M == TMEM lanes
constexpr int kActThreads = 128;    // one thread per row / TMEM lane
constexpr int kActTmemCols = 256;   // power of two >= N1 + N2
constexpr uint32_t PURPOSE_POLICY = 6;

struct ActorArgs {
  const void *obs;         // [rows][D] float, or __nv_bfloat16 (k_actor3x<PRE, __nv_bfloat16>)
  const unsigned char *image;   // k_actor2: packed weight operands (k_actor_pack)
  const float *w1, *b1;    // [h1][D], [h1]
  const float *w2, *b2;    // [h2][h1], [h2]
  const float *w3, *b3;    // [2][h2], [2]
  uint8_t *actions;        // [rows]      1 = turn the HVAC on
  float *prob;             // [rows] or NULL: probability of the action that was drawn
  float *prob_on;          // [rows] or NULL: probability of action 1
  long long rows;          // R * Ns (padding slots included; they get action 0)
  int Ns, N, D, h1, h2;
  int K1, N1, K2, N2, K3;  // padded: K multiple of 8 (UMMA_K of tf32), N multiple of 16 (K3: k_actor2's output layer)
  int off_w1, off_w2, off_a1, off_a2, off_vec, off_bar, smem_bytes;
  unsigned long long *dbg; // DRSIM_ACTOR_DBG: clock64 stamps [tile < 8][role][16] of CTA 0 (k_actor3x)
  int off_w3, w_bytes;     // k_actor3x: the fp32 output layer in the image; size of one (hi or lo) weight block
  unsigned long long seed;
  long long step, rep_offset;
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
// operand split of k_actor3x ALU-bound (activations and weights are finite).
DRSIM_D float to_tf32(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
DRSIM_D void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
DRSIM_D void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
DRSIM_D void tmem_ld16(uint32_t taddr, float v[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
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
// k_actor2: the production variant.  Same network, but
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
// k_actor3x: the same network at fp32-grade accuracy on the same tensor cores ("3xTF32").
//
// A TF32 operand keeps 10 mantissa bits; splitting every operand into hi = tf32(x) and lo = tf32(x - hi) and
// accumulating  A_hi W_hi + A_lo W_hi + A_hi W_lo  in the fp32 accumulator recovers ~21 bits per product (the
// dropped A_lo W_lo term is 2^-22 relative): probabilities agree with a plain fp32 forward to ~1e-6 instead of
// the 5e-3 of the single-pass kernel.
//
// Structure: ONE CTA per SM, three warp-specialised roles decoupled by mbarriers (no CTA barrier in the loop):
//   * producers (warps 0-7, two threads per row): the observation rows of the NEXT tile wait in registers; they
//     are split into the hi / lo operands of layer 1 in shared memory (16-byte stores, canonical K-major layout),
//     and after GEMM1 the accumulator R1 is turned into the layer-2 operand IN tensor memory: ReLU, hi in place,
//     lo into a second column range L1.  This pass is pipelined with GEMM2 by 32-column chunks: a chunk's K steps
//     are issued as soon as all rows have published it, so the tensor pipe idles for the first chunk only;
//   * the MMA warp (warp 12, one thread): GEMM1 (shared x shared) and GEMM2 (A from tensor memory), three passes
//     per K step, completion by tcgen05.commit on mbarriers;
//   * consumers (warps 8-11, one thread per row): the layer-2 accumulator R2 is DOUBLE-buffered in tensor memory, so tile i's
//     epilogue overlaps tile i+1's GEMMs: ReLU + the 2-wide output layer in plain fp32 FMAs straight from the
//     tcgen05.ld registers (no third GEMM, no split, no write-back), softmax, Philox draw.
// Tensor memory: R1 | L1 | R2[0] | R2[1] = 2 N1 + 2 N2 <= 512 columns.  Weight image (k_actor_pack3x):
// [w1_hi | w2_hi | w1_lo | w2_lo | w3 fp32 [2][N2] zero-padded, b3[2]], one TMA bulk copy per CTA.
// ------------------------------------------------------------------------------------------------
constexpr int kAct3Threads = 416;    // 8 producer warps + 4 consumer warps + the MMA warp (13 warps: 128 registers each)
constexpr int kAct3MaxChunks = 5;    // 32-column chunks of the layer-2 operand (N1 <= 144)
constexpr int kAct3PreChunks = 9;    // most 16-byte K chunks in HALF an observation row (K1 <= 72); the kernel is instantiated
                                     // for 2 / 4 / 7 / 9 so that the unrolled row handling carries no predicated-off work

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

// O = element type of the observation rows.  bf16 rows are widened in the producers' load: a bf16 value is exact in
// TF32, so its hi half is the value itself, its lo half zero, and the products equal those on the widened fp32 rows.
template <int PRE, typename O = float>   // PRE: 16-byte K chunks per thread in the observation operand (>= K1 / 8)
__global__ void __launch_bounds__(kAct3Threads, 1) k_actor3x(ActorArgs a) {
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
  unsigned char *s_a1h = smem + a.off_a1, *s_a1l = s_a1h + kActRows * a.K1 * 4;   // observation operand, hi and lo

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
  if (tid == 0) {  // the packed weight image (hi + lo + output layer): one TMA bulk copy per CTA
    mbar_expect_tx(wbar, (uint32_t)a.off_a1);
    bulk_load_g2s(smem, a.image, (uint32_t)a.off_a1, wbar);
  }
  const uint32_t tmem = *s_tmem;
  const uint32_t R1 = tmem, L1 = tmem + (uint32_t)a.N1, R2 = tmem + (uint32_t)(2 * a.N1);   // R2 slot s at R2 + s * N2
  const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;   // this warp's TMEM lane quadrant
  const int ng = (a.K2 + 15) >> 4, nchunk = (ng + 1) >> 1;       // 16-column granules / 32-column chunks of the layer-2 operand

  if (role == 0) {
    // ---------------------------------------------------------------- producers
    const int nch = a.K1 >> 2, c_lo = part ? nch / 2 : 0, c_hi = part ? nch : nch / 2;   // this thread's 16-byte K chunks
    float pre[PRE * 4];
    auto fetch = [&](int tile) {
      const long long row = (long long)tile * kActRows + t;
      const bool live = row < a.rows;
      const O *g = static_cast<const O *>(a.obs) + (size_t)(live ? row : 0) * a.D;
      if ((a.D & 1) == 0) {
#pragma unroll
        for (int j = 0; j < PRE * 2; ++j) {
          const int k = c_lo * 4 + 2 * j;
          float2 v = make_float2(0.f, 0.f);
          if (live && k < c_hi * 4 && k < a.D) {
            if constexpr (sizeof(O) == 2) v = __bfloat1622float2(__ldg(reinterpret_cast<const __nv_bfloat162 *>(g + k)));
            else v = __ldg(reinterpret_cast<const float2 *>(g + k));
          }
          pre[2 * j] = v.x;
          pre[2 * j + 1] = v.y;
        }
      } else {
#pragma unroll
        for (int j = 0; j < PRE * 4; ++j) {
          const int k = c_lo * 4 + j;
          pre[j] = (live && k < c_hi * 4 && k < a.D) ? (float)__ldg(g + k) : 0.f;
        }
      }
    };
    if (n_my > 0) fetch((int)blockIdx.x);
    for (int it = 0; it < n_my; ++it) {
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      ACT3_STAMP(0);
      // layer-1 operand: [obs | 1 | 0 ...] as hi + lo, one 16-byte store per K chunk (consecutive rows are contiguous:
      // conflict-free).  The previous tile's GEMM1 has completed (bar1 was waited for below).
#pragma unroll
      for (int j = 0; j < PRE; ++j) {
        const int c = c_lo + j;
        if (c < c_hi) {
          float v[4], h[4], l[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            v[i] = (4 * c + i == a.D) ? 1.f : pre[4 * j + i];
            h[i] = to_tf32(v[i]);
            l[i] = to_tf32(v[i] - h[i]);
          }
          const int off = c * (kActRows * 16) + t * 16;   // = umma_kmajor_off(kActRows, t, 4 c)
          *reinterpret_cast<float4 *>(s_a1h + off) = make_float4(h[0], h[1], h[2], h[3]);
          *reinterpret_cast<float4 *>(s_a1l + off) = make_float4(l[0], l[1], l[2], l[3]);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(a1_ready);
      ACT3_STAMP(1);
      if (it + 1 < n_my) fetch(tile + (int)gridDim.x);   // in flight during the rest of the round
      ACT3_STAMP(2);
      // layer-2 operand: A2 = relu(D1) as hi (in place) + lo, published chunk by chunk.  bar1 also covers GEMM2 of the
      // previous tile (commit tracks everything issued before it): L1 is free to overwrite.
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
            uint32_t l[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float x = fmaxf(__uint_as_float(r[k & 1][j]), 0.f);
              const float hi = to_tf32(x);
              r[k & 1][j] = __float_as_uint(hi);
              l[j] = __float_as_uint(to_tf32(x - hi));
            }
            tmem_st16(R1 + lane_off + (uint32_t)(16 * g), r[k & 1]);
            tmem_st16(L1 + lane_off + (uint32_t)(16 * g), l);
            tmem_wait_st();
          }
          tc_fence_before();
          mbar_arrive(a2_ready + k);
          ACT3_STAMP(4 + k);
        }
      }
    }
  } else if (role == 2) {
    // ---------------------------------------------------------------- MMA warp: one thread issues everything
    if (n_my > 0 && elect_one_lane()) {
      const uint32_t idesc1 = umma_instr_desc_tf32(kActRows, a.N1), idesc2 = umma_instr_desc_tf32(kActRows, a.N2);
      const uint32_t w1h = (uint32_t)__cvta_generic_to_shared(smem + a.off_w1), w2h = (uint32_t)__cvta_generic_to_shared(smem + a.off_w2);
      const uint32_t w1l = w1h + (uint32_t)a.w_bytes, w2l = w2h + (uint32_t)a.w_bytes;
      const uint32_t a1h = (uint32_t)__cvta_generic_to_shared(s_a1h), a1l = (uint32_t)__cvta_generic_to_shared(s_a1l);
      const uint32_t lbo_a = (kActRows / 8) * 128, lbo_w1 = (a.N1 / 8) * 128, lbo_w2 = (a.N2 / 8) * 128;
      const int ks1 = a.K1 >> 3, ks2 = a.K2 >> 3;
      mbar_wait_bounded(wbar, 0);   // the weight image has landed (async proxy -> tensor core: no proxy fence)
      for (int it = 0; it < n_my; ++it) {
        const int s = it & 1;
        const uint32_t d2 = R2 + (uint32_t)(s * a.N2);
        mbar_wait_bounded(a1_ready, (uint32_t)(it & 1));
        tc_fence_after();
        ACT3_STAMP(0);
        for (int ks = 0; ks < ks1; ++ks) {      // layer 1: D1[128 x N1] = [obs | 1] . [W1 | b1]^T -- hi.hi, lo.hi, hi.lo
          const uint64_t dah = umma_smem_desc(a1h + ks * 2 * lbo_a, lbo_a, 128), dal = umma_smem_desc(a1l + ks * 2 * lbo_a, lbo_a, 128);
          const uint64_t dbh = umma_smem_desc(w1h + ks * 2 * lbo_w1, lbo_w1, 128), dbl = umma_smem_desc(w1l + ks * 2 * lbo_w1, lbo_w1, 128);
          umma_tf32_ss(R1, dah, dbh, idesc1, ks > 0);
          umma_tf32_ss(R1, dal, dbh, idesc1, 1);
          umma_tf32_ss(R1, dah, dbl, idesc1, 1);
        }
        umma_commit(bar1);
        ACT3_STAMP(1);
        for (int k = 0; k < nchunk; ++k) {      // layer 2: D2[128 x N2] = A2 (tensor memory) . [W2 | b2]^T, chunk by chunk
          mbar_wait_bounded(a2_ready + k, (uint32_t)(it & 1));
          if (k == 0 && it >= 2) mbar_wait_bounded(r2_free + s, (uint32_t)(((it >> 1) & 1) ^ 1));   // tile it - 2 has left the slot
          tc_fence_after();
          ACT3_STAMP(2 + k);
          const int ke = min(4 * k + 4, ks2);
          for (int ks = 4 * k; ks < ke; ++ks) {
            const uint64_t dbh = umma_smem_desc(w2h + ks * 2 * lbo_w2, lbo_w2, 128), dbl = umma_smem_desc(w2l + ks * 2 * lbo_w2, lbo_w2, 128);
            umma_tf32_ts(d2, R1 + (uint32_t)(ks * 8), dbh, idesc2, ks > 0);
            umma_tf32_ts(d2, L1 + (uint32_t)(ks * 8), dbh, idesc2, 1);
            umma_tf32_ts(d2, R1 + (uint32_t)(ks * 8), dbl, idesc2, 1);
          }
        }
        umma_commit(bar2 + s);
        ACT3_STAMP(7);
      }
    }
  } else {
    // ---------------------------------------------------------------- consumers
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
