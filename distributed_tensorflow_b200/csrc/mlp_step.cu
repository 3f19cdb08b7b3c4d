// One worker training step of the reference MLP as ONE kernel (SURVEY 7.4 #1, K1-K4 + C1 + C2 + C5 fused):
//
//   token wait -> h = relu(x.W1 + b1) -> logits, softmax, clipped batch-SUM cross-entropy, dlogits -> dW2, db2, db1,
//   dh -> dW1 = x^T.dh -> gradients pushed to the ps slots -> stamp + arrival
//   (/root/reference/distributed_mnist.py:109-113,126 = one `mon_sess.run(train_step)` of a worker, :152)
//
// fp32 end to end in memory like the reference model (:98-107); the two large GEMMs run on the tensor cores as TF32
// (tcgen05.mma.kind::tf32, fp32 accumulate in TMEM), everything else in fp32 on the CUDA cores.
//
// Decomposition: G CTAs, CTA c owns the input-feature slice [c*ds, c*ds + ds) (ds a multiple of 8; 784 = 7 x 112).
//   phase 1  TMA-loads its slice of x ([128, ds], issued BEFORE the token wait: the batch does not depend on the
//            parameters) and -- after acquiring the ps token -- its ds rows of W1 straight from the parameter
//            replica / the ps GPU's memory (the pull is the B operand of the first GEMM); ds/8 MMAs give the partial
//            pre-activation [128, H] of the slice in TMEM; it is written to a scratch buffer in L2.
//   phase 2  (after a device-scope counter says all G partials landed) CTA c finalises batch rows [c*R, c*R + R):
//            h = relu(sum of partials + b1), logits, softmax, loss, dlogits, dh rows (-> scratch), and its partial
//            sums of dW2 / db2 / db1 (-> scratch).
//   phase 3  (after a second counter) CTA c sums its share of the G head partials in CTA order and stores it into the
//            gradient slot (a fixed order of additions: the step is bitwise reproducible, unlike fp32 atomics);
//            TMA-loads all of dh; dW1^T[H, slice] = dh^T . x_slice with the SAME slice of the
//            batch, re-fetched from L2 into the same shared-memory buffer while phase 2 runs (tcgen05 wants 32-bit
//            MN-major operands in the SWIZZLE_128B_BASE32B arrangement, the K-major A of phase 1 in SWIZZLE_128B: same
//            bytes, different swizzle, so TMA writes them twice); the epilogue stores the slice's rows of dW1 from TMEM
//            into the gradient slot (local symmetric memory under NVLS, the ps GPU's HBM over NVLink otherwise), then
//            ONE system-scope fence + release-increment of the arrival counter per CTA.
// The split of F1 along K is the split of dW1 along M: CTA c pulls and pushes the SAME rows of W1 / dW1 and reads only
// its slice of the batch from HBM.  Cross-CTA exchange goes through L2 (two counters, ~57 KB written / read per CTA): measured
// DSMEM bandwidth (~20 B/clk/SM) makes a cluster exchange no faster, and a plain grid has no cluster-shape constraint.
//
// DTF_HOST_EMU: compiled by g++ against tests/emu/host_emu.h with the TMA / tcgen05 parts replaced by scalar loops
// (the accumulator rows are recomputed from global memory where the hardware reads TMEM); the three phases are then
// launched one after another (phase_mask), because emulated blocks run sequentially.  The same phase-by-phase mode
// exists on hardware (debugging aid: it removes the inter-CTA waits from the picture).
#include <algorithm>
#include <cstdio>
#include <cstring>

#ifdef DTF_HOST_EMU
#include "host_emu.h"
#else
#include "common.cuh"
#endif
#include "ps_control.h"

namespace dtf {

static constexpr int kStepThreads = 256;
static constexpr int kXChunkBytes = 128 * 128;     // one 32-feature-wide chunk of the batch tile: 128 rows x 128 bytes
// one CTA's partial sums of the head gradients: dW2 [128][16], then db2 [16], then db1 [128]
static constexpr int kHeadPart = 128 * 16 + 16 + 128;

struct MlpStepParams {
  int B, D, H, C;              // batch <= 128, input features, hidden <= 128, classes <= 16
  int G, ds;                   // CTAs (= slices) and slice width (multiple of 8; G * ds >= D)
  int rows_per_cta;            // batch rows finalised per CTA in phase 2 (<= 16)
  int phase_mask;              // bit 0 / 1 / 2: run phase 1 / 2 / 3 (7 = fused; anything else = one phase per launch)
  int n1, n2, kb;              // MMA N of F1 (H rounded to 16), MMA N of B3 (ds rounded to 16), batch rounded to 8
  // ---- inputs: a device-resident dataset walked by the device step counter, or a staged batch (nbatches == 0)
  const float* x;              // [rows, ldx] fp32 (also described by map_x)
  long long ldx;
  const float* labels;         // [rows, ldl] fp32 one-hot
  long long ldl;
  long long nbatches, bstride, boffset;
  // ---- parameters (fp32): the worker's replica, or the ps GPU's master buffers (peer pointers)
  const float* w1;             // [D, ldw1] (also described by map_w1)
  long long ldw1;
  const float* b1;
  const float* w2;             // [H, ldw2]
  long long ldw2;
  const float* b2;
  // ---- scratch (worker-local, L2 resident)
  float* hpart;                // [G][128][n1 + 4] partial pre-activations (row pitch n1 + 4: conflict-free staging rows)
  float* dh;                   // [128][lddh] (rows >= B and columns >= H stay zero)
  long long lddh;
  unsigned int* flags;         // [8]: {partials written, dh rows written, CTAs finished (all monotonic: G per launch), launch
                               //       epoch} for training launches, the same four again for forward-only launches
  float* head_part;            // [G][kHeadPart] per-CTA partial sums of dW2 / db2 / db1
  // ---- gradient slots
  float* gw1;                  // [D, ldgw1]
  long long ldgw1;
  float* gb1;
  float* gw2;                  // [H, ldgw2]
  long long ldgw2;
  float* gb2;
  // ---- loss / bookkeeping
  float clip_min;
  float* loss_out;             // [G] per-CTA partials of the batch-sum loss
  float* logits_out;           // optional [B, C] (forward-only launches: validation / predict)
  unsigned long long* step_counter;     // device step counter (read at entry, incremented by CTA 0 at exit)
  int forward_only;            // 1: stop after the loss / logits (no gradients, no arrival)
  // ---- ps protocol
  int num_tokens;
  const unsigned long long* token[4];   // per ps shard holding a parameter: wait until *token >= step * token_scale
  unsigned long long token_scale[4];    // 1: mailbox token (= global step); G_ps: counter bumped once per ps_apply CTA
  unsigned long long token_base[4];     // the shard's global step when this worker adopted it (checkpoint restore / fabric
                                        // re-formation): step k waits for token >= k * scale + base
  int stamp_step;                       // 1 (sync): the push is stamped with the step; 0 (async): with *stamp_src (version)
  const unsigned long long* consumed[4]; // optional (backup workers, replicas_to_aggregate < replicas): the ps's count of this
                                        // worker's arrivals it has consumed OR dropped -- the slot is rewritten only once the
                                        // previous push (step * G arrivals so far) is no longer needed
  int num_signals;
  unsigned long long* arrivals[4];      // ps arrival counters (+1 per CTA per push)
  unsigned long long* stamp_dst[4];
  const unsigned long long* stamp_src[4];
  int sys_scope;               // 0: the ps shares this GPU (gpu-scope fences suffice)
  unsigned long long timeout_ns;
  unsigned int* err;
  unsigned long long* trace;   // optional [G][32] %globaltimer stamps (profiling / Timeline)
  int clustered;               // 1: the G CTAs are ONE thread-block cluster: the two exchanges are ordered by barrier.cluster
                               //    (release / acquire at cluster scope, ~0.2 us) instead of fence + counter + poll through L2
  int dbg;                     // debugging knobs: bit 0 skip the dW1 stores, bit 1 skip their TMEM loads
  unsigned long long* ring;    // optional worker ring [ring_cap][8] u64 (always-on tracing for the Timeline): CTA 0 writes
  int ring_cap;                //   {kind 2|3, t_entry, t_token, t_forward_end, t_head_end, t_exit, step, G} per launch
};

#ifndef DTF_HOST_EMU
DTF_DEVICE void red_relaxed_sys_add_u64_(unsigned long long* p, unsigned long long v) {
  asm volatile("red.relaxed.sys.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
DTF_DEVICE unsigned int ld_acquire_gpu_u32_(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
DTF_DEVICE unsigned int ld_relaxed_gpu_u32_(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// bring a tile into L2 only (no shared-memory destination, no completion tracking): next step's batch slice
DTF_DEVICE void tma_prefetch_l2_2d(const CUtensorMap* map, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1)
               : "memory");
}
// bulk (TMA) store of a contiguous shared-memory tile to global memory: one instruction by one thread, the copy engine
// streams it out (the destination may be peer memory: the unicast fabric's gradient slot in the ps GPU's HBM)
DTF_DEVICE void bulk_store_1d(void* gdst, const void* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
DTF_DEVICE void bulk_commit_and_wait() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
DTF_DEVICE void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
#else
static inline void red_relaxed_sys_add_u64_(unsigned long long* p, unsigned long long v) { __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
static inline unsigned int ld_acquire_gpu_u32_(const unsigned int* p) { return __atomic_load_n(p, __ATOMIC_SEQ_CST); }
static inline unsigned int ld_relaxed_gpu_u32_(const unsigned int* p) { return __atomic_load_n(p, __ATOMIC_SEQ_CST); }
#endif

// wait until a device-scope counter reaches `target` (bounded); one thread calls it
DTF_DEVICE bool wait_counter_ge(const unsigned int* ctr, unsigned int target, unsigned long long timeout_ns) {
  if ((int)(ld_acquire_gpu_u32_(ctr) - target) >= 0) return true;
  const unsigned long long t0 = globaltimer_ns();
  unsigned int spins = 0;
  while ((int)(ld_relaxed_gpu_u32_(ctr) - target) < 0) {
    if ((++spins & 0x3FF) == 0 && (globaltimer_ns() - t0) > timeout_ns) return false;
  }
  return (int)(ld_acquire_gpu_u32_(ctr) - target) >= 0;
}

#ifndef DTF_HOST_EMU
#define DTF_STEP_MAPS const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_x2, \
                      const __grid_constant__ CUtensorMap map_w1, const __grid_constant__ CUtensorMap map_dh,
#else
#define DTF_STEP_MAPS
#endif

__global__ void __launch_bounds__(kStepThreads, 1) mlp_step_kernel(DTF_STEP_MAPS const MlpStepParams p) {
  DTF_DYN_SMEM(unsigned char, smem_raw);
  __shared__ unsigned long long bars[8];               // mbarriers (8-byte aligned by type)
  __shared__ unsigned int tmem_holder;
  __shared__ unsigned long long s_step;
  __shared__ unsigned int s_epoch;
  __shared__ float s_red[16];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cta = blockIdx.x;
  const int d0 = cta * p.ds;
  const bool fused = p.phase_mask == 7;
  unsigned long long* tr = p.trace ? p.trace + 32 * cta : nullptr;
#define STAMP(slot) do { if (tr && tid == 0) tr[slot] = globaltimer_ns(); } while (0)
  STAMP(0);
  // worker ring: thread 0 of CTA 0 keeps five %globaltimer reads in registers and writes ONE 64-byte row at exit
  const bool ringer = p.ring != nullptr && cta == 0 && tid == 0;
  unsigned long long rt_entry = 0, rt_token = 0, rt_fwd = 0, rt_head = 0;
  if (ringer) rt_entry = globaltimer_ns();

  // ---- shared memory carve-up: [x tile | W1 slice / dh tile | head scratch]
#ifndef DTF_HOST_EMU
  unsigned char* tiles = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
#else
  unsigned char* tiles = smem_raw;
#endif
  const int nqx = (p.ds + 31) / 32;                       // 32-feature chunks of the batch tile
  const int nq1 = (p.n1 + 31) / 32;                       // 32-unit chunks of the W1 slice
  const int w_chunk = p.ds * 128;                         // bytes of one W1 chunk ([ds rows] x 128 B)
  const int dh_chunk = p.kb * 128;                        // bytes of one dh chunk ([kb rows] x 128 B)
  unsigned char* x_sm = tiles;
  unsigned char* w_sm = x_sm + nqx * kXChunkBytes;
  const int hpp = p.n1 + 4;                               // row pitch of the partial-pre-activation tile (smem staging == global)
  const int w_region = max(max(nq1 * w_chunk, 4 * dh_chunk), 128 * hpp * 4);
  float* hs = reinterpret_cast<float*>(w_sm + ((w_region + 1023) & ~1023));
  constexpr int HP = 132;                                 // padded row of the [16][128] activation tiles
  float* s_h = hs;                                        // [16][HP]
  float* s_dh = s_h + 16 * HP;                            // [16][HP]
  constexpr int WS = 20;                                  // row stride of the [128][16] W2 tile: 80 B keeps float4 rows of
                                                          // consecutive hidden units on distinct banks
  float* s_w2 = s_dh + 16 * HP;                           // [128][WS]
  float* s_b1 = s_w2 + 128 * WS;                          // [128]
  float* s_dl = s_b1 + 128;                               // [16][16]
  float* s_lab = s_dl + 256;                              // [16][16]
  float* s_b2 = s_lab + 256;                              // [16]

  unsigned int* fl = p.flags + (p.forward_only ? 4 : 0);
  // programmatic dependent launch: the kernel behind this one in the stream (the ps's apply when it shares the GPU, the next
  // step otherwise) may start ITS prologue now; ours -- barriers, tensor memory, descriptor prefetch -- runs under the tail of
  // the kernel in front of us, and nothing that kernel wrote (step counter, launch epoch, tokens, parameters) is read before
  // griddep_wait() below
  griddep_launch_dependents();
#ifndef DTF_HOST_EMU
  uint64_t* bar_x = reinterpret_cast<uint64_t*>(&bars[0]);
  uint64_t* bar_w = reinterpret_cast<uint64_t*>(&bars[1]);
  uint64_t* bar_m1 = reinterpret_cast<uint64_t*>(&bars[2]);
  uint64_t* bar_dh = reinterpret_cast<uint64_t*>(&bars[3]);
  uint64_t* bar_m2 = reinterpret_cast<uint64_t*>(&bars[4]);
  uint64_t* bar_x2 = reinterpret_cast<uint64_t*>(&bars[5]);
  if (tid == 0) {
    for (int i = 0; i < 6; ++i) mbar_init(reinterpret_cast<uint64_t*>(&bars[i]), 1);
    fence_mbar_init();
    tma_prefetch_desc(&map_x);
    tma_prefetch_desc(&map_x2);
    tma_prefetch_desc(&map_w1);
    tma_prefetch_desc(&map_dh);
  }
  if (warp == 1) {
    tmem_alloc(&tmem_holder, 256);
    tmem_relinquish();
  }
  tc_fence_before();
#endif
  griddep_wait();
  if (tid == 0) {
    s_step = p.step_counter ? *p.step_counter : 0ull;
    s_epoch = ld_relaxed_gpu_u32_(&fl[3]);
  }
  __syncthreads();
#ifndef DTF_HOST_EMU
  tc_fence_after();
  const uint32_t tmem_d1 = tmem_holder;                   // F1 accumulator: columns [0, n1)
  const uint32_t tmem_d2 = tmem_holder + 128;             // B3 accumulator: columns [128, 128 + n2)
#endif
  const unsigned long long step = s_step;
  const unsigned int sync_target = (unsigned int)p.G * (s_epoch + 1u);      // what the monotonic counters reach in THIS launch
  const long long row0 = p.nbatches > 0
      ? (long long)((step * (unsigned long long)p.bstride + (unsigned long long)p.boffset) % (unsigned long long)p.nbatches) * p.B
      : 0ll;
#ifndef DTF_HOST_EMU
  if (fused && !p.forward_only && p.nbatches > 0 && warp == 2 && lane == 0) {
    // the dataset is larger than L2 (172 MB): start pulling the NEXT step's slice of the batch into L2 now, a whole step
    // ahead, so that step's TMA finds it there instead of paying HBM latency on 128-byte pieces
    const long long row_next = (long long)(((step + 1ull) * (unsigned long long)p.bstride + (unsigned long long)p.boffset) %
                                           (unsigned long long)p.nbatches) * p.B;
    for (int q = 0; q < nqx; ++q) tma_prefetch_l2_2d(&map_x, d0 + 32 * q, (int32_t)row_next);
  }
#endif
  const int r_lo = cta * p.rows_per_cta;                  // batch rows this CTA finalises in phase 2
  const int nrows = max(0, min(p.rows_per_cta, p.B - r_lo));
  STAMP(1);

  // =====================================================================================================
  // phase 1: partial pre-activation of this feature slice
  // =====================================================================================================
  if (p.phase_mask & 3) {
    if (tid == 0) {
#ifndef DTF_HOST_EMU
      if (p.phase_mask & 1) {
        mbar_arrive_expect_tx(bar_x, (uint32_t)(nqx * kXChunkBytes));
        for (int q = 0; q < nqx; ++q) tma_load_2d(x_sm + q * kXChunkBytes, &map_x, bar_x, d0 + 32 * q, (int32_t)row0);
      }
#endif
      // the parameters behind every later read were published by the ps: acquire its token(s) for this step
      for (int i = 0; i < p.num_tokens; ++i)
        if (!wait_flag_ge_u64(reinterpret_cast<const uint64_t*>(p.token[i]), step * p.token_scale[i] + p.token_base[i], p.timeout_ns) && p.err)
          atomicExch(p.err, 1u);
      // backup workers: a straggler holds the next token while its late push still waits in the slot for the ps to fold it
      // in or drop it as stale -- do not overwrite a gradient the ps may be reading (TF's accumulator copies under a lock)
      for (int i = 0; i < p.num_signals; ++i)
        if (p.consumed[i] != nullptr && !p.forward_only &&
            !wait_flag_ge_u64(reinterpret_cast<const uint64_t*>(p.consumed[i]), step * (unsigned long long)p.G, p.timeout_ns) && p.err)
          atomicExch(p.err, 6u);
      // (colocated: the ps kernel that released this token finished before this kernel started -- stream order -- so the
      //  acquire's fast path is a single already-satisfied load)
#ifndef DTF_HOST_EMU
      fence_proxy_async();
      if (p.phase_mask & 1) {
        mbar_arrive_expect_tx(bar_w, (uint32_t)(nq1 * w_chunk));
        for (int q = 0; q < nq1; ++q) tma_load_2d(w_sm + q * w_chunk, &map_w1, bar_w, 32 * q, d0);   // box {32 units, ds rows}
      }
#endif
    }
    if (ringer) rt_token = globaltimer_ns();
    __syncthreads();                                       // token acquired (thread 0's acquire + barrier)
    STAMP(2);
  }
  // small parameters and this CTA's label rows -> shared memory, by warps 1..7 (warp 0's elected thread walks the
  // TMA -> MMA chain and must not wait on global loads); each thread's loads are issued as one independent batch
  if ((p.phase_mask & 2) && warp > 0) {
    const int t = tid - 32, nt = kStepThreads - 32;
    float v[10];
#pragma unroll
    for (int u = 0; u < 10; ++u) {
      const int i = t + u * nt;                             // 2048 (j, c) pairs over 224 threads
      const int j = i >> 4, c = i & 15;
      v[u] = (i < 128 * 16 && j < p.H && c < p.C) ? p.w2[(long long)j * p.ldw2 + c] : 0.f;
    }
    const float vb1 = t < p.H ? p.b1[t] : 0.f;
    const float vb2 = t < p.C ? p.b2[t] : 0.f;
    float vl[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = t + u * nt;
      const int r = i >> 4, c = i & 15;
      vl[u] = (i < 256 && r < nrows && c < p.C) ? p.labels[(row0 + r_lo + r) * p.ldl + c] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 10; ++u) {
      const int i = t + u * nt;
      if (i < 128 * 16) s_w2[(i >> 4) * WS + (i & 15)] = v[u];
    }
    if (t < 128) s_b1[t] = vb1;
    if (t < 16) s_b2[t] = vb2;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = t + u * nt;
      if (i < 256) s_lab[i] = vl[u];
    }
  }
  if (p.phase_mask & 1) {
#ifndef DTF_HOST_EMU
    if (tid == 0) {
      mbar_wait(bar_x, 0);
      STAMP(11);
      mbar_wait(bar_w, 0);
      STAMP(12);
      tc_fence_after();
      const uint32_t idesc = make_idesc(128, (uint32_t)p.n1, 0, 1, 1);       // A = x: K-major; B = W1[i][j]: MN-major
      const uint32_t xa = smem_u32(x_sm), wa = smem_u32(w_sm);
      for (int s = 0; s < p.ds / 8; ++s) {
        const uint64_t a_desc = make_smem_desc_sw128(xa + (s >> 2) * kXChunkBytes + (s & 3) * 32, 16, 1024);
        const uint64_t b_desc = make_smem_desc(wa + s * 1024, (uint32_t)w_chunk, 512, 1);      // 32-bit MN-major: BASE32B atoms
        umma_tf32(tmem_d1, a_desc, b_desc, idesc, s > 0 ? 1u : 0u);
      }
      umma_commit(bar_m1);
      STAMP(13);
      if (fused && !p.forward_only) {
        // the tensor core is done with the K-major copy of the batch slice: fetch the MN-major arrangement for phase 3
        // into the same buffer now, under the shadow of phase 2
        mbar_wait(bar_m1, 0);
        mbar_arrive_expect_tx(bar_x2, (uint32_t)(nqx * kXChunkBytes));
        for (int q = 0; q < nqx; ++q) tma_load_2d(x_sm + q * kXChunkBytes, &map_x2, bar_x2, d0 + 32 * q, (int32_t)row0);
        STAMP(14);
      }
    }
#endif
  }
  if (p.phase_mask & 1) {
#ifndef DTF_HOST_EMU
    mbar_wait(bar_m1, 0);
    tc_fence_after();
#endif
    STAMP(3);
    if (ringer) rt_fwd = globaltimer_ns();
    // epilogue 1: TMEM (lane = batch row, column = hidden unit) -> hpart[cta][row][0..n1)
    const int q = warp & 3, half = warp >> 2;
    const int b = q * 32 + lane;
    const int nchunks = p.n1 / 8;
    const int c_lo = half * ((nchunks + 1) / 2), c_hi = half ? nchunks : (nchunks + 1) / 2;
    float* dst = p.hpart + ((long long)cta * 128 + b) * hpp;
#ifndef DTF_HOST_EMU
    {
      // all of this warp's TMEM loads in flight at once (<= 8 chunks of 8 columns), ONE wait; the rows are parked in shared
      // memory (the W1 tile is dead: its MMAs completed) and leave as ONE bulk store -- hpart[cta] is that same [rows][hpp]
      // block in global memory
      float* stage = reinterpret_cast<float*>(w_sm) + b * hpp;
      uint32_t r[8][8];
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (c_lo + u < c_hi) tmem_ld_32x32b_x8(tmem_d1 + ((uint32_t)(q * 32) << 16) + (uint32_t)((c_lo + u) * 8), r[u]);
      tmem_ld_wait();
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (c_lo + u < c_hi) {
          float4* o = reinterpret_cast<float4*>(stage + (c_lo + u) * 8);
          o[0] = make_float4(__uint_as_float(r[u][0]), __uint_as_float(r[u][1]), __uint_as_float(r[u][2]), __uint_as_float(r[u][3]));
          o[1] = make_float4(__uint_as_float(r[u][4]), __uint_as_float(r[u][5]), __uint_as_float(r[u][6]), __uint_as_float(r[u][7]));
        }
      fence_proxy_async_smem();
      __syncthreads();
      if (tid == 0) {
        bulk_store_1d(p.hpart + (long long)cta * 128 * hpp, w_sm, (uint32_t)(p.B * hpp * 4));
        bulk_commit_and_wait();
      }
    }
#else
    for (int ch = c_lo; ch < c_hi; ++ch) {
      float v[8];
      for (int u = 0; u < 8; ++u) {
        const int j = ch * 8 + u;
        float a = 0.f;
        if (b < p.B && j < p.H)
          for (int i = d0; i < min(d0 + p.ds, p.D); ++i) a += p.x[(row0 + b) * p.ldx + i] * p.w1[(long long)i * p.ldw1 + j];
        v[u] = a;
      }
      if (b < p.B) {
        reinterpret_cast<float4*>(dst + ch * 8)[0] = make_float4(v[0], v[1], v[2], v[3]);
        reinterpret_cast<float4*>(dst + ch * 8)[1] = make_float4(v[4], v[5], v[6], v[7]);
      }
    }
    (void)dst;
#endif
#ifndef DTF_HOST_EMU
    if (fused && p.clustered) {
      cluster_sync_all();            // every CTA's partials are written and visible to every CTA of the cluster
    } else
#endif
    {
      __syncthreads();
      if (tid == 0) {
        __threadfence();
        atomicAdd(&fl[0], 1u);
      }
    }
    STAMP(4);
  }

  // =====================================================================================================
  // phase 2: finalise this CTA's batch rows -- h, logits, softmax / loss / dlogits, dh, dW2 / db2 / db1 partials
  // =====================================================================================================
  if (p.phase_mask & 2) {
    if (fused && !p.clustered) {
      if (tid == 0 && !wait_counter_ge(&fl[0], sync_target, p.timeout_ns) && p.err) atomicExch(p.err, 4u);
    }
    __syncthreads();
    STAMP(5);
    // h[r][j] = relu(sum_c hpart[c][r_lo + r][j] + b1[j]); the G partials of a position are loaded as ONE batch of
    // independent L2 requests (a serial loop would pay G round trips)
    const int n1v = p.n1 / 4;
    for (int idx = tid; idx < 16 * n1v; idx += kStepThreads) {
      const int r = idx / n1v, j4 = idx - r * n1v;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nrows) {
        const float4* base = reinterpret_cast<const float4*>(p.hpart + (long long)(r_lo + r) * hpp) + j4;
        const long long cstride = (long long)128 * hpp / 4;
        for (int c0 = 0; c0 < p.G; c0 += 8) {
          float4 t[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) t[u] = (c0 + u < p.G) ? __ldcg(base + (c0 + u) * cstride) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int u = 0; u < 8; ++u) { a.x += t[u].x; a.y += t[u].y; a.z += t[u].z; a.w += t[u].w; }
        }
        a.x = fmaxf(a.x + s_b1[4 * j4], 0.f);
        a.y = fmaxf(a.y + s_b1[4 * j4 + 1], 0.f);
        a.z = fmaxf(a.z + s_b1[4 * j4 + 2], 0.f);
        a.w = fmaxf(a.w + s_b1[4 * j4 + 3], 0.f);
      }
      float* o = s_h + r * HP + 4 * j4;
      o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w;
    }
    __syncthreads();
    STAMP(15);
    // logits / softmax / loss / dlogits.  Thread = (row r, quarter jq of the hidden units, class quad cq): one scalar + one
    // 16-byte shared-memory load per 4 FMAs; the four jq partials meet by shuffles, the 16 classes of a row = 4 lanes x 4.
    float my_loss = 0.f;
    {
      const int r = tid >> 4, jq = (tid >> 2) & 3, cq = tid & 3;
      const int jn = p.n1 >> 2;                                  // n1 is a multiple of 16
      const float* hr = s_h + r * HP + jq * jn;
      const float* wr = s_w2 + (jq * jn) * WS + 4 * cq;
      float z[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
      for (int j = 0; j < jn; ++j) {                             // rows of s_h / s_w2 beyond H are zero
        const float hv = hr[j];
        const float4 w = *reinterpret_cast<const float4*>(wr + j * WS);
        z[0] = fmaf(hv, w.x, z[0]); z[1] = fmaf(hv, w.y, z[1]); z[2] = fmaf(hv, w.z, z[2]); z[3] = fmaf(hv, w.w, z[3]);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        z[k] += __shfl_xor_sync(0xffffffffu, z[k], 4);
        z[k] += __shfl_xor_sync(0xffffffffu, z[k], 8);
      }
      bool live[4];
      float mx = -INFINITY;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        live[k] = 4 * cq + k < p.C;
        z[k] = live[k] ? z[k] + s_b2[4 * cq + k] : -INFINITY;
        mx = fmaxf(mx, z[k]);
      }
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      float e[4], se = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        e[k] = live[k] ? __expf(z[k] - mx) : 0.f;
        se += e[k];
      }
      se += __shfl_xor_sync(0xffffffffu, se, 1);
      se += __shfl_xor_sync(0xffffffffu, se, 2);
      const float inv = 1.f / se, lse = mx + __logf(se);
      const float4 lab4 = *reinterpret_cast<const float4*>(s_lab + r * 16 + 4 * cq);
      const float lab[4] = {lab4.x, lab4.y, lab4.z, lab4.w};
      float t[4], y[4], tsum = 0.f, lterm = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        y[k] = e[k] * inv;
        t[k] = 0.f;
        if (live[k]) {
          if (p.clip_min > 0.f) {
            lterm -= lab[k] * fmaxf(z[k] - lse, __logf(p.clip_min));   // log(clamp(y, clip, 1)) = max(log y, log clip), y <= 1
            t[k] = (y[k] >= p.clip_min) ? lab[k] : 0.f;
          } else {
            lterm -= lab[k] * (z[k] - lse);
            t[k] = lab[k];
          }
        }
        tsum += t[k];
      }
      tsum += __shfl_xor_sync(0xffffffffu, tsum, 1);
      tsum += __shfl_xor_sync(0xffffffffu, tsum, 2);
      const bool rlive = r < nrows;
      if (jq == 0) {                                             // one writer per (row, quad)
        float4 g4;
        g4.x = (live[0] && rlive) ? y[0] * tsum - t[0] : 0.f;
        g4.y = (live[1] && rlive) ? y[1] * tsum - t[1] : 0.f;
        g4.z = (live[2] && rlive) ? y[2] * tsum - t[2] : 0.f;
        g4.w = (live[3] && rlive) ? y[3] * tsum - t[3] : 0.f;
        *reinterpret_cast<float4*>(s_dl + r * 16 + 4 * cq) = g4;
        if (p.logits_out && rlive) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (live[k]) p.logits_out[(long long)(r_lo + r) * p.C + 4 * cq + k] = z[k];
        }
      }
      my_loss = (jq == 0 && rlive) ? lterm : 0.f;
      for (int o = 16; o > 0; o >>= 1) my_loss += __shfl_xor_sync(0xffffffffu, my_loss, o);
      if (lane == 0) s_red[warp] = my_loss;
    }
    __syncthreads();
    STAMP(16);
    if (tid == 0) {
      float t = 0.f;
      for (int i = 0; i < kStepThreads / 32; ++i) t += s_red[i];
      p.loss_out[cta] = t;
    }
    if (!p.forward_only) {
      // dh[r][j] = (h > 0) * dl[r][:] . W2[j][:] and db1[j] = sum_r dh[r][j].  Thread = (hidden unit j, row group): the W2 row
      // stays in registers across the group's 8 rows, the dl row is a broadcast; dh rows go to the L2 scratch (coalesced over j)
      {
        const int j = tid & 127, rg = tid >> 7;
        float4 w[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) w[c] = *reinterpret_cast<const float4*>(s_w2 + j * WS + 4 * c);
        float db1 = 0.f;
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          const int r = rg * 8 + rr;
          const float4* dl = reinterpret_cast<const float4*>(s_dl + r * 16);
          float d = 0.f, d1 = 0.f;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float4 a4 = dl[c];
            d = fmaf(a4.x, w[c].x, d); d1 = fmaf(a4.y, w[c].y, d1);
            d = fmaf(a4.z, w[c].z, d); d1 = fmaf(a4.w, w[c].w, d1);
          }
          d = (j < p.n1 && s_h[r * HP + j] > 0.f) ? d + d1 : 0.f;   // rows >= nrows / units >= H: h == 0 -> 0
          if (r < nrows && j < p.n1) p.dh[(long long)(r_lo + r) * p.lddh + j] = d;
          db1 += d;
        }
        s_dh[rg * 128 + j] = db1;                                // combine the two row groups below
      }
      STAMP(17);
      // this CTA's partials of dW2[j][4cq .. 4cq+3] = sum_r h[r][j] * dl[r][4cq .. 4cq+3]: one scalar + one 16-byte load
      // per 4 FMAs; db2 and db1 behind them (phase 3 adds the G partials up)
      float* part = p.head_part + (long long)cta * kHeadPart;
      for (int it = tid; it < 128 * 4; it += kStepThreads) {
        const int j = it >> 2, cq = it & 3;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < p.H && 4 * cq < p.C) {
#pragma unroll
          for (int r = 0; r < 16; ++r) {                         // row slots beyond nrows hold zeros in s_h and s_dl
            const float hv = s_h[r * HP + j];
            const float4 d4 = *reinterpret_cast<const float4*>(s_dl + r * 16 + 4 * cq);
            a.x = fmaf(hv, d4.x, a.x); a.y = fmaf(hv, d4.y, a.y); a.z = fmaf(hv, d4.z, a.z); a.w = fmaf(hv, d4.w, a.w);
          }
        }
        reinterpret_cast<float4*>(part)[it] = a;
      }
      if (tid < 16) {
        float a = 0.f;
#pragma unroll
        for (int r = 0; r < 16; ++r) a += s_dl[r * 16 + tid];
        part[128 * 16 + tid] = a;
      }
      __syncthreads();
      STAMP(18);
      if (tid < 128) part[128 * 16 + 16 + tid] = s_dh[tid] + s_dh[128 + tid];
#ifndef DTF_HOST_EMU
      if (fused && p.clustered) {
        STAMP(19);
        cluster_sync_all();          // every CTA's dh rows are in L2 and visible to the cluster
      } else
#endif
      {
        __syncthreads();
        STAMP(19);
        if (tid == 0) {
          __threadfence();
          atomicAdd(&fl[1], 1u);
        }
      }
    }
    STAMP(6);
    if (ringer) rt_head = globaltimer_ns();
  }

  // =====================================================================================================
  // phase 3: dW1 rows of this slice = x_slice^T . dh, pushed from TMEM into the gradient slot; arrival
  // =====================================================================================================
  if ((p.phase_mask & 4) && !p.forward_only) {
#ifndef DTF_HOST_EMU
    if (tid == 0) {
      if (fused && !p.clustered && !wait_counter_ge(&fl[1], sync_target, p.timeout_ns) && p.err) atomicExch(p.err, 5u);
      fence_proxy_async();
      mbar_arrive_expect_tx(bar_dh, (uint32_t)(4 * dh_chunk));
      for (int q = 0; q < 4; ++q) tma_load_2d(w_sm + q * dh_chunk, &map_dh, bar_dh, 32 * q, 0);      // box {32 units, kb rows}
      if (!fused) {
        mbar_arrive_expect_tx(bar_x2, (uint32_t)(nqx * kXChunkBytes));
        for (int q = 0; q < nqx; ++q) tma_load_2d(x_sm + q * kXChunkBytes, &map_x2, bar_x2, d0 + 32 * q, (int32_t)row0);
      }
      STAMP(20);
      mbar_wait(bar_x2, 0);
      mbar_wait(bar_dh, 0);
      STAMP(21);
      tc_fence_after();
      const uint32_t idesc = make_idesc(128, (uint32_t)p.n2, 1, 1, 1);       // A = dh[b][j]: MN-major; B = x[b][i]: MN-major
      const uint32_t xa = smem_u32(x_sm), da = smem_u32(w_sm);
      for (int s = 0; s < p.kb / 8; ++s) {
        const uint64_t a_desc = make_smem_desc(da + s * 1024, (uint32_t)dh_chunk, 512, 1);
        const uint64_t b_desc = make_smem_desc(xa + s * 1024, (uint32_t)kXChunkBytes, 512, 1);
        umma_tf32(tmem_d2, a_desc, b_desc, idesc, s > 0 ? 1u : 0u);
      }
      umma_commit(bar_m2);
    }
#else
    if (fused) { /* emulated blocks run one after another: the fused mode is hardware-only */ }
#endif
    // while the MMAs run: the head gradients of this CTA's share of [0, kHeadPart), the G partials added in CTA order.
    // Thread 0 acquired the phase-2 counter above (clustered: the cluster barrier did), so every partial is in L2
    __syncthreads();
    {
      const int share = (kHeadPart + p.G - 1) / p.G;
      const int e_hi = min(kHeadPart, (cta + 1) * share);
      for (int e = cta * share + tid; e < e_hi; e += kStepThreads) {
        float* dst;
        if (e < 128 * 16) dst = (e / 16 < p.H && e % 16 < p.C) ? p.gw2 + (long long)(e / 16) * p.ldgw2 + e % 16 : nullptr;
        else if (e < 128 * 16 + 16) dst = (e - 128 * 16 < p.C) ? p.gb2 + (e - 128 * 16) : nullptr;
        else dst = (e - 128 * 16 - 16 < p.H) ? p.gb1 + (e - 128 * 16 - 16) : nullptr;
        if (dst == nullptr) continue;
        const float* src = p.head_part + e;
        float a = 0.f;
        for (int c0 = 0; c0 < p.G; c0 += 8) {
          float t[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) t[u] = (c0 + u < p.G) ? __ldcg(src + (long long)(c0 + u) * kHeadPart) : 0.f;
#pragma unroll
          for (int u = 0; u < 8; ++u) a += t[u];
        }
        *dst = a;
      }
    }
#ifndef DTF_HOST_EMU
    mbar_wait(bar_m2, 0);
    tc_fence_after();
#endif
    STAMP(7);
    // epilogue 2: TMEM (lane = hidden unit j, column = feature i of the slice) -> gw1[d0 + i][j]: a warp stores 32
    // consecutive j per feature = one 128-byte line per instruction
    {
      const int q = warp & 3, half = warp >> 2;
      const int j = q * 32 + lane;
      const int nchunks = p.n2 / 8;
      const int c_lo = half * ((nchunks + 1) / 2), c_hi = half ? nchunks : (nchunks + 1) / 2;
#ifndef DTF_HOST_EMU
      {
        uint32_t r[8][8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (c_lo + u < c_hi && !(p.dbg & 2)) tmem_ld_32x32b_x8(tmem_d2 + ((uint32_t)(q * 32) << 16) + (uint32_t)((c_lo + u) * 8), r[u]);
        tmem_ld_wait();
        const int ncols = min(p.ds, p.D - d0);                 // features of this slice that exist
        if (p.ldgw1 == 128) {
          // the slot's rows are 128 floats: the slice's rows form ONE contiguous block [ncols][128] -- park the tile in
          // shared memory (the batch tile is dead: the B3 MMAs completed; lanes = consecutive j -> conflict-free) and
          // push it with one bulk store.  Hidden units >= H are rows of exact zeros (dh's padding), like the slot's padding.
          float* stage = reinterpret_cast<float*>(x_sm);
#pragma unroll
          for (int u = 0; u < 8; ++u)
            if (c_lo + u < c_hi) {
#pragma unroll
              for (int v = 0; v < 8; ++v) stage[((c_lo + u) * 8 + v) * 128 + j] = __uint_as_float(r[u][v]);
            }
          fence_proxy_async_smem();
          __syncthreads();
          if (tid == 0 && ncols > 0 && !(p.dbg & 1)) {
            bulk_store_1d(p.gw1 + (long long)d0 * 128, x_sm, (uint32_t)(ncols * 512));
            bulk_commit_and_wait();
          }
        } else if (j < p.H && !(p.dbg & 1)) {
          float* g = p.gw1 + (long long)(d0 + c_lo * 8) * p.ldgw1 + j;
#pragma unroll
          for (int u = 0; u < 8; ++u)
            if (c_lo + u < c_hi) {
#pragma unroll
              for (int v = 0; v < 8; ++v)
                if ((c_lo + u) * 8 + v < ncols) g[(long long)(u * 8 + v) * p.ldgw1] = __uint_as_float(r[u][v]);
            }
        }
      }
#else
      for (int ch = c_lo; ch < c_hi; ++ch) {
        float v[8];
        for (int u = 0; u < 8; ++u) {
          const int i = d0 + ch * 8 + u;
          float a = 0.f;
          if (j < p.H && i < p.D)
            for (int b = 0; b < p.B; ++b) a += p.x[(row0 + b) * p.ldx + i] * p.dh[(long long)b * p.lddh + j];
          v[u] = a;
        }
        if (j < p.H) {
          for (int u = 0; u < 8; ++u) {
            const int il = ch * 8 + u;
            if (il < p.ds && d0 + il < p.D) p.gw1[(long long)(d0 + il) * p.ldgw1 + j] = v[u];
          }
        }
      }
#endif
    }
    __syncthreads();
    STAMP(8);
    if (tid == 0) {
      // CTA 0 stamps the push FIRST; then ONE fence by one thread per CTA after the CTA barrier (release is cumulative: it
      // covers the bulk store waited for above, the head's stores and the stamp), then a RELAXED arrival.  The ps acts on
      // the push only once all G arrivals are in, CTA 0's included, so the stamp is visible by then.  When the ps shares this
      // GPU AND this stream (colocated), its kernel starts after this one has completed: no fence at all.
      if (cta == 0)
        for (int i = 0; i < p.num_signals; ++i)
          if (p.stamp_dst[i]) st_relaxed_sys_u64(reinterpret_cast<uint64_t*>(p.stamp_dst[i]), p.stamp_step ? step : *p.stamp_src[i]);
      if (p.sys_scope) fence_acq_rel_sys();
      for (int i = 0; i < p.num_signals; ++i) {
        if (p.sys_scope) red_relaxed_sys_add_u64_(p.arrivals[i], 1ull);
        else atomicAdd(reinterpret_cast<unsigned long long*>(p.arrivals[i]), 1ull);
      }
    }
    STAMP(9);
  }
  // launch epoch (+ the device step counter of training launches): advanced by the LAST CTA to get here (ticket), i.e.
  // after every CTA of this launch has read them
  const bool last_phase = p.forward_only ? (p.phase_mask & 2) != 0 : (p.phase_mask & 4) != 0;
  if (last_phase && tid == 0) {
    const unsigned int ticket = atomicAdd(&fl[2], 1u);
    if (ticket + 1u == sync_target) {
      fl[3] = s_epoch + 1u;
      if (p.step_counter && !p.forward_only) *p.step_counter = step + 1ull;
    }
  }
#ifndef DTF_HOST_EMU
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_holder, 256);
#endif
  STAMP(10);
  if (ringer && last_phase) {
    unsigned long long* row = p.ring + (step % (unsigned long long)p.ring_cap) * 8ull;
    if (p.forward_only) row = p.ring + (unsigned long long)p.ring_cap * 8ull;      // one extra row: the last forward-only launch
    row[1] = rt_entry; row[2] = rt_token; row[3] = rt_fwd; row[4] = rt_head; row[5] = globaltimer_ns();
    row[6] = step; row[7] = (unsigned long long)p.G;
    row[0] = p.forward_only ? 3ull : 2ull;
  }
#undef STAMP
}

}  // namespace dtf

#ifndef DTF_HOST_EMU
namespace dtf {
// tensor-map cache of csrc/gemm_tcgen05.cu
int cached_map_f32(CUtensorMap* out, const void* ptr, long long rows, long long cols, long long ld, int box_cols, int box_rows,
                   int sw32);
}
#endif

extern "C" {
using namespace dtf;

struct DtfMlpStepArgs {
  int B, D, H, C;
  int G;                       // 0: auto
  int phase_mask;              // 0 -> 7 (fused)
  const float* x; long long ldx; long long x_rows;
  const float* labels; long long ldl;
  long long nbatches, bstride, boffset;
  const float* w1; long long ldw1;
  const float* b1;
  const float* w2; long long ldw2;
  const float* b2;
  float* hpart; float* dh; long long lddh; unsigned int* flags;
  float* gw1; long long ldgw1; float* gb1; float* gw2; long long ldgw2; float* gb2;
  float clip_min;
  float* loss_out; float* logits_out;
  unsigned long long* step_counter;
  int forward_only;
  int num_tokens; const unsigned long long* token[4]; unsigned long long token_scale[4]; unsigned long long token_base[4];
  int stamp_step;
  const unsigned long long* consumed[4];
  int num_signals; unsigned long long* arrivals[4]; unsigned long long* stamp_dst[4]; const unsigned long long* stamp_src[4];
  int sys_scope;
  unsigned long long timeout_ns;
  unsigned int* err;
  unsigned long long* trace;
  int no_cluster;              // 1: plain grid + L2 counters even when the CTAs would fit one cluster
  int dbg;
  unsigned long long* ring; int ring_cap;      // optional worker trace ring: (ring_cap + 1) rows of 8 u64
  float* head_part;            // [G][dtf_mlp_step_head_part_floats()] scratch (training launches)
};

// Slices: at least ceil(B / 16) CTAs (phase 2 finalises <= 16 batch rows per CTA), at most 16; among those the widest
// slice (a multiple of 8, <= 128) that divides D evenly, else the widest.  784 features, batch 100 -> 7 x 112.
int dtf_mlp_step_slices(int D, int B, int* ds_out) {
  const int g_min = (B + 15) / 16;
  int g_any = 0, ds_any = 0;
  for (int ds = 128; ds >= 8; ds -= 8) {
    const int g = (D + ds - 1) / ds;
    if (g > 16) break;
    if (g < g_min) continue;
    if (D % ds == 0) {
      if (ds_out) *ds_out = ds;
      return g;
    }
    if (!g_any) { g_any = g; ds_any = ds; }
  }
  if (!g_any) {            // few features: more CTAs than slices (the extra ones own empty slices and only do phase 2)
    g_any = g_min;
    ds_any = ((D + g_min - 1) / g_min + 7) / 8 * 8;
  }
  if (ds_out) *ds_out = ds_any;
  return g_any;
}

// scratch sizes (floats): hpart = G * 128 * (n1 + 4), dh = 128 * 128
long long dtf_mlp_step_scratch_floats(int D, int B, int H) {
  int ds = 0;
  const int g = dtf_mlp_step_slices(D, B, &ds);
  const int n1 = (H + 15) / 16 * 16;
  return (long long)g * 128 * (n1 + 4) + 128 * 128 + 64;
}

int dtf_mlp_step(const DtfMlpStepArgs* a, cudaStream_t s) {
  if (a->B < 1 || a->B > 128 || a->H < 1 || a->H > 128 || a->C < 1 || a->C > 16 || a->D < 8) return -2;
  if ((a->ldx % 4) || (a->ldw1 % 4) || (a->lddh % 4) || a->lddh < 128) return -3;
  MlpStepParams p;
  memset(&p, 0, sizeof(p));
  p.B = a->B; p.D = a->D; p.H = a->H; p.C = a->C;
  int ds = 0;
  int g = dtf_mlp_step_slices(a->D, a->B, &ds);
  if (a->G > 0) { g = a->G; ds = ((a->D + g - 1) / g + 7) / 8 * 8; }
  if (ds > 128 || ds < 8 || g > 64) return -2;
  p.G = g; p.ds = ds;
  p.rows_per_cta = (a->B + g - 1) / g;
  if (p.rows_per_cta > 16) return -2;
  p.phase_mask = a->phase_mask ? a->phase_mask : 7;
  p.n1 = (a->H + 15) / 16 * 16;
  p.n2 = (ds + 15) / 16 * 16;
  p.kb = (a->B + 7) / 8 * 8;
  p.x = a->x; p.ldx = a->ldx; p.labels = a->labels; p.ldl = a->ldl;
  p.nbatches = a->nbatches; p.bstride = a->bstride; p.boffset = a->boffset;
  p.w1 = a->w1; p.ldw1 = a->ldw1; p.b1 = a->b1; p.w2 = a->w2; p.ldw2 = a->ldw2; p.b2 = a->b2;
  p.hpart = a->hpart; p.dh = a->dh; p.lddh = a->lddh; p.flags = a->flags;
  p.gw1 = a->gw1; p.ldgw1 = a->ldgw1; p.gb1 = a->gb1; p.gw2 = a->gw2; p.ldgw2 = a->ldgw2; p.gb2 = a->gb2;
  p.head_part = a->head_part;
  if (!a->forward_only && a->head_part == nullptr) return -3;
  p.clip_min = a->clip_min; p.loss_out = a->loss_out; p.logits_out = a->logits_out;
  p.step_counter = a->step_counter; p.forward_only = a->forward_only;
  if (a->num_tokens > 4 || a->num_signals > 4) return -2;
  p.num_tokens = a->num_tokens;
  p.num_signals = a->num_signals;
  for (int i = 0; i < 4; ++i) {
    p.consumed[i] = a->consumed[i];
    p.token[i] = a->token[i]; p.token_scale[i] = a->token_scale[i] ? a->token_scale[i] : 1ull; p.token_base[i] = a->token_base[i]; p.arrivals[i] = a->arrivals[i]; p.stamp_dst[i] = a->stamp_dst[i]; p.stamp_src[i] = a->stamp_src[i];
  }
  p.sys_scope = a->sys_scope; p.stamp_step = a->stamp_step;
  p.timeout_ns = a->timeout_ns ? a->timeout_ns : 2000000000ull;
  p.err = a->err; p.trace = a->trace; p.dbg = a->dbg;
  p.ring = a->ring_cap > 0 ? a->ring : nullptr; p.ring_cap = a->ring_cap;
  const int nqx = (ds + 31) / 32, nq1 = (p.n1 + 31) / 32;
  const int w_region = (std::max(std::max(nq1 * ds * 128, 4 * p.kb * 128), 128 * (p.n1 + 4) * 4) + 1023) & ~1023;
  const size_t head_floats = 2 * 16 * 132 + 128 * 20 + 128 + 256 + 256 + 16;
  const size_t smem = 1024 + (size_t)nqx * kXChunkBytes + w_region + head_floats * 4;
#ifdef DTF_HOST_EMU
  const int masks[3] = {1, 2, 4};
  for (int ph = 0; ph < 3; ++ph) {
    if (!(p.phase_mask & masks[ph])) continue;
    MlpStepParams q = p;
    q.phase_mask = masks[ph];
    DTF_LAUNCH_SMEM(mlp_step_kernel, g, kStepThreads, smem, s, q);
  }
  return 0;
#else
  CUtensorMap mx, mx2, mw, md;
  // x: [rows, D] box {32 features, 128 rows}, once per swizzle (K-major A of F1 / MN-major B of B3);
  // W1: [D, H] box {32 units, ds rows}; dh: [128, 128] box {32 units, kb rows} -- both MN-major operands
  int rc = cached_map_f32(&mx, a->x, a->x_rows, a->D, a->ldx, 32, 128, 0);
  if (rc) return rc < 0 ? -7 : 1000 + rc;
  rc = cached_map_f32(&mx2, a->x, a->x_rows, a->D, a->ldx, 32, 128, 1);
  if (rc) return rc < 0 ? -7 : 1000 + rc;
  // W1 rows padded to whole 32-unit chunks (the engine's tf32 layout: zero padding that no update ever changes): describe
  // the padded width, so that every box row is one aligned, fully in-bounds 128-byte line
  const long long wcols = (a->ldw1 >= 32 * nq1) ? 32 * nq1 : a->H;
  rc = cached_map_f32(&mw, a->w1, a->D, wcols, a->ldw1, 32, ds, 1);
  if (rc) return rc < 0 ? -7 : 1000 + rc;
  rc = cached_map_f32(&md, a->dh, 128, 128, a->lddh, 32, p.kb, 1);
  if (rc) return rc < 0 ? -7 : 1000 + rc;
  static bool configured[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(mlp_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return 2000 + (int)e;
    configured[dev] = true;
  }
  if (smem > 200 * 1024) return -2;
  if (p.phase_mask == 7 && g <= 8 && !a->no_cluster) {
    // the G CTAs as ONE cluster (co-scheduled on one GPC): barrier.cluster orders the two exchanges
    p.clustered = 1;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(g, 1, 1);
    cfg.blockDim = dim3(kStepThreads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = g;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    // programmatic launch only where it was measured to pay: ps and worker on ONE GPU and stream (N = 1: 25.9 -> 24.6 us per
    // step).  Across GPUs the next step's prologue already hides under its token wait, so the launch path stays the plain one
    cfg.numAttrs = (pdl_enabled() && !a->sys_scope) ? 2 : 1;
    return (int)cudaLaunchKernelEx(&cfg, mlp_step_kernel, mx, mx2, mw, md, p);
  } else if (p.phase_mask == 7) {
    mlp_step_kernel<<<g, kStepThreads, smem, s>>>(mx, mx2, mw, md, p);
  } else {
    const int masks[3] = {1, 2, 4};
    for (int ph = 0; ph < 3; ++ph) {
      if (!(p.phase_mask & masks[ph])) continue;
      MlpStepParams q = p;
      q.phase_mask = masks[ph];
      // phase-by-phase launches leave the step counter to the last phase
      mlp_step_kernel<<<g, kStepThreads, smem, s>>>(mx, mx2, mw, md, q);
    }
  }
  return (int)cudaGetLastError();
#endif
}

int dtf_sizeof_mlp_step_args() { return (int)sizeof(DtfMlpStepArgs); }
int dtf_mlp_step_head_part_floats() { return kHeadPart; }

}  // extern "C"
