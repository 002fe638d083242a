// Row-block resident executor of recurrent_inference for both Hanabi networks (hanabizero_b200/plan.py; the function of
// /root/reference/core/model.py:74-84 over config/hanabi_control/model.py:127-335 in eval mode, BatchNorm folded):
// ONE launch per simulation in which every CTA owns 128 rows of the batch for the WHOLE chain
//
// MuZeroNetFull (Hanabi-Full, hz_rowchain_create):
//   y1 = relu(W1 [s | onehot(a)] + b1)  ->  y2 = relu(W2 y1 + b2)  ->  s' = relu(W3 y2 + b3 + s)            (dynamics)
//   value / reward:  relu(Wh1 s')  ->  relu(WB2 .)  ->  WB3 .   (201-wide support logits, padded to P3)
//   policy:          h = relu(Wh1 s')  ->  a1 = relu(WB2 h)  ->  a2 = relu(Wa2 a1 + h)  ->  WB3 a2
// MuZeroNet (Hanabi-Small, hz_rowchain_create_small; the skip joins after bn1, heads 128 wide, one layer each):
//   y1 = relu(W1 [s | onehot(a)] + b1 + s)  ->  y2 = relu(W2 y1 + b2)  ->  s' = relu(W3 y2 + b3)
//   h = relu(Wh1 s') = [value | reward | policy]  ->  WB3[i] h_i   (51 / 51 / 11 logits, padded to 64)
//
// Why this shape.  The seven library GEMMs of this chain are single waves of 128x128 tiles: every CTA pulls 256 KB of
// operands through its SM's ~165 GB/s L2 port for 1 us of tensor work, so at 4096 rows the whole device is held for
// 35 us by 9 us of math.  With several searches in flight (SearchPipeline) what counts is SM-time per simulation, not
// the latency of one chain.  Here the activations of a 128-row block never leave the SM: they sit in shared memory in
// the K-major 128-byte-swizzled layout tcgen05.mma reads, each layer's accumulators (128 x 512 fp32 = all 512 TMEM
// columns) are drained by the epilogue warps straight back into that layout, and only the weights stream in (3.2 MB
// per row block, L2-resident, TMA into a 3 x 32 KB ring).  A 4096-row batch occupies 32 SMs instead of 148.
//
//   warp 0      TMA producer: weight tiles [N <= 256 out-columns x 64 k] in the static order of the job table
//   warp 1      tcgen05.mma issuer (one lane), M = 128, N = 256 | 208 (Full) | 256 | 128 | 64 (Small), K = 16,
//               fp16 x fp16 -> fp32 in TMEM
//   warps 2-17  epilogue: tcgen05.ld -> + bias (+ residual) -> ReLU -> fp16 -> back into the activation tile (swizzled),
//               in place; one of its threads moves whole tiles between shared and global memory as bulk tensor copies
//               (s in, s' out to the pool and back in for the policy branch, logits out)
//
// The kernel walks a job table built on the host.  Hanabi-Full: ten phases, fc1 | fc2 | fc3 + s | value, reward first
// layers | their second layers | their logits | policy h | a1 | a2 | policy logits.  Hanabi-Small: six, fc1 + s | fc2 |
// fc3 | the three first layers (N 256 + 128) | value, reward logits | policy logits (N 64).  A phase = one or two jobs
// (one per TMEM half) of MMAs, then their drains; the next phase's first MMAs start as soon as the first job is drained
// (ready0).  Each job's weight map has a box of exactly its N rows (the producer's expect_tx counts N rows per K-block);
// create checks that and the table's other bounds on the host.  The kernel is instantiated per network (kSmall), so the
// Hanabi-Full launch runs none of Hanabi-Small's code.
//
// The one-hot action columns of fc1 are not multiplied: row r adds column a_r of W1's action block (a 32 x 512 or
// 16 x 512 table, W1aT) in the epilogue, which is the same sum.  Full: fc3's residual s is copied back into the
// consumed tile and read from shared memory; the value/reward branch runs first on the resident s', the policy branch
// re-reads s' (already stored to the pool) afterwards, because three 256-wide first layers need 768 TMEM columns.
// Small: fc1's residual s is fc1's own A operand, still in the tile when fc1 drains; its three first layers fit the
// 384 TMEM columns at once.
//
// fp16 plans of these two networks only (F = 512, H = 256 or 128); everything else stays on the library chain.
// Measurements, stamps and what bounds it: profiles/r02_rowchain.md (Full), profiles/r03_rowchain_small.md (Small).
#include <cuda.h>
#include <cuda_fp16.h>

#include <stdlib.h>
#include <string.h>

#include "hz_common.cuh"

namespace hz {

constexpr int kBM = 128, kBK = 64, kF = 512, kH = 256;
constexpr int kHSmall = 128, kP3Small = 64;        // Hanabi-Small: heads 128 wide, 51 support logits padded to 64
constexpr int kKB = kBM * kBK * 2;                 // one K-block of the activation tile: 128 rows x 128 bytes
constexpr int kActBytes = kBM * kF * 2;            // 128 KB: 8 K-blocks
constexpr int kWSlot = 256 * kBK * 2;              // 32 KB: a weight tile of up to 256 output columns x 64 k
constexpr int kWSlots = 3;
constexpr int kOffW = kActBytes, kOffAux = kOffW + kWSlots * kWSlot;
constexpr int kAuxBytes = 128 + 1024;              // barriers + the phase's biases (2 jobs x 256 halfs)
constexpr int kRowSmem = kOffAux + kAuxBytes + 1024;   // + alignment slack: 231 552 bytes (limit 232 448)
constexpr int kEpiWarps = 16, kEpiThreads = kEpiWarps * 32, kRowThreads = 64 + kEpiThreads;
constexpr int kMaxPhases = 10, kMaps = 10;          // 7 weight maps + x0, state, out
constexpr int kMapX0 = 7, kMapState = 8, kMapOut = 9;
constexpr unsigned kSpin = 1u << 26;               // a stuck wait traps instead of hanging the GPU

struct RowJob {
  int32_t map, n0, batch, num_k, a_kb, n, half;   // weight tile source, A K-block offset, MMA N, TMEM half
  int32_t relu, dst_kb;                           // dst_kb >= 0: write fp16 into activation K-blocks dst_kb..
  int32_t res, res_off;                           // 0 none | 1 W1aT[action] + res_off | 2 x0 hidden + res_off (global) | 3 tile K-block res_off
                                                  // | 4 W1aT[action] + n0 and tile K-block res_off
  int32_t gout, gb;                               // 0 none | 1 TMA-store the tile to `state` | 2 TMA-store K-blocks dst_kb.. to out[gb]
  int32_t kb1;                                    // MMA: K-blocks before this one need only the previous phase's FIRST job drained
  const __half* bias;
};
struct RowPhase {
  int32_t njobs, after;                           // after: 0 nothing | 1 reload s' | 2 load the next row block's s
  int32_t a_wait, res_load;                       // the MMAs also wait for a TMA-loaded activation tile | the drain first
                                                  // brings s back into the (consumed) tile as its residual
  RowJob job[2];
};
struct alignas(64) RowParams {
  CUtensorMap maps[kMaps];
  RowPhase phase[kMaxPhases];
  int32_t n_phases, rows, row_blocks, p3;
  const __half* x0; int64_t ld_x0;                // [rows][ld_x0]: 512 hidden | 32 (Full) or 16 (Small) one-hot columns
  const __half* w1a_t;                            // [32 or 16][512]
  __half* state;                                  // [rows][512]
  __half* out;                                    // [3][rows][p3]
  unsigned long long* trace;                      // optional [grid][kMaxPhases][4] globaltimer stamps
};

namespace rc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (unsigned spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (spin > kSpin) __trap();
  }
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
      ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_all_but_last() { asm volatile("cp.async.bulk.wait_group 1;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile, rows of 128 bytes, 128-byte swizzle: 8-row groups 1024 bytes apart (SBO), descriptor
// version 1 (sm_100), layout type 2 (SWIZZLE_128B).  +32 bytes along K = +2 in the start-address field.
__device__ __forceinline__ uint64_t umma_desc_k128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffffu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
// byte offset, inside the activation tile, of the 16-byte chunk holding columns [8 ch, 8 ch + 8) of row r
// (ch = 0..63): K-block ch / 8, 8-row group r / 8, row r % 8, chunk (ch % 8) XOR (r % 8)
__device__ __forceinline__ uint32_t act_off(int r, int ch) {
  return (uint32_t)((ch >> 3) * kKB + (r >> 3) * 1024 + (r & 7) * 128 + ((((ch & 7) ^ (r & 7))) << 4));
}
__device__ __forceinline__ void stamp(const RowParams& P, int phase, int slot) {
  if (P.trace) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    P.trace[((size_t)blockIdx.x * kMaxPhases + phase) * 4 + slot] = t;
  }
}

}  // namespace rc

using namespace rc;

// kSmall: the Hanabi-Small instantiation (16 one-hot columns, residual mode 4).  The Hanabi-Full one compiles without
// any of it, so Hanabi-Small costs the Full launch nothing.
template <bool kSmall>
__global__ void __launch_bounds__(kRowThreads, 1) k_row_chain(const __grid_constant__ RowParams P) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // swizzle-128B tiles need 1024-byte alignment
  const uint32_t act = base, wbase = base + kOffW, aux = base + kOffAux;
  auto w_full = [&](int s) { return aux + 8u * s; };
  auto w_empty = [&](int s) { return aux + 8u * (kWSlots + s); };
  auto acc_full = [&](int h) { return aux + 8u * (2 * kWSlots + h); };
  // epilogue -> MMA, per phase: ready0 = the first job is drained (its TMEM half is free, its K-blocks of the tile are
  // written), ready1 = the whole phase is (second job, stores, tile loads issued).  The next phase's first MMAs need
  // ready0 only, so the second job's drain runs under them.
  const uint32_t ready0 = aux + 8u * (2 * kWSlots + 2), ready1 = ready0 + 8u;
  const uint32_t a_full = ready1 + 8u;          // a TMA-loaded activation tile (s, or s' coming back) has landed
  const uint32_t res_full = a_full + 8u;        // ... the residual tile has landed (epilogue waits)
  const uint32_t tmem_slot = res_full + 8u;
  const uint32_t sbias = aux + 128u;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kWSlots; ++s) { mbar_init(w_full(s), 1); mbar_init(w_empty(s), 1); }
    mbar_init(acc_full(0), 1);
    mbar_init(acc_full(1), 1);
    mbar_init(ready0, kEpiWarps);
    mbar_init(ready1, kEpiWarps);
    mbar_init(a_full, 1);
    mbar_init(res_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int m = 0; m < kMaps; ++m) tma_prefetch_desc(&P.maps[m]);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  if (warp == 0) {
    // ===== weight producer: walks the job table, never waits for activations =====
    const bool leader = elect_one();
    uint32_t slot = 0, e_par = 0xffffffffu;   // fresh barrier: waiting for parity 1 passes
    for (int rb = blockIdx.x; rb < P.row_blocks; rb += gridDim.x) {
      for (int ph = 0; ph < P.n_phases; ++ph) {
        const RowPhase& F = P.phase[ph];
        for (int j = 0; j < F.njobs; ++j) {
          const RowJob& J = F.job[j];
          const uint32_t bytes = (uint32_t)J.n * (kBK * 2);
          for (int kb = 0; kb < J.num_k; ++kb) {
            mbar_wait(w_empty(slot), (e_par >> slot) & 1u);
            e_par ^= 1u << slot;
            if (leader) {
              mbar_expect_tx(w_full(slot), bytes);
              tma_load_3d(wbase + slot * kWSlot, &P.maps[J.map], w_full(slot), kb * kBK, J.n0, J.batch);
            }
            __syncwarp();
            if (++slot == kWSlots) slot = 0;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    const bool leader = elect_one();
    uint32_t slot = 0, f_par = 0, r0_par = 0, r1_par = 0, af_par = 0;
    bool first_rb = true;
    for (int rb = blockIdx.x; rb < P.row_blocks; rb += gridDim.x) {
      for (int ph = 0; ph < P.n_phases; ++ph) {
        const RowPhase& F = P.phase[ph];
        mbar_wait(ready0, r0_par);
        r0_par ^= 1u;
        tc_fence_after();
        bool got1 = false;
        auto need_all = [&]() {              // everything the previous phase wrote, drained and loaded
          mbar_wait(ready1, r1_par);
          r1_par ^= 1u;
          if (F.a_wait) {
            mbar_wait(a_full, af_par);
            af_par ^= 1u;
          }
          tc_fence_after();
          got1 = true;
        };
        if (leader && first_rb) stamp(P, ph, 0);
        for (int j = 0; j < F.njobs; ++j) {
          const RowJob& J = F.job[j];
          const uint32_t d_tmem = tmem_base + (uint32_t)J.half * 256u;
          const uint32_t idesc = (1u << 4) | ((uint32_t)(J.n >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
          uint64_t da = umma_desc_k128(act + (uint32_t)J.a_kb * kKB);
          for (int kb = 0; kb < J.num_k; ++kb) {
            if (!got1 && (j > 0 || kb >= J.kb1)) need_all();
            mbar_wait(w_full(slot), (f_par >> slot) & 1u);
            f_par ^= 1u << slot;
            tc_fence_after();
            if (leader) {
              const uint64_t dw = umma_desc_k128(wbase + slot * kWSlot);
#pragma unroll
              for (int k16 = 0; k16 < kBK / 16; ++k16) {
                tc_mma_f16(d_tmem, da + (uint64_t)(2 * k16), dw + (uint64_t)(2 * k16), idesc, (kb | k16) != 0);
              }
              tc_commit(w_empty(slot));
            }
            __syncwarp();
            da += (uint64_t)(kKB >> 4);
            if (++slot == kWSlots) slot = 0;
          }
          if (leader) tc_commit(acc_full(J.half));
          __syncwarp();
        }
        if (!got1) need_all();
        if (leader && first_rb) stamp(P, ph, 1);
      }
      first_rb = false;
    }
  } else {
    // ===== epilogue warps 2..17: TMEM lane quarter = warp % 4, the four warps of a quarter split the columns =====
    const int q = warp & 3, part = (warp - 2) >> 2, et = threadIdx.x - 64;
    const int rloc = q * 32 + lane;
    uint32_t a_par = 0;                        // bit h: parity of acc_full(h)'s next completion
    bool first_rb = true;
    // all traffic between the activation tile and global memory is bulk-asynchronous and issued by ONE thread (et 0):
    // loads of s / s' complete on a_full, stores of s' and of the logits are bulk groups it waits for before the tile
    // is reused
    auto load_tile = [&](int map, int rb_, uint32_t bar) {
      mbar_expect_tx(bar, kActBytes);
#pragma unroll
      for (int kb = 0; kb < kF / kBK; ++kb) tma_load_3d(act + kb * kKB, &P.maps[map], bar, kb * kBK, rb_ * kBM, 0);
    };
    uint32_t rf_par = 0, ea_par = 0;
    if (et == 0) load_tile(kMapX0, blockIdx.x, a_full);
    __syncwarp();
    if (lane == 0) { mbar_arrive(ready0); mbar_arrive(ready1); }
    for (int rb = blockIdx.x; rb < P.row_blocks; rb += gridDim.x) {
      const int row = rb * kBM + rloc;
      const bool live = row < P.rows;
      for (int ph = 0; ph < P.n_phases; ++ph) {
        const RowPhase& F = P.phase[ph];
        // ---- while the MMAs run: this phase's biases -> shared memory, residual rows resolved, first chunks requested
        if (et == 0) tma_wait_read_all();   // bulk stores issued so far have read the tile: it may be overwritten again
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");    // ... and the previous phase's bias readers are done
        {
          const int j = et >> 8, col = et & 255;
          if (j < F.njobs && col < F.job[j].n) {
            const unsigned short bv = __half_as_ushort(F.job[j].bias[col]);
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(sbias + 2u * et), "h"(bv) : "memory");
          }
        }
        const __half* crow[2] = {nullptr, nullptr};
        uint4 ef0 = make_uint4(0, 0, 0, 0), ef1 = ef0;    // job 0's first residual chunk, requested before the wait
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (j >= F.njobs) continue;
          const RowJob& J = F.job[j];
          if ((J.res == 1 || (kSmall && J.res == 4)) && live) {
            // only the row's own one-hot columns: past them lie the next row's state columns, and any of those that
            // is exactly 1.0 would read as an action
            const uint4* oh = reinterpret_cast<const uint4*>(P.x0 + (size_t)row * P.ld_x0 + kF);
            constexpr int n_oh = kSmall ? 2 : 4;   // 16-byte chunks of 8 one-hot columns
            int a = -1;
#pragma unroll
            for (int v = 0; v < 4; ++v) {
              if (v >= n_oh) break;               // (compile-time)
              const uint4 w = oh[v];
              const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                if ((u[t] & 0xffffu) == 0x3c00u) a = v * 8 + t * 2;
                if ((u[t] >> 16) == 0x3c00u) a = v * 8 + t * 2 + 1;
              }
            }
            if (a >= 0) crow[j] = P.w1a_t + (size_t)a * kF + (J.res == 1 ? J.res_off : J.n0);
          } else if (J.res == 2 && live) {
            crow[j] = P.x0 + (size_t)row * P.ld_x0 + J.res_off;
          }
          if (j == 0 && crow[0]) {   // (res 4: only warms L1 with the W1aT chunk; the residual read is the tile's)
            const int c0 = ((part * (J.n >> 4)) >> 2) * 16;
            ef0 = __ldg(reinterpret_cast<const uint4*>(crow[0] + c0));
            ef1 = __ldg(reinterpret_cast<const uint4*>(crow[0] + c0 + 8));
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");    // biases staged
        // every job of the phase must have finished reading the activation tile before any of it is overwritten
        for (int j = 0; j < F.njobs; ++j) {
          const int h = F.job[j].half;
          mbar_wait(acc_full(h), (a_par >> h) & 1u);
          a_par ^= 1u << h;
        }
        tc_fence_after();
        if (kSmall && F.a_wait) {
          // a residual read from the tile the TMA loaded for this phase: wait for that load here too, so the bulk
          // copy's writes are visible to these threads (the MMAs that read it have completed, so this never blocks)
          if (F.job[0].res == 4 || F.job[1].res == 4) mbar_wait(a_full, ea_par);
          ea_par ^= 1u;
        }
        if (et == 0 && first_rb) stamp(P, ph, 2);
        if (F.res_load) {
          // the tile has been consumed: the input state s comes back into it (bulk copy) and is read as the residual
          // at shared-memory speed, in place (each thread reads a chunk of s before it writes the same chunk of s')
          if (et == 0) load_tile(kMapX0, rb, res_full);
          mbar_wait(res_full, rf_par);
          rf_par ^= 1u;
        }
        bool any_store = false;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (j >= F.njobs) continue;
          const RowJob& J = F.job[j];
          const int n16 = J.n >> 4;
          const int c_begin = ((part * n16) >> 2) * 16, c_end = (((part + 1) * n16) >> 2) * 16;
          const uint32_t t_addr = tmem_base + (uint32_t)J.half * 256u + ((uint32_t)(q * 32) << 16);
          const uint32_t sb = sbias + (uint32_t)j * 512u;
          const __half* cr = crow[j];
          const int res = J.res, relu = J.relu, dst_kb = J.dst_kb, res_off = J.res_off;
          any_store |= J.gout != 0;
          // residual of columns [c, c + 16) of this thread's row (zero when the row has none)
          auto fetch_res = [&](int c, uint4& e0, uint4& e1) {
            if (res == 3 || (kSmall && res == 4)) {
              const int ch = res_off * 8 + (c >> 3);
              e0 = ld_shared_v4(act + act_off(rloc, ch));
              e1 = ld_shared_v4(act + act_off(rloc, ch + 1));
            } else if (cr) {
              e0 = __ldg(reinterpret_cast<const uint4*>(cr + c));
              e1 = __ldg(reinterpret_cast<const uint4*>(cr + c + 8));
            }
          };
          auto emit = [&](const uint32_t (&r)[16], const uint4& e0, const uint4& e1, int c) {
            const uint4 b0 = ld_shared_v4(sb + 2u * (uint32_t)c), b1 = ld_shared_v4(sb + 2u * (uint32_t)c + 16u);
            float v[16];
            const __half2* h0 = reinterpret_cast<const __half2*>(&b0);
            const __half2* h1 = reinterpret_cast<const __half2*>(&b1);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float2 f0 = __half22float2(h0[t]), f1 = __half22float2(h1[t]);
              v[2 * t] = __uint_as_float(r[2 * t]) + f0.x;
              v[2 * t + 1] = __uint_as_float(r[2 * t + 1]) + f0.y;
              v[8 + 2 * t] = __uint_as_float(r[8 + 2 * t]) + f1.x;
              v[8 + 2 * t + 1] = __uint_as_float(r[8 + 2 * t + 1]) + f1.y;
            }
            if (res != 0) {
              const __half2* g0 = reinterpret_cast<const __half2*>(&e0);
              const __half2* g1 = reinterpret_cast<const __half2*>(&e1);
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const float2 x0 = __half22float2(g0[t]), x1 = __half22float2(g1[t]);
                v[2 * t] += x0.x; v[2 * t + 1] += x0.y; v[8 + 2 * t] += x1.x; v[8 + 2 * t + 1] += x1.y;
              }
            }
            if (kSmall && res == 4 && cr) {   // fc1's action column on top of the state residual (L1-resident table)
              const uint4 w0 = __ldg(reinterpret_cast<const uint4*>(cr + c));
              const uint4 w1 = __ldg(reinterpret_cast<const uint4*>(cr + c + 8));
              const __half2* g0 = reinterpret_cast<const __half2*>(&w0);
              const __half2* g1 = reinterpret_cast<const __half2*>(&w1);
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const float2 x0 = __half22float2(g0[t]), x1 = __half22float2(g1[t]);
                v[2 * t] += x0.x; v[2 * t + 1] += x0.y; v[8 + 2 * t] += x1.x; v[8 + 2 * t + 1] += x1.y;
              }
            }
            uint4 o0, o1;
            __half2* p0 = reinterpret_cast<__half2*>(&o0);
            __half2* p1 = reinterpret_cast<__half2*>(&o1);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              p0[t] = __floats2half2_rn(v[2 * t], v[2 * t + 1]);
              p1[t] = __floats2half2_rn(v[8 + 2 * t], v[8 + 2 * t + 1]);
            }
            if (relu) {   // rounding is monotonic and keeps the sign: max(round(x), 0) == round(max(x, 0))
              // NaN stays NaN, as in the library chain's ReLU epilogue (plain __hmax2 would return the 0)
              const __half2 z = __float2half2_rn(0.0f);
#pragma unroll
              for (int t = 0; t < 4; ++t) { p0[t] = __hmax2_nan(p0[t], z); p1[t] = __hmax2_nan(p1[t], z); }
            }
            if (dst_kb >= 0) {
              const int ch = dst_kb * 8 + (c >> 3);
              st_shared_v4(act + act_off(rloc, ch), o0);
              st_shared_v4(act + act_off(rloc, ch + 1), o1);
            }
          };
          uint32_t ra[16], rb2[16];
          uint4 ea0 = ef0, ea1 = ef1, eb0 = make_uint4(0, 0, 0, 0), eb1 = eb0;
          if (j == 1 || res == 3 || (kSmall && res == 4)) {
            ea0 = ea1 = make_uint4(0, 0, 0, 0);
            fetch_res(c_begin, ea0, ea1);
          }
          // a warp may own no columns (jobs narrower than 64): it must not issue a load it never waits for
          if (c_begin < c_end) tc_ld16(t_addr + (uint32_t)c_begin, ra);
          for (int c = c_begin; c < c_end; c += 32) {
            tc_wait_ld();
            const bool more1 = c + 16 < c_end;
            if (more1) {                         // the next chunk's accumulators and residual travel while this one is processed
              tc_ld16(t_addr + (uint32_t)(c + 16), rb2);
              if (res != 0) fetch_res(c + 16, eb0, eb1);
            }
            emit(ra, ea0, ea1, c);
            if (more1) {
              tc_wait_ld();
              if (c + 32 < c_end) {
                tc_ld16(t_addr + (uint32_t)(c + 32), ra);
                if (res != 0) fetch_res(c + 32, ea0, ea1);
              }
              emit(rb2, eb0, eb1, c + 16);
            }
          }
          if (j == 0) {   // the first job's half of TMEM and its K-blocks of the tile are ready for the next phase
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(ready0);
          }
        }
        if (any_store || F.after != 0) {
          // the tile (s', or the staged logits) goes out as bulk tensor stores; what comes in next follows them
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
          if (et == 0) {
            for (int j = 0; j < F.njobs; ++j) {
              const RowJob& J = F.job[j];
              if (J.gout == 1 && j == 0) {
                for (int kb = 0; kb < kF / kBK; ++kb) tma_store_3d(&P.maps[kMapState], act + kb * kKB, kb * kBK, rb * kBM, 0);
              } else if (J.gout == 2) {
                for (int i = 0; i * kBK < P.p3; ++i)
                  tma_store_3d(&P.maps[kMapOut], act + (J.dst_kb + i) * kKB, i * kBK, rb * kBM, J.gb);
              }
            }
            if (any_store) tma_commit();
            if (F.after == 1) {
              // the value/reward branch is done with the tile: s' comes back for the policy branch once its own store
              // (an earlier group) is complete and the logits just issued have been read
              tma_wait_all_but_last();
              tma_wait_read_all();
              asm volatile("fence.proxy.async;" ::: "memory");
              load_tile(kMapState, rb, a_full);
            } else if (F.after == 2 && rb + (int)gridDim.x < P.row_blocks) {
              tma_wait_read_all();
              load_tile(kMapX0, rb + gridDim.x, a_full);
            }
          }
        }
        if (et == 0 && first_rb) stamp(P, ph, 3);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(ready1);
      }
      first_rb = false;
    }
  }

  if (threadIdx.x == 64) tma_wait_all();   // the bulk stores read this CTA's shared memory
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
  }
}

// ---- host side ----------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess) {
      p = nullptr;
    }
    cudaGetLastError();
    return (EncodeTiledFn)p;
  }();
  return fn;
}

// fp16 weights [batch][n][k] (nn.Linear layout) with row stride ld: box = [1][box_n][64], 128-byte swizzle
static bool make_w_map(CUtensorMap* map, const void* ptr, int64_t k, int64_t n, int64_t batch, int64_t ld, int box_n) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {(cuuint64_t)k, (cuuint64_t)n, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)(n * ld) * 2};
  cuuint32_t box[3] = {(cuuint32_t)kBK, (cuuint32_t)box_n, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The kernel trusts its job table.  The one invariant it cannot survive: the producer expects J.n * 128 bytes per
// K-block but a TMA load moves its map's whole box, so a box of other than J.n rows leaves a wait unsatisfied and the
// kernel traps (kSpin).  Checked on the host with the table's other bounds, so a wrong table is an argument error.
static const char* table_error(const RowParams& P, const int* box_rows, bool small) {
  for (int p = 0; p < P.n_phases; ++p) {
    const RowPhase& F = P.phase[p];
    for (int j = 0; j < F.njobs; ++j) {
      const RowJob& J = F.job[j];
      const int kbs = (J.n + kBK - 1) / kBK, tile_kbs = kF / kBK;
      if (J.map < 0 || J.map >= kMapX0 || box_rows[J.map] != J.n) return "a weight map's box is not the job's N rows";
      if (J.n < 16 || J.n > 256 || J.n % 16) return "N must be a multiple of 16 between 16 and 256";
      if (J.half < 0 || J.half > 1 || J.half * 256 + J.n > 512) return "accumulators past the 512 TMEM columns";
      if (J.num_k < 1 || J.a_kb < 0 || J.a_kb + J.num_k > tile_kbs) return "A operand K-blocks outside the tile";
      if (J.dst_kb >= 0 && J.dst_kb + kbs > tile_kbs) return "destination K-blocks outside the tile";
      if (J.res >= 3 && (J.res_off < 0 || J.res_off + kbs > tile_kbs)) return "residual K-blocks outside the tile";
      if (J.res == 4 && (!small || !F.a_wait)) return "a tile + action residual is Hanabi-Small's, in a phase with a_wait";
    }
  }
  return nullptr;
}

}  // namespace hz

using namespace hz;

struct hz_rowchain {
  int device = 0, grid = 0, sms = 0;
  bool small = false;                 // which job table (and kernel instantiation): Hanabi-Small or Hanabi-Full
  RowParams params;
  unsigned long long* trace = nullptr;
};

// Job table + weight maps of either network (arguments already checked by the entry points), then the launch setup.
static int rowchain_create(const char* who, bool small, hz_rowchain** out, int device, const hz_rowchain_weights* w,
                           int rows, const void* x0, int64_t ld_x0, void* state, void* out_logits) {
  const int p3 = w->logit_cols;
  // fp16 weights [batch][n][k] with row stride ld, loaded as boxes of `box` rows x 64 k (one per job's K-block)
  struct WMap { const void* ptr; int64_t k, n, batch, ld; int box; };
  WMap wm[kMapX0];
  if (!small) {
    wm[0] = {w->w1, kF, kF, 1, w->ld_w1, 256};       // action columns are added in the epilogue
    wm[1] = {w->w2, kF, kF, 1, kF, 256};
    wm[2] = {w->w3, kF, kF, 1, kF, 256};
    wm[3] = {w->wh1, kF, 3 * kH, 1, kF, 256};
    wm[4] = {w->wb2, kH, kH, 3, kH, 256};
    wm[5] = {w->wa2, kH, kH, 1, kH, 256};
    wm[6] = {w->wb3, kH, p3, 3, kH, p3};
  } else {
    wm[0] = {w->w1, kF, kF, 1, w->ld_w1, 256};
    wm[1] = {w->w2, kF, kF, 1, kF, 256};
    wm[2] = {w->w3, kF, kF, 1, kF, 256};
    wm[3] = {w->wh1, kF, 3 * kHSmall, 1, kF, 256};           // rows 0..255: value | reward
    wm[4] = {w->wh1, kF, 3 * kHSmall, 1, kF, 128};           // rows 256..383: actor
    wm[5] = {w->wb3, kHSmall, kP3Small, 3, kHSmall, kP3Small};
    wm[6] = wm[5];                                           // unused; a valid descriptor for the kernel's prefetch
  }
  int box_rows[kMapX0];
  for (int m = 0; m < kMapX0; ++m) box_rows[m] = wm[m].box;

  hz_rowchain* e = new hz_rowchain;
  e->device = device;
  RowParams& P = e->params;
  memset(&P, 0, sizeof(P));
  const __half *b1 = (const __half*)w->b1, *b2 = (const __half*)w->b2, *b3 = (const __half*)w->b3,
               *bh1 = (const __half*)w->bh1, *bb2 = (const __half*)w->bb2, *ba2 = (const __half*)w->ba2,
               *bb3 = (const __half*)w->bb3;
  auto job = [](int map, int n0, int batch, int num_k, int a_kb, int n, int half, const __half* bias, int relu,
                int dst_kb, int res = 0, int res_off = 0, int gout = 0, int gb = 0) {
    RowJob j;
    memset(&j, 0, sizeof(j));
    j.map = map; j.n0 = n0; j.batch = batch; j.num_k = num_k; j.a_kb = a_kb; j.n = n; j.half = half;
    j.bias = bias; j.relu = relu; j.dst_kb = dst_kb; j.res = res; j.res_off = res_off; j.gout = gout; j.gb = gb;
    return j;
  };
  int np = 0;
  auto phase = [&](int after, RowJob j0, const RowJob* j1 = nullptr, int a_wait = 0) {
    RowPhase& F = P.phase[np++];
    F.after = after; F.njobs = j1 ? 2 : 1; F.job[0] = j0; F.a_wait = a_wait;
    if (j1) F.job[1] = *j1;
  };
  RowJob t;
  if (!small) {
    // dynamics
    t = job(0, 256, 0, 8, 0, 256, 1, b1 + 256, 1, 4, 1, 256);  phase(0, job(0, 0, 0, 8, 0, 256, 0, b1, 1, 0, 1, 0), &t, 1);
    t = job(1, 256, 0, 8, 0, 256, 1, b2 + 256, 1, 4);          phase(0, job(1, 0, 0, 8, 0, 256, 0, b2, 1, 0), &t);
    t = job(2, 256, 0, 8, 0, 256, 1, b3 + 256, 1, 4, 3, 4, 1);
    phase(0, job(2, 0, 0, 8, 0, 256, 0, b3, 1, 0, 3, 0, 1), &t);
    P.phase[np - 1].res_load = 1;                                      // + s, reloaded into the consumed tile
    // value | reward branch on the resident s' (Wh1 rows: actor 0..255, value 256..511, reward 512..767)
    t = job(3, 512, 0, 8, 0, 256, 1, bh1 + 512, 1, 4);         phase(0, job(3, 256, 0, 8, 0, 256, 0, bh1 + 256, 1, 0), &t);
    t = job(4, 0, 2, 4, 4, 256, 1, bb2 + 512, 1, 4);           phase(0, job(4, 0, 1, 4, 0, 256, 0, bb2 + 256, 1, 0), &t);
    // the logits are staged in the (now idle) tile, K-blocks 0..3 / 4..7, and leave as bulk stores
    t = job(6, 0, 1, 4, 4, p3, 1, bb3 + p3, 0, 4, 0, 0, 2, 1);
    phase(1, job(6, 0, 0, 4, 0, p3, 0, bb3, 0, 0, 0, 0, 2, 0), &t);
    // policy branch on the reloaded s'
    phase(0, job(3, 0, 0, 8, 0, 256, 0, bh1, 1, 0), nullptr, 1);       // h  -> K-blocks 0..3
    phase(0, job(4, 0, 0, 4, 0, 256, 1, bb2, 1, 4));                   // a1 -> K-blocks 4..7
    phase(0, job(5, 0, 0, 4, 4, 256, 0, ba2, 1, 0, 3, 0));             // a2 = relu(Wa2 a1 + h) -> K-blocks 0..3
    phase(2, job(6, 0, 2, 4, 0, p3, 1, bb3 + 2 * p3, 0, 4, 0, 0, 2, 2));   // policy logits staged in K-blocks 4..7
  } else {
    // dynamics: fc1's skip s joins after bn1; s is fc1's own A operand, still in the tile when its drain runs
    t = job(0, 256, 0, 8, 0, 256, 1, b1 + 256, 1, 4, 4, 4);    phase(0, job(0, 0, 0, 8, 0, 256, 0, b1, 1, 0, 4, 0), &t, 1);
    t = job(1, 256, 0, 8, 0, 256, 1, b2 + 256, 1, 4);          phase(0, job(1, 0, 0, 8, 0, 256, 0, b2, 1, 0), &t);
    t = job(2, 256, 0, 8, 0, 256, 1, b3 + 256, 1, 4);          phase(0, job(2, 0, 0, 8, 0, 256, 0, b3, 1, 0, 0, 0, 1), &t);
    // the three heads' first layers on the resident s' (Wh1 rows: value 0..127, reward 128..255, actor 256..383)
    t = job(4, 256, 0, 8, 0, 128, 1, bh1 + 256, 1, 4);         phase(0, job(3, 0, 0, 8, 0, 256, 0, bh1, 1, 0), &t);
    // logits staged in tile K-blocks the heads no longer need (value 6, reward 7, then policy 0), out as bulk stores
    t = job(5, 0, 1, 2, 2, p3, 1, bb3 + p3, 0, 7, 0, 0, 2, 1);
    phase(0, job(5, 0, 0, 2, 0, p3, 0, bb3, 0, 6, 0, 0, 2, 0), &t);
    phase(2, job(5, 0, 2, 2, 4, p3, 0, bb3 + 2 * p3, 0, 0, 0, 0, 2, 2));
  }
  // how far a phase's first job may run on the previous phase's first job alone (see ready0 / ready1 in the kernel)
  for (int p = 0; p < np; ++p) {
    RowPhase& F = P.phase[p];
    F.job[0].kb1 = 0;
    F.job[1].kb1 = 0;
    if (p == 0 || F.a_wait) continue;
    const RowJob& A = P.phase[p - 1].job[0];
    RowJob& J = F.job[0];
    if (J.half != A.half || A.dst_kb < 0 || P.phase[p - 1].after != 0) continue;
    const int w0 = (A.n + kBK - 1) / kBK;
    int k = 0;
    while (k < J.num_k && J.a_kb + k >= A.dst_kb && J.a_kb + k < A.dst_kb + w0) ++k;
    J.kb1 = k;
  }
  P.n_phases = np;
  if (const char* bad = table_error(P, box_rows, small)) {
    delete e;
    set_error("%s: job table: %s", who, bad);
    return HZ_ERR_ARG;
  }
  DeviceGuard dg(device);
  if (!dg.ok) { delete e; set_error("%s: cannot select device %d", who, device); return HZ_ERR_CUDA; }
  if (!encode_fn()) { delete e; set_error("%s: cuTensorMapEncodeTiled unavailable", who); return HZ_ERR_CUDA; }
  bool ok = true;
  for (int m = 0; m < kMapX0; ++m)
    ok = ok && make_w_map(&P.maps[m], wm[m].ptr, wm[m].k, wm[m].n, wm[m].batch, wm[m].ld, wm[m].box);
  // activations: boxes of 128 rows x 64 columns, the K-blocks of the tile (rows past the end read as zero and are not
  // written)
  ok = ok && make_w_map(&P.maps[kMapX0], x0, kF, rows, 1, ld_x0, kBM) &&
       make_w_map(&P.maps[kMapState], state, kF, rows, 1, kF, kBM) &&
       make_w_map(&P.maps[kMapOut], out_logits, p3, rows, 3, p3, kBM);
  if (!ok) { delete e; set_error("%s: cuTensorMapEncodeTiled failed", who); return HZ_ERR_CUDA; }
  P.rows = rows;
  P.row_blocks = (rows + kBM - 1) / kBM;
  P.p3 = p3;
  P.x0 = (const __half*)x0;
  P.ld_x0 = ld_x0;
  P.w1a_t = (const __half*)w->w1a_t;
  P.state = (__half*)state;
  P.out = (__half*)out_logits;
  e->small = small;
  cudaError_t err = small ? cudaFuncSetAttribute(k_row_chain<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRowSmem)
                          : cudaFuncSetAttribute(k_row_chain<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRowSmem);
  cudaDeviceProp prop;
  if (err == cudaSuccess) err = cudaGetDeviceProperties(&prop, device);
  if (err != cudaSuccess) { delete e; return fail_cuda(err, who); }
  e->sms = prop.multiProcessorCount;
  e->grid = P.row_blocks < e->sms ? P.row_blocks : e->sms;
  *out = e;
  return HZ_OK;
}

extern "C" {
#pragma GCC visibility push(default)

int hz_rowchain_create(hz_rowchain** out, int device, const hz_rowchain_weights* w, int rows, const void* x0,
                       int64_t ld_x0, void* state, void* out_logits) {
  if (!out || !w || rows <= 0 || !x0 || !state || !out_logits) { set_error("hz_rowchain_create: bad argument"); return HZ_ERR_ARG; }
  if (w->state_cols != kF || w->head_cols != kH || w->onehot_cols != 32 || w->logit_cols <= 0 || w->logit_cols > 256 ||
      w->logit_cols % 16 || ld_x0 < kF + 32 || ld_x0 % 8 || w->ld_w1 < kF + 32 || w->ld_w1 % 8) {
    set_error("hz_rowchain_create: this executor is built for state 512 / heads 256 / one-hot 32 / logits <= 256 (multiple of 16)");
    return HZ_ERR_ARG;
  }
  const void* ptrs[] = {w->w1, w->w1a_t, w->b1, w->w2, w->b2, w->w3, w->b3, w->wh1, w->bh1, w->wb2, w->bb2,
                        w->wa2, w->ba2, w->wb3, w->bb3, x0, state, out_logits};
  for (const void* p : ptrs) {
    if (!p || ((uintptr_t)p & 15)) { set_error("hz_rowchain_create: null or unaligned pointer"); return HZ_ERR_ARG; }
  }
  return rowchain_create("hz_rowchain_create", false, out, device, w, rows, x0, ld_x0, state, out_logits);
}

int hz_rowchain_create_small(hz_rowchain** out, int device, const hz_rowchain_weights* w, int rows, const void* x0,
                             int64_t ld_x0, void* state, void* out_logits) {
  if (!out || !w || rows <= 0 || !x0 || !state || !out_logits) { set_error("hz_rowchain_create_small: bad argument"); return HZ_ERR_ARG; }
  if (w->state_cols != kF || w->head_cols != kHSmall || w->onehot_cols != 16 || w->logit_cols != kP3Small ||
      ld_x0 < kF + 16 || ld_x0 % 8 || w->ld_w1 < kF + 16 || w->ld_w1 % 8) {
    set_error("hz_rowchain_create_small: this executor is built for state 512 / heads 128 / one-hot 16 / logits 64");
    return HZ_ERR_ARG;
  }
  if (w->wb2 || w->bb2 || w->wa2 || w->ba2) {
    set_error("hz_rowchain_create_small: wb2 / bb2 / wa2 / ba2 belong to the Hanabi-Full heads and must be NULL");
    return HZ_ERR_ARG;
  }
  const void* ptrs[] = {w->w1, w->w1a_t, w->b1, w->w2, w->b2, w->w3, w->b3, w->wh1, w->bh1, w->wb3, w->bb3,
                        x0, state, out_logits};
  for (const void* p : ptrs) {
    if (!p || ((uintptr_t)p & 15)) { set_error("hz_rowchain_create_small: null or unaligned pointer"); return HZ_ERR_ARG; }
  }
  return rowchain_create("hz_rowchain_create_small", true, out, device, w, rows, x0, ld_x0, state, out_logits);
}

int hz_rowchain_destroy(hz_rowchain* e) {
  if (!e) return HZ_OK;
  DeviceGuard dg(e->device);
  if (e->trace) cudaFree(e->trace);
  delete e;
  return HZ_OK;
}

int hz_rowchain_set_state(hz_rowchain* e, void* state) {
  if (!e || !state || ((uintptr_t)state & 15)) { set_error("hz_rowchain_set_state: bad argument"); return HZ_ERR_ARG; }
  if (state == (void*)e->params.state) return HZ_OK;
  if (!make_w_map(&e->params.maps[kMapState], state, kF, e->params.rows, 1, kF, kBM)) {
    set_error("hz_rowchain_set_state: cuTensorMapEncodeTiled failed");
    return HZ_ERR_CUDA;
  }
  e->params.state = (__half*)state;
  return HZ_OK;
}

int hz_rowchain_set_trace(hz_rowchain* e, int enable) {
  if (!e) { set_error("hz_rowchain_set_trace: bad argument"); return HZ_ERR_ARG; }
  DeviceGuard dg(e->device);
  if (enable && !e->trace) {
    const size_t bytes = (size_t)e->sms * kMaxPhases * 4 * sizeof(unsigned long long);
    HZ_CUDA(cudaMalloc(&e->trace, bytes));
    HZ_CUDA(cudaMemset(e->trace, 0, bytes));
  }
  e->params.trace = enable ? e->trace : nullptr;
  return HZ_OK;
}

int hz_rowchain_read_trace(hz_rowchain* e, uint64_t* host_out, int64_t count) {
  if (!e || !e->trace || !host_out || count <= 0) { set_error("hz_rowchain_read_trace: no trace"); return HZ_ERR_ARG; }
  DeviceGuard dg(e->device);
  const int64_t have = (int64_t)e->grid * kMaxPhases * 4;
  HZ_CUDA(cudaMemcpy(host_out, e->trace, (size_t)(count < have ? count : have) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return HZ_OK;
}

int hz_rowchain_grid(const hz_rowchain* e) { return e ? e->grid : 0; }

int hz_rowchain_run(hz_rowchain* e, void* stream) {
  if (!e) { set_error("hz_rowchain_run: bad argument"); return HZ_ERR_ARG; }
  DeviceGuard dg(e->device);
  if (e->small) k_row_chain<true><<<e->grid, kRowThreads, kRowSmem, (cudaStream_t)stream>>>(e->params);
  else k_row_chain<false><<<e->grid, kRowThreads, kRowSmem, (cudaStream_t)stream>>>(e->params);
  HZ_LAUNCH_CHECK("k_row_chain");
  return HZ_OK;
}

#pragma GCC visibility pop
}  // extern "C"
