// mlp_dev.cuh -- constants, launch parameters and PTX wrappers shared by the tensor-core chain kernels
// (mlp_tc.cu: host side + legacy kernel; mlp_pipe.cu: role-specialised pipelined kernel).
#pragma once
#include <math_constants.h>

#include "common.cuh"

namespace prb {

constexpr int TM = 128;              // rows per tile (= TMEM lanes, UMMA M)
constexpr int KC = 32;               // K columns per chunk (128 bytes of fp32/tf32)
constexpr int A_STAGE_BYTES = TM * KC * 4;        // 16 KB
constexpr int B_TILE_ROWS = 256;                  // max N per MMA / per weight tile
constexpr int MAX_STAGES = 4;        // ring depth upper bound (runtime depth in ChainParams)
constexpr int MAX_LAYERS = 3;
constexpr int MAX_NP = 512;

enum { IN_SA = 0, IN_FP = 1, IN_DIRECT = 2 };
// kernel build of IN_SA whose gather warps evaluate layer 0 themselves (ChainParams.sa_l0); not a ChainParams.mode_in value
enum { IN_SA_L0 = 3 };
constexpr int L0_IN = 8;             // layer-0 inputs of the direct form: [dx, dy, dz, up to 5 feature channels]
enum { OUT_ROWS = 0, OUT_SA_MAX = 1, OUT_FP = 2 };

struct ChainParams {
    int mode_in, mode_out, num_layers;
    int nchunks[MAX_LAYERS];   // K chunks per layer
    int np[MAX_LAYERS];        // padded N (multiple of 32)
    int dcol[MAX_LAYERS];      // TMEM column of the accumulator
    const float *w[MAX_LAYERS];      // packed weight images
    const float *scale[MAX_LAYERS];  // np floats (zero padded); unused when unit_scale
    int w_resident;                  // 1: the weight rings hold a whole tile's stages, filled once (no recycling)
    int sleepy_ns;                   // poll interval of the run-ahead roles in the narrow builds (ns)
    int sleepy;                      // bit 0: MMA issuer waits with a suspend hint, bit 1: weight producer does
    int a_tmem;                      // layers >= 1 take their A operand from tensor memory: the epilogue rewrites the
                                     // previous accumulator IN PLACE (relu(x + t) -> tf32), no shared-memory stage, no proxy fence
    int trace;                       // debug: record phase time stamps (see g_trace)
    int unit_scale;                  // 1: the per-channel scale is folded into the packed weights, epilogues only add shift
    const float *shift[MAX_LAYERS];
    // resources (sized per launch so that small layers run several CTAs per SM)
    int na, nb;                // ring depths
    int b_stage_bytes;         // weight stage size = min(256, max np) * 128
    int tmem_cols;             // power of two >= 32
    int gather_mode;           // layer-0 row gather: 0 registers (+cvt.rna), 1 cp.async.cg, 2 cp.async.ca
    int linear_last;           // the last layer of the chain has no ReLU (heads: y = W x + shift)
    int round_out;             // OUT_ROWS: round to tf32 (intermediate segment of a split chain)
    // layer-0 K segments (each padded to a multiple of KC)
    int nseg, seg_chunks[2], seg_width[2];
    long total_rows;
    int num_tiles;
    // SA
    int n, npoint, ns, log_ns, c_feat;
    const float *xyz, *new_xyz, *feats_pm;
    const int *idx;
    // SA, layer 0 in the gather warps (c_feat <= 5): the gather warps write relu_tf32(W0 . [dxyz, f] + shift0) into the A
    // ring, so the tensor-core chain starts at the original layer 1 (K = l0_np).  l0_w: l0_c rows of L0_IN floats (BN scale
    // folded, not yet rounded), l0_shift: l0_c floats; padded to l0_np (multiple of KC) with zeros in shared memory
    int sa_l0, l0_c, l0_np;
    const float *l0_w, *l0_shift;
    // FP
    int m, c_known, c_skip;
    const float *known_pm, *weight, *skip;
    // DIRECT
    const float *x_rows;
    int x_pitch;
    const float *x2_rows;   // IN_DIRECT, second K segment (nullptr: one segment)
    int x2_pitch;
    // output
    float *out;
    float *out_pm;       // optional second copy of the final output in point-major layout (rows x out_stride_c)
    int c_last;          // true channel count of the last layer
    int out_stride_c, out_c_off, out_pitch;
    // ---- pipelined kernel (mlp_pipe.cu) only
    int rcol[MAX_LAYERS];            // TMEM column of the accumulator of layer l < num_layers-1 (each has its own region)
    int zcol[2], zs, nslice, nbuf;   // last layer: computed in `nslice` column slices of `zs` columns, `nbuf` TMEM buffers
    int nb0, nb1;                    // weight ring depths: layer 0 / layers >= 1
    int b0_stage_bytes, b1_stage_bytes;
    int b_rows;                      // rows of a weight stage = N of one MMA
    int nsplit, split_w;             // single-layer launches: a tile's output columns are dealt to `nsplit` work items
    int num_items;                   // num_tiles * nsplit
    int rows32;                      // total_rows as int (< 2^31, checked on the host)
    int pool_mode;                   // SA max-pool over 16 / 32 samples: 0 = CREDUX (one warp-wide max per channel), 1 = shuffle butterfly
};

// ------------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t s2u(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra D_%=;\n\t"
        "bra W_%=;\n\t"
        "D_%=:\n\t}" ::"r"(bar), "r"(parity)
        : "memory");
}
// same, with a suspend-time hint: the single producer / MMA-issuer threads should sleep in hardware instead of
// spinning in the issue slots of the row warps that share their scheduler
__device__ __forceinline__ void mbar_wait_sleepy(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra D_%=;\n\t"
        "bra W_%=;\n\t"
        "D_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(20000u)
        : "memory");
}
// one non-blocking probe of a phase (true = completed)
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// 16-byte asynchronous global->shared copy (LDGSTS); src_bytes = 0 zero-fills the destination
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async16_ca(uint32_t dst, const void *src, uint32_t src_bytes) {   // also allocates in L1
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {   // ncols: power of two >= 32
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, tf32 inputs, fp32 accumulate, M=128
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// same with the A operand in tensor memory: lane = row, one 32-bit column per K element (8 columns per K=8 step)
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns from registers (thread i writes lane base+i)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
        "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// arrives on the mbarrier once all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp receives lane (base+i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 16 lanes x 16 consecutive fp32 columns in the "quad" register layout (measured, scripts/micro/tmem_layout.cu): thread t gets
//   r0,r1 = row t/4,     columns 2(t%4), +1      r2,r3 = row t/4 + 8, same columns
//   r4,r5 = row t/4,     columns 8 + 2(t%4), +1  r6,r7 = row t/4 + 8, same columns
// i.e. a thread holds 2 rows x 4 columns instead of 1 row x 8 columns: a reduction over ROWS (max-pool over the samples of a
// centre) needs 3 cross-lane stages instead of 5.  No wait inside: issue both halves of a warp's 32 lanes, then tmem_ld_wait.
__device__ __forceinline__ void tmem_ld_quad16(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 32 consecutive 32-bit columns in one instruction each way
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
        "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
        "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
        "r"(r[31])
        : "memory");
}
// relu + round-to-nearest-even to tf32 in ONE instruction (F2FP.RELU.TF32.F32)
__device__ __forceinline__ float relu_to_tf32(float x) {
    uint32_t r;
    asm("cvt.rn.relu.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// round-to-nearest-even to tf32: one F2FP instruction (cvt.rna expands to a 4-instruction sequence)
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rn.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// UMMA shared-memory descriptor: K-major, SWIZZLE_128B, 8-row atoms of 1024 bytes (SBO), version 1
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);   // start address
    d |= (uint64_t)1 << 16;                         // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;               // stride byte offset
    d |= (uint64_t)1 << 46;                         // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                         // SWIZZLE_128B
    return d;
}
__host__ __device__ constexpr uint32_t make_idesc(int n) {
    // c=f32 (1<<4), a=tf32 (2<<7), b=tf32 (2<<10), a,b K-major, N>>3 at bit 17, M>>4 at bit 24
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
}
// byte offset of (row r, 16-byte unit j) inside a K-major SWIZZLE_128B stage
__device__ __forceinline__ uint32_t swz(int r, int j) { return (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4)); }

// Shared memory is carved at run time (ring depths and the weight-stage size depend on the chain), so that
// narrow layers (SA1/SA2) fit 2 CTAs per SM and overlap their latency-bound gathers.
// warp-level float max over the lanes named by MASK (CREDUX.MAX.F32: ~28 cycles dependent, pipelined when independent)
template <unsigned MASK>
__device__ __forceinline__ float redux_max_f32(float v) {
    float r;
    asm volatile("redux.sync.max.f32 %0, %1, %2;" : "=f"(r) : "f"(v), "n"(MASK));
    return r;
}

constexpr int POOL_STRIDE = 20;      // floats per row of the max-pool staging tile (80 B: conflict-free 128-bit stores)
struct SmemFixed {
    int row_src[TM][3];      // SA: global point row (slot 0); FP: 3 known rows
    float row_aux[TM][3];    // SA: centre xyz; FP: 3 weights
    int row_valid[TM];
    uint64_t a_full[MAX_STAGES], a_empty[MAX_STAGES], b_full[MAX_STAGES], b_empty[MAX_STAGES], d_full[MAX_LAYERS];
    uint32_t tmem_base;
};

__host__ __device__ inline size_t chain_smem_bytes(int ng, int na, int nb, int b_stage_bytes, int np_total) {
    return 1024 /*alignment slack*/ + (size_t)na * A_STAGE_BYTES + (size_t)nb * b_stage_bytes + (size_t)2 * np_total * sizeof(float) +
           (size_t)ng * (TM * POOL_STRIDE + 8 * 16) * sizeof(float) + sizeof(SmemFixed) + 64;
}

struct RingPos {
    uint32_t stage, phase;
    __device__ void advance(int depth) {
        if (++stage == (uint32_t)depth) { stage = 0; phase ^= 1; }
    }
};

// barrier over one row group (128 threads) / over all row threads
__device__ __forceinline__ void bar_group(int grp) {
    if (grp == 0) asm volatile("bar.sync 2, 128;" ::: "memory");
    else if (grp == 1) asm volatile("bar.sync 3, 128;" ::: "memory");
    else asm volatile("bar.sync 4, 128;" ::: "memory");
}
template <int NG>
__device__ __forceinline__ void bar_rows() { asm volatile("bar.sync 1, %0;" ::"n"(128 * NG) : "memory"); }

}  // namespace prb
