// mlp_pipe.cu -- the shared-MLP chain as a ROLE-SPECIALISED, tile-pipelined tcgen05 kernel.
//
// Same contract as the legacy kernel in mlp_tc.cu (gather -> SharedMLP layers -> max-pool / channel-major store;
// replaces pointnet2_utils.py:249-257 + pointnet2_modules.py:40-52,144-156 + pytorch_utils.py:5-101 for eval-mode
// forward), but the phases of consecutive 128-row tiles overlap instead of running one after another:
//
//   gather warps   (4*NGW) build the layer-0 A operand of tile i+1, i+2, ... in a shared-memory ring (K-major
//                  SWIZZLE_128B chunks of 32 K-columns) while the tensor core and the epilogue warps are still busy
//                  with tile i: neighbour-row gathers are L2 latency, and no longer hold tensor memory;
//   issuer A       (1 thread) layer-0 MMAs: A from the ring, accumulator region X of tensor memory;
//   issuer B       (1 thread) layers >= 1: A operand straight from tensor memory (the previous accumulator rewritten in
//                  place by the epilogue warps), own accumulator regions Y / Z -- so X is free again as soon as layer 1 has
//                  consumed it and tile i+1's layer 0 runs under tile i's later layers;
//   producers      (2 threads) stream pre-packed weight tiles with cp.async.bulk into two rings (layer 0 / layers >= 1);
//   epilogue warps (4*NE) mid layers: tcgen05.ld -> +shift -> relu -> tf32 -> tcgen05.st in place, chunk by chunk (the
//                  next layer's MMAs start on the first chunk); last layer: computed in column SLICES through one or two
//                  small TMEM buffers, so that pooling / storing slice s overlaps the MMAs of slice s+1 and a 256-wide
//                  last layer does not need 256 columns next to its 224-column input.
//
// Tensor-memory plan: region l < L-1 at rcol[l] (np[l] columns each), last layer: nbuf buffers of zs columns at zcol[].
// Hazards: X is released to issuer A by a tcgen05.commit of issuer B after layer 1's MMAs; regions written and read
// by issuer B alone are ordered by the in-order execution of one thread's MMAs; slice buffers cycle through
// z_full (commit) / z_free (epilogue arrive) barriers.
#include <type_traits>

#include <map>
#include <mutex>

#include "mlp_dev.cuh"

namespace prb {

constexpr int PIPE_MAX_A = 8;      // A-ring depth upper bound
constexpr int PIPE_MAX_B = 12;    // weight rings: many SMALL stages (64 rows x 128 B) -> enough bytes in flight to cover the L2 latency

struct PipeSmem {
    uint64_t a_full[PIPE_MAX_A], a_empty[PIPE_MAX_A];
    uint64_t b0_full[PIPE_MAX_B], b0_empty[PIPE_MAX_B], b1_full[PIPE_MAX_B], b1_empty[PIPE_MAX_B];
    uint64_t r_full[2];          // accumulator of mid layer l complete
    uint64_t x_free;             // region 0 consumed by layer 1
    uint64_t ready[2][16];       // chunk kc of region l rewritten as the next layer's A operand
    uint64_t z_full[2], z_free[2];
    uint32_t tmem_base;
    int row_src[2][TM][3];       // double-buffered by item parity. SA: global point row (slot 0); FP: 3 known rows
    float row_aux[2][TM][3];     // SA: centre xyz; FP: 3 weights
    int row_valid[2][TM];
};

// `pool`: the max-pool staging tiles exist only for SA outputs (the last region of the layout: other modes never touch it)
// `l0_np`: layer-0 channels evaluated by the gather warps (ChainParams.sa_l0), L0_IN weights + 1 shift each; 0 otherwise
__host__ __device__ inline size_t pipe_smem_bytes(int ne, int na, int nb0, int b0_bytes, int nb1, int b1_bytes, int np_total, bool pool,
                                                  int l0_np) {
    return 1024 /*alignment slack*/ + (size_t)na * A_STAGE_BYTES + (size_t)nb0 * b0_bytes + (size_t)nb1 * b1_bytes +
           (size_t)l0_np * (L0_IN + 1) * sizeof(float) + (size_t)2 * np_total * sizeof(float) +
           (pool ? (size_t)ne * (TM * POOL_STRIDE + 8 * 16) * sizeof(float) : 0) + 64;
}

// round to tf32, nearest with ties away from zero: the same bits as the host packer's tf32_rna_host (mlp_tc.cu), so that
// layer-0 weights evaluated on the CUDA cores are the operands the tensor core would have seen
__device__ __forceinline__ float tf32_rna_bits(float x) {
    uint32_t u = __float_as_uint(x);
    if ((u & 0x7f800000u) != 0x7f800000u) u += 0x1000u;
    return __uint_as_float(u & 0xffffe000u);
}

__device__ __forceinline__ void bar_named(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// position of a running element index inside consecutive segments ("scenes") of `period` elements: advanced by a
// constant stride per tile without any division in the loop
struct Cursor {
    int scene, pos, adv_scene, adv_pos, period;
    __device__ __forceinline__ void init(int start, int step, int per) {
        period = per;
        scene = start / per; pos = start - scene * per;
        adv_scene = step / per; adv_pos = step - adv_scene * per;
    }
    __device__ __forceinline__ void advance() {
        scene += adv_scene; pos += adv_pos;
        if (pos >= period) { pos -= period; ++scene; }
    }
    __device__ __forceinline__ void at(int off, int &sc, int &ps) const {
        sc = scene; ps = pos + off;
        while (ps >= period) { ps -= period; ++sc; }
    }
};

// The four single-role warps (two weight producers, two MMA issuers) run their loops WARP-UNIFORMLY and only the
// instruction that must come from one thread (bulk copy, tcgen05.mma, tcgen05.commit, expect_tx) sits under elect.sync.
// Inside `if (lane == 0) { loops }` every descriptor lives in vector registers and ptxas wraps each UTCHMMA / UBLKCP in an
// ELECT + 6 x R2UR.BROADCAST waterfall loop (~12 instructions per MMA, measured: the single-thread issue rate bounded the
// wide levels); with uniform control flow the operands stay in uniform registers.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// every wait parks the warp in hardware (try_wait with a suspend hint) instead of spinning in the issue slots
__device__ __forceinline__ void bwait(uint64_t *bar, uint32_t parity) { mbar_wait_sleepy(s2u(bar), parity); }
// roles that run AHEAD of their consumer (gather warps, weight producers: a full ring is the normal state) poll rarely:
// a try_wait wakes on every barrier event of the CTA, ~100 polls per tile and warp were 23 % of all issued instructions
// ... but only where the ring has slack (narrow chains, two CTAs per SM): on the wide chains the weight ring IS the critical
// resource and a 400 ns poll interval on 41 stage refills per tile cost 10 % (SA3 0.131 -> 0.144 ms)
__device__ __forceinline__ void bwait_lazy(uint64_t *bar, uint32_t parity, int lazy_ns) {
    const uint32_t b = s2u(bar);
    if (lazy_ns > 0) { while (!mbar_test(b, parity)) __nanosleep((unsigned)lazy_ns); }
    else mbar_wait_sleepy(b, parity);
}

// SA max-pool of one 16-column batch when the nsample rows of a centre are lanes of ONE warp (NS = 16 / 32).
// POOL 0: one warp-wide (half-warp-wide) CREDUX.MAX per channel, then every lane picks the channel named by its low four
// lane bits through a 15-select tree.  POOL 1: halving shuffle butterfly.  Returns the pooled value of channel `ch(lane)`.
template <int NS, int POOL>
__device__ __forceinline__ float pool_batch(float (&v)[16], int lane) {
    if (POOL == 0) {
        if (NS == 32) {
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = redux_max_f32<0xffffffffu>(v[q]);
        } else if (lane < 16) {
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = redux_max_f32<0x0000ffffu>(v[q]);
        } else {
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = redux_max_f32<0xffff0000u>(v[q]);
        }
        const bool b0 = lane & 1, b1 = lane & 2, b2 = lane & 4, b3 = lane & 8;
        float t8[8], t4[4];
#pragma unroll
        for (int i = 0; i < 8; ++i) t8[i] = b0 ? v[2 * i + 1] : v[2 * i];
#pragma unroll
        for (int i = 0; i < 4; ++i) t4[i] = b1 ? t8[2 * i + 1] : t8[2 * i];
        const float t20 = b2 ? t4[1] : t4[0], t21 = b2 ? t4[3] : t4[2];
        return b3 ? t21 : t20;                      // channel lane & 15
    }
    float w8[8], w4[4], w2[2], x;
    if (NS == 32) {
        const bool b4 = lane & 16;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float keep = b4 ? v[i + 8] : v[i], send = b4 ? v[i] : v[i + 8];
            w8[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 16));
        }
        const bool b3 = lane & 8;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float keep = b3 ? w8[i + 4] : w8[i], send = b3 ? w8[i] : w8[i + 4];
            w4[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 8));
        }
        const bool b2 = lane & 4;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float keep = b2 ? w4[i + 2] : w4[i], send = b2 ? w4[i] : w4[i + 2];
            w2[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 4));
        }
        const bool b1 = lane & 2;
        x = fmaxf(b1 ? w2[1] : w2[0], __shfl_xor_sync(0xffffffffu, b1 ? w2[0] : w2[1], 2));
        return fmaxf(x, __shfl_xor_sync(0xffffffffu, x, 1));      // channel (lane >> 1) & 15
    }
    const bool b3 = lane & 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float keep = b3 ? v[i + 8] : v[i], send = b3 ? v[i] : v[i + 8];
        w8[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 8));
    }
    const bool b2 = lane & 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float keep = b2 ? w8[i + 4] : w8[i], send = b2 ? w8[i] : w8[i + 4];
        w4[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 4));
    }
    const bool b1 = lane & 2;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const float keep = b1 ? w4[i + 2] : w4[i], send = b1 ? w4[i] : w4[i + 2];
        w2[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 2));
    }
    const bool b0 = lane & 1;
    return fmaxf(b0 ? w2[1] : w2[0], __shfl_xor_sync(0xffffffffu, b0 ? w2[0] : w2[1], 1));   // channel bit-reversed-ish, see caller
}

// Max-pool of 16 accumulator columns straight from tensor memory in the quad layout (tmem_ld_quad16): the warp's 32 rows are
// read as two 16-lane halves A (rows 0-15) and B (rows 16-31), a thread then owns rows {g, g+8} of each half (g = lane / 4)
// for the 4 columns col(k) = 2 (lane % 4) + (k & 1) + 8 (k >> 1).  `act(x, col)` is applied to every element first (identity
// when the activation commutes with the max and is applied after pooling).
//   NS == 32: one centre per warp -> 12 in-thread maxima, then 3 halving exchange stages over lane bits 4, 3, 2 (4 shuffles);
//             lanes with bit 2 clear own column  2 (lane % 4) + bit3 + 8 bit4
//   NS == 16: half A is centre 0, half B centre 1 -> 8 in-thread maxima, 7 shuffles; lane owns centre bit4, column
//             2 (lane % 4) + bit2 + 8 bit3
// ~30 / ~40 instructions per 16-column batch against ~80 for the one-row-per-thread layout (16 CREDUX + 16 UR->R + 15 selects).
template <int NS, class Act>
__device__ __forceinline__ float pool_quad(uint32_t taddr, int lane, Act &&act) {
    uint32_t A[8], B[8];
    tmem_ld_quad16(taddr, A);
    tmem_ld_quad16(taddr + (16u << 16), B);
    tmem_ld_wait();
    const int cb = 2 * (lane & 3);
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
    if (NS == 32) {
        float v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int q = (k & 1) + 4 * (k >> 1), col = cb + (k & 1) + 8 * (k >> 1);
            v[k] = fmaxf(fmaxf(act(__uint_as_float(A[q]), col), act(__uint_as_float(A[q + 2]), col)),
                         fmaxf(act(__uint_as_float(B[q]), col), act(__uint_as_float(B[q + 2]), col)));
        }
        float k0 = b4 ? v[2] : v[0], k1 = b4 ? v[3] : v[1];
        k0 = fmaxf(k0, __shfl_xor_sync(0xffffffffu, b4 ? v[0] : v[2], 16));
        k1 = fmaxf(k1, __shfl_xor_sync(0xffffffffu, b4 ? v[1] : v[3], 16));
        float x = fmaxf(b3 ? k1 : k0, __shfl_xor_sync(0xffffffffu, b3 ? k0 : k1, 8));
        return fmaxf(x, __shfl_xor_sync(0xffffffffu, x, 4));
    } else {
        float a[4], b[4], w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int q = (k & 1) + 4 * (k >> 1), col = cb + (k & 1) + 8 * (k >> 1);
            a[k] = fmaxf(act(__uint_as_float(A[q]), col), act(__uint_as_float(A[q + 2]), col));
            b[k] = fmaxf(act(__uint_as_float(B[q]), col), act(__uint_as_float(B[q + 2]), col));
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = fmaxf(b4 ? b[k] : a[k], __shfl_xor_sync(0xffffffffu, b4 ? a[k] : b[k], 16));
        const float u0 = fmaxf(b3 ? w[2] : w[0], __shfl_xor_sync(0xffffffffu, b3 ? w[0] : w[2], 8));
        const float u1 = fmaxf(b3 ? w[3] : w[1], __shfl_xor_sync(0xffffffffu, b3 ? w[1] : w[3], 8));
        return fmaxf(b2 ? u1 : u0, __shfl_xor_sync(0xffffffffu, b2 ? u0 : u1, 4));
    }
}

// optional wait-time trace (prb_options.mlp_trace): CTA 0 accumulates the cycles each role spends in each class of wait
// and the total cycles of its item loop; read back with prb_debug_pipe_trace.  Slots: 0 issuer A {x_free|z_free, a_full,
// b0_full, total}, 1 issuer B {z_free, ready, b1_full, total}, 2 producer 0 {b0_empty, total}, 3 producer 1 {b1_empty,
// total}, 4 gather warp 0 {a_empty, total}, 5 epilogue warp 0 {r_full, z_full, total}
__device__ long long g_pipe_trace[8][8];
__shared__ unsigned int s_trace_acc[8][8];             // [slot][class]: cycles, accumulated by lane 0 of the traced warps of CTA 0
struct TraceTimer {
    int slot;                                           // -1: not traced (one register; the sums live in shared memory)
    long long t0;
    __device__ __forceinline__ void start(bool enable, int slot_) {
        slot = enable ? slot_ : -1;
        t0 = enable ? clock64() : 0;
        if (enable && (threadIdx.x & 31) == 0)
            for (int k = 0; k < 8; ++k) s_trace_acc[slot_][k] = 0u;
    }
    template <class F>
    __device__ __forceinline__ void timed(int k, F &&f) {
        if (slot >= 0) {
            const long long t = clock64();
            f();
            if ((threadIdx.x & 31) == 0) s_trace_acc[slot][k] += (unsigned int)(clock64() - t);
        } else f();
    }
    __device__ __forceinline__ void finish() {
        if (slot < 0 || (threadIdx.x & 31) != 0) return;
        for (int k = 0; k < 7; ++k) g_pipe_trace[slot][k] = (long long)s_trace_acc[slot][k];
        g_pipe_trace[slot][7] = clock64() - t0;
    }
};

// registers per thread of each role.  Launch allocation = 65536 / (threads x CTAs per SM) rounded down to 8 (what
// __launch_bounds__ makes ptxas assume); the misc warpgroup releases down to MISC, the others raise to EPI / GATHER:
//   128 * (MISC + NE * EPI + NGW * GATHER) <= 65536 / MINB
template <int NE, int NGW, int MINB> struct RegPlan;
template <> struct RegPlan<1, 1, 2> { static constexpr int MISC = 56, EPI = 96, GATHER = 88; };     // 384 x 2: base 80
template <> struct RegPlan<2, 2, 1> { static constexpr int MISC = 56, EPI = 112, GATHER = 96; };    // 640: base 96
template <> struct RegPlan<1, 1, 3> { static constexpr int MISC = 40, EPI = 80, GATHER = 48; };     // 384 x 3: base 56 (narrow SA levels)
template <> struct RegPlan<2, 3, 1> { static constexpr int MISC = 56, EPI = 80, GATHER = 88; };     // 768: base 80
// BASE = the launch allocation (what ptxas pins the kernel at when setmaxnreg is present): raise or release relative to it
template <int BASE, int N>
__device__ __forceinline__ void reg_set() {
    if (N > BASE) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
    else if (N < BASE) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

template <int NE, int NGW, int MINB, int MIN, int MOUT>
__global__ void __launch_bounds__((NE + NGW + 1) * 128, MINB) mlp_pipe_kernel(const __grid_constant__ ChainParams p) {
    constexpr int NTHREADS = (NE + NGW + 1) * 128;
    constexpr int REG_BASE = (65536 / (NTHREADS * MINB)) / 8 * 8 > 255 ? 255 : (65536 / (NTHREADS * MINB)) / 8 * 8;
    static_assert(128 * (RegPlan<NE, NGW, MINB>::MISC + NE * RegPlan<NE, NGW, MINB>::EPI + NGW * RegPlan<NE, NGW, MINB>::GATHER) <= NTHREADS * REG_BASE,
                  "register plan exceeds the CTA's launch allocation");
    constexpr int W_GATHER = 4 * NE, W_MISC = 4 * (NE + NGW);
    extern __shared__ uint8_t smem_raw[];
    __shared__ PipeSmem S;
    uint8_t *base = smem_raw + ((1024u - (s2u(smem_raw) & 1023u)) & 1023u);
    const int L = p.num_layers;
    // offset of layer l's scale / shift inside the shared copies (no dynamically indexed local array: it would live on the stack)
    auto sc_off = [&](int l) { return l == 0 ? 0 : (l == 1 ? p.np[0] : p.np[0] + p.np[1]); };
    static_assert(MAX_LAYERS == 3, "sc_off assumes at most three layers");
    const int np_total = sc_off(L - 1) + p.np[L - 1];
    uint8_t *sA = base;
    uint8_t *sB0 = sA + (size_t)p.na * A_STAGE_BYTES;
    uint8_t *sB1 = sB0 + (size_t)p.nb0 * p.b0_stage_bytes;
    float *s_l0w = reinterpret_cast<float *>(sB1 + (size_t)p.nb1 * p.b1_stage_bytes);   // IN_SA_L0: l0_np x L0_IN weights
    float *s_l0sh = s_l0w + (size_t)p.l0_np * L0_IN;                                     // ... and l0_np shifts
    float *s_scale = s_l0sh + p.l0_np;
    float *s_shift = s_scale + np_total;
    float *s_pool = s_shift + np_total;                                  // NE x (TM x POOL_STRIDE + 8 x 16)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int i = 0; i < PIPE_MAX_A; ++i) { mbar_init(s2u(&S.a_full[i]), 128); mbar_init(s2u(&S.a_empty[i]), 1); }
        for (int i = 0; i < PIPE_MAX_B; ++i) {
            mbar_init(s2u(&S.b0_full[i]), 1); mbar_init(s2u(&S.b0_empty[i]), 1);
            mbar_init(s2u(&S.b1_full[i]), 1); mbar_init(s2u(&S.b1_empty[i]), 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(s2u(&S.r_full[i]), 1);
            mbar_init(s2u(&S.z_full[i]), 1); mbar_init(s2u(&S.z_free[i]), 128 * NE);
            for (int k = 0; k < 16; ++k) mbar_init(s2u(&S.ready[i][k]), 128);
        }
        mbar_init(s2u(&S.x_free), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == W_MISC + 2) tmem_alloc(s2u(&S.tmem_base), (uint32_t)p.tmem_cols);
    for (int l = 0; l < L; ++l)
        for (int i = tid; i < p.np[l]; i += NTHREADS) { s_scale[sc_off(l) + i] = p.unit_scale ? 1.f : p.scale[l][i]; s_shift[sc_off(l) + i] = p.shift[l][i]; }
    if (MIN == IN_SA_L0) {
        for (int i = tid; i < p.l0_np * L0_IN; i += NTHREADS) s_l0w[i] = (i / L0_IN) < p.l0_c ? tf32_rna_bits(p.l0_w[i]) : 0.f;
        for (int i = tid; i < p.l0_np; i += NTHREADS) s_l0sh[i] = i < p.l0_c ? p.l0_shift[i] : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = S.tmem_base;
    // work items: the grid is a multiple of nsplit, so a CTA keeps its column group and walks tiles with a fixed stride
    const int brows = p.b_rows;          // rows (output channels) per weight stage / per MMA
    const int nsplit = p.nsplit;
    const int sj = (int)blockIdx.x % nsplit;
    const int tile0 = (int)blockIdx.x / nsplit, tstep = (int)gridDim.x / nsplit;
    const int ntiles = p.num_tiles;
    const bool resident = p.w_resident != 0;   // all weight stages of a tile fit the rings: loaded once, never recycled (narrow chains)
    const int lazy = NE == 1 ? p.sleepy_ns : 0;   // the two-/three-CTA builds run the narrow chains: rings with slack -> poll interval in ns
    TraceTimer tt;
    // traced warps of CTA 0 (warp-uniform): issuer A -> slot 0, issuer B 1, producers 2 / 3, gather warp 0 -> 4, epilogue warp 0 -> 5
    tt.start(p.trace != 0 && blockIdx.x == 0 && (warp >= W_MISC || warp == W_GATHER || warp == 0),
             warp == W_MISC + 2 ? 0 : warp == W_MISC + 3 ? 1 : warp == W_MISC ? 2 : warp == W_MISC + 1 ? 3 : warp == W_GATHER ? 4 : 5);

    // Register budget per role (setmaxnreg, warpgroup granularity): the four single-thread roles give most of theirs
    // back, the epilogue and gather warps -- which hold 32-column accumulator chunks / 12 gathered float4 per lane --
    // take it (RegPlan).  Without this every thread of the CTA is allocated the same count and the row warps spill.
    if (warp >= W_MISC) {
    reg_set<REG_BASE, RegPlan<NE, NGW, MINB>::MISC>();
    if (warp == W_MISC) {
        // ===================================================== weight producer, layer 0
        {
            RingPos rb = {0, 0};
            const int col0 = sj * p.split_w;
            const int width = L == 1 ? min(p.split_w, p.np[0] - col0) : p.np[0];
            const int halves = (width + brows - 1) / brows;
            const int nch = p.nchunks[0], nb = p.nb0;
            const uint32_t stage_bytes = (uint32_t)p.b0_stage_bytes;
            const float *w0 = p.w[0] + (size_t)col0 * KC;
            const size_t chunk_stride = (size_t)p.np[0] * KC;
            for (int tile = tile0; tile < ntiles; tile += tstep) {
                if (p.w_resident && tile != tile0) break;      // every stage was filled once and is never recycled
                const float *src = w0;
                for (int kc = 0; kc < nch; ++kc, src += chunk_stride)
                    for (int h = 0; h < halves; ++h) {
                        const uint32_t bytes = (uint32_t)min(brows, width - h * brows) * KC * 4;
                        tt.timed(0, [&] { bwait_lazy(&S.b0_empty[rb.stage], rb.phase ^ 1, lazy); });
                        if (elect_one()) {
                            mbar_expect_tx(s2u(&S.b0_full[rb.stage]), bytes);
                            bulk_g2s(s2u(sB0) + rb.stage * stage_bytes, src + (size_t)h * brows * KC, bytes, s2u(&S.b0_full[rb.stage]));
                        }
                        rb.advance(nb);
                    }
            }
        }
    } else if (warp == W_MISC + 1) {
        // ===================================================== weight producer, layers >= 1
        if (L > 1) {
            RingPos rb = {0, 0};
            const int nb = p.nb1;
            const uint32_t stage_bytes = (uint32_t)p.b1_stage_bytes;
            for (int tile = tile0; tile < ntiles; tile += tstep) {
                if (p.w_resident && tile != tile0) break;
                for (int l = 1; l < L; ++l) {
                    const bool last = l == L - 1;
                    const int nsl = last ? p.nslice : 1;
                    const int width = last ? p.zs : p.np[l];
                    const int halves = (width + brows - 1) / brows;
                    const int nch = p.nchunks[l];
                    const size_t chunk_stride = (size_t)p.np[l] * KC;
                    for (int s = 0; s < nsl; ++s) {
                        const float *src = p.w[l] + (size_t)s * width * KC;
                        for (int kc = 0; kc < nch; ++kc, src += chunk_stride)
                            for (int h = 0; h < halves; ++h) {
                                const uint32_t bytes = (uint32_t)min(brows, width - h * brows) * KC * 4;
                                tt.timed(0, [&] { bwait_lazy(&S.b1_empty[rb.stage], rb.phase ^ 1, lazy); });
                                if (elect_one()) {
                                    mbar_expect_tx(s2u(&S.b1_full[rb.stage]), bytes);
                                    bulk_g2s(s2u(sB1) + rb.stage * stage_bytes, src + (size_t)h * brows * KC, bytes, s2u(&S.b1_full[rb.stage]));
                                }
                                rb.advance(nb);
                            }
                    }
                }
            }
        }
    } else if (warp == W_MISC + 2) {
        // ===================================================== MMA issuer A: layer 0 (A operand from the shared-memory ring)
        {
            RingPos ra = {0, 0}, rb = {0, 0};
            const int width = L == 1 ? min(p.split_w, p.np[0] - sj * p.split_w) : p.np[0];
            const int halves = (width + brows - 1) / brows;
            const int nch = p.nchunks[0], na = p.na, nb = p.nb0;
            const uint32_t a_base = s2u(sA), b_base = s2u(sB0), b_bytes = (uint32_t)p.b0_stage_bytes;
            const uint32_t nbuf = (uint32_t)p.nbuf;
            uint32_t it = 0;
            for (int tile = tile0; tile < ntiles; tile += tstep, ++it) {
                uint32_t dcol, buf = 0;
                if (L > 1) {
                    tt.timed(0, [&] { bwait(&S.x_free, (it & 1) ^ 1); });       // layer 1 of the previous item has consumed X
                    dcol = (uint32_t)p.rcol[0];
                } else {
                    buf = nbuf == 2 ? (it & 1) : 0u;
                    tt.timed(0, [&] { bwait(&S.z_free[buf], ((nbuf == 2 ? (it >> 1) : it) & 1) ^ 1); });
                    dcol = (uint32_t)p.zcol[buf];
                }
                tc_fence_after();
                for (int kc = 0; kc < nch; ++kc) {
                    int c = kc, sg = 0;
                    if (p.nseg > 1 && c >= p.seg_chunks[0]) { c -= p.seg_chunks[0]; sg = 1; }
                    const int ksteps = (min(KC, p.seg_width[sg] - c * KC) + 7) >> 3;
                    tt.timed(1, [&] { bwait(&S.a_full[ra.stage], ra.phase); });
                    const uint64_t adesc = make_desc(a_base + ra.stage * A_STAGE_BYTES);
                    for (int h = 0; h < halves; ++h) {
                        const int rows = min(brows, width - h * brows);
                        if (!(resident && it > 0)) tt.timed(2, [&] { bwait(&S.b0_full[rb.stage], rb.phase); });
                        tc_fence_after();
                        const uint64_t bdesc = make_desc(b_base + rb.stage * b_bytes);
                        const uint32_t idesc = make_idesc(rows);
                        const uint32_t d = tmem + dcol + (uint32_t)(h * brows);
                        if (elect_one()) {
                            for (int ks = 0; ks < ksteps; ++ks)  // +32 bytes (= 2 x 16 B) per K=8 step inside the swizzle row
                                umma_tf32(d, adesc + (uint64_t)(2 * ks), bdesc + (uint64_t)(2 * ks), idesc, (kc > 0 || ks > 0) ? 1u : 0u);
                            if (!resident) umma_commit(s2u(&S.b0_empty[rb.stage]));
                            if (h == halves - 1) umma_commit(s2u(&S.a_empty[ra.stage]));
                            if (h == halves - 1 && kc == nch - 1) umma_commit(L > 1 ? s2u(&S.r_full[0]) : s2u(&S.z_full[buf]));
                        }
                        rb.advance(nb);
                    }
                    ra.advance(na);
                }
            }
        }
    } else if (warp == W_MISC + 3) {
        // ===================================================== MMA issuer B: layers >= 1 (A operand from tensor memory)
        if (L > 1) {
            RingPos rb = {0, 0};
            const int nb = p.nb1;
            const uint32_t b_base = s2u(sB1), b_bytes = (uint32_t)p.b1_stage_bytes;
            const uint32_t nbuf = (uint32_t)p.nbuf, nslice = (uint32_t)p.nslice;
            uint32_t it = 0, u = 0;      // u: running slice number (buffer = u mod nbuf)
            for (int tile = tile0; tile < ntiles; tile += tstep, ++it) {
                for (int l = 1; l < L; ++l) {
                    const bool last = l == L - 1;
                    const uint32_t nsl = last ? nslice : 1u;
                    const int width = last ? p.zs : p.np[l];
                    const int halves = (width + brows - 1) / brows;
                    const int nch = p.nchunks[l];
                    const uint32_t a_col = tmem + (uint32_t)p.rcol[l - 1];
                    for (uint32_t s = 0; s < nsl; ++s) {
                        uint32_t dcol, buf = 0;
                        if (last) {
                            buf = nbuf == 2 ? (u & 1) : 0u;
                            tt.timed(0, [&] { bwait(&S.z_free[buf], ((nbuf == 2 ? (u >> 1) : u) & 1) ^ 1); });   // the epilogue has drained this buffer
                            dcol = (uint32_t)p.zcol[buf];
                            ++u;
                        } else {
                            dcol = (uint32_t)p.rcol[l];
                        }
                        for (int kc = 0; kc < nch; ++kc) {
                            if (s == 0) tt.timed(1, [&] { bwait(&S.ready[l - 1][kc], it & 1); });   // chunk kc of the A operand is in place
                            tc_fence_after();
                            const uint32_t a_t = a_col + (uint32_t)(kc * KC);
                            for (int h = 0; h < halves; ++h) {
                                const int rows = min(brows, width - h * brows);
                                if (!(resident && it > 0)) tt.timed(2, [&] { bwait(&S.b1_full[rb.stage], rb.phase); });
                                tt.timed(3, [&] { tc_fence_after(); });
                                const uint64_t bdesc = make_desc(b_base + rb.stage * b_bytes);
                                const uint32_t idesc = make_idesc(rows);
                                const uint32_t d = tmem + dcol + (uint32_t)(h * brows);
                                tt.timed(4, [&] {
                                    if (elect_one()) {
#pragma unroll
                                        for (int ks = 0; ks < 4; ++ks)
                                            umma_tf32_ts(d, a_t + (uint32_t)(8 * ks), bdesc + (uint64_t)(2 * ks), idesc, (kc > 0 || ks > 0) ? 1u : 0u);
                                    }
                                });
                                tt.timed(5, [&] {
                                    if (elect_one()) {
                                        if (!resident) umma_commit(s2u(&S.b1_empty[rb.stage]));
                                        if (h == halves - 1 && kc == nch - 1) {
                                            umma_commit(last ? s2u(&S.z_full[buf]) : s2u(&S.r_full[l]));
                                            // region 0 may take the next item's layer 0 once layer 1 (all its slices) has read it
                                            if (l == 1 && s + 1 == nsl) umma_commit(s2u(&S.x_free));
                                        }
                                    }
                                });
                                rb.advance(nb);
                            }
                        }
                    }
                }
            }
        }
    }
    } else if (warp >= W_GATHER) {
        reg_set<REG_BASE, RegPlan<NE, NGW, MINB>::GATHER>();
        // ===================================================== gather warps: layer-0 A chunks, running ahead of the MMAs
        const int gw = warp - W_GATHER;
        const int wq = gw & 3, grp = gw >> 2;
        const int r = wq * 32 + lane;       // my row inside the tile
        const int j8 = lane & 7;            // my 16-byte unit inside a 128-byte row
        const int rsub = lane >> 3;         // which of the 4 rows a warp-wide gather step covers
        const int na = p.na, nch0 = p.nchunks[0];
        const int rows = p.rows32;
        RingPos ra = {0, 0};
        uint32_t cc = 0, it = 0;
        Cursor cur;
        if (MIN == IN_SA || MIN == IN_SA_L0) cur.init(tile0 * (TM >> p.log_ns), tstep * (TM >> p.log_ns), p.npoint);
        else if (MIN == IN_FP) cur.init(tile0 * TM, tstep * TM, p.n);
        else cur.init(0, 0, 1);
        for (int tile = tile0; tile < ntiles; tile += tstep, ++it, cur.advance()) {
            const int R = tile * TM + r;
            const bool valid = R < rows;
            // ---- per-row metadata of this tile (registers; FP also a shared table: 8 lanes cooperate on one row)
            int src = -1;                     // SA: global point row of my sample (-1 = padding row)
            float cx = 0.f, cy = 0.f, cz = 0.f;
            int my_scene = 0, my_u = 0;
            const int par = it & 1;
            if (MIN == IN_SA || MIN == IN_SA_L0) {
                int sc, pp;
                cur.at(r >> p.log_ns, sc, pp);
                if (valid) {
                    src = sc * p.n + __ldg(p.idx + R);
                    const float *ctr = p.new_xyz + ((size_t)sc * p.npoint + pp) * 3;
                    cx = __ldg(ctr); cy = __ldg(ctr + 1); cz = __ldg(ctr + 2);
                }
            } else if (MIN == IN_FP) {
                cur.at(r, my_scene, my_u);
                int m_src[3] = {0, 0, 0};
                float m_w[3] = {0.f, 0.f, 0.f};
                if (valid) {
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        m_src[q] = my_scene * p.m + __ldg(p.idx + (size_t)R * 3 + q);
                        m_w[q] = __ldg(p.weight + (size_t)R * 3 + q);
                    }
                }
                if (grp == 0) {
                    S.row_valid[par][r] = valid;
#pragma unroll
                    for (int q = 0; q < 3; ++q) { S.row_src[par][r][q] = m_src[q]; S.row_aux[par][r][q] = m_w[q]; }
                }
                // one barrier per item: the table is double buffered, so the readers of item it-1 never see item it+1's rows
                bar_named(5, 128 * NGW);
            }
            // IN_SA_L0: my row's layer-0 inputs [dx, dy, dz, f0..f4], rounded to tf32 as the A operand of the MMA form is
            float in0[L0_IN];
            if (MIN == IN_SA_L0) {
#pragma unroll
                for (int k = 0; k < L0_IN; ++k) in0[k] = 0.f;
                if (valid) {
                    const float *q = p.xyz + (size_t)src * 3;
                    in0[0] = to_tf32(__ldg(q + 0) - cx);
                    in0[1] = to_tf32(__ldg(q + 1) - cy);
                    in0[2] = to_tf32(__ldg(q + 2) - cz);
                    const int cf = p.c_feat;
                    const float *f = p.feats_pm + (size_t)src * cf;
#pragma unroll
                    for (int k = 0; k < L0_IN - 3; ++k)
                        if (k < cf) in0[3 + k] = to_tf32(__ldg(f + k));
                }
            }
            // sources of the 8 rows my lane group helps to gather (rows of my own warp: shuffles instead of a table)
            int s8[8];
            if (MIN == IN_SA) {
#pragma unroll
                for (int i = 0; i < 8; ++i) s8[i] = __shfl_sync(0xffffffffu, src, rsub + 4 * i);
            } else if (MIN == IN_DIRECT) {
#pragma unroll
                for (int i = 0; i < 8; ++i) { const int rr = tile * TM + wq * 32 + rsub + 4 * i; s8[i] = rr < rows ? rr : -1; }
            }

            for (int kc = 0; kc < nch0; ++kc, ++cc, ra.advance(na)) {
                if (NGW > 1 && (int)(cc % NGW) != grp) continue;
                int c = kc, seg = 0;
                if (p.nseg > 1 && c >= p.seg_chunks[0]) { c -= p.seg_chunks[0]; seg = 1; }
                const int k0 = c * KC;                       // first column of this chunk inside its segment
                const int width = p.seg_width[seg];
                uint8_t *A = sA + (size_t)ra.stage * A_STAGE_BYTES;
                uint64_t *empty_bar = &S.a_empty[ra.stage];
                const uint32_t empty_par = ra.phase ^ 1;
                const bool rows_seg = (MIN == IN_DIRECT) || (MIN == IN_SA && seg == 0 && p.c_feat > 5) || (MIN == IN_FP && seg == 0);
                if (rows_seg) {
                    // point-major sources: 8 lanes cover one row's 128 bytes, a warp covers 4 rows per step, 8 steps.
                    // All loads of a (half) chunk are issued before the first use (memory-level parallelism).
                    const int kk = k0 + 4 * j8;
                    if (MIN == IN_FP) {
                        const int C = p.c_known;
                        const bool vec = (C & 3) == 0;
#pragma unroll
                        for (int half = 0; half < 2; ++half) {
                            float4 t0[4], t1[4], t2[4];
                            float w0[4], w1[4], w2[4];
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int rr = wq * 32 + rsub + 4 * (half * 4 + i);
                                t0[i] = t1[i] = t2[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                                w0[i] = S.row_aux[par][rr][0]; w1[i] = S.row_aux[par][rr][1]; w2[i] = S.row_aux[par][rr][2];
                                if (S.row_valid[par][rr] && kk < width) {
                                    const float *s0 = p.known_pm + (size_t)S.row_src[par][rr][0] * C + kk;
                                    const float *s1 = p.known_pm + (size_t)S.row_src[par][rr][1] * C + kk;
                                    const float *s2 = p.known_pm + (size_t)S.row_src[par][rr][2] * C + kk;
                                    if (vec) {
                                        t0[i] = __ldg((const float4 *)s0); t1[i] = __ldg((const float4 *)s1); t2[i] = __ldg((const float4 *)s2);
                                    } else {
                                        float a0[4], a1[4], a2[4];
#pragma unroll
                                        for (int q = 0; q < 4; ++q) {
                                            const bool in = kk + q < width;
                                            a0[q] = in ? __ldg(s0 + q) : 0.f; a1[q] = in ? __ldg(s1 + q) : 0.f; a2[q] = in ? __ldg(s2 + q) : 0.f;
                                        }
                                        t0[i] = make_float4(a0[0], a0[1], a0[2], a0[3]);
                                        t1[i] = make_float4(a1[0], a1[1], a1[2], a1[3]);
                                        t2[i] = make_float4(a2[0], a2[1], a2[2], a2[3]);
                                    }
                                }
                            }
                            if (half == 0) tt.timed(0, [&] { bwait_lazy(empty_bar, empty_par, lazy); });
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int rr = wq * 32 + rsub + 4 * (half * 4 + i);
                                // same contraction as three_interpolate (reference SASS): fma(w2,p2, fma(w0,p0, w1*p1))
                                float4 v;
                                v.x = to_tf32(__fmaf_rn(w2[i], t2[i].x, __fmaf_rn(w0[i], t0[i].x, __fmul_rn(w1[i], t1[i].x))));
                                v.y = to_tf32(__fmaf_rn(w2[i], t2[i].y, __fmaf_rn(w0[i], t0[i].y, __fmul_rn(w1[i], t1[i].y))));
                                v.z = to_tf32(__fmaf_rn(w2[i], t2[i].z, __fmaf_rn(w0[i], t0[i].z, __fmul_rn(w1[i], t1[i].z))));
                                v.w = to_tf32(__fmaf_rn(w2[i], t2[i].w, __fmaf_rn(w0[i], t0[i].w, __fmul_rn(w1[i], t1[i].w))));
                                *reinterpret_cast<float4 *>(A + swz(rr, j8)) = v;
                            }
                        }
                    } else {
                        const int pitch = MIN == IN_DIRECT ? (seg ? p.x2_pitch : p.x_pitch) : p.c_feat;
                        const float *srcbase = MIN == IN_DIRECT ? (seg ? p.x2_rows : p.x_rows) : p.feats_pm;
                        // 128-bit loads need 16-byte aligned rows (a column slice of wider rows is not)
                        const bool vec = ((pitch & 3) | (int)(reinterpret_cast<uintptr_t>(srcbase) & 15)) == 0;
                        float4 t[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            t[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (s8[i] >= 0 && kk < width) {
                                const float *sp = srcbase + (size_t)s8[i] * pitch + kk;
                                if (vec) {
                                    t[i] = __ldg((const float4 *)sp);
                                } else {
                                    float o[4];
#pragma unroll
                                    for (int q = 0; q < 4; ++q) o[q] = (kk + q < width) ? __ldg(sp + q) : 0.f;
                                    t[i] = make_float4(o[0], o[1], o[2], o[3]);
                                }
                            }
                        }
                        tt.timed(0, [&] { bwait_lazy(empty_bar, empty_par, lazy); });
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int rr = wq * 32 + rsub + 4 * i;
                            float4 v = t[i];
                            v.x = to_tf32(v.x); v.y = to_tf32(v.y); v.z = to_tf32(v.z); v.w = to_tf32(v.w);
                            *reinterpret_cast<float4 *>(A + swz(rr, j8)) = v;
                        }
                    }
                } else if (MIN == IN_SA_L0) {
                    // layer 0 on the CUDA cores, one row per lane: channels k0 .. k0+31 = relu_tf32(W0 . in0 + shift0), written
                    // as the 128-byte A row of the first MMA layer (the original layer 1).  Weights and shifts are broadcast
                    // shared-memory reads; padding channels have zero weights and shifts, padding rows are zero.
                    tt.timed(0, [&] { bwait_lazy(empty_bar, empty_par, lazy); });
                    const float4 *w4 = reinterpret_cast<const float4 *>(s_l0w + (size_t)k0 * L0_IN);
                    const float4 *sh4 = reinterpret_cast<const float4 *>(s_l0sh + k0);
                    auto chunk = [&](auto wide_c) {
                        constexpr bool WIDE = decltype(wide_c)::value;      // more than one feature channel: 8 inputs, else 4
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 b = sh4[j];
                            float o[4];
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float4 wa = w4[2 * (4 * j + q)];
                                float acc = __fmul_rn(wa.x, in0[0]);
                                acc = __fmaf_rn(wa.y, in0[1], acc);
                                acc = __fmaf_rn(wa.z, in0[2], acc);
                                acc = __fmaf_rn(wa.w, in0[3], acc);
                                if (WIDE) {
                                    const float4 wb = w4[2 * (4 * j + q) + 1];
                                    acc = __fmaf_rn(wb.x, in0[4], acc);
                                    acc = __fmaf_rn(wb.y, in0[5], acc);
                                    acc = __fmaf_rn(wb.z, in0[6], acc);
                                    acc = __fmaf_rn(wb.w, in0[7], acc);
                                }
                                const float t = q == 0 ? b.x : q == 1 ? b.y : q == 2 ? b.z : b.w;
                                o[q] = valid ? relu_to_tf32(acc + t) : 0.f;
                            }
                            *reinterpret_cast<float4 *>(A + swz(r, j)) = make_float4(o[0], o[1], o[2], o[3]);
                        }
                    };
                    if (p.c_feat > 1) chunk(std::true_type{});
                    else chunk(std::false_type{});
                } else if (MIN == IN_SA) {
                    // relative xyz segment: [x - cx, y - cy, z - cz, (<= 5 feature channels,) 0 ...]; one K=8 step
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f), v2 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (valid) {
                        const float *q = p.xyz + (size_t)src * 3;
                        v.x = to_tf32(__ldg(q + 0) - cx);
                        v.y = to_tf32(__ldg(q + 1) - cy);
                        v.z = to_tf32(__ldg(q + 2) - cz);
                        const int cf = p.c_feat;
                        if (cf > 0 && cf <= 5) {
                            const float *f = p.feats_pm + (size_t)src * cf;
                            v.w = to_tf32(__ldg(f));
                            if (cf > 1) v2.x = to_tf32(__ldg(f + 1));
                            if (cf > 2) v2.y = to_tf32(__ldg(f + 2));
                            if (cf > 3) v2.z = to_tf32(__ldg(f + 3));
                            if (cf > 4) v2.w = to_tf32(__ldg(f + 4));
                        }
                    }
                    tt.timed(0, [&] { bwait_lazy(empty_bar, empty_par, lazy); });
                    *reinterpret_cast<float4 *>(A + swz(r, 0)) = v;
                    *reinterpret_cast<float4 *>(A + swz(r, 1)) = v2;
                } else if (MIN == IN_FP) {
                    // FP skip segment: channel-major (b, c_skip, n); lanes run along consecutive points
                    const float *bsrc = p.skip + (size_t)my_scene * p.c_skip * p.n + my_u;
                    float o[32];
#pragma unroll
                    for (int q = 0; q < 32; ++q) {
                        const int ch = k0 + q;
                        o[q] = (valid && ch < width) ? __ldg(bsrc + (size_t)ch * p.n) : 0.f;
                    }
                    tt.timed(0, [&] { bwait_lazy(empty_bar, empty_par, lazy); });
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float4 *>(A + swz(r, j)) =
                            make_float4(to_tf32(o[4 * j]), to_tf32(o[4 * j + 1]), to_tf32(o[4 * j + 2]), to_tf32(o[4 * j + 3]));
                }
                fence_async_smem();
                mbar_arrive(s2u(&S.a_full[ra.stage]));
            }
        }
    } else {
        reg_set<REG_BASE, RegPlan<NE, NGW, MINB>::EPI>();
        // ===================================================== epilogue warps (warps 0 .. 4*NE-1)
        const int wq = warp & 3, grp = warp >> 2;
        const int r = wq * 32 + lane;       // my row inside the tile / my TMEM lane
        const uint32_t trow = tmem + ((uint32_t)(wq * 32) << 16);
        float *pool = s_pool + grp * (TM * POOL_STRIDE + 128);
        float *pool2 = pool + TM * POOL_STRIDE;   // 8 x 16 partial maxima (nsample > 32)
        const int Cl = p.c_last;
        const int rows = p.rows32;
        const float *sc = s_scale + sc_off(L - 1), *sh = s_shift + sc_off(L - 1);
        const bool unit = p.unit_scale != 0;
        const bool pool_raw = unit && MOUT == OUT_SA_MAX;
        const float lo = p.linear_last ? -CUDART_INF_F : 0.f;    // ReLU = max(., 0); a linear last layer keeps the sign
        const uint32_t nbuf = (uint32_t)p.nbuf;
        const int nsl = L == 1 ? 1 : p.nslice;
        const int slice_w = L == 1 ? p.split_w : p.zs;
        const int ns = p.ns;
        // mid layer l of item number `itn`: accumulator -> +shift -> ReLU -> tf32, rewritten in place as the next layer's A operand
        auto mid_epilogue = [&](int l, uint32_t itn) {
            tt.timed(0, [&] { bwait(&S.r_full[l], itn & 1); });
            tc_fence_after();
            const int nch = p.np[l] / KC;
            const uint32_t col0 = trow + (uint32_t)p.rcol[l];
            for (int kc = grp; kc < nch; kc += NE) {
                uint32_t acc[32];
                tmem_ld32(col0 + (uint32_t)(kc * KC), acc);
                const float4 *sh4 = reinterpret_cast<const float4 *>(s_shift + sc_off(l) + kc * KC);
                if (unit) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 b = sh4[j];                 // broadcast LDS.128
                        acc[4 * j + 0] = __float_as_uint(relu_to_tf32(__uint_as_float(acc[4 * j + 0]) + b.x));
                        acc[4 * j + 1] = __float_as_uint(relu_to_tf32(__uint_as_float(acc[4 * j + 1]) + b.y));
                        acc[4 * j + 2] = __float_as_uint(relu_to_tf32(__uint_as_float(acc[4 * j + 2]) + b.z));
                        acc[4 * j + 3] = __float_as_uint(relu_to_tf32(__uint_as_float(acc[4 * j + 3]) + b.w));
                    }
                } else {
                    const float4 *sc4 = reinterpret_cast<const float4 *>(s_scale + sc_off(l) + kc * KC);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 a = sc4[j], b = sh4[j];
                        acc[4 * j + 0] = __float_as_uint(relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 0]), a.x, b.x)));
                        acc[4 * j + 1] = __float_as_uint(relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 1]), a.y, b.y)));
                        acc[4 * j + 2] = __float_as_uint(relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 2]), a.z, b.z)));
                        acc[4 * j + 3] = __float_as_uint(relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 3]), a.w, b.w)));
                    }
                }
                tmem_st32(col0 + (uint32_t)(kc * KC), acc);
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(s2u(&S.ready[l][kc]));
            }
        };
        // Skewed order: the first mid layer of item i+1 is handled BEFORE the last layer of item i.  Item i+1's layer-0
        // accumulator is complete by then (region X was released when layer 1 of item i had run), so the round trips
        // "rewritten chunk -> next layer's MMAs -> commit" of one item are covered by epilogue work of its neighbour
        // instead of idling the epilogue warps.  Not when the last layer IS layer 1 and has more slices than buffers:
        // X is released only after the last slice, which needs this item's final epilogue to drain buffers first.
        const bool skew = (L == 3) || (L == 2 && p.nslice <= p.nbuf);
        Cursor cur;
        if (MOUT == OUT_SA_MAX) cur.init(tile0 * (TM >> p.log_ns), tstep * (TM >> p.log_ns), p.npoint);
        else if (MOUT == OUT_FP) cur.init(tile0 * TM, tstep * TM, p.n);
        else cur.init(0, 0, 1);
        uint32_t it = 0, u = 0;
        int pool_par = 0;
        if (skew && tile0 < ntiles) mid_epilogue(0, 0u);
        for (int tile = tile0; tile < ntiles; tile += tstep, ++it, cur.advance()) {
            const int R = tile * TM + r;
            const bool valid = R < rows;
            if (skew) {
                for (int l = 1; l + 1 < L; ++l) mid_epilogue(l, it);
                if (tile + tstep < ntiles) mid_epilogue(0, it + 1);
            } else {
                for (int l = 0; l + 1 < L; ++l) mid_epilogue(l, it);
            }

            // ---- last layer, slice by slice: per-row output coordinates first
            size_t off_cm = 0, off_pm = 0;   // SA: (scene, centre) of my row / my 16-row segment; FP: (scene, point); ROWS: row
            bool ok = valid;
            if (MOUT == OUT_SA_MAX) {
                // 16 / 32 samples: the centre of my own row; other sample counts: the centre of my 16-row segment
                const int rowc = (ns >= 16) ? r : (r & ~15);
                int scn, pp;
                cur.at(rowc >> p.log_ns, scn, pp);
                ok = tile * TM + rowc < rows;
                off_cm = ((size_t)scn * p.out_stride_c + p.out_c_off) * p.npoint + pp;
                off_pm = ((size_t)scn * p.npoint + pp) * p.out_stride_c + p.out_c_off;
            } else if (MOUT == OUT_FP) {
                int scn, uu;
                cur.at(r, scn, uu);
                off_cm = ((size_t)scn * p.out_stride_c + p.out_c_off) * p.n + uu;
                off_pm = (size_t)R * p.out_stride_c + p.out_c_off;
            } else {
                off_cm = (size_t)R * p.out_pitch;
            }
            for (int s = 0; s < nsl; ++s, ++u) {
                const uint32_t buf = nbuf == 2 ? (u & 1) : 0u;
                const int s_lo = L == 1 ? sj * slice_w : s * slice_w;                  // first absolute column of this slice
                const int s_hi = min(Cl, s_lo + slice_w);
                tt.timed(1, [&] { bwait(&S.z_full[buf], (nbuf == 2 ? (u >> 1) : u) & 1); });
                tc_fence_after();
                const uint32_t zc = trow + (uint32_t)p.zcol[buf];
                if (MOUT == OUT_SA_MAX && (ns == 64 || ns == 128) && p.pool_mode != 3) {
                    // ---- 64 / 128 samples (RCNN stage): a centre spans 2 / 4 warps.  Every warp pools its 32 rows (quad layout,
                    // or the warp-wide reduction with pool_mode 2), the partial maxima of a centre's warps meet in a tiny
                    // double-buffered shared tile (one named barrier per batch instead of a 128 x 16 staging tile and three barriers)
                    const int wpc = ns >> 5;                          // warps per centre
                    const bool head = (wq & (wpc - 1)) == 0;
                    const bool quad = p.pool_mode == 0;
                    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
                    const int ch = quad ? 2 * (lane & 3) + (b3 ? 1 : 0) + (b4 ? 8 : 0) : (lane & 15);
                    const bool own = quad ? !b2 : lane < 16;          // lanes that hold a distinct column of the batch
                    const int c_first = s_lo + grp * 16;
                    float *ocm = p.out + off_cm + (size_t)(c_first + ch) * p.npoint;
                    float *opm = p.out_pm ? p.out_pm + off_pm + c_first + ch : nullptr;
                    const size_t cm_step = (size_t)(16 * NE) * p.npoint;
                    const float *shp = sh + c_first + ch;
                    uint32_t taddr = zc + (uint32_t)(c_first - s_lo);
                    const int n_ok = Cl - ch;
                    // pool_par toggles with EVERY batch of the kernel's lifetime (not per slice): a warp that runs ahead into the
                    // next slice must not overwrite the buffer its centre's head warp is still reading
                    for (int c0 = c_first; c0 < s_hi; c0 += 16 * NE, ocm += cm_step, shp += 16 * NE, taddr += 16 * NE, opm += (opm ? 16 * NE : 0), pool_par ^= 1) {
                        float x;
                        if (quad) {
                            if (pool_raw) {
                                x = pool_quad<32>(taddr, lane, [](float v, int) { return v; });
                            } else {
                                const float *sc0 = sc + c0, *sh0 = sh + c0;
                                x = pool_quad<32>(taddr, lane, [&](float v, int col) { return fmaxf(fmaf(v, sc0[col], sh0[col]), lo); });
                            }
                        } else {
                            uint32_t acc[16];
                            tmem_ld16(taddr, acc);
                            float v[16];
                            if (pool_raw) {
#pragma unroll
                                for (int q = 0; q < 16; ++q) v[q] = __uint_as_float(acc[q]);
                            } else {
                                const float4 *sh4 = reinterpret_cast<const float4 *>(sh + c0), *sc4 = reinterpret_cast<const float4 *>(sc + c0);
#pragma unroll
                                for (int j = 0; j < 4; ++j) {
                                    const float4 a = sc4[j], b = sh4[j];
                                    v[4 * j + 0] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 0]), a.x, b.x), lo);
                                    v[4 * j + 1] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 1]), a.y, b.y), lo);
                                    v[4 * j + 2] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 2]), a.z, b.z), lo);
                                    v[4 * j + 3] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 3]), a.w, b.w), lo);
                                }
                            }
                            x = pool_batch<32, 0>(v, lane);                    // max over my warp's 32 rows, channel lane & 15
                        }
                        float *tile2 = pool2 + pool_par * 64;                   // [4 warps][16 channels]
                        if (own) tile2[wq * 16 + ch] = x;
                        bar_named(2 + grp, 128);
                        if (head) {
                            for (int w2 = 1; w2 < wpc; ++w2) x = fmaxf(x, tile2[(wq + w2) * 16 + ch]);
                            if (pool_raw) x = fmaxf(x + *shp, lo);
                            if (ok && own && c0 < n_ok) {
                                *ocm = x;
                                if (opm) *opm = x;
                            }
                        }
                    }
                } else if (MOUT == OUT_SA_MAX && (ns == 32 || ns == 16)) {
                    // ---- fast path: dispatched ONCE per slice on (nsample, pooling kind); everything that does not depend on
                    // the 16-column batch is computed before the batch loop
                    auto quad_loop = [&](auto ns_c) {
                        constexpr int NSC = decltype(ns_c)::value;
                        const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
                        const int ch = 2 * (lane & 3) + (NSC == 32 ? (b3 ? 1 : 0) + (b4 ? 8 : 0) : (b2 ? 1 : 0) + (b3 ? 8 : 0));
                        const bool st_lane = ok && (NSC == 16 || !b2);
                        const int c_first = s_lo + grp * 16;
                        float *ocm = p.out + off_cm + (size_t)(c_first + ch) * p.npoint;
                        float *opm = p.out_pm ? p.out_pm + off_pm + c_first + ch : nullptr;
                        const size_t cm_step = (size_t)(16 * NE) * p.npoint;
                        const float *shp = sh + c_first + ch;
                        uint32_t taddr = zc + (uint32_t)(c_first - s_lo);
                        const int n_ok = Cl - ch;
                        for (int c0 = c_first; c0 < s_hi; c0 += 16 * NE, ocm += cm_step, shp += 16 * NE, taddr += 16 * NE, opm += (opm ? 16 * NE : 0)) {
                            float x;
                            if (pool_raw) {
                                x = pool_quad<NSC>(taddr, lane, [](float v, int) { return v; });
                                x = fmaxf(x + *shp, lo);
                            } else {
                                const float *sc0 = sc + c0, *sh0 = sh + c0;
                                x = pool_quad<NSC>(taddr, lane, [&](float v, int col) { return fmaxf(fmaf(v, sc0[col], sh0[col]), lo); });
                            }
                            if (st_lane && c0 < n_ok) {
                                *ocm = x;
                                if (opm) *opm = x;
                            }
                        }
                    };
                    auto slice_loop = [&](auto ns_c, auto pool_c) {
                        constexpr int NSC = decltype(ns_c)::value, POOLC = decltype(pool_c)::value;
                        const int ch = POOLC == 0 ? (lane & 15)
                                                  : (NSC == 32 ? ((lane >> 1) & 15)
                                                               : (((lane >> 3) & 1) * 8 + ((lane >> 2) & 1) * 4 + ((lane >> 1) & 1) * 2 + (lane & 1)));
                        const bool st_lane = ok && (NSC == 16 || (POOLC == 1 ? (lane & 1) == 0 : lane < 16));
                        const int c_first = s_lo + grp * 16;
                        float *ocm = p.out + off_cm + (size_t)(c_first + ch) * p.npoint;
                        float *opm = p.out_pm ? p.out_pm + off_pm + c_first + ch : nullptr;
                        const size_t cm_step = (size_t)(16 * NE) * p.npoint;
                        const float *shp = sh + c_first + ch;
                        uint32_t taddr = zc + (uint32_t)(c_first - s_lo);
                        const int n_ok = Cl - ch;                   // channel c0 + ch exists iff c0 < n_ok
                        for (int c0 = c_first; c0 < s_hi; c0 += 16 * NE, ocm += cm_step, shp += 16 * NE, taddr += 16 * NE, opm += (opm ? 16 * NE : 0)) {
                            uint32_t acc[16];
                            tmem_ld16(taddr, acc);
                            float v[16];
                            if (pool_raw) {
#pragma unroll
                                for (int q = 0; q < 16; ++q) v[q] = __uint_as_float(acc[q]);
                            } else {
                                // scale not folded (or a linear last layer): activation first, then the max
                                const float4 *sh4 = reinterpret_cast<const float4 *>(sh + c0), *sc4 = reinterpret_cast<const float4 *>(sc + c0);
#pragma unroll
                                for (int j = 0; j < 4; ++j) {
                                    const float4 a = sc4[j], b = sh4[j];
                                    v[4 * j + 0] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 0]), a.x, b.x), lo);
                                    v[4 * j + 1] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 1]), a.y, b.y), lo);
                                    v[4 * j + 2] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 2]), a.z, b.z), lo);
                                    v[4 * j + 3] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 3]), a.w, b.w), lo);
                                }
                            }
                            float x = pool_batch<NSC, POOLC>(v, lane);
                            if (pool_raw) x = fmaxf(x + *shp, lo);
                            if (st_lane && c0 < n_ok) {
                                *ocm = x;
                                if (opm) *opm = x;
                            }
                        }
                    };
                    using I16 = std::integral_constant<int, 16>;
                    using I32 = std::integral_constant<int, 32>;
                    using P0 = std::integral_constant<int, 0>;
                    using P1 = std::integral_constant<int, 1>;
                    if (ns == 32) { if (p.pool_mode == 0) quad_loop(I32{}); else if (p.pool_mode == 2) slice_loop(I32{}, P0{}); else slice_loop(I32{}, P1{}); }
                    else { if (p.pool_mode == 0) quad_loop(I16{}); else if (p.pool_mode == 2) slice_loop(I16{}, P0{}); else slice_loop(I16{}, P1{}); }
                } else
                for (int c0 = s_lo + grp * 16; c0 < s_hi; c0 += 16 * NE) {
                    uint32_t acc[16];
                    tmem_ld16(zc + (uint32_t)(c0 - s_lo), acc);
                    float v[16];
                    // folded scale + max-pool: max_s relu(x_s + t) == relu(max_s x_s + t), so the raw accumulators are
                    // pooled and shift / ReLU are applied once per (centre, channel) after the reduction
                    if (pool_raw) {
#pragma unroll
                        for (int q = 0; q < 16; ++q) v[q] = __uint_as_float(acc[q]);
                    } else if (unit) {
                        const float4 *sh4 = reinterpret_cast<const float4 *>(sh + c0);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float4 b = sh4[j];
                            v[4 * j + 0] = fmaxf(__uint_as_float(acc[4 * j + 0]) + b.x, lo);
                            v[4 * j + 1] = fmaxf(__uint_as_float(acc[4 * j + 1]) + b.y, lo);
                            v[4 * j + 2] = fmaxf(__uint_as_float(acc[4 * j + 2]) + b.z, lo);
                            v[4 * j + 3] = fmaxf(__uint_as_float(acc[4 * j + 3]) + b.w, lo);
                        }
                    } else {
                        const float4 *sc4 = reinterpret_cast<const float4 *>(sc + c0), *sh4 = reinterpret_cast<const float4 *>(sh + c0);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float4 a = sc4[j], b = sh4[j];
                            v[4 * j + 0] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 0]), a.x, b.x), lo);
                            v[4 * j + 1] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 1]), a.y, b.y), lo);
                            v[4 * j + 2] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 2]), a.z, b.z), lo);
                            v[4 * j + 3] = fmaxf(fmaf(__uint_as_float(acc[4 * j + 3]), a.w, b.w), lo);
                        }
                    }
                    if (MOUT == OUT_ROWS) {
                        if (valid) {
                            float *o = p.out + off_cm + c0;
                            if (p.round_out) {   // the next launch of a split chain reads these rows as its A operand
#pragma unroll
                                for (int q = 0; q < 16; ++q) v[q] = to_tf32(v[q]);
                            }
#pragma unroll
                            for (int q = 0; q < 16; q += 4)
                                *reinterpret_cast<float4 *>(o + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
                        }
                    } else if (MOUT == OUT_FP) {
                        if (valid) {
                            float *o = p.out + off_cm + (size_t)c0 * p.n;
#pragma unroll
                            for (int q = 0; q < 16; ++q)
                                if (c0 + q < Cl) o[(size_t)q * p.n] = v[q];
                            if (p.out_pm) {   // point-major copy for the next consumer (no transpose kernel)
                                float *o2 = p.out_pm + off_pm + c0;
                                if ((p.out_stride_c & 3) == 0 && c0 + 16 <= Cl) {
#pragma unroll
                                    for (int q = 0; q < 16; q += 4) *reinterpret_cast<float4 *>(o2 + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
                                } else {
#pragma unroll
                                    for (int q = 0; q < 16; ++q)
                                        if (c0 + q < Cl) o2[q] = v[q];
                                }
                            }
                        }
                    } else {
                        // other sample counts: max over the nsample consecutive rows of each centre through a staging tile:
                        // thread (seg, q) reduces the <=16 rows of one 16-row segment for channel c0+q
                        const int g16 = r >> 4, q = r & 15;
                        bar_named(2 + grp, 128);                     // previous readers of the staging tile are done
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            *reinterpret_cast<float4 *>(pool + r * POOL_STRIDE + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                        bar_named(2 + grp, 128);
                        if (ns >= 16) {
                            float x = pool[(g16 * 16) * POOL_STRIDE + q];
#pragma unroll
                            for (int t = 1; t < 16; ++t) x = fmaxf(x, pool[(g16 * 16 + t) * POOL_STRIDE + q]);
                            const int per = ns >> 4;
                            pool2[g16 * 16 + q] = x;
                            bar_named(2 + grp, 128);
                            const bool head = (g16 % per) == 0;
                            if (head) {
                                for (int t = 1; t < per; ++t) x = fmaxf(x, pool2[(g16 + t) * 16 + q]);
                            }
                            if (pool_raw) x = fmaxf(x + sh[c0 + q], lo);
                            if (ok && head && c0 + q < Cl) {
                                p.out[off_cm + (size_t)(c0 + q) * p.npoint] = x;
                                if (p.out_pm) p.out_pm[off_pm + c0 + q] = x;
                            }
                        } else {
                            // nsample 4 or 8: 128/ns centres per tile, 16 channels each -> (16/ns) items per thread
                            const int per16 = 16 / ns;
                            for (int t = 0; t < per16; ++t) {
                                const int row0 = g16 * 16 + t * ns;
                                float x = pool[row0 * POOL_STRIDE + q];
                                for (int t2 = 1; t2 < ns; ++t2) x = fmaxf(x, pool[(row0 + t2) * POOL_STRIDE + q]);
                                if (pool_raw) x = fmaxf(x + sh[c0 + q], lo);
                                int scn, pp;
                                cur.at(row0 >> p.log_ns, scn, pp);
                                if (tile * TM + row0 < rows && c0 + q < Cl) {
                                    p.out[((size_t)scn * p.out_stride_c + p.out_c_off + c0 + q) * p.npoint + pp] = x;
                                    if (p.out_pm) p.out_pm[((size_t)scn * p.npoint + pp) * p.out_stride_c + p.out_c_off + c0 + q] = x;
                                }
                            }
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive(s2u(&S.z_free[buf]));        // all 128*NE epilogue threads: this slice buffer may be overwritten
            }
        }
    }

    tt.finish();
    tc_fence_before();
    __syncthreads();
    if (warp == W_MISC + 2) tmem_dealloc(tmem, (uint32_t)p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------ host side
// Can this chain segment run on the pipelined kernel, and with which tensor-memory plan?  Fills the plan fields of p.
// Returns the CTAs per SM the plan allows (0 = not supported: the caller falls back to the legacy kernel).
struct PipePlan {
    int ne, ngw, occ, zs, nbuf, nslice, cols, na, nb0, nb1, b0_bytes, b1_bytes, nsplit, split_w, brows, resident;
    size_t smem;
};

// Plan rules (tunable through prb_options.mlp_ne / mlp_ngw / mlp_zs / mlp_nbuf for sweeps):
//  * last layer: slice width zs (divides np_last) x nbuf buffers next to the mid regions; prefer a plan of <= 256 columns
//    (two CTAs per SM), then double buffering, then wide slices;
//  * <= 256 columns: two CTAs of 4 epilogue + 4 gather warps (384 threads, 85 registers);
//    otherwise one CTA with 8 epilogue warps and 8 (layer 0 has >= 2 K chunks) or 4 gather warps.
static bool pipe_plan(const ChainParams &p, int max_optin, PipePlan *out, int force_occ = 0, int force_ngw = 0) {
    const int L = p.num_layers;
    const int np_last = p.np[L - 1];
    int np_total = 0, mid = 0;
    for (int l = 0; l < L; ++l) { np_total += p.np[l]; if (l + 1 < L) mid += p.np[l]; }
    if (mid + 32 > 512) return false;
    const int k0 = p.nchunks[0];
    const prb_options &o = opts();
    PipePlan best;
    long best_score = -1;
    for (int nbuf = 2; nbuf >= 1; --nbuf) {
        if (o.mlp_nbuf && nbuf != o.mlp_nbuf) continue;
        for (int zs = 256; zs >= 32; zs -= 32) {
            int nslice = 1, nsplit = 1, split_w = np_last, z = zs;
            if (L == 1) {
                // single layer: no slicing (the A chunks stream by once); wide layers are dealt to nsplit work items
                if (zs != 256) continue;
                // ... and launches with few tiles are dealt to MORE items than the accumulator width requires, until every SM
                // has one (each item re-gathers its A rows from L2; the small levels -- 32 to 256 tiles -- otherwise run on a
                // fraction of the GPU with one long K loop per CTA)
                nsplit = (np_last + 255) / 256;
                const int want = (num_sms() + p.num_tiles - 1) / p.num_tiles;
                if (want > nsplit && o.mlp_fill) nsplit = want;
                if (nsplit > np_last / 64) nsplit = np_last / 64 > 0 ? np_last / 64 : 1;
                if (nsplit < (np_last + 255) / 256) nsplit = (np_last + 255) / 256;
                if (o.mlp_zs >= 32 && o.mlp_zs < np_last) nsplit = (np_last + o.mlp_zs - 1) / o.mlp_zs;
                split_w = ((np_last + nsplit - 1) / nsplit + 31) / 32 * 32;
                nsplit = (np_last + split_w - 1) / split_w;
                z = split_w;
            } else {
                if (zs > np_last || np_last % zs) continue;
                if (o.mlp_zs && zs != o.mlp_zs) continue;
                nslice = np_last / zs;
            }
            const int need = mid + nbuf * z;
            if (need > 512) continue;
            int cols = 32;
            while (cols < need) cols <<= 1;
            PipePlan pl;
            pl.zs = z; pl.nbuf = nbuf; pl.nslice = nslice; pl.cols = cols; pl.nsplit = nsplit; pl.split_w = split_w;
            pl.occ = cols <= 256 ? 2 : 1;
            if (o.mlp_occ == 1 || force_occ == 1) pl.occ = 1;
            if (force_occ == 2 && pl.occ != 2) continue;
            if (force_occ == 3) {                          // three CTAs per SM: <= 128 columns each, SA gather without row segments
                if (cols > 128 || p.mode_in != IN_SA || p.mode_out != OUT_SA_MAX || p.c_feat > 5 || !(p.ns == 16 || p.ns == 32)) continue;   // also the IN_SA_L0 build
                pl.occ = 3;
            }
            pl.ne = pl.ngw = pl.occ >= 2 ? 1 : 2;         // builds: 4+4 row warps x 2 (or 3) CTAs, or 8+8 row warps x 1 CTA
            if (o.mlp_ne == 1) pl.ne = pl.ngw = 1;
            if (o.mlp_ne == 2) { pl.ne = pl.ngw = 2; pl.occ = 1; }
            if (pl.ne == 2 && (o.mlp_ngw == 3 || force_ngw == 3)) pl.ngw = 3;     // third build: 8 epilogue + 12 gather warps
            // weight stages: up to BROWS rows (output channels) of one 32-column K chunk.  Measured (profiles/r2_notes.md): 64-row
            // stages with 8-12 deep rings are SLOWER than 256-row stages 3 deep (SA3 0.178 vs 0.131 ms, FP1 0.242 vs 0.158):
            // every stage costs two single-thread barrier round trips and an N=64 MMA per K step, which outweighs the
            // extra bytes in flight.
            const int brows = o.mlp_brows >= 32 ? o.mlp_brows : 256;
            pl.brows = brows;
            int b0_rows = L == 1 ? z : p.np[0], b1_rows = 32;
            for (int l = 1; l < L; ++l) { const int w = (l == L - 1) ? z : p.np[l]; if (w > b1_rows) b1_rows = w; }
            if (b0_rows > brows) b0_rows = brows;
            if (b1_rows > brows) b1_rows = brows;
            pl.b0_bytes = b0_rows * KC * 4; pl.b1_bytes = L > 1 ? b1_rows * KC * 4 : 0;
            const size_t budget = (size_t)(227 * 1024) / pl.occ - 1024 - sizeof(PipeSmem) - 512;
            bool ok = false;
            pl.resident = 0;
            // resident weights: when every weight stage a tile needs fits next to a useful A ring, the rings are as deep as
            // one tile, filled once and never recycled -- no weight traffic, no stage barriers, no empty commits per tile
            if (o.mlp_resident) {
                const int halves0 = ((L == 1 ? z : p.np[0]) + brows - 1) / brows;
                int st0 = p.nchunks[0] * halves0, st1 = 0;
                for (int l = 1; l < L; ++l) {
                    const int w = (l == L - 1) ? z : p.np[l];
                    st1 += (l == L - 1 ? nslice : 1) * p.nchunks[l] * ((w + brows - 1) / brows);
                }
                if (st0 <= PIPE_MAX_B && st1 <= PIPE_MAX_B) {
                    const int na_min = k0 + 1 < PIPE_MAX_A ? (k0 + 1 > 3 ? k0 + 1 : 3) : PIPE_MAX_A;
                    for (int na = (k0 + 2 < PIPE_MAX_A ? (k0 + 2 > 3 ? k0 + 2 : 3) : PIPE_MAX_A); na >= na_min && !ok; --na) {
                        const size_t smem = pipe_smem_bytes(pl.ne, na, st0, pl.b0_bytes, st1, pl.b1_bytes, np_total,
                                                            p.mode_out == OUT_SA_MAX && !(p.ns == 16 || p.ns == 32), p.sa_l0 ? p.l0_np : 0);
                        if (smem <= budget && smem <= (size_t)max_optin) {
                            pl.na = na; pl.nb0 = st0; pl.nb1 = st1; pl.smem = smem; pl.resident = 1; ok = true;
                        }
                    }
                }
            }
            // weight rings 3 deep (2 if tight); the A ring as deep as fits, up to one whole item + 2
            for (int nb = 3; nb >= 2 && !ok; --nb)
                for (int na = (k0 + 2 < PIPE_MAX_A ? (k0 + 2 > 3 ? k0 + 2 : 3) : PIPE_MAX_A); na >= 2 && !ok; --na) {
                    const size_t smem = pipe_smem_bytes(pl.ne, na, nb, pl.b0_bytes, L > 1 ? nb : 0, pl.b1_bytes, np_total,
                                                        p.mode_out == OUT_SA_MAX && !(p.ns == 16 || p.ns == 32),   // 16 / 32 samples pool in registers
                                                        p.sa_l0 ? p.l0_np : 0);
                    if (smem <= budget && smem <= (size_t)max_optin && (nb == 2 || na >= (k0 < 4 ? k0 : 4))) {
                        pl.na = na; pl.nb0 = nb; pl.nb1 = L > 1 ? nb : 0; pl.smem = smem; ok = true;
                    }
                }
            if (!ok) continue;
            const long score = (long)pl.occ * 1000000L + nbuf * 1000L + z;
            if (score > best_score) { best_score = score; best = pl; }
        }
    }
    if (best_score < 0) return false;
    *out = best;
    return true;
}

// apply a plan to the launch parameters and launch
static int launch_with_plan(ChainParams &p, const PipePlan &pl, cudaStream_t st) {
    const int L = p.num_layers;
    int col = 0;
    for (int l = 0; l + 1 < L; ++l) { p.rcol[l] = col; col += p.np[l]; }
    p.zcol[0] = col; p.zcol[1] = col + pl.zs;
    p.zs = pl.zs; p.nslice = pl.nslice; p.nbuf = pl.nbuf;
    p.tmem_cols = pl.cols;
    p.na = pl.na; p.nb0 = pl.nb0; p.nb1 = pl.nb1 > 0 ? pl.nb1 : 1;
    p.b0_stage_bytes = pl.b0_bytes; p.b1_stage_bytes = pl.b1_bytes;
    p.nsplit = pl.nsplit; p.split_w = pl.split_w;
    p.b_rows = pl.brows;
    p.w_resident = pl.resident;
    p.num_items = p.num_tiles * pl.nsplit;
    int sms = num_sms();
    if (const int v = opts().mlp_sms; v >= 1 && v < sms) sms = v;
    int grid = sms * pl.occ;
    if (grid > p.num_items) grid = p.num_items;
    grid = grid / pl.nsplit * pl.nsplit;         // a CTA keeps its column group: tiles advance by grid / nsplit
    if (grid < pl.nsplit) grid = pl.nsplit;
    p.trace = opts().mlp_trace ? 1 : 0;
    p.rows32 = (int)p.total_rows;
    p.pool_mode = opts().mlp_pool;
    p.sleepy_ns = opts().mlp_lazy_ns > 0 ? opts().mlp_lazy_ns : 400;
    const size_t smem = pl.smem;
#define PRB_LAUNCH_PIPE(NE, NGW, MB, MI, MO)                                                                                   \
    do {                                                                                                                       \
        PRB_CUDA(cudaFuncSetAttribute(mlp_pipe_kernel<NE, NGW, MB, MI, MO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        mlp_pipe_kernel<NE, NGW, MB, MI, MO><<<grid, (NE + NGW + 1) * 128, smem, st>>>(p);                                      \
    } while (0)
#define PRB_LAUNCH_PIPE_IO(NE, NGW, MB)                                                                    \
    do {                                                                                                   \
        const int key = (p.sa_l0 ? IN_SA_L0 : p.mode_in) * 3 + p.mode_out;                                \
        switch (key) {                                                                                     \
            case IN_SA * 3 + OUT_ROWS: PRB_LAUNCH_PIPE(NE, NGW, MB, IN_SA, OUT_ROWS); break;              \
            case IN_SA * 3 + OUT_SA_MAX: PRB_LAUNCH_PIPE(NE, NGW, MB, IN_SA, OUT_SA_MAX); break;          \
            case IN_SA_L0 * 3 + OUT_SA_MAX: PRB_LAUNCH_PIPE(NE, NGW, MB, IN_SA_L0, OUT_SA_MAX); break;    \
            case IN_FP * 3 + OUT_ROWS: PRB_LAUNCH_PIPE(NE, NGW, MB, IN_FP, OUT_ROWS); break;              \
            case IN_FP * 3 + OUT_FP: PRB_LAUNCH_PIPE(NE, NGW, MB, IN_FP, OUT_FP); break;                  \
            case IN_DIRECT * 3 + OUT_ROWS: PRB_LAUNCH_PIPE(NE, NGW, MB, IN_DIRECT, OUT_ROWS); break;      \
            case IN_DIRECT * 3 + OUT_SA_MAX: PRB_LAUNCH_PIPE(NE, NGW, MB, IN_DIRECT, OUT_SA_MAX); break;  \
            case IN_DIRECT * 3 + OUT_FP: PRB_LAUNCH_PIPE(NE, NGW, MB, IN_DIRECT, OUT_FP); break;          \
            default: set_error("mlp: unsupported input / output mode pair %d / %d", p.mode_in, p.mode_out); return -1; \
        }                                                                                                  \
    } while (0)
    if (pl.occ == 3 && p.sa_l0) PRB_LAUNCH_PIPE(1, 1, 3, IN_SA_L0, OUT_SA_MAX);
    else if (pl.occ == 3) PRB_LAUNCH_PIPE(1, 1, 3, IN_SA, OUT_SA_MAX);
    else if (pl.ne == 1 && pl.ngw == 1) PRB_LAUNCH_PIPE_IO(1, 1, 2);      // launch bounds only cap the registers; occ 1 runs the same build
    else if (pl.ngw == 3) PRB_LAUNCH_PIPE_IO(2, 3, 1);
    else PRB_LAUNCH_PIPE_IO(2, 2, 1);
#undef PRB_LAUNCH_PIPE_IO
#undef PRB_LAUNCH_PIPE
    return check_launch("mlp_pipe_kernel");
}

// Which build runs a given chain shape -- two CTAs per SM of 4 epilogue + 4 gather warps, one CTA of 8 + 8 with twice the
// tensor memory (double-buffered last layer), or one CTA of 8 + 12 for gather-bound shapes -- is MEASURED, not guessed: the
// first eager launch of a shape times them
// (CUDA events on the launching stream, best of 2 after a warm-up; the launches are idempotent and every plan computes
// bit-identical results, K order and per-element arithmetic do not depend on the plan) and the winner is cached per
// device and shape.  Launches inside a stream capture, traced launches and launches with any plan option forced through
// prb_options use the rule-based plan (prefer two CTAs per SM).  profiles/r2_notes.md: SA2 scale 1 0.152 -> 0.139 ms,
// FP0 0.150 -> 0.125, FP3 0.122 -> 0.085 on the wide build; SA1 0.207 -> 0.266 the other way.
struct TuneKey {
    int dev, mode_in, mode_out, L, ns, k0, tiles, np[3];
    bool operator<(const TuneKey &o) const { return memcmp(this, &o, sizeof(TuneKey)) < 0; }
};
static std::mutex g_tune_mu;
struct TuneVal { int choice; int nc; int code[4]; float ms[4]; };
static std::map<TuneKey, TuneVal> g_tune;      // -> winning build: 2 = two CTAs per SM (4+4 row warps), 1 = one CTA 8+8, 3 = one CTA 8+12, 4 = three CTAs

static bool tuning_allowed(cudaStream_t st) {
    const prb_options &o = opts();
    if (!o.mlp_tune || o.mlp_trace || o.mlp_occ || o.mlp_ne || o.mlp_ngw || o.mlp_zs || o.mlp_nbuf) return false;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return false; }
    return cs == cudaStreamCaptureStatusNone;
}

// launch one fused segment on the pipelined kernel
int launch_chain_pipe(ChainParams &p, cudaStream_t st) {
    int max_optin = 0, dev = 0;
    PRB_CUDA(cudaGetDevice(&dev));
    PRB_CUDA(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    p.num_tiles = (int)((p.total_rows + TM - 1) / TM);
    if (p.num_tiles == 0) return 0;
    PipePlan pl;
    if (!(opts().mlp_occ == 3 && pipe_plan(p, max_optin, &pl, 3, 0)))       // mlp_occ = 3 forces the three-CTA build where it applies
        PRB_REQUIRE(pipe_plan(p, max_optin, &pl), "mlp: no tensor-memory / shared-memory plan for this chain segment");
    // candidates: the rule-based plan first, then the one-CTA builds it did not pick (8 + 8 and 8 + 12 row warps)
    PipePlan cand[4];
    int code[4], nc = 0;
    cand[nc] = pl; code[nc++] = pl.occ == 2 ? 2 : (pl.ngw == 3 ? 3 : 1);
    if (pl.occ == 2 && opts().mlp_occ != 2 && pipe_plan(p, max_optin, &cand[nc], 3, 0)) code[nc++] = 4;      // three CTAs per SM
    if (pl.occ == 2 && pipe_plan(p, max_optin, &cand[nc], 1, 0)) code[nc++] = 1;
    if (pl.ngw != 3 && pipe_plan(p, max_optin, &cand[nc], 1, 3) && cand[nc].ngw == 3) code[nc++] = 3;
    if (nc > 1) {
        TuneKey key;
        memset(&key, 0, sizeof(key));
        key.dev = dev; key.mode_in = p.sa_l0 ? IN_SA_L0 : p.mode_in; key.mode_out = p.mode_out; key.L = p.num_layers; key.ns = p.ns;
        key.k0 = p.nchunks[0]; key.tiles = p.num_tiles;
        for (int l = 0; l < p.num_layers; ++l) key.np[l] = p.np[l];
        int choice = 0;
        {
            std::lock_guard<std::mutex> g(g_tune_mu);
            auto it = g_tune.find(key);
            if (it != g_tune.end()) choice = it->second.choice;
        }
        if (choice == 0 && tuning_allowed(st)) {
            cudaEvent_t e0, e1;
            PRB_CUDA(cudaEventCreate(&e0));
            PRB_CUDA(cudaEventCreate(&e1));
            float best[4] = {1e30f, 1e30f, 1e30f, 1e30f};
            int rc = 0;
            for (int c = 0; c < nc && !rc; ++c)
                for (int rep = 0; rep < 3 && !rc; ++rep) {
                    ChainParams q = p;
                    cudaEventRecord(e0, st);
                    rc = launch_with_plan(q, cand[c], st);
                    cudaEventRecord(e1, st);
                    if (cudaEventSynchronize(e1) != cudaSuccess) rc = rc ? rc : -1;
                    float ms = 0.f;
                    cudaEventElapsedTime(&ms, e0, e1);
                    if (rep > 0 && ms < best[c]) best[c] = ms;
                }
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
            if (rc) return rc;
            int win = 0;
            for (int c = 1; c < nc; ++c)
                if (best[c] < 0.97f * best[win]) win = c;       // a later candidate has to win by a margin
            choice = code[win];
            TuneVal tv;
            memset(&tv, 0, sizeof(tv));
            tv.choice = choice; tv.nc = nc;
            for (int c = 0; c < nc; ++c) { tv.code[c] = code[c]; tv.ms[c] = best[c]; }
            std::lock_guard<std::mutex> g(g_tune_mu);
            g_tune[key] = tv;
        }
        for (int c = 0; c < nc; ++c)
            if (code[c] == choice) pl = cand[c];
    }
    return launch_with_plan(p, pl, st);
}

// tuned plans so far: n entries of 18 ints {mode_in, mode_out, layers, nsample, k chunks, tiles, np0, np1, np2, winner,
// 4 x (candidate build, measured microseconds)}
int pipe_tuned_plans(int *dst, int max_entries) {
    std::lock_guard<std::mutex> g(g_tune_mu);
    int n = 0;
    for (const auto &kv : g_tune) {
        if (n >= max_entries) break;
        const TuneKey &k = kv.first;
        int *d = dst + 18 * n++;
        d[0] = k.mode_in == IN_SA_L0 ? IN_SA : k.mode_in;       // reported as an SA chain (one layer shorter)
        d[1] = k.mode_out; d[2] = k.L; d[3] = k.ns; d[4] = k.k0; d[5] = k.tiles; d[6] = k.np[0]; d[7] = k.np[1]; d[8] = k.np[2];
        d[9] = kv.second.choice;
        for (int c = 0; c < 4; ++c) {       // candidates: build code (0 = none) and measured microseconds
            d[10 + 2 * c] = c < kv.second.nc ? kv.second.code[c] : 0;
            d[11 + 2 * c] = c < kv.second.nc ? (int)(kv.second.ms[c] * 1000.f + 0.5f) : 0;
        }
    }
    return n;
}

}  // namespace prb

// wait-time trace of the last traced pipelined launch: 8 roles x {up to 7 classes, total cycles in slot 7} (see g_pipe_trace)
extern "C" int prb_debug_tuned_plans(int *dst, int max_entries) { return prb::pipe_tuned_plans(dst, max_entries); }

extern "C" int prb_debug_pipe_trace(long long *dst) {
    PRB_CUDA(cudaDeviceSynchronize());
    PRB_CUDA(cudaMemcpyFromSymbol(dst, prb::g_pipe_trace, sizeof(long long) * 64));
    static long long zeros[64];
    PRB_CUDA(cudaMemcpyToSymbol(prb::g_pipe_trace, zeros, sizeof(zeros)));
    return 0;
}
