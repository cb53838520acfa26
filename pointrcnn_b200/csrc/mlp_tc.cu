// mlp_tc.cu -- the per-group / per-point shared MLP as a tcgen05 (5th-gen tensor core) layer chain.
//
// Replaces, for eval-mode forward, everything between the ball query and the next level's features:
//   grouping_operation x2 + cat + SharedMLP (Conv2d 1x1 -> BN -> ReLU) x L + max_pool2d
//     (pointnet2_lib/pointnet2/pointnet2_utils.py:249-257, pointnet2_modules.py:40-52, pytorch_utils.py:5-101)
//   three_interpolate + cat + SharedMLP x L
//     (pointnet2_modules.py:144-156)
// The reference materialises every (B,C,npoint,nsample) tensor in HBM between ~10 library kernels per
// scale; here a 128-row tile never leaves the SM between its gather and its pooled output.
//
// Structure (one CTA per SM, persistent over 128-row tiles; rows = (centre, sample) pairs or points):
//   warps 0-3  "row threads": build the A operand of every layer, chunk by chunk (32 K-columns =
//              one 128-byte swizzle row), into a ring of shared-memory stages:
//                layer 0  : gathered neighbour features / interpolated + skip features / plain rows
//                layer l>0: tcgen05.ld of layer l-1's accumulator columns -> scale/shift/ReLU -> tf32
//              and run the final epilogue (max over nsample / channel-major store).
//   warp 4     weight producer: one thread streams pre-packed weight tiles (already in the UMMA
//              K-major SWIZZLE_128B image, see prb_mlp_pack_weights) with cp.async.bulk + mbarrier tx.
//   warp 5     MMA issuer: one thread issues tcgen05.mma kind::tf32 (M=128, N<=256, K=8) with fp32
//              accumulators in TMEM; tcgen05.commit releases stages / publishes finished layers.
// TMEM plan: layer 0 at column 0, layer 1 at the top (512-N1), layer 2 at column 0 again; chains that
// do not fit (N_l + N_{l+1} > 512) are split into several launches by the host wrapper.
// Precision: operands are rounded to TF32 (cvt.rna), products accumulate in fp32 -- the same contract
// as the reference's cuDNN convolutions under torch's default allow_tf32=True (SURVEY.md 8c).
#include <string.h>

#include <vector>

#include "mlp_dev.cuh"

namespace prb {

// ------------------------------------------------------------------------------------------------ kernel
// NG row groups of 4 warps each (warp w: TMEM lane quarter w%4, group w/4) + producer warp + MMA warp.
// The A chunks (and the 16-column epilogue batches) of a tile are dealt round-robin to the groups, so 4*NG warps
// hide each other's latencies while the stage order seen by the MMA issuer stays sequential.
// optional phase trace (PRB_MLP_TRACE=1): CTA 0 stamps clock64 at the phase boundaries of its first 32 tiles
__device__ long long g_trace[32 * 16];
#define PRB_TRACE(slot) do { if (p.trace && blockIdx.x == 0 && tcount < 32 && r == 0) g_trace[tcount * 16 + (slot)] = clock64(); } while (0)

template <int NG, int MINB>
__global__ void __launch_bounds__(128 * NG + 64, MINB) mlp_chain_kernel(const ChainParams p) {
    constexpr int NTHREADS = 128 * NG + 64;
    extern __shared__ uint8_t smem_raw[];
    __shared__ SmemFixed S;
    // keep the pointer arithmetic on the __shared__ symbol itself so the compiler emits LDS/STS, not generic accesses
    uint8_t *base = smem_raw + ((1024u - (s2u(smem_raw) & 1023u)) & 1023u);
    const int L = p.num_layers;
    int np_total = 0, sc_off[MAX_LAYERS];
    for (int l = 0; l < L; ++l) { sc_off[l] = np_total; np_total += p.np[l]; }
    uint8_t *sA = base;
    uint8_t *sB = sA + (size_t)p.na * A_STAGE_BYTES;
    float *s_scale = reinterpret_cast<float *>(sB + (size_t)p.nb * p.b_stage_bytes);
    float *s_shift = s_scale + np_total;
    float *s_pool = s_shift + np_total;                                  // NG x (TM x POOL_STRIDE + 8 x 16)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NA = p.na, NB = p.nb;

    if (tid == 0) {
        for (int i = 0; i < NA; ++i) { mbar_init(s2u(&S.a_full[i]), 128); mbar_init(s2u(&S.a_empty[i]), 1); }
        for (int i = 0; i < NB; ++i) { mbar_init(s2u(&S.b_full[i]), 1); mbar_init(s2u(&S.b_empty[i]), 1); }
        for (int i = 0; i < MAX_LAYERS; ++i) mbar_init(s2u(&S.d_full[i]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4 * NG + 1) tmem_alloc(s2u(&S.tmem_base), (uint32_t)p.tmem_cols);
    for (int l = 0; l < L; ++l)
        for (int i = tid; i < p.np[l]; i += NTHREADS) { s_scale[sc_off[l] + i] = p.unit_scale ? 1.f : p.scale[l][i]; s_shift[sc_off[l] + i] = p.shift[l][i]; }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = S.tmem_base;

    if (warp == 4 * NG) {
        // ===================================================== weight producer
        if (lane == 0) {
            RingPos rb = {0, 0};
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
                for (int l = 0; l < L; ++l) {
                    const int halves = (p.np[l] + B_TILE_ROWS - 1) / B_TILE_ROWS;
                    for (int kc = 0; kc < p.nchunks[l]; ++kc)
                        for (int h = 0; h < halves; ++h) {
                            const int rows = min(B_TILE_ROWS, p.np[l] - h * B_TILE_ROWS);
                            const uint32_t bytes = (uint32_t)rows * KC * 4;
                            if (p.sleepy & 2) mbar_wait_sleepy(s2u(&S.b_empty[rb.stage]), rb.phase ^ 1); else mbar_wait(s2u(&S.b_empty[rb.stage]), rb.phase ^ 1);
                            mbar_expect_tx(s2u(&S.b_full[rb.stage]), bytes);
                            const float *src = p.w[l] + ((size_t)kc * p.np[l] + (size_t)h * B_TILE_ROWS) * KC;
                            bulk_g2s(s2u(sB + (size_t)rb.stage * p.b_stage_bytes), src, bytes, s2u(&S.b_full[rb.stage]));
                            rb.advance(NB);
                        }
                }
            }
        }
    } else if (warp == 4 * NG + 1) {
        // ===================================================== MMA issuer
        if (lane == 0) {
            RingPos ra = {0, 0}, rb = {0, 0};
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
                for (int l = 0; l < L; ++l) {
                    const int halves = (p.np[l] + B_TILE_ROWS - 1) / B_TILE_ROWS;
                    for (int kc = 0; kc < p.nchunks[l]; ++kc) {
                        // valid K in this chunk -> number of K=8 steps
                        int valid = KC;
                        if (l == 0) {
                            int c = kc, s = 0;
                            if (p.nseg > 1 && c >= p.seg_chunks[0]) { c -= p.seg_chunks[0]; s = 1; }
                            valid = min(KC, p.seg_width[s] - c * KC);
                        }
                        const int ksteps = (valid + 7) >> 3;
                        if (p.sleepy & 1) mbar_wait_sleepy(s2u(&S.a_full[ra.stage]), ra.phase); else mbar_wait(s2u(&S.a_full[ra.stage]), ra.phase);
                        const uint64_t adesc = make_desc(s2u(sA + (size_t)ra.stage * A_STAGE_BYTES));
                        for (int h = 0; h < halves; ++h) {
                            const int rows = min(B_TILE_ROWS, p.np[l] - h * B_TILE_ROWS);
                            if (p.sleepy & 1) mbar_wait_sleepy(s2u(&S.b_full[rb.stage]), rb.phase); else mbar_wait(s2u(&S.b_full[rb.stage]), rb.phase);
                            tc_fence_after();
                            const uint64_t bdesc = make_desc(s2u(sB + (size_t)rb.stage * p.b_stage_bytes));
                            const uint32_t idesc = make_idesc(rows);
                            const uint32_t d = tmem + (uint32_t)(p.dcol[l] + h * B_TILE_ROWS);
                            if (p.a_tmem && l > 0) {   // A = the rewritten accumulator of layer l-1: columns kc*32 + ks*8 ...
                                const uint32_t a_t = tmem + (uint32_t)(p.dcol[l - 1] + kc * KC);
                                for (int ks = 0; ks < ksteps; ++ks)
                                    umma_tf32_ts(d, a_t + (uint32_t)(8 * ks), bdesc + (uint64_t)(2 * ks), idesc, (kc > 0 || ks > 0) ? 1u : 0u);
                            } else {
                                for (int ks = 0; ks < ksteps; ++ks)  // +32 bytes (= 2 x 16 B) per K=8 step inside the swizzle row
                                    umma_tf32(d, adesc + (uint64_t)(2 * ks), bdesc + (uint64_t)(2 * ks), idesc, (kc > 0 || ks > 0) ? 1u : 0u);
                            }
                            umma_commit(s2u(&S.b_empty[rb.stage]));
                            rb.advance(NB);
                        }
                        umma_commit(s2u(&S.a_empty[ra.stage]));
                        ra.advance(NA);
                    }
                    umma_commit(s2u(&S.d_full[l]));
                }
            }
        }
    } else {
        // ===================================================== row threads (warps 0 .. 4*NG-1)
        RingPos ra = {0, 0};
        uint32_t dphase = 0;
        const int wq = warp & 3, grp = warp >> 2;
        const int r = wq * 32 + lane;       // my row inside the tile / my TMEM lane
        const uint32_t lane_base = (uint32_t)(wq * 32) << 16;
        const int j8 = lane & 7;            // my 16-byte unit inside a 128-byte row (gathers)
        const int rsub = lane >> 3;         // which of the 4 rows a warp-wide gather step covers
        uint32_t cc = 0;                    // chunk counter: chunk cc belongs to group cc % NG
        float *pool = s_pool + grp * (TM * POOL_STRIDE + 128);
        float *pool2 = pool + TM * POOL_STRIDE;   // 8 x 16 partial maxima (nsample > 32)

        // tile metadata is fetched one tile ahead (global loads of idx / centres / weights overlap the MMAs)
        int m_src[3] = {0, 0, 0};
        float m_aux[3] = {0.f, 0.f, 0.f};
        bool m_valid = false;
        int m_scene = 0, m_u = 0;            // FP: scene / point index of my row
        auto fetch_meta = [&](int tile) {
            const unsigned R = (unsigned)tile * TM + r;          // total_rows < 2^31 (checked on the host)
            m_valid = tile < p.num_tiles && (long)R < p.total_rows;
            if (p.mode_in == IN_SA) {
                const unsigned pr = m_valid ? (R >> p.log_ns) : 0u;     // global centre index (nsample is a power of two)
                const unsigned scene = pr / (unsigned)p.npoint;
                m_src[0] = (int)scene * p.n + (m_valid ? __ldg(p.idx + R) : 0);
                m_aux[0] = __ldg(p.new_xyz + (size_t)pr * 3 + 0);
                m_aux[1] = __ldg(p.new_xyz + (size_t)pr * 3 + 1);
                m_aux[2] = __ldg(p.new_xyz + (size_t)pr * 3 + 2);
            } else if (p.mode_in == IN_FP || p.mode_out == OUT_FP) {
                const unsigned rr = m_valid ? R : 0u;
                const unsigned scene = rr / (unsigned)p.n;
                m_scene = (int)scene; m_u = (int)(rr - scene * (unsigned)p.n);
                if (p.mode_in == IN_FP) {
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        m_src[q] = (int)scene * p.m + __ldg(p.idx + (size_t)rr * 3 + q);
                        m_aux[q] = __ldg(p.weight + (size_t)rr * 3 + q);
                    }
                }
            }
        };
        fetch_meta(blockIdx.x);

        int tcount = -1;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            ++tcount;
            PRB_TRACE(0);
            const long R = (long)tile * TM + r;
            const bool valid = m_valid;
            const int my_scene = m_scene, my_u = m_u;
            bar_rows<NG>();  // previous tile's readers of S.row_* are done
            if (grp == 0) {
                S.row_valid[r] = valid;
#pragma unroll
                for (int q = 0; q < 3; ++q) { S.row_src[r][q] = m_src[q]; S.row_aux[r][q] = m_aux[q]; }
            }
            bar_rows<NG>();

            // ---- layer 0: build A chunks from global memory
            // Feature rows with a 16-byte aligned pitch are gathered with cp.async straight into the swizzled stage
            // (no registers, up to two chunks of loads in flight per group); their fp32 bits reach the tensor core
            // unrounded, which then drops the low 13 mantissa bits itself.
            uint32_t pend_bar[2] = {0u, 0u};
            int npend = 0;
            // publish every chunk whose cp.async copies are still pending (all of them: groups complete in order)
            auto retire_all = [&]() {
                if (npend > 0) {
                    cp_async_wait<0>();
                    fence_async_smem();
                    mbar_arrive(pend_bar[0]);
                    if (npend == 2) mbar_arrive(pend_bar[1]);
                    npend = 0;
                }
            };
            // claim the next ring stage.  Never block on the consumer while own chunks are unpublished: the stage we
            // wait for may only be released after one of them has been consumed (deadlock otherwise).
            auto acquire_stage = [&]() {
                if (!mbar_test(s2u(&S.a_empty[ra.stage]), ra.phase ^ 1)) {
                    retire_all();
                    mbar_wait(s2u(&S.a_empty[ra.stage]), ra.phase ^ 1);
                }
            };
            for (int kc = 0; kc < p.nchunks[0]; ++kc, ++cc, ra.advance(NA)) {
                if ((int)(cc % NG) != grp) continue;
                int c = kc, seg = 0;
                if (p.nseg > 1 && c >= p.seg_chunks[0]) { c -= p.seg_chunks[0]; seg = 1; }
                const int k0 = c * KC;                       // first column of this chunk inside its segment
                const int width = p.seg_width[seg];
                uint8_t *A = sA + (size_t)ra.stage * A_STAGE_BYTES;
                const bool rows_seg = (p.mode_in == IN_DIRECT) || (p.mode_in == IN_SA && seg == 0 && p.c_feat > 5) ||
                                      (p.mode_in == IN_FP && seg == 0);
                if (rows_seg) {
                    // point-major sources: 8 lanes cover one row's 128 bytes, a warp covers 4 rows per step, 8 steps.
                    // All loads of the chunk are issued before the first use (memory-level parallelism).
                    const int kk = k0 + 4 * j8;
                    if (p.mode_in == IN_FP) {
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
                                w0[i] = S.row_aux[rr][0]; w1[i] = S.row_aux[rr][1]; w2[i] = S.row_aux[rr][2];
                                if (S.row_valid[rr] && kk < width) {
                                    const float *s0 = p.known_pm + (size_t)S.row_src[rr][0] * C + kk;
                                    const float *s1 = p.known_pm + (size_t)S.row_src[rr][1] * C + kk;
                                    const float *s2 = p.known_pm + (size_t)S.row_src[rr][2] * C + kk;
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
                            if (half == 0) acquire_stage();
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
                        const int pitch = p.mode_in == IN_DIRECT ? p.x_pitch : p.c_feat;
                        if ((pitch & 3) == 0 && p.gather_mode != 0) {
                            // asynchronous path: width is a multiple of 4 too, so a unit is either all data or all padding
                            acquire_stage();
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const int rr = wq * 32 + rsub + 4 * i;
                                const bool ok = S.row_valid[rr] && kk < width;
                                const float *src = p.mode_in == IN_DIRECT ? p.x_rows + ((size_t)tile * TM + rr) * pitch + kk
                                                                          : p.feats_pm + (size_t)S.row_src[rr][0] * pitch + kk;
                                if (p.gather_mode == 1) cp_async16(s2u(A + swz(rr, j8)), ok ? src : (const float *)p.w[0], ok ? 16u : 0u);
                                else cp_async16_ca(s2u(A + swz(rr, j8)), ok ? src : (const float *)p.w[0], ok ? 16u : 0u);
                            }
                            cp_async_commit();
                            if (npend == 2) {          // retire the oldest chunk: its copies have landed
                                cp_async_wait<2>();
                                fence_async_smem();
                                mbar_arrive(pend_bar[0]);
                                pend_bar[0] = pend_bar[1];
                                npend = 1;
                            }
                            pend_bar[npend++] = s2u(&S.a_full[ra.stage]);
                            continue;                  // (the for-increment advances cc and the ring)
                        }
                        float4 t[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int rr = wq * 32 + rsub + 4 * i;
                            t[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (S.row_valid[rr] && kk < width) {
                                const float *src = p.mode_in == IN_DIRECT ? p.x_rows + ((size_t)tile * TM + rr) * pitch + kk
                                                                          : p.feats_pm + (size_t)S.row_src[rr][0] * pitch + kk;
                                if ((pitch & 3) == 0) {
                                    t[i] = __ldg((const float4 *)src);
                                } else {
                                    float o[4];
#pragma unroll
                                    for (int q = 0; q < 4; ++q) o[q] = (kk + q < width) ? __ldg(src + q) : 0.f;
                                    t[i] = make_float4(o[0], o[1], o[2], o[3]);
                                }
                            }
                        }
                        acquire_stage();
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int rr = wq * 32 + rsub + 4 * i;
                            float4 v = t[i];
                            v.x = to_tf32(v.x); v.y = to_tf32(v.y); v.z = to_tf32(v.z); v.w = to_tf32(v.w);
                            *reinterpret_cast<float4 *>(A + swz(rr, j8)) = v;
                        }
                    }
                } else if (p.mode_in == IN_SA) {
                    // relative xyz segment: [x - cx, y - cy, z - cz, (<= 5 feature channels,) 0 ...]; one K=8 step
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f), v2 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (valid) {
                        const float *q = p.xyz + (size_t)m_src[0] * 3;
                        v.x = to_tf32(__ldg(q + 0) - m_aux[0]);
                        v.y = to_tf32(__ldg(q + 1) - m_aux[1]);
                        v.z = to_tf32(__ldg(q + 2) - m_aux[2]);
                        if (p.c_feat > 0 && p.c_feat <= 5) {
                            const float *f = p.feats_pm + (size_t)m_src[0] * p.c_feat;
                            v.w = to_tf32(__ldg(f));
                            if (p.c_feat > 1) v2.x = to_tf32(__ldg(f + 1));
                            if (p.c_feat > 2) v2.y = to_tf32(__ldg(f + 2));
                            if (p.c_feat > 3) v2.z = to_tf32(__ldg(f + 3));
                            if (p.c_feat > 4) v2.w = to_tf32(__ldg(f + 4));
                        }
                    }
                    acquire_stage();
                    *reinterpret_cast<float4 *>(A + swz(r, 0)) = v;
                    *reinterpret_cast<float4 *>(A + swz(r, 1)) = v2;
                } else {
                    // FP skip segment: channel-major (b, c_skip, n); lanes run along consecutive points
                    const float *bsrc = p.skip + (size_t)my_scene * p.c_skip * p.n + my_u;
                    float o[32];
#pragma unroll
                    for (int q = 0; q < 32; ++q) {
                        const int ch = k0 + q;
                        o[q] = (valid && ch < width) ? __ldg(bsrc + (size_t)ch * p.n) : 0.f;
                    }
                    acquire_stage();
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float4 *>(A + swz(r, j)) =
                            make_float4(to_tf32(o[4 * j]), to_tf32(o[4 * j + 1]), to_tf32(o[4 * j + 2]), to_tf32(o[4 * j + 3]));
                }
                fence_async_smem();
                mbar_arrive(s2u(&S.a_full[ra.stage]));
            }

            retire_all();
            PRB_TRACE(1);

            // next tile's metadata: issue the loads now, consume them at the top of the next iteration
            fetch_meta(tile + gridDim.x);

            // ---- layers 1..L-1: previous accumulator -> scale/shift/ReLU -> next A operand
            for (int l = 1; l < L; ++l) {
                mbar_wait(s2u(&S.d_full[l - 1]), dphase);
                tc_fence_after();
                PRB_TRACE(2 * l);
                for (int kc = 0; kc < p.nchunks[l]; ++kc, ++cc, ra.advance(NA)) {
                    if ((int)(cc % NG) != grp) continue;
                    mbar_wait(s2u(&S.a_empty[ra.stage]), ra.phase ^ 1);
                    uint8_t *A = sA + (size_t)ra.stage * A_STAGE_BYTES;
                    if (p.a_tmem) {
                        // in place: D_{l-1}[:, chunk] -> relu(. + shift) as tf32 bit patterns -> the same TMEM columns
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            const uint32_t col = tmem + lane_base + (uint32_t)(p.dcol[l - 1] + kc * KC + hh * 16);
                            uint32_t acc[16];
                            tmem_ld16(col, acc);
                            const float4 *sc4 = reinterpret_cast<const float4 *>(s_scale + sc_off[l - 1] + kc * KC + hh * 16);
                            const float4 *sh4 = reinterpret_cast<const float4 *>(s_shift + sc_off[l - 1] + kc * KC + hh * 16);
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float4 a = sc4[j], b = sh4[j];
                                acc[4 * j + 0] = __float_as_uint(relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 0]), a.x, b.x)));
                                acc[4 * j + 1] = __float_as_uint(relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 1]), a.y, b.y)));
                                acc[4 * j + 2] = __float_as_uint(relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 2]), a.z, b.z)));
                                acc[4 * j + 3] = __float_as_uint(relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 3]), a.w, b.w)));
                            }
                            tmem_st16(col, acc);
                        }
                        tmem_st_wait();
                        tc_fence_before();
                        mbar_arrive(s2u(&S.a_full[ra.stage]));
                        continue;
                    }
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        uint32_t acc[16];
                        tmem_ld16(tmem + lane_base + (uint32_t)(p.dcol[l - 1] + kc * KC + hh * 16), acc);
                        const float4 *sc4 = reinterpret_cast<const float4 *>(s_scale + sc_off[l - 1] + kc * KC + hh * 16);
                        const float4 *sh4 = reinterpret_cast<const float4 *>(s_shift + sc_off[l - 1] + kc * KC + hh * 16);
                        if (p.unit_scale) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float4 b = sh4[j];                 // broadcast LDS.128
                                float4 o;
                                o.x = relu_to_tf32(__uint_as_float(acc[4 * j + 0]) + b.x);
                                o.y = relu_to_tf32(__uint_as_float(acc[4 * j + 1]) + b.y);
                                o.z = relu_to_tf32(__uint_as_float(acc[4 * j + 2]) + b.z);
                                o.w = relu_to_tf32(__uint_as_float(acc[4 * j + 3]) + b.w);
                                *reinterpret_cast<float4 *>(A + swz(r, hh * 4 + j)) = o;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float4 a = sc4[j], b = sh4[j];     // broadcast LDS.128
                                float4 o;
                                o.x = relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 0]), a.x, b.x));
                                o.y = relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 1]), a.y, b.y));
                                o.z = relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 2]), a.z, b.z));
                                o.w = relu_to_tf32(fmaf(__uint_as_float(acc[4 * j + 3]), a.w, b.w));
                                *reinterpret_cast<float4 *>(A + swz(r, hh * 4 + j)) = o;
                            }
                        }
                    }
                    tc_fence_before();
                    fence_async_smem();
                    mbar_arrive(s2u(&S.a_full[ra.stage]));
                }
                PRB_TRACE(2 * l + 1);
            }

            // ---- final epilogue: 16-column batches dealt round-robin to the row groups
            mbar_wait(s2u(&S.d_full[L - 1]), dphase);
            tc_fence_after();
            PRB_TRACE(2 * L);
            const int Cl = p.c_last;
            const float *sc = s_scale + sc_off[L - 1], *sh = s_shift + sc_off[L - 1];
            // SA max-pool: thread (g16, q) owns 16-row segment g16 and channel q of every batch
            size_t e_off = 0, e_pm = 0;
            bool e_ok = false;
            // butterfly pooling (nsample 16 / 32): my centre is the one my own row belongs to
            size_t b_off = 0, b_pm = 0;
            bool b_ok = false;
            if (p.mode_out == OUT_SA_MAX && (p.ns == 16 || p.ns == 32)) {
                const unsigned Rg = (unsigned)tile * TM + (unsigned)r;
                b_ok = (long)Rg < p.total_rows;
                const unsigned pr = Rg >> p.log_ns, scene = pr / (unsigned)p.npoint, pp = pr - scene * (unsigned)p.npoint;
                b_off = ((size_t)scene * p.out_stride_c + p.out_c_off) * p.npoint + pp;
                b_pm = ((size_t)scene * p.npoint + pp) * p.out_stride_c + p.out_c_off;
            }
            if (p.mode_out == OUT_SA_MAX && p.ns >= 16) {
                const unsigned Rg = (unsigned)tile * TM + (unsigned)(r >> 4) * 16u;
                e_ok = (long)Rg < p.total_rows && (((r >> 4) & ((p.ns >> 4) - 1)) == 0);
                const unsigned pr = Rg >> p.log_ns, scene = pr / (unsigned)p.npoint, pp = pr - scene * (unsigned)p.npoint;
                e_off = ((size_t)scene * p.out_stride_c + p.out_c_off + (r & 15)) * p.npoint + pp;
                e_pm = ((size_t)scene * p.npoint + pp) * p.out_stride_c + p.out_c_off + (r & 15);
            }
            for (int c0 = grp * 16; c0 < Cl; c0 += 16 * NG) {
                uint32_t acc[16];
                tmem_ld16(tmem + lane_base + (uint32_t)(p.dcol[L - 1] + c0), acc);
                float v[16];
                // folded scale + max-pool: max_s relu(x_s + t) == relu(max_s x_s + t), so the raw accumulators are
                // pooled and shift / ReLU are applied once per (centre, channel) after the reduction
                const bool pool_raw = p.unit_scale && p.mode_out == OUT_SA_MAX;
                const float lo = p.linear_last ? -CUDART_INF_F : 0.f;    // ReLU = max(., 0); a linear last layer keeps the sign
                if (pool_raw) {
#pragma unroll
                    for (int q = 0; q < 16; ++q) v[q] = __uint_as_float(acc[q]);
                } else if (p.unit_scale) {
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
                if (p.mode_out == OUT_ROWS) {
                    if (valid) {
                        float *o = p.out + (size_t)R * p.out_pitch + c0;
                        if (p.round_out) {   // the next launch of a split chain reads these rows as its A operand
#pragma unroll
                            for (int q = 0; q < 16; ++q) v[q] = to_tf32(v[q]);
                        }
#pragma unroll
                        for (int q = 0; q < 16; q += 4)
                            *reinterpret_cast<float4 *>(o + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
                    }
                } else if (p.mode_out == OUT_FP) {
                    if (valid) {
                        float *o = p.out + ((size_t)my_scene * p.out_stride_c + p.out_c_off + c0) * p.n + my_u;
#pragma unroll
                        for (int q = 0; q < 16; ++q)
                            if (c0 + q < Cl) o[(size_t)q * p.n] = v[q];
                        if (p.out_pm) {   // point-major copy for the next consumer (no transpose kernel)
                            float *o2 = p.out_pm + (size_t)R * p.out_stride_c + p.out_c_off + c0;
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
                    // max over the nsample consecutive rows of each centre, through a shared staging tile:
                    // thread (seg, q) reduces the <=16 rows of one segment for channel c0+q; segments of a centre
                    // with nsample > 16 are combined with one shuffle (32) or a second tiny tile (64, 128).
                    // Groups are whole (total_rows is a multiple of nsample): tail groups past total_rows are skipped.
                    const int ns = p.ns;
                    const int g16 = r >> 4, q = r & 15;          // (segment of 16 rows, channel) handled by this thread
                    if (ns == 32 || ns == 16) {
                        // The nsample rows of a centre are lanes of ONE warp: halving butterfly, no staging tile and
                        // no barriers.  Each step a lane keeps half of its channels (chosen by one lane-id bit),
                        // sends the other half to its partner and takes the max -- 8+4+2+1 shuffles leave one channel
                        // per lane: channel (lane>>1)&15 for 32 samples (one more step joins lanes 2k, 2k+1), channel
                        // lane&15 for 16 samples.  (Measured per 16-column batch under load, scripts/mlp_trace.py:
                        // staged tile + two named barriers ~1000 cycles, 16 CREDUX ~860, this butterfly see notes.)
                        float w8[8], w4[4], w2[2], x;
                        if (ns == 32) {
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
                            x = fmaxf(x, __shfl_xor_sync(0xffffffffu, x, 1));
                        } else {
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
                            x = fmaxf(b0 ? w2[1] : w2[0], __shfl_xor_sync(0xffffffffu, b0 ? w2[0] : w2[1], 1));
                        }
                        // my channel and whether I store it: 32 samples -> even lanes, channel (lane >> 1) & 15;
                        // 16 samples -> every lane, channel = the bit pattern the halving steps selected
                        const int ch = ns == 32 ? ((lane >> 1) & 15) : (((lane >> 3) & 1) * 8 + ((lane >> 2) & 1) * 4 + ((lane >> 1) & 1) * 2 + (lane & 1));
                        if (pool_raw) x = fmaxf(x + sh[c0 + ch], lo);
                        if (b_ok && (ns == 16 || (lane & 1) == 0) && c0 + ch < Cl) {
                            p.out[b_off + (size_t)(c0 + ch) * p.npoint] = x;
                            if (p.out_pm) p.out_pm[b_pm + c0 + ch] = x;
                        }
                        continue;
                    }
                    bar_group(grp);                              // previous readers of the staging tile are done
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<float4 *>(pool + r * POOL_STRIDE + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    bar_group(grp);
                    if (ns >= 16) {
                        float x = pool[(g16 * 16) * POOL_STRIDE + q];
#pragma unroll
                        for (int s = 1; s < 16; ++s) x = fmaxf(x, pool[(g16 * 16 + s) * POOL_STRIDE + q]);
                        if (ns == 32) x = fmaxf(x, __shfl_xor_sync(0xffffffffu, x, 16));
                        if (ns > 32) {
                            pool2[g16 * 16 + q] = x;
                            bar_group(grp);
                            const int per = ns >> 4;
                            if ((g16 % per) == 0) {
                                for (int s = 1; s < per; ++s) x = fmaxf(x, pool2[(g16 + s) * 16 + q]);
                            }
                        }
                        if (pool_raw) x = fmaxf(x + sh[c0 + q], lo);
                        if (e_ok && c0 + q < Cl) {
                            p.out[e_off + (size_t)c0 * p.npoint] = x;
                            if (p.out_pm) p.out_pm[e_pm + c0] = x;
                        }
                    } else {
                        // nsample 4 or 8: 128/ns centres per tile, 16 channels each -> (16/ns) items per thread
                        const int per16 = 16 / ns;
                        for (int t = 0; t < per16; ++t) {
                            const int row0 = g16 * 16 + t * ns;
                            float x = pool[row0 * POOL_STRIDE + q];
                            for (int s = 1; s < ns; ++s) x = fmaxf(x, pool[(row0 + s) * POOL_STRIDE + q]);
                            if (pool_raw) x = fmaxf(x + sh[c0 + q], lo);
                            const unsigned Rg = (unsigned)tile * TM + (unsigned)row0;
                            if ((long)Rg < p.total_rows && c0 + q < Cl) {
                                const unsigned pr = Rg >> p.log_ns, scene = pr / (unsigned)p.npoint, pp = pr - scene * (unsigned)p.npoint;
                                p.out[((size_t)scene * p.out_stride_c + p.out_c_off + c0 + q) * p.npoint + pp] = x;
                                if (p.out_pm) p.out_pm[((size_t)scene * p.npoint + pp) * p.out_stride_c + p.out_c_off + c0 + q] = x;
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            dphase ^= 1;
            PRB_TRACE(2 * L + 1);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 4 * NG + 1) tmem_dealloc(tmem, (uint32_t)p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------ host side
static inline int round_up(int a, int b) { return (a + b - 1) / b * b; }

struct LayerGeom {
    int k_chunks;  // K chunks
    int np;        // padded N
    size_t w_off;  // float offset of this layer's image in the packed buffer
};

// K layout of layer 0 = the given segments, each padded to KC; deeper layers: previous np
static void chain_geometry(int L, int nseg, const int *seg_width, const int *c_out, LayerGeom *g, size_t *total_floats) {
    size_t off = 0;
    for (int l = 0; l < L; ++l) {
        int chunks = 0;
        if (l == 0) for (int s = 0; s < nseg; ++s) chunks += round_up(seg_width[s], KC) / KC;
        else chunks = g[l - 1].np / KC;
        g[l].k_chunks = chunks;
        g[l].np = round_up(c_out[l], 32);
        g[l].w_off = off;
        off += (size_t)chunks * g[l].np * KC;
    }
    if (total_floats) *total_floats = off;
}

static inline float tf32_rna_host(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7f800000u) != 0x7f800000u) u += 0x1000u;  // round to nearest, ties away (cvt.rna)
    u &= 0xffffe000u;
    float r;
    memcpy(&r, &u, 4);
    return r;
}

}  // namespace prb

using namespace prb;

// segment description used by the packer: our K order is seg 0 then seg 1; each segment names the first
// column it takes from the ORIGINAL (c_out0, c_in) weight and its width
struct PackSegs {
    int nseg;
    int src_off[2], width[2];
};

static void default_segs(int kind, int c_in, int a, PackSegs *ps) {
    // kind 0 (SA): original columns [xyz(3), feats(a)] -> ours [feats(a), xyz(3)];  a = c_feat
    // kind 1 (FP): original [interp(a), skip(c_in-a)] kept in order, split in two padded segments
    // kind 2 (DIRECT): one segment
    if (kind == 0) {
        // a handful of feature channels (e.g. the intensity of the first RPN level) ride in the xyz chunk: [xyz, feats]
        if (a > 0 && a <= 5) { ps->nseg = 1; ps->src_off[0] = 0; ps->width[0] = 3 + a; }
        else if (a > 0) { ps->nseg = 2; ps->src_off[0] = 3; ps->width[0] = a; ps->src_off[1] = 0; ps->width[1] = 3; }
        else { ps->nseg = 1; ps->src_off[0] = 0; ps->width[0] = 3; }
    } else if (kind == 1 && c_in - a > 0) {
        ps->nseg = 2; ps->src_off[0] = 0; ps->width[0] = a; ps->src_off[1] = a; ps->width[1] = c_in - a;
    } else {
        ps->nseg = 1; ps->src_off[0] = 0; ps->width[0] = c_in;
    }
}

extern "C" {

// extended packing entry points (kind / split) -- the header's prb_mlp_packed_bytes / prb_mlp_pack_weights
// are the DIRECT (kind 2) forms
PRB_API size_t prb_mlp_packed_bytes_ex(int kind, int split, int num_layers, int c_in, const int *c_out) {
    PackSegs ps;
    default_segs(kind, c_in, split, &ps);
    LayerGeom g[MAX_LAYERS];
    size_t total = 0;
    chain_geometry(num_layers, ps.nseg, ps.width, c_out, g, &total);
    return total * sizeof(float);
}

PRB_API int prb_mlp_pack_weights_ex(int kind, int split, int num_layers, int c_in, const int *c_out, const float *const *w, void *dst) {
    PRB_REQUIRE(num_layers >= 1 && num_layers <= MAX_LAYERS && w && dst && c_out, "mlp_pack: bad arguments");
    PackSegs ps;
    default_segs(kind, c_in, split, &ps);
    LayerGeom g[MAX_LAYERS];
    size_t total = 0;
    chain_geometry(num_layers, ps.nseg, ps.width, c_out, g, &total);
    float *out = (float *)dst;
    memset(out, 0, total * sizeof(float));
    for (int l = 0; l < num_layers; ++l) {
        const int np = g[l].np;
        const int kin = l == 0 ? c_in : c_out[l - 1];
        // map our K index -> original column (or -1 for padding)
        std::vector<int> kmap((size_t)g[l].k_chunks * KC, -1);
        if (l == 0) {
            int base = 0;
            for (int s = 0; s < ps.nseg; ++s) {
                for (int i = 0; i < ps.width[s]; ++i) kmap[base + i] = ps.src_off[s] + i;
                base += round_up(ps.width[s], KC);
            }
        } else {
            for (int i = 0; i < kin; ++i) kmap[i] = i;
        }
        for (int kc = 0; kc < g[l].k_chunks; ++kc)
            for (int n = 0; n < np; ++n)
                for (int kk = 0; kk < KC; ++kk) {
                    const int src = kmap[(size_t)kc * KC + kk];
                    float v = 0.f;
                    if (n < c_out[l] && src >= 0) v = tf32_rna_host(w[l][(size_t)n * kin + src]);
                    // K-major SWIZZLE_128B image of an (np x 32) tile: row n at n*128 B, 16-B unit j at j ^ (n & 7)
                    const int j = kk >> 2, q = kk & 3;
                    const size_t o = g[l].w_off + (size_t)kc * np * KC + (size_t)n * KC + (size_t)(((j ^ (n & 7)) << 2) + q);
                    out[o] = v;
                }
    }
    return 0;
}

size_t prb_mlp_packed_bytes(int num_layers, int c_in, const int *c_out) {
    return prb_mlp_packed_bytes_ex(2, 0, num_layers, c_in, c_out);
}
int prb_mlp_pack_weights(int num_layers, int c_in, const int *c_out, const float *const *w, void *dst) {
    return prb_mlp_pack_weights_ex(2, 0, num_layers, c_in, c_out, w, dst);
}

}  // extern "C"

namespace prb {

int launch_chain_pipe(ChainParams &p, cudaStream_t st);   // mlp_pipe.cu

// the pipelined kernel takes every segment unless the caller asks for the legacy one (prb_options.mlp_pipeline = 0) or
// for the cp.async gather experiment, which only the legacy kernel implements
static bool use_pipe() { return opts().mlp_pipeline != 0 && opts().mlp_gather == 0; }

// launch one fused segment of the chain: size rings / TMEM to the segment, pick the CTAs-per-SM it allows
static int launch_chain(ChainParams &p, cudaStream_t st) {
    if (use_pipe()) return launch_chain_pipe(p, st);
    int max_optin = 0;
    {
        int dev = 0;
        PRB_CUDA(cudaGetDevice(&dev));
        PRB_CUDA(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    }
    p.num_tiles = (int)((p.total_rows + TM - 1) / TM);
    if (p.num_tiles == 0) return 0;
    p.gather_mode = opts().mlp_gather;   // default 0; measured (profiles/r1_notes.md): register gather 1.53 ms, cp.async.cg 1.66, cp.async.ca 1.67 per batch of SA chains
    const int L = p.num_layers;
    int np_total = 0, np_max = 0;
    for (int l = 0; l < L; ++l) { np_total += p.np[l]; np_max = p.np[l] > np_max ? p.np[l] : np_max; }
    p.b_stage_bytes = (np_max < B_TILE_ROWS ? np_max : B_TILE_ROWS) * KC * 4;
    int need = p.np[0];
    if (L >= 2) need = p.np[0] + p.np[1];
    if (L >= 3 && p.np[1] + p.np[2] > need) need = p.np[1] + p.np[2];
    int cols = 32;
    while (cols < need) cols <<= 1;
    p.tmem_cols = cols;
    p.dcol[0] = 0;
    if (L >= 2) p.dcol[1] = cols - p.np[1];
    if (L >= 3) p.dcol[2] = 0;
    // Row-thread parallelism: NG groups of 4 row warps in one CTA (chunks dealt round-robin), or -- when TMEM and
    // shared memory allow several CTAs per SM -- NG=1 with 2 or 3 independent CTAs (the 3-CTA build is capped at 112
    // registers per thread).
    const int sm_smem = 227 * 1024;
    int ng = opts().mlp_ng;
    const bool ng_forced = ng != 0;
    int occ = 1;
    if (ng == 0) ng = (cols <= 256) ? 1 : 2;
    if (ng == 1) occ = 512 / cols > 3 ? 3 : 512 / cols;
    // 129..256 TMEM columns: two CTAs fit either way, and two CTAs of 8 row warps beat two of 4 (measured per level,
    // profiles/r1_notes.md: FP0 0.201 -> 0.165 ms, SA2 0.311 -> 0.295); the 3-CTA build stays best below 128 columns
    if (!ng_forced && ng == 1 && occ == 2) ng = 2;
    if (ng == 2) occ = 512 / cols >= 2 ? 2 : 1;
    if (const int o = opts().mlp_occ; o >= 1 && o < occ) occ = o;
    size_t smem = 0;
    for (;; --occ) {
        int depth = occ >= 2 ? 3 : 4;
        for (; depth >= 2; --depth) {
            smem = chain_smem_bytes(ng, depth, depth, p.b_stage_bytes, np_total);
            if ((smem + 1024 + 3744) * occ <= (size_t)sm_smem && smem <= (size_t)max_optin) { p.na = p.nb = depth; break; }
        }
        if (depth >= 2 || occ == 1) break;
    }
    PRB_REQUIRE(smem <= (size_t)max_optin, "mlp: %zu bytes of shared memory needed, %d available", smem, max_optin);
    // Tiles are dealt statically (tile += gridDim.x), so a CTA that cannot start with the first wave doubles the
    // kernel's duration.  When other streams hold SMs (BatchPipeline: the single-CTA-per-scene FPS of the next
    // batches), PRB_MLP_SMS sizes the grid for the SMs that are actually free.
    int sms = num_sms();
    if (const int v = opts().mlp_sms; v >= 1 && v < sms) sms = v;
    int grid = sms * occ;
    if (grid > p.num_tiles) grid = p.num_tiles;
#define PRB_LAUNCH_CHAIN(NGV, MB)                                                                                              \
    do {                                                                                                                       \
        PRB_CUDA(cudaFuncSetAttribute(mlp_chain_kernel<NGV, MB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));    \
        mlp_chain_kernel<NGV, MB><<<grid, 128 * NGV + 64, smem, st>>>(p);                                                     \
    } while (0)
    if (ng == 1 && occ >= 3) PRB_LAUNCH_CHAIN(1, 3);
    else if (ng == 1) PRB_LAUNCH_CHAIN(1, 2);
    else if (ng == 2 && occ >= 2) PRB_LAUNCH_CHAIN(2, 2);
    else if (ng == 2) PRB_LAUNCH_CHAIN(2, 1);
    else PRB_LAUNCH_CHAIN(3, 1);
#undef PRB_LAUNCH_CHAIN
    return check_launch("mlp_chain_kernel");
}

// TMEM feasibility of fusing layers [l0, l1).  Legacy kernel: accumulators ping-pong between column 0 and the top.
// Pipelined kernel: every mid layer owns a region, the last layer needs at least one 32-column slice buffer.
static bool fits_legacy(const LayerGeom *g, int l0, int l1) {
    const int n = l1 - l0;
    if (n == 1) return g[l0].np <= 512;
    if (n == 2) return g[l0].np + g[l0 + 1].np <= 512;
    return g[l0].np + g[l0 + 1].np <= 512 && g[l0 + 2].np + g[l0 + 1].np <= 512;
}
static bool fits_pipe(const LayerGeom *g, int l0, int l1) {
    int mid = 0;
    for (int l = l0; l + 1 < l1; ++l) mid += g[l].np;
    // keep at least two 64-column slice buffers (or the whole last layer) next to the mid regions
    const int last = g[l1 - 1].np;
    const int z = last < 64 ? last : 64;
    return g[l1 - 1].np <= 512 && mid + (l1 - l0 > 1 ? 2 * z : 0) <= 512;
}
static bool fits(const LayerGeom *g, int l0, int l1) { return use_pipe() ? fits_pipe(g, l0, l1) : fits_legacy(g, l0, l1); }

struct ChainIO {
    int kind, split;          // packing kind (0 SA, 1 FP, 2 DIRECT) and its split argument
    ChainParams base;         // mode_in / sources / output filled by the caller
    long rows;
};

static size_t chain_workspace_bytes(long rows, int L, int kind, int c_in, int split, const int *c_out) {
    PackSegs ps;
    default_segs(kind, c_in, split, &ps);
    LayerGeom g[MAX_LAYERS];
    chain_geometry(L, ps.nseg, ps.width, c_out, g, nullptr);
    // worst case: two ping-pong row buffers of the widest padded layer
    int wmax = 0;
    for (int l = 0; l < L; ++l) wmax = g[l].np > wmax ? g[l].np : wmax;
    bool split_needed = !fits_legacy(g, 0, L) || !fits_pipe(g, 0, L);   // either kernel may be chosen at launch time
    const size_t rows_pad = (size_t)((rows + TM - 1) / TM * TM);
    return split_needed ? 2 * (rows_pad * wmax * sizeof(float) + 256) : 256;
}

// run the whole chain, splitting where TMEM cannot hold two consecutive accumulators
static int run_chain(const ChainIO &io, const prb_mlp_desc *mlp, void *workspace, size_t workspace_bytes, cudaStream_t st) {
    const int L = mlp->num_layers;
    PRB_REQUIRE(io.rows < 0x7fffff00L, "mlp: %ld rows exceed the 2^31 row limit", io.rows);
    PRB_REQUIRE(L >= 1 && L <= MAX_LAYERS, "mlp: num_layers %d unsupported", L);
    PackSegs ps;
    default_segs(io.kind, mlp->c_in, io.split, &ps);
    LayerGeom g[MAX_LAYERS];
    chain_geometry(L, ps.nseg, ps.width, mlp->c_out, g, nullptr);
    for (int l = 0; l < L; ++l) PRB_REQUIRE(g[l].np <= MAX_NP, "mlp: layer width %d > %d unsupported", mlp->c_out[l], MAX_NP);
    size_t soff[MAX_LAYERS];
    size_t so = 0;
    for (int l = 0; l < L; ++l) { soff[l] = so; so += (size_t)g[l].np; }

    const long rows_pad = (io.rows + TM - 1) / TM * TM;
    int l0 = 0;
    const float *cur_rows = nullptr;
    int cur_pitch = 0;
    int pingpong = 0;
    while (l0 < L) {
        int l1 = L;
        while (l1 > l0 + 1 && !fits(g, l0, l1)) --l1;
        ChainParams p = io.base;
        p.unit_scale = mlp->scale ? 0 : 1;
        p.linear_last = (l1 == L && (mlp->flags & 1)) ? 1 : 0;
        p.trace = opts().mlp_trace ? 1 : 0;
        p.a_tmem = opts().mlp_atmem ? 1 : 0;   // default 1; measured (profiles/r1_notes.md): SA chains 1.124 -> 1.088 ms per batch; 0 = shared-memory stages
        p.sleepy = opts().mlp_sleepy;
        p.total_rows = io.rows;
        p.num_layers = l1 - l0;
        for (int l = l0; l < l1; ++l) {
            const int i = l - l0;
            p.nchunks[i] = g[l].k_chunks;
            p.np[i] = g[l].np;
            p.w[i] = mlp->packed_w + g[l].w_off;
            p.scale[i] = mlp->scale ? mlp->scale + soff[l] : nullptr;
            p.shift[i] = mlp->shift + soff[l];
        }
        if (l0 > 0) {  // continue from materialised rows
            p.mode_in = IN_DIRECT;
            p.x_rows = cur_rows;
            p.x_pitch = cur_pitch;
            p.x2_rows = nullptr;
            p.nseg = 1; p.seg_chunks[0] = g[l0].k_chunks; p.seg_width[0] = cur_pitch;
        } else {
            p.nseg = ps.nseg;
            for (int s = 0; s < ps.nseg; ++s) { p.seg_chunks[s] = round_up(ps.width[s], KC) / KC; p.seg_width[s] = ps.width[s]; }
        }
        if (l1 < L) {  // materialise this segment's activations as rows
            size_t buf_bytes = (size_t)rows_pad * g[l1 - 1].np * sizeof(float);
            PRB_REQUIRE(workspace && workspace_bytes >= 2 * buf_bytes, "mlp: workspace too small (%zu < %zu)", workspace_bytes, 2 * buf_bytes);
            float *dst = (float *)((char *)workspace + (pingpong ? workspace_bytes / 2 / 256 * 256 : 0));
            p.mode_out = OUT_ROWS;
            p.round_out = 1;
            p.out_pm = nullptr;
            p.out = dst;
            p.out_pitch = g[l1 - 1].np;
            p.c_last = g[l1 - 1].np;
            int rc = launch_chain(p, st);
            if (rc) return rc;
            cur_rows = dst;
            cur_pitch = g[l1 - 1].np;
            pingpong ^= 1;
        } else {
            // row-major output: write the padded width so the padding channels are defined (zero)
            p.c_last = p.mode_out == OUT_ROWS ? g[L - 1].np : mlp->c_out[L - 1];
            int rc = launch_chain(p, st);
            if (rc) return rc;
        }
        l0 = l1;
    }
    return 0;
}

}  // namespace prb

extern "C" {

// debug: copy the phase trace of the last traced launch (32 tiles x 16 stamps, clock64 of CTA 0's row thread 0)
PRB_API int prb_debug_mlp_trace(long long *dst) {
    PRB_CUDA(cudaDeviceSynchronize());
    PRB_CUDA(cudaMemcpyFromSymbol(dst, g_trace, sizeof(long long) * 32 * 16));
    static long long zeros[32 * 16];
    PRB_CUDA(cudaMemcpyToSymbol(g_trace, zeros, sizeof(zeros)));
    return 0;
}

PRB_API size_t prb_sa_workspace_bytes(int b, int npoint, int nsample, int c_feat, int num_layers, const int *c_out) {
    return chain_workspace_bytes((long)b * npoint * nsample, num_layers, 0, 3 + c_feat, c_feat, c_out);
}
PRB_API size_t prb_fp_workspace_bytes(int b, int n, int c_known, int c_skip, int num_layers, const int *c_out) {
    return chain_workspace_bytes((long)b * n, num_layers, 1, c_known + c_skip, c_known, c_out);
}
PRB_API size_t prb_rows_workspace_bytes(long rows, int c_in, int num_layers, const int *c_out) {
    return chain_workspace_bytes(rows, num_layers, 2, c_in, 0, c_out);
}

PRB_API int prb_sa_group_mlp_max_ws(int b, int n, int npoint, int nsample, int c_feat, const float *xyz, const float *new_xyz,
                                    const float *feats_pm, const int *idx, const prb_mlp_desc *mlp, float *out, float *out_pm,
                                    int out_stride_c, int out_c_off, void *workspace, size_t workspace_bytes, void *stream) {
    PRB_REQUIRE(b >= 0 && n > 0 && npoint > 0 && nsample > 0 && xyz && new_xyz && idx && mlp && out, "sa_group_mlp_max: bad arguments");
    PRB_REQUIRE(mlp->c_in == 3 + c_feat, "sa_group_mlp_max: c_in %d != 3 + c_feat %d", mlp->c_in, c_feat);
    PRB_REQUIRE(c_feat == 0 || feats_pm, "sa_group_mlp_max: features missing");
    PRB_REQUIRE(nsample >= 4 && nsample <= 128 && (nsample & (nsample - 1)) == 0, "sa_group_mlp_max: nsample %d must be a power of two in [4,128]", nsample);
    if (b == 0) return 0;
    ChainIO io;
    memset(&io, 0, sizeof(io));
    io.kind = 0; io.split = c_feat;
    io.rows = (long)b * npoint * nsample;
    io.base.mode_in = IN_SA; io.base.mode_out = OUT_SA_MAX;
    io.base.n = n; io.base.npoint = npoint; io.base.ns = nsample; io.base.c_feat = c_feat;
    io.base.log_ns = 0;
    while ((1 << io.base.log_ns) < nsample) ++io.base.log_ns;
    io.base.xyz = xyz; io.base.new_xyz = new_xyz; io.base.feats_pm = feats_pm; io.base.idx = idx;
    io.base.out = out; io.base.out_pm = out_pm; io.base.out_stride_c = out_stride_c; io.base.out_c_off = out_c_off;
    return run_chain(io, mlp, workspace, workspace_bytes, (cudaStream_t)stream);
}

// SA chains with c_feat <= 5, layer 0 outside the tensor core: the gather warps evaluate relu(W0 . [x_j - c, f_j] + shift0)
// (l0_w: c0 x 8 floats per channel [wx, wy, wz, wf0 .. wf4], BN scale folded, zero beyond 3 + c_feat; l0_shift: c0 floats;
// both device) and write it as the A operand of `mlp`, the chain of the original layers 1 .. L-1 packed as plain rows
// (kind 2, c_in = c0).  One tensor-memory hand-off per tile fewer than prb_sa_group_mlp_max_ws with the same operands
// (tf32-rounded inputs and weights); the chain must fit one launch.
PRB_API int prb_sa_group_mlp_max_l0(int b, int n, int npoint, int nsample, int c_feat, const float *xyz, const float *new_xyz,
                                    const float *feats_pm, const int *idx, int c0, const float *l0_w, const float *l0_shift,
                                    const prb_mlp_desc *mlp, float *out, float *out_pm, int out_stride_c, int out_c_off, void *stream) {
    PRB_REQUIRE(b >= 0 && n > 0 && npoint > 0 && nsample > 0 && xyz && new_xyz && idx && mlp && out && l0_w && l0_shift,
                "sa_group_mlp_max_l0: bad arguments");
    PRB_REQUIRE(c_feat >= 0 && c_feat <= L0_IN - 3, "sa_group_mlp_max_l0: c_feat %d > %d", c_feat, L0_IN - 3);
    PRB_REQUIRE(c_feat == 0 || feats_pm, "sa_group_mlp_max_l0: features missing");
    PRB_REQUIRE(c0 >= 1 && c0 <= MAX_NP && mlp->c_in == c0, "sa_group_mlp_max_l0: layer-0 width %d / chain input %d", c0, mlp->c_in);
    PRB_REQUIRE(mlp->scale == nullptr, "sa_group_mlp_max_l0: the BN scale must be folded into the weights");
    PRB_REQUIRE(nsample >= 4 && nsample <= 128 && (nsample & (nsample - 1)) == 0, "sa_group_mlp_max_l0: nsample %d must be a power of two in [4,128]", nsample);
    PRB_REQUIRE(use_pipe(), "sa_group_mlp_max_l0: needs the pipelined kernel (mlp_pipeline = 1, mlp_gather = 0)");
    const int L = mlp->num_layers;
    PRB_REQUIRE(L >= 1 && L <= MAX_LAYERS, "sa_group_mlp_max_l0: num_layers %d unsupported", L);
    LayerGeom g[MAX_LAYERS];
    chain_geometry(L, 1, &c0, mlp->c_out, g, nullptr);
    PRB_REQUIRE(fits_pipe(g, 0, L), "sa_group_mlp_max_l0: the chain does not fit one launch");
    if (b == 0) return 0;
    ChainIO io;
    memset(&io, 0, sizeof(io));
    io.kind = 2; io.split = 0;
    io.rows = (long)b * npoint * nsample;
    io.base.mode_in = IN_SA; io.base.mode_out = OUT_SA_MAX;
    io.base.sa_l0 = 1; io.base.l0_c = c0; io.base.l0_np = round_up(c0, KC); io.base.l0_w = l0_w; io.base.l0_shift = l0_shift;
    io.base.n = n; io.base.npoint = npoint; io.base.ns = nsample; io.base.c_feat = c_feat;
    io.base.log_ns = 0;
    while ((1 << io.base.log_ns) < nsample) ++io.base.log_ns;
    io.base.xyz = xyz; io.base.new_xyz = new_xyz; io.base.feats_pm = feats_pm; io.base.idx = idx;
    io.base.out = out; io.base.out_pm = out_pm; io.base.out_stride_c = out_stride_c; io.base.out_c_off = out_c_off;
    return run_chain(io, mlp, nullptr, 0, (cudaStream_t)stream);
}

PRB_API int prb_fp_interp_mlp_ws(int b, int n, int m, int c_known, int c_skip, const float *known_pm, const int *idx,
                                 const float *weight, const float *skip, const prb_mlp_desc *mlp, float *out, float *out_pm,
                                 void *workspace, size_t workspace_bytes, void *stream) {
    PRB_REQUIRE(b >= 0 && n > 0 && m > 0 && c_known > 0 && known_pm && idx && weight && mlp && out, "fp_interp_mlp: bad arguments");
    PRB_REQUIRE(mlp->c_in == c_known + c_skip, "fp_interp_mlp: c_in %d != %d + %d", mlp->c_in, c_known, c_skip);
    PRB_REQUIRE(c_skip == 0 || skip, "fp_interp_mlp: skip features missing");
    if (b == 0) return 0;
    ChainIO io;
    memset(&io, 0, sizeof(io));
    io.kind = 1; io.split = c_known;
    io.rows = (long)b * n;
    io.base.mode_in = IN_FP; io.base.mode_out = OUT_FP;
    io.base.n = n; io.base.m = m; io.base.c_known = c_known; io.base.c_skip = c_skip;
    io.base.known_pm = known_pm; io.base.idx = idx; io.base.weight = weight; io.base.skip = skip;
    io.base.out = out; io.base.out_pm = out_pm; io.base.out_stride_c = mlp->c_out[mlp->num_layers - 1]; io.base.out_c_off = 0;
    return run_chain(io, mlp, workspace, workspace_bytes, (cudaStream_t)stream);
}

// plain rows -> MLP -> rows (also the unit-test doorway of the tensor-core chain)
PRB_API int prb_mlp_rows(long rows, int c_in, const float *x_rows, const prb_mlp_desc *mlp, float *out_rows, int out_pitch,
                         void *workspace, size_t workspace_bytes, void *stream) {
    PRB_REQUIRE(rows >= 0 && c_in > 0 && x_rows && mlp && out_rows, "mlp_rows: bad arguments");
    PRB_REQUIRE(mlp->c_in == c_in, "mlp_rows: c_in mismatch");
    const int np_last = (mlp->c_out[mlp->num_layers - 1] + 31) / 32 * 32;
    PRB_REQUIRE(out_pitch >= np_last && (out_pitch & 3) == 0, "mlp_rows: out_pitch %d must be >= %d and a multiple of 4", out_pitch, np_last);
    if (rows == 0) return 0;
    ChainIO io;
    memset(&io, 0, sizeof(io));
    io.kind = 2; io.split = 0;
    io.rows = rows;
    io.base.mode_in = IN_DIRECT; io.base.mode_out = OUT_ROWS;
    io.base.x_rows = x_rows; io.base.x_pitch = c_in;
    io.base.out = out_rows; io.base.out_pitch = out_pitch;
    return run_chain(io, mlp, workspace, workspace_bytes, (cudaStream_t)stream);
}

PRB_API size_t prb_rows2_workspace_bytes(long rows, int c_a, int c_b, int num_layers, const int *c_out) {
    return chain_workspace_bytes(rows, num_layers, c_b > 0 ? 1 : 2, c_a + c_b, c_b > 0 ? c_a : 0, c_out);
}

PRB_API int prb_mlp_rows2(long rows, int c_a, const float *a_rows, int a_pitch, int c_b, const float *b_rows, int b_pitch,
                          const prb_mlp_desc *mlp, float *out_rows, int out_pitch, void *workspace, size_t workspace_bytes,
                          void *stream) {
    PRB_REQUIRE(rows >= 0 && c_a > 0 && a_rows && a_pitch >= c_a && mlp && out_rows, "mlp_rows2: bad arguments");
    PRB_REQUIRE(c_b >= 0 && (c_b == 0 || (b_rows && b_pitch >= c_b)), "mlp_rows2: bad second segment");
    PRB_REQUIRE(mlp->c_in == c_a + c_b, "mlp_rows2: c_in %d != %d + %d", mlp->c_in, c_a, c_b);
    PRB_REQUIRE(c_b == 0 || use_pipe(), "mlp_rows2: two input segments need the pipelined kernel (mlp_pipeline = 1, mlp_gather = 0)");
    const int np_last = (mlp->c_out[mlp->num_layers - 1] + 31) / 32 * 32;
    PRB_REQUIRE(out_pitch >= np_last && (out_pitch & 3) == 0, "mlp_rows2: out_pitch %d must be >= %d and a multiple of 4", out_pitch, np_last);
    if (rows == 0) return 0;
    ChainIO io;
    memset(&io, 0, sizeof(io));
    io.kind = c_b > 0 ? 1 : 2; io.split = c_b > 0 ? c_a : 0;      // weights packed with prb_mlp_pack_weights_ex(kind, split, ...)
    io.rows = rows;
    io.base.mode_in = IN_DIRECT; io.base.mode_out = OUT_ROWS;
    io.base.x_rows = a_rows; io.base.x_pitch = a_pitch;
    io.base.x2_rows = c_b > 0 ? b_rows : nullptr; io.base.x2_pitch = b_pitch;
    io.base.out = out_rows; io.base.out_pitch = out_pitch;
    return run_chain(io, mlp, workspace, workspace_bytes, (cudaStream_t)stream);
}

// header forms without an explicit workspace: valid only for chains that need no split
int prb_sa_group_mlp_max(int b, int n, int npoint, int nsample, int c_feat, const float *xyz, const float *new_xyz,
                         const float *feats_pm, const int *idx, const prb_mlp_desc *mlp, float *out, int out_stride_c,
                         int out_c_off, void *stream) {
    return prb_sa_group_mlp_max_ws(b, n, npoint, nsample, c_feat, xyz, new_xyz, feats_pm, idx, mlp, out, nullptr, out_stride_c,
                                   out_c_off, nullptr, 0, stream);
}
int prb_fp_interp_mlp(int b, int n, int m, int c_known, int c_skip, const float *known_pm, const int *idx, const float *weight,
                      const float *skip, const prb_mlp_desc *mlp, float *out, void *stream) {
    return prb_fp_interp_mlp_ws(b, n, m, c_known, c_skip, known_pm, idx, weight, skip, mlp, out, nullptr, nullptr, 0, stream);
}

}  // extern "C"
