// smenv_mlp.cuh -- the one dense contraction of the step loop on the 5th-generation tensor cores: batched inference of
// the risk network and of the backup policy (safe_motions_base.py:1498-1603, actions.py:303-340;
// keras_fcnet_last_layer_activation.py:86-136, :187-202; train_risk_network.py).
//
//   risk(obs, action) = sigmoid(W4 selu(W3 selu(W2 selu(W1 [obs, action]))))      30 -> 512 -> 256 -> 128 -> 1
//   backup(obs)       = tanh(W3 swish(W2 swish(W1 obs)))[0:7]                      23 -> 256 -> 128 -> 14
//
// One CTA (512 threads) owns a tile of 128 envs = the 128 rows of a tcgen05.mma (cta_group::1, M = 128) and runs the
// whole network on it without leaving the SM:
//   * activations live in shared memory as fp16 in the canonical K-major no-swizzle UMMA layout (8x16-byte core
//     matrices, SBO = 128 B between 8-row groups, LBO = 2048 B between 8-column groups), weights are packed into the
//     same layout on the host once and streamed through shared memory in 64-column K chunks;
//   * one thread issues tcgen05.mma.kind::f16 (fp16 x fp16 -> fp32) into TMEM (N = 512 as two N = 256 instructions),
//     tcgen05.commit signals an mbarrier;
//   * the epilogue reads the accumulator row of each env with tcgen05.ld (four threads per TMEM lane, a quarter of
//     the columns each: the epilogue is latency-bound, more warps hide it), adds the bias,
//     applies selu / swish and writes the next layer's operand straight back to shared memory; the last hidden layer
//     is contracted with the tiny output layer on the CUDA cores while it is still in registers.
//   * the weight chunks stream through two 32 KB buffers with 1-D bulk TMA (cp.async.bulk -> mbarrier complete_tx),
//     issued two chunks ahead by the MMA-issuing thread, across layer and tile boundaries, so that the copies overlap
//     the MMAs and the epilogues.
#pragma once
#include <cuda_fp16.h>

#include "smenv_device.cuh"

#define MLP_MAX_TC 3
#define MLP_MAX_OUT 16 /* outputs of the CUDA-core output layer; stored padded to 8 or 16 columns (MlpNet.out_pad) */
#define MLP_WOUT_FLOATS 2048 /* shared-memory floats of the output layer: last hidden width x out_pad */
#define MLP_TILE_M 128
#define MLP_THREADS 512 /* four warps per TMEM lane quarter: each handles a quarter of the accumulator columns */
#define MLP_PARTS (MLP_THREADS / MLP_TILE_M)
#define MLP_CHUNK_K 64
#define MLP_MAX_WIDTH 512

// K columns of a layer's weights staged per chunk: at most MLP_CHUNK_K and at most 32 KB of shared memory
__host__ __device__ __forceinline__ int mlp_chunk_k(int N, int K) {
    int c = K < MLP_CHUNK_K ? K : MLP_CHUNK_K;
    const int cap = 16384 / N;   // 32768 bytes / (N rows * 2 bytes)
    return c < cap ? c : cap;
}

enum { MLP_ACT_SELU = 0, MLP_ACT_SWISH = 1 };
enum { MLP_OUT_SIGMOID = 0, MLP_OUT_TANH = 1 };

struct MlpNet {
    int n_tc;                 // tensor-core layers
    int n_in, k_in;           // real and padded (16, 32 or 64) input width
    int dims[MLP_MAX_TC];     // widths of the tensor-core layers (multiples of 16; > 256 only as 512)
    int hidden_act, out_act;
    int n_out;                // outputs of the final CUDA-core layer (<= MLP_MAX_OUT)
    int out_pad;              // 8 or 16: column stride of w_out / b_out
    const __half* w[MLP_MAX_TC];  // packed K chunks, canonical layout
    const float* b[MLP_MAX_TC];
    const float* w_out;       // [dims[n_tc-1]][out_pad]
    const float* b_out;       // [out_pad]
    const float* w32[MLP_MAX_TC];  // float32 kernels [in][out] row-major of the hidden layers (exact evaluation of a few rows)
};

struct MlpArgs {
    MlpNet net;
    int n;                    // rows (envs)
    const float* in[3];            // input row = [segment 0, segment 1, segment 2, zero padding]
    int in_stride[3], in_w[3];     // row stride (floats) and width of every segment (pointers are pre-offset)
    float* out; int out_stride;
};

// ------------------------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------------------------
// shared-memory matrix descriptor: K-major, no swizzle (layout type 0), version 1 (sm_100)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3ffffu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
// instruction descriptor of kind::f16: D = f32, A = B = f16, both K-major, M x N
__device__ __forceinline__ uint32_t umma_idesc_f16(int m, int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
                 :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// 32 consecutive accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* r) {
    uint32_t u[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
          "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]),
          "=r"(u[16]), "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]),
          "=r"(u[24]), "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) r[i] = __uint_as_float(u[i]);
}

// 16 consecutive accumulator columns, asynchronously: the registers are valid after tmem_wait16 on the same array (the
// wait names them as in/out operands, so the compiler cannot move their uses in front of it)
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t* u) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
          "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait16(uint32_t* u) {
    asm volatile("tcgen05.wait::ld.sync.aligned;\n"
                 : "+r"(u[0]), "+r"(u[1]), "+r"(u[2]), "+r"(u[3]), "+r"(u[4]), "+r"(u[5]), "+r"(u[6]), "+r"(u[7]),
                   "+r"(u[8]), "+r"(u[9]), "+r"(u[10]), "+r"(u[11]), "+r"(u[12]), "+r"(u[13]), "+r"(u[14]), "+r"(u[15])
                 :: "memory");
}

__device__ __forceinline__ float mlp_hidden_act(float x, int act) {
    if (act == MLP_ACT_SELU) return 1.0507009873554805f * (x > 0.0f ? x : 1.6732632423543772f * (__expf(x) - 1.0f));
    return x / (1.0f + __expf(-x));  // swish
}

// shared memory carve-up (bytes)
#define MLP_W_BUF_BYTES 32768
#define MLP_MAX_LAST 256                                   /* widest last hidden layer */
#define MLP_SM_ACT 0                                       /* 128 x 512 fp16 */
#define MLP_SM_W (MLP_TILE_M * MLP_MAX_WIDTH * 2)         /* two weight chunks: <= 512 x 32 or 256 x 64 fp16 each */
#define MLP_SM_IN (MLP_SM_W + 2 * MLP_W_BUF_BYTES)         /* 128 x 64 fp16 */
#define MLP_SM_WOUT (MLP_SM_IN + MLP_TILE_M * 64 * 2)      /* last hidden width x out_pad floats (<= MLP_WOUT_FLOATS) */
#define MLP_SM_BIAS (MLP_SM_WOUT + MLP_WOUT_FLOATS * 4)
#define MLP_SM_BAR (MLP_SM_BIAS + MLP_MAX_TC * MLP_MAX_WIDTH * 4)
#define MLP_SM_BYTES (MLP_SM_BAR + 64)

__global__ void __launch_bounds__(MLP_THREADS, 1) mlp_kernel(MlpArgs A) {
    extern __shared__ __align__(1024) unsigned char mlp_smem[];
    unsigned char* a_act = mlp_smem + MLP_SM_ACT;
    unsigned char* w_buf = mlp_smem + MLP_SM_W;
    unsigned char* a_in = mlp_smem + MLP_SM_IN;
    float* w_out = reinterpret_cast<float*>(mlp_smem + MLP_SM_WOUT);
    float* bias = reinterpret_cast<float*>(mlp_smem + MLP_SM_BIAS);
    // partial outputs of the column quarters of a row: [MLP_PARTS][128][MLP_MAX_OUT] floats in the activation buffer,
    // which is free once the MMAs of the last tensor-core layer are done
    float* part = reinterpret_cast<float*>(mlp_smem + MLP_SM_ACT);
    uint64_t* bar = reinterpret_cast<uint64_t*>(mlp_smem + MLP_SM_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mlp_smem + MLP_SM_BAR + 48);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int rtid = tid & (MLP_TILE_M - 1);   // row of the tile this thread serves
    const int half = tid >> 7;                 // which quarter of the columns / input segments this thread handles
    const int quarter = warp & 3;              // TMEM lane quarter the warp may access
    const MlpNet& net = A.net;
    const int n_last = net.dims[net.n_tc - 1];

    // ---------------- one-time setup: barrier, tensor memory, small parameters
    uint64_t* bar_full = bar;        // [2] weight chunk landed in buffer b
    uint64_t* bar_empty = bar + 2;   // [2] the MMAs reading buffer b are done
    uint64_t* bar_done = bar + 4;    // all MMAs of a layer are done
    if (tid == 0) {
        for (int i = 0; i < 5; ++i) mbar_init(bar + i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" :: "r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    for (int l = 0; l < net.n_tc; ++l)
        for (int i = tid; i < net.dims[l]; i += MLP_THREADS) bias[l * MLP_MAX_WIDTH + i] = __ldg(net.b[l] + i);
    const int out_pad = net.out_pad;
    for (int i = tid; i < n_last * out_pad; i += MLP_THREADS) w_out[i] = __ldg(net.w_out + i);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    uint32_t done_phase = 0;
    const int n_tiles = (A.n + MLP_TILE_M - 1) / MLP_TILE_M;
    // ---------------- weight streaming state of the issuing thread: chunks are numbered g = 0, 1, ... over all layers
    // of all tiles of this CTA; chunk g uses buffer g & 1 for the (g >> 1)-th time
    int chunks_per_tile = 0;
    {
        int K = net.k_in;
        for (int l = 0; l < net.n_tc; ++l) { chunks_per_tile += K / mlp_chunk_k(net.dims[l], K); K = net.dims[l]; }
    }
    const int my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    int pf_left = chunks_per_tile * my_tiles, pf_g = 0, pf_layer = 0, pf_chunk = 0, pf_K = net.k_in;  // prefetch cursor
    int g = 0;                                                                                      // consume cursor
    auto prefetch = [&]() {
        if (pf_left == 0) return;
        const int b = pf_g & 1, u = pf_g >> 1;
        if (u > 0) mbar_wait(&bar_empty[b], (uint32_t)(u - 1) & 1u);   // the previous user of the buffer is done
        const int N = net.dims[pf_layer];
        const int ck = mlp_chunk_k(N, pf_K);
        const uint32_t bytes = (uint32_t)(N * ck * 2);
        mbar_expect_tx(&bar_full[b], bytes);
        tma_bulk_g2s(w_buf + b * MLP_W_BUF_BYTES, reinterpret_cast<const unsigned char*>(net.w[pf_layer]) + (size_t)pf_chunk * bytes,
                     bytes, &bar_full[b]);
        ++pf_g; --pf_left;
        if (++pf_chunk == pf_K / ck) {
            pf_chunk = 0; pf_K = N;
            if (++pf_layer == net.n_tc) { pf_layer = 0; pf_K = net.k_in; }
        }
    };
    if (tid == 0) { prefetch(); prefetch(); }
    // this thread's slot inside an 8-row core-matrix group (row = tid): byte offset of its 16-byte row segment
    const uint32_t row_off = (uint32_t)(rtid >> 3) * 128u + (uint32_t)(rtid & 7) * 16u;

#pragma unroll 1
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int row = tile * MLP_TILE_M + rtid;
        const bool valid = row < A.n;
        // ---------------- input rows -> fp16 operand of the first layer
        for (int kc = half; kc < net.k_in / 8; kc += MLP_PARTS) {
            __align__(16) __half h[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int k = kc * 8 + i;
                float x = 0.0f;
                if (valid) {
                    if (k < A.in_w[0]) x = A.in[0][(size_t)row * A.in_stride[0] + k];
                    else if (k < A.in_w[0] + A.in_w[1]) x = A.in[1][(size_t)row * A.in_stride[1] + (k - A.in_w[0])];
                    else if (k < A.in_w[0] + A.in_w[1] + A.in_w[2])
                        x = A.in[2][(size_t)row * A.in_stride[2] + (k - A.in_w[0] - A.in_w[1])];
                }
                h[i] = __float2half_rn(x);
            }
            *reinterpret_cast<uint4*>(a_in + kc * 2048 + row_off) = *reinterpret_cast<const uint4*>(h);
        }
        fence_async_smem();
        __syncthreads();
        uint32_t a_src = smem_u32(a_in);
        int K = net.k_in;
        float acc_out[MLP_MAX_OUT];
#pragma unroll
        for (int o = 0; o < MLP_MAX_OUT; ++o) acc_out[o] = 0.0f;
#pragma unroll 1
        for (int l = 0; l < net.n_tc; ++l) {
            const int N = net.dims[l];
            const int chunk_k = mlp_chunk_k(N, K);
            const int n_chunks = K / chunk_k;
            const uint32_t lbo_b = (uint32_t)(N / 8) * 128u;
            // ---- one thread: wait for each weight chunk, issue its MMAs, release the buffer, fetch two chunks ahead
            if (tid == 0) {
#pragma unroll 1
                for (int c = 0; c < n_chunks; ++c) {
                    const int b = g & 1;
                    mbar_wait(&bar_full[b], (uint32_t)(g >> 1) & 1u);
                    tc_fence_after();
                    const uint32_t wb = smem_u32(w_buf + b * MLP_W_BUF_BYTES);
                    for (int kk = 0; kk < chunk_k / 16; ++kk) {
                        const uint64_t adesc = umma_desc(a_src + (uint32_t)((c * chunk_k + kk * 16) / 8) * 2048u, 2048u, 128u);
                        for (int nh = 0; nh * 256 < N; ++nh) {
                            const int n_mma = N - nh * 256 < 256 ? N - nh * 256 : 256;
                            const uint64_t bdesc = umma_desc(wb + (uint32_t)(kk * 2) * lbo_b + (uint32_t)nh * 32u * 128u, lbo_b, 128u);
                            umma_f16(tmem + (uint32_t)nh * 256u, adesc, bdesc, umma_idesc_f16(MLP_TILE_M, n_mma),
                                     (c > 0 || kk > 0) ? 1u : 0u);
                        }
                    }
                    umma_commit(&bar_empty[b]);
                    ++g;
                    if (c == n_chunks - 1) umma_commit(bar_done);
                    prefetch();
                }
            }
            mbar_wait(bar_done, done_phase);   // all MMAs of the layer are done: the accumulator may be read
            done_phase ^= 1u;
            tc_fence_after();
            // ---------------- epilogue: accumulator row of this env -> bias, activation -> next operand / output
            const bool last = l == net.n_tc - 1;
            const float* bl = bias + l * MLP_MAX_WIDTH;
            // 16 columns at a time, the next 16 in flight while these go through the activation (the load latency of
            // the tensor memory hides behind the arithmetic)
            {
                const uint32_t tbase = tmem + ((uint32_t)(quarter * 32) << 16);
                // blocks of 16 columns; this thread takes blocks half, half + MLP_PARTS, ... (any width that is a multiple of
                // 16: narrow layers leave some of the four column groups idle)
                const int nblk = N / 16;
                const int hidden_act = net.hidden_act, n_out = net.n_out;
                auto process16 = [&](const uint32_t* u, int c) {
                    float r[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) r[j] = mlp_hidden_act(__uint_as_float(u[j]) + bl[c + j], hidden_act);
                    if (!last) {
#pragma unroll
                        for (int g2 = 0; g2 < 2; ++g2) {
                            __align__(16) __half h[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) h[i] = __float2half_rn(r[8 * g2 + i]);
                            *reinterpret_cast<uint4*>(a_act + (uint32_t)((c + 8 * g2) / 8) * 2048u + row_off) =
                                *reinterpret_cast<const uint4*>(h);
                        }
                    } else if (n_out == 1) {   // the risk network: one output column
#pragma unroll
                        for (int j = 0; j < 16; ++j) acc_out[0] = fmaf(r[j], w_out[(c + j) * out_pad], acc_out[0]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float4 wa = *reinterpret_cast<const float4*>(w_out + (c + j) * out_pad);
                            const float4 wb = *reinterpret_cast<const float4*>(w_out + (c + j) * out_pad + 4);
                            acc_out[0] = fmaf(r[j], wa.x, acc_out[0]); acc_out[1] = fmaf(r[j], wa.y, acc_out[1]);
                            acc_out[2] = fmaf(r[j], wa.z, acc_out[2]); acc_out[3] = fmaf(r[j], wa.w, acc_out[3]);
                            acc_out[4] = fmaf(r[j], wb.x, acc_out[4]); acc_out[5] = fmaf(r[j], wb.y, acc_out[5]);
                            acc_out[6] = fmaf(r[j], wb.z, acc_out[6]); acc_out[7] = fmaf(r[j], wb.w, acc_out[7]);
                            if (out_pad == 16) {   // stochastic policies: means and log-std outputs (16 columns)
                                const float4 wc = *reinterpret_cast<const float4*>(w_out + (c + j) * 16 + 8);
                                const float4 wd = *reinterpret_cast<const float4*>(w_out + (c + j) * 16 + 12);
                                acc_out[8] = fmaf(r[j], wc.x, acc_out[8]); acc_out[9] = fmaf(r[j], wc.y, acc_out[9]);
                                acc_out[10] = fmaf(r[j], wc.z, acc_out[10]); acc_out[11] = fmaf(r[j], wc.w, acc_out[11]);
                                acc_out[12] = fmaf(r[j], wd.x, acc_out[12]); acc_out[13] = fmaf(r[j], wd.y, acc_out[13]);
                                acc_out[14] = fmaf(r[j], wd.z, acc_out[14]); acc_out[15] = fmaf(r[j], wd.w, acc_out[15]);
                            }
                        }
                    }
                };
                uint32_t ua[16], ub[16];
                if (half < nblk) {
                    tmem_ld16_issue(tbase + (uint32_t)(half * 16), ua);
                    tmem_wait16(ua);
                }
#pragma unroll 1
                for (int bi = half; bi < nblk; bi += 2 * MLP_PARTS) {
                    const bool second = bi + MLP_PARTS < nblk, third = bi + 2 * MLP_PARTS < nblk;
                    if (second) tmem_ld16_issue(tbase + (uint32_t)((bi + MLP_PARTS) * 16), ub);
                    process16(ua, bi * 16);
                    if (second) {
                        tmem_wait16(ub);
                        if (third) tmem_ld16_issue(tbase + (uint32_t)((bi + 2 * MLP_PARTS) * 16), ua);
                        process16(ub, (bi + MLP_PARTS) * 16);
                        if (third) tmem_wait16(ua);
                    }
                }
            }
            tc_fence_before();
            fence_async_smem();
            __syncthreads();   // operand of the next layer complete; accumulator free for the next MMAs
            a_src = smem_u32(a_act);
            K = N;
        }
        // the column quarters of a row meet in shared memory and are added in a fixed order (bit-reproducible results;
        // the MMAs that read the activation buffer are done, the next tile writes it only after two more barriers)
#pragma unroll
        for (int o = 0; o < MLP_MAX_OUT; ++o) part[(half * MLP_TILE_M + rtid) * MLP_MAX_OUT + o] = acc_out[o];
        __syncthreads();
        if (valid && half == 0) {
            for (int o = 0; o < net.n_out; ++o) {
                float x = part[rtid * MLP_MAX_OUT + o];
#pragma unroll
                for (int q = 1; q < MLP_PARTS; ++q) x += part[(q * MLP_TILE_M + rtid) * MLP_MAX_OUT + o];
                x += __ldg(net.b_out + o);
                A.out[(size_t)row * A.out_stride + o] = net.out_act == MLP_OUT_SIGMOID ? 1.0f / (1.0f + __expf(-x)) : tanhf(x);
            }
        }
        __syncthreads();   // the partial sums are read before the next tile's first layer overwrites the buffer
    }
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem) : "memory");
}

// risky actions are replaced by the backup policy's (actions.py:328-337); risk >= threshold (safe_motions_base.py:1601).
// exec == actions: in place (the stand-alone gate); otherwise the executed actions go to their own buffer and `actions`
// keeps what the policy proposed (the reward's action punishment rates the proposal, safe_motions_base.py:1066).
__global__ void risk_gate_kernel(const float* actions, float* exec, const float* risk, const float* backup, int backup_stride,
                                 int nj, int n, float threshold, uint8_t* risky) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= n) return;
    const bool r = risk[env] >= threshold;
    if (risky) risky[env] = r ? 1 : 0;
    for (int j = 0; j < nj; ++j) {
        const float u = r ? backup[(size_t)env * backup_stride + j] : actions[(size_t)env * nj + j];
        if (r || exec != actions) exec[(size_t)env * nj + j] = u;
    }
}

// get_random_action (safe_motions_base.py:1327-1328) materialised, for the gate in front of smenv_step_random
__global__ void random_actions_kernel(float* actions, int nj, int n, int env_base, uint32_t step_counter, uint32_t k0,
                                      uint32_t k1) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int env = t / nj, j = t % nj;
    if (env >= n) return;
    uint4 r = philox((uint32_t)(env + env_base), step_counter, (uint32_t)j, 0xAC71u, k0, k1);
    actions[t] = 2.0f * u01f(r.x) - 1.0f;
}

// The agent's DiagGaussian head (smenv_step_agent): thread = (env, joint), the eight lanes of an env side by side.
struct AgentArgs {
    const float* policy_out;   // [n][MLP_MAX_OUT] tanh outputs of the agent: nj means, then nj log-std pre-activations
    float* actions;            // [n][nj] clip(sample, -1, 1): what the env executes (or the gate rates)
    float* sample;             // [n][nj] unclipped sample, or NULL
    float* logp;               // [n] log-likelihood of the unclipped sample, or NULL
    float* dist;               // [n][2 nj] mean, log_std, or NULL
    int n, nj, env_base, explore;
    uint32_t step_counter, k0, k1;
    float lo, span;            // log_std = lo + (t + 1) / 2 * span
};

__global__ void agent_action_kernel(AgentArgs A) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int env = t >> 3, j = t & 7;
    const bool live = env < A.n && j < A.nj;
    float eps = 0.0f, log_std = 0.0f;
    if (live) {
        const float* o = A.policy_out + (size_t)env * MLP_MAX_OUT;
        const float mean = o[j];
        float sample = mean;
        if (A.explore) {
            const uint4 r = philox((uint32_t)(env + A.env_base), A.step_counter, (uint32_t)j, 0xA6E7u, A.k0, A.k1);
            sample = diag_gaussian_sample(mean, o[A.nj + j], A.lo, A.span, r, log_std, eps);
        } else {
            log_std = A.lo + 0.5f * (o[A.nj + j] + 1.0f) * A.span;
        }
        A.actions[(size_t)env * A.nj + j] = fminf(1.0f, fmaxf(-1.0f, sample));   // RLlib's clip_actions
        if (A.sample) A.sample[(size_t)env * A.nj + j] = sample;
        if (A.dist) {
            A.dist[(size_t)env * 2 * A.nj + j] = mean;
            A.dist[(size_t)env * 2 * A.nj + A.nj + j] = log_std;
        }
    }
    // DiagGaussian logp of the unclipped sample, summed by lane 0 of the env over the joints in order (bit-reproducible);
    // explore = 0 reports 0 (RLlib's StochasticSampling with explore=False).  Every lane of the warp takes part.
    float sq = 0.0f, ls = 0.0f;
    for (int k = 0; k < A.nj; ++k) {
        const float e = __shfl_sync(FULL, eps, k, 8), l = __shfl_sync(FULL, log_std, k, 8);
        sq = fmaf(e, e, sq);
        ls += l;
    }
    if (j == 0 && env < A.n && A.logp)
        A.logp[env] = A.explore ? -0.5f * sq - ls - 0.91893853320467274f * (float)A.nj : 0.0f;   // 0.5 log(2 pi) per joint
}

// ------------------------------------------------------------------------------------------------------------------
// Exact (float32, CUDA cores) evaluation of a network on a LIST of rows: the tensor-core pass rates every env with fp16
// operands; rows whose risk lies within a band around the threshold are re-rated here so that the gate decision equals the
// float32 decision of the reference's TensorFlow model (safe_motions_base.py:1597-1603), and the backup policy's action
// of the risky envs is computed here in float32 as well (actions.py:328-333).  One CTA = sixteen rows; a thread owns output
// columns, the weights stream through L2 once per sixteen rows.
// ------------------------------------------------------------------------------------------------------------------
#define MLP_EXACT_ROWS 16
#define MLP_EXACT_SMEM (2 * MLP_EXACT_ROWS * MLP_MAX_WIDTH * 4)
struct MlpExactArgs {
    MlpNet net;
    const int* rows;      // [*n_rows] row indices, or NULL: rows 0 .. *n_rows - 1
    const int* n_rows;    // device counter
    int n_rows_host;      // used when n_rows == NULL
    const float* in[3];
    int in_stride[3], in_w[3];
    float* out;
    int out_stride, n_write;   // the first n_write outputs of every listed row are written
};

__device__ __forceinline__ float mlp_hidden_act_exact(float x, int act) {
    if (act == MLP_ACT_SELU) return 1.0507009873554805f * (x > 0.0f ? x : 1.6732632423543772f * (expf(x) - 1.0f));
    return x / (1.0f + expf(-x));
}

__global__ void __launch_bounds__(256) mlp_exact_kernel(MlpExactArgs A) {
    extern __shared__ __align__(16) unsigned char exact_smem[];
    float (*xa)[MLP_MAX_WIDTH] = reinterpret_cast<float (*)[MLP_MAX_WIDTH]>(exact_smem);
    float (*xb)[MLP_MAX_WIDTH] = xa + MLP_EXACT_ROWS;
    __shared__ int row_id[MLP_EXACT_ROWS];
    const int n_rows = A.n_rows ? *A.n_rows : A.n_rows_host;
    const MlpNet& net = A.net;
    const int tid = threadIdx.x;
#pragma unroll 1
    for (int base = blockIdx.x * MLP_EXACT_ROWS; base < n_rows; base += gridDim.x * MLP_EXACT_ROWS) {
        __syncthreads();
        if (tid < MLP_EXACT_ROWS) row_id[tid] = base + tid < n_rows ? (A.rows ? A.rows[base + tid] : base + tid) : -1;
        __syncthreads();
        for (int i = tid; i < MLP_EXACT_ROWS * net.n_in; i += blockDim.x) {
            const int r = i / net.n_in, k = i - r * net.n_in, row = row_id[r];
            float x = 0.0f;
            if (row >= 0) {
                if (k < A.in_w[0]) x = A.in[0][(size_t)row * A.in_stride[0] + k];
                else if (k < A.in_w[0] + A.in_w[1]) x = A.in[1][(size_t)row * A.in_stride[1] + (k - A.in_w[0])];
                else x = A.in[2][(size_t)row * A.in_stride[2] + (k - A.in_w[0] - A.in_w[1])];
            }
            xa[r][k] = x;
        }
        __syncthreads();
        float (*src)[MLP_MAX_WIDTH] = xa;
        float (*dst)[MLP_MAX_WIDTH] = xb;
        int K = net.n_in;
#pragma unroll 1
        for (int l = 0; l < net.n_tc; ++l) {
            const int N = net.dims[l];
            const float* W = net.w32[l];
#pragma unroll 1
            for (int n = tid; n < N; n += blockDim.x) {
                float acc[MLP_EXACT_ROWS];
                const float b = __ldg(net.b[l] + n);
#pragma unroll
                for (int r = 0; r < MLP_EXACT_ROWS; ++r) acc[r] = b;
#pragma unroll 4
                for (int k = 0; k < K; ++k) {
                    const float w = __ldg(W + (size_t)k * N + n);
#pragma unroll
                    for (int r = 0; r < MLP_EXACT_ROWS; ++r) acc[r] = fmaf(src[r][k], w, acc[r]);
                }
#pragma unroll
                for (int r = 0; r < MLP_EXACT_ROWS; ++r) dst[r][n] = mlp_hidden_act_exact(acc[r], net.hidden_act);
            }
            __syncthreads();
            float (*t)[MLP_MAX_WIDTH] = src; src = dst; dst = t;
            K = N;
        }
        for (int idx = tid; idx < MLP_EXACT_ROWS * A.n_write; idx += blockDim.x) {
            const int tid2 = idx;
            const int r = tid2 / A.n_write, o = tid2 - r * A.n_write, row = row_id[r];
            if (row >= 0) {
                float acc = __ldg(net.b_out + o);
                for (int k = 0; k < K; ++k) acc = fmaf(src[r][k], __ldg(net.w_out + (size_t)k * net.out_pad + o), acc);
                A.out[(size_t)row * A.out_stride + o] = net.out_act == MLP_OUT_SIGMOID ? 1.0f / (1.0f + expf(-acc)) : tanhf(acc);
            }
        }
    }
}

// the look-ahead's risk (smenv_set_risk_lookahead): 1 once a sub-step of the env's shadow copy ended its episode for a
// reason other than the trajectory length (risk_ground_truth's labelling rule, safe_motions_base.py:1520-1592)
__global__ void lookahead_latch_kernel(float* risk, const uint8_t* done, const int32_t* term_reason, int n) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env < n && done[env] && term_reason[env] != SM_TERM_TRAJECTORY_LENGTH) risk[env] = 1.0f;
}

// rows whose tensor-core risk lies within `band` of the threshold -> list (re-rated exactly before the gate decides)
__global__ void gate_band_kernel(const float* risk, int n, float threshold, float band, int* list, int* count) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool near = env < n && fabsf(risk[env] - threshold) < band;
    const unsigned m = __ballot_sync(FULL, near);
    if (m) {
        int b0 = 0;
        if (lane == __ffs(m) - 1) b0 = atomicAdd(count, __popc(m));
        b0 = __shfl_sync(FULL, b0, __ffs(m) - 1);
        if (near) list[b0 + __popc(m & ((1u << lane) - 1u))] = env;
    }
}

// the gate decision; risky envs are listed so that their backup action can be computed (exact mode)
__global__ void risk_decide_kernel(const float* actions, float* exec, const float* risk, int nj, int n, float threshold,
                                   uint8_t* risky, int* list, int* count) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool r = env < n && risk[env] >= threshold;
    if (env < n) {
        if (risky) risky[env] = r ? 1 : 0;
        if (exec != actions)
            for (int j = 0; j < nj; ++j) exec[(size_t)env * nj + j] = actions[(size_t)env * nj + j];
    }
    const unsigned m = __ballot_sync(FULL, r);
    if (m) {
        int b0 = 0;
        if (lane == __ffs(m) - 1) b0 = atomicAdd(count, __popc(m));
        b0 = __shfl_sync(FULL, b0, __ffs(m) - 1);
        if (r) list[b0 + __popc(m & ((1u << lane) - 1u))] = env;
    }
}
