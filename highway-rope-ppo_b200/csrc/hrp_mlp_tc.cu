// hrp_mlp_tc.cu -- tcgen05 (5th-gen tensor core) GEMM for the policy/value MLP of ppo/agent.py:12-84.
//
//   C[M,N] (+)= sum_k A(m,k) * B(n,k)      A(m,k) = A[m*sam + k*sak],  B(n,k) = B[n*sbn + k*sbk]
//
// with the same fused epilogue as the SIMT kernel in hrp_ppo.cu (+C, +bias[n], ReLU, ReLU-mask) and the same
// deterministic split-K (gridDim.z partial tiles).  Arbitrary element strides cover every GEMM of the
// forward and backward pass without transposed activation copies: nn.Linear forward (A = activations [B,K], B =
// weight [N,K], both K-contiguous), dX = dY W^T-copy (K-contiguous against the transposed weight copies of
// hrp_ppo.cu), dW = dY^T X (both operands batch-major, i.e. "MN-contiguous").  An N-segmented B operand lets two
// weight matrices that are not adjacent in the flat parameter buffer act as one [N, K] operand.
//
// Structure (one CTA = one 128 x {64, 128} output tile; 8 loader / epilogue warps + 1 MMA warp):
//   * operands are fp32 in HBM and are multiplied as TF32 on the tensor cores (kind::tf32); in the default
//     3xTF32 mode every operand is split into hi = trunc_tf32(x) and lo = x - hi while it is staged, and
//     D += Alo*Bhi + Ahi*Blo + Ahi*Bhi is accumulated in fp32 in TMEM, which recovers fp32-level accuracy
//     (the dropped Alo*Blo term is ~2^-22 relative);
//   * tiles are staged global -> registers (two K-blocks ahead) -> shared memory in the canonical K-major
//     SWIZZLE_128B layout (8-row x 128-byte atoms, 16-byte chunk index XOR row%8); 2 (3xTF32) or 4 (TF32)
//     shared-memory stages, full / empty mbarrier rings, the empty side signalled by tcgen05.commit; the
//     single-pass TF32 mode stages with cp.async instead;
//   * one elected lane of the MMA warp issues the tcgen05.mma instructions (UMMA 128 x BN x 8); the accumulator
//     lives in BN TMEM columns; the epilogue reads it with tcgen05.ld (32 lanes x 16 columns at a time), stages the
//     tile in shared memory and writes 128-bit coalesced rows;
//   * launched with programmatic stream serialisation: the prologue overlaps the previous kernel's tail.
// Where the time goes (phase clocks below, DESIGN.md 3.2): the 3xTF32 main loop is bound by shared-memory
// bandwidth (48 KB of tile writes + 72 KB of UMMA operand reads per K-block), not by tensor-pipe time.
// Plain ld.global staging (no TMA) is deliberate: the weight matrices live at 8-byte-aligned offsets of the
// flat parameter buffer and half of the backward operands are MN-contiguous, neither of which a 128B-swizzled
// tensor map accepts without extra copies.  The matrices are small (<= 4 MB) and L2-resident.
#include "hrp_internal.cuh"

// phase clocks of CTA (0,0,0), thread 0 (+ the MMA warp's lane 0): see hrp_debug_gemm_phases
__device__ long long g_tc_phase[16];
// -- compiled in only by a profiling build (HRP_PHASE_CLOCKS=1 python highway-rope-ppo_b200/build.py --force, for
// tools/gemm_one.py); the production kernel carries no clock reads or global stores for them
#ifdef HRP_PHASE_CLOCKS
#define TC_PHASE(i) do { if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (tid == 0 || tid == TC_THREADS)) g_tc_phase[(i)] = clock64(); } while (0)
#else
#define TC_PHASE(i) do { } while (0)
#endif

namespace {

constexpr int BM = 128, BK = 32;                  // BK * 4 B = 128 B = one swizzle row; BN is 64 or 128
constexpr int TC_THREADS = 256;                    // loader / epilogue threads (8 warps)
constexpr int TC_LAUNCH_THREADS = TC_THREADS + 32;  // + one warp that only issues tcgen05.mma
constexpr int A_TILE_BYTES = BM * BK * 4;         // 16 KB per part of the A tile

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4,
// LBO = 1 (unused for swizzled K-major), SBO = 1024 B (one 8-row atom), version 1 (Blackwell), layout 2
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// cute::UMMA::InstrDescriptor: D = F32 (bits 4-5 = 1), A = B = TF32 (2 at bits 7-9, 10-12), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28
__host__ __device__ constexpr uint32_t make_idesc(int m, int n)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// byte offset of element (row, k) inside a [rows x 32 fp32] K-major SWIZZLE_128B tile
__device__ __forceinline__ uint32_t swz(int r, int k)
{
    return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((((k >> 2) ^ (r & 7)) & 7) << 4) + ((k & 3) << 2));
}

// ---- operand staging: global -> registers (fetch) -> swizzled shared tile(s) (stash) --------------------------
// MODE 0: scalar, K-contiguous (a warp reads one 128-byte row)      1: scalar, MN-contiguous (32 rows at one k)
// MODE 2: 16-byte vectors along K (needs 16 B alignment)           3: 8-byte vectors along K (flat-buffer weights)
// MODE 4: 16-byte vectors along MN (4 rows at one k; batch-major operands of the weight gradient)
// MODE 5: MN-contiguous, lanes along MN and 4 consecutive k per thread: four coalesced scalar loads, then ONE
//         16-byte shared-memory store per part (MODE 4 needs four scalar stores per part for the same data)
enum { ST_K1 = 0, ST_MN1 = 1, ST_K4 = 2, ST_K2 = 3, ST_MN4 = 4, ST_MNK4 = 5 };

template <int MODE, int ROWS>
struct Stager {
    static constexpr int ELEMS = ROWS * BK / TC_THREADS;   // fp32 values per thread and K-block
    float v[ELEMS];

    // scalar element of thread-slot idx.  K-contiguous: a warp covers one 128-byte row (coalesced, and the 32
    // words of a swizzled row hit 32 banks).  MN-contiguous: a warp covers 8 rows x 4 k -- four fully used
    // 32-byte sectors in global memory, and (chunk ^ row%8, k%4) is a bijection onto the 32 banks.
    static __device__ __forceinline__ void coord1(int idx, int &r, int &k)
    {
        if (MODE == ST_K1) { r = idx >> 5; k = idx & 31; }
        else {
            int lane = idx & 31, unit = idx >> 5;
            r = (unit % (ROWS / 8)) * 8 + (lane >> 2);
            k = (unit / (ROWS / 8)) * 4 + (lane & 3);
        }
    }
    // 4-row vector of thread-slot idx (ST_MN4): lane <-> k, so that each of the four scalar shared-memory
    // stores of a warp goes to 32 different banks (k/4 ^ const covers the 8 chunks, k%4 the words)
    static __device__ __forceinline__ void coord_mn4(int idx, int &r, int &k)
    {
        k = idx & 31;
        r = (idx >> 5) * 4;
    }

    // P(row, k) = P[row * srow + k * sk]; rows >= nrows and k >= kend read as zero
    __device__ __forceinline__ void fetch(const float *__restrict__ P, long long srow, long long sk, int row0,
                                          int nrows, int k0, int kend, int tid)
    {
        if (MODE == ST_K1 || MODE == ST_MN1) {
#pragma unroll
            for (int i = 0; i < ELEMS; ++i) {
                int r, k;
                coord1(tid + i * TC_THREADS, r, k);
                int gr = row0 + r, gk = k0 + k;
                v[i] = (gr < nrows && gk < kend) ? __ldg(P + (long long)gr * srow + (long long)gk * sk) : 0.f;
            }
        } else if (MODE == ST_K4) {
#pragma unroll
            for (int i = 0; i < ELEMS / 4; ++i) {
                int idx = tid + i * TC_THREADS;
                int r = idx >> 3, k = (idx & 7) * 4;
                int gr = row0 + r, gk = k0 + k;
                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                if (gr < nrows && gk < kend) t = __ldg(reinterpret_cast<const float4 *>(P + (long long)gr * srow + gk));
                v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
            }
        } else if (MODE == ST_K2) {
#pragma unroll
            for (int i = 0; i < ELEMS / 2; ++i) {
                int idx = tid + i * TC_THREADS;
                int r = idx >> 4, k = (idx & 15) * 2;
                int gr = row0 + r, gk = k0 + k;
                float2 t = make_float2(0.f, 0.f);
                if (gr < nrows && gk < kend) t = __ldg(reinterpret_cast<const float2 *>(P + (long long)gr * srow + gk));
                v[2 * i] = t.x; v[2 * i + 1] = t.y;
            }
        } else if (MODE == ST_MN4) {
#pragma unroll
            for (int i = 0; i < ELEMS / 4; ++i) {
                int r, k;
                coord_mn4(tid + i * TC_THREADS, r, k);
                int gr = row0 + r, gk = k0 + k;
                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                if (gr < nrows && gk < kend) t = __ldg(reinterpret_cast<const float4 *>(P + (long long)gk * sk + gr));
                v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
            }
        } else {  // ST_MNK4: thread-slot idx -> row idx % ROWS, k chunk idx / ROWS
#pragma unroll
            for (int i = 0; i < ELEMS / 4; ++i) {
                const int idx = tid + i * TC_THREADS, r = idx % ROWS, k = (idx / ROWS) * 4;
                const int gr = row0 + r;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int gk = k0 + k + j;
                    v[4 * i + j] = (gr < nrows && gk < kend) ? __ldg(P + (long long)gk * sk + (long long)gr * srow) : 0.f;
                }
            }
        }
    }

    template <int NSPLIT>
    __device__ __forceinline__ void put(uint8_t *hi_tile, int part_bytes, uint32_t o, float x) const
    {
        if (NSPLIT == 3) {
            float hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
            *(float *)(hi_tile + o) = hi;
            *(float *)(hi_tile + part_bytes + o) = x - hi;
        } else {
            *(float *)(hi_tile + o) = x;
        }
    }

    // hi part at hi_tile, lo part (3xTF32) at hi_tile + part_bytes
    template <int NSPLIT>
    __device__ __forceinline__ void stash(uint8_t *hi_tile, int part_bytes, int tid) const
    {
        if (MODE == ST_K1 || MODE == ST_MN1) {
#pragma unroll
            for (int i = 0; i < ELEMS; ++i) {
                int r, k;
                coord1(tid + i * TC_THREADS, r, k);
                put<NSPLIT>(hi_tile, part_bytes, swz(r, k), v[i]);
            }
        } else if (MODE == ST_K4) {
#pragma unroll
            for (int i = 0; i < ELEMS / 4; ++i) {
                int idx = tid + i * TC_THREADS;
                uint32_t o = swz(idx >> 3, (idx & 7) * 4);   // one whole 16-byte chunk
                float4 x = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                if (NSPLIT == 3) {
                    float4 h;
                    h.x = __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                    h.y = __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                    h.z = __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                    h.w = __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                    *(float4 *)(hi_tile + o) = h;
                    *(float4 *)(hi_tile + part_bytes + o) = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
                } else {
                    *(float4 *)(hi_tile + o) = x;
                }
            }
        } else if (MODE == ST_K2) {
#pragma unroll
            for (int i = 0; i < ELEMS / 2; ++i) {
                int idx = tid + i * TC_THREADS;
                uint32_t o = swz(idx >> 4, (idx & 15) * 2);  // half of a 16-byte chunk
                float2 x = make_float2(v[2 * i], v[2 * i + 1]);
                if (NSPLIT == 3) {
                    float2 h;
                    h.x = __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                    h.y = __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                    *(float2 *)(hi_tile + o) = h;
                    *(float2 *)(hi_tile + part_bytes + o) = make_float2(x.x - h.x, x.y - h.y);
                } else {
                    *(float2 *)(hi_tile + o) = x;
                }
            }
        } else if (MODE == ST_MN4) {  // four rows at one k
#pragma unroll
            for (int i = 0; i < ELEMS / 4; ++i) {
                int r, k;
                coord_mn4(tid + i * TC_THREADS, r, k);
#pragma unroll
                for (int j = 0; j < 4; ++j) put<NSPLIT>(hi_tile, part_bytes, swz(r + j, k), v[4 * i + j]);
            }
        } else {  // ST_MNK4: one whole 16-byte chunk of row r; 8 consecutive rows hit 8 different bank groups
#pragma unroll
            for (int i = 0; i < ELEMS / 4; ++i) {
                const int idx = tid + i * TC_THREADS;
                const uint32_t o = swz(idx % ROWS, (idx / ROWS) * 4);
                float4 x = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                if (NSPLIT == 3) {
                    float4 h;
                    h.x = __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                    h.y = __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                    h.z = __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                    h.w = __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                    *(float4 *)(hi_tile + o) = h;
                    *(float4 *)(hi_tile + part_bytes + o) = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
                } else {
                    *(float4 *)(hi_tile + o) = x;
                }
            }
        }
    }
};

template <int NSPLIT, int BN, bool ASYNC>
__host__ __device__ constexpr int tc_stages()
{
    constexpr int stage = (NSPLIT == 3 ? 2 : 1) * (A_TILE_BYTES + BN * BK * 4);
    // register-staged path: <= 96 KB per CTA so that two CTAs share an SM; cp.async path: as deep as 200 KB allow
    return ASYNC ? (4 * stage <= 200 * 1024 ? 4 : 3) : (NSPLIT == 3 ? 2 : 4);
}

// ---- epilogue shared by both main loops: TMEM -> registers -> shared (row-major, padded) -> coalesced global rows
// Optional fused consumer (TcDots, hrp_ppo.cu's act path): the output is [a1 | c1], the hidden activations of the two
// heads, and all the policy needs of it are A + 1 dot products per row -- mean_a = a1 . Wa2[a], value = c1 . Wc2.  A tile
// lies entirely in a1 or in c1 (H % BN == 0, checked by the host); every thread multiplies its four columns of a row
// by the head weights it keeps in registers, the CQ threads of the row add up by shuffles, and the tile leaves NP
// partial sums per row in out[tile][row][NP]; a tiny kernel adds the tiles (heads_finish_kernel, NP = 4 for the
// Gaussian head; heads_finish_cat_kernel, NP = 4 or 8 for the categorical one).  With skip_store the activation itself
// is never written.
template <int BN, bool DUAL, int NP>
__device__ __forceinline__ void tc_epilogue(uint8_t *smem, uint64_t *bar_done_p, uint32_t tmem_d, int nkb, int M, int N,
                                            int m0, int n0, int bn0, float *__restrict__ C, int ldc,
                                            const float *__restrict__ biasp, int relu, const float *__restrict__ mask,
                                            int ldm, int accumulate, float *__restrict__ C_lo, const TcDots &dots)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // ---- epilogue: TMEM -> registers -> shared (row-major, padded) -> coalesced global rows.
    // Warp w reads TMEM lanes 32 (w % 4) .., columns (BN / 2) (w / 4) ..; the operand stages are free by now.
    if (nkb > 0) mbar_wait(bar_done_p, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (tid == 0) TC_PHASE(5);   // accumulator ready
    constexpr int LDS = BN + 4;   // row pitch: 16-byte aligned rows; 128-bit accesses of 8 consecutive rows or chunks hit 32 banks
    float *stage_c = (float *)smem;
    if (warp < TC_THREADS / 32) {
        const int trow = 32 * (warp & 3) + lane;
#pragma unroll 1
        for (int c0 = (BN / 2) * (warp >> 2); c0 < (BN / 2) * (warp >> 2) + BN / 2; c0 += 16) {
            uint32_t v[16];
            if (nkb > 0) {
                uint32_t taddr = tmem_d + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)c0;
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, "
                    "%13, %14, %15}, [%16];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                      "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
                      "=r"(v[15])
                    : "r"(taddr));
                if (DUAL) {   // 3xTF32: columns [BN, 2 BN) hold the A_hi x B_lo part of the same tile
                    uint32_t u[16];
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, "
                        "%13, %14, %15}, [%16];"
                        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
                          "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]),
                          "=r"(u[15])
                        : "r"(taddr + (uint32_t)BN));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
                } else {
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = 0u;
            }
#pragma unroll
            for (int j = 0; j < 16; j += 4)
                *(uint4 *)(stage_c + trow * LDS + c0 + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
    }
    __syncthreads();
    if (tid == 0) TC_PHASE(6);   // tile staged in shared memory
    float *Cz = C + (size_t)blockIdx.z * M * ldc;
    // optional "lo" twin of the output, x - trunc_tf32(x): the pre-split operand of the TMA-fed kernel (hrp_gemm_tma.cu)
    float *Clz = C_lo ? C_lo + (size_t)blockIdx.z * M * ldc : nullptr;
    const bool vec = n0 + BN <= N && ldc % 4 == 0 && ((uintptr_t)Cz & 15) == 0 && (!Clz || ((uintptr_t)Clz & 15) == 0) &&
                     (mask == nullptr || (ldm % 4 == 0 && ((uintptr_t)mask & 15) == 0));
    if (vec && tid < TC_THREADS) {
        // whole tile inside the matrix and 16-byte aligned rows: a warp writes 512 contiguous bytes per instruction.
        // Thread t owns the column quad t % (BN / 4); rows advance by TC_THREADS / (BN / 4), four rows per round trip.
        constexpr int CQ = BN / 4, RSTEP = TC_THREADS / CQ, GROUP = 4;
        const int cq = tid % CQ, gn = n0 + 4 * cq;
        float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (biasp) bv = make_float4(biasp[bn0 + 4 * cq], biasp[bn0 + 4 * cq + 1], biasp[bn0 + 4 * cq + 2], biasp[bn0 + 4 * cq + 3]);
        float *crow = Cz + (size_t)(m0 + tid / CQ) * ldc + gn;
        const float *mrow = mask ? mask + (size_t)(m0 + tid / CQ) * ldm + gn : nullptr;
        const float *srow = stage_c + (tid / CQ) * LDS + 4 * cq;
        float4 hwv[NP];
        if (dots.out) {
            const bool actor = n0 < dots.H;
            const int nd = actor ? dots.A : 1;
#pragma unroll
            for (int a = 0; a < NP; ++a) {
                const float *w = actor ? dots.wa + (size_t)a * dots.H + gn : dots.wc + (gn - dots.H);
                hwv[a] = a < nd ? make_float4(w[0], w[1], w[2], w[3]) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll 1
        for (int rb = tid / CQ; rb < BM; rb += RSTEP * GROUP) {
            float4 prev[GROUP], mk[GROUP];
#pragma unroll
            for (int j = 0; j < GROUP; ++j) {
                const bool ok = m0 + rb + j * RSTEP < M;
                prev[j] = (accumulate && ok) ? *(const float4 *)(crow + (size_t)j * RSTEP * ldc) : make_float4(0.f, 0.f, 0.f, 0.f);
                mk[j] = (mask && ok) ? __ldg((const float4 *)(mrow + (size_t)j * RSTEP * ldm)) : make_float4(1.f, 1.f, 1.f, 1.f);
            }
#pragma unroll
            for (int j = 0; j < GROUP; ++j) {
                float4 x = *(const float4 *)(srow + j * RSTEP * LDS);
                x.x += bv.x + prev[j].x; x.y += bv.y + prev[j].y; x.z += bv.z + prev[j].z; x.w += bv.w + prev[j].w;
                if (relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
                x.x = mk[j].x > 0.f ? x.x : 0.f; x.y = mk[j].y > 0.f ? x.y : 0.f;
                x.z = mk[j].z > 0.f ? x.z : 0.f; x.w = mk[j].w > 0.f ? x.w : 0.f;
                if (dots.out) {
                    float d[NP];
#pragma unroll
                    for (int a = 0; a < NP; ++a) {
                        d[a] = fmaf(x.w, hwv[a].w, fmaf(x.z, hwv[a].z, fmaf(x.y, hwv[a].y, x.x * hwv[a].x)));
#pragma unroll
                        for (int off = CQ / 2; off > 0; off >>= 1) d[a] += __shfl_xor_sync(0xffffffffu, d[a], off);
                    }
                    if (cq == 0 && m0 + rb + j * RSTEP < M) {
                        float *o = dots.out + ((size_t)blockIdx.x * M + (m0 + rb + j * RSTEP)) * NP;
#pragma unroll
                        for (int q = 0; q < NP; q += 4) *(float4 *)(o + q) = make_float4(d[q], d[q + 1], d[q + 2], d[q + 3]);
                    }
                }
                if (m0 + rb + j * RSTEP < M && !dots.skip_store) {
                    *(float4 *)(crow + (size_t)j * RSTEP * ldc) = x;
                    if (Clz) {
                        float4 l;
                        l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                        l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                        l.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                        l.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                        *(float4 *)(Clz + (crow - Cz) + (size_t)j * RSTEP * ldc) = l;
                    }
                }
            }
            crow += (size_t)RSTEP * GROUP * ldc;
            if (mask) mrow += (size_t)RSTEP * GROUP * ldm;
            srow += RSTEP * GROUP * LDS;
        }
    } else if (!vec) {
        // ragged or unaligned tile: thread t writes column t % BN, rows advance by TC_THREADS / BN, eight rows per
        // memory round trip
        constexpr int RSTEP = TC_THREADS / BN, GROUP = 8;
        const int c = tid % BN, gn = n0 + c;
        const float bv = (biasp && gn < N) ? biasp[bn0 + c] : 0.f;
        if (gn < N && tid < TC_THREADS) {
#pragma unroll 1
            for (int rb = tid / BN; rb < BM; rb += RSTEP * GROUP) {
                float prev[GROUP], mk[GROUP];
#pragma unroll
                for (int j = 0; j < GROUP; ++j) {
                    const int gm = m0 + rb + j * RSTEP;
                    const bool ok = gm < M;
                    prev[j] = (accumulate && ok) ? Cz[(size_t)gm * ldc + gn] : 0.f;
                    mk[j] = (mask && ok) ? __ldg(mask + (size_t)gm * ldm + gn) : 1.f;
                }
#pragma unroll
                for (int j = 0; j < GROUP; ++j) {
                    const int r = rb + j * RSTEP, gm = m0 + r;
                    float x = stage_c[r * LDS + c] + bv + prev[j];
                    if (relu) x = fmaxf(x, 0.f);
                    x = mk[j] > 0.f ? x : 0.f;
                    if (gm < M) {
                        Cz[(size_t)gm * ldc + gn] = x;
                        if (Clz) Clz[(size_t)gm * ldc + gn] = x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
                    }
                }
            }
        }
    }
    if (tid == 0) TC_PHASE(7);   // tile written
}

template <int AMODE, int BMODE, int NSPLIT, int BN, bool ASYNC, int NP>
__global__ void __launch_bounds__(TC_LAUNCH_THREADS)
tc_gemm_kernel(int M, int N, int K, const float *__restrict__ A, long long sam, long long sak,
               const float *__restrict__ B, long long sbn, long long sbk, float *__restrict__ C, int ldc,
               const float *__restrict__ bias, int relu, const float *__restrict__ mask, int ldm, int accumulate,
               int k_chunk, int nseg, const float *__restrict__ B2, const float *__restrict__ bias2, float *__restrict__ C_lo,
               const TcDots dots)
{
    constexpr int PARTS = NSPLIT == 3 ? 2 : 1;                  // hi (+ lo) copy of every operand tile
    constexpr int B_TILE_BYTES = BN * BK * 4;
    constexpr int STAGE_BYTES = PARTS * (A_TILE_BYTES + B_TILE_BYTES);
    constexpr int STAGES = tc_stages<NSPLIT, BN, ASYNC>();
    // 3xTF32 accumulates in 2 BN columns: [0, BN) <- A_hi B_hi + A_lo B_hi, [BN, 2 BN) <- A_hi B_lo (summed in the
    // epilogue).  The hi and lo tiles of B are adjacent in a stage, so ONE UMMA with N = 2 BN multiplies A_hi by both:
    // two instructions per k-step instead of three (the UMMA stream paces the main loop, ~88 cycles per instruction)
    constexpr int TM_COLS = NSPLIT == 3 ? 2 * BN : BN;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ uint64_t bar_full[4], bar_empty[4], bar_done;
    __shared__ uint32_t tmem_base_s;
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    hrp_pdl_release();   // the next kernel of the stream may set itself up while this one runs
    if (tid == 0) TC_PHASE(0);
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    // N-segmented B operand: output columns >= nseg multiply the rows of a second matrix (two weight matrices that
    // are not adjacent in memory act as one [N, K] operand; tiles never straddle the boundary, see hrp_tc_gemm)
    const bool seg2 = nseg > 0 && n0 >= nseg;
    const float *__restrict__ Bp = seg2 ? B2 : B;
    const float *__restrict__ biasp = seg2 ? bias2 : bias;
    const int bn0 = seg2 ? n0 - nseg : n0;                       // first row of this tile inside Bp
    const int bN = nseg > 0 ? (seg2 ? N - nseg : nseg) : N;      // rows of Bp
    const int kbeg = blockIdx.z * k_chunk, kend = min(K, kbeg + k_chunk);
    const int nkb = (kend - kbeg + BK - 1) / BK;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&bar_full[s], TC_THREADS);   // every loader thread arrives once its part of the stage is written
            mbar_init(&bar_empty[s], 1);           // tcgen05.commit arrives when the MMAs have read the stage
        }
        mbar_init(&bar_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                     "n"(TM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = tmem_base_s;
    constexpr uint32_t idesc = make_idesc(BM, BN);
    constexpr uint32_t idesc2 = make_idesc(BM, 2 * BN);   // A_hi against the stacked [B_hi ; B_lo] tile
    hrp_pdl_wait();      // everything above overlapped the previous kernel's tail; its results are visible from here
    if (tid == 0) TC_PHASE(1);

    if (ASYNC && warp < TC_THREADS / 32) {
        // ===== loader warps, cp.async path (A: 16-byte, B: 8-byte aligned K-contiguous operands).
        // The tensor core TRUNCATES fp32 operands to TF32 (tools/tf32_probe.py), so the raw fp32 tile is the
        // "hi" operand as it is: raw tiles go global -> shared with cp.async, STAGES - 1 K-blocks in flight, no
        // registers involved; each thread then derives the "lo" tile (x - trunc(x)) from the chunks it copied.
        constexpr int P = STAGES - 1;
        constexpr int B_CHUNKS = BN * BK / 2 / TC_THREADS;     // 8-byte chunks of B per thread
        auto issue = [&](int kb) {
            const int s = kb % STAGES, k0 = kbeg + kb * BK;
            const uint32_t a_raw = smem_u32(smem + s * STAGE_BYTES), b_raw = a_raw + PARTS * A_TILE_BYTES;
#pragma unroll
            for (int i = 0; i < BM * BK / 4 / TC_THREADS; ++i) {
                const int idx = tid + i * TC_THREADS, r = idx >> 3, k = (idx & 7) * 4;
                const int gr = m0 + r, gk = k0 + k;
                const bool ok = gr < M && gk < kend;
                const float *src = ok ? A + (long long)gr * sam + gk : A;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(a_raw + swz(r, k)), "l"(src),
                             "r"(ok ? 16 : 0)
                             : "memory");
            }
#pragma unroll
            for (int i = 0; i < B_CHUNKS; ++i) {
                const int idx = tid + i * TC_THREADS, r = idx >> 4, k = (idx & 15) * 2;
                const int gr = bn0 + r, gk = k0 + k;
                const bool ok = gr < bN && gk < kend;
                const float *src = ok ? Bp + (long long)gr * sbn + gk : Bp;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(b_raw + swz(r, k)), "l"(src),
                             "r"(ok ? 8 : 0)
                             : "memory");
            }
        };
        for (int kb = 0; kb < P; ++kb) {
            if (kb < nkb) issue(kb);
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            asm volatile("cp.async.wait_group %0;" ::"n"(P - 1) : "memory");   // this thread's chunks of block kb landed
            if (NSPLIT == 3) {
                uint8_t *a_raw = smem + s * STAGE_BYTES, *b_raw = a_raw + PARTS * A_TILE_BYTES;
#pragma unroll
                for (int i = 0; i < BM * BK / 4 / TC_THREADS; ++i) {
                    const int idx = tid + i * TC_THREADS;
                    const uint32_t o = swz(idx >> 3, (idx & 7) * 4);
                    const float4 x = *(const float4 *)(a_raw + o);
                    float4 l;
                    l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                    l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                    l.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                    l.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                    *(float4 *)(a_raw + A_TILE_BYTES + o) = l;
                }
#pragma unroll
                for (int i = 0; i < B_CHUNKS; ++i) {
                    const int idx = tid + i * TC_THREADS;
                    const uint32_t o = swz(idx >> 4, (idx & 15) * 2);
                    const float2 x = *(const float2 *)(b_raw + o);
                    float2 l;
                    l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                    l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                    *(float2 *)(b_raw + B_TILE_BYTES + o) = l;
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bar_full[s])) : "memory");
            const int nx = kb + P;                           // refill the stage that block kb - 1 used
            if (nx < nkb) {
                if (nx >= STAGES) mbar_wait(&bar_empty[nx % STAGES], (uint32_t)(((nx / STAGES) - 1) & 1));
                issue(nx);
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
    } else if (warp < TC_THREADS / 32) {
        // ===== loader warps: global -> registers (PF K-blocks ahead) -> swizzled shared stage -> bar_full.
        // Measured (tools/gemm_one.py phase clocks, 4096 x 256 x 256): a K-block takes ~920 cycles with PF = 2 and
        // with PF = 4 alike -- the 3xTF32 main loop is bound by shared-memory bandwidth (48 KB of tile writes plus
        // 72 KB of operand reads by the 12 UMMAs per K-block at 128 B/cycle), not by the L2 round trip.
        constexpr int PF = 2;
        Stager<AMODE, BM> sa0, sa1, sa2, sa3;   // named, not an array: the register sets must never be indexed dynamically
        Stager<BMODE, BN> sb0, sb1, sb2, sb3;
        auto step = [&](int kb, Stager<AMODE, BM> &ra, Stager<BMODE, BN> &rb) {
            const int s = kb % STAGES;
            if (kb == 4 && tid == 0) TC_PHASE(10);
            if (kb >= STAGES) mbar_wait(&bar_empty[s], (uint32_t)(((kb / STAGES) - 1) & 1));  // MMAs of kb - STAGES retired
            if (kb == 4 && tid == 0) TC_PHASE(11);
            uint8_t *a_hi = smem + s * STAGE_BYTES, *b_hi = a_hi + PARTS * A_TILE_BYTES;
            ra.template stash<NSPLIT>(a_hi, A_TILE_BYTES, tid);
            rb.template stash<NSPLIT>(b_hi, B_TILE_BYTES, tid);
            if (kb == 4 && tid == 0) TC_PHASE(12);
            if (kb + PF < nkb) {                            // refill this register set: in flight for PF blocks
                const int k0 = kbeg + (kb + PF) * BK;
                ra.fetch(A, sam, sak, m0, M, k0, kend, tid);
                rb.fetch(Bp, sbn, sbk, bn0, bN, k0, kend, tid);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bar_full[s])) : "memory");
            if (kb == 4 && tid == 0) TC_PHASE(13);
        };
#define HRP_TC_PREFETCH(j, ra, rb)                                               \
        if (j < nkb) {                                                              \
            ra.fetch(A, sam, sak, m0, M, kbeg + j * BK, kend, tid);                 \
            rb.fetch(Bp, sbn, sbk, bn0, bN, kbeg + j * BK, kend, tid);              \
        }
        HRP_TC_PREFETCH(0, sa0, sb0)
        HRP_TC_PREFETCH(1, sa1, sb1)
        if (PF > 2) { HRP_TC_PREFETCH(2, sa2, sb2) }
        if (PF > 3) { HRP_TC_PREFETCH(3, sa3, sb3) }
#undef HRP_TC_PREFETCH
        if (tid == 0) TC_PHASE(2);   // first loads issued
        for (int kb = 0; kb < nkb; kb += PF) {
            step(kb, sa0, sb0);
            if (kb + 1 < nkb) step(kb + 1, sa1, sb1);
            if (PF > 2 && kb + 2 < nkb) step(kb + 2, sa2, sb2);
            if (PF > 3 && kb + 3 < nkb) step(kb + 3, sa3, sb3);
            if (kb == 0 && tid == 0) TC_PHASE(3);
        }
        if (tid == 0) TC_PHASE(4);   // loaders done
    } else {
        // ===== MMA warp: waits for a full stage, one elected lane issues the UMMAs, tcgen05.commit frees the stage
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            mbar_wait(&bar_full[s], (uint32_t)((kb / STAGES) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (kb == 4) TC_PHASE(14);
            if (lane == 0) {
                const uint32_t a_s = smem_u32(smem + s * STAGE_BYTES), b_s = a_s + PARTS * A_TILE_BYTES;
                // descriptors differ only in the start-address field (bits 0-13, units of 16 bytes)
                const uint64_t da_hi = make_desc(a_s), db_hi = make_desc(b_s);
                const uint64_t da_lo = da_hi + (A_TILE_BYTES >> 4);   // B_lo follows B_hi: rows BN .. 2 BN - 1 of the stacked tile
#pragma unroll
                for (int kk = 0; kk < BK / 8; ++kk) {       // UMMA_K = 8 tf32 = 32 bytes = 2 address units
                    const uint64_t o = (uint64_t)(kk * 2);
                    const uint32_t acc = (kb > 0 || kk > 0) ? 1u : 0u;
                    if (NSPLIT == 3) {
                        umma_tf32(tmem_d, da_hi + o, db_hi + o, idesc2, acc);   // [A_hi B_hi | A_hi B_lo]
                        umma_tf32(tmem_d, da_lo + o, db_hi + o, idesc, 1u);     // + A_lo B_hi into the first half
                    } else {
                        umma_tf32(tmem_d, da_hi + o, db_hi + o, idesc, acc);
                    }
                }
                umma_commit(&bar_empty[s]);
                if (kb + 1 == nkb) umma_commit(&bar_done);  // accumulator complete
                if (kb == 4) TC_PHASE(15);
                if (kb == 0) TC_PHASE(8);
                if (kb + 1 == nkb) TC_PHASE(9);
            }
            __syncwarp();
        }
    }

    tc_epilogue<BN, NSPLIT == 3, NP>(smem, &bar_done, tmem_d, nkb, M, N, m0, n0, bn0, C, ldc, biasp, relu, mask, ldm, accumulate, C_lo, dots);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(TM_COLS) : "memory");
}

// Two variants that kept the A operand in tensor memory (tcgen05.st of the hi / lo halves, TS-form
// `tcgen05.mma [d], [a], b_desc`) were built and are parity-green in the history of this file: one with row-per-
// thread global loads (1030 vs 920 cycles per K-block, twice as slow for batch-major A) and one that kept the
// coalesced loads and passed the raw tile through a shared-memory transposition buffer (7.97k vs 7.29k main-loop
// cycles at 4096 x 256 x 256).  Neither beat the SS path: the per-K-block phase clocks (slots 10-15 of
// hrp_debug_gemm_phases) show that the MMA warp needs ~1050 cycles to push the 12 UMMAs of a K-block through the
// tensor pipe (~88 cycles per 128 x 64 x 8 instruction) while a stash takes ~580 and the stage hand-over ~430, i.e.
// the main loop is paced by the UMMA stream itself, whichever memory the A operand comes from.

// NP: partial sums per row of the fused row-dot epilogue (TcDots): 4, or 8 for a categorical head of more than four logits
template <int AMODE, int BMODE, int NSPLIT, int BN, bool ASYNC = false, int NP = 4>
int launch(dim3 grid, cudaStream_t s, int M, int N, int K, const float *A, long long sam, long long sak,
           const float *B, long long sbn, long long sbk, float *C, int ldc, const float *bias, int relu,
           const float *mask, int ldm, int accumulate, int k_chunk, int nseg, const float *B2, const float *bias2, float *C_lo,
           const TcDots &dots)
{
    constexpr int PARTS = NSPLIT == 3 ? 2 : 1;
    constexpr int STAGES = tc_stages<NSPLIT, BN, ASYNC>();
    constexpr int OPERANDS = STAGES * PARTS * (A_TILE_BYTES + BN * BK * 4);
    constexpr int EPILOGUE = BM * (BN + 4) * 4;
    constexpr int SMEM = (OPERANDS > EPILOGUE ? OPERANDS : EPILOGUE) + 1024;
    // the attribute is per device (a process may drive several GPUs)
    static bool configured[HRP_MAX_DEVICES] = {false};
    auto kern = tc_gemm_kernel<AMODE, BMODE, NSPLIT, BN, ASYNC, NP>;
    int dev = 0;
    HRP_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= HRP_MAX_DEVICES) { hrp_set_error("device index %d not supported", dev); return -1; }
    if (!configured[dev]) {
        HRP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        configured[dev] = true;
    }
    HRP_CUDA_OK(hrp_launch_pdl(kern, grid, dim3(TC_LAUNCH_THREADS), (size_t)SMEM, s, M, N, K, A, sam, sak, B, sbn, sbk, C, ldc,
                               bias, relu, mask, ldm, accumulate, k_chunk, nseg, B2, bias2, C_lo, dots));
    return 0;
}

template <int AMODE, int BMODE, int NP = 4>
int dispatch(int bn, int nsplit, dim3 grid, cudaStream_t s, int M, int N, int K, const float *A, long long sam,
             long long sak, const float *B, long long sbn, long long sbk, float *C, int ldc, const float *bias,
             int relu, const float *mask, int ldm, int accumulate, int k_chunk, int nseg, const float *B2,
             const float *bias2, float *C_lo, const TcDots &dots)
{
#define HRP_TC_ARGS grid, s, M, N, K, A, sam, sak, B, sbn, sbk, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk, nseg, B2, bias2, C_lo, dots
    if constexpr (NP == 4)   // (never with the fused epilogue, the only user of NP = 8)
        if (bn == 32 && nsplit == 3) return launch<AMODE, BMODE, 3, 32>(HRP_TC_ARGS);
    if (bn <= 64)
        return nsplit == 3 ? launch<AMODE, BMODE, 3, 64, false, NP>(HRP_TC_ARGS) : launch<AMODE, BMODE, 1, 64, false, NP>(HRP_TC_ARGS);
    return nsplit == 3 ? launch<AMODE, BMODE, 3, 128, false, NP>(HRP_TC_ARGS) : launch<AMODE, BMODE, 1, 128, false, NP>(HRP_TC_ARGS);
#undef HRP_TC_ARGS
}

// forward-pass operands (activations x weights, both K-contiguous and aligned): cp.async staging
template <int NP = 4>
int dispatch_async(int bn, int nsplit, dim3 grid, cudaStream_t s, int M, int N, int K, const float *A, long long sam,
                   long long sak, const float *B, long long sbn, long long sbk, float *C, int ldc, const float *bias,
                   int relu, const float *mask, int ldm, int accumulate, int k_chunk, int nseg, const float *B2,
                   const float *bias2, float *C_lo, const TcDots &dots)
{
#define HRP_TC_ARGS grid, s, M, N, K, A, sam, sak, B, sbn, sbk, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk, nseg, B2, bias2, C_lo, dots
    if (bn == 64)
        return nsplit == 3 ? launch<ST_K4, ST_K2, 3, 64, true, NP>(HRP_TC_ARGS) : launch<ST_K4, ST_K2, 1, 64, true, NP>(HRP_TC_ARGS);
    return nsplit == 3 ? launch<ST_K4, ST_K2, 3, 128, true, NP>(HRP_TC_ARGS) : launch<ST_K4, ST_K2, 1, 128, true, NP>(HRP_TC_ARGS);
#undef HRP_TC_ARGS
}

inline bool aligned(const void *p, int bytes) { return ((uintptr_t)p % bytes) == 0; }

}  // namespace

// the N-tile width hrp_tc_gemm picks (the fused row-dot epilogue's caller sizes its partial buffer with it)
int hrp_tc_gemm_bn(int M, int N, int splits, int nseg, int narrow)
{
    const int mt = (M + BM - 1) / BM, sp = splits > 1 ? splits : 1;
    int bn = (N <= 64 || mt * ((N + 127) / 128) * sp < 120) ? 64 : 128;
    if (nseg > 0 && nseg % 128 != 0) bn = 64;
    (void)narrow;   // (64-wide instead of 128-wide tiles for the 2 H-wide head GEMM were measured slower: 40.6 against 38.2 us)
    return bn;
}

// Strided tcgen05 GEMM; returns the number of K splits actually used (partials at C + z*M*ldc), <0 on error.
// nsplit: 3 = 3xTF32 (fp32-grade accuracy), 1 = single TF32 pass.
int hrp_tc_gemm(int M, int N, int K, const float *A, long long sam, long long sak, const float *B, long long sbn,
                long long sbk, float *C, int ldc, const float *bias, int relu, const float *mask, int ldm,
                int accumulate, int splits, int nsplit, cudaStream_t s, int nseg, const float *B2, const float *bias2,
                float *C_lo, const TcDots *dots_in, int narrow)
{
    const TcDots dots = dots_in ? *dots_in : TcDots{nullptr, nullptr, 0, 0, nullptr, 0};
    int k_chunk = K;
    if (splits > 1) {
        k_chunk = ((K + splits - 1) / splits + BK - 1) / BK * BK;
        splits = (K + k_chunk - 1) / k_chunk;
    } else {
        splits = 1;
    }
    // 64-wide N tiles when 128-wide ones would leave most of the 148 SMs idle
    const int mt = (M + BM - 1) / BM;
    if (nseg > 0 && (nseg % 64 != 0 || nseg >= N || B2 == nullptr)) { hrp_set_error("hrp_tc_gemm: bad N segmentation"); return -1; }
    int bn = hrp_tc_gemm_bn(M, N, splits, nseg, narrow);   // (a tile never straddles the two B matrices of a segmented operand)
    // `narrow` (the forward chains, where nothing else runs beside the GEMM): 32-wide N tiles when 64-wide ones leave at
    // most one CTA per SM -- two CTAs (80 KB of stages each) then share an SM and the prologue / epilogue of one overlaps
    // the main loop of the other: policy forward 43.3 -> 38.2 us.  Not for the backward pass, whose GEMMs already share
    // the machine with the weight-gradient GEMMs of the side streams (optimizer step 127 -> 141 us with it).
    // HRP_BN32=0 switches it off.
    static const bool bn32 = !(getenv("HRP_BN32") && getenv("HRP_BN32")[0] == '0');
    if (narrow && bn32 && bn == 64 && nsplit == 3 && N % 32 == 0 && N >= 64 && mt * ((N + 63) / 64) * splits <= 148 && !dots.out)
        bn = 32;
    dim3 grid((N + bn - 1) / bn, mt, splits);
    if (dots.out && (splits != 1 || dots.H % bn != 0 || N % bn != 0 || ldc % 4 != 0 || !aligned(C, 16) || mask || C_lo ||
                     dots.A < 1 || dots.A > 8)) {
        hrp_set_error("hrp_tc_gemm: the fused row-dot epilogue needs whole, aligned tiles that do not straddle H, and 1..8 "
                      "head rows");
        return -1;
    }
    const bool akc = sak == 1, bkc = sbk == 1;
    // vectorised staging where strides and base addresses allow it
    const bool a_k4 = akc && K % 4 == 0 && sam % 4 == 0 && aligned(A, 16);
    const bool b_k2 = bkc && K % 2 == 0 && sbn % 2 == 0 && aligned(B, 8) && (nseg == 0 || aligned(B2, 8));
    const bool b_k4 = bkc && K % 4 == 0 && sbn % 4 == 0 && aligned(B, 16) && (nseg == 0 || aligned(B2, 16));
#define HRP_TC_GO(am, bm) dispatch<am, bm>(bn, nsplit, grid, s, M, N, K, A, sam, sak, B, sbn, sbk, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk, nseg, B2, bias2, C_lo, dots)
    int rc;
    if (dots.out && dots.A > 4) {
        // a categorical head of more than four logits: eight partial sums per row.  Only the operand layouts of the act
        // path are instantiated (K-contiguous activations and weights), chosen by the rule below; the alignment of
        // critic.0 in the flat buffer follows n (offset = n mod 4 floats past a 16-byte boundary)
#define HRP_TC_GO8(am, bm) dispatch<am, bm, 8>(bn, nsplit, grid, s, M, N, K, A, sam, sak, B, sbn, sbk, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk, nseg, B2, bias2, C_lo, dots)
        if (a_k4 && b_k2 && nsplit == 1)
            rc = dispatch_async<8>(bn, nsplit, grid, s, M, N, K, A, sam, sak, B, sbn, sbk, C, ldc, bias, relu, mask, ldm, accumulate,
                                   k_chunk, nseg, B2, bias2, C_lo, dots);
        else if (a_k4 && b_k4) rc = HRP_TC_GO8(ST_K4, ST_K4);
        else if (a_k4 && b_k2) rc = HRP_TC_GO8(ST_K4, ST_K2);
        else if (akc && bkc) rc = HRP_TC_GO8(ST_K1, ST_K1);
        else {
            hrp_set_error("hrp_tc_gemm: the eight-wide fused row-dot epilogue needs K-contiguous operands");
            return -1;
        }
#undef HRP_TC_GO8
        return rc < 0 ? rc : splits;
    }
    // cp.async staging pays off for the single-pass mode only (measured: 3xTF32 hidden forward 12.6 us register-staged
    // vs 14.5 us cp.async -- the lo tiles need a second pass through shared memory; TF32 H=512 19.6 -> 16.6 us)
    if (a_k4 && b_k2 && nsplit == 1) rc = dispatch_async(bn, nsplit, grid, s, M, N, K, A, sam, sak, B, sbn, sbk, C, ldc, bias, relu, mask, ldm, accumulate, k_chunk, nseg, B2, bias2, C_lo, dots);
    else if (a_k4 && b_k4) rc = HRP_TC_GO(ST_K4, ST_K4);
    else if (a_k4 && b_k2) rc = HRP_TC_GO(ST_K4, ST_K2);
    else if (a_k4 && sbn == 1) rc = HRP_TC_GO(ST_K4, ST_MN1);
    else if (sam == 1 && sbn == 1 && nseg == 0) rc = HRP_TC_GO(ST_MNK4, ST_MNK4);
    else if (akc && bkc) rc = HRP_TC_GO(ST_K1, ST_K1);
    else if (akc) rc = HRP_TC_GO(ST_K1, ST_MN1);
    else if (bkc) rc = HRP_TC_GO(ST_MN1, ST_K1);
    else rc = HRP_TC_GO(ST_MN1, ST_MN1);
#undef HRP_TC_GO
    return rc < 0 ? rc : splits;
}

// debugging aid (not part of include/hrp.h): SM clock at the phase boundaries of the last GEMM's first CTA
extern "C" int hrp_debug_gemm_phases(long long *out16)
{
    HRP_CUDA_OK(cudaDeviceSynchronize());
    HRP_CUDA_OK(cudaMemcpyFromSymbol(out16, g_tc_phase, sizeof(long long) * 16));
    return 0;
}
