// Kernel (a): query x reference distance stage (replaces apples/distance.py:718-745 jc69 and :681-715 scoredist
// as called from apples/Reference.py:138-152).
//
// Nucleotide: sequences are three bit-planes (lo, hi, valid) of 32-site words.  For a (query, reference) pair
//   valid    = popc(qv & rv)                                    distance.py:733-734
//   mismatch = popc(((qlo ^ rlo) | (qhi ^ rhi)) & qv & rv)      distance.py:737
// The dense kernel gets both from two cheaper counts.  With the code bits cleared at invalid sites (done when the
// operands are laid out), x = qv ^ rv marks the sites where exactly one side is valid, and
// z = (qlo ^ rlo) | (qhi ^ rhi) | x marks those plus the mismatching valid sites, so
//   E1 = popc(x),  D = popc(z):   mismatch = D - E1,   valid = (nq + nr - E1) / 2
// (nq, nr = valid sites of the two rows, counted once per row): 3 LOP3 per 32 sites instead of 4.
// The dense kernel computes all pairs of a query block against all representatives with a GEMM-like tiling:
// operands are stored tile-major ([row tile][32-word chunk][plane][word][row in tile]) so that one pipeline stage of a
// tile is one contiguous block; thread 0 keeps a 2-stage shared-memory ring full with 1-D TMA bulk copies
// (cp.async.bulk + mbarrier complete_tx, two copies per stage), 16 warps hold a 4x4 register tile of pairs per thread
// (CTA tile 128 queries x 64 representatives, one persistent CTA per SM, 128 registers per thread) and do the
// LOP3/POPC work.  The binding resources are the integer pipes (ALU LOP3, XU POPC), not HBM (DESIGN.md, "rooflines").
#include "common.cuh"
#include <type_traits>

// ---------------------------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + 1-D bulk async copy (TMA)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
#ifdef DT_PRODUCER_SLEEP
        __nanosleep(DT_PRODUCER_SLEEP);
#endif
    }
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// which of a thread's 16 pairs also carry-save their mismatch words (DT_MCSA pairs, spread over the 4x4 block)
#ifndef DT_MCSA
#define DT_MCSA 13  // measured optimum on B200 (profiles/dense_variants_r01.txt)
#endif
__host__ __device__ constexpr int mcsa_slot(int i, int j) { return ((i * 4 + ((j + i) & 3)) * DT_MCSA) / 16; }
__host__ __device__ constexpr bool mcsa_pair(int i, int j) {
    const int p = i * 4 + ((j + i) & 3);
    return DT_MCSA > 0 && (p == 0 ? true : (p * DT_MCSA) / 16 != ((p - 1) * DT_MCSA) / 16);
}

// three-input logic op with an explicit truth table (a = 0xf0, b = 0xcc, c = 0xaa)
template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(d) : "r"(a), "r"(b), "r"(c), "n"(LUT));
    return d;
}

// ---------------------------------------------------------------------------------------------------------------
// row-major [rows][3][W]  ->  tile-major [rows_pad / T][Wp / WC][3][WC][T]   (padding must be pre-zeroed by the caller)
// One pipeline stage of a tile -- 3 planes x WC words x T rows -- is one contiguous block: a single bulk copy.
// ---------------------------------------------------------------------------------------------------------------
__global__ void transpose_nuc_kernel(const uint32_t* __restrict__ rm, int rows, int W, uint32_t* __restrict__ wm, int Wp,
                                     int rows_pad, int T) {
    __shared__ uint32_t tile[32][33];
    const int plane = blockIdx.z;
    const int r0 = blockIdx.y * 32, w0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int r = r0 + i, w = w0 + threadIdx.x;
        uint32_t x = 0u;
        if (r < rows && w < W) {
            x = rm[((size_t)r * 3 + plane) * W + w];
            if (plane < 2) x &= rm[((size_t)r * 3 + 2) * W + w];  // code bits are zero where the site is invalid
        }
        tile[i][threadIdx.x] = x;
    }
    __syncthreads();
    const int n_chunks = Wp / DT_WC;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int w = w0 + i, r = r0 + threadIdx.x;
        if (w < Wp && r < rows_pad) {
            const size_t blk = (size_t)(r / T) * n_chunks + w / DT_WC;
            wm[((blk * 3 + plane) * DT_WC + w % DT_WC) * T + r % T] = tile[threadIdx.x][i];
        }
    }
}

void launch_transpose_nuc(const uint32_t* rm, int rows, int W, uint32_t* wm, int Wp, int rows_pad, int tile_rows,
                          cudaStream_t s) {
    dim3 grid((Wp + 31) / 32, (rows_pad + 31) / 32, 3), block(32, 8);
    transpose_nuc_kernel<<<grid, block, 0, s>>>(rm, rows, W, wm, Wp, rows_pad, tile_rows);
}

// valid sites per row (one warp per row); rows >= `rows` (padding) get 0
__global__ void row_valid_kernel(const uint32_t* __restrict__ rm, int rows, int W, uint32_t* __restrict__ nv, int rows_pad) {
    const int r = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32, lane = threadIdx.x % 32;
    if (r >= rows_pad) return;
    uint32_t c = 0;
    if (r < rows)
        for (int w = lane; w < W; w += 32) c += __popc(rm[((size_t)r * 3 + 2) * W + w]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) nv[r] = c;
}

void launch_row_valid(const uint32_t* rm, int rows, int W, uint32_t* nv, int rows_pad, cudaStream_t s) {
    row_valid_kernel<<<(rows_pad + 7) / 8, 256, 0, s>>>(rm, rows, W, nv, rows_pad);
}

// ---------------------------------------------------------------------------------------------------------------
// dense nucleotide kernel
// ---------------------------------------------------------------------------------------------------------------
struct DenseNucArgs {
    const uint32_t* q_wm;  // [q_pad / TQ][Wp / WC][3][WC][TQ]
    const uint32_t* r_wm;  // [r_pad / TR][Wp / WC][3][WC][TR]
    const uint32_t* q_nv;  // [q_pad] valid sites per query row
    const uint32_t* r_nv;  // [r_pad]
    int q_pad, r_pad, W, Wp;  // W words hold sites, Wp = W rounded up to whole pipeline stages (zero words)
    // keys epilogue
    uint32_t* keys;
    int64_t ldk;
    uint32_t k_one, k_two17;  // 1 and 1 << 17 (see the consumer loop)
    unsigned long long* clk;  // optional: {clock64, globaltimer} of CTA 0 at start and end -> effective SM clock
    // full epilogue (parity export)
    int nq, n_ref, vmin;
    uint32_t* mism;
    uint32_t* valid;
    double* dist;
};

template <bool FULL>
__global__ void __launch_bounds__(DT_THREADS, DT_MINBLOCKS) dense_nuc_kernel(const DenseNucArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint32_t* stage_base = reinterpret_cast<uint32_t*>(smem_raw);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_raw + DT_STAGES * DT_STAGE_BYTES);
    uint64_t* empty_bar = full_bar + DT_STAGES;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int n_rt = a.r_pad / DT_TR;
    const int n_tiles = (a.q_pad / DT_TQ) * n_rt;
    const int n_chunks = a.Wp / DT_WC;

    if (tid == 0 && blockIdx.x == 0 && a.clk) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        a.clk[0] = (unsigned long long)clock64();
        a.clk[1] = t;
    }
    if (tid == 0) {
        for (int s = 0; s < DT_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], DT_CONSUMERS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // one pipeline stage of a tile is contiguous in global memory (tile-major layout): two bulk copies per stage,
    // issued by one thread
    auto issue_stage = [&](uint32_t git, int tile, int c) {
        const int s = git % DT_STAGES;
        const int qt = tile / n_rt, rt = tile % n_rt;
        mbar_arrive_expect_tx(&full_bar[s], DT_STAGE_BYTES);
        uint32_t* sq = stage_base + (size_t)s * DT_STAGE_WORDS;
        uint32_t* sr = sq + 3 * DT_WC * DT_TQ;
        tma_bulk_g2s(sq, a.q_wm + ((size_t)qt * n_chunks + c) * (3 * DT_WC * DT_TQ), 3 * DT_WC * DT_TQ * 4, &full_bar[s]);
        tma_bulk_g2s(sr, a.r_wm + ((size_t)rt * n_chunks + c) * (3 * DT_WC * DT_TR), 3 * DT_WC * DT_TR * 4, &full_bar[s]);
    };
#if DT_SELF_PRODUCE
    // No producer warp (a 17th warp would cap the kernel at 96 registers per thread: 5 warps on one scheduler).  Thread
    // 0 keeps the ring full: before computing chunk `it` it issues every chunk < it + STAGES whose stage has been
    // released (non-blocking test), and blocks only if chunk `it` itself has not been issued yet.
    uint32_t p_it = 0;
    int p_c = 0;
    int p_tile = blockIdx.x;
    auto produce = [&](uint32_t it_now) {
        while (p_tile < n_tiles && p_it < it_now + DT_STAGES) {
            const int ps = p_it % DT_STAGES;
            const uint32_t pph = ((p_it / DT_STAGES) & 1) ^ 1;
            if (p_it == it_now) {
                mbar_wait(&empty_bar[ps], pph);
            } else if (!mbar_try_wait(&empty_bar[ps], pph)) {
                break;
            }
            issue_stage(p_it, p_tile, p_c);
            ++p_it;
            if (++p_c == n_chunks) { p_c = 0; p_tile += gridDim.x; }
        }
    };
#else
    if (warp == DT_CONSUMERS / 32) {
        // ===== producer warp =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                for (int c = 0; c < n_chunks; ++c, ++it) {
                    mbar_wait(&empty_bar[it % DT_STAGES], ((it / DT_STAGES) & 1) ^ 1);
                    issue_stage(it, tile, c);
                }
            }
        }
        return;
    }
#endif

    // ===== consumers: thread (tq, tr) owns queries 4*tq..+3 and representatives 4*tr..+3 of the tile =====
#ifdef DT_MAP_TR_FAST
    const int tr = tid % (DT_TR / 4), tq = tid / (DT_TR / 4);
#else
    const int tq = tid % (DT_TQ / 4), tr = tid / (DT_TQ / 4);
#endif
    uint32_t it = 0;
    const uint32_t k_one = a.k_one, k_two17 = a.k_two17;  // run-time multipliers: keeps the accumulations IMADs
    const uint32_t k_two = a.k_two17 >> 16;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int qt = tile / n_rt, rt = tile % n_rt;
        // per pair: acc = D (low 16 bits) | E1 (high 16 bits); `ones` is the weight-1 plane of a carry-save counter over
        // the x words: two words are folded with one full adder (2 LOP3) and only the carry (weight 2) is popcounted,
        // which moves POPC work from the XU pipe to the ALU pipe; DT_MCSA of the 16 pairs do the same for their z
        // words, which levels the two pipes (DESIGN.md "rooflines")
        uint32_t acc[4][4], ones[4][4];
        uint32_t onesM[DT_MCSA > 0 ? DT_MCSA : 1];
#pragma unroll
        for (int i = 0; i < (DT_MCSA > 0 ? DT_MCSA : 1); ++i) onesM[i] = 0u;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[i][j] = ones[i][j] = 0u;
            }

        for (int c = 0; c < n_chunks; ++c, ++it) {
            const int s = it % DT_STAGES;
            const uint32_t ph = (it / DT_STAGES) & 1;
#if DT_SELF_PRODUCE
            if (tid == 0) produce(it);
            if (warp == 0) __syncwarp();
#endif
            mbar_wait(&full_bar[s], ph);
            const uint32_t* sq = stage_base + (size_t)s * DT_STAGE_WORDS;
            const uint32_t* sr = sq + 3 * DT_WC * DT_TQ;
            // the zero words that pad the last stage are not computed on
            const int wend = min(DT_WC, ((a.W + 1) & ~1) - c * DT_WC);
#pragma unroll 1
            for (int w = 0; w < wend; w += 2) {
                uint32_t qlo[2][4], qhi[2][4], qva[2][4], rlo[2][4], rhi[2][4], rva[2][4];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint4 ql = *reinterpret_cast<const uint4*>(sq + (0 * DT_WC + w + h) * DT_TQ + 4 * tq);
                    const uint4 qh = *reinterpret_cast<const uint4*>(sq + (1 * DT_WC + w + h) * DT_TQ + 4 * tq);
                    const uint4 qv = *reinterpret_cast<const uint4*>(sq + (2 * DT_WC + w + h) * DT_TQ + 4 * tq);
                    const uint4 rl = *reinterpret_cast<const uint4*>(sr + (0 * DT_WC + w + h) * DT_TR + 4 * tr);
                    const uint4 rh = *reinterpret_cast<const uint4*>(sr + (1 * DT_WC + w + h) * DT_TR + 4 * tr);
                    const uint4 rv = *reinterpret_cast<const uint4*>(sr + (2 * DT_WC + w + h) * DT_TR + 4 * tr);
                    qlo[h][0] = ql.x; qlo[h][1] = ql.y; qlo[h][2] = ql.z; qlo[h][3] = ql.w;
                    qhi[h][0] = qh.x; qhi[h][1] = qh.y; qhi[h][2] = qh.z; qhi[h][3] = qh.w;
                    qva[h][0] = qv.x; qva[h][1] = qv.y; qva[h][2] = qv.z; qva[h][3] = qv.w;
                    rlo[h][0] = rl.x; rlo[h][1] = rl.y; rlo[h][2] = rl.z; rlo[h][3] = rl.w;
                    rhi[h][0] = rh.x; rhi[h][1] = rh.y; rhi[h][2] = rh.z; rhi[h][3] = rh.w;
                    rva[h][0] = rv.x; rva[h][1] = rv.y; rva[h][2] = rv.z; rva[h][3] = rv.w;
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        // 6 LOP3 per pair per two words (+ 2 per carry-save adder), pinned with explicit LUTs
                        const uint32_t x0 = lop3<0x3c>(qva[0][i], rva[0][j], 0u);            // exactly one side valid
                        const uint32_t x1 = lop3<0x3c>(qva[1][i], rva[1][j], 0u);
                        const uint32_t y0 = lop3<0xbe>(qlo[0][i], rlo[0][j], x0);            // (qlo ^ rlo) | x
                        const uint32_t y1 = lop3<0xbe>(qlo[1][i], rlo[1][j], x1);
                        const uint32_t m0 = lop3<0xbe>(qhi[0][i], rhi[0][j], y0);            // (qhi ^ rhi) | y
                        const uint32_t m1 = lop3<0xbe>(qhi[1][i], rhi[1][j], y1);
                        const uint32_t o = ones[i][j];
                        const uint32_t carry = lop3<0xe8>(o, x0, x1);                        // full adder: majority
                        ones[i][j] = lop3<0x96>(o, x0, x1);                                  //             parity
                        // the accumulations go to the (idle) FMA pipe as IMADs: the multipliers are opaque
                        // registers so that ptxas cannot turn them back into ALU-pipe adds / shifts
                        if (mcsa_pair(i, j)) {
                            // DT_MCSA of the 16 pairs also fold their two mismatch words with a full adder (2 more
                            // LOP3, 1 POPC less): levels the XU (POPC) and ALU (LOP3) pipes
                            const uint32_t om = onesM[mcsa_slot(i, j)];
                            const uint32_t cm = lop3<0xe8>(om, m0, m1);
                            onesM[mcsa_slot(i, j)] = lop3<0x96>(om, m0, m1);
                            acc[i][j] = __popc(cm) * k_two + acc[i][j];
                        } else {
                            acc[i][j] = __popc(m0) * k_one + acc[i][j];
                            acc[i][j] = __popc(m1) * k_one + acc[i][j];
                        }
                        acc[i][j] = __popc(carry) * k_two17 + acc[i][j];
                    }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[s]);
        }
        uint32_t accM[4][4], accV[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t a2 = acc[i][j] + (__popc(ones[i][j]) << 16) +
                                    (mcsa_pair(i, j) ? __popc(onesM[mcsa_slot(i, j)]) : 0);
                accM[i][j] = a2 & 0xffffu;  // D
                accV[i][j] = a2 >> 16;      // E1
            }

        // ---- epilogue ----
        const int q0 = qt * DT_TQ + 4 * tq, r0 = rt * DT_TR + 4 * tr;
        {
            const uint4 nq = *reinterpret_cast<const uint4*>(a.q_nv + q0);
            const uint4 nr = *reinterpret_cast<const uint4*>(a.r_nv + r0);
            const uint32_t nqa[4] = {nq.x, nq.y, nq.z, nq.w}, nra[4] = {nr.x, nr.y, nr.z, nr.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t D = accM[i][j], E1 = accV[i][j];
                    accM[i][j] = D - E1;                         // mismatching valid sites
                    accV[i][j] = (nqa[i] + nra[j] - E1) >> 1;    // sites valid on both sides
                }
        }
        if (!FULL) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                uint4 o;
                o.x = accM[i][0] | (accV[i][0] << 16);
                o.y = accM[i][1] | (accV[i][1] << 16);
                o.z = accM[i][2] | (accV[i][2] << 16);
                o.w = accM[i][3] | (accV[i][3] << 16);
                *reinterpret_cast<uint4*>(a.keys + (size_t)(q0 + i) * a.ldk + r0) = o;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int q = q0 + i, r = r0 + j;
                    if (q < a.nq && r < a.n_ref) {
                        const size_t o = (size_t)q * a.n_ref + r;
                        a.mism[o] = accM[i][j];
                        a.valid[o] = accV[i][j];
                        a.dist[o] = jc69_from_counts(accM[i][j], accV[i][j], a.vmin);
                    }
                }
        }
    }
    if (tid == 0 && blockIdx.x == 0 && a.clk) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        a.clk[2] = (unsigned long long)clock64();
        a.clk[3] = t;
    }
}

cudaError_t dense_nuc_configure() {
    cudaError_t e = cudaFuncSetAttribute(dense_nuc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DT_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(dense_nuc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DT_SMEM_BYTES);
}

static int dense_grid(int q_pad, int r_pad, int num_sms) {
    int tiles = (q_pad / DT_TQ) * (r_pad / DT_TR);
    int g = DT_MINBLOCKS * num_sms;  // resident CTAs per SM, persistent over tiles
    return tiles < g ? tiles : g;
}

void launch_dense_nuc_keys(const uint32_t* q_wm, const uint32_t* q_nv, int q_pad, const uint32_t* r_wm,
                           const uint32_t* r_nv, int r_pad, int W, int Wp, uint32_t* keys,
                           int64_t ldk, unsigned long long* clk, int num_sms, cudaStream_t s) {
    DenseNucArgs a{};
    a.clk = clk;
    a.q_wm = q_wm; a.r_wm = r_wm; a.q_nv = q_nv; a.r_nv = r_nv; a.q_pad = q_pad; a.r_pad = r_pad; a.W = W; a.Wp = Wp; a.keys = keys; a.ldk = ldk;
    a.k_one = 1u; a.k_two17 = 1u << 17;
    dense_nuc_kernel<false><<<dense_grid(q_pad, r_pad, num_sms), DT_THREADS, DT_SMEM_BYTES, s>>>(a);
}

// line minima of a key block written by dense_nuc_kernel<false> (the tensor-core kernel folds them in its epilogue): one
// thread per line, the same helpers, so the two count paths agree bit for bit
__global__ void __launch_bounds__(256) line_minima_kernel(const uint32_t* __restrict__ keys, int rows, int64_t ldk, uint32_t vmin1,
                                                          uint32_t* __restrict__ kmin) {
    const int64_t nl = ldk / 32;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)rows * nl) return;
    const uint4* src = reinterpret_cast<const uint4*>(keys + i * 32);   // row r, line l starts at r * ldk + 32 l = 32 i
    uint32_t k[32];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint4 x = src[j];
        k[4 * j] = line_usable(x.x, vmin1);
        k[4 * j + 1] = line_usable(x.y, vmin1);
        k[4 * j + 2] = line_usable(x.z, vmin1);
        k[4 * j + 3] = line_usable(x.w, vmin1);
    }
    kmin[i] = line_min32(k);
}

void launch_line_minima(const uint32_t* keys, int rows, int64_t ldk, int vmin, uint32_t* kmin, cudaStream_t s) {
    const int64_t n = (int64_t)rows * (ldk / 32);
    if (n <= 0) return;
    line_minima_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(keys, rows, ldk, (uint32_t)(vmin > 1 ? vmin : 1), kmin);
}

void launch_dense_nuc_full(const uint32_t* q_wm, const uint32_t* q_nv, int q_pad, int nq, const uint32_t* r_wm,
                           const uint32_t* r_nv, int r_pad, int n_ref, int W, int Wp,
                           int vmin, uint32_t* mism, uint32_t* valid, double* dist, int num_sms,
                           cudaStream_t s) {
    DenseNucArgs a{};
    a.q_wm = q_wm; a.r_wm = r_wm; a.q_nv = q_nv; a.r_nv = r_nv; a.q_pad = q_pad; a.r_pad = r_pad; a.W = W; a.Wp = Wp;
    a.k_one = 1u; a.k_two17 = 1u << 17;
    a.nq = nq; a.n_ref = n_ref; a.vmin = vmin; a.mism = mism; a.valid = valid; a.dist = dist;
    dense_nuc_kernel<true><<<dense_grid(q_pad, r_pad, num_sms), DT_THREADS, DT_SMEM_BYTES, s>>>(a);
}

// ---------------------------------------------------------------------------------------------------------------
// dense amino-acid kernel: dist[q][r] = scoredist(q, r)  (distance.py:681-715)
//
// Work per (query, reference, site): one BLOSUM45 lookup and one accumulation -- a table-lookup kernel, bound by the
// shared-memory pipe, not by HBM or the fp64 pipe.  Design:
//   * codes are one byte per site (0..19 amino acids in a2i order, 20 = gap).  The north star sketches 5-bit packing; with
//     a lookup per site the code is an ADDRESS, so a byte per site (no shift / mask per lookup) is the faster form of
//     the same 21-letter alphabet, and the operands are small anyway (1.6 kB per sequence at config 3);
//   * the table is held in shared memory as 44-bit FIXED POINT split into two 22-bit limbs (two uint32 tables of 21 rows
//     x 32 columns): value = round(B * 2^43).  The integer sums are exact and order-independent; the quantisation is
//     2^-44 per site (5e-14 relative on a sum of ~1e3, four orders below the 1e-9 parity tolerance, and below the
//     summation-order noise of the reference's BLAS ddot).  A row has 21 used columns, so the 32 lanes of a warp -- same
//     query symbol, 32 different references -- hit 21 distinct banks or broadcast: both lookups are conflict-free
//     (an fp64 table is 2-way conflicted by construction: 21 entries on 16 eight-byte banks);
//   * reference tiles (256 references x 64 sites = 16 KB, tile-major in global memory so a stage is one contiguous block)
//     and query tiles (8 queries x 64 sites) are staged by 1-D TMA bulk copies (cp.async.bulk + mbarrier), two stages;
//   * a thread owns 2 references x 8 queries: the reference bytes of 8 sites are unpacked once into table column
//     offsets and reused for the 8 queries; the query codes are expanded once per stage into table row offsets
//     (broadcast LDS.128), so a lookup costs 1 address add + 2 LDS.32 + 1 accumulation (IADD3 takes two sites);
//   * 32-bit limb sums are flushed into a 64-bit total every 1024 sites; valid-site counts come from bit-planes
//     (aa_valid_kernel, popc(qv & rv)) computed beside the codes.
// ---------------------------------------------------------------------------------------------------------------
// codes [rows][Lp] -> tile-major [rows_pad / T][n_chunks][T][AA_CH] (padding = gap) and valid bit-planes, word-major
// [Wv][rows_pad] (bit s % 32 of word s / 32 = site s is not a gap); block (32, 8): x = site in a 32-site word
__global__ void aa_layout_kernel(const uint8_t* __restrict__ codes, int rows, int Lp, int T, int rows_pad, int n_chunks,
                                 uint8_t* __restrict__ tm, uint32_t* __restrict__ vm) {
    const int r = blockIdx.y * blockDim.y + threadIdx.y;
    const int s = blockIdx.x * 32 + threadIdx.x;
    if (r >= rows_pad) return;
    uint8_t c = 20;
    if (r < rows && s < Lp) c = codes[(size_t)r * Lp + s];
    tm[(((size_t)(r / T) * n_chunks + s / AA_CH) * T + r % T) * AA_CH + s % AA_CH] = c;
    const uint32_t v = __ballot_sync(0xffffffffu, c != 20);
    if (threadIdx.x == 0) vm[(size_t)blockIdx.x * rows_pad + r] = v;
}

void launch_aa_layout(const uint8_t* codes, int rows, int Lp, int T, int rows_pad, uint8_t* tm, uint32_t* vm, cudaStream_t s) {
    const int n_chunks = (Lp + AA_CH - 1) / AA_CH;
    dim3 grid(n_chunks * (AA_CH / 32), (rows_pad + 7) / 8), block(32, 8);
    aa_layout_kernel<<<grid, block, 0, s>>>(codes, rows, Lp, T, rows_pad, n_chunks, tm, vm);
}

// valid[q][r] = sites where neither sequence has a gap (distance.py:698-699); lanes = consecutive references
__global__ void aa_valid_kernel(const uint32_t* __restrict__ qv, int q_pad, int nq, const uint32_t* __restrict__ rv, int r_pad,
                                int n_r, int Wv, uint32_t* __restrict__ valid, int64_t ldv) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const int q0 = blockIdx.y * 8;
    if (r >= n_r) return;
    uint32_t c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int w = 0; w < Wv; ++w) {
        const uint32_t x = rv[(size_t)w * r_pad + r];
#pragma unroll
        for (int k = 0; k < 8; ++k) c[k] += __popc(x & qv[(size_t)w * q_pad + min(q0 + k, q_pad - 1)]);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if (q0 + k < nq) valid[(size_t)(q0 + k) * ldv + r] = c[k];
}

struct DenseAaArgs {
    const uint8_t* q_tm;     // [q_pad / AA_TQ][n_chunks][AA_TQ][AA_CH]
    const uint8_t* r_tm;     // [r_pad / AA_TR][n_chunks][AA_TR][AA_CH]
    const uint32_t* tab;     // [2][21][AA_TABW] limbs (high, low)
    const uint32_t* valid;   // [nq][ldv] from aa_valid_kernel
    int64_t ldv;
    int nq, n_r, n_chunks, L;
    double overlap;
    double* dist;            // [nq][ldd]
    int64_t ldd;
};

__global__ void __launch_bounds__(AA_THREADS) dense_aa_kernel(const DenseAaArgs a) {
    constexpr int STAGE_BYTES = (AA_TR + AA_TQ) * AA_CH;
    __shared__ __align__(128) unsigned char s_stage[2][STAGE_BYTES];
    __shared__ __align__(16) uint32_t s_qoff[AA_TQ][AA_CH];   // table row offsets (bytes) of the stage's query codes
    __shared__ uint32_t s_tab[2 * 21 * AA_TABW];
    __shared__ uint64_t s_bar[2];
    const int tid = threadIdx.x;
    const int rt = blockIdx.x, qt = blockIdx.y;
    for (int i = tid; i < 2 * 21 * AA_TABW; i += AA_THREADS) s_tab[i] = a.tab[i];
    if (tid == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int c) {
        const int st = c & 1;
        mbar_arrive_expect_tx(&s_bar[st], STAGE_BYTES);
        tma_bulk_g2s(s_stage[st], a.r_tm + ((size_t)rt * a.n_chunks + c) * (AA_TR * AA_CH), AA_TR * AA_CH, &s_bar[st]);
        tma_bulk_g2s(s_stage[st] + AA_TR * AA_CH, a.q_tm + ((size_t)qt * a.n_chunks + c) * (AA_TQ * AA_CH), AA_TQ * AA_CH,
                     &s_bar[st]);
    };
    if (tid == 0) issue(0);

    uint32_t ah[AA_TQ][2], al[AA_TQ][2];
    uint64_t tot[AA_TQ][2];
#pragma unroll
    for (int q = 0; q < AA_TQ; ++q)
#pragma unroll
        for (int j = 0; j < 2; ++j) { ah[q][j] = al[q][j] = 0u; tot[q][j] = 0ull; }
    const uint32_t tab_base = smem_u32(s_tab);

    for (int c = 0; c < a.n_chunks; ++c) {
        const int st = c & 1;
        if (tid == 0 && c + 1 < a.n_chunks) issue(c + 1);   // the other buffer was released by the barrier below
        mbar_wait(&s_bar[st], (c >> 1) & 1);
        // query codes -> table row offsets, once per stage (AA_TQ * AA_CH = 512 codes, 4 per thread)
        {
            const unsigned char* qs = s_stage[st] + AA_TR * AA_CH;
            const uint32_t w = *reinterpret_cast<const uint32_t*>(qs + 4 * tid);
            uint4 o;
            o.x = (w & 0xffu) * (AA_TABW * 4);
            o.y = ((w >> 8) & 0xffu) * (AA_TABW * 4);
            o.z = ((w >> 16) & 0xffu) * (AA_TABW * 4);
            o.w = (w >> 24) * (AA_TABW * 4);
            *reinterpret_cast<uint4*>(&s_qoff[0][0] + 4 * tid) = o;
        }
        __syncthreads();
        const unsigned char* r0 = s_stage[st] + (size_t)tid * AA_CH;
        const unsigned char* r1 = s_stage[st] + (size_t)(tid + AA_THREADS) * AA_CH;
#pragma unroll 1
        for (int g = 0; g < AA_CH / 8; ++g) {
            const uint2 b0 = *reinterpret_cast<const uint2*>(r0 + 8 * g);
            const uint2 b1 = *reinterpret_cast<const uint2*>(r1 + 8 * g);
            uint32_t ro[8][2];   // table column offsets (bytes) of the two references' next 8 sites, + the table base
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t w0 = k < 4 ? b0.x : b0.y, w1 = k < 4 ? b1.x : b1.y;
                ro[k][0] = tab_base + (((w0 >> (8 * (k & 3))) & 0xffu) << 2);
                ro[k][1] = tab_base + (((w1 >> (8 * (k & 3))) & 0xffu) << 2);
            }
#pragma unroll
            for (int q = 0; q < AA_TQ; ++q) {
                const uint4 qa = *reinterpret_cast<const uint4*>(&s_qoff[q][8 * g]);       // broadcast
                const uint4 qb = *reinterpret_cast<const uint4*>(&s_qoff[q][8 * g + 4]);
                const uint32_t qo[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
#pragma unroll
                for (int k = 0; k < 8; ++k)
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const uint32_t addr = qo[k] + ro[k][j];
                        uint32_t h, l;
                        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(h) : "r"(addr));
                        asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(l) : "r"(addr), "n"(21 * AA_TABW * 4));
                        ah[q][j] += h;
                        al[q][j] += l;
                    }
            }
        }
        if ((c & 15) == 15 || c + 1 == a.n_chunks) {   // 16 stages = 1024 sites: the 22-bit limbs cannot overflow 32 bits
#pragma unroll
            for (int q = 0; q < AA_TQ; ++q)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    tot[q][j] += ((uint64_t)ah[q][j] << AA_LIMB) + al[q][j];
                    ah[q][j] = al[q][j] = 0u;
                }
        }
        __syncthreads();   // every thread is done with this stage's buffers (and with s_qoff)
    }
    // ---- epilogue: fixed point -> fp64, scoredist correction in-register.  The conversion is exact while the BLOSUM sum
    // is below 1024 (total < 2^53); beyond, it rounds at 2^-53 relative, far below the 1e-9 tolerance ----
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int r = rt * AA_TR + tid + j * AA_THREADS;
        if (r >= a.n_r) continue;
#pragma unroll
        for (int q = 0; q < AA_TQ; ++q) {
            const int qi = qt * AA_TQ + q;
            if (qi >= a.nq) continue;
            const double sum = (double)tot[q][j] * (1.0 / 8796093022208.0);   // 2^-43
            const uint32_t v = a.valid[(size_t)qi * a.ldv + r];
            a.dist[(size_t)qi * a.ldd + r] = scoredist_from_sum(sum, v, a.L, a.overlap);
        }
    }
}

// dist[nq][ldd] (and valid[nq][ldv]) from the tile-major operands; `valid` is a scratch / output buffer of nq * ldv words
void launch_dense_aa(const uint8_t* q_tm, const uint32_t* q_vm, int q_pad, int nq, const uint8_t* r_tm, const uint32_t* r_vm,
                     int r_pad, int n_r, int Lp, int L, double overlap, const uint32_t* tab, uint32_t* valid, int64_t ldv,
                     double* dist, int64_t ldd, cudaStream_t s) {
    const int n_chunks = (Lp + AA_CH - 1) / AA_CH;
    const int Wv = n_chunks * (AA_CH / 32);
    {
        dim3 grid((n_r + 127) / 128, (nq + 7) / 8);
        aa_valid_kernel<<<grid, 128, 0, s>>>(q_vm, q_pad, nq, r_vm, r_pad, n_r, Wv, valid, ldv);
    }
    DenseAaArgs a;
    a.q_tm = q_tm; a.r_tm = r_tm; a.tab = tab; a.valid = valid; a.ldv = ldv; a.nq = nq; a.n_r = n_r; a.n_chunks = n_chunks;
    a.L = L; a.overlap = overlap; a.dist = dist; a.ldd = ldd;
    dim3 grid(r_pad / AA_TR, q_pad / AA_TQ);
    dense_aa_kernel<<<grid, AA_THREADS, 0, s>>>(a);
}

// the two limb tables of round(BLOSUM45 * 2^43) (21 x 21 with a zero gap row / column, rows padded to AA_TABW words)
void aa_build_tables(const double* blosum441, uint32_t* out) {
    for (int i = 0; i < 2 * 21 * AA_TABW; ++i) out[i] = 0u;
    for (int a = 0; a < 21; ++a)
        for (int b = 0; b < 21; ++b) {
            const double x = blosum441[a * 21 + b];
            const uint64_t v = (uint64_t)(x * 8796093022208.0 + 0.5);
            out[a * AA_TABW + b] = (uint32_t)(v >> AA_LIMB);
            out[21 * AA_TABW + a * AA_TABW + b] = (uint32_t)(v & ((1u << AA_LIMB) - 1));
        }
}

// ---------------------------------------------------------------------------------------------------------------
// byte-compare fallback of the nucleotide distance stage: the reference's definition applied to the raw bytes
// (distance.py:733-737), for inputs the 2-bit planes cannot carry -- alignments longer than 65 535 columns (16-bit
// counts) and bytes other than A,C,G,T,- that survive fasta2dic (non-letters such as '.', '*', '?', digits) and count as
// ordinary characters.  One block per query, one warp per representative (grid-stride), 4 sites per lane and step; keys
// are (mismatch | valid << 32).  ~30x slower than the bit-plane kernel: a correctness path for rare inputs.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t nz_bytes(uint32_t x) { return (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u; }

__global__ void __launch_bounds__(256) dense_bytes_kernel(const uint8_t* __restrict__ q, int64_t q_stride, int nq,
                                                          const uint8_t* __restrict__ r, int64_t r_stride, int n_r, int Lp,
                                                          unsigned long long* __restrict__ keys, int64_t ldk) {
    const int qi = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t* qrow = reinterpret_cast<const uint32_t*>(q + (size_t)qi * q_stride);
    const int nw = Lp / 4;
    for (int ri = warp; ri < n_r; ri += 8) {
        const uint32_t* rrow = reinterpret_cast<const uint32_t*>(r + (size_t)ri * r_stride);
        uint32_t m = 0, v = 0;
        for (int w = lane; w < nw; w += 32) {
            const uint32_t a = qrow[w], b = rrow[w];
            const uint32_t both = nz_bytes(a ^ 0x2d2d2d2du) & nz_bytes(b ^ 0x2d2d2d2du);
            v += __popc(both);
            m += __popc(nz_bytes(a ^ b) & both);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m += __shfl_xor_sync(0xffffffffu, m, o);
            v += __shfl_xor_sync(0xffffffffu, v, o);
        }
        if (lane == 0) keys[(size_t)qi * ldk + ri] = (unsigned long long)m | ((unsigned long long)v << 32);
    }
}

void launch_dense_bytes(const uint8_t* q, int64_t q_stride, int nq, const uint8_t* r, int64_t r_stride, int n_r, int Lp,
                        unsigned long long* keys, int64_t ldk, cudaStream_t s) {
    if (nq <= 0) return;
    dense_bytes_kernel<<<nq, 256, 0, s>>>(q, q_stride, nq, r, r_stride, n_r, Lp, keys, ldk);
}

// parity export in byte mode: mism / valid / jc69 of every (query, reference) pair
__global__ void bytes_keys_to_counts_kernel(const unsigned long long* __restrict__ keys, int64_t n, int vmin, uint32_t* mism,
                                            uint32_t* valid, double* dist) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t m = (uint32_t)(keys[i] & 0xffffffffull), v = (uint32_t)(keys[i] >> 32);
    mism[i] = m;
    valid[i] = v;
    dist[i] = jc69_from_counts(m, v, vmin);
}

void launch_bytes_keys_to_counts(const unsigned long long* keys, int64_t n, int vmin, uint32_t* mism, uint32_t* valid, double* dist,
                                 cudaStream_t s) {
    if (n <= 0) return;
    bytes_keys_to_counts_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(keys, n, vmin, mism, valid, dist);
}
