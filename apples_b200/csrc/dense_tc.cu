// Kernel (a1): the query x representative count stage (apples/distance.py:733-737 as called from
// apples/Reference.py:138-142) on the 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in TMEM),
// bit-identical to the LOP3/POPC kernel of distance.cu (which stays selectable: apples_ctx_set_dense_mode(ctx, 0)).
// The block-scaled fp4 kernel at the end of this file (kernel (a), the default) takes alignments up to FP4_MAX_L sites;
// this one takes the rest up to TC_MAX_L.
//
// BASELINE.json's north star says "no tensor cores are used, since nothing here is a dense contraction".  The mismatch
// count IS a contraction once the alphabet is embedded in a regular simplex: with
//     A = (+,+,+)  C = (+,-,-)  G = (-,+,-)  T = (-,-,+)          (dot = 3 for equal symbols, -1 for different ones)
// scaled by 126 and a fourth component that is 125 on the query side and 127 on the reference side for a valid site (all
// four components are 0 at a gap), one site contributes
//     126^2 * (3 or -1) + 125 * 127 = 63503 (match)  or  -1 (mismatch)  or  0 (a gap on either side)
// to an int8 dot product with K = 4 L.  One s32 accumulator S = 63503 * match - mismatch therefore carries BOTH counts
// exactly (|S| < 2^31 for L <= 33 816):
//     match = (S + 63503) div 63504,   mismatch = 63503 * match - S,   valid = match + mismatch.
// Measured at config 5 on B200: 29.8 ms per 125 000 x 21 924 x 5000 step against 137.1 ms for the integer-pipe kernel at
// 0.78 of its pipe roofline (DESIGN.md section 3a): the stage is compute-bound, so it belongs on the tensor cores.
//
// Kernel: persistent, one CTA per SM: warp 0 = TMA producer (1-D bulk copies of pre-arranged operand images), warp 1 = MMA
// issuer (one thread), warps 2-9 = epilogue (tcgen05.ld, decode, 32-bit keys identical to distance.cu's, and the line
// minima of those keys, common.cuh).
// CTA tile 256 queries x 256 representatives = two M=128, N=256 accumulators (all 512 TMEM columns) sharing the B operand in
// shared memory, 3 stages of 32 sites (128 bytes of K per row: A 32 KB + B 32 KB).  Operands are K-major, no swizzle: an
// operand image is [k16 = 8][row block = 32][8 rows][16 bytes], i.e. 128-byte core matrices with SBO = 128 B between row
// blocks and LBO = 4096 B between the 16-byte K slices (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp).
#include "common.cuh"

constexpr int TC_TM = 256;                 // query rows per CTA tile
constexpr int TC_TN = 256;                 // representative rows per CTA tile
constexpr int TC_KS = 128;                 // K bytes per row and stage = 32 sites = one plane word
constexpr int TC_STAGES = 3;
constexpr int TC_IMG = TC_TM * TC_KS;      // bytes of one operand image (32 KB)
constexpr int TC_EPI_WARPS = 8;           // two per TMEM lane quarter, each takes half of the 256 columns
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;
constexpr int TC_XPOSE = 32 * 33 * 4;       // per epilogue warp: a 32 x 32 block of keys, row pitch 33 words
constexpr int TC_SMEM = TC_STAGES * 2 * TC_IMG + 1024 + 256 + TC_EPI_WARPS * TC_XPOSE;   // + alignment slack + barriers + staging
constexpr int TC_W = 63504;                // 4 * 126^2
constexpr int TC_MAX_L = 33816;            // 63503 * L < 2^31

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void tc_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(tc_smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tc_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc_smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(tc_smem_u32(bar))
                 : "memory");
}

// K-major, no swizzle: start address, LBO (K direction) and SBO (row-block direction) in 16-byte units, version 1 (sm_100)
__device__ __forceinline__ uint64_t tc_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((smem_addr & 0x3ffffu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
           (1ull << 46);
}
// kind::i8: D = s32 (2), A = B = signed int8 (1), both K-major, N >> 3 at bit 17, M >> 4 at bit 24 (UMMA::InstrDescriptor)
constexpr uint32_t TC_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TC_TN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(TC_IDESC), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// operand images: bit-planes [rows][3][W] -> int8 [rows_pad / 256][n_w][8][32][8][16]  (one 32 KB image per tile and word).
// One block per (tile of 256 rows, chunk of 32 words): the plane words are read coalesced along the row (32 consecutive
// words = 128 bytes per warp load) into shared memory, then every thread writes 16-byte pieces (4 sites x 4 components) so
// that a warp writes 512 contiguous bytes.  `vw` = the value of the fourth component (125 queries / 127 references).
// HBM-bound: 128 bytes written per 12 bytes read.
// ---------------------------------------------------------------------------------------------------------------
constexpr int TCI_WCH = 32;   // words per block
__global__ void __launch_bounds__(256) tc_image_kernel(const uint32_t* __restrict__ planes, int rows, int W, int n_w, int vw,
                                                       uint4* __restrict__ out) {
    extern __shared__ uint32_t sp[];   // [3][256][TCI_WCH + 1]
    const int tile = blockIdx.y, w0 = blockIdx.x * TCI_WCH;
    const int row0 = tile * TC_TM;
    for (int idx = threadIdx.x; idx < 3 * TC_TM * TCI_WCH; idx += 256) {
        const int wl = idx % TCI_WCH, p = (idx / TCI_WCH) % 3, r = idx / (3 * TCI_WCH);
        uint32_t x = 0;
        if (row0 + r < rows && w0 + wl < n_w) x = planes[((size_t)(row0 + r) * 3 + p) * W + w0 + wl];
        sp[(p * TC_TM + r) * (TCI_WCH + 1) + wl] = x;
    }
    __syncthreads();
    const int nwl = min(TCI_WCH, n_w - w0);
    for (int wl = 0; wl < nwl; ++wl) {
        uint4* img = out + ((size_t)tile * n_w + w0 + wl) * (TC_IMG / 16);
#pragma unroll
        for (int i = 0; i < TC_IMG / 16 / 256; ++i) {
            const int t = threadIdx.x + 256 * i;          // uint4 index inside the image: ((k16 * 32 + rb) * 8 + r8)
            const int r = ((t >> 3) & 31) * 8 + (t & 7), k16 = t >> 8;
            const uint32_t lo = sp[(0 * TC_TM + r) * (TCI_WCH + 1) + wl], hi = sp[(1 * TC_TM + r) * (TCI_WCH + 1) + wl],
                           va = sp[(2 * TC_TM + r) * (TCI_WCH + 1) + wl];
            uint32_t o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int s = k16 * 4 + j;
                const uint32_t l = (lo >> s) & 1u, h = (hi >> s) & 1u, v = (va >> s) & 1u;
                // A(0)=(+,+,+) C(1)=(+,-,-) G(2)=(-,+,-) T(3)=(-,-,+), code = lo | hi << 1; 0x7e = +126, 0x82 = -126
                const uint32_t x = h ? 0x82u : 0x7eu;
                const uint32_t y = l ? 0x82u : 0x7eu;
                const uint32_t z = (l ^ h) ? 0x82u : 0x7eu;
                o[j] = v ? (x | (y << 8) | (z << 16) | ((uint32_t)vw << 24)) : 0u;
            }
            img[t] = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
}

static const int TCI_SMEM = 3 * TC_TM * (TCI_WCH + 1) * 4;

void launch_tc_image(const uint32_t* planes, int rows, int W, int n_w, int rows_pad, int vw, void* out, cudaStream_t s) {
    if (rows_pad <= 0 || n_w <= 0) return;
    dim3 grid((n_w + TCI_WCH - 1) / TCI_WCH, rows_pad / TC_TM);
    tc_image_kernel<<<grid, 256, TCI_SMEM, s>>>(planes, rows, W, n_w, vw, (uint4*)out);
}

struct TcArgs {
    const uint8_t* a_img;   // [q_pad / 256][n_w][32 KB]
    const uint8_t* b_img;   // [r_pad / 256][n_w][32 KB]
    int q_pad, r_pad, n_w;
    uint32_t* keys;         // [q_pad][ldk] (mismatch | valid << 16)
    int64_t ldk;
    uint32_t* kmin;         // [q_pad][ldk / 32] line minima of the keys (common.cuh)
    uint32_t vmin1;         // max(vmin, 1): the overlap gate of the line minima
    int sq, sr;             // super-tile shape (query tiles x representative tiles) of the L2-friendly tile order
};

// tile index -> (query tile, representative tile) of an n_qt x n_rt tile grid: super-tiles of sq x sr tiles, so that the
// ~148 CTAs of a wave share a few operand images in L2 instead of streaming all representatives for every pair of query
// tiles
__device__ __forceinline__ void super_tile(int n_qt, int n_rt, int sq, int sr, int t, int& qt, int& rt) {
    const int per_band = sq * n_rt;                // tiles of a band of sq query tiles
    const int band = t / per_band, in_band = t % per_band;
    const int q0 = band * sq;
    const int qh = min(sq, n_qt - q0);             // the last band may be thinner
    const int col = in_band / (qh * sr);           // super-tile column inside the band
    const int rem = in_band % (qh * sr);
    const int r0 = col * sr;
    const int rw = min(sr, n_rt - r0);
    // inside a (qh x rw) super-tile: row-major over its tiles; in_band was laid out with full-width columns of qh * sr tiles
    // except the last column, which holds qh * rw tiles
    qt = q0 + rem / rw;
    rt = r0 + rem % rw;
}
__device__ __forceinline__ void tc_tile(const TcArgs& a, int t, int& qt, int& rt) {
    super_tile(a.q_pad / TC_TM, a.r_pad / TC_TN, a.sq, a.sr, t, qt, rt);
}

__global__ void __launch_bounds__(TC_THREADS, 1) dense_tc_kernel(const TcArgs a) {
    extern __shared__ unsigned char tc_smem_raw[];
    // operand images need 16-byte alignment only (no swizzle); keep 1024 for good measure
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + TC_STAGES * 2 * TC_IMG);
    uint64_t* empty = full + TC_STAGES;
    uint64_t* tfull = empty + TC_STAGES;
    uint64_t* tempty = tfull + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = (a.q_pad / TC_TM) * (a.r_pad / TC_TN);

    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            tc_mbar_init(&full[s], 1);
            tc_mbar_init(&empty[s], 1);
        }
        tc_mbar_init(tfull, 1);
        tc_mbar_init(tempty, TC_EPI_WARPS);   // one arrival per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // TMEM: all 512 columns (two 128 x 256 s32 accumulators)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tc_smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        // ===== producer =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                int qt, rt;
                tc_tile(a, t, qt, rt);
                for (int w = 0; w < a.n_w; ++w, ++it) {
                    const int s = it % TC_STAGES;
                    tc_mbar_wait(&empty[s], ((it / TC_STAGES) & 1) ^ 1);
                    tc_mbar_expect_tx(&full[s], 2 * TC_IMG);
                    unsigned char* sa = smem + (size_t)s * 2 * TC_IMG;
                    tc_bulk_g2s(sa, a.a_img + ((size_t)qt * a.n_w + w) * TC_IMG, TC_IMG, &full[s]);
                    tc_bulk_g2s(sa + TC_IMG, a.b_img + ((size_t)rt * a.n_w + w) * TC_IMG, TC_IMG, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            uint32_t it = 0, tl = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tl) {
                tc_mbar_wait(tempty, (tl & 1) ^ 1);   // the epilogue has drained the accumulators of the previous tile
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                for (int w = 0; w < a.n_w; ++w, ++it) {
                    const int s = it % TC_STAGES;
                    tc_mbar_wait(&full[s], (it / TC_STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t sa = tc_smem_u32(smem + (size_t)s * 2 * TC_IMG), sb = sa + TC_IMG;
#pragma unroll
                    for (int k = 0; k < TC_KS / 32; ++k) {          // 4 MMAs of K = 32 bytes
                        const uint64_t bd = tc_desc(sb + 2 * k * 4096, 4096, 128);
#pragma unroll
                        for (int h = 0; h < 2; ++h) {               // the two 128-row halves of the query image
                            const uint64_t ad = tc_desc(sa + h * 2048 + 2 * k * 4096, 4096, 128);
                            tc_mma(tmem + (uint32_t)h * TC_TN, ad, bd, (w > 0 || k > 0) ? 1u : 0u);
                        }
                    }
                    tc_commit(&empty[s]);      // arrives when the MMAs above have read their operands
                }
                tc_commit(tfull);              // accumulators complete
            }
        }
    } else {
        // ===== epilogue: a warp can read the TMEM lanes 32 * (warp % 4) .. + 31; two warps share a quarter, 128 columns each =====
        const int quarter = warp & 3;
        const int c0 = ((warp - 2) >> 2) * (TC_TN / 2);
        uint32_t* xp = reinterpret_cast<uint32_t*>(smem + TC_STAGES * 2 * TC_IMG + 256) + (size_t)(warp - 2) * (TC_XPOSE / 4);
        uint32_t tl = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tl) {
            int qt, rt;
            tc_tile(a, t, qt, rt);
            tc_mbar_wait(tfull, tl & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {
                const int row0 = qt * TC_TM + h * 128 + quarter * 32;   // first of the warp's 32 rows
                // the minima of the lane's row in the warp's 4 lines, shifted in one line per 32 columns
                uint32_t lm0 = LINE_NONE, lm1 = LINE_NONE, lm2 = LINE_NONE, lm3 = LINE_NONE;
#pragma unroll 1
                for (int c = c0; c < c0 + TC_TN / 2; c += 32) {
                    uint32_t v[32];
                    const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(h * TC_TN + c);
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                        : "r"(taddr)
                        : "memory");
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    // decode, then transpose the warp's 32 rows x 32 columns through shared memory: a lane holds one ROW of
                    // the block, but a store instruction should write whole 128-byte row segments (4 rows x 128 B per
                    // instruction instead of 32 rows x 16 B: 8x fewer lines per store).
                    // The line minimum in registers: the lane holds the whole line of its row (no shuffles).  Folded on
                    // (mismatch, match) in column order: m / v orders as m / match, and a key under the overlap gate never
                    // replaces the running minimum (which starts at "none", 1 / 0); whether the winner passes 4 m < 3 v is
                    // decided once per line below.  Same result as line_usable / line_min32 (common.cuh)
                    uint32_t bmi = 1u, bma = 0u;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int S = (int)v[j];
                        const uint32_t match = (uint32_t)(S + (TC_W - 1)) / (uint32_t)TC_W;
                        const uint32_t mism = (uint32_t)((int)((TC_W - 1) * match) - S);
                        xp[lane * 33 + j] = mism | ((match + mism) << 16);
                        const bool lower = match + mism >= a.vmin1 && mism * bma < bmi * match;
                        bmi = lower ? mism : bmi;
                        bma = lower ? match : bma;
                    }
                    lm0 = lm1;
                    lm1 = lm2;
                    lm2 = lm3;
                    lm3 = (bmi < 3u * bma) ? (bmi | ((bmi + bma) << 16)) : LINE_NONE;
                    __syncwarp();
#pragma unroll
                    for (int r0 = 0; r0 < 32; r0 += 4) {
                        const int rr = r0 + (lane >> 3), cc = (lane & 7) * 4;
                        const uint4 o = make_uint4(xp[rr * 33 + cc], xp[rr * 33 + cc + 1], xp[rr * 33 + cc + 2], xp[rr * 33 + cc + 3]);
                        // streaming store: the 1.8 GB of keys of a launch must not evict the operand images from L2
                        __stcs(reinterpret_cast<uint4*>(a.keys + (size_t)(row0 + rr) * a.ldk + (size_t)rt * TC_TN + c + cc), o);
                    }
                    __syncwarp();
                }
                // one 16-byte store per row: lines (rt * 256 + c0) / 32 .. + 3 (ldk is a multiple of 256)
                __stcs(reinterpret_cast<uint4*>(a.kmin + (size_t)(row0 + lane) * (a.ldk / 32) + ((size_t)rt * TC_TN + c0) / 32),
                       make_uint4(lm0, lm1, lm2, lm3));
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) tc_mbar_arrive(tempty);
        }
    }
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// ===============================================================================================================
// Kernel (a) on block-scaled fp4 (tcgen05.mma kind::mxf4, all scale factors 1.0): the default for alignments of up to
// FP4_MAX_L sites.  The kind::i8 kernel above needs 4 operand bytes per site because one s32 accumulator carries both
// counts through the weight 63503; fp4 cannot hold those weights, so the counts go to TWO fp32 accumulators instead,
// and each operand element goes to exactly one of them:
//     D1 = sum of the three +-1 simplex components   = 3 match - mismatch   (in [-L, 3L])
//     D2 = sum of the validity component (1 or 0)    = match + mismatch     (in [0, L])
// Both are small integers, exact in fp32 (tests/test_gpu_count_fp4.py checks the whole range on the device), and
//     match = (D1 + D2) / 4,   mismatch = D2 - match.
// A site is 4 e2m1 elements = 2 bytes of K instead of 4.
//
// Kernel: the same persistent structure as dense_tc_kernel (producer warp, MMA warp, 8 epilogue warps, super-tile order,
// streaming key stores, line minima).  CTA tile 128 queries x 224 representatives: D1 in TMEM columns 0..223, D2 in
// 256..479, the constant scale factors in 480..511.  A stage is 64 sites = 128 bytes of K per row (A 16 KB + B 28 KB),
// 4 stages.  Per stage the MMA warp issues 4 MMAs of K = 64: the x, y and z slices into D1, the validity slice into D2.
// Operand images are K-major, no swizzle, in 128-byte core matrices as above: [k16 = 8][row block = R / 8][8 rows][16 B]
// with R = 128 or 224 rows, so LBO = 16 R bytes; the 16-byte piece k16 = 2 * component + (word & 1) holds the 32 sites
// of one plane word, site s in nibble s.  The MMA sums over all of K, so only the SAME order on both sides matters.
//
// The K2P instantiation (dense_fp4_kernel<true>) counts transitions and transversions apart.  With code = lo | hi << 1
// (A=0 C=1 G=2 T=3), lo separates purines from pyrimidines, so over a valid pair the y product is -1 exactly for a
// transversion, and x x' + z z' is +2 for a match, -2 for a transition and 0 for a transversion.  The y slice goes to a
// third accumulator D3 instead of D1 (still 4 MMAs per stage, no operand byte added):
//     D1' = sum (x + z) = 2 (match - ts),   D2 = valid,   D3 = sum y = valid - 2 tv
// so tv = (D2 - D3) / 2 and ts = (D2 - tv - D1' / 2) / 2, all integers within +-2 L (exact in fp32).  Three 128 x N fp32
// accumulators and the 32 scale-factor columns fit 512 TMEM columns for N = 160: D1' at 0, D2 at 160, D3 at 320, scale
// factors at 480 / 496 as above.  The tile is 128 x 160 (5 whole 32-key lines); the epilogue writes 64-bit keys
// ts | tv << 16 | valid << 32 and folds no line minima.
// ===============================================================================================================
#ifndef FP4_MAX_L_V
#define FP4_MAX_L_V 33816
#endif
constexpr int FP4_MAX_L = FP4_MAX_L_V;      // longest alignment of the fp4 kernel (build-time knob for measurements)
constexpr int F4_TM = 128;                  // query rows per CTA tile
constexpr int F4_TN = 224;                  // representative rows per CTA tile (whole 32-key lines: 7)
constexpr int F4_KS = 128;                  // K bytes per row and stage = 64 sites x 4 components x 4 bits
constexpr int F4_STAGES = 4;
constexpr int F4_A = F4_TM * F4_KS;         // 16 KB
constexpr int F4_B = F4_TN * F4_KS;         // 28 KB
constexpr int F4_STAGE = F4_A + F4_B;
constexpr int F4_SMEM = F4_STAGES * F4_STAGE + 1024 + 256 + TC_EPI_WARPS * TC_XPOSE;
constexpr uint32_t F4_D2 = 256, F4_SFA = 480, F4_SFB = 496;   // TMEM columns of D2 and of the scale factors
// K2P instantiation: 128 x 160 tiles, D2 and D3 at TMEM columns 160 and 320, a 64-bit key transpose block per warp
constexpr int F4K_TN = 160;
constexpr int F4K_B = F4K_TN * F4_KS;       // 20 KB
constexpr int F4K_STAGE = F4_A + F4K_B;
constexpr int F4K_XPOSE = 32 * 33 * 8;
constexpr int F4K_SMEM = F4_STAGES * F4K_STAGE + 1024 + 256 + TC_EPI_WARPS * F4K_XPOSE;
constexpr uint32_t F4K_D2 = 160, F4K_D3 = 320;
// kind::mxf4 (UMMA::InstrDescriptorBlockScaled): A = B = E2M1 (1) at bits 7 and 10, both K-major, N >> 3 at bit 17,
// scale format UE8M0 at bit 23, M >> 4 at bit 24, scale-factor ids 0, K = 64
template <int TN>
constexpr uint32_t F4_IDESC = (1u << 7) | (1u << 10) | ((uint32_t)(TN >> 3) << 17) | (1u << 23) | ((uint32_t)(F4_TM >> 4) << 24);
constexpr uint32_t F4_ONES = 0x7f7f7f7fu;   // four UE8M0 scale factors of 2^0

template <int TN>
__device__ __forceinline__ void f4_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t sfa, uint32_t sfb,
                                       uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.scale_vec::2X [%0], %1, %2, %3, [%4], [%5], p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(F4_IDESC<TN>), "r"(sfa), "r"(sfb), "r"(accumulate)
        : "memory");
}

// 32 consecutive TMEM columns of the warp's 32 lanes
__device__ __forceinline__ void f4_ld32(uint32_t taddr, uint32_t* d) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]), "=r"(d[4]), "=r"(d[5]), "=r"(d[6]), "=r"(d[7]),
          "=r"(d[8]), "=r"(d[9]), "=r"(d[10]), "=r"(d[11]), "=r"(d[12]), "=r"(d[13]), "=r"(d[14]), "=r"(d[15]),
          "=r"(d[16]), "=r"(d[17]), "=r"(d[18]), "=r"(d[19]), "=r"(d[20]), "=r"(d[21]), "=r"(d[22]), "=r"(d[23]),
          "=r"(d[24]), "=r"(d[25]), "=r"(d[26]), "=r"(d[27]), "=r"(d[28]), "=r"(d[29]), "=r"(d[30]), "=r"(d[31])
        : "r"(taddr)
        : "memory");
}
// an fp32 accumulator holding an integer of magnitude < 2^22 -> that integer (the 1.5 * 2^23 shift)
__device__ __forceinline__ int f4_int(uint32_t d) {
    return __float_as_int(__int_as_float((int)d) + 12582912.0f) - 0x4b400000;
}

// 8 bits -> bit i at bit 4 i
__device__ __forceinline__ uint32_t f4_spread(uint32_t b) {
    b = (b | (b << 12)) & 0x000f000fu;
    b = (b | (b << 6)) & 0x03030303u;
    return (b | (b << 3)) & 0x11111111u;
}
// the 32 sites of one component as e2m1 nibbles: +1 = 0x2, -1 = 0xa (neg = sign bits), 0 where `valid` is clear
__device__ __forceinline__ uint4 f4_nibbles(uint32_t valid, uint32_t neg) {
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = (f4_spread((valid >> (8 * j)) & 0xffu) << 1) | (f4_spread((neg >> (8 * j)) & 0xffu) << 3);
    return make_uint4(o[0], o[1], o[2], o[3]);
}

// fp4 operand images: bit-planes [rows][3][W] -> [rows_pad / R][n_c][R * 128 bytes], n_c = ceil(n_w / 2) chunks of 64
// sites (a missing odd word is all gaps).  One thread per (row, word): a warp takes 32 rows of one word, so each of its
// four 16-byte stores per thread covers 512 contiguous bytes; the 8 warps of a block take 8 consecutive words of the same
// rows, which share the 32-byte sectors of the plane reads.  The validity component is 1 at every valid site on both sides.
__global__ void __launch_bounds__(256) fp4_image_kernel(const uint32_t* __restrict__ planes, int rows, int W, int n_w, int R,
                                                        uint4* __restrict__ out) {
    const int n_c = (n_w + 1) / 2;
    const int r = blockIdx.y * 32 + (threadIdx.x & 31);
    const int w = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (w >= 2 * n_c) return;
    uint32_t lo = 0, hi = 0, va = 0;
    if (r < rows && w < n_w) {
        const uint32_t* p = planes + (size_t)r * 3 * W + w;
        lo = p[0];
        hi = p[W];
        va = p[2 * W];
    }
    const int rr = r % R;
    uint4* img = out + ((size_t)(r / R) * n_c + (w >> 1)) * (R * 8) + (rr >> 3) * 8 + (rr & 7);
    // A(0)=(+,+,+) C(1)=(+,-,-) G(2)=(-,+,-) T(3)=(-,-,+), code = lo | hi << 1 (as tc_image_kernel)
    const int k = w & 1;
    img[(0 + k) * R] = f4_nibbles(va, hi & va);          // k16 piece = R / 8 core matrices = R * 8 uint4
    img[(2 + k) * R] = f4_nibbles(va, lo & va);
    img[(4 + k) * R] = f4_nibbles(va, (lo ^ hi) & va);
    img[(6 + k) * R] = f4_nibbles(va, 0u);
}

// K2P = false: JC69 keys and line minima (D1, D2); K2P = true: the K2P keys (D1', D2, D3), see above
template <bool K2P>
__global__ void __launch_bounds__(TC_THREADS, 1) dense_fp4_kernel(const TcArgs a) {   // a.n_w = chunks of 64 sites
    constexpr int TN = K2P ? F4K_TN : F4_TN;
    constexpr int B_BYTES = TN * F4_KS;
    constexpr int STAGE = F4_A + B_BYTES;
    extern __shared__ unsigned char tc_smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + F4_STAGES * STAGE);
    uint64_t* empty = full + F4_STAGES;
    uint64_t* tfull = empty + F4_STAGES;
    uint64_t* tempty = tfull + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_qt = a.q_pad / F4_TM, n_rt = a.r_pad / TN;
    const int n_tiles = n_qt * n_rt;

    if (tid == 0) {
        for (int s = 0; s < F4_STAGES; ++s) {
            tc_mbar_init(&full[s], 1);
            tc_mbar_init(&empty[s], 1);
        }
        tc_mbar_init(tfull, 1);
        tc_mbar_init(tempty, TC_EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tc_smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    // scale factors: 1.0 in every byte of columns 480..511 of all 128 lanes, by warps 2..5 (one per lane quarter)
    if (warp >= 2 && warp < 6) {
        const uint32_t taddr = tmem + ((uint32_t)((warp & 3) * 32) << 16) + F4_SFA;
        const uint32_t o = F4_ONES;
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
            "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
            "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(o)
            : "memory");
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    if (warp == 0) {
        // ===== producer =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                int qt, rt;
                super_tile(n_qt, n_rt, a.sq, a.sr, t, qt, rt);
                for (int c = 0; c < a.n_w; ++c, ++it) {
                    const int s = it % F4_STAGES;
                    tc_mbar_wait(&empty[s], ((it / F4_STAGES) & 1) ^ 1);
                    tc_mbar_expect_tx(&full[s], STAGE);
                    unsigned char* sa = smem + (size_t)s * STAGE;
                    tc_bulk_g2s(sa, a.a_img + ((size_t)qt * a.n_w + c) * F4_A, F4_A, &full[s]);
                    tc_bulk_g2s(sa + F4_A, a.b_img + ((size_t)rt * a.n_w + c) * B_BYTES, B_BYTES, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            const uint32_t sfa = tmem + F4_SFA, sfb = tmem + F4_SFB;
            uint32_t it = 0, tl = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tl) {
                tc_mbar_wait(tempty, (tl & 1) ^ 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                for (int c = 0; c < a.n_w; ++c, ++it) {
                    const int s = it % F4_STAGES;
                    tc_mbar_wait(&full[s], (it / F4_STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t sa = tc_smem_u32(smem + (size_t)s * STAGE), sb = sa + F4_A;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {   // components x, y, z into D1, validity into D2 (K2P: y into D3)
                        const uint64_t ad = tc_desc(sa + 2 * k * (F4_TM * 16), F4_TM * 16, 128);
                        const uint64_t bd = tc_desc(sb + 2 * k * (TN * 16), TN * 16, 128);
                        if (K2P && k == 1)
                            f4_mma<TN>(tmem + F4K_D3, ad, bd, sfa, sfb, c > 0 ? 1u : 0u);
                        else if (k < 3)
                            f4_mma<TN>(tmem, ad, bd, sfa, sfb, (c > 0 || k > 0) ? 1u : 0u);
                        else
                            f4_mma<TN>(tmem + (K2P ? F4K_D2 : F4_D2), ad, bd, sfa, sfb, c > 0 ? 1u : 0u);
                    }
                    tc_commit(&empty[s]);
                }
                tc_commit(tfull);
            }
        }
    } else if constexpr (K2P) {
        // ===== K2P epilogue: two warps per TMEM lane quarter; g = 0 takes the lines 0..2 of the tile row, g = 1 the lines 3..4 =====
        const int quarter = warp & 3, g = (warp - 2) >> 2;
        const int c0 = g * 96, c1 = g ? F4K_TN : 96;
        unsigned long long* xp =
            reinterpret_cast<unsigned long long*>(smem + F4_STAGES * STAGE + 256) + (size_t)(warp - 2) * (F4K_XPOSE / 8);
        unsigned long long* keys = reinterpret_cast<unsigned long long*>(a.keys);
        uint32_t tl = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tl) {
            int qt, rt;
            super_tile(n_qt, n_rt, a.sq, a.sr, t, qt, rt);
            tc_mbar_wait(tfull, tl & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int row0 = qt * F4_TM + quarter * 32;
#pragma unroll 1
            for (int c = c0; c < c1; c += 32) {
                uint32_t d1[32], d2[32], d3[32];
                const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c;
                f4_ld32(taddr, d1);
                f4_ld32(taddr + F4K_D2, d2);
                f4_ld32(taddr + F4K_D3, d3);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int mts2 = f4_int(d1[j]), valid = f4_int(d2[j]), y = f4_int(d3[j]);
                    const int tv = (valid - y) >> 1;
                    const int ts = (valid - tv - (mts2 >> 1)) >> 1;
                    xp[lane * 33 + j] = (unsigned long long)(uint32_t)(ts | (tv << 16)) | ((unsigned long long)valid << 32);
                }
                __syncwarp();
                // 2 rows x 256 bytes per store instruction
#pragma unroll
                for (int r0 = 0; r0 < 32; r0 += 2) {
                    const int rr = r0 + (lane >> 4), cc = (lane & 15) * 2;
                    const ulonglong2 o = make_ulonglong2(xp[rr * 33 + cc], xp[rr * 33 + cc + 1]);
                    __stcs(reinterpret_cast<ulonglong2*>(keys + (size_t)(row0 + rr) * a.ldk + (size_t)rt * F4K_TN + c + cc), o);
                }
                __syncwarp();
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) tc_mbar_arrive(tempty);
        }
    } else {
        // ===== epilogue: two warps per TMEM lane quarter; g = 0 takes the lines 0..3 of the tile row, g = 1 the lines 4..6 =====
        const int quarter = warp & 3, g = (warp - 2) >> 2;
        const int c0 = g * 128, c1 = g ? F4_TN : 128;
        uint32_t* xp = reinterpret_cast<uint32_t*>(smem + F4_STAGES * STAGE + 256) + (size_t)(warp - 2) * (TC_XPOSE / 4);
        uint32_t tl = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tl) {
            int qt, rt;
            super_tile(n_qt, n_rt, a.sq, a.sr, t, qt, rt);
            tc_mbar_wait(tfull, tl & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int row0 = qt * F4_TM + quarter * 32;
            uint32_t lm0 = LINE_NONE, lm1 = LINE_NONE, lm2 = LINE_NONE, lm3 = LINE_NONE;
#pragma unroll 1
            for (int c = c0; c < c1; c += 32) {
                uint32_t d1[32], d2[32];
                const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c;
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(d1[0]), "=r"(d1[1]), "=r"(d1[2]), "=r"(d1[3]), "=r"(d1[4]), "=r"(d1[5]), "=r"(d1[6]), "=r"(d1[7]),
                      "=r"(d1[8]), "=r"(d1[9]), "=r"(d1[10]), "=r"(d1[11]), "=r"(d1[12]), "=r"(d1[13]), "=r"(d1[14]), "=r"(d1[15]),
                      "=r"(d1[16]), "=r"(d1[17]), "=r"(d1[18]), "=r"(d1[19]), "=r"(d1[20]), "=r"(d1[21]), "=r"(d1[22]), "=r"(d1[23]),
                      "=r"(d1[24]), "=r"(d1[25]), "=r"(d1[26]), "=r"(d1[27]), "=r"(d1[28]), "=r"(d1[29]), "=r"(d1[30]), "=r"(d1[31])
                    : "r"(taddr)
                    : "memory");
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(d2[0]), "=r"(d2[1]), "=r"(d2[2]), "=r"(d2[3]), "=r"(d2[4]), "=r"(d2[5]), "=r"(d2[6]), "=r"(d2[7]),
                      "=r"(d2[8]), "=r"(d2[9]), "=r"(d2[10]), "=r"(d2[11]), "=r"(d2[12]), "=r"(d2[13]), "=r"(d2[14]), "=r"(d2[15]),
                      "=r"(d2[16]), "=r"(d2[17]), "=r"(d2[18]), "=r"(d2[19]), "=r"(d2[20]), "=r"(d2[21]), "=r"(d2[22]), "=r"(d2[23]),
                      "=r"(d2[24]), "=r"(d2[25]), "=r"(d2[26]), "=r"(d2[27]), "=r"(d2[28]), "=r"(d2[29]), "=r"(d2[30]), "=r"(d2[31])
                    : "r"(taddr + F4_D2)
                    : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                // decode and line minimum as in dense_tc_kernel.  fp32 -> integer by the 1.5 * 2^23 shift (exact for
                // |x| < 2^22): D1 + D2 = 4 match and D2 = valid are integers in [0, 4 L]
                uint32_t bmi = 1u, bma = 0u;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float f1 = __int_as_float((int)d1[j]), f2 = __int_as_float((int)d2[j]);
                    const uint32_t m4 = (uint32_t)__float_as_int((f1 + f2) + 12582912.0f) - 0x4b400000u;
                    const uint32_t valid = (uint32_t)__float_as_int(f2 + 12582912.0f) - 0x4b400000u;
                    const uint32_t match = m4 >> 2;
                    const uint32_t mism = valid - match;
                    xp[lane * 33 + j] = mism | (valid << 16);
                    const bool lower = valid >= a.vmin1 && mism * bma < bmi * match;
                    bmi = lower ? mism : bmi;
                    bma = lower ? match : bma;
                }
                lm0 = lm1;
                lm1 = lm2;
                lm2 = lm3;
                lm3 = (bmi < 3u * bma) ? (bmi | ((bmi + bma) << 16)) : LINE_NONE;
                __syncwarp();
#pragma unroll
                for (int r0 = 0; r0 < 32; r0 += 4) {
                    const int rr = r0 + (lane >> 3), cc = (lane & 7) * 4;
                    const uint4 o = make_uint4(xp[rr * 33 + cc], xp[rr * 33 + cc + 1], xp[rr * 33 + cc + 2], xp[rr * 33 + cc + 3]);
                    __stcs(reinterpret_cast<uint4*>(a.keys + (size_t)(row0 + rr) * a.ldk + (size_t)rt * F4_TN + c + cc), o);
                }
                __syncwarp();
            }
            // the warp's lines of its row: lm0..lm3 = lines 0..3 (g = 0), lm1..lm3 = lines 4..6 (g = 1)
            uint32_t* mrow = a.kmin + (size_t)(row0 + lane) * (a.ldk / 32) + (size_t)rt * (F4_TN / 32) + 3 * g;
            if (g == 0) __stcs(mrow, lm0);
            __stcs(mrow + 1, lm1);
            __stcs(mrow + 2, lm2);
            __stcs(mrow + 3, lm3);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) tc_mbar_arrive(tempty);
        }
    }
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// function attributes are per device: called by apples_ctx_create on the context's device
cudaError_t dense_tc_configure() {
    cudaError_t e = cudaFuncSetAttribute(tc_image_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TCI_SMEM);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(dense_fp4_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, F4_SMEM);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(dense_fp4_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, F4K_SMEM);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(dense_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
}

int dense_fp4_max_sites() { return FP4_MAX_L < TC_MAX_L ? FP4_MAX_L : TC_MAX_L; }
int dense_fp4_tile_rows(int side, bool k2p) { return side ? (k2p ? F4K_TN : F4_TN) : F4_TM; }
size_t dense_fp4_image_bytes(int rows_pad, int n_w) { return (size_t)rows_pad * ((n_w + 1) / 2) * F4_KS; }

void launch_fp4_image(const uint32_t* planes, int rows, int W, int n_w, int rows_pad, int tile_rows, void* out, cudaStream_t s) {
    if (rows_pad <= 0 || n_w <= 0) return;
    const int n_c = (n_w + 1) / 2;
    dim3 grid((2 * n_c + 7) / 8, rows_pad / 32);
    fp4_image_kernel<<<grid, 256, 0, s>>>(planes, rows, W, n_w, tile_rows, (uint4*)out);
}

void launch_dense_fp4(const void* a_img, int q_pad, const void* b_img, int r_pad, int n_w, uint32_t* keys, int64_t ldk,
                      uint32_t* kmin, int vmin, int num_sms, cudaStream_t s) {
    TcArgs a;
    a.a_img = (const uint8_t*)a_img;
    a.b_img = (const uint8_t*)b_img;
    a.q_pad = q_pad;
    a.r_pad = r_pad;
    a.n_w = (n_w + 1) / 2;
    a.keys = keys;
    a.ldk = ldk;
    a.kmin = kmin;
    a.vmin1 = (uint32_t)(vmin > 1 ? vmin : 1);
    a.sq = 12;
    a.sr = 12;
    const int tiles = (q_pad / F4_TM) * (r_pad / F4_TN);
    dense_fp4_kernel<false><<<tiles < num_sms ? tiles : num_sms, TC_THREADS, F4_SMEM, s>>>(a);
}

void launch_dense_fp4_k2p(const void* a_img, int q_pad, const void* b_img, int r_pad, int n_w, unsigned long long* keys,
                          int64_t ldk, int num_sms, cudaStream_t s) {
    TcArgs a;
    a.a_img = (const uint8_t*)a_img;
    a.b_img = (const uint8_t*)b_img;
    a.q_pad = q_pad;
    a.r_pad = r_pad;
    a.n_w = (n_w + 1) / 2;
    a.keys = reinterpret_cast<uint32_t*>(keys);
    a.ldk = ldk;
    a.kmin = nullptr;
    a.vmin1 = 1;
    a.sq = 12;
    a.sr = 12;
    const int tiles = (q_pad / F4_TM) * (r_pad / F4K_TN);
    dense_fp4_kernel<true><<<tiles < num_sms ? tiles : num_sms, TC_THREADS, F4K_SMEM, s>>>(a);
}

int dense_tc_max_sites() { return TC_MAX_L; }
int dense_tc_tile_rows() { return TC_TM; }
size_t dense_tc_image_bytes(int rows_pad, int n_w) { return (size_t)(rows_pad / TC_TM) * n_w * TC_IMG; }

void launch_dense_tc(const void* a_img, int q_pad, const void* b_img, int r_pad, int n_w, uint32_t* keys, int64_t ldk,
                     uint32_t* kmin, int vmin, int num_sms, cudaStream_t s) {
    TcArgs a;
    a.a_img = (const uint8_t*)a_img;
    a.b_img = (const uint8_t*)b_img;
    a.q_pad = q_pad;
    a.r_pad = r_pad;
    a.n_w = n_w;
    a.keys = keys;
    a.ldk = ldk;
    a.kmin = kmin;
    a.vmin1 = (uint32_t)(vmin > 1 ? vmin : 1);
    // super-tiles of about one wave: 12 x 12 tiles = 144 CTAs share 12 + 12 operand images per K step (shapes from 7 x 7 to
    // 37 x 4 measure within 2% of each other, profiles/tc_tile_sweep_r02.txt; only 1-wide strips lose, 11%)
    a.sq = 12;
    a.sr = 12;
    const int tiles = (q_pad / TC_TM) * (r_pad / TC_TN);
    dense_tc_kernel<<<tiles < num_sms ? tiles : num_sms, TC_THREADS, TC_SMEM, s>>>(a);
}
