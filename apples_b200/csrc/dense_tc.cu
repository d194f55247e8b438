// Kernel (a), default for nucleotide alignments: the query x representative count stage (apples/distance.py:733-737 as
// called from apples/Reference.py:138-142) on the 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in TMEM),
// bit-identical to the LOP3/POPC kernel of distance.cu (which stays selectable: apples_ctx_set_dense_mode(ctx, 0)).
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

// tile index -> (query tile, representative tile): super-tiles of sq x sr tiles, so that the ~148 CTAs of a wave share a
// few operand images in L2 instead of streaming all representatives for every pair of query tiles
__device__ __forceinline__ void tc_tile(const TcArgs& a, int t, int& qt, int& rt) {
    const int n_qt = a.q_pad / TC_TM, n_rt = a.r_pad / TC_TN;
    const int per_band = a.sq * n_rt;              // tiles of a band of sq query tiles
    const int band = t / per_band, in_band = t % per_band;
    const int q0 = band * a.sq;
    const int qh = min(a.sq, n_qt - q0);           // the last band may be thinner
    const int col = in_band / (qh * a.sr);         // super-tile column inside the band
    const int rem = in_band % (qh * a.sr);
    const int r0 = col * a.sr;
    const int rw = min(a.sr, n_rt - r0);
    // inside a (qh x rw) super-tile: row-major over its tiles; in_band was laid out with full-width columns of qh * sr tiles
    // except the last column, which holds qh * rw tiles
    qt = q0 + rem / rw;
    rt = r0 + rem % rw;
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

// function attributes are per device: called by apples_ctx_create on the context's device
cudaError_t dense_tc_configure() {
    cudaError_t e = cudaFuncSetAttribute(tc_image_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TCI_SMEM);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(dense_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
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
