// sp_kernel_w.cuh — the warp-synchronous render kernel for the reference's everyday sizes, N = P x T = 64 .. 1024
// (lib/example.html:23-84 offers 128 .. 1024, lib/spectroplot.js:254 defaults to 512).
//
// A warp transforms FW = 32 / T frames at a time; a thread holds P complex points (P = 8, 16 or 32, T <= P):
//   pass A   dft<P> over the slow input digit (stride T), twiddle W_N^{t k0};
//   exchange ONE trip through a per-warp shared-memory buffer, fenced by __syncwarp only - no block or named barrier
//            anywhere in the transform, so the 8 - 16 FFT warps of a CTA drift freely and cover each other's latencies
//            (render_rc_kernel holds 64 points per thread: 232 registers, 8 warps, three named barriers per frame);
//   pass B   P / T transforms dft<T> per thread: thread u owns rows k0 = u + T q, bins k0 + P k1.
// The window coefficients and the twiddles of a thread never change, so they live in registers.
// The raw bytes of the warp's next FW frames are prefetched by TMA bulk copies into the warp's exchange buffer; when the
// frames overlap (hop < N, the reference's normal operating point: width ~3000 frames over a short capture) the whole
// span is copied ONCE and every frame decodes from its own offset, i.e. the overlapping samples are re-read from shared
// memory, not from L2 / HBM.
// Epilogue, joint histogram (one shared-memory atomic per pixel), colour bytes staged in two halves, store warpgroup
// with full / empty mbarriers and setmaxnreg: as in render_r64_kernel.  The staging tile is transposed ([word][frame]),
// so a store warp reads 8 frames of a word with vector loads and its lanes cover 8-frame groups that are adjacent in the
// image row: a row receives 256 B .. 1 KB of contiguous bytes per store instruction.
// Spectrogram and waterfall layout, split-real (OPT), cmap_len <= 256, whole groups of 8 frames inside the buffer; everything else
// (dB tap, longer colormaps, remainder frames) stays on render_kernel.  Replaces the hot loops of reference lib/worker.js:68-137 (+ lib/samples.js:313-400,
// lib/fft_nayuki.js:54-96).
#pragma once
#include "sp_fused.cuh"

namespace sp {

// The shape of render_w_kernel for N = 2^log2n, which the engine's tile count needs as well: N = P x T with P = 8, 16, 32;
// NW FFT warps (A/B: profiles/r02_w_kernel_tuning.txt; for P = 32 8 warps of 232 registers that hold the twiddles beat
// 12 warps of 152 that read them from shared memory); WSH warp-steps of FW = 32 / T frames per warp and staging half.
constexpr int w_log2p(int log2n) { return log2n <= 6 ? 3 : (log2n <= 8 ? 4 : 5); }
constexpr int w_warps(int P) { return P <= 16 ? 16 : 8; }
constexpr int w_steps(int N) { return N == 64 ? 4 : 2; }
constexpr int w_tile_frames(int log2n)              // frames of a tile: two staging halves
{
    return 2 * w_warps(1 << w_log2p(log2n)) * w_steps(1 << log2n) * (32 >> (log2n - w_log2p(log2n)));
}

template <int LOG2P, int LOG2T, int FMT> struct WCfg {
    static constexpr int P = 1 << LOG2P, T = 1 << LOG2T, N = P * T, FW = 32 / T, Q = P / T;
    static_assert(LOG2P == w_log2p(LOG2P + LOG2T), "the P x T split of N is w_log2p's");
    static constexpr int NW = w_warps(P);                                        // FFT warps
    static_assert(NW % 4 == 0, "setmaxnreg is a warpgroup (4 warps) operation: the FFT warps must fill whole warpgroups (a mixed one hangs)");
    static constexpr int FFT_THREADS = 32 * NW, STORE_THREADS = 128, THREADS = FFT_THREADS + STORE_THREADS;
    static constexpr int STORE_REGS = 40;
    // registers: the CTA's allocation at launch is THREADS x (65536 / THREADS rounded down to 8); setmaxnreg moves registers inside it
    static constexpr int LAUNCH_REGS = (65536 / THREADS) / 8 * 8 > 255 ? 248 : (65536 / THREADS) / 8 * 8;
    static constexpr int FFT_REGS_RAW = (THREADS * LAUNCH_REGS - STORE_THREADS * STORE_REGS) / FFT_THREADS / 8 * 8;
    static constexpr int FFT_REGS = FFT_REGS_RAW > 232 ? 232 : FFT_REGS_RAW;
    static constexpr int WSH = w_steps(N);                                       // warp-steps per warp and staging half
    static constexpr int F = w_tile_frames(LOG2P + LOG2T), HF = F / 2;           // frames per tile / staging half (NW * WSH * FW)
    static constexpr int SWB = sample_width(FMT == FMT_RUNTIME ? CF64 : FMT);
    static constexpr bool OK = (FMT != FMT_RUNTIME) && SWB <= 8 && T <= P && T >= 8;
    static constexpr int XP = T + 2;                                             // exchange row pitch (float2): LDS.128 of 8 lanes conflict-free
    static constexpr int FSTR = P * XP + ((T == 8 && (P * XP) % 16 != 8) ? 8 : 0);   // float2 per frame: STS.64 of two frames in a half-warp conflict-free
    // bytes per raw frame slot: the frame, 16 bytes of alignment slack at either end, and a pad that puts the FW frames a warp
    // decodes with ONE load instruction (T lanes x SWB bytes each) into different banks
    // (a multiple of 16 bytes: bulk-copy destination)
    static constexpr int RAWP = N * SWB + ((T * SWB >= 128 || T * SWB < 16 || (T * SWB) % 16 != 0) ? 32 : (T * SWB >= 32 ? T * SWB : T * SWB + 128));
    static_assert(RAWP % 16 == 0, "raw slots are bulk-copy destinations");
    static constexpr int FPITCH = (HF + 31) / 32 * 32 + FW;                      // staging words per word column: STS.32 of a warp conflict-free
    static constexpr int HALF_WORDS = (N / 4) * FPITCH;
    // The bulk copy, its position arithmetic (double) and its barrier serve TWO consecutive warp-steps = 2 FW consecutive frames wherever
    // the doubled raw area still fits shared memory (every shape for samples of up to 4 bytes): ncu put 22 % of the FFT warps' time of
    // the N = 128 kernel, and 11 % at N = 512, into that per-step bookkeeping
    static constexpr size_t SMEM_REST = (size_t)2 * HALF_WORDS * 4 + (size_t)JH_SIZE * 4 + 1024 /* LUT */
                                      + (size_t)F * 8 /* s_mm */ + (size_t)NW * 8 + 64 + 128 + 1024 /* LUT alignment */;
    static constexpr size_t SMEM_SG2 = (size_t)NW * (((2 * FW * RAWP + 15) & ~15) + ((FW * FSTR * 8 + 15) & ~15)) + (size_t)NW * 2 * 2 * FW * 4 + SMEM_REST;
    static constexpr int SG = (WSH % 2 == 0 && SMEM_SG2 <= 232448) ? 2 : 1, FWS = FW * SG;
    // the raw frames and the exchange area of a warp do not share bytes: the exchange stores need no "raw frame consumed" fence (they
    // ride between the twiddle products) and the next frames' bulk copy starts as soon as the warp has decoded, not after pass B
    static constexpr int RAW_BYTES = (FWS * RAWP + 15) & ~15;
    static constexpr int XBYTES = RAW_BYTES + ((FW * FSTR * 8 + 15) & ~15);
    static constexpr size_t SMEM_BYTES = (size_t)NW * XBYTES + (size_t)NW * 2 * FWS * 4 /* s_off */ + SMEM_REST;
};

// min / max over the T lanes of a frame (aligned groups of T lanes).  A __reduce_*_sync with a partial mask makes the warp's
// FW groups run the collective one after the other (ncu: 10 % of the stall samples of the N = 128 kernel sat there as
// branch_resolving); an xor butterfly over log2 T steps keeps all 32 lanes together.
template <int T> __device__ __forceinline__ unsigned group_min(unsigned v)
{
    if constexpr (T == 32) return __reduce_min_sync(0xffffffffu, v);
    else {
#pragma unroll
        for (int o = 1; o < T; o <<= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
        return v;
    }
}
template <int T> __device__ __forceinline__ unsigned group_max(unsigned v)
{
    if constexpr (T == 32) return __reduce_max_sync(0xffffffffu, v);
    else {
#pragma unroll
        for (int o = 1; o < T; o <<= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
        return v;
    }
}

// twW: [P][T] float2 = W_N^{t*k} (k = 0 .. P-1; double -> fp32 once)
// OPT = true: the same kernel with the split-real post-process (lib/fft_nayuki.js:103-119) compiled in; the launcher takes it
// for channelMode messages only, so the plain kernel carries neither its registers nor its code.
template <int LOG2P, int LOG2T, int FMT, bool OPT = false>
__global__ void __launch_bounds__(WCfg<LOG2P, LOG2T, FMT>::THREADS, 1) render_w_kernel(const Params p, const float2 *__restrict__ twW)
{
    using B = WCfg<LOG2P, LOG2T, FMT>;
    constexpr int P = B::P, T = B::T, N = B::N, FW = B::FW, Q = B::Q, NW = B::NW, HF = B::HF, F = B::F, SG = B::SG, FWS = B::FWS;
    static_assert(B::WSH % SG == 0, "a stage group must not straddle staging halves");
    constexpr bool FLOAT_IN = FMT == CF32 || FMT == CF64 || FMT == FMT_RUNTIME;   // |X|^2 may be +inf / NaN
    extern __shared__ __align__(128) unsigned char smem_w[];
    const unsigned lut_base = (smem_u32(smem_w) + 1023u) & ~1023u;               // see render_r64_kernel
    unsigned char *s_x = smem_w + (lut_base - smem_u32(smem_w)) + 1024;          // [NW][XBYTES] exchange / raw frames
    unsigned *s_lut = reinterpret_cast<unsigned *>(s_x - 1024);                  // [256] RGBA indexed by the staged byte
    unsigned *s_stage = reinterpret_cast<unsigned *>(s_x + NW * B::XBYTES);      // [2][N/4][FPITCH] colour bytes: word column x frame
    unsigned *s_jh = s_stage + 2 * B::HALF_WORDS;                                // [JH_SIZE] joint histogram
    uint2 *s_mm = reinterpret_cast<uint2 *>(s_jh + JH_SIZE);                     // [F] per-frame min/max bit patterns of |X|^2
    uint64_t *s_mbar = reinterpret_cast<uint64_t *>(s_mm + F);                   // [NW] raw frames landed
    uint64_t *s_full = s_mbar + NW;                                              // [2] staging half holds HF finished frames
    uint64_t *s_empty = s_full + 2;                                              // [2] staging half has been stored
    int *s_off = reinterpret_cast<int *>(s_empty + 2);                           // [NW][2][FW] byte offset of each staged frame in the warp's buffer

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int f = lane / T, t = lane % T;   // frame of the warp-step, column
    unsigned char *xs = s_x + (size_t)(warp < NW ? warp : 0) * B::XBYTES;
    float2 *X = reinterpret_cast<float2 *>(xs + B::RAW_BYTES) + f * B::FSTR;     // this frame's exchange area
    uint64_t *mbar = s_mbar + (warp < NW ? warp : 0);

    const JhConst jc = fused_prologue(p, s_jh, s_lut, tid, B::THREADS);
    const unsigned jh_base = smem_u32(s_jh) - (JH_MAGIC_BITS << 2);
    const int nfull = p.n_full;

    // a warp: start the bulk copies of the FW frames xr .. xr + FW - 1 (chunk relative) into the warp's buffer (issued by lane 0)
    auto stage = [&](long long xr, unsigned par) {
        // called by the whole warp.  FW = 4 (N = 64, 128): lane i works out the position of frame i (double arithmetic,
        // lib/worker.js:72) and lane 0 collects them - four positions in the time of one while the warp would otherwise wait for a
        // serial loop in lane 0 (+4 % at N = 128, +3 % at N = 64; with one or two frames per warp the warp-wide double
        // instructions cost more than they save: -2 .. -4 %, so those keep the loop in lane 0)
        long long p0[FWS];
        if constexpr (FWS >= 4) {
            const int i = lane < FWS ? lane : FWS - 1;
            const long long xc = xr + i < p.chunk_frames ? xr + i : p.chunk_frames - 1;   // partial last tile: redo the last frame
            const long long xgl = p.frame_first + p.chunk_first + xc;
            const long long mine = frame_pos(p.stride, xgl) - p.sample_base;
#pragma unroll
            for (int k = 0; k < FWS; k++) p0[k] = __shfl_sync(0xffffffffu, mine, k);
            if (lane != 0) return;
        } else {
            if (lane != 0) return;
#pragma unroll
            for (int i = 0; i < FWS; i++) {
                const long long xc = xr + i < p.chunk_frames ? xr + i : p.chunk_frames - 1;
                const long long xgl = p.frame_first + p.chunk_first + xc;
                p0[i] = frame_pos(p.stride, xgl) - p.sample_base;
            }
        }
        int *off = s_off + (warp * 2 + par) * FWS;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        // overlapping frames (hop < N): ONE copy of the span, every frame decodes from its own offset in it
        const long long span = p0[FWS - 1] - p0[0] + N;
        if (FWS > 1 && span < (long long)FWS * N && span * B::SWB + 32 <= FWS * B::RAWP) {
            // staged_extent(p0[0], B::SWB, span), written out: the call changes this kernel's machine code
            const unsigned long long o0 = (unsigned long long)p0[0] * B::SWB, a0 = o0 & ~15ull;
            const unsigned bytes = (unsigned)(((o0 - a0) + (unsigned long long)span * B::SWB + 15) & ~15ull);
#pragma unroll
            for (int i = 0; i < FWS; i++) off[i] = (int)((o0 - a0) + (unsigned long long)(p0[i] - p0[0]) * B::SWB);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32(xs)), "l"(p.buf + a0), "r"(bytes), "r"(smem_u32(mbar)) : "memory");
        } else {
            unsigned total = 0;
            Extent e[FWS];
#pragma unroll
            for (int i = 0; i < FWS; i++) {
                e[i] = staged_extent(p0[i], B::SWB, N);
                off[i] = i * B::RAWP + e[i].skew;
                total += e[i].bytes;
            }
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(total) : "memory");
#pragma unroll
            for (int i = 0; i < FWS; i++)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(smem_u32(xs + i * B::RAWP)), "l"(p.buf + e[i].src), "r"(e[i].bytes), "r"(smem_u32(mbar)) : "memory");
        }
    };

    if (lane == 0 && warp < NW) mbar_init(mbar, 1);
    if (tid == 0) {
        for (int h = 0; h < 2; h++) { mbar_init(s_full + h, NW); mbar_init(s_empty + h, B::STORE_THREADS / 32); }
    }
    if (lane == 0) asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    long long tile = blockIdx.x;
    unsigned kk = 0;                        // tiles done by this CTA (phase of the full / empty barriers)

    if (tid >= B::FFT_THREADS) {
        // ================= store warps: staged colour bytes -> LUT -> image rows (lib/worker.js:115-121) =================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(B::STORE_REGS));
        const int ht = tid - B::FFT_THREADS;
        const bool rows_aligned = (p.nframes % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.image) & 31) == 0);
        constexpr int G8 = HF / 8;                                               // 8-frame groups per half
        for (; tile < p.ntiles; tile += gridDim.x, kk++) {
            const long long xr0 = tile * F;
#pragma unroll 1
            for (int h = 0; h < 2; h++) {
                mbar_wait(s_full + h, kk & 1);
                const size_t x0 = (size_t)(p.chunk_first + xr0) + HF * h;
                const unsigned *half = s_stage + h * B::HALF_WORDS;
                if (p.waterfall) {
                    // waterfall layout (lib/worker.js:116): frame x is image row nframes - 1 - x, bin b is column (b + n/2 - 1) mod n.
                    // Item = (frame, word column): the T lanes that share (q, m) hold T consecutive bins, i.e. T consecutive
                    // columns - every store instruction writes runs of 4 T contiguous bytes; the staged words of those lanes are
                    // FPITCH apart (conflict-free, like the FFT warps' writes).
#pragma unroll 1
                    for (int id = ht; id < HF * (N / 4); id += B::STORE_THREADS) {
                        const int wcol = id % (N / 4), fl = id / (N / 4);
                        if (xr0 + HF * h + fl >= p.chunk_frames) break;                   // partial last tile
                        const int u = wcol % T, qm = wcol / T, m = qm % (T / 4), q = qm / (T / 4);
                        const unsigned w = half[wcol * B::FPITCH + fl];
                        uint32_t *rowp = reinterpret_cast<uint32_t *>(p.image) + (size_t)N * (size_t)(p.nframes - 1 - (long long)(x0 + fl));
#pragma unroll
                        for (int j = 0; j < 4; j++) rowp[waterfall_col((u + T * q) + P * (4 * m + j), N)] = lut_at(lut_base, w, j);
                    }
                }
#pragma unroll 1
                for (int id = ht; id < (p.waterfall ? 0 : (N / 4) * G8); id += B::STORE_THREADS) {
                    // item = (word column, 8-frame group): adjacent lanes take adjacent groups of the same image rows
                    const int g = id % G8, wcol = id / G8;
                    if (xr0 + HF * h + 8 * g >= p.chunk_frames) continue;         // partial last tile (chunk_frames % 8 == 0)
                    const int u = wcol % T, qm = wcol / T, m = qm % (T / 4), q = qm / (T / 4);
                    const unsigned *src = half + wcol * B::FPITCH + 8 * g;
                    unsigned w[8];
                    if constexpr (FW == 4) {
                        const uint4 a = *reinterpret_cast<const uint4 *>(src), b = *reinterpret_cast<const uint4 *>(src + 4);
                        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
                    } else if constexpr (FW == 2) {
#pragma unroll
                        for (int i = 0; i < 4; i++) { const uint2 a = *reinterpret_cast<const uint2 *>(src + 2 * i); w[2 * i] = a.x; w[2 * i + 1] = a.y; }
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; i++) w[i] = src[i];
                    }
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const int bin = (u + T * q) + P * (4 * m + j);
                        uint32_t *rowp = reinterpret_cast<uint32_t *>(p.image) + (size_t)p.nframes * (size_t)image_row(bin, nfull) + x0 + 8 * g;
                        uint4 a, b;
                        lut_row8(lut_base, w, j, a, b);
                        store_row8(rowp, a, b, rows_aligned);
                    }
                }
                for (int fl = ht; fl < HF; fl += B::STORE_THREADS) {
                    // per-frame min / max of the half's frames as dB
                    if (xr0 + HF * h + fl >= p.chunk_frames) break;
                    const long long xl = p.chunk_first + xr0 + HF * h + fl;
                    const uint2 mm = s_mm[HF * h + fl];
                    const float2 db = frame_db(mm.x, mm.y, p);
                    p.fmin[xl] = db.x;
                    p.fmax[xl] = db.y;
                }
                __syncwarp();                                   // this warp is done reading the half (and s_mm)
                if ((ht & 31) == 0) mbar_arrive(s_empty + h);
            }
        }
    } else {
    // ================= FFT warps: every warp walks its own warp-steps of FW frames =================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(B::FFT_REGS));
    unsigned fpar = 0;                      // parity of this warp's step counter (mbarrier phase, s_off slot)
    // thread-invariant tables: window coefficient of sample t + T a; twiddle W_N^{t k0}
    float win[P];
#pragma unroll
    for (int a = 0; a < P; a++) win[a] = p.window[t + T * a];
    float2 tw[P];
#pragma unroll
    for (int k = 1; k < P; k++) tw[k] = twW[k * T + t];
    // frames of warp-step (h, j) of a tile: h*HF + ((j/SG)*NW + warp)*FWS + (j%SG)*FW .. + FW - 1 (a warp's SG consecutive steps = FWS consecutive frames)
    auto step_first = [&](long long tl, int h, int j) -> long long { return tl * F + h * HF + ((j / SG) * NW + warp) * FWS + (j % SG) * FW; };
    if (tile < p.ntiles) stage(step_first(tile, 0, 0), 0);

    while (tile < p.ntiles) {
        const long long next_tile = tile + gridDim.x;
#pragma unroll 1
        for (int hj = 0; hj < 2 * B::WSH; hj++) {
            int h = hj / B::WSH;
            const int j = hj % B::WSH;
            asm volatile("" : "+r"(h));                                 // (see render_r64_kernel: keeps the mbarrier address arithmetic opaque)
            const long long xr = step_first(tile, h, j) + f;            // chunk-relative frame of this thread
            const int fh = ((j / SG) * NW + warp) * FWS + (j % SG) * FW + f;   // frame within the half
            const int r = j % SG;                                       // step within the stage group
            const bool valid = xr < p.chunk_frames;                     // false: past the end of a partial last tile (outputs suppressed)
            const unsigned dump = smem_u32(s_jh + JH_SIZE - 1);         // histogram atomics of such frames land in an unused counter
            cf v[P];
            // ---------------- load + decode + window (lib/worker.js:70-75) ----------------
            if (r == 0) mbar_wait(mbar, fpar);
            {
                const unsigned char *rp = xs + s_off[(warp * 2 + fpar) * FWS + r * FW + f];
#pragma unroll
                for (int a = 0; a < P; a++) v[a] = decode_raw_cf<FMT>(rp, T * a + t, p.format);
                if (t == 0 && valid) p.fmid[p.chunk_first + xr] = raw_mid<FMT>(v[P / 2]);
#pragma unroll
                for (int a = 0; a < P; a++) v[a] = cscale(v[a], win[a]);
            }
            if (r == SG - 1) fpar ^= 1;

            // ---------------- pass A: DFT-P over the slow input digit, twiddle W_N^{t*k0} ----------------
            dft<P>(v);
            cst(X + t, v[0]);
#pragma unroll
            for (int k = 1; k < P; k++) { v[k] = cmul(v[k], tw[k]); cst(X + k * B::XP + t, v[k]); }   // Z[k0][t], between the products
            __syncwarp();                                               // the rows are complete (and every lane has decoded its raw frame)
            auto prefetch = [&]() {
                if (hj + 1 < 2 * B::WSH) stage(step_first(tile, (hj + 1) / B::WSH, (hj + 1) % B::WSH), fpar);
                else if (next_tile < p.ntiles) stage(step_first(next_tile, 0, 0), fpar);
            };
            if (r == SG - 1) prefetch();                                // the raw area is free: start the bulk copy of the warp's next frames
            // ---------------- pass B: thread u = t owns rows k0 = u + T*q: Q transforms of length T ----------------
#pragma unroll
            for (int q = 0; q < Q; q++) {
                const float4 *row = reinterpret_cast<const float4 *>(X + (t + T * q) * B::XP);
#pragma unroll
                for (int i = 0; i < T / 2; i++) {
                    const float4 z = row[i];
                    v[q * T + 2 * i] = cpk(z.x, z.y); v[q * T + 2 * i + 1] = cpk(z.z, z.w);
                }
            }
            __syncwarp();                                               // the exchange area is free (next step's stores, split-real below)
            const bool split = OPT && p.channel_mode;
            if (j == 0) mbar_wait(s_empty + h, (kk + 1) & 1);           // the store warps are done with this staging half (previous tile)
#pragma unroll
            for (int q = 0; q < Q; q++) {
                cf u_[T];
#pragma unroll
                for (int i = 0; i < T; i++) u_[i] = v[q * T + i];
                dft<T>(u_);                                             // u_[k1] is bin (t + T*q) + P*k1
#pragma unroll
                for (int i = 0; i < T; i++) v[q * T + i] = u_[i];
            }
            if constexpr (OPT) {
                if (split) {
                    // ---------------- split-real post-process (lib/fft_nayuki.js:103-119) ----------------
                    // bin i pairs with bin n - i, which lives in lane (T - t) mod T of the same frame: one more trip through the
                    // frame's exchange area, this time indexed by bin (writes and reads of a warp instruction are consecutive
                    // words: conflict-free).  Bins below n/2 are the registers k1 < T/2, bins above it k1 >= T/2; bin 0 and
                    // bin n/2 are lane 0's registers (q = 0, k1 = 0 / T/2).
#pragma unroll
                    for (int r = 0; r < P; r++) cst(X + (t + T * (r / T) + P * (r % T)), v[r]);
                    __syncwarp();
#pragma unroll
                    for (int r = 0; r < P; r++) {
                        const int q = r / T, k1 = r % T;
                        const int b = t + T * q + P * k1;
                        const cf w = cld(X + ((N - b) & (N - 1)));
                        const float2 fa = cun(v[r]);
                        cf nv;
                        if (k1 < T / 2) nv = split_lo(v[r], w);
                        else nv = split_hi(v[r], w);
                        if (q == 0 && k1 == 0 && t == 0) nv = split_dc(fa);
                        if (q == 0 && k1 == T / 2 && t == 0) nv = split_nyquist();
                        v[r] = nv;
                    }
                    __syncwarp();                                       // now the buffer is free
                }
            }

            // ---------------- per-bin epilogue (lib/worker.js:85-122) ----------------
            BinMinMax<FLOAT_IN> bm;
            unsigned *stg = s_stage + h * B::HALF_WORDS + t * B::FPITCH + fh;
#pragma unroll
            for (int q = 0; q < Q; q++)
#pragma unroll
                for (int m = 0; m < T / 4; m++)     // bins (t + T*q) + P*(4m .. 4m+3): four colour bytes in one word of column (q*(T/4) + m)*T + t
                    stg[((q * (T / 4) + m) * T) * B::FPITCH] = epilogue4(v + q * T + 4 * m, bm, jc, jh_base, valid, dump);
            auto gmin = [](unsigned x) { return group_min<T>(x); };
            auto gmax = [](unsigned x) { return group_max<T>(x); };
            unsigned umn = gmin(bm.lo()), umx = gmax(bm.hi());
            if (__any_sync(0xffffffffu, umn < 0x00800000u || umx >= 0x7f800000u))   // rare (warp-uniform)
                fixup_nonfinite(v, valid, lane == 0, true, s_jh, jc, gmin, gmax, umn, umx);
            if (t == 0) s_mm[h * HF + fh] = make_uint2(umn, umx);
            if (j == B::WSH - 1) {          // this warp has staged its last frames of the half (and their s_mm entries)
                __syncwarp();
                if (lane == 0) mbar_arrive(s_full + h);
            }
        } // warp-steps
        tile = next_tile;
        kk++;
    } // tiles
    } // FFT warps

    __syncthreads();
    flush_joint_hist(p, s_jh, tid, B::THREADS);
}

} // namespace sp
