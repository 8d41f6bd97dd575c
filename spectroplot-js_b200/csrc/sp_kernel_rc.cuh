// sp_kernel_rc.cuh — the 64-points-per-thread render kernel for N = 2048 = 64 x C, C = 32.
//
// Same machine as render_r64_kernel (sp_kernel_r64.cuh), with the frame folded differently:
//   * N = 64 x C: C = 32 threads (one warp) transform a frame, each holding 64 complex points: dft<64> over the slow input
//     digit (stride C), twiddle W_N^{t*k0}, ONE shared-memory exchange, then RPT = 64 / C = 2 row transforms dft<C> per
//     thread (thread t owns rows k0 = 2t, 2t + 1, bins k0 + 64*k1);
//   * a stream of 64 threads therefore works on FS = 2 frames at a time, its raw frames prefetched by FS bulk copies
//     (TMA) on one mbarrier into the stream's exchange buffer;
//   * joint histogram (one shared-memory atomic per pixel), colour bytes staged in two halves of 16 frames, store
//     warpgroup with full / empty mbarriers, setmaxnreg — exactly as in render_r64_kernel; a lane of the store warps
//     still writes one 32-byte sector (8 frames of one row), and adjacent lanes take the two 8-frame groups of a half,
//     so a row receives 64 contiguous bytes per instruction.
// Only full tiles of 32 frames inside the buffer come here (spectrogram layout, cmap_len <= 256); the engine routes
// everything else through render_kernel.
// Replaces the hot loops of reference lib/worker.js:68-137 (+ lib/samples.js:313-400, lib/fft_nayuki.js:54-96).
#pragma once
#include "sp_fused.cuh"

namespace sp {

template <int FMT> struct RcCfg {
    static constexpr int C = 32, N = 64 * C, RPT = 64 / C, FS = 64 / C;          // threads per frame, rows per thread, frames per stream step
    static constexpr int STREAMS = 4, FFT_THREADS = 256, STORE_THREADS = 128, THREADS = FFT_THREADS + STORE_THREADS;
    static constexpr int STEPS = 4, SF = STREAMS * FS, F = STEPS * SF, HF = F / 2;  // frames per step / tile / staging half
    static constexpr int FFT_REGS = 232, STORE_REGS = 40;
    static constexpr int SWB = sample_width(FMT == FMT_RUNTIME ? CF64 : FMT);
    static constexpr bool OK = (FMT != FMT_RUNTIME) && SWB <= 8;
    static constexpr int XP = 66;                                                // float2 per 64-point chunk (LDS.128 conflict-free)
    static constexpr int FP = C * XP;                                            // float2 per frame of the exchange buffer
    static constexpr int RAWP = N * SWB + 32;                                    // bytes per raw frame slot
    static constexpr int X_BYTES = (FS * FP * 8 > FS * RAWP ? FS * FP * 8 : FS * RAWP) + 15 & ~15;
    static constexpr int G = HF / 8;                                             // adjacent lanes of a store warp = adjacent 8-frame groups
    static constexpr int FPW = N / 4 + 2;                                        // staging words per frame
    static constexpr int HALF_WORDS = HF * FPW;
    static constexpr int TW_PITCH = 14;
    static constexpr size_t SMEM_BYTES = (size_t)STREAMS * X_BYTES + (size_t)2 * HALF_WORDS * 4 + (size_t)JH_SIZE * 4 + (size_t)N * 4
                                       + (size_t)C * TW_PITCH * 8 + 1024 /* LUT */ + (size_t)F * 8 /* s_mm */
                                       + (size_t)STREAMS * 2 * FS * 4 /* s_off */ + 128 + 1024 /* LUT alignment */;
};

// tw14: [C][14] float2 = W_N^{t*k}, k = 1..7, 8, 16, 24, 32, 40, 48, 56
template <int FMT>
__global__ void __launch_bounds__(384, 1) render_rc_kernel(const Params p, const float2 *__restrict__ tw14)
{
    using B = RcCfg<FMT>;
    constexpr int C = B::C, N = B::N, RPT = B::RPT, FS = B::FS, F = B::F, HF = B::HF;
    constexpr bool FLOAT_IN = FMT == CF32 || FMT == CF64 || FMT == FMT_RUNTIME;   // |X|^2 may be +inf / NaN
    extern __shared__ __align__(128) unsigned char smem_rc[];
    const unsigned lut_base = (smem_u32(smem_rc) + 1023u) & ~1023u;              // see render_r64_kernel
    unsigned char *s_x = smem_rc + (lut_base - smem_u32(smem_rc)) + 1024;        // [4][X_BYTES] exchange / raw frames
    unsigned *s_lut = reinterpret_cast<unsigned *>(s_x - 1024);                  // [256] RGBA indexed by the staged byte
    unsigned *s_stage = reinterpret_cast<unsigned *>(s_x + B::STREAMS * B::X_BYTES);   // [2][HF][FPW] colour bytes (4 bins per word)
    unsigned *s_jh = s_stage + 2 * B::HALF_WORDS;                                // [JH_SIZE] joint histogram
    float *s_win = reinterpret_cast<float *>(s_jh + JH_SIZE);                    // [C][64] (row t: window[C a + t] at (a + 4t) mod 64)
    float2 *s_tw = reinterpret_cast<float2 *>(s_win + N);                        // [C][14]
    uint2 *s_mm = reinterpret_cast<uint2 *>(s_tw + C * B::TW_PITCH);             // [F] per-frame min/max bit patterns of |X|^2
    uint64_t *s_mbar = reinterpret_cast<uint64_t *>(s_mm + F);                   // [4] raw frames landed
    uint64_t *s_full = s_mbar + B::STREAMS;                                      // [2] staging half holds HF finished frames
    uint64_t *s_empty = s_full + 2;                                              // [2] staging half has been stored
    int *s_off = reinterpret_cast<int *>(s_empty + 2);                           // [4][2][FS] misalignment of the staged frames

    const int tid = threadIdx.x;
    const int s = tid >> 6;                 // stream
    const int ts = tid & 63;                // thread of the stream
    const int fi = ts / C, t = ts % C;      // frame of the stream step, column
    unsigned char *xs = s_x + (size_t)s * B::X_BYTES;
    float2 *X = reinterpret_cast<float2 *>(xs) + fi * B::FP;                     // this frame's exchange area
    uint64_t *mbar = s_mbar + s;

    const JhConst jc = fused_prologue(p, s_jh, s_lut, tid, B::THREADS);
    for (int i = tid; i < C * B::TW_PITCH; i += B::THREADS) s_tw[i] = tw14[i];
    for (int i = tid; i < N; i += B::THREADS) s_win[(i % C) * 64 + (((i / C) + 4 * (i % C)) & 63)] = p.window[i];
    const unsigned jh_base = smem_u32(s_jh) - (JH_MAGIC_BITS << 2);
    const int nfull = p.n_full;

    // ts == 0 of a stream: start the bulk copies of the FS frames xr .. xr + FS - 1 (chunk relative) into the stream's buffer
    auto stage = [&](long long xr, unsigned par) {
        unsigned total = 0;
        const void *src[FS];
        unsigned bytes[FS];
#pragma unroll
        for (int i = 0; i < FS; i++) {
            const long long xc = xr + i < p.chunk_frames ? xr + i : p.chunk_frames - 1;   // partial last tile: redo the last frame
            const long long xgl = p.frame_first + p.chunk_first + xc;
            const long long p0 = (long long)__dadd_rn(0.5, __dmul_rn(p.stride, (double)xgl)) - p.sample_base;   // lib/worker.js:72
            const unsigned long long off = (unsigned long long)p0 * B::SWB, a0 = off & ~15ull;
            src[i] = p.buf + a0;
            bytes[i] = (unsigned)(((off - a0) + (unsigned long long)N * B::SWB + 15) & ~15ull);
            s_off[(s * 2 + par) * FS + i] = (int)(off - a0);
            total += bytes[i];
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(total) : "memory");
#pragma unroll
        for (int i = 0; i < FS; i++)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32(xs + i * B::RAWP)), "l"(src[i]), "r"(bytes[i]), "r"(smem_u32(mbar)) : "memory");
    };

    if (ts == 0 && tid < B::FFT_THREADS) mbar_init(mbar, 1);
    if (tid == 0) {
        for (int h = 0; h < 2; h++) { mbar_init(s_full + h, B::FFT_THREADS / 32); mbar_init(s_empty + h, B::STORE_THREADS / 32); }
    }
    if (ts == 0) asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    long long tile = blockIdx.x;
    unsigned kk = 0;                        // tiles done by this CTA (phase of the full / empty barriers)

    if (tid >= B::FFT_THREADS) {
        // ================= store warps: staged colour bytes -> LUT -> image rows (lib/worker.js:115-121) =================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(B::STORE_REGS));
        const int ht = tid - B::FFT_THREADS;
        const bool rows_aligned = (p.nframes % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.image) & 31) == 0);
        for (; tile < p.ntiles; tile += gridDim.x, kk++) {
            const long long xr0 = tile * F;
#pragma unroll 1
            for (int h = 0; h < 2; h++) {
                mbar_wait(s_full + h, kk & 1);
                const size_t x0 = (size_t)(p.chunk_first + xr0) + HF * h;
                const unsigned *half = s_stage + h * B::HALF_WORDS;
                if (p.waterfall) {
                    // waterfall layout (lib/worker.js:116): frame x is image row nframes - 1 - x, bin b is column (b + n/2 - 1) mod n.
                    // Item = (frame, m, o): o = tc*RPT + r runs over 64 consecutive bins, so the lanes of a store write
                    // consecutive columns (128 contiguous bytes); the staged word of (m, o) sits at m*64 + r*C + tc.
                    constexpr int MG = C / 4;                           // 64-bin groups per staged byte position
#pragma unroll 1
                    for (int i = 0; i < HF * MG * 64 / B::STORE_THREADS; i++) {
                        const int id = ht + B::STORE_THREADS * i, o = id & 63, rest = id >> 6;
                        const int m = rest % MG, fl = rest / MG;
                        if (xr0 + HF * h + fl >= p.chunk_frames) continue;               // partial last tile
                        const unsigned w = half[fl * B::FPW + m * 64 + (o % RPT) * C + o / RPT];
                        uint32_t *rowp = reinterpret_cast<uint32_t *>(p.image) + (size_t)N * (size_t)(p.nframes - 1 - (long long)(x0 + fl));
#pragma unroll
                        for (int j = 0; j < 4; j++) rowp[(o + 64 * (4 * m + j) + N / 2 - 1) & (N - 1)] = lut_at(lut_base, w, j);
                    }
                }
#pragma unroll 1
                for (int i = 0; i < (p.waterfall ? 0 : (HF / 8) * (N / 4) / B::STORE_THREADS); i++) {
                    // item = (8-frame group g, word w): word w = m*64 + r*C + tc holds bins (tc*RPT + r) + 64*(4m + j), j = 0..3
                    const int id = ht + B::STORE_THREADS * i;
                    const int g = id % B::G, rest = id / B::G;
                    const int wq = rest % (N / 4), g2 = rest / (N / 4);
                    const int grp = g2 * B::G + g;
                    const int tc = wq % C, r = (wq / C) % RPT, m = wq / 64;
                    if (xr0 + HF * h + 8 * grp >= p.chunk_frames) continue;       // partial last tile (chunk_frames % 8 == 0)
                    const unsigned *src = half + (8 * grp) * B::FPW + wq;
                    unsigned w[8];
#pragma unroll
                    for (int f = 0; f < 8; f++) w[f] = src[f * B::FPW];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const int bin = tc * RPT + r + 64 * (4 * m + j);
                        const int y = (nfull / 2 - bin) & (nfull - 1);                         // lib/worker.js:90
                        uint32_t *rowp = reinterpret_cast<uint32_t *>(p.image) + (size_t)p.nframes * (size_t)y + x0 + 8 * grp;   // :117
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
    // ================= FFT warps: four streams of FS frames each =================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(B::FFT_REGS));
    unsigned fpar = 0;                      // parity of this stream's step counter (mbarrier phase, s_off slot)
    if (ts == 0 && tile < p.ntiles) stage(tile * F + s * FS, 0);

    while (tile < p.ntiles) {
        const long long xr0 = tile * F;
        const long long next_tile = tile + gridDim.x;

#pragma unroll 1
        for (int step = 0; step < B::STEPS; step++) {
            const int fl = step * B::SF + s * FS + fi;                  // frame of the tile handled by this thread now
            const bool valid = xr0 + fl < p.chunk_frames;               // false: past the end of a partial last tile (outputs suppressed)
            const unsigned dump = smem_u32(s_jh + JH_SIZE - 1);         // histogram atomics of such frames land in an unused counter
            int half = step >> 1;                                       // staging half of this step
            asm volatile("" : "+r"(half));                              // (see render_r64_kernel: keeps nvcc from folding 8*(step >> 1))
            cf v[64];
            // ---------------- load + decode + window (lib/worker.js:70-75) ----------------
            mbar_wait(mbar, fpar);
            {
                const unsigned char *rp = xs + fi * B::RAWP + s_off[(s * 2 + fpar) * FS + fi];
#pragma unroll
                for (int a = 0; a < 64; a++) v[a] = decode_raw_cf<FMT>(rp, C * a + t, p.format);
                // raw sample at p0 + n/2 (lib/worker.js:131-133); the power-of-two scale is exact
                if (t == 0 && valid) p.fmid[p.chunk_first + xr0 + fl] = make_float2(cre(v[32]) * raw_scale<FMT>(), cim(v[32]) * raw_scale<FMT>());
                const float4 *wrow = reinterpret_cast<const float4 *>(s_win + t * 64);
#pragma unroll
                for (int q = 0; q < 16; q++) {
                    const float4 w = wrow[(q + t) & 15];
                    v[4 * q] = cscale(v[4 * q], w.x);         v[4 * q + 1] = cscale(v[4 * q + 1], w.y);
                    v[4 * q + 2] = cscale(v[4 * q + 2], w.z); v[4 * q + 3] = cscale(v[4 * q + 3], w.w);
                }
            }
            fpar ^= 1;

            // ---------------- pass A: DFT-64 over the slow input digit, twiddle W_N^{t*k0} ----------------
            dft64_between(v, [&] { stream_barrier(s); });               // every thread of the stream has consumed its raw frame
            {
                // each twiddled row goes straight to the 64-point chunk k0 / RPT (owner thread) at (k0 % RPT) * C + t: the
                // exchange stores ride between the twiddle products
                const float4 *twp = reinterpret_cast<const float4 *>(s_tw + t * B::TW_PITCH);
                float2 w[8], hi[8];                                     // w[j] = W^{t*j}, hi[i] = W^{t*8i}
                const float4 a = twp[0], b = twp[1], c = twp[2], d = twp[3], e = twp[4], f = twp[5], g = twp[6];
                w[1] = make_float2(a.x, a.y); w[2] = make_float2(a.z, a.w); w[3] = make_float2(b.x, b.y); w[4] = make_float2(b.z, b.w);
                w[5] = make_float2(c.x, c.y); w[6] = make_float2(c.z, c.w); w[7] = make_float2(d.x, d.y);
                hi[1] = make_float2(d.z, d.w); hi[2] = make_float2(e.x, e.y); hi[3] = make_float2(e.z, e.w); hi[4] = make_float2(f.x, f.y);
                hi[5] = make_float2(f.z, f.w); hi[6] = make_float2(g.x, g.y); hi[7] = make_float2(g.z, g.w);
#pragma unroll
                for (int j = 1; j < 8; j++) v[j] = cmul(v[j], w[j]);
#pragma unroll
                for (int k = 0; k < 8; k++) cst(X + (k / RPT) * B::XP + (k % RPT) * C + t, v[k]);
#pragma unroll
                for (int i = 1; i < 8; i++) {
                    v[8 * i] = cmul(v[8 * i], hi[i]);
#pragma unroll
                    for (int j = 1; j < 8; j++) v[8 * i + j] = cmul(v[8 * i + j], cun(cmul(cpk(hi[i]), w[j])));
#pragma unroll
                    for (int k = 8 * i; k < 8 * i + 8; k++) cst(X + (k / RPT) * B::XP + (k % RPT) * C + t, v[k]);
                }
            }
            stream_barrier(s);
            // ---------------- pass B: thread t owns rows t*RPT .. t*RPT + RPT - 1: RPT transforms of length C ----------------
            {
                const float4 *row = reinterpret_cast<const float4 *>(X + t * B::XP);
#pragma unroll
                for (int m = 0; m < 32; m++) {
                    const float4 q = row[m];
                    v[2 * m] = cpk(q.x, q.y); v[2 * m + 1] = cpk(q.z, q.w);
                }
            }
            stream_barrier(s);                                          // the exchange buffer is free: prefetch the stream's next frames
            if (ts == 0) {
                if (step < B::STEPS - 1) stage(xr0 + (step + 1) * B::SF + s * FS, fpar);
                else if (next_tile < p.ntiles) stage(next_tile * F + s * FS, fpar);
            }
            if ((step & 1) == 0) mbar_wait(s_empty + half, (kk + 1) & 1);   // the store warps are done with this staging half
#pragma unroll
            for (int r = 0; r < RPT; r++) {
                cf u[C];
#pragma unroll
                for (int i = 0; i < C; i++) u[i] = v[r * C + i];
                dft<C>(u);                                              // u[k1] is bin (t*RPT + r) + 64*k1
#pragma unroll
                for (int i = 0; i < C; i++) v[r * C + i] = u[i];
            }

            // ---------------- per-bin epilogue (lib/worker.js:85-122) ----------------
            BinMinMax<FLOAT_IN> bm;
            unsigned *stg = s_stage + half * B::HALF_WORDS + (fl - half * HF) * B::FPW + t;
#pragma unroll
            for (int r = 0; r < RPT; r++)
#pragma unroll
                for (int m = 0; m < C / 4; m++)     // bins (t*RPT + r) + 64*(4m .. 4m+3): four colour bytes in one word at m*64 + r*C + t
                    stg[m * 64 + r * C] = epilogue4(v + r * C + 4 * m, bm, jc, jh_base, valid, dump);
            unsigned umn = __reduce_min_sync(0xffffffffu, bm.lo()), umx = __reduce_max_sync(0xffffffffu, bm.hi());
            if (__any_sync(0xffffffffu, umn < 0x00800000u || umx >= 0x7f800000u))   // rare (warp-uniform)
                fixup_nonfinite(v, valid, (ts & 31) == 0, true, s_jh, jc, WarpMin(), WarpMax(), umn, umx);
            if (t == 0) s_mm[fl] = make_uint2(umn, umx);
            if (step & 1) {                 // this warp has staged its last frames of the half (and their s_mm entries)
                __syncwarp();
                if ((ts & 31) == 0) mbar_arrive(s_full + half);
            }
        } // steps
        tile = next_tile;
        kk++;
    } // tiles
    } // FFT warps

    __syncthreads();
    flush_joint_hist(p, s_jh, tid, B::THREADS);
}

} // namespace sp
