// sp_kernels.cuh — the fused render kernel: decode + window + FFT + dB + colormap + RGBA
// + histograms + per-frame min/max in ONE pass (replaces the hot loops of reference
// lib/worker.js:68-137 together with lib/samples.js:313-400 and lib/fft_nayuki.js:54-119).
//
// Work decomposition (N = FFT size):
//   * a "slot" of T = N/16 threads owns one frame at a time; each thread keeps 16 complex
//     points in registers.  The FFT is a decimation-in-frequency 16 x 16 x R transform
//     (1, 2 or 3 register passes) with shared-memory exchanges in padded, bank-conflict-free
//     layouts; twiddles are expanded from 4 table loads per pass.
//   * a slot renders 8 CONSECUTIVE frames and keeps their colour indices packed in registers
//     (16 bins x 8 bytes), so each image row is written as one aligned 32-byte segment
//     (2 x STG.128) — the transposed store of lib/worker.js:117 without a shared-memory tile.
//   * a CTA of 256 threads is persistent: it loops over tiles of 8*SLOTS frames and keeps the
//     two histograms in shared memory, flushing them to 64-bit global counters once.
#pragma once
#include "sp_device.cuh"

namespace sp {

struct Params {
    // input
    const uint8_t *buf;            // shard bytes; sample `sample_base` is at buf[0]
    unsigned long long valid_bytes;
    long long sample_base;
    int format;                    // runtime format (used by FMT_RUNTIME kernels and slow paths)
    int n_full;                    // FFT size of the message (n)
    double stride;                 // global fractional hop (lib/worker.js:50)
    long long frame_first;         // global index of local frame 0
    long long nframes;             // frames rendered by this launch (image width in pixels)
    const float *window;           // n_full fp32 coefficients (rounded once from double)
    const float4 *window_t;        // render_r64_kernel: the same coefficients as [16][64] float4, element (q, t) = w[64*(4q + i) + t], i = 0..3
    const float2 *twA;             // pass-A twiddles [15][T]:  W_N^{t*k},      k = 1..15 (N = kernel size, T = N/16)
    const float2 *twB;             // pass-B twiddles [15][RL]: W_{N/16}^{b*k}, k = 1..15 (3-pass sizes only)
    // dB / colour mapping
    float c0, c1;                  // d0 = c1 * log2(|X|^2) + c0
    float gn, gc, cmaxf;           // gray = trunc(0.5 + clamp(gn * d0 + gc, 0, cmax))
    int cmap_len;
    const uint32_t *lut;           // cmap_len packed RGBA words
    // output
    uint8_t *image;                // may be null
    int waterfall, channel_mode;
    float *fmin, *fmax;            // per local frame: min / max of d0 (reference init 0 / -200)
    float2 *fmid;                  // per local frame: raw mid sample (amp gauge)
    unsigned long long *cb_hist, *c_hist;
    float *db_out;                 // optional [nframes][n_full] d0 tap
    float2 *spec_out;              // optional [chunk frames][n_full] complex spectrum tap: the kernel stops after the FFT
                                   // (split-real for n_full > 4096 is finished by spectrum_epilogue_kernel)
    // sub-frame mode (n_full > kernel N): the kernel transforms n_full/sub_r point
    // sub-sequences produced by the radix-sub_r pre-pass; sub-frame (x, k0) yields the
    // bins k0 + sub_r*k'.  sub_r == 1 is the ordinary mode.
    int sub_r;
    const float2 *sub_in;          // [chunk frames][sub_r][N] complex, frame-major
    long long chunk_first;         // first local frame of this launch (multiple of 8)
    long long chunk_frames;        // frames rendered by this launch (== nframes when not chunked)
    long long ntiles;
    // joint (dB bin, colour index) histogram of render_r64_kernel (decoded by finalize_kernel)
    unsigned long long *j_hist;    // [JH_SIZE]
    float jA, jB, jC, jD;          // see jh_eval()
    int use_tma;                   // render_r64_kernel: image rows leave through tensor-TMA stores (width % 4 == 0, 16-byte aligned image)
    int dbg;                       // SP_DEBUG_SKIP bit mask (performance experiments only): 1 image stores, 4 LUT lookups (store warps of render_r64_kernel),
                                   // 16 no span staging in render_w_kernel (every frame copied on its own)
    unsigned long long *tile_ctr;  // render_r64_kernel: the launch's tile counter, zero at launch and left at zero by the launch
    unsigned long long *t_stamp;   // render_r64_kernel: %globaltimer at the start of CTA 0 goes to t_stamp[0] (null: not recorded)
};

// Programmatic dependent launch (render_r64_kernel, finalize_kernel).  wait: the grid this one was launched behind has completed
// and its memory operations are visible (returns at once without such a grid).  launch_dependents: the next grid of the stream,
// launched with cudaLaunchAttributeProgrammaticStreamSerialization, may start once every CTA of this grid has executed it or exited.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

template <int LOG2N> struct Cfg {
    static constexpr int N = 1 << LOG2N;
    static constexpr int P = N >= 16 ? 16 : N;          // points per thread
    static constexpr int T = N / P;                     // threads per frame
    static constexpr int PASSES = LOG2N <= 4 ? 1 : (LOG2N <= 8 ? 2 : 3);
    static constexpr int RL = PASSES == 1 ? P : (PASSES == 2 ? N / 16 : N / 256);   // last radix
    static constexpr int NB = P / RL;                   // butterflies per thread in the last pass
    static constexpr int THREADS = 256;
    static constexpr int SLOTS = THREADS / T;
    static constexpr int FRAMES_PER_SLOT = 8;
    static constexpr int TILE = SLOTS * FRAMES_PER_SLOT;
    // exchange layouts in float2 units (see DESIGN.md "shared-memory layouts")
    static constexpr int N1 = N / 16;
    static constexpr int PITCH_A = PASSES == 3 ? N1 + (RL % 16) : (T + 1);
    static constexpr int SIZE_A = PASSES >= 2 ? 16 * PITCH_A + (PASSES == 2 ? 1 : 0) : 0;
    static constexpr int P1 = RL + 1;
    static constexpr int PITCH_B = 16 * P1 + (RL % 16);
    static constexpr int SIZE_B = PASSES == 3 ? 16 * PITCH_B : 0;
    static constexpr int WPS = T > 32 ? T / 32 : 1;     // warps per slot
    static constexpr int SMEM_X = SLOTS * (SIZE_A + SIZE_B) > N * SLOTS ? SLOTS * (SIZE_A + SIZE_B) : N * SLOTS;
};

constexpr int CB_BINS = 1000;     // lib/worker.js:41
// Shared-memory dB histogram is indexed by the RAW saturating conversion r = u32(2.5 - 10*d0):
//   r == 0            d0 > +0.15 dB: the reference's negative index, not counted   (lib/worker.js:106)
//   r == 1, 2         bin 0        (~~ truncates toward zero: (-1, 1) -> 0)
//   3 <= r <= 1001    bin r - 2
//   1002 <= r < CAP   bin 999      (cBabs >= 1000)
//   r == CAP          d0 == -inf (|X|^2 == 0): ~~(+Infinity) == 0 -> bin 0
// so the per-pixel work is FFMA + F2I + IMNMX + ATOMS with no compare / select; the mapping is
// applied once per CTA when the counters are flushed.  The engine rejects block_norm so small that a
// finite d0 could reach CAP (10*log10(block_norm) < -75 dB).
constexpr int CB_RAW_CAP = 3071;
constexpr int CB_RAW = CB_RAW_CAP + 1;

__host__ __device__ inline size_t main_smem_bytes(int smem_x_float2, int cmap_len, int twb_float2)
{
    return (size_t)smem_x_float2 * 8 + (size_t)CB_RAW * 4 + (size_t)cmap_len * 8 + 64 * 8 + (size_t)twb_float2 * 8;
}

// ---------------------------------------------------------------------------------------------
// Joint histogram (render_r64_kernel).  Per pixel, with l2 = log2|X|^2 and d0 = c1*l2 + c0 (= dBfs - gain):
//   r  = RN(sat(jA*l2 + jB) * RCAP),  jA*l2 + jB = (2.0 - 10*d0) / RCAP   : RN(x - 0.5) == trunc(x) for the
//        x = 2.5 - 10*d0 of the table above (off quantisation ties), saturating at 0 and RCAP = 1003
//   g' = RN(sat(jC*l2 + jD) * cmax) subtracted from cmax (as is when range < 0), jC*l2 + jD = (cmax - (d0 + gain)*color_norm) / cmax
//        (lib/worker.js:111-112: the colour index g = cmax - g', clamped by the saturation)
// Both roundings are done by adding 2^23 inside an FFMA, so S = 2^23 + r + g' and Y = 2^23 + g' come out of
// four FMA-pipe instructions with no F2I and no integer clamp.  r falls and g rises with l2, so j = r + g'
// is monotone and (r, g') is a function of j: ONE shared-memory atomic per pixel.  jh_decode() inverts j
// by bisection over the ordered floats with the SAME jh_eval().  Non-finite pixels (|X|^2 flushed to 0,
// +inf, NaN) take the ordinary path and are corrected per frame through two extra counters:
//   JH_ZERO  pixels with d0 = -inf: counted as r = RCAP (bin 999) -> move them to bin 0  (~~(+Infinity) == 0)
//   JH_BAD   pixels with d0 = +inf or NaN: counted as r = 0 (dropped) -> add them to bin 0
//   JH_NAN   NaN pixels: sat(NaN) = 0 gives them the joint index of some ordinary level; the kernel takes them out of that
//            counter again and counts them here -> colour index 0 (the dB bin comes from JH_BAD)
// ---------------------------------------------------------------------------------------------
constexpr int JH_RCAP = 1003;
constexpr int JH_BINS = JH_RCAP + 1 + 256;
constexpr int JH_ZERO = JH_BINS, JH_BAD = JH_BINS + 1, JH_NAN = JH_BINS + 2, JH_SIZE = JH_BINS + 4;
constexpr unsigned JH_MAGIC_BITS = 0x4B000000u;       // 2^23

struct JhConst { float A, B, C, D, rcap, ncmax, ymagic; int rev; };
__host__ __device__ __forceinline__ JhConst jh_const(const Params &p)
{
    JhConst c;
    c.A = p.jA; c.B = p.jB; c.C = p.jC; c.D = p.jD;
    c.rcap = (float)JH_RCAP;
    // the second term must fall with l2 like r does: cmax - g when the colour index rises with the level (range > 0),
    // g itself when it falls (range < 0)
    c.rev = p.jC >= 0.0f;
    c.ncmax = c.rev ? -(float)(p.cmap_len - 1) : (float)(p.cmap_len - 1);
    c.ymagic = (c.rev ? (float)(p.cmap_len - 1) : 0.0f) + 8388608.0f;
    return c;
}
// returns S = 2^23 + r + g'; Y = 2^23 + g'
__device__ __forceinline__ float jh_eval(float l2, const JhConst &c, float &Y)
{
    const float kx = __saturatef(fmaf(l2, c.A, c.B));
    const float ky = __saturatef(fmaf(l2, c.C, c.D));
    Y = fmaf(ky, c.ncmax, c.ymagic);
    return fmaf(kx, c.rcap, Y);
}

__device__ __forceinline__ int cb_bin_of_raw(int r)
{
    return r == 0 ? -1 : (r <= 2 ? 0 : (r <= 1001 ? r - 2 : (r < CB_RAW_CAP ? CB_BINS - 1 : 0)));
}

// first output bin of butterfly j of thread t in the last pass (bin = kbase + kstep * k)
template <class C> __device__ __forceinline__ int kbase_of(int t, int j)
{
    if constexpr (C::PASSES == 1) return 0;
    else if constexpr (C::PASSES == 2) return t + C::T * j;
    else { const int q = t + C::T * j; return (q / 16) + 16 * (q % 16); }
}

// order-preserving float <-> uint mapping for atomic min / max on floats
__device__ __forceinline__ unsigned f2ord(float f)
{
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u)
{
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// joint index j -> (dB bin or -1, colour index); false when no log2|X|^2 maps to j
__device__ inline bool jh_decode(int j, const JhConst &c, int cmax, int &bin, int &g)
{
    unsigned lo = f2ord(__int_as_float(0xff800000)), hi = f2ord(__int_as_float(0x7f800000));   // -inf .. +inf, no NaN between
    float Y;
    while (lo < hi) {                                  // smallest l2 with J(l2) <= j (J is non-increasing)
        const unsigned mid = lo + (hi - lo) / 2;
        const int J = (int)(__float_as_uint(jh_eval(ord2f(mid), c, Y)) - JH_MAGIC_BITS);
        if (J <= j) hi = mid; else lo = mid + 1;
    }
    const int J = (int)(__float_as_uint(jh_eval(ord2f(lo), c, Y)) - JH_MAGIC_BITS);
    const int gp = (int)(__float_as_uint(Y) - JH_MAGIC_BITS);
    const int r = J - gp;
    g = c.rev ? cmax - gp : gp;
    bin = r == 0 ? -1 : (r <= 2 ? 0 : (r <= 1001 ? r - 2 : CB_BINS - 1));
    return J == j;
}

// shared-memory counters -> 64-bit global histograms (raw dB index mapped to the reference's bins)
__device__ __forceinline__ void flush_hist(unsigned *s_cb, uint2 *s_col, const Params &p, int tid, int nthreads, bool clear)
{
    for (int i = tid; i < CB_RAW; i += nthreads) {
        const unsigned c = s_cb[i];
        if (c) {
            const int b = cb_bin_of_raw(i);
            if (b >= 0) atomicAdd(&p.cb_hist[b], (unsigned long long)c);
            if (clear) s_cb[i] = 0;
        }
    }
    for (int i = tid; i < p.cmap_len; i += nthreads) {
        const unsigned c = s_col[i].y;
        if (c) {
            atomicAdd(&p.c_hist[i], (unsigned long long)c);
            if (clear) s_col[i].y = 0;
        }
    }
}

template <int LOG2N, int FMT>
__global__ void __launch_bounds__(256, 2) render_kernel(const Params p)
{
    using C = Cfg<LOG2N>;
    constexpr int N = C::N, P = C::P, T = C::T;
    constexpr int kstep = C::PASSES == 1 ? 1 : (C::PASSES == 2 ? 16 : 256);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2 *xbuf = reinterpret_cast<float2 *>(smem_raw);
    unsigned *s_cb = reinterpret_cast<unsigned *>(xbuf + C::SMEM_X);           // [CB_RAW] raw dB histogram
    uint2 *s_col = reinterpret_cast<uint2 *>(s_cb + CB_RAW);                    // [cmap_len] {RGBA, count}
    float2 *s_mm = reinterpret_cast<float2 *>(s_col + p.cmap_len);              // [64] per-warp min/max partials
    float2 *s_twB = s_mm + 64;                                                  // [15][RL] pass-B twiddles

    const int tid = threadIdx.x;
    const int slot = tid / T;
    const int t = tid % T;
    float2 *bufA = xbuf + slot * (C::SIZE_A + C::SIZE_B);
    float2 *bufB = bufA + C::SIZE_A;
    (void)bufA; (void)bufB;

    for (int i = tid; i < CB_RAW; i += C::THREADS) s_cb[i] = 0;
    for (int i = tid; i < p.cmap_len; i += C::THREADS) s_col[i] = make_uint2(p.lut[i], 0u);
    if constexpr (C::PASSES == 3)
        for (int i = tid; i < 15 * C::RL; i += C::THREADS) s_twB[i] = p.twB[i];
    const unsigned cmax_u = (unsigned)(p.cmap_len - 1);
    const float gc5 = p.gc + 0.5f;
    const float l2c_k = -10.0f * p.c1, l2c_k0 = fmaf(-10.0f, p.c0, 2.5f);       // raw cB index = l2c_k * log2|X|^2 + l2c_k0
    const float l2c_g = p.gn * p.c1, l2c_g0 = fmaf(p.gn, p.c0, gc5);             // colour index  = l2c_g * log2|X|^2 + l2c_g0
    const cf l2c_kg = cpk(l2c_k, l2c_g), l2c_kg0 = cpk(l2c_k0, l2c_g0);

    const bool sub = p.sub_r > 1;
    const int nfull = p.n_full;
    const int sub_r = p.sub_r;

    // thread-invariant window coefficients (element T*a + t of the frame); ones in sub-frame mode
    float win[P];
#pragma unroll
    for (int a = 0; a < P; a++) win[a] = sub ? 1.0f : p.window[T * a + t];
    int kbase[C::NB];
#pragma unroll
    for (int j = 0; j < C::NB; j++) kbase[j] = kbase_of<C>(t, j);

    const bool wide_rows = !p.waterfall && p.image && p.cmap_len <= 256 && (p.nframes % 4 == 0)
                           && ((reinterpret_cast<uintptr_t>(p.image) & 15) == 0);
    const bool direct = p.image && !wide_rows;     // per-pixel 4-byte stores
    unsigned long long px_since_flush = 0;
    __syncthreads();

    for (long long tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        // tile -> (first chunk-relative frame of this slot, sub-sequence index)
        long long xg; int k0sub = 0;
        if (sub) { k0sub = (int)(tile % sub_r); xg = tile / sub_r; } else xg = tile;
        const long long xr0 = xg * C::TILE + (long long)slot * C::FRAMES_PER_SLOT;   // chunk relative
        unsigned glo[P], ghi[P];
#pragma unroll
        for (int i = 0; i < P; i++) { glo[i] = 0; ghi[i] = 0; }

#pragma unroll 1
        for (int f = 0; f < C::FRAMES_PER_SLOT; f++) {
            const bool active = xr0 + f < p.chunk_frames;
            const long long xr = active ? xr0 + f : p.chunk_frames - 1;   // inactive slots redo the last frame
            const long long xl = p.chunk_first + xr;                      // local frame == image column
            cf v[P];
            bool ragged = false;                                          // frame reads past the end of the buffer
            // two-pass sizes (N <= 256): a slot's T <= 16 threads sit in one warp and the only barrier of a frame is the one
            // between the pass-A writes and the last-pass reads of bufA; order this frame's writes after the previous
            // frame's reads explicitly (compute-sanitizer racecheck flagged the intra-warp write-after-read)
            if constexpr (C::PASSES == 2) __syncwarp();
            // ---------------- load + decode + window (lib/worker.js:70-75) ----------------
            if (sub) {
                const float2 *src = p.sub_in + ((size_t)xr * sub_r + k0sub) * N;
#pragma unroll
                for (int a = 0; a < P; a++) v[a] = cld(src + T * a + t);
            } else {
                const long long xgl = p.frame_first + xl;
                // ~~(0.5 + stride * x): separate multiply and add like JavaScript (no FMA)
                const long long p0 = (long long)__dadd_rn(0.5, __dmul_rn(p.stride, (double)xgl)) - p.sample_base;
                const bool inside = p0 >= 0 &&
                    (unsigned long long)(p0 + N) * (unsigned)sample_width(FMT == FMT_RUNTIME ? p.format : FMT) <= p.valid_bytes;
                if (inside) {
#pragma unroll
                    for (int a = 0; a < P; a++) v[a] = cpk(decode_raw<FMT>(p.buf, p0 + T * a + t, p.format));
                } else {                                       // slow path: frames touching a ragged buffer end
                    ragged = true;
                    const float inv = 1.0f / raw_scale<FMT>();
#pragma unroll
                    for (int a = 0; a < P; a++) {
                        const float2 d = decode_checked(p.buf, p0 + T * a + t, p.format, p.valid_bytes);
                        v[a] = cpk(d.x * inv, d.y * inv);
                    }
                }
                // raw sample at p0 + n/2 (lib/worker.js:131-133); the power-of-two scale is exact
                if (t == 0 && active) p.fmid[xl] = make_float2(cre(v[P / 2]) * raw_scale<FMT>(), cim(v[P / 2]) * raw_scale<FMT>());
#pragma unroll
                for (int a = 0; a < P; a++) v[a] = cscale(v[a], win[a]);
            }

            // ---------------- FFT pass A: radix P over the slowest input digit ----------------
            dft<P>(v);
            if constexpr (C::PASSES >= 2) {
#pragma unroll
                for (int k = 1; k < 16; k++) v[k] = cmul(v[k], __ldg(p.twA + (k - 1) * T + t));   // W_N^{t*k}
#pragma unroll
                for (int k = 0; k < 16; k++) cst(&bufA[k * C::PITCH_A + t], v[k]);
                __syncthreads();
            }
            if constexpr (C::PASSES == 3) {
                // ------------ pass B: thread <-> (k0, b1), radix 16 over a1 ------------
                constexpr int R2 = C::RL;
                const int k0 = t / R2, b1 = t % R2;
#pragma unroll
                for (int a = 0; a < 16; a++) v[a] = cld(&bufA[k0 * C::PITCH_A + R2 * a + b1]);
                dft<16>(v);
#pragma unroll
                for (int k = 1; k < 16; k++) v[k] = cmul(v[k], s_twB[(k - 1) * R2 + b1]);         // W_{N/16}^{b1*k}
#pragma unroll
                for (int k = 0; k < 16; k++) cst(&bufB[k0 * C::PITCH_B + k * C::P1 + b1], v[k]);
                __syncthreads();
            }
            // ---------------- last pass: NB radix-RL butterflies; v[j*RL + k] is bin kbase[j] + kstep*k ------
            if constexpr (C::PASSES == 2) {
#pragma unroll
                for (int j = 0; j < C::NB; j++) {
                    const int k0 = t + T * j;
                    cf u[C::RL];
#pragma unroll
                    for (int b = 0; b < C::RL; b++) u[b] = cld(&bufA[k0 * C::PITCH_A + b]);
                    dft<C::RL>(u);
#pragma unroll
                    for (int b = 0; b < C::RL; b++) v[j * C::RL + b] = u[b];
                }
            } else if constexpr (C::PASSES == 3) {
#pragma unroll
                for (int j = 0; j < C::NB; j++) {
                    const int q = t + T * j, k1 = q % 16, k0 = q / 16;
                    cf u[C::RL];
#pragma unroll
                    for (int b = 0; b < C::RL; b++) u[b] = cld(&bufB[k0 * C::PITCH_B + k1 * C::P1 + b]);
                    dft<C::RL>(u);
#pragma unroll
                    for (int b = 0; b < C::RL; b++) v[j * C::RL + b] = u[b];
                }
            }

            // ---------------- optional spectrum tap: hand the bins to spectrum_epilogue_kernel ----------------
            if (p.spec_out) {
                if (active) {
#pragma unroll
                    for (int j = 0; j < C::NB; j++)
#pragma unroll
                        for (int k = 0; k < C::RL; k++) {
                            const int kk = kbase[j] + kstep * k;
                            cst(p.spec_out + (size_t)xr * nfull + (sub ? k0sub + sub_r * kk : kk), v[j * C::RL + k]);
                        }
                }
                continue;
            }

            // ---------------- optional split-real post-process (lib/fft_nayuki.js:103-119) ----------------
            if (p.channel_mode) {
                // (the engine never combines channel mode with sub-frame mode, see sp_engine.cu)
                __syncthreads();                               // everyone is done reading bufA / bufB
                float2 *X = xbuf + slot * N;
#pragma unroll
                for (int j = 0; j < C::NB; j++)
#pragma unroll
                    for (int k = 0; k < C::RL; k++) cst(&X[kbase[j] + kstep * k], v[j * C::RL + k]);
                __syncthreads();
#pragma unroll
                for (int j = 0; j < C::NB; j++)
#pragma unroll
                    for (int k = 0; k < C::RL; k++) {
                        const int bin = kbase[j] + kstep * k;
                        const float2 a = cun(v[j * C::RL + k]);
                        const float2 b = X[(N - bin) & (N - 1)];
                        float2 r;
                        if (bin == 0) r = make_float2(fmaf(0.0f, a.y, a.x), 0.f); // a NaN in imag[0] reaches real[0] in the reference (its butterflies multiply by every twiddle, NaN * 0 = NaN): keep that
                        else if (bin == N / 2) r = make_float2(0.f, 0.f);
                        else if (bin < N / 2) r = make_float2(0.5f * (a.x + b.x), 0.5f * (a.y - b.y));
                        else r = make_float2(0.5f * (b.y + a.y), 0.5f * (-b.x + a.x));
                        v[j * C::RL + k] = cpk(r);
                    }
                __syncthreads();                               // X aliases the exchange buffers
            }

            // ---------------- per-bin epilogue (lib/worker.js:85-122) ----------------
            // min / max are tracked on |X|^2 (log2 and the FMA are monotone), converted once per thread
            float amin = __int_as_float(0x7f800000), amax = 0.0f;
            float vabs[P / 2 > 0 ? P / 2 : 1];
#pragma unroll
            for (int i = 0; i < P; i++) {
                const float2 vi = cun(v[i]);
                const float abs2 = fmaf(vi.x, vi.x, vi.y * vi.y);
                if (i & 1) {                                 // 3-input min / max (NaN never wins, like `<` in JS)
                    const float prev = vabs[i >> 1];
                    amin = fmin3(amin, prev, abs2);
                    amax = fmax3(amax, prev, abs2);
                } else vabs[i >> 1] = abs2;
                const float l2 = fast_log2(abs2);                              // dBfs - gain = c1*l2 + c0 (lib/worker.js:93)
                // saturating float->uint conversions do the clamping: negative / NaN -> 0, +inf -> max
                const float2 kg = cun(cfma2(cpk(l2, l2), l2c_kg, l2c_kg0));     // one FFMA2: (raw cB index, colour index)
                const float kf = kg.x;
                unsigned cr = min(__float2uint_rz(kf), (unsigned)CB_RAW_CAP);                             // :105-106
                if ((FMT == CF32 || FMT == CF64 || FMT == FMT_RUNTIME) || ragged)
                    if (!(fabsf(kf) <= 3.0e9f)) cr = 1;     // NaN / -inf (float input, or `undefined` past a ragged end): ~~v == 0 -> bin 0
                const unsigned g = min(__float2uint_rz(kg.y), cmax_u);                                    // :111-112
                if (active) {
                    atomicAdd(&s_cb[cr], 1u);
                    atomicAdd(&s_col[g].y, 1u);                             // :113
                }
                // byte f of (ghi:glo) = colour index of frame f of this slot
                glo[i] = __funnelshift_r(glo[i], ghi[i], 8);
                ghi[i] = __funnelshift_r(ghi[i], g, 8);
            }
            float mn = fminf(0.0f, fmaf(fast_log2(amin), p.c1, p.c0));        // lib/worker.js:82,102
            float mx = fmaxf(-200.0f, fmaf(fast_log2(amax), p.c1, p.c0));     // lib/worker.js:83,103

            // slow outputs (uniform branch, once per frame): per-pixel stores and the dB tap
            if ((direct | (p.db_out != nullptr)) && active) {
#pragma unroll 1
                for (int j = 0; j < C::NB; j++)
#pragma unroll 1
                    for (int k = 0; k < C::RL; k++) {
                        const int i = j * C::RL + k;
                        cf vsel = v[0];
#pragma unroll
                        for (int q = 0; q < P; q++) if (q == i) vsel = v[q];   // register select, no local memory
                        const float2 vi = cun(vsel);
                        const int kb = kbase_of<C>(t, j);
                        const int bin = sub ? k0sub + sub_r * (kb + kstep * k) : kb + kstep * k;
                        const float abs2 = fmaf(vi.x, vi.x, vi.y * vi.y);
                        const float d0 = fmaf(fast_log2(abs2), p.c1, p.c0);
                        const unsigned gi = min(__float2uint_rz(fmaf(fast_log2(abs2), l2c_g, l2c_g0)), cmax_u);   // (cmap_len may exceed 256)
                        if (p.db_out) p.db_out[(size_t)xl * nfull + bin] = d0;
                        if (direct) {
                            const int y = (nfull / 2 - bin) & (nfull - 1);                     // lib/worker.js:90
                            const size_t px = p.waterfall
                                ? (size_t)nfull * (size_t)(p.nframes - 1 - xl) + (size_t)(nfull - 1 - y)   // :116
                                : (size_t)xl + (size_t)p.nframes * (size_t)y;                              // :117
                            reinterpret_cast<uint32_t *>(p.image)[px] = s_col[gi].x;
                        }
                    }
            }

            // ---------------- per-frame min / max (lib/worker.js:102-103) ----------------
#pragma unroll
            for (int off = (T < 32 ? T : 32) / 2; off > 0; off >>= 1) {
                mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            }
            if constexpr (T <= 32) {
                if (t == 0 && active) {
                    if (sub) {
                        atomicMin(reinterpret_cast<unsigned *>(p.fmin) + xl, f2ord(mn));
                        atomicMax(reinterpret_cast<unsigned *>(p.fmax) + xl, f2ord(mx));
                    } else { p.fmin[xl] = mn; p.fmax[xl] = mx; }
                }
            } else {
                if ((t & 31) == 0) s_mm[(slot * C::FRAMES_PER_SLOT + f) * C::WPS + t / 32] = make_float2(mn, mx);
            }
        } // frames of the slot

        // ---------------- row stores: 8 frames x 4 bytes = one 32-byte segment per bin ----------------
        if (wide_rows && xr0 < p.chunk_frames) {
            const bool full8 = xr0 + 8 <= p.chunk_frames;
            const size_t x0 = (size_t)(p.chunk_first + xr0);
#pragma unroll
            for (int j = 0; j < C::NB; j++)
#pragma unroll
                for (int k = 0; k < C::RL; k++) {
                    const int i = j * C::RL + k;
                    const int bin = sub ? k0sub + sub_r * (kbase[j] + kstep * k) : kbase[j] + kstep * k;
                    const int y = (nfull / 2 - bin) & (nfull - 1);
                    uint32_t *row = reinterpret_cast<uint32_t *>(p.image) + (size_t)p.nframes * (size_t)y + x0;
                    uint4 a, b;
                    a.x = s_col[glo[i] & 255].x; a.y = s_col[(glo[i] >> 8) & 255].x;
                    a.z = s_col[(glo[i] >> 16) & 255].x; a.w = s_col[glo[i] >> 24].x;
                    reinterpret_cast<uint4 *>(row)[0] = a;
                    if (full8) {                               // else nframes % 4 == 0: exactly 4 frames left
                        b.x = s_col[ghi[i] & 255].x; b.y = s_col[(ghi[i] >> 8) & 255].x;
                        b.z = s_col[(ghi[i] >> 16) & 255].x; b.w = s_col[ghi[i] >> 24].x;
                        reinterpret_cast<uint4 *>(row)[1] = b;
                    }
                }
        }

        // ---------------- per-frame min/max across the warps of a slot ----------------
        if constexpr (T > 32) {
            __syncthreads();
            if (tid < C::SLOTS * C::FRAMES_PER_SLOT && !p.spec_out) {
                const int s = tid / C::FRAMES_PER_SLOT, f = tid % C::FRAMES_PER_SLOT;
                const long long xr = xg * C::TILE + (long long)s * C::FRAMES_PER_SLOT + f;
                if (xr < p.chunk_frames) {
                    const long long xl = p.chunk_first + xr;
                    float mn = 0.0f, mx = -200.0f;
                    for (int w = 0; w < C::WPS; w++) {
                        const float2 m = s_mm[(s * C::FRAMES_PER_SLOT + f) * C::WPS + w];
                        mn = fminf(mn, m.x); mx = fmaxf(mx, m.y);
                    }
                    if (sub) {
                        atomicMin(reinterpret_cast<unsigned *>(p.fmin) + xl, f2ord(mn));
                        atomicMax(reinterpret_cast<unsigned *>(p.fmax) + xl, f2ord(mx));
                    } else { p.fmin[xl] = mn; p.fmax[xl] = mx; }
                }
            }
            // s_mm is next written after the __syncthreads of the next tile's first frame
        }

        // keep the 32-bit shared counters from wrapping on very long captures
        px_since_flush += (unsigned long long)C::TILE * N;
        if (px_since_flush >= (1ull << 31)) {
            __syncthreads();
            flush_hist(s_cb, s_col, p, tid, C::THREADS, true);
            px_since_flush = 0;
            __syncthreads();
        }
    } // tiles

    __syncthreads();
    flush_hist(s_cb, s_col, p, tid, C::THREADS, false);
}

// ---------------------------------------------------------------------------------------------
// Radix-R pre-pass for n_full = R * 4096 (R = 2, 4, 8, 16): decode + window + DFT_R over the
// slowest input digit + twiddle W_n^{b*k0}; writes R sub-sequences of 4096 points per frame,
// which render_kernel<12> then transforms in sub-frame mode (four-step FFT, scratch kept
// L2-resident by chunking the frames).
// ---------------------------------------------------------------------------------------------
template <int R, int FMT>
__global__ void __launch_bounds__(256) prepass_kernel(const Params p, float2 *__restrict__ out, const float2 *__restrict__ tw_full)
{
    constexpr int NS = 4096;
    const long long gid = (long long)blockIdx.x * 256 + threadIdx.x;
    const long long xr = gid / NS;                 // chunk-relative frame
    const int b = (int)(gid % NS);
    if (xr >= p.chunk_frames) return;
    const long long xl = p.chunk_first + xr;
    const long long xgl = p.frame_first + xl;
    const long long p0 = (long long)__dadd_rn(0.5, __dmul_rn(p.stride, (double)xgl)) - p.sample_base;
    const bool inside = p0 >= 0 &&
        (unsigned long long)(p0 + (long long)R * NS) * (unsigned)sample_width(FMT == FMT_RUNTIME ? p.format : FMT) <= p.valid_bytes;
    cf v[R];
    if (inside) {
#pragma unroll
        for (int a = 0; a < R; a++) v[a] = cpk(decode_raw<FMT>(p.buf, p0 + NS * a + b, p.format));
    } else {
        const float inv = 1.0f / raw_scale<FMT>();
#pragma unroll
        for (int a = 0; a < R; a++) {
            const float2 d = decode_checked(p.buf, p0 + NS * a + b, p.format, p.valid_bytes);
            v[a] = cpk(d.x * inv, d.y * inv);
        }
    }
    if (b == 0) p.fmid[xl] = make_float2(cre(v[R / 2]) * raw_scale<FMT>(), cim(v[R / 2]) * raw_scale<FMT>());   // sample p0 + n/2
#pragma unroll
    for (int a = 0; a < R; a++) v[a] = cscale(v[a], p.window[NS * a + b]);
    dft<R>(v);
#pragma unroll
    for (int k = 1; k < R; k++) v[k] = cmul(v[k], tw_full[b * k]);
    float2 *dst = out + (size_t)xr * R * NS + b;
#pragma unroll
    for (int k = 0; k < R; k++) cst(dst + (size_t)k * NS, v[k]);
}

// ---------------------------------------------------------------------------------------------
// Per-bin epilogue over a complex spectrum held in global memory (one thread per bin): optional
// split-real (lib/fft_nayuki.js:103-119), then dB, histograms, colour, pixel, per-frame min / max
// exactly as render_kernel does them (lib/worker.js:85-125).  Used where the post-process needs
// bins of different sub-sequences of the four-step FFT together: channelMode with n > 4096.
// p.fmin / p.fmax hold order-preserving uints (init_minmax_kernel), as in sub-frame mode.
// ---------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256) spectrum_epilogue_kernel(const Params p, const float2 *__restrict__ spec)
{
    extern __shared__ unsigned s_epi[];
    unsigned *s_cb = s_epi, *s_cnt = s_epi + CB_RAW;
    for (int i = threadIdx.x; i < CB_RAW + p.cmap_len; i += 256) s_epi[i] = 0;
    __syncthreads();
    const int n = p.n_full, per_frame = n / 256;
    const unsigned cmax_u = (unsigned)(p.cmap_len - 1);
    const float gc5 = p.gc + 0.5f;
    const float l2c_k = -10.0f * p.c1, l2c_k0 = fmaf(-10.0f, p.c0, 2.5f);
    const float l2c_g = p.gn * p.c1, l2c_g0 = fmaf(p.gn, p.c0, gc5);
    const long long total = p.chunk_frames * per_frame;
    for (long long tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const long long xr = tile / per_frame, xl = p.chunk_first + xr;
        const int bin = (int)(tile % per_frame) * 256 + threadIdx.x;
        const float2 *X = spec + (size_t)xr * n;
        float2 r = X[bin];
        if (p.channel_mode) {
            const float2 a = r, b = X[(n - bin) & (n - 1)];
            if (bin == 0) r = make_float2(fmaf(0.0f, a.y, a.x), 0.f); // a NaN in imag[0] reaches real[0] in the reference (its butterflies multiply by every twiddle, NaN * 0 = NaN): keep that
            else if (bin == n / 2) r = make_float2(0.f, 0.f);
            else if (bin < n / 2) r = make_float2(0.5f * (a.x + b.x), 0.5f * (a.y - b.y));
            else r = make_float2(0.5f * (b.y + a.y), 0.5f * (-b.x + a.x));
        }
        const float abs2 = fmaf(r.x, r.x, r.y * r.y);
        const float l2 = fast_log2(abs2);
        const float d0 = fmaf(l2, p.c1, p.c0);
        const float kf = fmaf(l2, l2c_k, l2c_k0);
        unsigned cr = min(__float2uint_rz(kf), (unsigned)CB_RAW_CAP);
        if (!(fabsf(kf) <= 3.0e9f)) cr = 1;                                      // NaN / -inf -> bin 0
        const unsigned g = min(__float2uint_rz(fmaf(l2, l2c_g, l2c_g0)), cmax_u);
        atomicAdd(&s_cb[cr], 1u);
        atomicAdd(&s_cnt[g], 1u);
        if (p.db_out) p.db_out[(size_t)xl * n + bin] = d0;
        if (p.image) {
            const int y = (n / 2 - bin) & (n - 1);                                // lib/worker.js:90
            const size_t px = p.waterfall ? (size_t)n * (size_t)(p.nframes - 1 - xl) + (size_t)(n - 1 - y)   // :116
                                          : (size_t)xl + (size_t)p.nframes * (size_t)y;                      // :117
            reinterpret_cast<uint32_t *>(p.image)[px] = p.lut[g];
        }
        float mn = fminf(0.0f, d0), mx = fmaxf(-200.0f, d0);                      // NaN never wins (lib/worker.js:102-103)
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(reinterpret_cast<unsigned *>(p.fmin) + xl, f2ord(mn));
            atomicMax(reinterpret_cast<unsigned *>(p.fmax) + xl, f2ord(mx));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < CB_RAW; i += 256) {
        const unsigned c = s_cb[i];
        if (c) {
            const int b = cb_bin_of_raw(i);
            if (b >= 0) atomicAdd(&p.cb_hist[b], (unsigned long long)c);
        }
    }
    for (int i = threadIdx.x; i < p.cmap_len; i += 256)
        if (s_cnt[i]) atomicAdd(&p.c_hist[i], (unsigned long long)s_cnt[i]);
}

} // namespace sp
