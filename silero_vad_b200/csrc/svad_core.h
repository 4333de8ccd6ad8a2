// svad_core.h -- per-thread arithmetic of the fused fp32 Silero-VAD kernel (sm_100a).
//
// One CTA (256 threads) owns a tile of up to 32 stream "slots" and walks them through time.
// Everything a thread does between two CTA barriers is a function in this header, written so
// that the same source compiles (a) as __device__ code for the CUDA kernel in
// svad_kernel_fp32.cu and (b) as plain C++ for the barrier-phase emulator tests/emu/ uses to
// check layouts and index algebra on a machine without a GPU.  No warp shuffles in here for
// that reason; cross-thread traffic goes through shared memory only.
//
// What is computed (reference: silero_vad.jit::_model / _model_8k, SURVEY.md Appendix A):
//   STFT   4 Hann-windowed N-point real DFTs per chunk (N = 256 @16k / 128 @8k), hop N/2, over
//          [context | chunk | reflect-pad]; done as a two-pass FFT (N = 16*NQ): pass A = NQ-point
//          DFTs over q for each residue r (two real sequences per complex FFT), twiddle, pass C =
//          16-point DFTs over r.  Equivalent to the reference's conv with forward_basis_buffer
//          (silero_vad.jit::_model.stft.transform_).
//   enc0-3 Conv1d k=3 pad=1 strides 1,2,2,1 + ReLU with the zero-padding taps skipped.
//   LSTM   gates = [x ; h] . [W_ih ; W_hh]^T + b, order i,f,g,o (torch.lstm_cell).
//   head   sigmoid(w . relu(h') + b).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define SVAD_HD __host__ __device__ __forceinline__
#define SVAD_COLD __host__ __device__ __noinline__
#else
#define SVAD_HD inline
#define SVAD_COLD inline
#endif

namespace svad {

constexpr int kThreads = 256;
constexpr int kSlots = 32;   // stream slots per CTA tile (row dimension of every GEMM)
constexpr int kHid = 128;
constexpr int kGates = 512;
constexpr int kStageBytes = 32768;  // one weight-tape slab buffer
constexpr int kStages = 2;
constexpr int kTcStageBytes = 16384;  // tensor-core kernel: 4 x 16 KB stages, up to 3-4 TMA copies in flight
constexpr int kTcStages = 4;

#if defined(__CUDACC__)
using f4 = float4;
using f2 = float2;
#else
struct alignas(16) f4 { float x, y, z, w; };
struct alignas(8) f2 { float x, y; };
#endif

// Packed fp32 FMA (Blackwell FFMA2 / fma.rn.f32x2): {a, a} * b + c in one issue slot.  The fp32 pipe tops out at the
// same ~110 FMA/clk/SM either way (tools/ubench_fma.cu), but FFMA2 needs half the issue slots, which is what the
// operand loads and address arithmetic of the GEMM loops compete for.  Per-lane results are IEEE fmaf.
SVAD_HD f2 ffma2_s(float a, f2 b, f2 c) {
#if defined(__CUDA_ARCH__)
    return __ffma2_rn(make_float2(a, a), b, c);
#else
    return f2{fmaf(a, b.x, c.x), fmaf(a, b.y, c.y)};
#endif
}

// ---------------------------------------------------------------- branch geometry
template <bool SR16>
struct Geo {
    static constexpr int n = SR16 ? 512 : 256;     // chunk samples
    static constexpr int ctx = SR16 ? 64 : 32;     // context_size_samples
    static constexpr int N = SR16 ? 256 : 128;     // filter_length
    static constexpr int hop = N / 2;              // hop_length
    static constexpr int F = N / 2 + 1;            // bins: 129 / 65
    static constexpr int NQ = N / 16;              // pass-A DFT length: 16 / 8
    static constexpr int L1 = ctx + n;             // 576 / 288
    // enc0 slabs: channels per slab (each channel = 3 taps x 128 floats = 1536 B)
    static constexpr int e0_nslab = SR16 ? 7 : 4;
    static constexpr int e0_cps = SR16 ? 19 : 17;  // max channels per slab (<= 21)
    static constexpr int nslab = e0_nslab + 4 + 1 + 1 + 16;
    static constexpr int nslab_enc = nslab - 16;   // features mode: the encoder slabs only (the tape's first nslab_enc slabs)
};

// ---------------------------------------------------------------- shared-memory map (float offsets)
// mag  [4][F][32]      (later aliased by e1 [2][64][32], e2 [64][32], e3 [128][32])
// e0   [4][128][32]    (aliased by the FFT exchange planes Zre/Zim [32][257] during the STFT)
// h    [128][32]
// consts: b0[128] b1[64] b2[64] b3[128] bl[512] wout[128] bout[1] pad[3] win[256] twr[256] twi[256]
struct SmemMap {
    static constexpr bool kTC = false;
    static constexpr int mag = 0;
    static constexpr int mag_floats = 4 * 129 * kSlots;          // 16512
    static constexpr int e1 = mag;                               // [2][64][32]
    static constexpr int e2 = e1 + 2 * 64 * kSlots;              // [64][32]
    static constexpr int e3 = e2 + 64 * kSlots;                  // [128][32]
    static constexpr int e0 = mag + mag_floats;
    static constexpr int zpitch = 257;
    static constexpr int e0_floats = 2 * kSlots * zpitch;        // 16448 >= 4*128*32
    static constexpr int zre = e0;
    static constexpr int zim = e0 + kSlots * zpitch;
    static constexpr int h = e0 + e0_floats;
    static constexpr int consts = h + kHid * kSlots;
    static constexpr int c_b0 = 0, c_b1 = 128, c_b2 = 192, c_b3 = 256, c_bl = 384, c_wout = 896, c_bout = 1024, c_win = 1028;
    static constexpr int c_twr = c_win + 256, c_twi = c_twr + 256;   // pass-A twiddles W_N^{k1 r} at [k1*16 + r]
    static constexpr int consts_floats = c_twi + 256;
    static constexpr int headp = consts + consts_floats;         // [32] probabilities of this step
    static constexpr int stage = headp + kSlots;                 // must be 16B aligned (x4 bytes)
    static constexpr int stage_floats = kStageBytes / 4;
    static constexpr int total_floats = stage + kStages * stage_floats;
};
// Shared-memory map of the tensor-core kernel (svad_tc.h).  Same regions, but every buffer an MMA reads directly
// (mag, e3, h and the "lo" staging tiles) is a stack of tcgen05 MN-major SWIZZLE_128B_BASE32B atoms: rows of 32
// floats (one per channel k), 32-byte chunk index XORed with k & 3, 512-byte aligned bases, mag frames padded to
// 132 rows so every frame starts on an atom boundary.  Weight stages hold K-major SWIZZLE_128B tiles (1 KB aligned).
struct SmemMapTC {
    static constexpr bool kTC = true;
    static constexpr int mag_pitch = 132;                        // rows per frame
    static constexpr int h = 0;                                  // LSTM hidden state [128][32]; below its lo rows (descriptor strides are unsigned)
    static constexpr int mag = h + kHid * kSlots;
    static constexpr int mag_floats = 4 * mag_pitch * kSlots;    // 16896 floats = 132 x 512 B
    // activations after enc0 (all as tcgen05 B rows; hi = the fp32 value, lo = its tf32 truncation error), over the dead mag rows
    static constexpr int e1 = mag;                               // [2][64][32]
    static constexpr int e1lo = e1 + 2 * 64 * kSlots;
    static constexpr int e2 = e1lo + 2 * 64 * kSlots;            // [64][32]
    static constexpr int e2lo = e2 + 64 * kSlots;
    static constexpr int e3 = e1;                                // [128][32] (over e1, dead once enc2 has run)
    static constexpr int e0 = mag + mag_floats;
    static constexpr int zpitch = 257;
    static constexpr int e0_floats = 129 * 128;                  // 66048 B >= Z planes (2*32*257) and e0 (4*128*32)
    static constexpr int zre = e0;
    static constexpr int zim = e0 + kSlots * zpitch;
    static constexpr int lo0 = e0;                               // enc0 lo tiles [4][Kt][32] (after the STFT, before e0 is written)
    static constexpr int e0lo = mag;                             // lo parts of e0 [4][128][32] (enc1's second B operand; mag is dead by then)
    static constexpr int lol_x = e1lo;                           // LSTM lo rows of e3 [128][32] (over e1lo), one N atom above e3
    static constexpr int lol_h = e2lo + 64 * kSlots;             // LSTM lo rows of h  [128][32]
    static constexpr int consts = e0 + e0_floats;
    static constexpr int c_b0 = 0, c_b1 = 128, c_b2 = 192, c_b3 = 256, c_bl = 384, c_wout = 896, c_bout = 1024, c_win = 1028;
    static constexpr int c_twr = c_win + 256, c_twi = c_twr + 256;
    static constexpr int c_wnyq = c_twi + 256;                   // enc0 weights of the Nyquist bin: [3 taps][128]
    static constexpr int c_nyq = c_wnyq + 384;                   // |X| of the Nyquist bin, [4 frames][32 slots] (copied out of mag before e0lo overwrites it)
    static constexpr int consts_floats = c_nyq + 4 * kSlots;
    static constexpr int headp = consts + consts_floats;
    static constexpr int stage = (headp + kSlots + 255) / 256 * 256;   // 1 KB aligned
    static constexpr int stage_floats = kTcStageBytes / 4;
    static constexpr int total_floats = stage + kTcStages * stage_floats;
};
static_assert(SmemMapTC::e0 % 256 == 0 && SmemMapTC::h % 128 == 0 && SmemMapTC::e3 % 128 == 0 && SmemMapTC::lol_x % 128 == 0, "atom / tile alignment");
static_assert(SmemMapTC::lol_h + 128 * kSlots <= SmemMapTC::mag + SmemMapTC::mag_floats && SmemMapTC::lol_x > SmemMapTC::e3 && SmemMapTC::lol_h > SmemMapTC::h && SmemMapTC::e0_floats >= 4 * SmemMapTC::stage_floats, "LSTM-phase borrowings");
static_assert(SmemMapTC::e0_floats >= 2 * kSlots * SmemMapTC::zpitch, "Z planes");
static_assert((size_t)SmemMapTC::total_floats * 4 + 256 <= 232448, "shared memory budget");
static_assert(SmemMap::e0_floats >= 4 * 128 * kSlots, "e0 region too small");
static_assert(SmemMap::e3 + 128 * kSlots <= SmemMap::mag + SmemMap::mag_floats, "e1/e2/e3 alias overflow");
static_assert(SmemMap::stage % 4 == 0, "stage alignment");

// tcgen05 MN-major SWIZZLE_128B_BASE32B row: 32-byte chunk (slot >> 3) XOR (row & 3)
SVAD_HD int tc_slot(int slot, int row) { return (((slot >> 3) ^ (row & 3)) << 3) | (slot & 7); }
SVAD_HD int tc_f4(int g, int row) { return (((g >> 1) ^ (row & 3)) << 1) | (g & 1); }   // physical float4 index of logical float4 g

// ---------------------------------------------------------------- thread coordinates
struct Tc {
    int tid, warp, lane, lm, ln;
    SVAD_HD explicit Tc(int t) : tid(t), warp(t >> 5), lane(t & 31), lm((t >> 3) & 3), ln(t & 7) {}
    // the 8 row slots of this thread are two float4 groups: [4*lm, 4*lm+4) and [16+4*lm, 16+4*lm+4)
    SVAD_HD int row0() const { return 4 * lm; }
    SVAD_HD int row1() const { return 16 + 4 * lm; }
};

// Slot validity for tiles of 4*RM streams (RM in [4,8]): every thread owns rows {4lm..4lm+3} and the first
// RM-4 of {16+4lm..16+4lm+3}.  Streams are numbered over the valid slots in increasing slot order.
template <int RM>
SVAD_HD bool slot_valid(int s) { return s < 16 || (s & 3) < RM - 4; }
template <int RM>
SVAD_HD int slot_to_local(int s) {  // local stream index of a valid slot
    return s < 16 ? s : 16 + (RM - 4) * ((s - 16) >> 2) + (s & 3);
}

// ---------------------------------------------------------------- persistent per-thread registers
struct Regs {
    f2 acc[32];      // GEMM accumulators of the current layer (column or row pairs, see each layer)
    float c[16];     // LSTM cell state: [row i][unit u] -> c[i*2+u]
};

// ---------------------------------------------------------------- small complex FFTs
// X[k] = sum_n x[n] exp(-2 pi i k n / NP), in place, compile-time indices only.
template <int K, int NP>
SVAD_HD void tw_mul(float& re, float& im) {  // (re,im) *= exp(-2 pi i K / NP)
    constexpr int k = ((K % NP) + NP) % NP;
    if constexpr (k == 0) {
    } else if constexpr (4 * k == NP) {          // -i
        float t = re; re = im; im = -t;
    } else if constexpr (2 * k == NP) {          // -1
        re = -re; im = -im;
    } else if constexpr (4 * k == 3 * NP) {      // +i
        float t = re; re = -im; im = t;
    } else if constexpr (8 * k == NP) {          // (1 - i)/sqrt2
        constexpr float s = 0.70710678118654752440f;
        float a = (re + im) * s, b = (im - re) * s; re = a; im = b;
    } else if constexpr (8 * k == 3 * NP) {      // (-1 - i)/sqrt2
        constexpr float s = 0.70710678118654752440f;
        float a = (im - re) * s, b = -(re + im) * s; re = a; im = b;
    } else if constexpr (8 * k == 5 * NP) {      // (-1 + i)/sqrt2
        constexpr float s = 0.70710678118654752440f;
        float a = -(re + im) * s, b = (re - im) * s; re = a; im = b;
    } else if constexpr (8 * k == 7 * NP) {      // (1 + i)/sqrt2
        constexpr float s = 0.70710678118654752440f;
        float a = (re - im) * s, b = (re + im) * s; re = a; im = b;
    } else {
        // general: only k/NP in {1,3,5,7,...}/16 reach here (NP == 16)
        constexpr double ang = -2.0 * 3.14159265358979323846 * (double)k / (double)NP;
        // constexpr cos/sin are not available in C++17; table for sixteenths
        constexpr float c16[16] = {1.0f, 0.92387953251128675613f, 0.70710678118654752440f, 0.38268343236508977173f,
                                   0.0f, -0.38268343236508977173f, -0.70710678118654752440f, -0.92387953251128675613f,
                                   -1.0f, -0.92387953251128675613f, -0.70710678118654752440f, -0.38268343236508977173f,
                                   0.0f, 0.38268343236508977173f, 0.70710678118654752440f, 0.92387953251128675613f};
        static_assert(NP == 16, "general twiddle only for 16ths");
        (void)ang;
        constexpr float wr = c16[k];                 // cos(2 pi k/16)
        constexpr float wi = -c16[(k + 12) % 16];    // -sin(2 pi k/16) ; sin(x) = cos(x - pi/2) = c16[k-4]
        float a = re * wr - im * wi, b = re * wi + im * wr; re = a; im = b;
    }
}

// radix-2 decimation-in-frequency, natural order in, bit-reversed order out (bin k at index bitrev(k)).
template <int NP, int LEN, int START>
struct Dif {
    SVAD_HD static void run(float (&re)[NP], float (&im)[NP]) {
        if constexpr (LEN >= 2) {
            constexpr int H = LEN / 2;
            Bfly<0>(re, im);
            Dif<NP, H, START>::run(re, im);
            Dif<NP, H, START + H>::run(re, im);
        }
    }
    template <int I>
    SVAD_HD static void Bfly(float (&re)[NP], float (&im)[NP]) {
        constexpr int H = LEN / 2;
        if constexpr (I < H) {
            float ar = re[START + I], ai = im[START + I], br = re[START + I + H], bi = im[START + I + H];
            re[START + I] = ar + br; im[START + I] = ai + bi;
            float dr = ar - br, di = ai - bi;
            tw_mul<I*(NP / LEN), NP>(dr, di);
            re[START + I + H] = dr; im[START + I + H] = di;
            Bfly<I + 1>(re, im);
        }
    }
};
SVAD_HD constexpr int bitrev(int x, int bits) { int r = 0; for (int i = 0; i < bits; i++) if (x & (1 << i)) r |= 1 << (bits - 1 - i); return r; }
SVAD_HD constexpr int ilog2(int x) { int r = 0; while ((1 << r) < x) r++; return r; }
// after fft_dif, bin k sits at index bitrev(k)
template <int NP>
SVAD_HD void fft_dif(float (&re)[NP], float (&im)[NP]) { Dif<NP, NP, 0>::run(re, im); }
template <int NP>
constexpr int binpos(int k) { return bitrev(k, ilog2(NP)); }

// ---------------------------------------------------------------- audio window fetch
// Sample `i` (0 <= i < L1 + N/4) of the padded window [context | chunk | reflect] of chunk t:
//   utils_vad.py:78 (context concat), silero_vad.jit::_model.stft.padding (reflect right by N/4),
//   utils_vad.py:100-102 (zero tail).  `ctx_in` (may be null) supplies samples before time 0.
// Samples are fp32 in [-1, 1) or int16 PCM; PCM is scaled by 2^-15 on load, which is exactly the float the
// reference's loaders produce (int16 / 32768: examples/cpp/wav.h:95-136, examples/onnx_sequence/run.py:115-119).
SVAD_HD float ld_sample(const float* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
SVAD_HD float ld_sample(const int16_t* p) {
#if defined(__CUDA_ARCH__)
    return (float)__ldg(p) * (1.0f / 32768.0f);
#else
    return (float)*p * (1.0f / 32768.0f);
#endif
}

// `dec` > 1: the row holds sr = dec * 16000 audio and only every dec-th sample is read -- the reference's `x[:, ::step]`
// (utils_vad.py:39-42, 301-305) done by the load instead of a host-side slice; L counts the decimated samples.
template <bool SR16, typename S>
SVAD_HD float window_sample(const S* audio, long L, const float* ctx_in, long t, int i, int dec = 1) {
    using G = Geo<SR16>;
    if (i >= G::L1) i = 2 * G::L1 - 2 - i;           // xp[L1 + j] = x1[L1 - 2 - j]
    long a = t * G::n - G::ctx + i;
    if (a < 0) return ctx_in ? ctx_in[G::ctx + a] : 0.0f;
    if (a >= L) return 0.0f;
    return ld_sample(audio + a * dec);
}

// ---------------------------------------------------------------- STFT pass A
// The STFT runs in 4 rounds; round (hs, fp) covers the 16 slots [16*hs, 16*hs+16) and the frame pair
// (2*fp, 2*fp+1).  Thread (half-warp hw = tid >> 4, residue r = tid & 15) owns slot 16*hs + hw and
// transforms the residue-r subsequences of BOTH frames with one complex NQ-point FFT (frame 2fp in the
// real part, frame 2fp+1 in the imaginary part -- two frames of the SAME stream, so no rounding noise
// ever crosses between streams), applies W_N^{k1 r} and stores Z_r[k1], k1 < NQ, into the exchange planes
// Z[item][k1*16 + r] with item = zitem(hw, fr).
SVAD_HD int zitem(int hw, int fr) { return (hw >> 1) + 8 * fr + 16 * (hw & 1); }   // bank-conflict-free stores
SVAD_HD int zitem_hw(int item) { return 2 * (item & 7) + (item >> 4); }
SVAD_HD int zitem_fr(int item) { return (item >> 3) & 1; }

// Raw (unwindowed) samples of one round for this thread: xa[q] = frame 2fp, xb[q] = frame 2fp+1, m = r + 16 q.
// Generic window fetch (context / reflect pad / zero tail resolved per sample): only the first and the last chunk of a
// row take it, so it is kept out of line -- the fused kernel's steady-state loop has to fit the instruction cache.
template <bool SR16, typename S>
SVAD_COLD void stft_load_generic(int r, int fp, const S* audio, const float* ctx_in, long L, long t, float* xa, float* xb, int dec) {
    using G = Geo<SR16>;
#pragma unroll 4
    for (int q = 0; q < G::NQ; q++) {
        const int m = r + 16 * q;
        xa[q] = window_sample<SR16, S>(audio, L, ctx_in, t, G::hop * (2 * fp) + m, dec);
        xb[q] = window_sample<SR16, S>(audio, L, ctx_in, t, G::hop * (2 * fp + 1) + m, dec);
    }
}

// `fast` (CTA-uniform; never with dec > 1): the whole padded window of chunk t lies inside the row, so the addresses are affine in
// (r, q) with the reflection resolved at compile time; otherwise the generic fetch handles context / zero tail.
template <bool SR16, typename S>
SVAD_HD void stft_load(int tid, int fp, const S* audio, const float* ctx_in, long L, long t, bool fast,
                       float (&xa)[Geo<SR16>::NQ], float (&xb)[Geo<SR16>::NQ], int dec = 1) {
    using G = Geo<SR16>;
    const int r = tid & 15;
    if (!audio) {
#pragma unroll
        for (int q = 0; q < G::NQ; q++) { xa[q] = 0.0f; xb[q] = 0.0f; }
        return;
    }
    if (fast) {
        const S* p = audio + t * G::n - G::ctx;   // window origin
#pragma unroll
        for (int q = 0; q < G::NQ; q++) {
            const int m = r + 16 * q;
            const int ia = G::hop * (2 * fp) + m, ib = G::hop * (2 * fp + 1) + m;   // ia < L1 always
            // frame 3 runs into the reflect pad for m >= L1 - 3 hop (a multiple of 16, so independent of r)
            const bool refl = (fp == 1) && (16 * q >= G::L1 - 3 * G::hop);
            const int jb = refl ? 2 * G::L1 - 2 - ib : ib;
            xa[q] = ld_sample(p + ia);
            xb[q] = ld_sample(p + jb);
        }
    } else {
        float ta[G::NQ], tb[G::NQ];   // address-taken copies: xa / xb themselves stay in registers
        stft_load_generic<SR16, S>(r, fp, audio, ctx_in, L, t, ta, tb, dec);
#pragma unroll
        for (int q = 0; q < G::NQ; q++) { xa[q] = ta[q]; xb[q] = tb[q]; }
    }
}

template <bool SR16, class M = SmemMap>
SVAD_HD void stft_pass_a(const Tc& tc, float* sm, const float (&xa)[Geo<SR16>::NQ], const float (&xb)[Geo<SR16>::NQ]) {
    using G = Geo<SR16>;
    constexpr int NQ = G::NQ;
    const int r = tc.tid & 15, hw = tc.tid >> 4;
    const float* win = sm + M::consts + M::c_win + r;
    const float* twr = sm + M::consts + M::c_twr + r;
    const float* twi = sm + M::consts + M::c_twi + r;
    float zr[NQ], zi[NQ];
#pragma unroll
    for (int q = 0; q < NQ; q++) {
        const float w = win[16 * q];  // 0.5 * periodic Hann at m = r + 16 q
        zr[q] = w * xa[q];
        zi[q] = w * xb[q];
    }
    fft_dif<NQ>(zr, zi);
    const int ia = zitem(hw, 0), ib = zitem(hw, 1);
    float* za_re = sm + M::zre + ia * M::zpitch + r;
    float* za_im = sm + M::zim + ia * M::zpitch + r;
    float* zb_re = sm + M::zre + ib * M::zpitch + r;
    float* zb_im = sm + M::zim + ib * M::zpitch + r;
#pragma unroll
    for (int k = 0; k < NQ; k++) {
        const int pk = bitrev(k, ilog2(NQ)), pn = bitrev((NQ - k) % NQ, ilog2(NQ));
        // Ya = Z[k] + conj(Z[-k]) ; Yb = -i (Z[k] - conj(Z[-k]))   (the 1/2 lives in the window)
        const float yar = zr[pk] + zr[pn], yai = zi[pk] - zi[pn];
        const float ybr = zi[pk] + zi[pn], ybi = zr[pn] - zr[pk];
        const float wr = twr[k * 16], wi = twi[k * 16];
        za_re[k * 16] = yar * wr - yai * wi;
        za_im[k * 16] = yar * wi + yai * wr;
        zb_re[k * 16] = ybr * wr - ybi * wi;
        zb_im[k * 16] = ybr * wi + ybi * wr;
    }
}

// ---------------------------------------------------------------- STFT pass C
// Thread (lane = exchange item -> slot, frame) takes k1 and runs the 16-point DFT over r;
// bins k1 + NQ*k2, k2 < 8 (and N/2 for k1 = 0) of that (slot, frame) go to mag[frame][bin][slot].
template <bool SR16, class M = SmemMap>
SVAD_HD void stft_pass_c(const Tc& tc, float* sm, int hs, int fp, int k1) {
    using G = Geo<SR16>;
    constexpr int pitch = M::kTC ? 132 : G::F;
    const int item = tc.lane;
    const int slot = 16 * hs + zitem_hw(item), f = 2 * fp + zitem_fr(item);
    const float* zre = sm + M::zre + item * M::zpitch + k1 * 16;
    const float* zim = sm + M::zim + item * M::zpitch + k1 * 16;
    float xr[16], xi[16];
#pragma unroll
    for (int r = 0; r < 16; r++) { xr[r] = zre[r]; xi[r] = zim[r]; }
    fft_dif<16>(xr, xi);
    float* mg = sm + M::mag + (f * pitch) * kSlots;
#pragma unroll
    for (int k2 = 0; k2 < 8; k2++) {
        const int p = bitrev(k2, 4), bin = k1 + G::NQ * k2;
        mg[bin * kSlots + (M::kTC ? tc_slot(slot, bin) : slot)] = sqrtf(xr[p] * xr[p] + xi[p] * xi[p]);
    }
    if (k1 == 0) {
        const int p = bitrev(8, 4);
        mg[(G::N / 2) * kSlots + slot] = sqrtf(xr[p] * xr[p] + xi[p] * xi[p]);   // N/2 is a multiple of 4: identity swizzle
    }
}

// ---------------------------------------------------------------- helpers
// Activation rows are 32 slots = 8 float4 groups; group g of channel ch is stored at physical group g ^ key(ch)
// so that the 8 lanes of a warp that write 8 different channels of the same row group hit 8 different bank
// groups (STS.128 conflict-free) while a reader, for whom ch is warp-uniform, just follows the permutation.
SVAD_HD int key_hi(int ch) { return (ch >> 1) & 7; }   // e0, e3, h   (writers own channel pairs)
SVAD_HD int key_lo(int ch) { return ch & 7; }          // e1, e2      (writers own single channels)
SVAD_HD int swz_slot(int slot, int key) { return (((slot >> 2) ^ key) << 2) | (slot & 3); }
SVAD_HD void load8(const float* row, int lm, int key, float (&x)[8]) {
    f4 a = *reinterpret_cast<const f4*>(row + ((lm ^ key) << 2));
    f4 b = *reinterpret_cast<const f4*>(row + (((4 + lm) ^ key) << 2));
    x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
}
SVAD_HD void store8(float* row, int lm, int key, const float (&x)[8]) {
    f4 a{x[0], x[1], x[2], x[3]}, b{x[4], x[5], x[6], x[7]};
    *reinterpret_cast<f4*>(row + ((lm ^ key) << 2)) = a;
    *reinterpret_cast<f4*>(row + (((4 + lm) ^ key) << 2)) = b;
}
SVAD_HD void store8_tc(float* row, int lm, int ch, const float (&x)[8]) {
    f4 a{x[0], x[1], x[2], x[3]}, b{x[4], x[5], x[6], x[7]};
    *reinterpret_cast<f4*>(row + (tc_f4(lm, ch) << 2)) = a;
    *reinterpret_cast<f4*>(row + (tc_f4(4 + lm, ch) << 2)) = b;
}
SVAD_HD float relu(float v) { return v > 0.0f ? v : 0.0f; }   // NaN -> 0 like fmaxf(v, 0)
SVAD_HD float sigmoid_acc(float v) { return 1.0f / (1.0f + expf(-v)); }
// Gate math of the tensor-core kernel: one MUFU.EX2 + one MUFU.RCP (+ one Newton step) per activation instead of libm expf /
// tanhf / IEEE division (~35 instead of ~115 instructions per LSTM cell).  Absolute error ~1e-7 per activation (ex2.approx: 2 ulp
// of e^x, which enters scaled by <= 1/4 resp. 1/2), saturating correctly for large |v| (e^x = inf -> 0 / 1).
SVAD_HD float rcp_newton(float y) {   // 1 / y for y in [1, inf]
#if defined(__CUDA_ARCH__)
    const float r = __fdividef(1.0f, y);
    return (y < 1e30f) ? fmaf(r, fmaf(-y, r, 1.0f), r) : r;   // no refinement near overflow (y * r would be inf * 0)
#else
    return 1.0f / y;
#endif
}
SVAD_HD float sigmoid_fast(float v) {
#if defined(__CUDA_ARCH__)
    return rcp_newton(1.0f + __expf(-v));
#else
    return 1.0f / (1.0f + expf(-v));
#endif
}
SVAD_HD float tanh_fast(float v) {
#if defined(__CUDA_ARCH__)
    return fmaf(-2.0f, rcp_newton(1.0f + __expf(2.0f * v)), 1.0f);
#else
    return tanhf(v);
#endif
}

// ---------------------------------------------------------------- enc0
// acc[t][i] = (col u=0, col u=1) for t<4 frames, i<8 rows -> rg.acc[t*8+i]; cols 16*warp + 2*ln + u.
// slab = W0p[c][j][128] for channels [c0, c1).
template <bool SR16, int RM>
SVAD_HD void enc0_init(const Tc& tc, const float* sm, Regs& rg) {
    const f2 b0 = *reinterpret_cast<const f2*>(sm + SmemMap::consts + SmemMap::c_b0 + 16 * tc.warp + 2 * tc.ln);
#pragma unroll
    for (int k = 0; k < 32; k++) rg.acc[k] = b0;
}
template <bool SR16>
SVAD_HD void enc0_fetch(const Tc& tc, const float* mag, const float* wp, int c, float (&x)[4][8], f2 (&w)[3]) {
    using G = Geo<SR16>;
#pragma unroll
    for (int f = 0; f < 4; f++) load8(mag + (f * G::F + c) * kSlots, tc.lm, 0, x[f]);
#pragma unroll
    for (int j = 0; j < 3; j++) w[j] = *reinterpret_cast<const f2*>(wp + j * 128);
}
template <int RM>
SVAD_HD void enc0_fma(const float (&x)[4][8], const f2 (&w)[3], Regs& rg) {
#pragma unroll
    for (int t = 0; t < 4; t++)
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const int fi = t + j - 1;
            if (fi < 0 || fi > 3) continue;
#pragma unroll
            for (int i = 0; i < RM; i++) rg.acc[t * 8 + i] = ffma2_s(x[fi][i], w[j], rg.acc[t * 8 + i]);
        }
}
// Operands of channel c+1 are fetched before the 70-80 FFMA2 of channel c issue (register double buffer), so a
// warp never sits on LDS latency with an idle FMA pipe even when its SMSP partner runs in lockstep.
template <bool SR16, int RM>
SVAD_HD void enc0_slab(const Tc& tc, const float* sm, const float* slab, Regs& rg, int c0, int c1) {
    const int oc = 16 * tc.warp + 2 * tc.ln;
    const float* mag = sm + SmemMap::mag;
    const float* wp = slab + oc;
    float xa[4][8], xb[4][8];
    f2 wa[3], wb[3];
    enc0_fetch<SR16>(tc, mag, wp, c0, xa, wa);
    int c = c0;
#pragma unroll 1
    for (; c + 2 <= c1; c += 2) {
        enc0_fetch<SR16>(tc, mag, wp + (c + 1 - c0) * 384, c + 1, xb, wb);
        enc0_fma<RM>(xa, wa, rg);
        if (c + 2 < c1) enc0_fetch<SR16>(tc, mag, wp + (c + 2 - c0) * 384, c + 2, xa, wa);
        enc0_fma<RM>(xb, wb, rg);
    }
    if (c < c1) enc0_fma<RM>(xa, wa, rg);
}
template <bool SR16, int RM>
SVAD_HD void enc0_store(const Tc& tc, float* sm, const Regs& rg) {
    const int oc = 16 * tc.warp + 2 * tc.ln;
#pragma unroll
    for (int t = 0; t < 4; t++) {
        float v0[8], v1[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            v0[i] = (i < RM) ? relu(rg.acc[t * 8 + i].x) : 0.0f;
            v1[i] = (i < RM) ? relu(rg.acc[t * 8 + i].y) : 0.0f;
        }
        store8(sm + SmemMap::e0 + (t * 128 + oc) * kSlots, tc.lm, key_hi(oc), v0);
        store8(sm + SmemMap::e0 + (t * 128 + oc + 1) * kSlots, tc.lm, key_hi(oc), v1);
    }
}

// ---------------------------------------------------------------- enc1: 128 -> 64, stride 2, T 4 -> 2
// t=0 sees frames (-1,0,1) -> taps 1,2 ; t=1 sees frames (1,2,3).  Only 64 output columns: a thread owns a column PAIR
// (oc = 16*(warp&3) + 2*ln, packed FFMA2 with the activation as the scalar operand, like enc0) and the input channels of
// every slab are split between the two warp groups (warps 0-3 / 4-7); the two partial sums meet in shared memory.
// rg.acc[t*8 + i] = (col oc, col oc+1) for out-frame t, row i.  slab = W1p[c][j][64] for channels [c0, c1).
SVAD_HD void load8p(const float* row, int lm, int key, f2 (&x)[4]) {
    f4 a = *reinterpret_cast<const f4*>(row + ((lm ^ key) << 2));
    f4 b = *reinterpret_cast<const f4*>(row + (((4 + lm) ^ key) << 2));
    x[0] = f2{a.x, a.y}; x[1] = f2{a.z, a.w}; x[2] = f2{b.x, b.y}; x[3] = f2{b.z, b.w};
}
template <int RM, class M = SmemMap>
SVAD_HD void enc1_init(const Tc& tc, const float* sm, Regs& rg) {
    const int oc = 16 * (tc.warp & 3) + 2 * tc.ln;
    const f2 b = (tc.warp < 4) ? *reinterpret_cast<const f2*>(sm + M::consts + M::c_b1 + oc) : f2{0.0f, 0.0f};
#pragma unroll
    for (int k = 0; k < 16; k++) rg.acc[k] = b;
}
SVAD_HD void enc1_fetch(const Tc& tc, const float* e0, const float* wp, int c, float (&x)[4][8], f2 (&w)[3]) {
#pragma unroll
    for (int f = 0; f < 4; f++) load8(e0 + (f * 128 + c) * kSlots, tc.lm, key_hi(c), x[f]);
#pragma unroll
    for (int j = 0; j < 3; j++) w[j] = *reinterpret_cast<const f2*>(wp + j * 64);
}
template <int RM>
SVAD_HD void enc1_fma(const float (&x)[4][8], const f2 (&w)[3], Regs& rg) {
#pragma unroll
    for (int i = 0; i < RM; i++) {
        rg.acc[i] = ffma2_s(x[0][i], w[1], rg.acc[i]);
        rg.acc[i] = ffma2_s(x[1][i], w[2], rg.acc[i]);
        rg.acc[8 + i] = ffma2_s(x[1][i], w[0], rg.acc[8 + i]);
        rg.acc[8 + i] = ffma2_s(x[2][i], w[1], rg.acc[8 + i]);
        rg.acc[8 + i] = ffma2_s(x[3][i], w[2], rg.acc[8 + i]);
    }
}
template <int RM, class M = SmemMap>
SVAD_HD void enc1_slab(const Tc& tc, const float* sm, const float* slab, Regs& rg, int c0, int c1) {
    const int hc = (c1 - c0) >> 1, cb = c0 + (tc.warp >> 2) * hc;   // this warp group's channels [cb, cb + hc), hc even
    const float* wp = slab + (cb - c0) * 192 + 16 * (tc.warp & 3) + 2 * tc.ln;
    const float* e0 = sm + M::e0;
    float xa[4][8], xb[4][8];
    f2 wa[3], wb[3];
    enc1_fetch(tc, e0, wp, cb, xa, wa);
#pragma unroll 1
    for (int c = 0; c < hc; c += 2) {
        enc1_fetch(tc, e0, wp + (c + 1) * 192, cb + c + 1, xb, wb);
        enc1_fma<RM>(xa, wa, rg);
        if (c + 2 < hc) enc1_fetch(tc, e0, wp + (c + 2) * 192, cb + c + 2, xa, wa);
        enc1_fma<RM>(xb, wb, rg);
    }
}
// after the last slab: warps 4-7 park their partial sums (scratch above e3), barrier, warps 0-3 add, ReLU, store e1
template <int RM, class M = SmemMap>
SVAD_HD void enc1_park(const Tc& tc, float* sm, const Regs& rg) {
    if (tc.warp < 4) return;
    float* scr = sm + M::e3 + 128 * kSlots;
    const int oc = 16 * (tc.warp & 3) + 2 * tc.ln;
#pragma unroll
    for (int t = 0; t < 2; t++) {
        float v0[8], v1[8];
#pragma unroll
        for (int i = 0; i < 8; i++) { v0[i] = rg.acc[t * 8 + i].x; v1[i] = rg.acc[t * 8 + i].y; }
        store8(scr + (t * 64 + oc) * kSlots, tc.lm, key_hi(oc), v0);
        store8(scr + (t * 64 + oc + 1) * kSlots, tc.lm, key_hi(oc), v1);
    }
}
template <int RM, class M = SmemMap>
SVAD_HD void enc1_store(const Tc& tc, float* sm, const Regs& rg) {
    if (tc.warp >= 4) return;
    const float* scr = sm + M::e3 + 128 * kSlots;
    const int oc = 16 * tc.warp + 2 * tc.ln;
#pragma unroll
    for (int t = 0; t < 2; t++) {
        float p0[8], p1[8], v0[8], v1[8];
        load8(scr + (t * 64 + oc) * kSlots, tc.lm, key_hi(oc), p0);
        load8(scr + (t * 64 + oc + 1) * kSlots, tc.lm, key_hi(oc), p1);
#pragma unroll
        for (int i = 0; i < 8; i++) {
            v0[i] = (i < RM) ? relu(rg.acc[t * 8 + i].x + p0[i]) : 0.0f;
            v1[i] = (i < RM) ? relu(rg.acc[t * 8 + i].y + p1[i]) : 0.0f;
        }
        store8(sm + M::e1 + (t * 64 + oc) * kSlots, tc.lm, key_lo(oc), v0);
        store8(sm + M::e1 + (t * 64 + oc + 1) * kSlots, tc.lm, key_lo(oc + 1), v1);
    }
}

// ---------------------------------------------------------------- enc2: 64 -> 64, stride 2, T 2 -> 1 (taps 1,2 live)
// slab = W2p[c][jj][64], jj=0 <-> tap 1 (frame 0), jj=1 <-> tap 2 (frame 1); one slab, 64 channels.  Row pairs.
template <int RM, class M = SmemMap>
SVAD_HD void enc2_all(const Tc& tc, float* sm, const float* slab, Regs& rg) {
    const int o = 8 * tc.warp + tc.ln;
    const float b = sm[M::consts + M::c_b2 + o];
    f2 acc[4];
#pragma unroll
    for (int ip = 0; ip < 4; ip++) acc[ip] = f2{b, b};
#pragma unroll 4
    for (int c = 0; c < 64; c++) {
        f2 x0[4], x1[4];
        load8p(sm + M::e1 + c * kSlots, tc.lm, key_lo(c), x0);
        load8p(sm + M::e1 + (64 + c) * kSlots, tc.lm, key_lo(c), x1);
        const float w0 = slab[c * 128 + o], w1 = slab[c * 128 + 64 + o];
#pragma unroll
        for (int ip = 0; ip < 4; ip++) { acc[ip] = ffma2_s(w0, x0[ip], acc[ip]); acc[ip] = ffma2_s(w1, x1[ip], acc[ip]); }
    }
    float v[8];
#pragma unroll
    for (int ip = 0; ip < 4; ip++) {
        v[2 * ip] = (2 * ip < RM) ? relu(acc[ip].x) : 0.0f;
        v[2 * ip + 1] = (2 * ip + 1 < RM) ? relu(acc[ip].y) : 0.0f;
    }
    store8(sm + M::e2 + o * kSlots, tc.lm, key_lo(o), v);
    (void)rg;
}

// ---------------------------------------------------------------- enc3: 64 -> 128, T 1 -> 1 (tap 1 live)
// slab = W3p[c][128]; cols 16*warp + 2*ln + u (column pairs).
template <int RM, class M = SmemMap>
SVAD_HD void enc3_all(const Tc& tc, float* sm, const float* slab, Regs& rg) {
    const int oc = 16 * tc.warp + 2 * tc.ln;
    const f2 b3 = *reinterpret_cast<const f2*>(sm + M::consts + M::c_b3 + oc);
    f2 acc[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = b3;
#pragma unroll 4
    for (int c = 0; c < 64; c++) {
        float x[8];
        load8(sm + M::e2 + c * kSlots, tc.lm, key_lo(c), x);
        const f2 w = *reinterpret_cast<const f2*>(slab + c * 128 + oc);
#pragma unroll
        for (int i = 0; i < RM; i++) acc[i] = ffma2_s(x[i], w, acc[i]);
    }
    float v0[8], v1[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { v0[i] = (i < RM) ? relu(acc[i].x) : 0.0f; v1[i] = (i < RM) ? relu(acc[i].y) : 0.0f; }
    if constexpr (M::kTC) {   // e3 is read by the LSTM MMAs: tcgen05 atom rows
        store8_tc(sm + M::e3 + oc * kSlots, tc.lm, oc, v0);
        store8_tc(sm + M::e3 + (oc + 1) * kSlots, tc.lm, oc + 1, v1);
    } else {
        store8(sm + M::e3 + oc * kSlots, tc.lm, key_hi(oc), v0);
        store8(sm + M::e3 + (oc + 1) * kSlots, tc.lm, key_hi(oc), v1);
    }
    (void)rg;
}

// ---------------------------------------------------------------- LSTM
// Columns are permuted on the host: n' = 64*warp + 32*u + 4*ln + g  <->  gate g of hidden unit j = 16*warp + 2*ln + u.
// rg.acc[i*4 + 2u + p] = gates (2p, 2p+1) of unit u for row i.  slab = Wl[k][512] for k in [k0, k0+16);
// k < 128 reads e3, else h.
template <int RM>
SVAD_HD void lstm_init(const Tc& tc, const float* sm, Regs& rg) {
    const float* bl = sm + SmemMap::consts + SmemMap::c_bl + 64 * tc.warp + 4 * tc.ln;
    const f4 b0 = *reinterpret_cast<const f4*>(bl), b1 = *reinterpret_cast<const f4*>(bl + 32);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        rg.acc[i * 4 + 0] = f2{b0.x, b0.y}; rg.acc[i * 4 + 1] = f2{b0.z, b0.w};
        rg.acc[i * 4 + 2] = f2{b1.x, b1.y}; rg.acc[i * 4 + 3] = f2{b1.z, b1.w};
    }
}
SVAD_HD void lstm_fetch(const Tc& tc, const float* a, const float* wrow, int kk, float (&x)[8], f2 (&w)[4]) {
    load8(a + kk * kSlots, tc.lm, key_hi(kk), x);
    const f4 w0 = *reinterpret_cast<const f4*>(wrow + kk * kGates);
    const f4 w1 = *reinterpret_cast<const f4*>(wrow + kk * kGates + 32);
    w[0] = f2{w0.x, w0.y}; w[1] = f2{w0.z, w0.w}; w[2] = f2{w1.x, w1.y}; w[3] = f2{w1.z, w1.w};
}
template <int RM>
SVAD_HD void lstm_fma(const float (&x)[8], const f2 (&w)[4], Regs& rg) {
#pragma unroll
    for (int i = 0; i < RM; i++)
#pragma unroll
        for (int p = 0; p < 4; p++) rg.acc[i * 4 + p] = ffma2_s(x[i], w[p], rg.acc[i * 4 + p]);
}
template <int RM>
SVAD_HD void lstm_slab(const Tc& tc, const float* sm, const float* slab, Regs& rg, int k0) {
    const float* wrow = slab + 64 * tc.warp + 4 * tc.ln;
    const float* a = (k0 < kHid) ? sm + SmemMap::e3 + k0 * kSlots : sm + SmemMap::h + (k0 - kHid) * kSlots;
    float xa[8], xb[8];
    f2 wa[4], wb[4];
    lstm_fetch(tc, a, wrow, 0, xa, wa);
#pragma unroll 2
    for (int kk = 0; kk < 16; kk += 2) {
        lstm_fetch(tc, a, wrow, kk + 1, xb, wb);
        lstm_fma<RM>(xa, wa, rg);
        if (kk + 2 < 16) lstm_fetch(tc, a, wrow, kk + 2, xa, wa);
        lstm_fma<RM>(xb, wb, rg);
    }
}
// gate nonlinearity + state update; writes h' into smem (after the barrier that ends the last slab).
template <int RM>
SVAD_HD void lstm_epilogue(const Tc& tc, float* sm, Regs& rg) {
    const int j0 = 16 * tc.warp + 2 * tc.ln;
#pragma unroll
    for (int u = 0; u < 2; u++) {
        float hv[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            if (i < RM) {
                const f2 g01 = rg.acc[i * 4 + 2 * u], g23 = rg.acc[i * 4 + 2 * u + 1];
                float ig = sigmoid_acc(g01.x), fg = sigmoid_acc(g01.y), gg = tanhf(g23.x), og = sigmoid_acc(g23.y);
                float cn = fmaf(fg, rg.c[i * 2 + u], ig * gg);
                rg.c[i * 2 + u] = cn;
                hv[i] = og * tanhf(cn);
            } else {
                hv[i] = 0.0f;
            }
        }
        store8(sm + SmemMap::h + (j0 + u) * kSlots, tc.lm, key_hi(j0), hv);
    }
}
// head: thread tid < 32 (slot = tid): p = sigmoid(sum_j wout[j] relu(h'[j]) + bout)
SVAD_HD float head_prob(const float* sm, int slot) {
    const float* wout = sm + SmemMap::consts + SmemMap::c_wout;
    const float* h = sm + SmemMap::h;
    float a0 = sm[SmemMap::consts + SmemMap::c_bout], a1 = 0.f;
#pragma unroll 8
    for (int j = 0; j < kHid; j += 2) {   // units j, j+1 share a swizzle key
        const int ps = swz_slot(slot, key_hi(j));
        a0 = fmaf(wout[j], relu(h[j * kSlots + ps]), a0);
        a1 = fmaf(wout[j + 1], relu(h[(j + 1) * kSlots + ps]), a1);
    }
    return sigmoid_acc(a0 + a1);
}

}  // namespace svad
