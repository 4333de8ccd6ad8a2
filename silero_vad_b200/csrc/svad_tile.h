// svad_tile.h -- barrier-level schedule of one CTA of the fused fp32 kernel: a tile of up to 4*RM
// streams is carried through all T chunk steps; (h, c) and the audio context never leave the SM.
//
// `Env` hides what differs between the GPU and the CPU emulator:
//   int tid();  float* smem();  void sync();                      CTA barrier
//   const float* slab_acquire(long it, long total);               thread 0 first refills the ring (waits until every warp
//                                                                 released slab it-1, issues slab it+1); then all wait
//                                                                 until tape slab #it has landed in its stage
//   void slab_done(long it);                                      this thread is finished reading slab #it
// Weight slabs are handed over with full/empty mbarriers, so warps are NOT barrier-synchronised per slab; CTA
// barriers remain only where activations cross threads: 8 for the STFT, one per layer boundary, 2 around the
// LSTM epilogue / head (15 per step instead of 45).
#pragma once
#include "svad_core.h"
#include "svad_pack.h"

namespace svad {

struct TileArgs {
    const void* audio;      // [B][ld] samples (fp32 or int16 PCM, see run_cta's S), device (or host in the emulator)
    long ld, L;             // row stride (in stored samples), valid samples per row AFTER decimation (tail is zero-padded to T*n)
    int dec;                // sample stride within a row: 1, or k for sr = k * 16000 input (utils_vad.py:39-42)
    int B;                  // streams
    long T;                 // chunk steps = ceil(L / n)
    const float* state_in;  // [2][B][128] or null (zeros)
    const float* ctx_in;    // [B] rows of ctx floats, row stride ctx_ld, or null (zeros)
    long ctx_ld;
    float* state_out;       // [2][B][128] or null
    float* ctx_out;         // [B][ctx] or null
    float* probs;           // [B][ldp]
    long ldp;
    const float* tape;      // weight tape (Tape<SR16>::total floats)
    const float* consts;    // SmemMap::consts_floats floats
    long long* dbg;         // optional: per-phase clock64 stamps of CTA 0 (tensor-core kernel, profiling builds)
};

// FEAT: features mode (encoder-feature export for decoder fine-tuning).  The step ends after enc3: its rows go to a.probs, which
// then holds [B][ldp][128] floats (the post-ReLU enc3 output of chunk t of stream g, i.e. the LSTM input, at row g * ldp + t), and
// the LSTM, the head and the state / context write-back are skipped.  (TileArgs keeps its layout: a field added for this mode
// changed the register allocation of the inference instantiations.)  The tape walk then has G::nslab_enc slabs per step (the
// LSTM slabs are never issued), so Env must be instantiated with the same FEAT.
template <bool SR16, int RM, typename S, bool FEAT = false, class Env>
SVAD_HD void run_cta(Env& env, const TileArgs& a, int first_tile, int tile_stride, int ntiles) {
    using G = Geo<SR16>;
    constexpr int kNslab = FEAT ? G::nslab_enc : G::nslab;
    using TP = Tape<SR16>;
    const Tc tc(env.tid());
    float* sm = env.smem();
    const S* audio = static_cast<const S*>(a.audio);
    Regs rg;
    constexpr int BT = 4 * RM;

    // constants -> smem; pass-A twiddle table W_N^{k1 r} (k1 < NQ, r < 16) computed in place
    for (int i = tc.tid; i < SmemMap::c_twr; i += kThreads) sm[SmemMap::consts + i] = a.consts[i];
    {
        const int k = tc.tid >> 4, r = tc.tid & 15;
        float s = 0.0f, c = 1.0f;
        if (k < G::NQ) {
            const float x = -2.0f * (float)((k * r) % G::N) / (float)G::N;  // angle / pi
#if defined(__CUDA_ARCH__)
            sincospif(x, &s, &c);
#else
            s = (float)sin(M_PI * (double)x); c = (float)cos(M_PI * (double)x);
#endif
        }
        sm[SmemMap::consts + SmemMap::c_twr + tc.tid] = c;
        sm[SmemMap::consts + SmemMap::c_twi + tc.tid] = s;
    }
    int my_tiles = 0;
    for (int tile = first_tile; tile < ntiles; tile += tile_stride) my_tiles++;
    const long total_slabs = (long)my_tiles * a.T * kNslab;
    long it = 0;  // running slab counter of this CTA

    for (int tile = first_tile; tile < ntiles; tile += tile_stride) {
        const int g0 = tile * BT;
        // ---- tile init: h -> smem, c -> registers
        env.sync();  // previous tile's readers of h / consts writers done
        for (int i = tc.tid; i < kHid * kSlots; i += kThreads) {
            const int j = i >> 5, s = i & 31;
            const int g = g0 + slot_to_local<RM>(s);
            float v = 0.0f;
            if (a.state_in && slot_valid<RM>(s) && g < a.B) v = a.state_in[(long)g * kHid + j];
            sm[SmemMap::h + j * kSlots + swz_slot(s, key_hi(j))] = v;
        }
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int s = (i < 4) ? tc.row0() + i : tc.row1() + (i - 4);
                const int g = g0 + slot_to_local<RM>(s);
                const int j = 16 * tc.warp + 2 * tc.ln + u;
                float v = 0.0f;
                if (a.state_in && i < RM && g < a.B) v = a.state_in[((long)a.B + g) * kHid + j];
                rg.c[i * 2 + u] = v;
            }
        // audio rows of the two slots (one per 16-slot half) this thread feeds in STFT pass A
        const S* aud[2];
        const float* cxp[2];
#pragma unroll
        for (int hs = 0; hs < 2; hs++) {
            const int sl = 16 * hs + (tc.tid >> 4);
            const int gs = g0 + slot_to_local<RM>(sl);
            const bool v = slot_valid<RM>(sl) && gs < a.B;
            aud[hs] = v ? audio + (long)gs * a.ld : nullptr;
            cxp[hs] = (v && a.ctx_in) ? a.ctx_in + (long)gs * a.ctx_ld : nullptr;
        }
        env.sync();

        float xa[G::NQ], xb[G::NQ];   // raw samples of the STFT round about to be transformed
        for (long t = 0; t < a.T; t++) {
            // ---------------- STFT: 4 rounds (slot half hs, frame pair fp); the raw samples of round i+1 are
            // fetched into registers while round i is transformed, round 0 of the next step at the end of this one.
            const bool fast = (t > 0) && ((t + 1) * G::n <= a.L) && a.dec == 1;
            if (t + 1 < a.T && a.dec == 1) {   // pull the next chunk of every stream of the tile into L2
                constexpr int kPerLine = 128 / (int)sizeof(S), kLines = G::n / kPerLine;
                for (int i = tc.tid; i < BT * kLines; i += kThreads) {
                    const int loc = i / kLines, line = i % kLines, g = g0 + loc;
                    const long off = (t + 1) * G::n + line * kPerLine;
                    if (g < a.B && off < a.L) env.prefetch_l2(audio + (long)g * a.ld + off);
                }
            }
            if (t == 0) stft_load<SR16, S>(tc.tid, 0, aud[0], cxp[0], a.L, t, fast, xa, xb, a.dec);
#pragma unroll 1
            for (int rnd = 0; rnd < 4; rnd++) {
                const int hs = rnd >> 1, fp = rnd & 1;
                float na[G::NQ], nb[G::NQ];
                if (rnd < 3) stft_load<SR16, S>(tc.tid, (rnd + 1) & 1, rnd >= 1 ? aud[1] : aud[0], rnd >= 1 ? cxp[1] : cxp[0], a.L, t, fast, na, nb, a.dec);
                stft_pass_a<SR16>(tc, sm, xa, xb);
                env.sync();
#pragma unroll
                for (int kk = 0; kk < G::NQ / 8; kk++) stft_pass_c<SR16>(tc, sm, hs, fp, tc.warp * (G::NQ / 8) + kk);
                env.sync();
                if (rnd < 3) {
#pragma unroll
                    for (int q = 0; q < G::NQ; q++) { xa[q] = na[q]; xb[q] = nb[q]; }
                }
            }
            // ---------------- enc0
            enc0_init<SR16, RM>(tc, sm, rg);
#pragma unroll 1
            for (int s = 0; s < G::e0_nslab; s++, it++) {
                const float* slab = env.slab_acquire(it, total_slabs);
                enc0_slab<SR16, RM>(tc, sm, slab, rg, TP::e0_c0(s), TP::e0_c0(s + 1));
                env.slab_done(it);
            }
            enc0_store<SR16, RM>(tc, sm, rg);
            env.sync();
            // ---------------- enc1
            enc1_init<RM>(tc, sm, rg);
#pragma unroll 1
            for (int s = 0; s < 4; s++, it++) {
                const float* slab = env.slab_acquire(it, total_slabs);
                enc1_slab<RM>(tc, sm, slab, rg, s * 32, s * 32 + 32);
                env.slab_done(it);
            }
            enc1_park<RM>(tc, sm, rg);
            env.sync();
            enc1_store<RM>(tc, sm, rg);
            env.sync();
            // ---------------- enc2, enc3
            {
                const float* slab = env.slab_acquire(it, total_slabs);
                enc2_all<RM>(tc, sm, slab, rg);
                env.slab_done(it);
                env.sync();
                it++;
                slab = env.slab_acquire(it, total_slabs);
                enc3_all<RM>(tc, sm, slab, rg);
                env.slab_done(it);
                env.sync();
                it++;
            }
            if constexpr (FEAT) {
                for (int i = tc.tid; i < kHid * kSlots; i += kThreads) {   // consecutive threads: consecutive channels of one slot
                    const int s = i >> 7, j = i & (kHid - 1);
                    const int g = g0 + slot_to_local<RM>(s);
                    if (slot_valid<RM>(s) && g < a.B) a.probs[((long)g * a.ldp + t) * kHid + j] = sm[SmemMap::e3 + j * kSlots + swz_slot(s, key_hi(j))];
                }
                env.sync();   // e3 is read before the next step's STFT overwrites the region
                if (t + 1 < a.T)
                    stft_load<SR16, S>(tc.tid, 0, aud[0], cxp[0], a.L, t + 1, ((t + 2) * G::n <= a.L) && a.dec == 1, xa, xb, a.dec);
                continue;
            }
            // ---------------- LSTM + head
            lstm_init<RM>(tc, sm, rg);
#pragma unroll 1
            for (int s = 0; s < 16; s++, it++) {
                const float* slab = env.slab_acquire(it, total_slabs);
                lstm_slab<RM>(tc, sm, slab, rg, s * 16);
                env.slab_done(it);
            }
            env.sync();   // every warp is done reading e3 / h
            lstm_epilogue<RM>(tc, sm, rg);
            env.sync();
            if (tc.tid < kSlots) {
                const int g = g0 + slot_to_local<RM>(tc.tid);
                if (slot_valid<RM>(tc.tid) && g < a.B) a.probs[(long)g * a.ldp + t] = head_prob(sm, tc.tid);
            }
            if (t + 1 < a.T)
                stft_load<SR16, S>(tc.tid, 0, aud[0], cxp[0], a.L, t + 1, ((t + 2) * G::n <= a.L) && a.dec == 1, xa, xb, a.dec);
        }
        // ---- tile exit: carry state / context out
        env.sync();
        if (FEAT) continue;
        if (a.state_out) {
            for (int i = tc.tid; i < kHid * kSlots; i += kThreads) {
                const int s = i & 31, j = i >> 5;
                const int g = g0 + slot_to_local<RM>(s);
                if (slot_valid<RM>(s) && g < a.B) a.state_out[(long)g * kHid + j] = sm[SmemMap::h + j * kSlots + swz_slot(s, key_hi(j))];
            }
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int s = (i < 4) ? tc.row0() + i : tc.row1() + (i - 4);
                    const int g = g0 + slot_to_local<RM>(s);
                    const int j = 16 * tc.warp + 2 * tc.ln + u;
                    if (i < RM && g < a.B) a.state_out[((long)a.B + g) * kHid + j] = rg.c[i * 2 + u];
                }
        }
        if (a.ctx_out) {
            for (int i = tc.tid; i < BT * G::ctx; i += kThreads) {
                const int loc = i / G::ctx, k = i % G::ctx, g = g0 + loc;
                if (g < a.B) {
                    // new context = last ctx samples of the (zero-padded) final window
                    const float* cx = a.ctx_in ? a.ctx_in + (long)g * a.ctx_ld : nullptr;
                    float v = (a.T > 0) ? window_sample<SR16, S>(audio + (long)g * a.ld, a.L, cx, a.T - 1, G::n + k, a.dec)
                                        : (cx ? cx[k] : 0.0f);
                    a.ctx_out[(long)g * G::ctx + k] = v;
                }
            }
        }
    }
}

}  // namespace svad
