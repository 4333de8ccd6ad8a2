// svad_emu_tune.cpp -- CPU emulation of the decoder fine-tuning device code (TEST INFRASTRUCTURE, never timed).
//   svad_emu_features   the fused fp32 kernel in features mode: svad::run_cta<..., FEAT = true> on 256 OS threads, a pthread
//                       barrier for __syncthreads and memcpy for the TMA bulk copies of the encoder-only weight-slab walk
//   svad_emu_cell_*     one step of the LSTM cell of the training kernels (svad_train_cell.h), for the float64 autograd check
#include <pthread.h>
#include <sched.h>

#include <atomic>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../silero_vad_b200/csrc/svad_tile.h"
#include "../../silero_vad_b200/csrc/svad_train_cell.h"

using namespace svad;

namespace {
struct Shared {
    std::vector<float> smem;
    pthread_barrier_t bar;
    const float* tape;
    std::atomic<long> issued{0};            // slabs copied into the ring so far
    std::atomic<long> released[kStages];    // per stage: thread arrivals so far
};

template <bool SR16>
struct EmuEnvFeat {
    static constexpr int kNslab = Geo<SR16>::nslab_enc;   // run_cta<..., FEAT = true> walks the encoder slabs only
    Shared* sh;
    int tid_;
    int tid() const { return tid_; }
    float* smem() { return sh->smem.data(); }
    void sync() { pthread_barrier_wait(&sh->bar); }
    void prefetch_l2(const void*) {}
    void issue(long it) {
        const int idx = (int)(it % kNslab), stage = (int)(it % kStages);
        memcpy(sh->smem.data() + SmemMap::stage + stage * SmemMap::stage_floats, sh->tape + Tape<SR16>::slab_off(idx),
               sizeof(float) * Tape<SR16>::slab_len(idx));
    }
    const float* slab_acquire(long it, long total) {
        if (tid_ == 0 && it >= 1 && it + 1 < total) {
            const long prev = it - 1;   // the stage slab it+1 goes into
            while (sh->released[prev % kStages].load(std::memory_order_acquire) < (long)kThreads * (prev / kStages + 1)) sched_yield();
            issue(it + 1);
            sh->issued.store(it + 2, std::memory_order_release);
        }
        while (sh->issued.load(std::memory_order_acquire) <= it) sched_yield();
        return sh->smem.data() + SmemMap::stage + (it % kStages) * SmemMap::stage_floats;
    }
    void slab_done(long it) { sh->released[it % kStages].fetch_add(1, std::memory_order_acq_rel); }
};

template <bool SR16, int RM>
void run_features(const TileArgs& a, int ntiles) {
    Shared sh;
    sh.smem.assign(SmemMap::total_floats, 0.0f);
    sh.tape = a.tape;
    pthread_barrier_init(&sh.bar, nullptr, kThreads);
    {
        EmuEnvFeat<SR16> e0{&sh, 0};
        const long total = (long)ntiles * a.T * EmuEnvFeat<SR16>::kNslab;
        for (int i = 0; i < kStages; i++) sh.released[i] = 0;
        long pre = 0;
        for (long i = 0; i < kStages && i < total; i++) { e0.issue(i); pre = i + 1; }
        sh.issued = pre;
    }
    std::vector<std::thread> th;
    for (int t = 0; t < kThreads; t++)
        th.emplace_back([&, t] {
            EmuEnvFeat<SR16> env{&sh, t};
            run_cta<SR16, RM, float, true>(env, a, 0, 1, ntiles);
        });
    for (auto& x : th) x.join();
    pthread_barrier_destroy(&sh.bar);
}
}  // namespace

// f32 audio [B][L] (L a multiple of n), optional per-row context [B][ctx] -> feat [B][L/n][128]
extern "C" int svad_emu_features(const char* weights, int sr, int rm, int B, long L, const float* audio, const float* ctx_in, float* feat) {
    TensorMap tm;
    std::string err;
    if (!read_container(weights, tm, err)) return -1;
    PackedBranch pb;
    const bool sr16 = sr == 16000;
    if (!(sr16 ? pack_branch<true>(tm, pb, err) : pack_branch<false>(tm, pb, err))) return -2;
    const int n = sr16 ? 512 : 256;
    if (L % n) return -4;
    TileArgs a{};
    a.audio = audio; a.ld = L; a.L = L; a.dec = 1; a.B = B; a.T = L / n;
    a.ctx_in = ctx_in; a.ctx_ld = sr16 ? 64 : 32;
    a.probs = feat; a.ldp = a.T;   // features mode: [B][T][128]
    a.tape = pb.tape.data(); a.consts = pb.consts.data();
    const int ntiles = (B + 4 * rm - 1) / (4 * rm);
    if (rm == 8) sr16 ? run_features<true, 8>(a, ntiles) : run_features<false, 8>(a, ntiles);
    else if (rm == 4) sr16 ? run_features<true, 4>(a, ntiles) : run_features<false, 4>(a, ntiles);
    else return -3;
    return 0;
}

extern "C" void svad_emu_cell_fwd(const float* pre, float c_prev, float* out) {   // pre[4] (i, f, g, o) -> out: i f g o c h
    const CellFwd r = lstm_cell_fwd(pre[0], pre[1], pre[2], pre[3], c_prev);
    out[0] = r.i; out[1] = r.f; out[2] = r.g; out[3] = r.o; out[4] = r.c; out[5] = r.h;
}
extern "C" void svad_emu_cell_bwd(const float* act, float c_prev, float c, float dh, float dc, float* out) {   // -> dpre[4], dc_prev
    const CellBwd r = lstm_cell_bwd(act[0], act[1], act[2], act[3], c_prev, c, dh, dc);
    out[0] = r.d_i; out[1] = r.d_f; out[2] = r.d_g; out[3] = r.d_o; out[4] = r.dc_prev;
}
