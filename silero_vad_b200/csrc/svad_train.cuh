// svad_train.cuh -- kernels for fine-tuning the VAD decoder (LSTMCell(128 -> 128) + Dropout -> ReLU -> Conv1d(128 -> 1) -> Sigmoid)
// on frozen encoder features, and the (enter, exit) threshold grid of the threshold search.  Instantiated in svad_api.cu.
//
// B streams x T steps, features x[B][T][128] (post-ReLU enc3 rows, svad_features_device).  The parameters are read from the
// caller's device tensors on every call (torch parameters updated by any optimizer):
//   W_ih, W_hh [512][128], b_ih, b_hh [512], w_head [128], b_head [1]; gate rows in torch.lstm_cell order i, f, g, o.
//
// Forward   dec_inproj  Gx[n][r] = b_ih[r] + b_hh[r] + x[n] . W_ih[r]          (n = b T + t; one parallel GEMM over all steps)
//           dec_fwd     the serial scan.  One CTA of 512 threads per group of G streams (G = 1, 2, 4 from B and the SM count);
//                       thread r owns gate row r: W_hh[r][0..96) is resident in shared memory (192 KB, k-major), W_hh[r][96..128)
//                       in 32 registers, so no weight byte leaves the SM during the scan.  Per step: gate row r of the G streams
//                       (h_{t-1} broadcast from shared memory) -> barrier -> thread (g, j) updates unit j of stream g (c stays
//                       in its register) and the head partial -> barrier -> probabilities.
//           Tape (optional, for the backward pass): activated gates [B][T][512] and c [B][T][128]; h = o tanh(c) is recomputed.
// Backward  dec_bwd     the reverse scan, same ownership with W_hh in row-major halves: thread (q, j) owns column j of the gate
//                       block q (rows 128 q + [0, 96) in shared memory, rows 128 q + [96, 128) in registers), so that
//                       dh_{t-1} = dgates_t . W_hh is four partials per unit summed in a fixed order.  Writes dgates [B][T][512]
//                       and per-stream head-gradient partials.
//           dec_wgrad   dW_ih = sum_n dgates[n]^T x[n], dW_hh = sum_n dgates[n]^T h_{n-1}, db = sum_n dgates[n]: 64 x 64 output
//                       tiles over fixed chunks of the n range, partials to the workspace;
//           dec_reduce  sums the chunk partials (and the per-stream head partials) in index order.
// No float atomics anywhere: two calls give bit-identical gradients.
#pragma once
#include "svad_train_cell.h"

namespace svad {

constexpr int kDecThreads = 512;
constexpr int kDecSmemK = 96;                       // rows of the 128-deep recurrent product held in shared memory (rest: registers)
constexpr int kDecRegK = kHid - kDecSmemK;          // 32
constexpr int kWgChunk = 4096;                      // dec_wgrad: rows n per partial (fixed, so results do not depend on the device)

// dynamic shared memory of the scans: the resident W_hh part plus per-step exchange buffers
template <int G>
constexpr size_t dec_fwd_smem_bytes() { return (size_t)(kDecSmemK * kGates + G * kGates + G * kHid + G * 4) * 4; }   // wt, pre, hs, hp
template <int G>
constexpr size_t dec_bwd_smem_bytes() { return (size_t)(kDecSmemK * kGates + G * kGates + 4 * G * kHid) * 4; }      // wb, dgs, part

// ---------------------------------------------------------------- Gx = x W_ih^T + b_ih + b_hh       grid (ceil(N / 64), 8), 256 thr
__global__ void __launch_bounds__(256) dec_inproj(const float* __restrict__ x, const float* __restrict__ w_ih, const float* __restrict__ b_ih,
                                                  const float* __restrict__ b_hh, float* __restrict__ gx, long N) {
    __shared__ __align__(16) float As[64][68];   // [k][m]
    __shared__ __align__(16) float Bs[64][68];   // [k][r]
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const long m0 = (long)blockIdx.x * 64;
    const int r0 = blockIdx.y * 64;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < kHid; k0 += 64) {
        for (int q = threadIdx.x; q < 64 * 64; q += 256) {
            const int mm = q >> 6, kk = q & 63;
            As[kk][mm] = (m0 + mm < N) ? x[(m0 + mm) * kHid + k0 + kk] : 0.0f;
            Bs[kk][mm] = w_ih[(long)(r0 + mm) * kHid + k0 + kk];
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < 64; kk++) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const long m = m0 + ty * 4 + i;
        if (m >= N) continue;
        float4 o;
        float* ov = &o.x;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int r = r0 + tx * 4 + j;
            ov[j] = acc[i][j] + (b_ih[r] + b_hh[r]);
        }
        *reinterpret_cast<float4*>(gx + m * kGates + r0 + tx * 4) = o;
    }
}

// ---------------------------------------------------------------- forward scan                       grid ceil(B / G), 512 threads
template <int G>
__global__ void __launch_bounds__(kDecThreads, 1) dec_fwd(const float* __restrict__ gx, const float* __restrict__ w_hh, const float* __restrict__ w_head,
                                                         const float* __restrict__ b_head, const float* __restrict__ drop, float* __restrict__ probs,
                                                         float* __restrict__ tape_gates, float* __restrict__ tape_c, int B, long T) {
    extern __shared__ __align__(16) float sm[];
    float* wt = sm;                                // [96][512]: W_hh[r][k] at wt[k * 512 + r]
    float* pre = wt + kDecSmemK * kGates;          // [G][512] gate pre-activations of this step
    float* hs = pre + G * kGates;                  // [G][128] h_{t-1}
    float* hp = hs + G * kHid;                     // [G][4] head partials (one per warp of a stream's 128 units)
    const int r = threadIdx.x, b0 = blockIdx.x * G;
    for (int q = threadIdx.x; q < kGates * kDecSmemK; q += kDecThreads) {
        const int rr = q / kDecSmemK, k = q % kDecSmemK;
        wt[k * kGates + rr] = w_hh[(long)rr * kHid + k];
    }
    float wr[kDecRegK];
#pragma unroll
    for (int k = 0; k < kDecRegK; k++) wr[k] = w_hh[(long)r * kHid + kDecSmemK + k];
    for (int q = threadIdx.x; q < G * kHid; q += kDecThreads) hs[q] = 0.0f;
    // unit thread: stream g = tid / 128, unit j = tid % 128
    const int ug = threadIdx.x >> 7, uj = threadIdx.x & (kHid - 1);
    const int ub = b0 + ug;
    const bool unit = ug < G && ub < B;
    const float wh = w_head[uj], bh = b_head[0];
    float c = 0.0f;
    __syncthreads();
    for (long t = 0; t < T; t++) {
        float acc[G];
#pragma unroll
        for (int g = 0; g < G; g++) acc[g] = (b0 + g < B) ? gx[((long)(b0 + g) * T + t) * kGates + r] : 0.0f;
#pragma unroll 4
        for (int k = 0; k < kDecSmemK; k += 4) {
            const float w0 = wt[k * kGates + r], w1 = wt[(k + 1) * kGates + r], w2 = wt[(k + 2) * kGates + r], w3 = wt[(k + 3) * kGates + r];
#pragma unroll
            for (int g = 0; g < G; g++) {
                const float4 h = *reinterpret_cast<const float4*>(hs + g * kHid + k);
                acc[g] = fmaf(w0, h.x, acc[g]); acc[g] = fmaf(w1, h.y, acc[g]); acc[g] = fmaf(w2, h.z, acc[g]); acc[g] = fmaf(w3, h.w, acc[g]);
            }
        }
#pragma unroll
        for (int k = 0; k < kDecRegK; k += 4) {
#pragma unroll
            for (int g = 0; g < G; g++) {
                const float4 h = *reinterpret_cast<const float4*>(hs + g * kHid + kDecSmemK + k);
                acc[g] = fmaf(wr[k], h.x, acc[g]); acc[g] = fmaf(wr[k + 1], h.y, acc[g]); acc[g] = fmaf(wr[k + 2], h.z, acc[g]); acc[g] = fmaf(wr[k + 3], h.w, acc[g]);
            }
        }
#pragma unroll
        for (int g = 0; g < G; g++) pre[g * kGates + r] = acc[g];
        __syncthreads();   // pre complete; every read of h_{t-1} done
        if (unit) {
            const float* pg = pre + ug * kGates;
            const CellFwd cf = lstm_cell_fwd(pg[uj], pg[kHid + uj], pg[2 * kHid + uj], pg[3 * kHid + uj], c);
            c = cf.c;
            hs[ug * kHid + uj] = cf.h;
            const long n = (long)ub * T + t;
            if (tape_gates) {
                float* tg = tape_gates + n * kGates;
                tg[uj] = cf.i; tg[kHid + uj] = cf.f; tg[2 * kHid + uj] = cf.g; tg[3 * kHid + uj] = cf.o;
                tape_c[n * kHid + uj] = cf.c;
            }
            const float m = drop ? drop[n * kHid + uj] : 1.0f;
            float part = wh * relu(cf.h * m);
#pragma unroll
            for (int s = 16; s >= 1; s >>= 1) part += __shfl_xor_sync(0xffffffffu, part, s);
            if ((uj & 31) == 0) hp[ug * 4 + (uj >> 5)] = part;
        }
        __syncthreads();   // h_t and the head partials complete
        if (threadIdx.x < G && b0 + (int)threadIdx.x < B) {
            const float* p = hp + threadIdx.x * 4;
            probs[(long)(b0 + threadIdx.x) * T + t] = sigmoid_acc(bh + ((p[0] + p[1]) + (p[2] + p[3])));
        }
    }
}

// ---------------------------------------------------------------- backward scan                      grid ceil(B / G), 512 threads
// head_part [B][129]: per stream sum_t ds_t relu(h_t m_t) (128) and sum_t ds_t.
template <int G>
__global__ void __launch_bounds__(kDecThreads, 1) dec_bwd(const float* __restrict__ w_hh, const float* __restrict__ w_head, const float* __restrict__ drop,
                                                         const float* __restrict__ probs, const float* __restrict__ dprobs,
                                                         const float* __restrict__ tape_gates, const float* __restrict__ tape_c,
                                                         float* __restrict__ dgates, float* __restrict__ head_part, int B, long T) {
    extern __shared__ __align__(16) float sm[];
    float* wb = sm;                                // [4][96][128]: W_hh[128 q + rr][j] at wb[(q * 96 + rr) * 128 + j]
    float* dgs = wb + kDecSmemK * kGates;          // [G][512] dgates of this step
    float* part = dgs + G * kGates;                // [4][G][128] partials of dh_{t-1}, one per gate block q
    const int q = threadIdx.x >> 7, j = threadIdx.x & (kHid - 1), b0 = blockIdx.x * G;
    for (int i = threadIdx.x; i < 4 * kDecSmemK * kHid; i += kDecThreads) {
        const int qq = i / (kDecSmemK * kHid), rr = (i / kHid) % kDecSmemK, jj = i % kHid;
        wb[i] = w_hh[(long)(qq * kHid + rr) * kHid + jj];
    }
    float wr[kDecRegK];
#pragma unroll
    for (int k = 0; k < kDecRegK; k++) wr[k] = w_hh[(long)(q * kHid + kDecSmemK + k) * kHid + j];
    for (int i = threadIdx.x; i < 4 * G * kHid; i += kDecThreads) part[i] = 0.0f;
    const int ug = q, ub = b0 + ug;              // unit thread (g, j) = (q, j) for q < G
    const bool unit = ug < G && ub < B;
    const float wh = w_head[j];
    float dc = 0.0f, dw_acc = 0.0f, db_acc = 0.0f;
    __syncthreads();
    for (long t = T - 1; t >= 0; t--) {
        if (unit) {
            const long n = (long)ub * T + t;
            const float* tg = tape_gates + n * kGates;
            const float gi = tg[j], gf = tg[kHid + j], gg = tg[2 * kHid + j], go = tg[3 * kHid + j];
            const float c = tape_c[n * kHid + j], c_prev = t > 0 ? tape_c[(n - 1) * kHid + j] : 0.0f;
            const float p = probs[n], ds = dprobs[n] * (p * (1.0f - p));
            const float m = drop ? drop[n * kHid + j] : 1.0f;
            const float z = go * tanhf(c) * m;
            const float* pp = part + ug * kHid + j;
            float dh = ((pp[0] + pp[G * kHid]) + pp[2 * G * kHid]) + pp[3 * G * kHid];   // dgates_{t+1} . W_hh, fixed order
            if (z > 0.0f) dh = fmaf(ds * wh, m, dh);
            dw_acc = fmaf(ds, relu(z), dw_acc);
            db_acc += ds;
            const CellBwd cb = lstm_cell_bwd(gi, gf, gg, go, c_prev, c, dh, dc);
            dc = cb.dc_prev;
            float* dg = dgs + ug * kGates;
            dg[j] = cb.d_i; dg[kHid + j] = cb.d_f; dg[2 * kHid + j] = cb.d_g; dg[3 * kHid + j] = cb.d_o;
            float* dgo = dgates + n * kGates;
            dgo[j] = cb.d_i; dgo[kHid + j] = cb.d_f; dgo[2 * kHid + j] = cb.d_g; dgo[3 * kHid + j] = cb.d_o;
        }
        __syncthreads();   // dgates_t complete; every read of the partials done
        float acc[G];
#pragma unroll
        for (int g = 0; g < G; g++) acc[g] = 0.0f;
        const float* wq = wb + q * kDecSmemK * kHid + j;
#pragma unroll 4
        for (int rr = 0; rr < kDecSmemK; rr += 4) {
            const float w0 = wq[rr * kHid], w1 = wq[(rr + 1) * kHid], w2 = wq[(rr + 2) * kHid], w3 = wq[(rr + 3) * kHid];
#pragma unroll
            for (int g = 0; g < G; g++) {
                const float4 d = *reinterpret_cast<const float4*>(dgs + g * kGates + q * kHid + rr);
                acc[g] = fmaf(w0, d.x, acc[g]); acc[g] = fmaf(w1, d.y, acc[g]); acc[g] = fmaf(w2, d.z, acc[g]); acc[g] = fmaf(w3, d.w, acc[g]);
            }
        }
#pragma unroll
        for (int k = 0; k < kDecRegK; k += 4) {
#pragma unroll
            for (int g = 0; g < G; g++) {
                const float4 d = *reinterpret_cast<const float4*>(dgs + g * kGates + q * kHid + kDecSmemK + k);
                acc[g] = fmaf(wr[k], d.x, acc[g]); acc[g] = fmaf(wr[k + 1], d.y, acc[g]); acc[g] = fmaf(wr[k + 2], d.z, acc[g]); acc[g] = fmaf(wr[k + 3], d.w, acc[g]);
            }
        }
#pragma unroll
        for (int g = 0; g < G; g++) part[(q * G + g) * kHid + j] = acc[g];
        __syncthreads();   // partials complete; dgs free
    }
    if (unit) {
        head_part[(long)ub * (kHid + 1) + j] = dw_acc;
        if (j == 0) head_part[(long)ub * (kHid + 1) + kHid] = db_acc;
    }
}

// ---------------------------------------------------------------- weight-gradient partials          grid (8, 4, nchunks), 256 threads
// wg_part[chunk][512][257]: columns 0..127 dW_ih, 128..255 dW_hh, 256 db; chunk = rows n in [chunk * kWgChunk, ...).
__global__ void __launch_bounds__(256) dec_wgrad(const float* __restrict__ dgates, const float* __restrict__ x, const float* __restrict__ tape_gates,
                                                 const float* __restrict__ tape_c, float* __restrict__ wg_part, long T, long N) {
    __shared__ __align__(16) float As[16][64];   // [n][r]
    __shared__ __align__(16) float Bs[16][64];   // [n][k]
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int r0 = blockIdx.x * 64, k0 = blockIdx.y * 64;   // k0 < 128: x columns, else h_{t-1} columns
    const long n_lo = (long)blockIdx.z * kWgChunk, n_hi = n_lo + kWgChunk < N ? n_lo + kWgChunk : N;
    float acc[4][4] = {}, dbacc[4] = {};
    for (long n0 = n_lo; n0 < n_hi; n0 += 16) {
        for (int qd = threadIdx.x; qd < 16 * 64; qd += 256) {
            const int nn = qd >> 6, c = qd & 63;
            const long n = n0 + nn;
            float a = 0.0f, b = 0.0f;
            if (n < n_hi) {
                a = dgates[n * kGates + r0 + c];
                if (k0 < kHid) b = x[n * kHid + k0 + c];
                else if (n % T) b = tape_gates[(n - 1) * kGates + 3 * kHid + (k0 - kHid) + c] * tanhf(tape_c[(n - 1) * kHid + (k0 - kHid) + c]);
            }
            As[nn][c] = a;
            Bs[nn][c] = b;
        }
        __syncthreads();
#pragma unroll
        for (int nn = 0; nn < 16; nn++) {
            const float4 a = *reinterpret_cast<const float4*>(&As[nn][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[nn][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; i++) {
                dbacc[i] += av[i];
#pragma unroll
                for (int jj = 0; jj < 4; jj++) acc[i][jj] = fmaf(av[i], bv[jj], acc[i][jj]);
            }
        }
        __syncthreads();
    }
    float* out = wg_part + (long)blockIdx.z * kGates * (2 * kHid + 1);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int r = r0 + ty * 4 + i;
#pragma unroll
        for (int jj = 0; jj < 4; jj++) out[(long)r * (2 * kHid + 1) + k0 + tx * 4 + jj] = acc[i][jj];
        if (blockIdx.y == 0 && tx == 0) out[(long)r * (2 * kHid + 1) + 2 * kHid] = dbacc[i];
    }
}

// ---------------------------------------------------------------- fixed-order sums of the partials
__global__ void dec_reduce(const float* __restrict__ wg_part, int nchunks, const float* __restrict__ head_part, int B, float* __restrict__ dw_ih,
                           float* __restrict__ dw_hh, float* __restrict__ db, float* __restrict__ dw_head, float* __restrict__ db_head) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    constexpr int W = 2 * kHid + 1;
    if (i < kGates * W) {
        float s = 0.0f;
        for (int c = 0; c < nchunks; c++) s += wg_part[(long)c * kGates * W + i];
        const int r = i / W, k = i % W;
        if (k < kHid) dw_ih[r * kHid + k] = s;
        else if (k < 2 * kHid) dw_hh[r * kHid + k - kHid] = s;
        else db[r] = s;
    } else if (i < kGates * W + kHid + 1) {
        const int j = i - kGates * W;
        float s = 0.0f;
        for (int b = 0; b < B; b++) s += head_part[(long)b * (kHid + 1) + j];
        if (j < kHid) dw_head[j] = s; else db_head[0] = s;
    }
}

// ---------------------------------------------------------------- threshold grid                     grid files, 192 threads
// Thread p < 190 runs the hysteresis scan of pair p (enter index a, exit index e < a, a outer / e inner as in the search loop)
// over the file's probabilities widened to double, and counts the chunks whose decision equals the target.
constexpr int kGridN = 20, kGridPairs = kGridN * (kGridN - 1) / 2, kGridStage = 4096;
__global__ void __launch_bounds__(192) threshold_grid(const float* __restrict__ probs, const float* __restrict__ gts, const long long* __restrict__ offsets,
                                                      const double* __restrict__ grid, long long* __restrict__ counts) {
    __shared__ float ps[kGridStage];
    __shared__ float gs[kGridStage];
    const int p = threadIdx.x;
    int a = 1, e = p;
    while (e >= a) { e -= a; a++; }
    const bool active = p < kGridPairs;
    const double enter = active ? grid[a] : 2.0, exit_ = active ? grid[e] : -1.0;
    const long long lo = offsets[blockIdx.x], hi = offsets[blockIdx.x + 1];
    bool speech = false;
    long long hits = 0;
    for (long long s0 = lo; s0 < hi; s0 += kGridStage) {
        const int len = (int)(hi - s0 < kGridStage ? hi - s0 : kGridStage);
        __syncthreads();
        for (int i = threadIdx.x; i < len; i += blockDim.x) { ps[i] = probs[s0 + i]; gs[i] = gts[s0 + i]; }
        __syncthreads();
        if (active)
            for (int i = 0; i < len; i++) {
                const double v = (double)ps[i];
                if (v >= enter) speech = true;
                else if (v <= exit_) speech = false;
                hits += (gs[i] == (speech ? 1.0f : 0.0f));
            }
    }
    if (active) counts[(long long)blockIdx.x * kGridPairs + p] = hits;
}

}  // namespace svad
