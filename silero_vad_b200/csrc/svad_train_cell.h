// svad_train_cell.h -- per-unit arithmetic of the decoder-training kernels (svad_train.cuh): one LSTM cell step forward and
// backward, and the head.  Plain fp32 with accurate expf / tanhf (not the MUFU approximations of the inference kernels): the
// gradients are judged against torch autograd.  Compiles for the device and, through tests/emu, as plain C++ so that one step
// can be checked against torch in float64 without a GPU.
//
// sigmoid_acc is svad_core.h's.
//
// Cell (torch.lstm_cell, gate order i, f, g, o):  c = f c' + i g,  h = o tanh(c).
// Head (VADDecoderRNNJIT.decoder: Dropout -> ReLU -> Conv1d(128, 1, 1) -> Sigmoid):  p = sigmoid(b + sum_j w_j relu(h_j m_j)),
// m the dropout multiplier (0 or 1 / (1 - p_drop); 1 in eval mode).  The recurrent h is not dropped.
#pragma once
#include "svad_core.h"

namespace svad {

struct CellFwd { float i, f, g, o, c, h; };

// pre-activations of the four gates and c_{t-1} -> activated gates, c_t, h_t
SVAD_HD CellFwd lstm_cell_fwd(float pi, float pf, float pg, float po, float c_prev) {
    CellFwd r;
    r.i = sigmoid_acc(pi);
    r.f = sigmoid_acc(pf);
    r.g = tanhf(pg);
    r.o = sigmoid_acc(po);
    r.c = fmaf(r.f, c_prev, r.i * r.g);
    r.h = r.o * tanhf(r.c);
    return r;
}

struct CellBwd { float d_i, d_f, d_g, d_o, dc_prev; };

// activated gates, c_{t-1}, c_t and the gradients arriving at h_t (head + recurrence) and at c_t (from step t+1) -> gradients of
// the four pre-activations and of c_{t-1}
SVAD_HD CellBwd lstm_cell_bwd(float i, float f, float g, float o, float c_prev, float c, float dh, float dc) {
    const float tc = tanhf(c);
    const float dct = fmaf(dh * o, 1.0f - tc * tc, dc);
    CellBwd r;
    r.d_o = dh * tc * (o * (1.0f - o));
    r.d_i = dct * g * (i * (1.0f - i));
    r.d_f = dct * c_prev * (f * (1.0f - f));
    r.d_g = dct * i * (1.0f - g * g);
    r.dc_prev = dct * f;
    return r;
}

}  // namespace svad
