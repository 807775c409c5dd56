// Recurrent kernels of the projected TT-LSTM (LSTMP, the `proj_size` of torch.nn.LSTM):
//
//   m_t = o_t * tanh(c_t)      (H)
//   h_t = W_hr m_t             (P < H)    h_t is the layer output and the next step's hh input
//
// W_hr is a second TT chain (H -> P) whose cores are staged in shared memory next to W_hh, and every step runs it
// between the gate math and the next step's hh chain.  These are the runtime-shape kernels k_rnn_fwd / k_rnn_bwd
// (tt_kernels.cuh) with that chain added; LSTM only.  Launch code is in ttrnn_capi.cu.
#pragma once
#include "tt_kernels.cuh"

struct RnnFwdProjArgs {
    ChainPlan p;            // hh chain: P -> 4H
    ChainPlan q;            // projection chain W_hr: H -> P
    int tile[TT_MAX_D], tile_q[TT_MAX_D];
    int R, H, P;
    int steps;              // timesteps in this launch
    long long B;
    const float *xg;        // ih projection of this chunk: row b, step t at xg + (b*xg_bstride + t*4H)
    long long xg_bstride;
    const float *cores;     // hh core blob
    const float *cores_q;   // hr core blob
    const float *h_in;      // (B,P) or null = zeros
    const float *c_in;      // (B,H) or null = zeros
    float *out;             // h_t of this chunk: out + b*out_bstride + t*P
    long long out_bstride;
    float *c_save;          // c_t: c_save + b*c_bstride + t*H, or null (inference)
    long long c_bstride;
    float *h_out;           // (B,P) state after the last step of this launch
    float *c_out;           // (B,H)
};

// ---------------------------------------------------------------------------
// Persistent projected forward.  Shared memory:
//   [W_hh][W_hr][c state R*H][xg tile R*4H][G R*p.g_BS][h slot R*p.in_BS][m slot R*q.in_BS][Gq R*q.g_BS][P][Q]
// P / Q are the ping-pong slots of whichever chain runs (sized for the larger of the two).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(TT_NTHREADS)
k_rnn_fwd_proj(const __grid_constant__ RnnFwdProjArgs a) {
    extern __shared__ __align__(16) float smem[];
    const ChainPlan &p = a.p, &q = a.q;
    const int tid = threadIdx.x;
    const int H = a.H, P = a.P, GH = 4 * a.H, R = a.R;
    float *wsm = smem;
    float *wsq = wsm + p.w_floats;
    float *csm = wsq + q.w_floats;
    float *xgs = csm + tt_round4(R * H);
    float *g = xgs + tt_round4(R * GH);
    float *hin = g + R * p.g_BS;
    float *min_ = hin + R * p.in_BS;
    float *gq = min_ + R * q.in_BS;
    float *PP = gq + R * q.g_BS;
    const int pp0 = p.pp_floats[0] > q.pp_floats[0] ? p.pp_floats[0] : q.pp_floats[0];
    float *QQ = PP + R * pp0;
    const int hBS = p.st[p.d - 1].BS, mBS = q.st[q.d - 1].BS;

    tt_stage_weights(p, a.cores, wsm, tid, TT_NTHREADS);
    tt_stage_weights(q, a.cores_q, wsq, tid, TT_NTHREADS);
    const long long ntiles = (a.B + R - 1) / R;
    for (long long tile_i = blockIdx.x; tile_i < ntiles; tile_i += gridDim.x) {
        const long long row0 = tile_i * R;
        __syncthreads();
        for (int e = tid; e < R * P; e += TT_NTHREADS) {
            const int b = e / P, j = e - b * P;
            const long long row = row0 + b;
            hin[b * hBS + tt_in_index(p, j)] = (row < a.B && a.h_in) ? __ldg(a.h_in + row * P + j) : 0.f;
        }
        for (int e = tid; e < R * H; e += TT_NTHREADS) {
            const long long row = row0 + e / H;
            csm[e] = (row < a.B && a.c_in) ? __ldg(a.c_in + row * H + (e % H)) : 0.f;
        }
        __syncthreads();

        const bool vec16 = (GH % 4 == 0);
        for (int t = 0; t < a.steps; ++t) {
            if (vec16) {
                for (int e = tid * 4; e < R * GH; e += TT_NTHREADS * 4) {
                    const int b = e / GH, c = e - b * GH;
                    if (row0 + b < a.B) tt_cp_async16(xgs + e, a.xg + (row0 + b) * a.xg_bstride + (long long)t * GH + c);
                }
            } else {
                for (int e = tid; e < R * GH; e += TT_NTHREADS) {
                    const int b = e / GH, c = e - b * GH;
                    if (row0 + b < a.B) tt_cp_async4(xgs + e, a.xg + (row0 + b) * a.xg_bstride + (long long)t * GH + c);
                }
            }
            // (1) hh chain on h_{t-1} (P inputs)
            for (int k = p.d - 1; k >= 0; --k) {
                const StagePlan &s = p.st[k];
                const float *X = (s.xpp == 0) ? hin : (s.xpp == 1 ? PP : QQ);
                float *Y = (k == 0) ? g : (p.st[k - 1].xpp == 1 ? PP : QQ);
                tt_stage_fwd(s, a.tile[k], R, X, wsm + s.w_off, Y, tid, TT_NTHREADS);
                if (k == 0) tt_cp_async_wait_all();
                __syncthreads();
            }
            // (2) gate math: c_t, and m_t into the projection chain's input slot
            for (int e = tid; e < R * H; e += TT_NTHREADS) {
                const int b = e / H, h = e - b * H;
                const long long row = row0 + b;
                float mv = 0.f;
                if (row < a.B) {
                    const float *gb = g + b * p.g_BS;
                    const float *xb = xgs + b * GH;
                    const float ig = tt_sigmoid(gb[tt_g_index(p, h)] + xb[h]);
                    const float fg = tt_sigmoid(gb[tt_g_index(p, H + h)] + xb[H + h]);
                    const float gg = tanhf(gb[tt_g_index(p, 2 * H + h)] + xb[2 * H + h]);
                    const float og = tt_sigmoid(gb[tt_g_index(p, 3 * H + h)] + xb[3 * H + h]);
                    const float cnew = fg * csm[e] + ig * gg;
                    mv = og * tanhf(cnew);
                    csm[e] = cnew;
                    if (a.c_save) a.c_save[row * a.c_bstride + (long long)t * H + h] = cnew;
                }
                min_[b * mBS + tt_in_index(q, h)] = mv;
            }
            __syncthreads();
            // (3) projection chain: h_t = W_hr m_t
            tt_chain_fwd_pp(q, a.tile_q, R, min_, PP, QQ, gq, wsq, tid);
            // (4) h_t -> out and the hh input slot
            for (int e = tid; e < R * P; e += TT_NTHREADS) {
                const int b = e / P, j = e - b * P;
                const long long row = row0 + b;
                const float hv = gq[b * q.g_BS + tt_g_index(q, j)];
                hin[b * hBS + tt_in_index(p, j)] = hv;
                if (row < a.B) a.out[row * a.out_bstride + (long long)t * P + j] = hv;
            }
            __syncthreads();
        }
        for (int e = tid; e < R * P; e += TT_NTHREADS) {
            const int b = e / P, j = e - b * P;
            const long long row = row0 + b;
            if (row < a.B && a.h_out) a.h_out[row * P + j] = hin[b * hBS + tt_in_index(p, j)];
        }
        for (int e = tid; e < R * H; e += TT_NTHREADS) {
            const long long row = row0 + e / H;
            if (row < a.B && a.c_out) a.c_out[row * H + (e % H)] = csm[e];
        }
    }
}

struct RnnBwdProjArgs {
    ChainPlan p, q;         // hh chain, projection chain (slot placement applied)
    int tile[TT_MAX_D], tile_bd[TT_MAX_D], mg[TT_MAX_D];
    int tile_q[TT_MAX_D], tile_bd_q[TT_MAX_D], mg_q[TT_MAX_D];
    int R, H, P;
    int t0, steps, T;       // this launch covers timesteps [t0, t0+steps) of a length-T sequence
    long long B;
    float *xg;              // chunk buffer (b, steps, 4H): ih projection in, delta_ih out
    long long xg_bstride;
    const float *cores, *cores_q;
    const float *hs;        // (B,T,P) outputs of this layer
    const float *cs;        // (B,T,H) cell states of this layer
    const float *h0;        // (B,P) or null
    const float *c0;        // (B,H) or null
    const float *dhs;       // (B,T,P) gradient wrt this layer's outputs, or null
    const float *dh_in;     // (B,P) gradient flowing into h_{t0+steps-1} from later steps, or null
    const float *dc_in;     // (B,H) same for c, or null
    float *dh_out;          // (B,P) gradient wrt h_{t0-1}
    float *dc_out;          // (B,H)
    float *partial;         // [gridDim.x][p.core_floats + q.core_floats]: hh core grads, then hr core grads
    float *spill;           // [gridDim.x][R * (p.spill_floats + q.spill_floats)] or null
};

// ---------------------------------------------------------------------------
// Reverse-time persistent BPTT of the projected LSTM.  Shared memory:
//   [W_hh][dW_hh][W_hr][dW_hr][hh x slots R*p.all_floats][hr x slots R*q.all_floats][G R*p.g_BS][Gq R*q.g_BS]
//   [xg tile R*4H][dh chain R*p.in_BS][dh direct R*P][dc R*H][c_prev R*H]
// Per step: recompute the hh chain and the gates (m_t), run the projection chain forward keeping its X_k, run it
// backward from dY_0 = the total dh_t (core gradients of W_hr, dm_t in the m slot), the gate backward with dm_t, and
// the hh chain backward (core gradients of W_hh, dh_{t-1}).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(TT_NTHREADS)
k_rnn_bwd_proj(const __grid_constant__ RnnBwdProjArgs a) {
    extern __shared__ __align__(16) float smem[];
    const ChainPlan &p = a.p, &q = a.q;
    const int tid = threadIdx.x, R = a.R, H = a.H, P = a.P, GH = 4 * a.H;
    float *wsm = smem;
    float *dws = wsm + p.w_floats;
    float *wsq = dws + p.w_floats;
    float *dwq = wsq + q.w_floats;
    float *xa = dwq + q.w_floats;
    float *xaq = xa + R * p.all_floats;
    float *g = xaq + R * q.all_floats;
    float *gq = g + R * p.g_BS;
    float *xgs = gq + R * q.g_BS;
    float *dhc = xgs + tt_round4(R * GH);
    float *dhd = dhc + R * p.in_BS;
    float *dcs = dhd + tt_round4(R * P);
    float *cps = dcs + tt_round4(R * H);
    float *spill = a.spill ? a.spill + (long long)blockIdx.x * R * (p.spill_floats + q.spill_floats) : nullptr;
    float *spillq = spill ? spill + (long long)R * p.spill_floats : nullptr;

    const int hBS = p.st[p.d - 1].BS, mBS = q.st[q.d - 1].BS;
    float *hslot = tt_slot(p, p.d - 1, R, xa, spill);
    float *mslot = tt_slot(q, q.d - 1, R, xaq, spillq);
    const bool vec16 = (GH % 4 == 0);

    tt_stage_weights(p, a.cores, wsm, tid, TT_NTHREADS);
    tt_stage_weights(q, a.cores_q, wsq, tid, TT_NTHREADS);
    for (int e = tid; e < p.w_floats; e += TT_NTHREADS) dws[e] = 0.f;
    for (int e = tid; e < q.w_floats; e += TT_NTHREADS) dwq[e] = 0.f;
    const long long ntiles = (a.B + R - 1) / R;
    for (long long tile_i = blockIdx.x; tile_i < ntiles; tile_i += gridDim.x) {
        const long long row0 = tile_i * R;
        __syncthreads();
        for (int e = tid; e < R * p.in_BS; e += TT_NTHREADS) dhc[e] = 0.f;
        for (int e = tid; e < R * P; e += TT_NTHREADS) {
            const long long row = row0 + e / P;
            dhd[e] = (row < a.B && a.dh_in) ? __ldg(a.dh_in + row * P + (e % P)) : 0.f;
        }
        for (int e = tid; e < R * H; e += TT_NTHREADS) {
            const long long row = row0 + e / H;
            dcs[e] = (row < a.B && a.dc_in) ? __ldg(a.dc_in + row * H + (e % H)) : 0.f;
        }
        __syncthreads();
        for (int t = a.steps - 1; t >= 0; --t) {
            const int tg = a.t0 + t;
            // ---- load h_{t-1} (P), c_{t-1} (H); prefetch the ih projection of step t
            if (vec16) {
                for (int e = tid * 4; e < R * GH; e += TT_NTHREADS * 4) {
                    const int b = e / GH, c = e - b * GH;
                    if (row0 + b < a.B) tt_cp_async16(xgs + e, a.xg + (row0 + b) * a.xg_bstride + (long long)t * GH + c);
                }
            } else {
                for (int e = tid; e < R * GH; e += TT_NTHREADS) {
                    const int b = e / GH, c = e - b * GH;
                    if (row0 + b < a.B) tt_cp_async4(xgs + e, a.xg + (row0 + b) * a.xg_bstride + (long long)t * GH + c);
                }
            }
            for (int e = tid; e < R * P; e += TT_NTHREADS) {
                const int b = e / P, j = e - b * P;
                const long long row = row0 + b;
                float hv = 0.f;
                if (row < a.B) {
                    if (tg > 0) hv = __ldg(a.hs + (row * a.T + (tg - 1)) * P + j);
                    else if (a.h0) hv = __ldg(a.h0 + row * P + j);
                }
                hslot[b * hBS + tt_in_index(p, j)] = hv;
            }
            for (int e = tid; e < R * H; e += TT_NTHREADS) {
                const int b = e / H, h = e - b * H;
                const long long row = row0 + b;
                float cv = 0.f;
                if (row < a.B) {
                    if (tg > 0) cv = __ldg(a.cs + (row * a.T + (tg - 1)) * H + h);
                    else if (a.c0) cv = __ldg(a.c0 + row * H + h);
                }
                cps[e] = cv;
            }
            __syncthreads();
            // ---- (1) recompute the hh chain, keeping every intermediate
            for (int k = p.d - 1; k >= 0; --k) {
                const StagePlan &s = p.st[k];
                const float *X = tt_slot(p, k, R, xa, spill);
                float *Y = (k == 0) ? g : tt_slot(p, k - 1, R, xa, spill);
                tt_stage_fwd(s, a.tile[k], R, X, wsm + s.w_off, Y, tid, TT_NTHREADS);
                if (k == 0) tt_cp_async_wait_all();
                __syncthreads();
            }
            // ---- gates -> m_t into the projection chain's input slot
            for (int e = tid; e < R * H; e += TT_NTHREADS) {
                const int b = e / H, h = e - b * H;
                float mv = 0.f;
                if (row0 + b < a.B) {
                    const float *gb = g + b * p.g_BS;
                    const float *xb = xgs + b * GH;
                    const float ig = tt_sigmoid(gb[tt_g_index(p, h)] + xb[h]);
                    const float fg = tt_sigmoid(gb[tt_g_index(p, H + h)] + xb[H + h]);
                    const float gg = tanhf(gb[tt_g_index(p, 2 * H + h)] + xb[2 * H + h]);
                    const float og = tt_sigmoid(gb[tt_g_index(p, 3 * H + h)] + xb[3 * H + h]);
                    mv = og * tanhf(fg * cps[e] + ig * gg);
                }
                mslot[b * mBS + tt_in_index(q, h)] = mv;
            }
            __syncthreads();
            // ---- (2) projection chain forward, keeping X_k (its output h_t is not needed)
            tt_chain_fwd_keep(q, a.tile_q, R, xaq, spillq, gq, wsq, /*kstop=*/1, tid);
            // ---- (3) dY_0 = total dh_t: direct (d_hT at the last step) + chain term from step t+1 + dhs[t]
            for (int e = tid; e < R * P; e += TT_NTHREADS) {
                const int b = e / P, j = e - b * P;
                const long long row = row0 + b;
                float dh = 0.f;
                if (row < a.B) {
                    dh = dhd[e] + dhc[b * hBS + tt_in_index(p, j)];
                    if (a.dhs) dh += __ldg(a.dhs + (row * a.T + tg) * P + j);
                }
                gq[b * q.g_BS + tt_g_index(q, j)] = dh;
                dhd[e] = 0.f;
            }
            __syncthreads();
            //      projection chain backward: W_hr core gradients, dm_t in place of m_t
            tt_chain_bwd(q, a.tile_bd_q, a.mg_q, R, xaq, spillq, gq, mslot, wsq, dwq, true, tid);
            // ---- (4) gate backward with dm_t; G <- delta_hh, xg (global) <- delta_ih
            for (int e = tid; e < R * H; e += TT_NTHREADS) {
                const int b = e / H, h = e - b * H;
                const long long row = row0 + b;
                float *gb = g + b * p.g_BS;
                const int gi0 = tt_g_index(p, h), gi1 = tt_g_index(p, H + h), gi2 = tt_g_index(p, 2 * H + h),
                          gi3 = tt_g_index(p, 3 * H + h);
                if (row >= a.B) {
                    gb[gi0] = 0.f; gb[gi1] = 0.f; gb[gi2] = 0.f; gb[gi3] = 0.f;
                    continue;
                }
                const float *xb = xgs + b * GH;
                const float dm = mslot[b * mBS + tt_in_index(q, h)];
                const float ig = tt_sigmoid(gb[gi0] + xb[h]);
                const float fg = tt_sigmoid(gb[gi1] + xb[H + h]);
                const float gg = tanhf(gb[gi2] + xb[2 * H + h]);
                const float og = tt_sigmoid(gb[gi3] + xb[3 * H + h]);
                const float cprev = cps[e];
                const float cnew = fg * cprev + ig * gg;
                const float tc = tanhf(cnew);
                const float dc = dcs[e] + dm * og * (1.0f - tc * tc);
                const float d_i = dc * gg * ig * (1.0f - ig);
                const float d_f = dc * cprev * fg * (1.0f - fg);
                const float d_g = dc * ig * (1.0f - gg * gg);
                const float d_o = dm * tc * og * (1.0f - og);
                dcs[e] = dc * fg;
                gb[gi0] = d_i; gb[gi1] = d_f; gb[gi2] = d_g; gb[gi3] = d_o;
                float *dxg = a.xg + row * a.xg_bstride + (long long)t * GH;
                dxg[h] = d_i; dxg[H + h] = d_f; dxg[2 * H + h] = d_g; dxg[3 * H + h] = d_o;
            }
            __syncthreads();
            // ---- (5) hh chain backward: W_hh core gradients and dh_{t-1} (P)
            tt_chain_bwd(p, a.tile_bd, a.mg, R, xa, spill, g, dhc, wsm, dws, true, tid);
        }
        for (int e = tid; e < R * P; e += TT_NTHREADS) {
            const int b = e / P, j = e - b * P;
            const long long row = row0 + b;
            if (row < a.B) a.dh_out[row * P + j] = dhd[e] + dhc[b * hBS + tt_in_index(p, j)];
        }
        for (int e = tid; e < R * H; e += TT_NTHREADS) {
            const long long row = row0 + e / H;
            if (row < a.B) a.dc_out[row * H + (e % H)] = dcs[e];
        }
    }
    __syncthreads();
    float *slot = a.partial + (long long)blockIdx.x * (p.core_floats + q.core_floats);
    tt_flush_partial(p, dws, nullptr, 0, slot, tid);
    tt_flush_partial(q, dwq, nullptr, 0, slot + p.core_floats, tid);
}
