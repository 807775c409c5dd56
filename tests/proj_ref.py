"""Reference for projected TT-LSTM stacks (LSTMP, `proj_size`), built from the unchanged oracle (test infrastructure only).

A projected layer is the oracle's TT-LSTM cell with one more TT matvec at the end of every step:

    m_t = o_t * tanh(c_t)      (H)
    h_t = W_hr m_t             (P)      the layer output and the next step's hh input (W_hh is 4H x P)

`lstmp_forward` has the signature of the oracle's lstm_forward, so the per-layer-state, bidirectional and dropout
compositions (tests/layer_states_ref.py, tests/bidir_ref.py, tests/dropout_ref.py) run it unchanged.
tests/test_proj_cpu.py pins it against torch.nn.LSTM(proj_size=P).
"""
import torch

from helpers import oracle


def lstmp_cell(p, x, h, c):
    hid = c.shape[1]
    gates = oracle.ttlinear(p["ih_cores"], p["ih_bias"], x) + oracle.ttlinear(p["hh_cores"], p["hh_bias"], h)
    i = torch.sigmoid(gates[:, :hid])
    f = torch.sigmoid(gates[:, hid:2 * hid])
    g = torch.tanh(gates[:, 2 * hid:3 * hid])
    o = torch.sigmoid(gates[:, 3 * hid:])
    c_new = f * c + i * g
    return oracle.tt_matvec(p["hr_cores"], o * torch.tanh(c_new)), c_new


def sizes(p):
    """(H, P) of one projected layer."""
    hr = p["hr_cores"]
    H = 1
    P = 1
    for c in hr:
        H *= int(c.shape[2])
        P *= int(c.shape[1])
    return H, P


def lstmp_forward(layers, x, init_states=None):
    """The oracle's lstm_forward loop with projected cells: one (h0 (B, P), c0 (B, H)) seeds every layer; returns
    (outputs (B, T, P), (h_T, c_T)) of the last layer."""
    batch, seq_len, _ = x.shape
    H, P = sizes(layers[0])
    if init_states is None:
        init_states = (torch.zeros(batch, P, dtype=x.dtype), torch.zeros(batch, H, dtype=x.dtype))
    state = [tuple(init_states)] * len(layers)
    outputs = []
    for t in range(seq_len):
        inp = x[:, t, :]
        for li, p in enumerate(layers):
            inp, c_new = lstmp_cell(p, inp, *state[li])
            state[li] = (inp, c_new)
        outputs.append(inp)
    return torch.stack(outputs, dim=1), state[-1]


def random_layers(I, H, P, L, n_cores, tt_rank, bias=True, seed=0, dtype=torch.float64, requires_grad=False, scale=1.0,
                  in_sizes=None):
    """Random projected layers with the oracle's Glorot core distribution.  in_sizes: the input width of each layer
    (default I, then P)."""
    g = torch.Generator().manual_seed(seed)
    layers = []
    for l in range(L):
        n_in = in_sizes[l] if in_sizes else (I if l == 0 else P)
        p = {}
        for short, (a, b, gates) in (("ih", (n_in, H, 4)), ("hh", (P, H, 4)), ("hr", (H, P, 1))):
            in_q, out_q = oracle.tt_shape(a, b, n_cores, gates)
            std = oracle.glorot_core_std(in_q, out_q, tt_rank) * scale
            ranks = [1] + [tt_rank] * (len(in_q) - 1) + [1]
            p[short + "_cores"] = [(torch.randn(ranks[k], out_q[k], in_q[k], ranks[k + 1], generator=g, dtype=torch.float64)
                                    * std).to(dtype).requires_grad_(requires_grad) for k in range(len(in_q))]
            if short != "hr":
                b_ = None
                if bias:
                    b_ = (1e-3 + 1e-2 * torch.randn(4 * H, generator=g, dtype=torch.float64)).to(dtype)
                    b_ = b_.requires_grad_(requires_grad)
                p[short + "_bias"] = b_
        layers.append(p)
    return layers


def flat_params(layers):
    """Parameters in blob order: per layer ih cores, ih bias, hh cores, hh bias, hr cores."""
    out = []
    for p in layers:
        for short in ("ih", "hh", "hr"):
            out += list(p[short + "_cores"])
            if p.get(short + "_bias") is not None:
                out.append(p[short + "_bias"])
    return out


def state_dict(layers, names=None):
    """Module state_dict of the layers; names: the cell name of each layer (default cell{l})."""
    sd = {}
    for l, p in enumerate(layers):
        cell = names[l] if names else "cell%d" % l
        for short, long in (("ih", "input_weights"), ("hh", "hidden_weights"), ("hr", "projection_weights")):
            for k, c in enumerate(p[short + "_cores"]):
                sd["%s.%s.parameters.%d" % (cell, long, k)] = c.detach().clone()
            if p.get(short + "_bias") is not None:
                sd["%s.%s.bias" % (cell, long)] = p[short + "_bias"].detach().clone()
    return sd


def torch_lstmp(pairs, x, states, I, H, P, bias=True):
    """torch.nn.LSTM(proj_size=P, batch_first=True) in FP64 with its weights formed inside the graph from the TT cores
    (tt_dense through torch.func.functional_call), so that autograd hands back core gradients.  pairs: per layer a tuple
    of one (or, bidirectional, two) layer dicts; states = (h0 (D*L, B, P), c0 (D*L, B, H))."""
    D = len(pairs[0])
    m = torch.nn.LSTM(I, H, len(pairs), bias=bias, batch_first=True, proj_size=P, bidirectional=D == 2).double()
    params = {}
    for l, pair in enumerate(pairs):
        for d, q in enumerate(pair):
            sfx = "_l%d%s" % (l, "_reverse" if d else "")
            params["weight_ih" + sfx] = oracle.tt_dense(q["ih_cores"])
            params["weight_hh" + sfx] = oracle.tt_dense(q["hh_cores"])
            params["weight_hr" + sfx] = oracle.tt_dense(q["hr_cores"])
            if bias:
                params["bias_ih" + sfx] = q["ih_bias"]
                params["bias_hh" + sfx] = q["hh_bias"]
    return torch.func.functional_call(m, params, (x, tuple(states)))
