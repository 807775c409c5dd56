"""Reference for per-layer states, built from the unchanged oracles (test infrastructure only).

The reference's loop is step-major / layer-minor (lstm.py:123-133), but layer l at step t only reads layer l's own state
and layer l - 1's output at step t, so running the stack one layer at a time over the whole sequence computes the same
values.  Run that way, each layer can start from its own initial state and hand back its own final state: the contract of
torch.nn.LSTM, (L, B, H) states in and out, which `forward_states` implements.
"""


def lstm_layer_states(forward, layers, x, states=None):
    """`forward` = an oracle's lstm_forward(layers, x, init_states).  states = (h0, c0), each (L, B, H), or None
    (zeros).  Returns (outputs of the last layer, [h_n, c_n]) with h_n, c_n (L, B, H)."""
    import torch
    inp, hs, cs = x, [], []
    for l, p in enumerate(layers):
        inp, (h, c) = forward([p], inp, None if states is None else (states[0][l], states[1][l]))
        hs.append(h)
        cs.append(c)
    return inp, [torch.stack(hs), torch.stack(cs)]


def gru_layer_states(forward, layers, x, states=None):
    """`forward` = an oracle's gru_forward(layers, x, init_states).  states (L, B, H) or None (zeros).  Returns
    (outputs of the last layer, [h_n]) with h_n (L, B, H)."""
    import torch
    inp, hs = x, []
    for l, p in enumerate(layers):
        inp, h = forward([p], inp, None if states is None else states[l])
        hs.append(h)
    return inp, [torch.stack(hs)]
