"""Reference for inter-layer dropout, built from the unchanged oracles (test infrastructure only).

The stack runs one layer at a time (as tests/layer_states_ref.py and tests/bidir_ref.py do), and the output of every layer
but the last is multiplied by a given mask before the next layer reads it.  A mask holds 0 or 1 / (1 - p) per element, so
the multiplication is the whole of dropout; where it comes from is up to the caller: torch's own draws on the CPU
(tests/test_dropout_cpu.py pins this composition against torch.nn.LSTM / GRU(dropout=p)), or the engine's mask kernel on
the GPU (ttrnn_dropout_apply on a block of ones).
"""


def dropout_layer_states(forward, cell, layers, x, masks, states=None):
    """`forward` = an oracle's lstm_forward / gru_forward(layers, x, init_states).  masks: L - 1 tensors (B, T, H).
    states: per state variable an (L, B, H) tensor, or None (zeros).  Returns (outputs of the last layer, [final states,
    each (L, B, H)]), the contract of torch.nn.LSTM / GRU(dropout=p, batch_first=True) in training mode."""
    import torch
    lstm = cell == "lstm"
    inp, fins = x, []
    for l, p in enumerate(layers):
        st = None
        if states is not None:
            st = (states[0][l], states[1][l]) if lstm else states[0][l]
        out, fin = forward([p], inp, st)
        fins.append(list(fin) if lstm else [fin])
        inp = out * masks[l] if l < len(layers) - 1 else out
    return inp, [torch.stack([f[k] for f in fins]) for k in range(len(fins[0]))]


def dropout_bidir_forward(forward, cell, pairs, x, masks, states=None):
    """Bidirectional form: pairs as tests/bidir_ref.bidir_layers returns them, masks: L - 1 tensors (B, T, 2H) applied to
    the joined output of each layer but the last; the next layer's reverse direction reads the masked values reversed in
    time.  states: per state variable a (2L, B, H) tensor, direction d of layer l at 2l + d, or None."""
    import torch
    lstm = cell == "lstm"
    inp, fins = x, []
    for l, (pf, pr) in enumerate(pairs):
        outs = []
        for d, (p, seq) in enumerate(((pf, inp), (pr, inp.flip(1)))):
            st = None
            if states is not None:
                st = (states[0][2 * l + d], states[1][2 * l + d]) if lstm else states[0][2 * l + d]
            out, fin = forward([p], seq, st)
            outs.append(out)
            fins.append(list(fin) if lstm else [fin])
        inp = torch.cat([outs[0], outs[1].flip(1)], dim=2)
        if l < len(pairs) - 1:
            inp = inp * masks[l]
    return inp, [torch.stack([f[k] for f in fins]) for k in range(len(fins[0]))]
