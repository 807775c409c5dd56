"""Reference for bidirectional stacks, composed from the unchanged oracles (test infrastructure only).

Per layer, the forward direction runs the oracle's one-layer loop on the layer input x; the reverse direction runs it
with its own parameters on x reversed in time, and its outputs are reversed back.  The next layer's input is the two
concatenated, (B, T, 2H).  This is the composition of torch.nn.LSTM / GRU(bidirectional=True), which
tests/test_bidirectional_cpu.py pins against torch itself, and the one `bidirectional_stack` implements.
"""


def bidir_layers(from_state_dict, sd, num_layers, **kw):
    """[(forward params, reverse params)] of each layer from a bidirectional module's state_dict (keys cell{l}.* and
    cell{l}_reverse.*), through an oracle's layers_from_state_dict."""
    pairs = []
    for l in range(num_layers):
        pair = []
        for prefix in ("cell%d." % l, "cell%d_reverse." % l):
            sub = {"cell0." + k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}
            pair.append(from_state_dict(sub, 1, **kw)[0])
        pairs.append(tuple(pair))
    return pairs


def flat_pairs(pairs):
    """The per-direction parameter dicts in module order: cell0, cell0_reverse, cell1, ..."""
    return [p for pair in pairs for p in pair]


def bidir_forward(forward, cell, pairs, x, states=None):
    """`forward` = an oracle's lstm_forward / gru_forward.  states: per state variable (h, and c for an LSTM) a
    (2L, B, H) tensor, direction d of layer l at 2l + d, or None (zeros).  Returns (out (B, T, 2H), [final states, each
    (2L, B, H)]), the contract of torch.nn.LSTM / GRU(bidirectional=True, batch_first=True)."""
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
    return inp, [torch.stack([f[k] for f in fins]) for k in range(len(fins[0]))]
