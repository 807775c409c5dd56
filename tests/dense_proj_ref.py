"""torch.nn.LSTM(proj_size=P, batch_first=True) with the weights of a dense `LSTM` copied in (test infrastructure only).

The gate order is i, f, g, o in both, so the state_dicts map one to one:
    cell{l}{sfx}.input_weights.weight      -> weight_ih_l{l}{sfx}
    (no ih bias)                           -> bias_ih_l{l}{sfx} = 0
    cell{l}{sfx}.hidden_weights.weight     -> weight_hh_l{l}{sfx}
    cell{l}{sfx}.hidden_weights.bias       -> bias_hh_l{l}{sfx}
    cell{l}{sfx}.projection_weights.weight -> weight_hr_l{l}{sfx}
sfx is "" or "_reverse".  No restated LSTMP math: torch itself is the oracle.
"""
import torch


def torch_names(m, l, sfx=""):
    """torch's parameter names of cell{l}{sfx} of dense LSTM `m`, in the order of that cell's flat_parameters()."""
    names = ["weight_ih_l%d%s", "weight_hh_l%d%s"] + (["bias_hh_l%d%s"] if m.bias else []) + \
        (["weight_hr_l%d%s"] if m.proj_size else [])
    return [n % (l, sfx) for n in names]


def _copy(t, m, l_src, l_dst, sfx):
    cell = getattr(m, "cell%d%s" % (l_src, sfx))
    with torch.no_grad():
        for name, p in zip(torch_names(m, l_dst, sfx), cell.flat_parameters()):
            getattr(t, name).copy_(p.detach().cpu())
        if m.bias:
            getattr(t, "bias_ih_l%d%s" % (l_dst, sfx)).zero_()


def _sfxs(m):
    return ("", "_reverse") if m.bidirectional else ("",)


def torch_lstm(m, dtype=torch.float64):
    """The whole stack of `m` as one torch.nn.LSTM on the CPU."""
    t = torch.nn.LSTM(m.input_size, m.hidden_size, m.num_layers, bias=bool(m.bias), batch_first=True,
                      bidirectional=m.bidirectional, proj_size=m.proj_size).to(dtype)
    for l in range(m.num_layers):
        for sfx in _sfxs(m):
            _copy(t, m, l, l, sfx)
    return t


def torch_layers(m, dtype=torch.float64):
    """One one-layer torch.nn.LSTM per layer of a unidirectional `m` (to compose with a given dropout mask)."""
    out = []
    for l in range(m.num_layers):
        in_size = m.input_size if l == 0 else m.output_size
        t = torch.nn.LSTM(in_size, m.hidden_size, 1, bias=bool(m.bias), batch_first=True, proj_size=m.proj_size).to(dtype)
        _copy(t, m, l, 0, "")
        out.append(t)
    return out


def torch_params(t, m):
    """The torch stack's parameters that correspond to m.flat_parameters(), in that order (no bias_ih)."""
    return [getattr(t, n) for l in range(m.num_layers) for sfx in _sfxs(m) for n in torch_names(m, l, sfx)]


def layers_params(layers, m):
    """The same for the one-layer modules of torch_layers."""
    return [getattr(t, n) for t in layers for n in torch_names(m, 0)]


def layer_forward(layers, x, st=None):
    """tests/dropout_ref.py's `forward` over a list holding one one-layer torch LSTM: st = (h (B, P), c (B, H)) or None."""
    (t,) = layers
    out, (h, c) = t(x, None if st is None else (st[0].unsqueeze(0), st[1].unsqueeze(0)))
    return out, (h[0], c[0])
