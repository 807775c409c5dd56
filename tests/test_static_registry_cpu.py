"""The registry of statically specialised kernels, without a GPU: the key table of ttrnn_static_kernel_keys(), the
launch counters, and that test_gpu_static_registry.py has a case for exactly the registered kernels (a new TTS_* line
without a case fails here)."""
import ctypes

from tensorized_rnn_b200 import _lib

import test_gpu_static_registry as reg


def _lines(fn):
    buf = ctypes.create_string_buffer(1 << 16)
    n = fn(buf, len(buf))
    assert 0 < n < len(buf) - 1
    return [ln.split("|") for ln in buf.value.decode().strip().splitlines()]


def test_key_table_matches_the_kernel_table_and_keys_are_unique():
    lib = _lib.load()
    table, keys_text = _lines(lib.ttrnn_static_kernel_table), _lines(lib.ttrnn_static_kernel_keys)
    assert all(len(r) == 5 for r in table), [r for r in table if len(r) != 5]
    assert all(len(r) == 8 for r in keys_text), [r for r in keys_text if len(r) != 8]
    # same entries in the same order: (kind, name, R) of line i agree
    assert [r[:3] for r in table] == [r[:3] for r in keys_text]
    keys = reg.registry_keys(lib)
    assert len(keys) == len(set(keys)), [k for k in keys if keys.count(k) > 1]
    for kind, name, R, cell, mode, saved, split, merged in keys:
        assert R >= 1 and split in (0, 1) and merged in (0, 1), (kind, name)
        if kind.startswith("rnn"):
            assert cell in (reg.LSTM, reg.GRU) and mode in (reg.XG, reg.RANK1) and saved in (0, 2), (kind, name)
            assert merged == ("(m01" in name), name
        else:
            assert (cell, mode, saved, merged) == (reg.NA, reg.NA, reg.NA, 0), (kind, name)


def test_launch_counters_cover_the_table():
    lib = _lib.load()
    n = lib.ttrnn_static_kernel_launches(None, 0, 1)
    assert n == len(_lines(lib.ttrnn_static_kernel_table))
    counts = (ctypes.c_int64 * (n + 3))(*([-1] * (n + 3)))
    assert lib.ttrnn_static_kernel_launches(counts, n + 3, 0) == n
    assert list(counts[:n]) == [0] * n and list(counts[n:]) == [-1] * 3       # no launch on the host, no overrun


def test_gpu_ledger_has_exactly_the_registered_kernels():
    keys = set(reg.registry_keys(_lib.load()))
    ledger = set(reg.LEDGER)
    assert not keys - ledger, "registered kernels without a case in test_gpu_static_registry.py: %s" % sorted(keys - ledger)
    assert not ledger - keys, "cases for kernels that are not registered: %s" % sorted(ledger - keys)
    targets = [k for c in reg.CASES for k in c.targets]
    assert len(targets) == len(set(targets)), "a kernel is the target of more than one case"
    assert len({c.id for c in reg.CASES}) == len(reg.CASES)
