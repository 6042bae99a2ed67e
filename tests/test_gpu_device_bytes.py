"""Device-byte counters (b200_device_bytes, b200_*_device_bytes): every buffer a handle allocates is charged to its owner and
released with it.  Two identical cycles of create / use / close on one Engine must leave the context's counter where the
first cycle left it (no drift, nothing left charged by a closed handle), and must give the dynamic handles the same sizes."""
import numpy as np
import pytest

from tests.util import synth_accounts, synth_storage

pytestmark = [pytest.mark.gpu]


def _cycle(eng, keys, accs, skeys, svals, offs, ins_keys, ins_accs):
    from reth_b200.engine import DynamicState, DynamicTrie, ResidentTrie, RootStream
    got = {}
    rt = ResidentTrie.create(eng, keys, accs)
    upd = accs[:50].copy()
    upd["nonce"] += 1
    rt.update(keys[:50], upd)
    _, rebuilt = rt.apply(ins_keys, ins_accs)
    assert rebuilt
    got["trie"] = rt.device_bytes()
    rt.close()

    dt = DynamicTrie.create(eng, keys, accs)
    dt.apply(keys[:100], accs[:100], present=np.r_[np.ones(60, np.uint8), np.zeros(40, np.uint8)])
    got["dtrie"] = dt.device_bytes()
    dt.close()

    ds = DynamicState.create(eng, keys, accs, skeys, svals, offs)
    got["dstate"] = ds.device_bytes()
    ds.close()

    st = RootStream(eng, retain_updates=True)
    h = len(keys) // 2
    sh = int(offs[h])
    st.push(keys[:h], accs[:h], skeys[:sh], svals[:sh], offs[:h + 1])
    st.push(keys[h:], accs[h:], skeys[sh:], svals[sh:], offs[h:] - offs[h])
    st.finish()
    st.close()
    got["engine"] = eng.device_bytes()
    return got


def test_device_bytes_stable_across_cycles():
    from reth_b200 import Engine
    n = 3000
    keys, accs = synth_accounts(41, n)
    skeys, svals, offs = synth_storage(42, np.arange(n) % 6)
    ins_keys, ins_accs = synth_accounts(43, 20)
    eng = Engine(0)
    try:
        first = _cycle(eng, keys, accs, skeys, svals, offs, ins_keys, ins_accs)
        second = _cycle(eng, keys, accs, skeys, svals, offs, ins_keys, ins_accs)
    finally:
        eng.close()
    assert all(v > 0 for v in first.values()), first
    assert second["engine"] == first["engine"]
    assert second["dtrie"] == first["dtrie"]
    assert second["dstate"] == first["dstate"]
