"""CPU: host-side logic of the drop-in -- checkpoint loading, state_dict contract, arch
inference, the C-ABI library's exported symbols -- and that the product path fails loudly
(no CPU fallback) when there is no GPU."""
import ctypes
import gzip
import os
import re

import numpy as np
import pytest
import torch

import tskd_b200
from tskd_b200 import capi
from tskd_b200.arch import BLOB_KEYS, INERT_KEYS, ArchConfig, arch_from_state_dict
from conftest import GOLDEN, ROOT, load_golden


def test_library_exports_every_declared_symbol():
    lib = tskd_b200.load_library()
    header = open(os.path.join(ROOT, "include", "b2cnn.h")).read()
    declared = set(re.findall(r"\b(b2cnn_[a-z_0-9]+)\s*\(", header))
    assert declared == set(capi.SYMBOLS), declared ^ set(capi.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.b2cnn_version()


def test_pure_host_entry_points():
    lib = tskd_b200.load_library()
    cfg = capi.make_config(tskd_b200.ARCH_PRESETS["mycnn5"])
    assert lib.b2cnn_l_out(ctypes.byref(cfg)) == 25
    assert lib.b2cnn_weight_count(ctypes.byref(cfg)) == 5370   # 5957 params minus the unused out1/out2/age_fn
    big = capi.make_config(tskd_b200.ARCH_PRESETS["mycnn5"].with_shape(3, 75000))
    assert lib.b2cnn_l_out(ctypes.byref(big)) == 18745
    old = capi.make_config(tskd_b200.ARCH_PRESETS["mycnn3"].with_shape(3, 75000))
    assert lib.b2cnn_l_out(ctypes.byref(old)) == 18747
    bad = capi.make_config(ArchConfig(window=12))
    assert lib.b2cnn_l_out(ctypes.byref(bad)) == -1


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_fails_loudly_without_gpu():
    lib = tskd_b200.load_library()
    cfg = capi.make_config(tskd_b200.ARCH_PRESETS["mycnn5"])
    h = ctypes.c_void_p()
    rc = lib.b2cnn_create(ctypes.byref(cfg), ctypes.byref(h))
    assert rc == capi.ECUDA and not h.value
    assert b"cuda" in lib.b2cnn_last_error().lower()
    m = tskd_b200.B200MyCNN()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 10, 120), torch.tensor([50.0]))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.predict(torch.zeros(4, 10, 120))


def test_product_never_imports_oracle():
    """No import / include / dlopen of anything under oracle/ from the shipped package (comments may cite the checker)."""
    import re
    pkg = os.path.join(ROOT, "time-series-kafka-demo_b200")
    bad = re.compile(r"""^\s*(from|import)\s+\.*oracle\b|__import__\(\s*['"]oracle|import_module\(\s*['"]oracle|"""
                     r"""#\s*include\s*["<][^">]*oracle|CDLL\([^)]*oracle|libmycnn_ref""", re.M)
    n = 0
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not bad.search(src), f
                n += 1
    assert n > 10
    for f in ("tskd_b200.py",):
        assert not bad.search(open(os.path.join(ROOT, f)).read()), f


def test_state_dict_contract(golden5):
    g, sd = golden5
    m = tskd_b200.B200MyCNN.from_reference(sd)
    assert m.arch == tskd_b200.ARCH_PRESETS["mycnn5"] and m.MAGICNUM == 25
    out = m.state_dict()
    assert list(out.keys()) == list(sd.keys())             # same names, same order
    for k in sd:
        assert out[k].shape == sd[k].shape and torch.equal(out[k], sd[k]), k
    assert set(BLOB_KEYS) | set(INERT_KEYS) == set(sd.keys())
    assert sum(v.numel() for v in sd.values()) == 5957      # explore_torch.ipynb:2117
    blob = m.packed_weights()
    assert blob.numel() == 5370
    assert torch.equal(blob[:400], sd["conv1.weight"].reshape(-1))
    with pytest.raises(RuntimeError):
        m.load_state_dict({k: v for k, v in sd.items() if k != "out.bias"})
    assert m.training is False
    with pytest.raises(NotImplementedError):
        m.train()
    assert m.eval() is m


@pytest.mark.parametrize("n,C,k1,pk,L", [(2, 7, 5, 2, 27), (3, 7, 5, 2, 27), (4, 10, 5, 2, 27)])
def test_arch_inference_older_checkpoints(n, C, k1, pk, L):
    g, sd = load_golden(f"mycnn{n}_ckpt.npz")
    a = arch_from_state_dict(sd, window=120)
    assert (a.in_channels, a.k1, a.pool_k, a.pool_s, a.l_out) == (C, k1, pk, 2, L)
    m = tskd_b200.B200MyCNN.from_reference(sd)
    assert "out1.weight" not in m.state_dict() and "age_fn.weight" in m.state_dict()


def test_view_contract_rejected():
    """L_out(window) != MAGICNUM must be an error, not a silent straddle (bin/models.py:29)."""
    g, sd = load_golden("mycnn5_xtestinput.npz")
    with pytest.raises((RuntimeError, ValueError)):
        tskd_b200.B200MyCNN.from_reference(sd, window=240)


@pytest.mark.parametrize("n", [2, 3, 4, 5])
def test_load_legacy_pickles(n, tmp_path):
    """The reference's shipped checkpoints model/MyCNN{n}.pth, stored byte for byte (gzip-compressed) under tests/golden/."""
    p = tmp_path / f"MyCNN{n}.pth"
    with gzip.open(os.path.join(GOLDEN, f"MyCNN{n}.pth.gz"), "rb") as f:
        p.write_bytes(f.read())
    ref = tskd_b200.load_reference_checkpoint(str(p))
    assert type(ref).__name__ == "PickledMyCNN" and ref.training is False
    m = tskd_b200.B200MyCNN.from_reference(ref)
    g, sd = load_golden("mycnn5_xtestinput.npz" if n == 5 else f"mycnn{n}_ckpt.npz")
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]), k


def test_restricted_unpickler_rejects_foreign_globals(tmp_path):
    import pickle
    p = tmp_path / "evil.pth"
    with open(p, "wb") as f:
        pickle.dump(os.system, f)
    with pytest.raises(Exception):
        tskd_b200.load_reference_checkpoint(str(p))


class _EvalPayload:
    def __reduce__(self):
        return (eval, ("__import__('os').getpid()",))


class _GetattrPayload:
    def __reduce__(self):
        return (getattr, ("abc", "upper"))


@pytest.mark.parametrize("payload", [_EvalPayload, _GetattrPayload])
@pytest.mark.parametrize("zipfile", [False, True])
def test_restricted_unpickler_rejects_builtins_and_torch_prefix(tmp_path, payload, zipfile):
    """ADVICE r1: builtins.eval / getattr (and anything merely *under* torch. or numpy.) must not unpickle --
    the allowlist is exact (module, name) pairs, not prefixes."""
    import pickle
    p = tmp_path / "evil.pth"
    torch.save(payload(), str(p), _use_new_zipfile_serialization=zipfile)
    with pytest.raises(pickle.UnpicklingError):
        tskd_b200.load_reference_checkpoint(str(p))
    from tskd_b200 import checkpoint
    up = checkpoint._Unpickler.__new__(checkpoint._Unpickler)
    for mod, name in (("builtins", "eval"), ("torch.serialization", "load"), ("numpy", "load"), ("_codecs", "encode"),
                      ("torch._utils", "_rebuild_tensor_v2x")):
        with pytest.raises(pickle.UnpicklingError):
            checkpoint._Unpickler.find_class(up, mod, name)


def test_synth_is_deterministic():
    a = tskd_b200.synth.make_windows(5, 3, 64, "physio", seed=1)
    b = tskd_b200.synth.make_windows(5, 3, 64, "physio", seed=1)
    assert torch.equal(a, b) and a.min() >= 0 and a.max() <= 200
    e = tskd_b200.synth.make_windows(4, 3, 64, "edge", seed=1)
    assert torch.isnan(e[0]).any() and torch.isinf(e[1]).any()
    ages = tskd_b200.synth.make_ages(100)
    assert ages.min() >= 15 and ages.max() <= 80


def test_train_entry_points_validate_without_a_gpu():
    """b2cnn_train_workspace_bytes is pure host arithmetic; b2cnn_train_step rejects bad arguments before touching CUDA."""
    import ctypes
    from tskd_b200 import capi
    lib = capi.load_library()
    cfg = capi.make_config(tskd_b200.ARCH_PRESETS["mycnn5"])
    n = lib.b2cnn_train_workspace_bytes(ctypes.byref(cfg), 32)
    assert n > 32 * (4 * 111 + 4 * 55 + 51 + 25) * 4
    bad = capi.make_config(tskd_b200.ARCH_PRESETS["mycnn5"].with_shape(10, 121))    # L_out(121) == 25 still; break the view instead
    bad.lstm_input = 24
    assert lib.b2cnn_train_workspace_bytes(ctypes.byref(bad), 32) < 0
    opt = capi.Adam(1e-3, 0.9, 0.999, 1e-8)
    rc = lib.b2cnn_train_step(ctypes.byref(cfg), None, None, None, None, 1, ctypes.byref(opt), 1, None, 4, None, None, 1, None, None,
                              None, None, 0, None)
    assert rc == capi.EINVAL and "null" in capi.last_error()


def test_zero_windows_and_trainer_argument_checks_need_no_gpu():
    """predict() over zero rows scores nothing (the per-row loop of bin/predictStream.py:70) and never reaches the library;
    the trainer rejects bad arguments before it looks for a device."""
    import tskd_b200
    from tskd_b200.trainer import B200Trainer
    m = tskd_b200.B200MyCNN(tskd_b200.ARCH_PRESETS["mycnn5"])
    out = m.predict(torch.zeros(0, 10, 120), 65.0)
    assert tuple(out.shape) == (0,) and out.dtype == torch.float32
    with pytest.raises(RuntimeError, match="expected input"):
        m.predict(torch.zeros(0, 9, 120), 65.0)
    with pytest.raises(ValueError, match="mode"):
        m.predict(torch.zeros(0, 10, 120), 65.0, mode="rows")
    with pytest.raises(ValueError, match="mode"):
        B200Trainer(m, mode="rows")
    with pytest.raises(ValueError, match="dropout"):
        B200Trainer(m, dropout=1.0)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA"):
            B200Trainer(m)
