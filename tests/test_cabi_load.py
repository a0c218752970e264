"""CPU tests: the C-ABI library loads, exports every symbol include/wwb200.h declares,
and fails loudly (no fallback) when there is no CUDA device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_weights
from wakeword_detection_b200 import _cabi


def header_symbols():
    text = open(os.path.join(ROOT, "include", "wwb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(wwb_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _cabi.load_library()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), "libwwb200.so does not export %s" % s
    assert sorted(_cabi.PROTOTYPES) == syms, "ctypes prototypes out of sync with the header"
    assert lib.wwb_version() == 100


def test_pure_helpers():
    lib = _cabi.load_library()
    assert lib.wwb_num_frames(511) == 0
    assert lib.wwb_num_frames(512) == 1
    assert lib.wwb_num_frames(32000) == 197
    assert lib.wwb_num_frames(176000) == 1097


def test_create_without_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = _cabi.load_library()
    w = load_weights("CRNN")
    st, keep = _cabi.make_weights_struct(w, w)
    ctx = C.c_void_p()
    rc = lib.wwb_create(0, C.byref(st), 0, C.byref(ctx))
    assert rc == -2 and not ctx.value
    assert b"no CPU fallback" in lib.wwb_last_error(None)
    with pytest.raises(RuntimeError):
        _cabi.Engine(w)


def test_bad_arguments_rejected_before_any_device_work():
    lib = _cabi.load_library()
    ctx = C.c_void_p()
    assert lib.wwb_create(0, None, 0, C.byref(ctx)) == -1
    w = load_weights("CRNN")
    st, keep = _cabi.make_weights_struct(w, w)
    st.n_bins = 129
    assert lib.wwb_create(0, C.byref(st), 0, C.byref(ctx)) == -1
    assert b"geometry" in lib.wwb_last_error(None)
    # WaveNet: the head is a 2-way softmax (a [1, 32] det2_w would be read as [2, 32]), and both WaveNet paths hold
    # windows of up to 182 frames (the fp32 path's shared buffer has 182 + 18 rows)
    w = load_weights("Wavenet")
    for field, value, msg in (("n_out", 1, b"n_out"), ("mel_length", 183, b"window"), ("mel_length", 192, b"window")):
        for precision in (0, 1):
            st, keep = _cabi.make_weights_struct(w, w)
            setattr(st, field, value)
            assert lib.wwb_create(0, C.byref(st), precision, C.byref(ctx)) == -1 and not ctx.value
            assert msg in lib.wwb_last_error(None)


def test_weights_struct_packing():
    for name in ("CRNN", "CRNN_arik_original", "Wavenet"):
        w = load_weights(name)
        st, keep = _cabi.make_weights_struct(w, w)
        assert st.n_mel == 40 and st.n_bins == 257
        assert st.mel_length == (182 if name == "Wavenet" else 151)
        assert st.n_out == (1 if name == "CRNN" else 2)
        assert abs(st.mel_floor - 1e-5) < 1e-9 and abs(st.mel_log_offset + 11.512925) < 1e-5
    fw = {k: load_weights("CRNN")[k] for k in ("mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale")}
    st, keep = _cabi.make_weights_struct(fw, fw)
    assert st.kind == -1
