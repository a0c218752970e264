"""Trained-weight extraction from the reference's model directories.

The reference builds `TFLiteModel(model_dir/{filter,encode,detect}.tflite)`
(reference: spokestack/wakeword/tflite.py:51-59, utils/evaluate_models.py:30-36)
and derives all geometry from the models' input/output shapes (:67-90).  Here the
same directory is read with `tflite_reader`, every trained tensor is located by
*walking the graph* (never by tensor name alone: SURVEY.md Appendix A4 lists the
misleading names) and returned as a flat dict of named float32 arrays.  A
directory holding a `weights.npz` written by `save_npz` is accepted as well, so
the GPU box does not need the `.tflite` files.

Canonical names
  filter : mel_w[40,257] mel_b[40] mel_floor[] mel_log_offset[] mel_scale[]
  CRNN   : conv_w[32,5,20] conv_b[32]
           gru{1,2}_{f,b}_w[96,in] gru*_u[96,32] gru*_bi[96] gru*_br[96]
           det1_w[64,64] det1_b[64] det2_w[n,64] det2_b[n]   (n=1 sigmoid | n=2 softmax)
  WaveNet: in_w[16,40] in_b[16]  bn_mul[24,16] bn_add[24,16] dilation[24]
           sig_w[24,16,3,16] sig_b[24,16] tanh_w[24,16,3,16] tanh_b[24,16]   (out, tap, in)
           res_w[23,16,16] res_b[23,16]  skip_w[24,32,16] skip_b[24,32]
           det1_w[32,32] det1_b[32] det2_w[2,32] det2_b[2]
  both   : mel_length[] (encoder window length in mel frames, read from the encoder's input shape: CRNN 17..256,
           shipped 151; WaveNet 17..182, shipped 182)
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import numpy as np

from . import tflite_reader as tr

F32 = np.float32
_PASS_THROUGH = ("RESHAPE", "BATCH_TO_SPACE_ND", "SPACE_TO_BATCH_ND", "PAD")


class _Walker:
    def __init__(self, g: tr.SubGraph) -> None:
        self.g = g
        self.producer: Dict[int, int] = {}
        self.consumers: Dict[int, List[int]] = {}
        for k, op in enumerate(g.ops):
            for o in op.outputs:
                self.producer[o] = k
            for i in op.inputs:
                if i >= 0:
                    self.consumers.setdefault(i, []).append(k)

    def const(self, t: int) -> Optional[np.ndarray]:
        return self.g.tensors[t].data if t >= 0 else None

    def data_input(self, op: tr.Op) -> int:
        """The first non-constant input of `op`."""
        for i in op.inputs:
            if i >= 0 and self.const(i) is None:
                return i
        raise ValueError("op %s has no data input" % op.name)

    def back(self, t: int, through=_PASS_THROUGH) -> int:
        """Follow tensor `t` backwards through layout-only ops; returns the op index
        that produced the first 'real' value (or -1 for a graph input)."""
        while True:
            k = self.producer.get(t, -1)
            if k < 0 or self.g.ops[k].name not in through:
                return k
            t = self.g.ops[k].inputs[0]

    def forward(self, t: int, through=_PASS_THROUGH) -> List[int]:
        """Op indices consuming `t`, looking through layout-only ops."""
        out = []
        for k in self.consumers.get(t, []):
            if self.g.ops[k].name in through:
                out += self.forward(self.g.ops[k].outputs[0], through)
            else:
                out.append(k)
        return out


# ----------------------------------------------------------------------------
def extract_filter(path: str) -> Dict[str, np.ndarray]:
    """filter.tflite: FC(257->40) -> MAXIMUM(floor) -> LOG -> SUB(offset) -> MUL(scale)
    (reference call site: spokestack/wakeword/tflite.py:181-184)."""
    g = tr.load(path).main
    out: Dict[str, np.ndarray] = {}
    for op in g.ops:
        consts = [g.tensors[i].data for i in op.inputs if i >= 0 and g.tensors[i].data is not None]
        if op.name == "FULLY_CONNECTED":
            out["mel_w"] = consts[0].astype(F32)
            out["mel_b"] = (consts[1] if len(consts) > 1 else np.zeros(consts[0].shape[0])).astype(F32)
        elif op.name == "MAXIMUM":
            out["mel_floor"] = np.asarray(consts[0], F32).reshape(())
        elif op.name == "SUB":
            out["mel_log_offset"] = np.asarray(consts[0], F32).reshape(())
        elif op.name == "MUL":
            out["mel_scale"] = np.asarray(consts[0], F32).reshape(())
    missing = {"mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale"} - set(out)
    if missing:
        raise ValueError("filter graph not recognised, missing %s" % sorted(missing))
    return out


def _extract_dense_head(path: str) -> Dict[str, np.ndarray]:
    g = tr.load(path).main
    fcs = [op for op in g.ops if op.name == "FULLY_CONNECTED"]
    if len(fcs) != 2:
        raise ValueError("CRNN detect graph not recognised")
    out = {}
    for k, op in enumerate(fcs, 1):
        out["det%d_w" % k] = g.tensors[op.inputs[1]].data.astype(F32)
        out["det%d_b" % k] = g.tensors[op.inputs[2]].data.astype(F32)
    last = g.ops[-1].name
    n = out["det2_w"].shape[0]
    if not ((last == "LOGISTIC" and n == 1) or (last == "SOFTMAX" and n == 2)):
        raise ValueError("unexpected detect head %s with %d outputs" % (last, n))
    return out


def extract_crnn(encode_path: str, detect_path: str) -> Dict[str, np.ndarray]:
    """CRNN encode/detect (SURVEY.md Appendix A2).  GRU weights are anonymous
    constants inside the four WHILE bodies: the FC fed by GATHER is the input
    projection, the FC fed by the carried state is the recurrent one; a WHILE whose
    sequence input comes from REVERSE_V2 is the backward direction."""
    m = tr.load(encode_path)
    g = m.main
    w = _Walker(g)
    out: Dict[str, np.ndarray] = {}
    conv = [op for op in g.ops if op.name == "CONV_2D"]
    if len(conv) != 1:
        raise ValueError("CRNN encoder: expected one CONV_2D")
    cw = g.tensors[conv[0].inputs[1]].data
    if cw.shape[3] != 1 or conv[0].options["stride_h"] != 2 or conv[0].options["stride_w"] != 8 \
            or conv[0].options["padding"] != 0 or conv[0].options["act"] != 1:
        raise ValueError("CRNN encoder: unexpected conv geometry")
    out["conv_w"] = cw[..., 0].astype(F32)
    out["mel_length"] = np.asarray(m.input_details()[0]["shape"][2], np.int32)
    out["conv_b"] = g.tensors[conv[0].inputs[2]].data.astype(F32)

    whiles = [op for op in g.ops if op.name == "WHILE"]
    if len(whiles) != 4:
        raise ValueError("CRNN encoder: expected four WHILE loops")
    seen = set()
    for op in whiles:
        seq_in = op.inputs[-1]
        backward = g.ops[w.producer[seq_in]].name == "REVERSE_V2" if seq_in in w.producer else False
        body = m.subgraphs[op.options["body"]]
        bw = _Walker(body)
        state_in = body.inputs[3]
        fcs = [o for o in body.ops if o.name == "FULLY_CONNECTED"]
        rec = [o for o in fcs if o.inputs[0] == state_in]
        inp = [o for o in fcs if o.inputs[0] != state_in
               and body.ops[bw.producer[o.inputs[0]]].name == "GATHER"]
        if len(rec) != 1 or len(inp) != 1:
            raise ValueError("CRNN encoder: WHILE body not recognised")
        W = body.tensors[inp[0].inputs[1]].data.astype(F32)
        layer = 1 if W.shape[1] == out["conv_w"].shape[0] * 20 else 2
        key = "gru%d_%s" % (layer, "b" if backward else "f")
        if key in seen:
            raise ValueError("CRNN encoder: duplicate %s" % key)
        seen.add(key)
        out[key + "_w"] = W
        out[key + "_bi"] = body.tensors[inp[0].inputs[2]].data.astype(F32)
        out[key + "_u"] = body.tensors[rec[0].inputs[1]].data.astype(F32)
        out[key + "_br"] = body.tensors[rec[0].inputs[2]].data.astype(F32)
    out.update(_extract_dense_head(detect_path))
    return out


def extract_wavenet(encode_path: str, detect_path: str) -> Dict[str, np.ndarray]:
    """WaveNet encode/detect (SURVEY.md Appendix A3), located by graph walking."""
    enc_model = tr.load(encode_path)
    g = enc_model.main
    w = _Walker(g)

    def eff_bias(k: int):
        """conv bias + the per-channel constant of the ADD that follows it; also the
        op index of whatever consumes the biased value and the fused activation."""
        op = g.ops[k]
        b = g.tensors[op.inputs[2]].data.astype(F32).copy()
        act = op.options["act"]
        nxt = w.forward(op.outputs[0])
        tail = op.outputs[0]
        if len(nxt) == 1 and g.ops[nxt[0]].name == "ADD":
            a = g.ops[nxt[0]]
            c = [w.const(i) for i in a.inputs]
            cc = [v for v in c if v is not None and v.ndim == 1 and v.shape[0] == b.shape[0]]
            if len(cc) == 1:
                b = b + cc[0].astype(F32)
                act = a.options.get("act", 0)
                tail = a.outputs[0]
                nxt = w.forward(tail)
        return b, act, tail, nxt

    convs = [k for k, op in enumerate(g.ops) if op.name == "CONV_2D"]
    shapes = {k: tuple(g.tensors[g.ops[k].inputs[1]].shape) for k in convs}
    first = [k for k in convs if shapes[k][3] == 40]
    if len(first) != 1:
        raise ValueError("WaveNet encoder: input conv not found")
    out: Dict[str, np.ndarray] = {}
    b, act, x_tensor, _ = eff_bias(first[0])
    if act != 1:
        raise ValueError("WaveNet encoder: input conv must be ReLU")
    out["in_w"] = g.tensors[g.ops[first[0]].inputs[1]].data[:, 0, 0, :].astype(F32)
    out["in_b"] = b
    out["mel_length"] = np.asarray(enc_model.input_details()[0]["shape"][1], np.int32)

    gate = [k for k in convs if shapes[k][2] == 3]
    sig, tanh = [], []
    for k in gate:
        b, act, tail, nxt = eff_bias(k)
        kind = g.ops[nxt[0]].name
        (sig if kind == "LOGISTIC" else tanh).append((k, b, nxt[0]))
        if kind not in ("LOGISTIC", "TANH") or act != 0:
            raise ValueError("WaveNet encoder: gate conv not followed by LOGISTIC/TANH")
    if len(sig) != len(tanh):
        raise ValueError("WaveNet encoder: gate convs unbalanced")
    nb = len(sig)
    out["bn_mul"] = np.zeros((nb, 16), F32); out["bn_add"] = np.zeros((nb, 16), F32)
    out["dilation"] = np.zeros((nb,), np.int32)
    out["sig_w"] = np.zeros((nb, 16, 3, 16), F32); out["sig_b"] = np.zeros((nb, 16), F32)
    out["tanh_w"] = np.zeros((nb, 16, 3, 16), F32); out["tanh_b"] = np.zeros((nb, 16), F32)
    out["skip_w"] = np.zeros((nb, 32, 16), F32); out["skip_b"] = np.zeros((nb, 32), F32)
    out["res_w"] = np.zeros((nb - 1, 16, 16), F32); out["res_b"] = np.zeros((nb - 1, 16), F32)
    gate_mul_to_block = {}
    for blk, ((ks, bs, ls), (kt, bt, lt)) in enumerate(zip(sig, tanh)):
        out["sig_w"][blk] = g.tensors[g.ops[ks].inputs[1]].data[:, 0, :, :]
        out["tanh_w"][blk] = g.tensors[g.ops[kt].inputs[1]].data[:, 0, :, :]
        out["sig_b"][blk], out["tanh_b"][blk] = bs, bt
        # both gate convs read the same padded tensor: PAD <- ADD(bn_add) <- MUL(bn_mul)
        t = g.ops[ks].inputs[0]
        pad_op = None
        while True:
            k = w.producer[t]
            if g.ops[k].name == "PAD":
                pad_op = g.ops[k]
            if g.ops[k].name not in _PASS_THROUGH:
                break
            t = g.ops[k].inputs[0]
        if pad_op is None or g.ops[k].name != "ADD":
            raise ValueError("WaveNet encoder: block %d BN/PAD chain not recognised" % blk)
        pads = g.tensors[pad_op.inputs[1]].data
        out["dilation"][blk] = int(pads[1][0]) // 2
        add = g.ops[k]
        out["bn_add"][blk] = [w.const(i) for i in add.inputs if w.const(i) is not None][0]
        mul = g.ops[w.producer[w.data_input(add)]]
        if mul.name != "MUL":
            raise ValueError("WaveNet encoder: block %d BN mul missing" % blk)
        out["bn_mul"][blk] = [w.const(i) for i in mul.inputs if w.const(i) is not None][0]
        # the gate product
        so, to = g.ops[ls].outputs[0], g.ops[lt].outputs[0]
        prod = [k2 for k2 in w.consumers[so] if g.ops[k2].name == "MUL" and to in g.ops[k2].inputs]
        if len(prod) != 1:
            raise ValueError("WaveNet encoder: block %d gate product missing" % blk)
        gate_mul_to_block[prod[0]] = blk

    n_res = 0
    for k in convs:
        if shapes[k][2] != 1 or shapes[k][3] != 16:
            continue
        src = w.back(g.ops[k].inputs[0])
        blk = gate_mul_to_block.get(src)
        if blk is None:
            raise ValueError("WaveNet encoder: 1x1 conv not fed by a gate product")
        b, act, _, _ = eff_bias(k)
        if act != 1:
            raise ValueError("WaveNet encoder: 1x1 conv must be ReLU")
        wk = g.tensors[g.ops[k].inputs[1]].data[:, 0, 0, :].astype(F32)
        if shapes[k][0] == 16:
            out["res_w"][blk], out["res_b"][blk] = wk, b
            n_res += 1
        else:
            out["skip_w"][blk], out["skip_b"][blk] = wk, b
    if n_res != nb - 1:
        raise ValueError("WaveNet encoder: expected %d residual convs, found %d" % (nb - 1, n_res))

    d = tr.load(detect_path).main
    dc = [op for op in d.ops if op.name == "CONV_2D"]
    if len(dc) != 2 or d.ops[0].name != "RELU" or d.ops[-1].name != "SOFTMAX":
        raise ValueError("WaveNet detect graph not recognised")
    dw = _Walker(d)
    out["det1_w"] = d.tensors[dc[0].inputs[1]].data[:, 0, 0, :].astype(F32)
    b1 = d.tensors[dc[0].inputs[2]].data.astype(F32).copy()
    for k in dw.forward(dc[0].outputs[0]):
        if d.ops[k].name == "ADD":
            b1 = b1 + [dw.const(i) for i in d.ops[k].inputs if dw.const(i) is not None][0]
    out["det1_b"] = b1
    out["det2_w"] = d.tensors[dc[1].inputs[1]].data[:, 0, 0, :].astype(F32)
    out["det2_b"] = d.tensors[dc[1].inputs[2]].data.astype(F32)
    return out


# ----------------------------------------------------------------------------
def model_kind(model_type: str) -> str:
    """'CRNN' or 'WAVENET' (the reference upper-cases: wakeword/tflite.py:62)."""
    k = model_type.upper()
    if k not in ("CRNN", "WAVENET"):
        raise ValueError("model_type must be 'CRNN' or 'Wavenet', got %r" % (model_type,))
    return k


# trained tensors of the encode / detect files (everything the converter's float16 option touches; filter.tflite is
# never converted with it)
_FILTER_KEYS = ("mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale")
_NOT_TRAINED = ("mel_length", "dilation", "quant_source")


def quantize_fp16(weights: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
    """The fp16-quantised variant of a model as the reference's converters produce it
    (`optimizations=[DEFAULT]`, `supported_types=[float16]`: wwdetect/CRNN/convert_CRNN_tflite.py:23-37,
    wwdetect/wavenet/wavenet_model.py:149-163): every trained float32 constant of encode / detect is stored as
    float16 and widened back at run time, the arithmetic stays float32.  Idempotent."""
    out = {}
    for k, v in weights.items():
        if k in _FILTER_KEYS or k in _NOT_TRAINED or not isinstance(v, np.ndarray) or v.dtype != np.float32:
            out[k] = v
        else:
            out[k] = v.astype(np.float16).astype(np.float32)
    out["quant_source"] = np.array("derived")
    return out


def load_model_dir(model_dir: str, model_type: str, quant: bool = False) -> Dict[str, np.ndarray]:
    """All trained tensors (filter + encode + detect) of a reference model directory.
    quant=True: the float16 variant - from `encode-quant.tflite` / `detect-quant.tflite` when the directory holds them
    (`quant_source` = "file"), otherwise derived from the float32 files by the converter's rounding ("derived")."""
    kind = model_kind(model_type)
    if quant:
        enc, det = os.path.join(model_dir, "encode-quant.tflite"), os.path.join(model_dir, "detect-quant.tflite")
        if os.path.isfile(enc) and os.path.isfile(det):
            m = extract_crnn(enc, det) if kind == "CRNN" else extract_wavenet(enc, det)
            m.update(extract_filter(os.path.join(model_dir, "filter.tflite")))
            m["quant_source"] = np.array("file")
            return m
        return quantize_fp16(load_model_dir(model_dir, model_type))
    npz = os.path.join(model_dir, "weights.npz")
    if os.path.isfile(npz) and not os.path.isfile(os.path.join(model_dir, "encode.tflite")):
        with np.load(npz) as z:
            out = {k: z[k] for k in z.files}
        have = "CRNN" if "conv_w" in out else "WAVENET"
        if have != kind:
            raise ValueError("%s holds %s weights, model_type says %s" % (npz, have, kind))
        return out
    f = extract_filter(os.path.join(model_dir, "filter.tflite"))
    enc, det = os.path.join(model_dir, "encode.tflite"), os.path.join(model_dir, "detect.tflite")
    m = extract_crnn(enc, det) if kind == "CRNN" else extract_wavenet(enc, det)
    m.update(f)
    return m


def save_npz(weights: Dict[str, np.ndarray], path: str) -> None:
    np.savez(path, **weights)


def geometry(weights: Dict[str, np.ndarray]) -> Dict[str, int]:
    """Shape-driven configuration, as the reference derives it from the models'
    input/output details (wakeword/tflite.py:67-90)."""
    fft = (weights["mel_w"].shape[1] - 1) * 2
    if "conv_w" in weights:
        return {"kind": 0, "fft": fft, "mel_width": 40, "mel_length": int(weights["mel_length"]),
                "encode_length": 1, "encode_width": 64,
                "n_out": int(weights["det2_w"].shape[0])}
    return {"kind": 1, "fft": fft, "mel_width": int(weights["in_w"].shape[1]), "mel_length": int(weights["mel_length"]),
            "encode_length": int(weights["mel_length"]), "encode_width": 32, "n_out": 2}
