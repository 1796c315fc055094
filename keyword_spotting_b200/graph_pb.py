"""Weight formats of the reference: reading the frozen ``graph.pb`` / ``graph_octbit.pb`` it deploys.

The reference freezes its deployment graph with ``convert_variables_to_constants`` (main.py:339-348) and
rewrites it for octbit (main.py:357-371, octbit/octbit_graph.py:404-550); ``detector.py:134-146`` then loads the
GraphDef.  TensorFlow is not a dependency of this package, so this module carries a minimal protobuf wire-format
reader for exactly the messages involved (GraphDef / NodeDef / AttrValue / TensorProto / TensorShapeProto, field
numbers from TensorFlow's public .proto files) and maps the variable names of models/rnn_ctc.py to
``ModelWeights``:

    model/drnn/multi_rnn_cell/cell_{l}/gru_cell/gates/{kernel|weights}, .../{bias|biases}      (:236-243, get_cell)
    model/drnn/multi_rnn_cell/cell_{l}/gru_cell/candidate/{kernel|weights}, .../{bias|biases}
    model/weightsClasses, model/biasesClasses                                                  (:265-273)
    the [fft_size/2 + 1, n_mel] float Const feeding model/mel                                             (:139-148)

and, for the octbit-rewritten graph, every ``OctbitMatMul`` node to (qint8 weight ``[out, in]``, ``scale``, ``bias``)
(octbit/octbit_graph.py:527-536).
"""
from __future__ import annotations

import re
import struct
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np

# tensorflow/core/framework/types.proto
_DTYPES = {1: np.float32, 2: np.float64, 3: np.int32, 4: np.uint8, 5: np.int16, 6: np.int8, 9: np.int64, 10: np.bool_,
           11: np.int8, 12: np.uint8, 13: np.int32, 17: np.uint16, 19: np.float16, 22: np.uint32, 23: np.uint64}
DT_QINT8 = 11


class GraphFormatError(ValueError):
    pass


def _varint(buf, pos):
    result = shift = 0
    while True:
        if pos >= len(buf):
            raise GraphFormatError("truncated varint")
        b = buf[pos]
        pos += 1
        result |= (b & 0x7F) << shift
        if not b & 0x80:
            return result, pos
        shift += 7
        if shift > 70:
            raise GraphFormatError("varint too long")


def _fields(buf):
    """Yield (field_number, wire_type, value) of one message; value is int or a memoryview."""
    buf = memoryview(buf)
    pos = 0
    n = len(buf)
    while pos < n:
        key, pos = _varint(buf, pos)
        fno, wt = key >> 3, key & 7
        if wt == 0:
            v, pos = _varint(buf, pos)
        elif wt == 1:
            v = buf[pos:pos + 8]
            pos += 8
        elif wt == 2:
            ln, pos = _varint(buf, pos)
            if pos + ln > n:
                raise GraphFormatError("truncated length-delimited field")
            v = buf[pos:pos + ln]
            pos += ln
        elif wt == 5:
            v = buf[pos:pos + 4]
            pos += 4
        else:
            raise GraphFormatError("unsupported wire type %d" % wt)
        yield fno, wt, v


def _signed64(v):
    return v - (1 << 64) if v >= (1 << 63) else v


def _parse_shape(buf):
    dims = []
    for fno, wt, v in _fields(buf):
        if fno == 2 and wt == 2:                      # Dim
            size = 0
            for f2, w2, v2 in _fields(v):
                if f2 == 1 and w2 == 0:
                    size = _signed64(v2)
            dims.append(size)
    return tuple(dims)


def _packed(v, wt, fmt, size):
    if wt == 2:                                       # packed
        return list(struct.unpack("<%d%s" % (len(v) // size, fmt), bytes(v)))
    return [struct.unpack("<" + fmt, bytes(v))[0]]


def _parse_tensor(buf):
    dtype, shape, content = 1, (), None
    floats, doubles, ints, int64s, bools, halfs = [], [], [], [], [], []
    for fno, wt, v in _fields(buf):
        if fno == 1 and wt == 0:
            dtype = v
        elif fno == 2 and wt == 2:
            shape = _parse_shape(v)
        elif fno == 4 and wt == 2:
            content = bytes(v)
        elif fno == 5:
            floats += _packed(v, wt, "f", 4)
        elif fno == 6:
            doubles += _packed(v, wt, "d", 8)
        elif fno in (7, 13, 10, 11):                  # int_val, half_val, int64_val, bool_val: varints
            dst = {7: ints, 13: halfs, 10: int64s, 11: bools}[fno]
            if wt == 2:
                pos = 0
                while pos < len(v):
                    x, pos = _varint(v, pos)
                    dst.append(x)
            else:
                dst.append(v)
    if dtype not in _DTYPES:
        raise GraphFormatError("unsupported tensor dtype %d" % dtype)
    np_dt = np.dtype(_DTYPES[dtype])
    count = int(np.prod(shape)) if shape else 1
    if content is not None:
        arr = np.frombuffer(content, dtype=np_dt.newbyteorder("<")).astype(np_dt)
    else:
        vals = floats or doubles or int64s or ints or bools
        if halfs:
            arr = np.asarray(halfs, np.uint16).view(np.float16)
        elif np_dt.kind in "iu" or np_dt.kind == "b":
            arr = np.asarray([_signed64(x) if x >= (1 << 63) else (x - (1 << 32) if np_dt.itemsize <= 4 and x >= (1 << 31) else x)
                              for x in vals], np.int64).astype(np_dt)
        else:
            arr = np.asarray(vals, np_dt)
        if arr.size == 1 and count > 1:               # a single value fills the tensor (TensorProto convention)
            arr = np.full(count, arr[0], np_dt)
        elif arr.size == 0:
            arr = np.zeros(count, np_dt)
        elif arr.size < count:                        # the last value repeats
            arr = np.concatenate([arr, np.full(count - arr.size, arr[-1], np_dt)])
    if arr.size != count:
        raise GraphFormatError("tensor has %d values for shape %r" % (arr.size, shape))
    return arr.reshape(shape), dtype


def _parse_attr(buf):
    for fno, wt, v in _fields(buf):
        if fno == 8 and wt == 2:
            return _parse_tensor(v)[0]
        if fno == 4 and wt == 5:
            return struct.unpack("<f", bytes(v))[0]
        if fno == 3 and wt == 0:
            return _signed64(v)
        if fno == 5 and wt == 0:
            return bool(v)
        if fno == 2 and wt == 2:
            return bytes(v)
        if fno == 6 and wt == 0:
            return ("dtype", v)
        if fno == 7 and wt == 2:
            return _parse_shape(v)
    return None


@dataclass
class Node:
    name: str = ""
    op: str = ""
    inputs: List[str] = field(default_factory=list)
    attrs: Dict[str, object] = field(default_factory=dict)


def parse_graph_def(data: bytes) -> List[Node]:
    nodes = []
    for fno, wt, v in _fields(data):
        if fno != 1 or wt != 2:
            continue                                   # versions, library
        node = Node()
        for f2, w2, v2 in _fields(v):
            if f2 == 1 and w2 == 2:
                node.name = bytes(v2).decode("utf-8")
            elif f2 == 2 and w2 == 2:
                node.op = bytes(v2).decode("utf-8")
            elif f2 == 3 and w2 == 2:
                node.inputs.append(bytes(v2).decode("utf-8"))
            elif f2 == 5 and w2 == 2:
                key, val = None, None
                for f3, w3, v3 in _fields(v2):
                    if f3 == 1 and w3 == 2:
                        key = bytes(v3).decode("utf-8")
                    elif f3 == 2 and w3 == 2:
                        val = _parse_attr(v3)
                if key is not None:
                    node.attrs[key] = val
        nodes.append(node)
    if not nodes:
        raise GraphFormatError("no NodeDef found: not a GraphDef")
    return nodes


def load_graph(path_or_bytes) -> List[Node]:
    if isinstance(path_or_bytes, (bytes, bytearray, memoryview)):
        return parse_graph_def(bytes(path_or_bytes))
    with open(path_or_bytes, "rb") as f:
        return parse_graph_def(f.read())


def constants(nodes: List[Node]) -> Dict[str, np.ndarray]:
    """name -> value of every Const node."""
    return {n.name: n.attrs["value"] for n in nodes if n.op == "Const" and isinstance(n.attrs.get("value"), np.ndarray)}


_CELL = re.compile(r"(?:^|/)cell_(\d+)/gru_cell/(gates|candidate)/(kernel|weights|bias|biases)$")


def rnn_ctc_weights(nodes: List[Node], n_mel: Optional[int] = None, scope: str = "model", fft_size: int = 400):
    """Frozen rnn_ctc deployment graph -> keyword_spotting_b200.ModelWeights (and the implied sizes)."""
    from .rnn_ctc import ModelWeights
    consts = constants(nodes)
    layers: Dict[int, Dict[str, np.ndarray]] = {}
    fc_w = fc_b = mel = None
    bins = fft_size // 2 + 1
    other = []
    for name, val in consts.items():
        if scope and not name.startswith(scope + "/"):
            continue
        m = _CELL.search(name)
        if m:
            l, part, kind = int(m.group(1)), m.group(2), m.group(3)
            if val.dtype != np.float32:
                raise GraphFormatError("%s is %s, not float32: an octbit-rewritten graph -- read it with octbit_nodes()"
                                       % (name, val.dtype))
            key = part + ("_kernel" if kind in ("kernel", "weights") else "_bias")
            layers.setdefault(l, {})[key] = val.astype(np.float32)
        elif name.endswith("/weightsClasses"):
            fc_w = val.astype(np.float32)
        elif name.endswith("/biasesClasses"):
            fc_b = val.astype(np.float32)
        elif val.dtype == np.float32 and val.ndim == 2 and (n_mel is None or val.shape[1] == n_mel):
            if val.shape[0] == bins:
                mel = val
            else:
                other.append(tuple(val.shape))
    if not layers or fc_w is None or fc_b is None:
        raise GraphFormatError("not an rnn_ctc deployment graph: GRU / FC constants missing under scope %r" % scope)
    L = max(layers) + 1
    for l in range(L):
        missing = {"gates_kernel", "gates_bias", "candidate_kernel", "candidate_bias"} - set(layers.get(l, {}))
        if missing:
            raise GraphFormatError("layer %d lacks %s" % (l, sorted(missing)))
    if mel is None:
        hint = ""
        if other:
            hint = " (float [rows, n_mel] Consts of other shapes: %s; a [fft_size/2 + 1, n_mel] basis needs that fft_size)" % (
                ", ".join("[%d, %d]" % s for s in other))
        raise GraphFormatError("the [%d, n_mel] mel basis Const of fft_size = %d was not found%s" % (bins, fft_size, hint))
    return ModelWeights.from_arrays(mel, [layers[l]["gates_kernel"] for l in range(L)],
                                    [layers[l]["gates_bias"] for l in range(L)],
                                    [layers[l]["candidate_kernel"] for l in range(L)],
                                    [layers[l]["candidate_bias"] for l in range(L)], fc_w, fc_b)


@dataclass
class OctbitNode:
    name: str
    weight_q: np.ndarray          # [out, in] int8 (already transposed, octbit_graph.py:191-215)
    scale: float
    bias: np.ndarray              # [out] float32
    x_input: str
    weight_name: str = ""         # name of the qint8 Const (the variable the MatMul read before the rewrite)


def octbit_nodes(nodes: List[Node]) -> List[OctbitNode]:
    """Every OctbitMatMul of an octbit-rewritten graph with its constant operands (octbit_graph.py:527-536)."""
    by_name = {n.name: n for n in nodes}

    def resolve(name):                                 # through Identity / Enter to the Const (octbit_graph.py:488-524)
        name = name.split(":")[0].lstrip("^")
        seen = 0
        while name in by_name and by_name[name].op in ("Identity", "Enter") and seen < 16:
            name = by_name[name].inputs[0].split(":")[0]
            seen += 1
        return by_name.get(name)

    out = []
    for n in nodes:
        if n.op != "OctbitMatMul":
            continue
        w = resolve(n.inputs[1]) if len(n.inputs) > 1 else None
        if w is None or w.op != "Const" or not isinstance(w.attrs.get("value"), np.ndarray):
            raise GraphFormatError("OctbitMatMul %s: weight Const not found" % n.name)
        wq = w.attrs["value"]
        if wq.dtype != np.int8 or wq.ndim != 2:
            raise GraphFormatError("OctbitMatMul %s: weight must be a rank-2 qint8 Const" % n.name)
        if n.attrs.get("transpose_b") is False or n.attrs.get("transpose_a") is True:
            raise GraphFormatError("OctbitMatMul %s: only transpose_a=False, transpose_b=True exist (octbit_mat_mul_op.cc:41-44)" % n.name)
        scale = n.attrs.get("scale")
        bias = n.attrs.get("bias")
        if not isinstance(scale, float) or not isinstance(bias, np.ndarray):
            raise GraphFormatError("OctbitMatMul %s: scale / bias attrs missing" % n.name)
        out.append(OctbitNode(n.name, np.ascontiguousarray(wq), float(scale), bias.astype(np.float32).reshape(-1), n.inputs[0],
                              w.name))
    return out


def rnn_ctc_octbit_weights(nodes: List[Node], n_mel: Optional[int] = None, scope: str = "model", fft_size: int = 400):
    """Octbit-rewritten rnn_ctc deployment graph (``graph_octbit.pb``, main.py:357-371) ->
    ``(ModelWeights, OctbitModelWeights)``.

    The float Consts that survive the rewrite (cell_0, every bias, the mel basis, and the FC when it was left float)
    are read as in ``rnn_ctc_weights``; every ``OctbitMatMul`` is mapped through the name of its qint8 Const
    (``.../cell_{l}/gru_cell/{gates,candidate}/{kernel,weights}`` or ``.../weightsClasses``).  The float kernels of
    converted MatMuls no longer exist in the graph; ``ModelWeights`` carries their dequantised image
    (``W_q^T * scale``) so that the container stays complete -- the octbit forward never reads it."""
    from .rnn_ctc import ModelWeights, OctbitMatrix, OctbitModelWeights
    octs = octbit_nodes(nodes)
    if not octs:
        raise GraphFormatError("no OctbitMatMul node: not an octbit-rewritten graph")
    ow = OctbitModelWeights()
    deq: Dict[str, np.ndarray] = {}
    for o in octs:
        mat = OctbitMatrix(o.weight_q, float(np.float32(o.scale)), o.bias)
        m = _CELL.search(o.weight_name)
        if m and m.group(3) in ("kernel", "weights"):
            (ow.gates if m.group(2) == "gates" else ow.candidate)[int(m.group(1))] = mat
        elif o.weight_name.endswith("/weightsClasses"):
            ow.fc = mat
        else:
            raise GraphFormatError("OctbitMatMul %s reads %s, which is not a GRU kernel or the FC of rnn_ctc" % (o.name, o.weight_name))
        deq[o.weight_name] = (o.weight_q.T.astype(np.float32) * np.float32(o.scale)).astype(np.float32)
    patched = []
    for n in nodes:
        if n.op == "Const" and n.name in deq:
            n2 = Node(name=n.name, op=n.op, inputs=list(n.inputs), attrs=dict(n.attrs))
            n2.attrs["value"] = deq[n.name]
            patched.append(n2)
        else:
            patched.append(n)
    return rnn_ctc_weights(patched, n_mel=n_mel, scope=scope, fft_size=fft_size), ow
