"""Reader for the reference's TensorFlow-1.14 ``.meta.txt`` graph files (text-proto MetaGraphDef).

The reference executes the graph through ``tensorflow::Session`` (``ppo2/session_creator.hpp:23-57``);
this framework has no TensorFlow, so the graph file is only *read*: hidden sizes come from the
``VariableV2`` shapes of ``model/{pi,vf}_fc{k}/w``, the initial weights from the ``Const``
``tensor_content`` of ``model/*/Initializer/*`` and the constants that the graph bakes in
(entropy coefficient ``loss/mul_4/y``, value coefficient ``loss/mul_5/y``, clip norm
``loss/clip_by_global_norm/mul/x``, Adam ``ppo2/_train/{beta1,beta2,epsilon}``) and which value loss the
graph builds (``vf_clip``, see ``classify_vf_clip``).

This is the Python twin of ``csrc/meta_parser.cpp`` (the one the product path uses); tests check that
both agree on the reference fixture.  No protobuf dependency: a 60-line recursive text-proto reader.
"""
from __future__ import annotations

import re
import struct
from dataclasses import dataclass, field
from typing import Dict, List, Tuple

import numpy as np

# Trainable tensors in the order of the graph's gradient list (GRAPH:23738-24074), then the
# untrained q head that the Saver still stores (GRAPH:32396).
TENSOR_ORDER = [
    "model/pi_fc0/w", "model/pi_fc0/b", "model/vf_fc0/w", "model/vf_fc0/b",
    "model/pi_fc1/w", "model/pi_fc1/b", "model/vf_fc1/w", "model/vf_fc1/b",
    "model/vf/w", "model/vf/b", "model/pi/w", "model/pi/b", "model/pi/logstd",
    "model/q/w", "model/q/b",
]
N_TRAINABLE_TENSORS = 13
LOGSTD = "model/pi/logstd"  # absent with a categorical head (Discrete action space): 14 tensors, 12 trainable

_TOKEN = re.compile(r'\s*(?:([A-Za-z_][A-Za-z0-9_]*)|([{}:])|("(?:[^"\\]|\\.)*")|([-+0-9.eE]+[A-Za-z]*|-?inf|nan))')


def _unescape(s: str) -> bytes:
    """C-style unescape of a text-proto string literal body (octal \\ooo, \\n, \\t, \\", \\\\ ...)."""
    out = bytearray()
    i, n = 0, len(s)
    simple = {"n": 10, "t": 9, "r": 13, '"': 34, "'": 39, "\\": 92, "a": 7, "b": 8, "f": 12, "v": 11}
    while i < n:
        c = s[i]
        if c != "\\":
            out += c.encode("latin-1") if ord(c) < 256 else c.encode("utf-8")
            i += 1
            continue
        i += 1
        c = s[i]
        if c in "01234567":
            j = i
            while j < n and j < i + 3 and s[j] in "01234567":
                j += 1
            out.append(int(s[i:j], 8) & 0xFF)
            i = j
        elif c == "x":
            j = i + 1
            while j < n and j < i + 3 and s[j] in "0123456789abcdefABCDEF":
                j += 1
            out.append(int(s[i + 1:j], 16))
            i = j
        else:
            out.append(simple[c])
            i += 1
    return bytes(out)


def _parse_block(text: str, pos: int) -> Tuple[dict, int]:
    """Parse fields until the matching '}' (or EOF). Returns ({name: [values...]}, new_pos)."""
    msg: Dict[str, list] = {}
    n = len(text)
    while True:
        m = _TOKEN.match(text, pos)
        if not m:
            return msg, n
        if m.group(2) == "}":
            return msg, m.end()
        key = m.group(1)
        if key is None:
            raise ValueError(f"text-proto: expected field name at offset {pos}: {text[pos:pos+40]!r}")
        pos = m.end()
        m = _TOKEN.match(text, pos)
        if m.group(2) == ":":
            pos = m.end()
            m = _TOKEN.match(text, pos)
        if m.group(2) == "{":
            val, pos = _parse_block(text, m.end())
        elif m.group(3) is not None:
            val, pos = _unescape(m.group(3)[1:-1]), m.end()
        elif m.group(4) is not None:
            val, pos = m.group(4), m.end()
        else:  # enum / bool identifier
            val, pos = m.group(1), m.end()
        msg.setdefault(key, []).append(val)


@dataclass
class MetaInfo:
    hidden: List[int]
    obs_dim: int
    act_dim: int
    tensors: Dict[str, np.ndarray]
    ent_coef: float
    vf_coef: float
    clip_norm: float
    beta1: float
    beta2: float
    adam_eps: float
    tf_version: str = ""
    vf_clip: str = "shared"
    activation: str = "tanh"
    action_space: str = "box"
    shapes: Dict[str, Tuple[int, ...]] = field(default_factory=dict)

    def flat_params(self, include_q: bool = True) -> np.ndarray:
        names = TENSOR_ORDER if include_q else TENSOR_ORDER[:N_TRAINABLE_TENSORS]
        return np.concatenate([self.tensors[n].ravel() for n in names if n in self.tensors]).astype(np.float32)


def _attr(node: dict, key: str) -> dict | None:
    for a in node.get("attr", []):
        if a["key"][0] == key.encode():
            return a["value"][0]
    return None


def _tensor_value(node: dict) -> np.ndarray:
    t = _attr(node, "value")["tensor"][0]
    dims = [int(d["size"][0]) for d in t.get("tensor_shape", [{}])[0].get("dim", [])]
    count = int(np.prod(dims)) if dims else 1
    if "tensor_content" in t:
        arr = np.frombuffer(t["tensor_content"][0], dtype="<f4").copy()
    elif "float_val" in t:
        vals = [float(v) for v in t["float_val"]]
        arr = np.full(count, vals[0], dtype=np.float32) if len(vals) == 1 else np.asarray(vals, np.float32)
    else:  # all-zero tensors carry neither field
        arr = np.zeros(count, dtype=np.float32)
    return arr.reshape(dims) if dims else arr.reshape(())


def _inputs(node: dict) -> List[str]:
    """Data inputs of a node ("name:0" -> "name"; control inputs "^name" skipped)."""
    return [i.decode().split(":")[0] for i in node.get("input", []) if not i.startswith(b"^")]


def classify_vf_clip(nodes: Dict[str, dict]) -> str:
    """The value loss of Stable-Baselines' PPO2, vf_loss = 0.5 * mean(max(square(vpred - R), square(vpred_clipped - R))):
    "none" (vpred_clipped is vpred), "shared" / "separate" (old_vpred_ph + clip_by_value(vpred - old_vpred_ph, -b, b) with
    b = loss/clip_range_ph / loss/clip_range_vf_ph), from the data flow behind the second operand of loss/Maximum.  A graph
    without loss/Maximum is "shared" (the shipped graph's form); any other shape raises ValueError.  Twin of
    classify_vf_clip in csrc/meta_parser.cpp."""
    def node(name, op):
        n = nodes.get(name)
        return n if n is not None and n["op"][0] == op.encode() else None

    def sub_of_square(sq):
        s = node(sq, "Square")
        if s is None or len(_inputs(s)) != 1:
            return None
        d = node(_inputs(s)[0], "Sub")
        return _inputs(d) if d is not None and len(_inputs(d)) == 2 else None

    if "loss/Maximum" not in nodes:
        return "shared"
    mx = node("loss/Maximum", "Maximum")
    mi = _inputs(mx) if mx is not None else []
    s1 = sub_of_square(mi[0]) if len(mi) == 2 else None
    s2 = sub_of_square(mi[1]) if len(mi) == 2 else None
    if s1 is None or s2 is None or s1[1] != s2[1]:
        raise ValueError("loss/Maximum is not max(square(vpred - R), square(vpred_clipped - R))")
    if s2[0] == s1[0]:
        return "none"
    add = node(s2[0], "Add")
    ai = _inputs(add) if add is not None else []
    if len(ai) == 2 and ai[1] == "loss/old_vpred_ph":
        ai = [ai[1], ai[0]]
    clip = node(ai[1], "Maximum") if len(ai) == 2 and ai[0] == "loss/old_vpred_ph" else None  # clip_by_value = max(min(x, b), -b)
    ci = _inputs(clip) if clip is not None else []
    mn = node(ci[0], "Minimum") if len(ci) == 2 else None
    neg = node(ci[1], "Neg") if len(ci) == 2 else None
    ni = _inputs(mn) if mn is not None else []
    gi = _inputs(neg) if neg is not None else []
    if len(ni) != 2 or len(gi) != 1 or ni[1] != gi[0]:
        raise ValueError(f"the clipped value {s2[0]} is neither vpred nor old_vpred_ph + clip_by_value(..., -b, b)")
    if ni[1] == "loss/clip_range_ph":
        return "shared"
    if ni[1] == "loss/clip_range_vf_ph":
        return "separate"
    raise ValueError(f"the value clip bound {ni[1]} is neither loss/clip_range_ph nor loss/clip_range_vf_ph")


_ACT_PAIRS = (("pi_fc0", "pi_fc1"), ("pi_fc1", "pi"), ("vf_fc0", "vf_fc1"), ("vf_fc1", "vf"))


def classify_activation(nodes: Dict[str, dict]) -> str:
    """The hidden-layer activation of Stable-Baselines' MlpPolicy, act(matmul(x, w) + b) with act = act_fun: for each
    (hidden layer L, reader N) pair, every forward MatMul (in the model/ or train_model/ scope, neither operand transposed;
    the gradient sub-graph's MatMuls also read the weights) whose weight operand is the read of model/N/w must take a Tanh
    or Relu of Add(MatMul(., read of model/L/w), read of model/L/b), and every pair has such a reader in both scopes.
    "tanh" / "relu" when all agree; a graph without forward nodes is "tanh"; anything else (another activation, mixed
    activations, a deeper or shared-trunk net_arch) raises ValueError.  Twin of classify_activation in csrc/meta_parser.cpp."""
    for v in ("model/pi_fc2/w", "model/vf_fc2/w", "model/shared_fc0/w"):
        if v in nodes:
            raise ValueError(f"variable {v}: only two hidden layers per tower, without a shared trunk, are supported")

    def op_of(name):
        n = nodes.get(name)
        return n["op"][0].decode() if n is not None else ""

    def is_read_of(name, var):
        return op_of(name) == "Identity" and _inputs(nodes[name]) == [var]

    def attr_true(node, key):
        v = _attr(node, key)
        return v is not None and v.get("b", ["false"])[0] == "true"

    def forward_scope(name):
        """0: model/, 1: train_model/, -1: neither or not a plain x * W product."""
        n = nodes.get(name)
        if n is None or op_of(name) != "MatMul" or attr_true(n, "transpose_a") or attr_true(n, "transpose_b"):
            return -1
        return 0 if name.startswith("model/") else 1 if name.startswith("train_model/") else -1

    first = None
    found = 0
    per_scope = [[0, 0] for _ in _ACT_PAIRS]
    for pi, (L, N) in enumerate(_ACT_PAIRS):
        for name in sorted(nodes):
            scope = forward_scope(name)
            if scope < 0:
                continue
            mi = _inputs(nodes[name])
            if len(mi) != 2 or not is_read_of(mi[1], f"model/{N}/w"):
                continue
            found += 1
            per_scope[pi][scope] += 1
            act, aop = mi[0], op_of(mi[0])
            if aop not in ("Tanh", "Relu"):
                raise ValueError(f"node {name} reads {act} (op {aop or 'missing'}), not a Tanh or Relu of layer {L}")
            ai = _inputs(nodes[act])
            add = ai[0] if len(ai) == 1 else ""
            di = _inputs(nodes[add]) if op_of(add) in ("Add", "AddV2", "BiasAdd") else []
            ok = False
            for s in range(2 if len(di) == 2 else 0):
                m, b = di[s], di[1 - s]
                if forward_scope(m) < 0 or not is_read_of(b, f"model/{L}/b"):
                    continue
                li = _inputs(nodes[m])
                ok = len(li) == 2 and is_read_of(li[1], f"model/{L}/w")
            if not ok:
                raise ValueError(f"activation node {act} (read by {name}) is not act(matmul(x, model/{L}/w) + model/{L}/b)")
            if first is None:
                first = (aop, act)
            elif aop != first[0]:
                raise ValueError(f"the graph mixes activations: {first[1]} is {first[0]}, {act} is {aop}")
    if found == 0:
        return "tanh"
    for (L, N), counts in zip(_ACT_PAIRS, per_scope):
        for scope, n in zip(("model/", "train_model/"), counts):
            if n == 0:
                raise ValueError(f"no forward MatMul under {scope} reads model/{N}/w")
    return "relu" if first[0] == "Relu" else "tanh"


def classify_action_space(nodes: Dict[str, dict], n: int) -> str:
    """The action space of Stable-Baselines' policy head: "box" (DiagGaussianProbabilityDistribution, with model/pi/logstd) or
    "discrete" (CategoricalProbabilityDistribution over the n logits of model/pi, no logstd).  PPO2's action placeholder
    loss/action_ph, when the graph has it, must agree: float [?, n] for "box", int32 / int64 [?] for "discrete"; otherwise
    ValueError naming the node.  Twin of classify_action_space in csrc/meta_parser.cpp."""
    box = LOGSTD in nodes
    ph = nodes.get("loss/action_ph")
    if ph is None:
        return "box" if box else "discrete"
    dt = _attr(ph, "dtype")
    dtype = dt["type"][0] if dt is not None and "type" in dt else ""
    shp = _attr(ph, "shape")
    dims = [int(d["size"][0]) for d in shp["shape"][0].get("dim", [])] if shp is not None and "shape" in shp else []
    if box and dtype == "DT_FLOAT" and len(dims) == 2 and dims[1] == n:
        return "box"
    if not box and dtype in ("DT_INT32", "DT_INT64") and len(dims) == 1:
        return "discrete"
    head = (f"Gaussian head (model/pi/logstd present): a Box space needs a float [?, {n}] placeholder" if box else
            "categorical head (no model/pi/logstd): a Discrete space needs an int32 / int64 [?] placeholder")
    raise ValueError(f"node loss/action_ph ({dtype or 'no dtype'}, rank {len(dims)}) contradicts the {head}")


def meta_action_space(path: str) -> str:
    """The action space of a graph file's policy head ("box" / "discrete"), read by this module's parser."""
    return parse_meta_txt(path).action_space


def meta_activation(path: str) -> str:
    """The hidden-layer activation of a graph file ("tanh" / "relu"), read by this module's parser."""
    return parse_meta_txt(path).activation


def parse_meta_txt(path: str) -> MetaInfo:
    with open(path, "r", encoding="latin-1") as f:
        text = f.read()
    root, _ = _parse_block(text, 0)
    graph = root["graph_def"][0]
    nodes = {n["name"][0].decode(): n for n in graph["node"]}

    shapes: Dict[str, Tuple[int, ...]] = {}
    tensors: Dict[str, np.ndarray] = {}
    for name in TENSOR_ORDER:
        if name == LOGSTD and name not in nodes:  # categorical head
            continue
        var = nodes[name]
        assert var["op"][0] == b"VariableV2", name
        shp = _attr(var, "shape")["shape"][0]
        shapes[name] = tuple(int(d["size"][0]) for d in shp.get("dim", []))
        init = None
        for suffix in ("initial_value", "Const", "zeros"):
            cand = nodes.get(f"{name}/Initializer/{suffix}")
            if cand is not None and cand["op"][0] == b"Const":
                init = _tensor_value(cand)
                break
        if init is None:
            raise ValueError(f"no Const initializer found for {name}")
        tensors[name] = np.ascontiguousarray(init.reshape(shapes[name]), dtype=np.float32)

    def scalar(name: str) -> float:
        return float(_tensor_value(nodes[name]).reshape(-1)[0])

    hidden = [shapes["model/pi_fc0/w"][1], shapes["model/pi_fc1/w"][1]]
    ver = ""
    try:
        ver = root["meta_info_def"][0]["tensorflow_version"][0].decode()
    except Exception:
        pass
    return MetaInfo(
        hidden=hidden,
        obs_dim=shapes["model/pi_fc0/w"][0],
        act_dim=shapes["model/pi/w"][1],
        tensors=tensors,
        ent_coef=scalar("loss/mul_4/y"),
        vf_coef=scalar("loss/mul_5/y"),
        clip_norm=scalar("loss/clip_by_global_norm/mul/x"),
        beta1=scalar("ppo2/_train/beta1"),
        beta2=scalar("ppo2/_train/beta2"),
        adam_eps=scalar("ppo2/_train/epsilon"),
        tf_version=ver,
        vf_clip=classify_vf_clip(nodes),
        activation=classify_activation(nodes),
        action_space=classify_action_space(nodes, shapes["model/pi/w"][1]),
        shapes=shapes,
    )


# TF Saver V2 bundle: the .data file is the tensors' raw bytes concatenated in the order of the
# (sorted) .index keys (ppo2/ppo2.hpp:107-131 runs the graph's Saver; GRAPH:32396 tensor_names).
CKPT_ORDER = sorted(TENSOR_ORDER)


def read_checkpoint_data(data_path: str, shapes: Dict[str, Tuple[int, ...]]) -> Dict[str, np.ndarray]:
    """The tensors of `shapes` (15, or 14 without logstd for a categorical head) from a Saver V2 .data file."""
    raw = np.fromfile(data_path, dtype="<f4")
    out, off = {}, 0
    for name in CKPT_ORDER:
        if name not in shapes:
            continue
        n = int(np.prod(shapes[name]))
        out[name] = raw[off:off + n].reshape(shapes[name]).copy()
        off += n
    if off != raw.size:
        raise ValueError(f"checkpoint data has {raw.size} floats, shapes need {off}")
    return out


def param_layout(obs_dim: int, act_dim: int, h1: int, h2: int, action_space: str = "box") -> Dict[str, Tuple[int, Tuple[int, ...]]]:
    """Offsets (in floats) of every tensor inside the flat parameter vector used by the core.  A categorical head
    (action_space "discrete", act_dim logits) has no logstd; the other tensors keep their order."""
    if action_space not in ("box", "discrete"):
        raise ValueError(f"action_space must be 'box' or 'discrete', not {action_space!r}")
    shp = {
        "model/pi_fc0/w": (obs_dim, h1), "model/pi_fc0/b": (h1,),
        "model/vf_fc0/w": (obs_dim, h1), "model/vf_fc0/b": (h1,),
        "model/pi_fc1/w": (h1, h2), "model/pi_fc1/b": (h2,),
        "model/vf_fc1/w": (h1, h2), "model/vf_fc1/b": (h2,),
        "model/vf/w": (h2, 1), "model/vf/b": (1,),
        "model/pi/w": (h2, act_dim), "model/pi/b": (act_dim,),
        "model/pi/logstd": (1, act_dim),
        "model/q/w": (h2, act_dim), "model/q/b": (act_dim,),
    }
    out, off = {}, 0
    for name in TENSOR_ORDER:
        if name == LOGSTD and action_space == "discrete":
            continue
        out[name] = (off, shp[name])
        off += int(np.prod(shp[name]))
    out["__total__"] = (off, ())
    return out


def _escape(b: bytes) -> str:
    out = []
    for c in b:
        if c == 0x5C:
            out.append("\\\\")
        elif c == 0x22:
            out.append('\\"')
        elif c == 0x27:
            out.append("\\'")
        elif 32 <= c < 127:
            out.append(chr(c))
        else:
            out.append("\\%03o" % c)
    return "".join(out)


def write_meta_txt(path: str, tensors: Dict[str, np.ndarray], ent_coef: float = 0.0, vf_coef: float = 0.5,
                   clip_norm: float = 0.5, beta1: float = 0.9, beta2: float = 0.999, adam_eps: float = 1e-5,
                   vf_clip: str | None = None, activation: str | None = None, action_space: str | None = None) -> None:
    """Write a minimal .meta.txt (variables + initialisers + baked constants) that both readers accept.

    The reference's graphs come from a Stable-Baselines/TensorFlow export script that is not part of the
    repo; this writer lets a user produce a graph file for other hidden sizes without TensorFlow.
    vf_clip = "shared" | "none" | "separate" adds the value-loss nodes that tell the readers which value loss the
    graph builds (Stable-Baselines' cliprange_vf None / < 0 / >= 0), named as Stable-Baselines names them;
    without it the file has no loss sub-graph and reads as "shared".
    activation = "tanh" | "relu" adds the forward nodes that tell the readers the hidden-layer activation (Stable-Baselines'
    act_fun), under model/ and train_model/ as Stable-Baselines names them; without it the file has none and reads as "tanh".
    action_space = "box" | "discrete" adds PPO2's action placeholder loss/action_ph (float [?, n] / int64 [?]); "discrete" also
    leaves model/pi/logstd out (a categorical head over the n columns of model/pi/w; `tensors` need not hold logstd).  Without it
    the file has no placeholder and a logstd, and reads as "box"."""
    if vf_clip not in (None, "shared", "none", "separate"):
        raise ValueError(f"vf_clip must be None, 'shared', 'none' or 'separate', not {vf_clip!r}")
    if activation not in (None, "tanh", "relu"):
        raise ValueError(f"activation must be None, 'tanh' or 'relu', not {activation!r}")
    if action_space not in (None, "box", "discrete"):
        raise ValueError(f"action_space must be None, 'box' or 'discrete', not {action_space!r}")
    def dims(shape, ind):
        return "".join(f"{ind}dim {{\n{ind}  size: {d}\n{ind}}}\n" for d in shape)

    def const_node(name, arr):
        arr = np.asarray(arr, np.float32)
        if arr.ndim == 0:
            val = f"          float_val: {float(arr)!r}\n"
        elif not arr.any():
            val = ""
        else:
            val = f'          tensor_content: "{_escape(arr.astype("<f4").tobytes())}"\n'
        return (f'  node {{\n    name: "{name}"\n    op: "Const"\n    attr {{\n      key: "dtype"\n      value {{\n        type: DT_FLOAT\n      }}\n    }}\n'
                f'    attr {{\n      key: "value"\n      value {{\n        tensor {{\n          dtype: DT_FLOAT\n          tensor_shape {{\n'
                f'{dims(arr.shape, "            ")}          }}\n{val}        }}\n      }}\n    }}\n  }}\n')

    def var_node(name, shape):
        return (f'  node {{\n    name: "{name}"\n    op: "VariableV2"\n    attr {{\n      key: "dtype"\n      value {{\n        type: DT_FLOAT\n      }}\n    }}\n'
                f'    attr {{\n      key: "shape"\n      value {{\n        shape {{\n{dims(shape, "          ")}        }}\n      }}\n    }}\n  }}\n')

    parts = ['meta_info_def {\n  tensorflow_version: "1.14.0"\n}\ngraph_def {\n']
    for name in TENSOR_ORDER:
        if name == LOGSTD and action_space == "discrete":
            continue
        arr = np.asarray(tensors[name], np.float32)
        parts.append(const_node(f"{name}/Initializer/initial_value", arr))
        parts.append(var_node(name, arr.shape))
    if action_space is not None:
        n = np.asarray(tensors["model/pi/w"]).shape[1]
        parts.append(_action_placeholder("DT_INT64", (-1,)) if action_space == "discrete" else _action_placeholder("DT_FLOAT", (-1, n)))
    if activation is not None:
        parts.append(_forward_nodes(activation))
    if vf_clip is not None:
        parts.append(_vf_loss_nodes(vf_clip))
    for name, val in (("loss/mul_4/y", ent_coef), ("loss/mul_5/y", vf_coef), ("loss/clip_by_global_norm/mul/x", clip_norm),
                      ("ppo2/_train/beta1", beta1), ("ppo2/_train/beta2", beta2), ("ppo2/_train/epsilon", adam_eps)):
        parts.append(const_node(name, np.float32(val)))
    parts.append("}\n")
    with open(path, "w", encoding="latin-1") as f:
        f.write("".join(parts))


def _action_placeholder(dtype: str, shape) -> str:
    """PPO2's loss/action_ph (train_model.pdtype.sample_placeholder([None])) with its dtype and shape attributes."""
    dims = "".join(f"          dim {{\n            size: {d}\n          }}\n" for d in shape)
    return (f'  node {{\n    name: "loss/action_ph"\n    op: "Placeholder"\n    attr {{\n      key: "dtype"\n      value {{\n        type: {dtype}\n      }}\n    }}\n'
            f'    attr {{\n      key: "shape"\n      value {{\n        shape {{\n{dims}        }}\n      }}\n    }}\n  }}\n')


def _op_node(name, kind, *inputs):
    ins = "".join(f'    input: "{i}"\n' for i in inputs)
    return f'  node {{\n    name: "{name}"\n    op: "{kind}"\n{ins}  }}\n'


def _forward_nodes(activation: str) -> str:
    """The forward pass of Stable-Baselines' MlpPolicy that classify_activation reads (ops and data inputs only): the
    variables' reads, then per scope (the act model, and train_model that reuses its variables) the hidden layers in
    mlp_extractor's order (pi_fc0, vf_fc0, pi_fc1, vf_fc1: activations Tanh, Tanh_1, ... or Relu, Relu_1, ...) and the heads."""
    kind = {"tanh": "Tanh", "relu": "Relu"}[activation]
    layers = ("pi_fc0", "pi_fc1", "vf_fc0", "vf_fc1", "vf", "pi")
    nodes = []
    for layer in layers:
        for v in ("w", "b"):
            nodes.append(_op_node(f"model/{layer}/{v}/read", "Identity", f"model/{layer}/{v}"))
    for scope in ("model", "train_model"):
        x = f"{scope}/flatten/Reshape"
        latent = {"pi": x, "vf": x}
        k = 0
        for idx in (0, 1):
            for tower in ("pi", "vf"):
                layer = f"{tower}_fc{idx}"
                act = f"{scope}/{kind}" + (f"_{k}" if k else "")
                k += 1
                nodes += [_op_node(f"{scope}/{layer}/MatMul", "MatMul", latent[tower], f"model/{layer}/w/read"),
                          _op_node(f"{scope}/{layer}/add", "Add", f"{scope}/{layer}/MatMul", f"model/{layer}/b/read"),
                          _op_node(act, kind, f"{scope}/{layer}/add")]
                latent[tower] = act
        for head, tower in (("vf", "vf"), ("pi", "pi")):
            nodes += [_op_node(f"{scope}/{head}/MatMul", "MatMul", latent[tower], f"model/{head}/w/read"),
                      _op_node(f"{scope}/{head}/add", "Add", f"{scope}/{head}/MatMul", f"model/{head}/b/read")]
    return "".join(nodes)


def _vf_loss_nodes(vf_clip: str) -> str:
    """The nodes of Stable-Baselines' value loss that classify_vf_clip reads (ops and data inputs only)."""
    def op(name, kind, *inputs):
        ins = "".join(f'    input: "{i}"\n' for i in inputs)
        return f'  node {{\n    name: "{name}"\n    op: "{kind}"\n{ins}  }}\n'

    v = "train_model/strided_slice"  # train_model.value_flat = vf[:, 0]
    nodes = [op("loss/rewards_ph", "Placeholder"), op("loss/old_vpred_ph", "Placeholder"), op("loss/clip_range_ph", "Placeholder"),
             op(v, "StridedSlice", "train_model/vf/add")]
    vc = v
    if vf_clip != "none":
        bound = "loss/clip_range_ph"
        if vf_clip == "separate":
            bound = "loss/clip_range_vf_ph"
            nodes.append(op(bound, "Placeholder"))
        nodes += [op("loss/sub", "Sub", v, "loss/old_vpred_ph"), op("loss/Neg", "Neg", bound),
                  op("loss/clip_by_value/Minimum", "Minimum", "loss/sub", bound),
                  op("loss/clip_by_value", "Maximum", "loss/clip_by_value/Minimum", "loss/Neg"),
                  op("loss/add", "Add", "loss/old_vpred_ph", "loss/clip_by_value")]
        vc = "loss/add"
    nodes += [op("loss/sub_1", "Sub", v, "loss/rewards_ph"), op("loss/Square_1", "Square", "loss/sub_1"),
              op("loss/sub_2", "Sub", vc, "loss/rewards_ph"), op("loss/Square_2", "Square", "loss/sub_2"),
              op("loss/Maximum", "Maximum", "loss/Square_1", "loss/Square_2")]
    return "".join(nodes)
