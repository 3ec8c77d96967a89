"""Generate tests/golden/*.npz by running the UNMODIFIED reference cell on the numpy TF1 shim.

    python oracle/gen_golden.py            # needs /root/reference (build container only)

For every case below this imports `/root/reference/{config,ops,mac_cell}.py` (never copied into the
repo), sets the reference's global `config` through its own `parseArgs()` (`config.py:95-424`),
restates the ten-line caller `MACnet.MACnetwork` (`model.py:428-458`: construct, zero_state, static
netLength unroll), and records per-step control / memory / info / contControl and the attention maps.
Variable *values* come from `mac_network_b200.params.init_params` (so the product, the oracle and the
reference all see identical weights); variable *names and shapes* are whatever the reference creates
and are stored in the fixture so the product's enumeration can be checked against them.

The fixtures pin `oracle/mac_oracle.py`; they cannot travel any other way, because neither
`/root/reference` nor TensorFlow exists on the GPU box.
"""
import importlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference"
sys.path.insert(0, os.path.join(HERE, "tf1_shim"))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import tensorflow as tf                      # noqa: E402  (the shim)
from mac_network_b200.config import MACConfig  # noqa: E402
from mac_network_b200.params import init_params, perturb_biases  # noqa: E402
from mac_network_b200.synthetic import make_inputs  # noqa: E402

COMMON = ["--memoryVariationalDropout", "--relu=ELU", "--controlContextual", "--readProjInputs",
          "--readMemConcatKB", "--readMemConcatProj", "--readMemProj", "--readCtrl", "--writeMemProj"]
ARGS = COMMON + ["--initCtrl=Q", "--controlInputUnshared"]
SMALL = dict(B=3, S=5, N=7, d=16, L=3)

# name -> (flag source, extra flags, shape, train?)
CASES = {
    # the five shipped flag files, read from the reference's own configs/ directory
    "args_small": ("@args.txt", [], SMALL, False),
    "args1_small": ("@args1.txt", [], SMALL, False),
    "args2_small": ("@args2.txt", [], SMALL, False),
    "args3_small": ("@args3.txt", [], SMALL, False),
    "args4_small": ("@args4.txt", [], SMALL, False),
    "gqa_small": ("@args3.txt", ["--writeGate"], dict(B=3, S=4, N=9, d=16, L=4), False),
    # training mode (dropouts at config.py:210-212 defaults, plus a write dropout)
    "args_train_small": ("@args.txt", [], SMALL, True),
    "args1_train_small": ("@args1.txt", [], SMALL, True),
    "gqa_train_small": ("@args3.txt", ["--writeGate", "--writeDropout=0.9"], dict(B=3, S=4, N=9, d=16, L=4), True),
    "novardp_train_small": (None, [f for f in ARGS if f != "--memoryVariationalDropout"], SMALL, True),
    # other working flags (SURVEY.md section 8(a) "P2")
    "p2_control": (None, ARGS + ["--controlConcatWords", "--controlProj", "--controlProjAct=TANH",
                                 "--controlInWordsProj"], SMALL, False),
    "p2_control_feed": (None, COMMON + ["--initCtrl=ZERO", "--controlFeedPrev", "--controlContAct=RELU",
                                        "--controlOutWordsProj", "--controlInputAct=RELU"], SMALL, False),
    "p2_ablations": (None, ARGS + ["--controlContinuous"], SMALL, False),
    "p2_wholeq": (None, ARGS + ["--controlWholeQ", "--initMem=Q"], SMALL, False),
    "p2_unshared": (None, ARGS + ["--unsharedCells", "1", "--initMem=ZERO"], SMALL, False),
    "p2_read_bl": (None, ARGS + ["--readMemAttType=BL", "--readCtrlAttType=BL", "--readProjShared",
                                 "--readMemAct=TANH", "--readCtrlAct=NON"], SMALL, False),
    "p2_read_add": (None, ARGS + ["--readMemAttType=ADD", "--readCtrlAttType=ADD", "--mulBias=0.5",
                                  "--readCtrlConcatKB", "--readCtrlConcatProj", "--readSmryKBProj"], SMALL, False),
    "p2_read_plain": (None, ["--relu=STD", "--controlContextual", "--readCtrl", "--readCtrlConcatKB",
                             "--mulBias=0.25", "--initCtrl=Q"], SMALL, False),
    "p2_read_noproj": (None, ["--relu=ELU", "--readProjInputs", "--readMemAct=NON"], SMALL, False),
    "p2_write_info": (None, ARGS + ["--writeInputs=INFO", "--writeInfoProj", "--writeInfoAct=RELU",
                                    "--writeMergeCtrl", "--writeMemAct=TANH"], SMALL, False),
    "p2_write_sum": (None, ARGS + ["--writeInputs=SUM", "--writeSelfAtt", "--writeGate",
                                   "--writeGateBias=-0.5"], SMALL, False),
    "p2_write_mem": (None, [f for f in ARGS if f != "--writeMemProj"] + ["--writeInputs=MEM"], SMALL, False),
    "p2_write_mul": (None, ARGS + ["--writeConcatMul", "--writeSelfAtt"], SMALL, False),
    # training mode on the composed path: which tensors the read unit drops there, and over what width (mac_cell.py:266)
    "p2_read_add_train": (None, ARGS + ["--readMemAttType=ADD", "--readCtrlAttType=ADD", "--mulBias=0.5",
                                        "--readCtrlConcatKB", "--readCtrlConcatProj", "--readSmryKBProj"], SMALL, True),
    "p2_read_plain_train": (None, ["--relu=STD", "--controlContextual", "--readCtrl", "--readCtrlConcatKB",
                                   "--mulBias=0.25", "--initCtrl=Q"], SMALL, True),
    # batch-normalised memory (mac_cell.py:369-373): stored statistics at eval, batch statistics + their update in training
    "p2_memory_bn": (None, ARGS + ["--memoryBN", "--bnCenter", "--bnScale", "--bnDecay=0.9"], SMALL, False),
    "p2_memory_bn_train": (None, ARGS + ["--memoryBN", "--bnCenter", "--bnDecay=0.9", "--writeGate"],
                           dict(B=5, S=5, N=7, d=16, L=3), True),
    # BASELINE.json configs[0]/[1]: S=20, 14x14 KB, d=512, netLength=4 (float32 storage) at B=16, half their batch, so
    # that the fixture stays under 1 MB (samples are independent at eval; the GPU tests still run B=32 against the oracle)
    "args_cpu_ref": ("@args.txt", [], dict(B=16, S=20, N=196, d=512, L=4), False),
    "gqa_mid": ("@args3.txt", ["--writeGate"], dict(B=8, S=30, N=49, d=512, L=6), False),
}

_ref_config = importlib.import_module("config")
_ref_ops = importlib.import_module("ops")
_ref_cell = importlib.import_module("mac_cell")


def set_reference_config(src, extra, shape, train):
    argv = ["gen_golden"]
    if src is not None:
        argv.append("@" + os.path.join(REF, "configs", src[1:]))
    argv += list(extra)
    argv += ["--netLength", str(shape["L"]), "--memDim", str(shape["d"]), "--ctrlDim", str(shape["d"]),
             "--attDim", str(shape["d"])]
    # a fresh namespace each time: parseArgs() fills the module-global `config` in place
    for k in list(vars(_ref_config.config).keys()):
        delattr(_ref_config.config, k)
    old = sys.argv
    sys.argv = argv
    try:
        _ref_config.parseArgs()
    finally:
        sys.argv = old
    return argv[1:]


def cell_flags_from_reference():
    """The cell-relevant flags, read back from the reference's parsed global config."""
    import dataclasses
    kw = {}
    for f in dataclasses.fields(MACConfig):
        if f.name in ("bnDecay", "bnCenter", "bnScale") and not _ref_config.config.memoryBN:
            continue          # recorded only where they matter, so the older fixtures regenerate byte for byte
        kw[f.name] = getattr(_ref_config.config, f.name)
    return kw


def run_case(name, src, extra, shape, train, seed=7):
    argv = set_reference_config(src, extra, shape, train)
    rc = _ref_config.config
    kw = cell_flags_from_reference()
    cfg = MACConfig(**kw).validate()
    B, S, N, d, L = (shape[k] for k in "BSNdL")
    inputs = make_inputs(B, S, N, d, seed=seed, dtype=np.float64)
    params = perturb_biases(init_params(cfg, L, seed=seed + 1, dtype=np.float64), seed=seed + 2)
    dp = {"memory": rc.memoryDropout, "read": rc.readDropout, "write": rc.writeDropout} if train else \
         {"memory": 1.0, "read": 1.0, "write": 1.0}          # model.py:118-125: 1.0 at eval
    store = tf.reset_shim(values=params, seed=seed + 3, dtype=np.float64)
    feed = {k: (tf.constant(v) if v.dtype != np.int32 else v) for k, v in inputs.items()}   # feed_dict analogue

    # ---- model.py:428-458 restated: MACnetwork scope, construct, zero_state, unroll
    conts = []
    with tf.variable_scope("MACnetwork"):
        cell = _ref_cell.MACCell(
            vecQuestions=feed["vecQuestions"], questionWords=feed["questionWords"],
            questionCntxWords=feed["questionCntxWords"], questionLengths=feed["questionLengths"],
            knowledgeBase=feed["knowledgeBase"], memoryDropout=dp["memory"], readDropout=dp["read"],
            writeDropout=dp["write"], batchSize=B, train=train, reuse=None)
        state = cell.zero_state(B, tf.float32)
        none = tf.zeros((B, 1), dtype=tf.float32)
        for i in range(rc.netLength):
            cell.iteration = i
            _, state = cell(none, state)
            conts.append(cell.contControl)

    created = {k: list(v.shape) for k, v in store.vars.items()}
    missing = sorted(set(created) - set(params))
    unused = sorted(set(params) - set(created))
    assert not missing and not unused, (name, "reference created but not enumerated:", missing,
                                        "enumerated but never created:", unused)
    big = d >= 256
    st = np.float32 if big else np.float64
    out = {
        "control": cell.controls[:, 1:].transpose(1, 0, 2).astype(st),
        "memory": cell.memories[:, 1:].transpose(1, 0, 2).astype(st),
        "info": cell.infos[:, 1:].transpose(1, 0, 2).astype(st),
        "contControl": np.stack(conts).astype(st),
        "final_control": np.asarray(state.control, st),
        "final_memory": np.asarray(state.memory, st),
        "att_question": np.stack(cell.attentions["question"]).astype(st),
        "att_kb": np.stack(cell.attentions["kb"]).astype(st),
    }
    if cell.attentions["gate"]:
        out["att_gate"] = np.stack(cell.attentions["gate"]).astype(st)
    for i, a in enumerate(cell.attentions["self"]):
        out["att_self_%d" % i] = np.asarray(a, st)
    for i, u in enumerate(store.uniform_draws):
        out["uniform_%03d" % i] = u.astype(np.float64)
    if rc.memoryBN:          # the stored statistics after the forward (moved by the training forward, untouched at eval)
        for k, v in store.vars.items():
            if "/BatchNorm/moving_" in k:
                out["final_bn_" + k.rsplit("/", 1)[-1]] = np.asarray(v, np.float64)
    # the cell must not modify its inputs (SURVEY 8(b) ownership)
    chk = make_inputs(B, S, N, d, seed=seed, dtype=np.float64)
    for k in chk:
        assert np.array_equal(chk[k], inputs[k]), k
    meta = {"case": name, "argv": [a.replace(REF + "/", "") for a in argv], "cell_flags": kw, "shape": shape,
            "train": train, "dropouts": dp, "input_seed": seed, "param_seed": seed + 1, "bias_seed": seed + 2,
            "variables": created, "n_uniform": len(store.uniform_draws), "reference_commit": "118d9b6a"}
    out["meta_json"] = np.frombuffer(json.dumps(meta, sort_keys=True).encode(), dtype=np.uint8)
    return out


def run_output_case(name, train, seed=17, B=6, d=16, A=12, hidden=(8,)):
    """Output unit + classifier + loss through the reference's own MACnet methods (model.py:512-528, 547-576, 593-596)."""
    import types
    ref_model = importlib.import_module("model")
    set_reference_config("@args.txt", ["--outClassifierDims"] + [str(h) for h in hidden], dict(L=1, d=d), train)
    rc = _ref_config.config
    rc.answerWordsNum = A
    from mac_network_b200.output_unit import output_specs, init_output_params
    specs = output_specs(d, d, list(hidden), A)
    params = init_output_params(specs, seed=seed, dtype=np.float64)
    rng = np.random.RandomState(seed + 1)
    memory, vecq = rng.standard_normal((B, d)), 0.5 * np.tanh(rng.standard_normal((B, d)))
    answers = rng.randint(0, A, size=(B,)).astype(np.int32)
    keep = rc.outputDropout if train else 1.0
    store = tf.reset_shim(values=params, seed=seed + 2, dtype=np.float64)
    me = types.SimpleNamespace(dropouts={"output": keep}, batchNorm=None, answerLossList=[])
    feats, dim = ref_model.MACnet.outputOp(me, tf.constant(memory), tf.constant(vecq), None, None)
    logits = ref_model.MACnet.classifier(me, feats, dim)
    loss, losses = ref_model.MACnet.addAnswerLossOp(me, logits, answers)
    created = {k: list(v.shape) for k, v in store.vars.items()}
    assert created == {k: list(v[0]) for k, v in specs.items()}, (created, specs)
    out = {"logits": np.asarray(logits), "losses": np.asarray(losses), "loss": np.asarray(loss),
           "memory": memory, "vecQuestions": vecq, "answers": answers}
    for i, u in enumerate(store.uniform_draws):
        out["uniform_%03d" % i] = u.astype(np.float64)
    if rc.memoryBN:          # the stored statistics after the forward (moved by the training forward, untouched at eval)
        for k, v in store.vars.items():
            if "/BatchNorm/moving_" in k:
                out["final_bn_" + k.rsplit("/", 1)[-1]] = np.asarray(v, np.float64)
    meta = {"case": name, "train": train, "keep": keep, "B": B, "d": d, "A": A, "hidden": list(hidden), "param_seed": seed,
            "relu": rc.relu, "variables": created, "n_uniform": len(store.uniform_draws)}
    out["meta_json"] = np.frombuffer(json.dumps(meta, sort_keys=True).encode(), dtype=np.uint8)
    return out


def run_stem_case(name, train, seed=23, B=2, H=5, W=4, cin=8, cout=8):
    """Image stem through the reference's own `ops.CNNLayer` as `MACnet.stem` calls it (model.py:165-204, ops.py:380-438)."""
    set_reference_config("@args.txt", ["--stemDim", str(cout)], dict(L=1, d=cout), train)
    rc = _ref_config.config
    from mac_network_b200.stem import stem_specs, init_stem_params
    specs = stem_specs(cin, cout, rc.stemNumLayers, rc.stemKernelSize)
    params = init_stem_params(specs, seed=seed, dtype=np.float64)
    images = np.maximum(np.random.RandomState(seed + 1).standard_normal((B, H, W, cin)), 0)    # post-ReLU ResNet features
    keep = rc.stemDropout if train else 1.0
    store = tf.reset_shim(values=params, seed=seed + 2, dtype=np.float64)
    dims = [cin] + [rc.stemDim] * (rc.stemNumLayers - 1) + [cout]
    with tf.variable_scope("stem"):
        feats = _ref_ops.CNNLayer(tf.constant(images), dims, batchNorm=None, dropout=keep,
                                  kernelSizes=rc.stemKernelSizes, strides=rc.stemStrideSizes)
        kb = tf.reshape(feats, (B, -1, cout))
    created = {k: list(v.shape) for k, v in store.vars.items()}
    assert created == {k: list(v[0]) for k, v in specs.items()}, (created, specs)
    out = {"images": images, "kb": np.asarray(kb)}
    for i, u in enumerate(store.uniform_draws):
        out["uniform_%03d" % i] = u.astype(np.float64)
    if rc.memoryBN:          # the stored statistics after the forward (moved by the training forward, untouched at eval)
        for k, v in store.vars.items():
            if "/BatchNorm/moving_" in k:
                out["final_bn_" + k.rsplit("/", 1)[-1]] = np.asarray(v, np.float64)
    meta = {"case": name, "train": train, "keep": keep, "shape": [B, H, W, cin, cout], "layers": rc.stemNumLayers,
            "ksize": rc.stemKernelSize, "param_seed": seed, "relu": rc.relu, "variables": created,
            "n_uniform": len(store.uniform_draws)}
    out["meta_json"] = np.frombuffer(json.dumps(meta, sort_keys=True).encode(), dtype=np.uint8)
    return out


def run_encoder_case(name, train, proj, seed=29, B=5, S=7, V=11, E=12, enc_dim=16, bi=True):
    """Question input unit through the reference's own `MACnet.qEmbeddingsOp` + `MACnet.encoder` (model.py:208-220, 279-307)
    -> `ops.RNNLayer` / `biRNNLayer` (ops.py:859-952) on the shim's BasicLSTMCell / bidirectional_dynamic_rnn."""
    import types
    ref_model = importlib.import_module("model")
    ctrl = enc_dim + 4 if proj else enc_dim
    extra = ["--encDim", str(enc_dim), "--wrdEmbDim", str(E)] + (["--encProj"] if proj else [])
    if bi:
        set_reference_config("@args.txt", extra, dict(L=1, d=ctrl), train)
    else:                                                      # args.txt without --encBi: ops.fwRNNLayer (ops.py:797-829)
        set_reference_config(None, [f for f in ARGS] + extra, dict(L=1, d=ctrl), train)
    rc = _ref_config.config
    assert rc.encBi == bi and rc.encType == "LSTM" and rc.encNumLayers == 1 and not rc.encVariationalDropout
    from mac_network_b200.encoder import encoder_specs, init_encoder_params
    specs = encoder_specs(V, E, enc_dim, ctrl_dim=ctrl, bi=bi, proj=proj)
    params = init_encoder_params(specs, seed=seed, dtype=np.float64)
    rng = np.random.RandomState(seed + 1)
    lengths = rng.randint(1, S + 1, size=(B,)).astype(np.int32)
    lengths[0] = S                                             # the batch is trimmed to its longest question (model.py:681-687)
    lengths[1] = 1
    q = rng.randint(1, V + 1, size=(B, S)).astype(np.int32)
    q[np.arange(S)[None, :] >= lengths[:, None]] = 0           # padding id
    keep_in, keep_q = (rc.encInputDropout, rc.qDropout) if train else (1.0, 1.0)
    store = tf.reset_shim(values=params, seed=seed + 2, dtype=np.float64)
    me = types.SimpleNamespace(dropouts={"encInput": keep_in, "question": keep_q, "stateInput": 1.0})
    emb_init = params["qEmbeddings/emb"]
    words, _ = ref_model.MACnet.qEmbeddingsOp(me, q, emb_init)
    projFlag = (rc.encDim != rc.ctrlDim) or rc.encProj                                   # model.py:786
    cntx, vecq = ref_model.MACnet.encoder(me, words, lengths, projFlag, projFlag, rc.ctrlDim)
    created = {k: list(v.shape) for k, v in store.vars.items()}
    assert created == {k: list(v[0]) for k, v in specs.items()}, (created, specs)
    out = {"qIndices": q, "questionLengths": lengths, "questionWords": np.asarray(words),
           "questionCntxWords": np.asarray(cntx), "vecQuestions": np.asarray(vecq)}
    for i, u in enumerate(store.uniform_draws):
        out["uniform_%03d" % i] = u.astype(np.float64)
    if rc.memoryBN:          # the stored statistics after the forward (moved by the training forward, untouched at eval)
        for k, v in store.vars.items():
            if "/BatchNorm/moving_" in k:
                out["final_bn_" + k.rsplit("/", 1)[-1]] = np.asarray(v, np.float64)
    meta = {"case": name, "train": train, "proj": proj, "bi": bi, "keep_input": keep_in, "keep_question": keep_q,
            "shape": {"B": B, "S": S, "V": V, "E": E, "encDim": enc_dim, "ctrlDim": ctrl}, "param_seed": seed,
            "variables": created, "n_uniform": len(store.uniform_draws)}
    out["meta_json"] = np.frombuffer(json.dumps(meta, sort_keys=True).encode(), dtype=np.uint8)
    return out


def main():
    outdir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    only = sys.argv[1:]
    for name, (src, extra, shape, train) in CASES.items():
        if only and name not in only:
            continue
        out = run_case(name, src, extra, shape, train)
        path = os.path.join(outdir, name + ".npz")
        np.savez_compressed(path, **out)
        print("%-22s %8.1f KB  vars=%d draws=%d" % (name, os.path.getsize(path) / 1024.0,
                                                     len(json.loads(bytes(out["meta_json"]).decode())["variables"]),
                                                     sum(k.startswith("uniform_") for k in out)))
    for name, train in (("stem_eval", False), ("stem_train", True)):
        if only and name not in only:
            continue
        out = run_stem_case(name, train)
        path = os.path.join(outdir, name + ".npz")
        np.savez_compressed(path, **out)
        print("%-22s %8.1f KB" % (name, os.path.getsize(path) / 1024.0))
    for name, train, proj, bi in (("encoder_eval", False, False, True), ("encoder_train", True, False, True),
                                  ("encoder_proj", False, True, True), ("encoder_uni", False, False, False)):
        if only and name not in only:
            continue
        out = run_encoder_case(name, train, proj, bi=bi)
        path = os.path.join(outdir, name + ".npz")
        np.savez_compressed(path, **out)
        print("%-22s %8.1f KB" % (name, os.path.getsize(path) / 1024.0))
    for name, train in (("output_eval", False), ("output_train", True)):
        if only and name not in only:
            continue
        out = run_output_case(name, train)
        path = os.path.join(outdir, name + ".npz")
        np.savez_compressed(path, **out)
        print("%-22s %8.1f KB" % (name, os.path.getsize(path) / 1024.0))


if __name__ == "__main__":
    main()
