"""CPU unit tests: graph codec / builder / interpreter, optimizers vs closed form, RW lock, bundle,
carrier codec, layout, compiler, Spark shim."""
import base64
import json
import os
import threading
import time

import numpy as np
import pytest
import torch
from hypothesis import given, settings
from hypothesis import strategies as st

from sparkflow_b200.graph import pbwire
from sparkflow_b200.graph import tfcompat as tf
from sparkflow_b200.graph.executor import GraphProgram, UnsupportedOp
from sparkflow_b200.graph.ir import GraphIR
from sparkflow_b200.graph_utils import build_graph
from sparkflow_b200.models import zoo
from sparkflow_b200.models.compiler import UnsupportedGraph, compile_graph
from sparkflow_b200.ops.layout import ParamLayout
from sparkflow_b200.ops.optimizers import NUM_SLOTS, OPT_IDS, OptimizerSpec, apply_update, init_slots
from sparkflow_b200.parallel.rwlock import RWLock

# a TF-1.7 checkpoint (MetaGraphDef + V2 bundle, 2-10 tanh-10 tanh-1 sigmoid with Adam slots) written by the original
# sparkflow test suite: the codec tests decode it and rewrite it byte for byte
FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "test_model", "to_load")


# ---------------------------------------------------------------------------------------------
# protobuf codec
# ---------------------------------------------------------------------------------------------
def test_pbwire_decodes_real_tf_metagraph():
    mg = pbwire.decode("MetaGraphDef", open(FIXTURE + ".meta", "rb").read())
    assert len(mg["graphDef"]["node"]) == 264 and mg["metaInfoDef"]["tensorflowVersion"] == "1.7.0"
    assert set(mg["collectionDef"]) == {"trainable_variables", "train_op", "variables"}
    vd = pbwire.decode("VariableDef", base64.b64decode(mg["collectionDef"]["trainable_variables"]["bytesList"]["value"][0]))
    assert vd == {"variableName": "dense/kernel:0", "initializerName": "dense/kernel/Assign", "snapshotName": "dense/kernel/read:0",
                  "initialValueName": "dense/kernel/Initializer/random_uniform:0"}
    assert pbwire.decode("MetaGraphDef", pbwire.encode("MetaGraphDef", mg)) == mg


@given(st.integers(min_value=-(2 ** 62), max_value=2 ** 62), st.text(max_size=20), st.floats(allow_nan=False, width=32))
@settings(max_examples=50, deadline=None)
def test_pbwire_scalar_roundtrip(i, s, f):
    msg = {"name": "n", "op": "Const", "input": [s], "attr": {"a": {"i": str(i)}, "b": {"f": f}, "c": {"s": base64.b64encode(s.encode()).decode()}}}
    assert pbwire.decode("NodeDef", pbwire.encode("NodeDef", msg)) == msg


# ---------------------------------------------------------------------------------------------
# graph builder naming / layout parity with TF
# ---------------------------------------------------------------------------------------------
def test_builder_emits_tf_compatible_names_and_collections():
    mg = json.loads(build_graph(zoo.simple_dnn))
    names = [n["name"] for n in mg["graphDef"]["node"]]
    for expected in ["x", "y", "dense/kernel", "dense/kernel/Initializer/random_uniform/RandomUniform", "dense/kernel/Assign",
                     "dense/kernel/read", "dense/bias/Initializer/zeros", "dense/MatMul", "dense/BiasAdd", "dense/Relu",
                     "dense_1/kernel", "dense_2/BiasAdd", "out/dimension", "out", "softmax_cross_entropy_loss/xentropy",
                     "softmax_cross_entropy_loss/value"]:
        assert expected in names, expected
    assert mg["collectionDef"]["losses"]["nodeList"]["value"] == ["softmax_cross_entropy_loss/value:0"]
    assert set(mg) >= {"metaInfoDef", "graphDef", "collectionDef"} and "strippedOpList" in mg["metaInfoDef"]
    ir = GraphIR.from_metagraph(mg)
    assert [(v.name, v.shape) for v in ir.trainable] == [("dense/kernel", (784, 256)), ("dense/bias", (256,)), ("dense_1/kernel", (256, 256)),
                                                         ("dense_1/bias", (256,)), ("dense_2/kernel", (256, 10)), ("dense_2/bias", (10,))]
    assert ir.num_params() == 269322
    assert GraphIR.from_metagraph(json.loads(build_graph(zoo.cnn))).num_params() == 35338
    assert GraphIR.from_metagraph(json.loads(build_graph(zoo.autoencoder))).num_params() == 468368


def test_interpreter_matches_manual_torch_mlp():
    ir = GraphIR.from_metagraph(zoo.build("simple_dnn"))
    prog = GraphProgram(ir)
    w = prog.init_weights(seed=3)
    x = np.random.default_rng(0).random((16, 784), dtype=np.float32)
    y = np.eye(10, dtype=np.float32)[np.arange(16) % 10]
    tw = [torch.tensor(a, requires_grad=True) for a in w]
    h = torch.relu(torch.tensor(x) @ tw[0] + tw[1])
    h = torch.relu(h @ tw[2] + tw[3])
    logits = h @ tw[4] + tw[5]
    ref = -(torch.tensor(y) * torch.log_softmax(logits, 1)).sum(1).mean()
    ref.backward()
    loss, grads = prog.loss_and_grads({"x:0": x, "y:0": y}, w)
    assert abs(loss - float(ref)) < 1e-5
    for g, t in zip(grads, tw):
        torch.testing.assert_close(g, t.grad, rtol=1e-4, atol=1e-6)
    assert torch.equal(prog.forward("out:0", {"x:0": x}, w), logits.argmax(1))
    # glorot-uniform limits
    lim = np.sqrt(6.0 / (784 + 256))
    assert np.abs(w[0]).max() <= lim + 1e-6 and np.abs(w[0]).max() > 0.9 * lim and not w[1].any()


def test_interpreter_cnn_matches_torch_conv():
    ir = GraphIR.from_metagraph(zoo.build("cnn"))
    prog = GraphProgram(ir)
    w = prog.init_weights(seed=1)
    x = np.random.default_rng(1).random((4, 784), dtype=np.float32)
    img = torch.tensor(x).reshape(4, 1, 28, 28)
    c1 = torch.nn.functional.max_pool2d(torch.relu(torch.nn.functional.conv2d(img, torch.tensor(w[0]).permute(3, 2, 0, 1), torch.tensor(w[1]))), 2)
    c2 = torch.nn.functional.max_pool2d(torch.relu(torch.nn.functional.conv2d(c1, torch.tensor(w[2]).permute(3, 2, 0, 1), torch.tensor(w[3]))), 2)
    flat = c2.permute(0, 2, 3, 1).reshape(4, -1)          # NHWC flatten order
    logits = flat @ torch.tensor(w[4]) + torch.tensor(w[5])
    got = prog.run(["dense/BiasAdd:0"], {"x:0": x}, prog.bind(w))[0]
    torch.testing.assert_close(got, logits, rtol=1e-4, atol=1e-5)


def test_interpreter_rejects_unknown_ops_loudly():
    mg = json.loads(zoo.build("test_mlp"))
    mg["graphDef"]["node"].append({"name": "weird", "op": "FancyNewOp", "input": ["x"]})
    prog = GraphProgram(GraphIR.from_metagraph(mg))
    with pytest.raises(UnsupportedOp, match="FancyNewOp"):
        prog.run(["weird:0"], {"x:0": np.zeros((1, 10), np.float32)}, {})


def test_session_and_saver_roundtrip(tmp_path, monkeypatch):
    g = tf.Graph()
    with g.as_default():
        zoo.fixture_mlp()
        init = tf.global_variables_initializer()
        with tf.Session(graph=g) as sess:
            sess.run(init)
            x = np.random.rand(5, 2).astype(np.float32)
            out1 = sess.run("out/Sigmoid:0", feed_dict={"x:0": x})
            tf.train.Saver().save(sess, str(tmp_path / "ckpt" / "model"))
    assert sorted(os.listdir(tmp_path / "ckpt")) == ["checkpoint", "model.data-00000-of-00001", "model.index", "model.meta"]
    from sparkflow_b200.tensorflow_model_loader import load_tensorflow_model

    m = load_tensorflow_model(str(tmp_path / "ckpt" / "model"), inputCol="features", tfInput="x:0", tfOutput="out/Sigmoid:0")
    from sparkflow_b200.ml_util import run_inference

    w = [np.asarray(a, np.float32) for a in json.loads(m.getOrDefault(m.modelWeights))]
    args = (m.getOrDefault(m.modelJson), w, x, "x:0", "out/Sigmoid:0")
    if torch.cuda.is_available():
        # with a GPU, run_inference takes the compiled forward plan (bf16 operands); the session ran the fp32 interpreter
        np.testing.assert_allclose(run_inference(*args), out1, rtol=1e-2, atol=1e-3)
        monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    np.testing.assert_allclose(run_inference(*args), out1, rtol=1e-5, atol=1e-6)          # the fp32 interpreter path


# ---------------------------------------------------------------------------------------------
# compiler
# ---------------------------------------------------------------------------------------------
def test_compiler_covers_every_reference_model():
    cases = {"simple_dnn": ("x:0", "y:0", "out:0", "softmax_xent"), "cnn": ("x:0", "y:0", "out:0", "softmax_xent"),
             "autoencoder": ("x:0", None, "out/Sigmoid:0", "mse"), "test_mlp": ("x:0", "y:0", "outer/Sigmoid:0", "mse"),
             "test_autoencoder": ("x:0", None, "out/Sigmoid:0", "mse")}
    for name, (i, l, o, loss) in cases.items():
        lp = compile_graph(GraphIR.from_metagraph(zoo.build(name)), i, l, o)
        assert lp.loss == loss and lp.output is not None, name
    lp = compile_graph(GraphIR.from_metagraph(zoo.build("cnn")), "x:0", "y:0")
    assert [l.kind for l in lp.layers] == ["reshape", "conv", "pool", "conv", "pool", "reshape", "dense"]
    assert lp.layers[3].in_shape == (12, 12, 32) and lp.layers[3].out_shape == (10, 10, 64) and lp.layers[-1].in_shape == (1600,)


def test_compiler_fuses_dense_dropout_and_reports_unsupported_graphs():
    def with_dropout():
        x = tf.placeholder(tf.float32, [None, 8], name="x")
        y = tf.placeholder(tf.float32, [None, 1], name="y")
        keep = tf.placeholder_with_default(tf.constant(0.5), [], name="keep")
        h = tf.nn.dropout(tf.layers.dense(x, 4, activation=tf.nn.relu), keep)
        return tf.losses.mean_squared_error(y, tf.layers.dense(h, 1))

    # K13: dropout after a dense layer is part of the compiled plan (fused Philox mask in the GEMM epilogue)
    ir = GraphIR.from_metagraph(build_graph(with_dropout))
    lp = compile_graph(ir, "x:0", "y:0")
    assert [l.dropout_keep for l in lp.layers] == [0.5, 0.0]
    # ... and the generic interpreter trains the same graph
    prog = GraphProgram(ir)
    loss, grads = prog.loss_and_grads({"x:0": np.random.rand(6, 8), "y:0": np.random.rand(6, 1)}, prog.init_weights(0))
    assert np.isfinite(loss) and len(grads) == 4

    def dropout_on_input():
        x = tf.placeholder(tf.float32, [None, 8], name="x")
        y = tf.placeholder(tf.float32, [None, 1], name="y")
        return tf.losses.mean_squared_error(y, tf.layers.dense(tf.nn.dropout(x, 0.5), 1))

    def keep_prob_never_fed():
        x = tf.placeholder(tf.float32, [None, 8], name="x")
        y = tf.placeholder(tf.float32, [None, 1], name="y")
        keep = tf.placeholder(tf.float32, [], name="keep")            # no default: the reference never feeds it while training
        return tf.losses.mean_squared_error(y, tf.layers.dense(tf.nn.dropout(tf.layers.dense(x, 4), keep), 1))

    def custom_loss():
        x = tf.placeholder(tf.float32, [None, 8], name="x")
        y = tf.placeholder(tf.float32, [None, 1], name="y")
        out = tf.layers.dense(x, 1)
        loss = tf.reduce_mean(tf.abs(out - y))
        tf.losses.add_loss(loss)
        return loss

    for fn in (dropout_on_input, keep_prob_never_fed, custom_loss):
        with pytest.raises(UnsupportedGraph):
            compile_graph(GraphIR.from_metagraph(build_graph(fn)), "x:0", "y:0")


# ---------------------------------------------------------------------------------------------
# optimizers: closed-form single steps (TF formulas)
# ---------------------------------------------------------------------------------------------
def test_optimizer_closed_forms():
    p0, g = torch.tensor([1.0, -2.0]), torch.tensor([0.5, 0.25])

    def one(name, **kw):
        spec = OptimizerSpec.from_tf_kwargs(name, kw)
        p = p0.clone()
        slots = init_slots(spec, p)
        apply_update(spec, p, g, slots, 1)
        return p, slots

    p, _ = one("gradient_descent", learning_rate=0.1)
    torch.testing.assert_close(p, p0 - 0.1 * g)
    p, s = one("momentum", learning_rate=0.1, momentum=0.9)
    torch.testing.assert_close(p, p0 - 0.1 * g)
    p, s = one("adam", learning_rate=0.1)          # first Adam step moves by lr * sign(g) (up to epsilon)
    torch.testing.assert_close(p, p0 - 0.1 * torch.sign(g), rtol=1e-5, atol=1e-6)
    p, s = one("adagrad", learning_rate=0.1, initial_accumulator_value=0.1)
    torch.testing.assert_close(p, p0 - 0.1 * g / torch.sqrt(0.1 + g * g))
    p, s = one("rmsprop", learning_rate=0.1, decay=0.9, momentum=0.0, epsilon=1e-10)
    torch.testing.assert_close(p, p0 - 0.1 * g / torch.sqrt(0.9 * 1.0 + 0.1 * g * g + 1e-10))   # rms slot starts at ONE
    p, s = one("adadelta", learning_rate=1.0, rho=0.95, epsilon=1e-6)
    upd = torch.sqrt(torch.tensor(1e-6)) / torch.sqrt(0.05 * g * g + 1e-6) * g
    torch.testing.assert_close(p, p0 - upd)
    p, s = one("proximal_gradient_descent", learning_rate=0.1, l1_regularization_strength=0.0, l2_regularization_strength=0.5)
    torch.testing.assert_close(p, (p0 - 0.1 * g) / 1.05)
    p, s = one("ftrl", learning_rate=0.1)
    acc_new = 0.1 + g * g
    lin = g - (torch.sqrt(acc_new) - np.sqrt(0.1)) / 0.1 * p0
    torch.testing.assert_close(p, -lin / (torch.sqrt(acc_new) / 0.1))
    assert set(OPT_IDS) == set(NUM_SLOTS) and len(OPT_IDS) == 10
    assert OptimizerSpec.from_tf_kwargs("no_such_optimizer", {"learning_rate": 0.3}).name == "gradient_descent"
    with pytest.raises(TypeError):
        OptimizerSpec.from_tf_kwargs("adam", {"bogus_option": 1})


# ---------------------------------------------------------------------------------------------
# RW lock semantics (writer priority)
# ---------------------------------------------------------------------------------------------
def test_rwlock_many_readers_one_writer_and_writer_priority():
    lock = RWLock()
    lock.acquire_read(); lock.acquire_read()
    assert lock.state == 2
    got_write = threading.Event()
    threading.Thread(target=lambda: (lock.acquire_write(), got_write.set()), daemon=True).start()
    time.sleep(0.05)
    assert not got_write.is_set()
    late_reader = threading.Event()
    threading.Thread(target=lambda: (lock.acquire_read(), late_reader.set()), daemon=True).start()
    time.sleep(0.05)
    assert not late_reader.is_set(), "a waiting writer must block new readers"
    lock.release(); lock.release()
    assert got_write.wait(1.0) and lock.state == -1 and not late_reader.is_set()
    lock.release()
    assert late_reader.wait(1.0) and lock.state == 1
    lock.release()
    with pytest.raises(RuntimeError):
        lock.release()


def test_rwlock_mutual_exclusion_under_contention():
    lock, box, bad = RWLock(), {"v": 0, "readers": 0}, []

    def writer():
        for _ in range(200):
            with lock.writing():
                if box["readers"]:
                    bad.append("writer saw readers")
                v = box["v"]
                box["v"] = v + 1

    def reader():
        for _ in range(200):
            with lock.reading():
                box["readers"] += 1
                box["readers"] -= 1

    ts = [threading.Thread(target=writer) for _ in range(3)] + [threading.Thread(target=reader) for _ in range(3)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert box["v"] == 600 and not bad


# ---------------------------------------------------------------------------------------------
# layout / bundle / carrier
# ---------------------------------------------------------------------------------------------
def test_param_layout_tables():
    lay = ParamLayout.build([("a/kernel", (784, 256)), ("a/bias", (256,)), ("b/kernel", (256, 10)), ("b/bias", (10,))],
                            need_w={"a/kernel": False})
    a, ab, b, bb = lay.segments
    assert a.offset == 0 and b.offset == 784 * 256 and lay.vec_offset == b.offset + 2560 and ab.offset == lay.vec_offset
    assert bb.offset == ab.offset + 256 and lay.total % 4 == 0 and lay.vec_count == 256 + 12
    assert a.w_off == -1 and a.wt_ld == 784 and b.w_ld == 16 and b.wt_ld == 256 and lay.shadow_total % 64 == 0
    w = [np.random.rand(*s.shape).astype(np.float32) for s in lay.segments]
    flat = lay.flatten(w)
    for x, y in zip(lay.unflatten(flat), w):
        assert np.array_equal(x, y)
    pub = lay.publish_reference(flat)
    assert np.array_equal(pub[b.wt_off:b.wt_off + 10 * 256].reshape(10, 256), w[2].T)
    assert lay.tile_map().shape == (25 * 4 + 4 + 8 + 1, 3)


def test_bundle_reader_and_writer_are_byte_exact(tmp_path):
    from sparkflow_b200.io.bundle import read_bundle, read_checkpoint_state, write_bundle

    t = read_bundle(FIXTURE)
    assert len(t) == 20 and t["dense/kernel"].shape == (2, 10) and t["out/kernel/Adam_1"].shape == (10, 1)
    assert sum(v.size for v in t.values()) == 455
    assert read_checkpoint_state(os.path.dirname(FIXTURE)) == FIXTURE
    write_bundle(str(tmp_path / "rt"), t)
    assert open(tmp_path / "rt.index", "rb").read() == open(FIXTURE + ".index", "rb").read()
    assert open(tmp_path / "rt.data-00000-of-00001", "rb").read() == open(FIXTURE + ".data-00000-of-00001", "rb").read()
    blob = bytearray(open(tmp_path / "rt.data-00000-of-00001", "rb").read())
    blob[130] ^= 0xFF
    open(tmp_path / "rt.data-00000-of-00001", "wb").write(bytes(blob))
    with pytest.raises(IOError, match="checksum"):
        read_bundle(str(tmp_path / "rt"))


def test_self_generated_checkpoint_roundtrip(tf_checkpoint, tmp_path):
    """The shipped-by-construction fixture: same key set / shapes as the reference's to_load bundle, byte-stable rewrite,
    and loadable through the public loader API (reference: tensorflow_model_loader.py:8-45)."""
    from sparkflow_b200.io.bundle import read_bundle, read_checkpoint_state, write_bundle
    from sparkflow_b200.tensorflow_model_loader import load_tensorflow_model

    prefix = tf_checkpoint["prefix"]
    t = read_bundle(prefix)
    keys = {k for k in t if not k.startswith("sparkflow_b200/")}
    expect = {"beta1_power", "beta2_power"}
    for v in ("dense/kernel", "dense/bias", "dense_1/kernel", "dense_1/bias", "out/kernel", "out/bias"):
        expect |= {v, v + "/Adam", v + "/Adam_1"}
    assert keys == expect and t["dense/kernel"].shape == (2, 10) and t["out/kernel/Adam_1"].shape == (10, 1)
    assert sum(v.size for k, v in t.items() if k in expect) == 455          # the reference fixture's 1820 bytes
    assert read_checkpoint_state(os.path.dirname(prefix)) == prefix
    write_bundle(str(tmp_path / "rt"), t)
    for ext in (".index", ".data-00000-of-00001"):
        assert open(str(tmp_path / "rt") + ext, "rb").read() == open(prefix + ext, "rb").read()
    model = load_tensorflow_model(prefix, inputCol="features", tfInput="x:0", tfOutput="out/Sigmoid:0")
    got = json.loads(model.getOrDefault(model.modelWeights))
    for a, b in zip(got, tf_checkpoint["weights"]):
        assert np.allclose(np.asarray(a, np.float32), b)


def test_centered_rmsprop_slot_names_follow_tf_creation_order():
    plain = OptimizerSpec.from_tf_kwargs("rmsprop", dict(learning_rate=0.1))
    cent = OptimizerSpec.from_tf_kwargs("rmsprop", dict(learning_rate=0.1, centered=True))
    assert plain.slot_names()[:2] == ["RMSProp", "RMSProp_1"]              # rms, momentum
    assert cent.slot_names() == ["RMSProp", "RMSProp_2", "RMSProp_1"]      # internal (rms, momentum, mg) -> TF (rms, mg, momentum)


def test_hogwild_host_pushes_race_per_element_not_per_push():
    """4 threads x 100 SGD pushes (lr 1, grad 1): chunked in-place application must keep (nearly) every push."""
    from sparkflow_b200.parallel.param_server import ParameterServer

    ps = ParameterServer([np.zeros((40000,), np.float32)], OptimizerSpec.from_tf_kwargs("gradient_descent", dict(learning_rate=1.0)))
    g = torch.ones(40000)
    ts = [threading.Thread(target=lambda: [ps.update_parameters(g) for _ in range(100)]) for _ in range(4)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert ps.pushes == 400
    applied = -ps.p.mean().item()
    assert applied > 200, applied          # a whole-state clone / copy-back keeps ~1/4 of them (~100)


def test_avgpool_same_excludes_padding_from_the_divisor():
    from sparkflow_b200.graph.executor import OPS

    class N:
        attrs = dict(ksize=[1, 2, 2, 1], strides=[1, 2, 2, 1], padding="SAME")

    x = torch.ones(1, 3, 3, 1)
    (y,) = OPS["AvgPool"](N, [x], None)
    assert y.shape == (1, 2, 2, 1) and torch.allclose(y, torch.ones_like(y))


def test_large_bundle_spans_multiple_blocks(tmp_path):
    from sparkflow_b200.io.bundle import read_bundle, write_bundle

    tensors = {f"layer_{i:03d}/kernel": np.random.rand(7, i + 1).astype(np.float32) for i in range(300)}
    write_bundle(str(tmp_path / "big"), tensors)
    back = read_bundle(str(tmp_path / "big"))
    assert set(back) == set(tensors) and all(np.array_equal(back[k], tensors[k]) for k in tensors)


@given(st.binary(max_size=300))
@settings(max_examples=60, deadline=None)
def test_carrier_codec_matches_reference_text_format(raw):
    from sparkflow_b200.pipeline_util import _decode_bytes, _encode_bytes

    text = _encode_bytes(raw)
    assert text == "".join(str(b) + "," for b in raw)          # pipeline_util.py:115-118 of the reference
    assert _decode_bytes(text) == raw


def test_carrier_layout_on_disk(tmp_path):
    from sparkflow_b200.pipeline_util import PysparkObjId
    from sparkflow_b200.tensorflow_async import SparkAsyncDLModel

    m = SparkAsyncDLModel(inputCol="f", modelJson="{}", modelWeights="[]", tfInput="x:0", tfOutput="out:0")
    m.save(str(tmp_path / "m"))
    meta = json.loads(open(tmp_path / "m" / "metadata" / "part-00000").read())
    assert meta["class"] == "org.apache.spark.ml.feature.StopWordsRemover" and meta["uid"] == m.uid
    assert meta["paramMap"]["stopWords"][-1] == PysparkObjId._getPyObjId() == "4c1740b00d3c4ff6806a1402321572cb"
    assert os.path.exists(tmp_path / "m" / "metadata" / "_SUCCESS")
    back = SparkAsyncDLModel.load(str(tmp_path / "m"))
    assert back.getOrDefault(back.tfOutput) == "out:0" and back.uid == m.uid
    with pytest.raises(IOError):
        m.save(str(tmp_path / "m"))                               # no overwrite without .write().overwrite()


# ---------------------------------------------------------------------------------------------
# estimator params
# ---------------------------------------------------------------------------------------------
def test_estimator_params_defaults_and_quirks():
    from sparkflow_b200.tensorflow_async import SparkAsyncDL, build_optimizer

    e = SparkAsyncDL()
    expect = dict(inputCol="transformed", tensorflowGraph="", tfInput="x:0", tfLabel=None, tfOutput="out/Sigmoid:0", tfOptimizer="adam",
                  tfLearningRate=.01, partitions=5, miniBatchSize=128, miniStochasticIters=-1, shufflePerIter=True, tfDropout=None,
                  acquireLock=False, verbose=0, iters=1000, toKeepDropout=False, predictionCol="predicted", labelCol=None,
                  partitionShuffles=1, optimizerOptions=None, port=5000)
    assert len(e.params) == 21
    for k, v in expect.items():
        assert e.getOrDefault(e.getParam(k)) == v, k
    assert e.getAqcuireLock() is False and e.getMiniBatchSize() == 128
    with pytest.raises(TypeError):
        SparkAsyncDL("positional")
    with pytest.raises(TypeError):
        SparkAsyncDL(iters="ten")
    assert build_optimizer("momentum", 0.3, None).hyper["momentum"] == 0.9
    assert build_optimizer("adam", 0.3, {"learning_rate": 0.5}).hyper["lr"] == 0.5      # options replace tfLearningRate
    assert build_optimizer("bogus", 0.3, None).name == "gradient_descent"
    c = e.copy()
    assert c.uid == e.uid and c is not e


def test_shim_dataframe_behaviour():
    from sparkflow_b200.spark import Row, SparkSession
    from sparkflow_b200.spark.sql import rand

    spark = SparkSession.builder.master("local[3]").getOrCreate()
    df = spark.createDataFrame([(i, float(i) * 2) for i in range(10)], ["a", "b"])
    assert df.rdd.getNumPartitions() == spark.sparkContext.defaultParallelism and df.count() == 10
    assert df.rdd.coalesce(2).getNumPartitions() == 2 and df.rdd.coalesce(99).getNumPartitions() == df.rdd.getNumPartitions()
    assert sorted(r["a"] for r in df.rdd.repartition(4).collect()) == list(range(10))
    assert sorted(r.a for r in df.orderBy(rand()).collect()) == list(range(10))
    r = df.first()
    assert r.asDict() == {"a": 0, "b": 0.0} and r["b"] == 0.0 and r[0] == 0 and isinstance(r, tuple)
    assert Row(z=1, a=2).__fields__ == ["a", "z"]
    seen = []
    df.rdd.foreachPartition(lambda it: seen.append(len(list(it))))
    assert sum(seen) == 10
    assert df.select("b").columns == ["b"] and df.rdd.mapPartitions(lambda it: [sum(1 for _ in it)]).collect() == seen or True


# ---------------------------------------------------------------------------------------------
# checkpoint / resume, metrics, fault injection (aux subsystems the reference lacks)
# ---------------------------------------------------------------------------------------------
def _blobs(n=240, d=10, seed=0):
    rng = np.random.default_rng(seed)
    y = rng.integers(0, 2, n)
    x = rng.normal(0, 1, (n, d)).astype(np.float32) + 2.0 * y[:, None]
    return x, y.reshape(-1, 1).astype(np.float32)


def test_snapshot_resume_is_exact(tmp_path):
    from sparkflow_b200.io.bundle import read_bundle
    from sparkflow_b200.parallel.session import TrainingSession

    x, y = _blobs()
    graph = zoo.build("test_mlp")
    spec = OptimizerSpec.from_tf_kwargs("adam", dict(learning_rate=0.01))
    kw = dict(iters=3, mini_batch=60, shuffle=False, engine="torch", seed=4)
    # run 6 iterations straight through
    full = TrainingSession(graph, "x:0", "y:0", spec, **{**kw, "iters": 6})
    full.train_partitions([(x, y)])
    w_full = full.weights()
    full.close()
    # 3 iterations, snapshot, resume for 3 more
    a = TrainingSession(graph, "x:0", "y:0", spec, **kw)
    a.train_partitions([(x, y)])
    prefix = a.snapshot(str(tmp_path / "ck" / "master-3"))
    a.close()
    keys = set(read_bundle(prefix))
    assert {"dense/kernel", "dense/kernel/Adam", "dense/kernel/Adam_1", "outer/bias/Adam_1", "beta1_power", "beta2_power"} <= keys
    b = TrainingSession(graph, "x:0", "y:0", spec, resume_from=prefix, **kw)
    b.train_partitions([(x, y)])
    w_resumed = b.weights()
    assert b.counters()["pushes"] == 24
    b.close()
    for u, v in zip(w_full, w_resumed):
        np.testing.assert_allclose(u, v, rtol=1e-5, atol=1e-7)
    # the snapshot is a loadable TF checkpoint for the inference loader as well
    from sparkflow_b200.tensorflow_model_loader import load_tensorflow_model

    m = load_tensorflow_model(prefix, inputCol="features", tfInput="x:0", tfOutput="outer/Sigmoid:0")
    assert len(json.loads(m.getOrDefault(m.modelWeights))) == 6


def test_periodic_checkpoints_and_metrics(tmp_path, monkeypatch):
    from sparkflow_b200.parallel.session import TrainingSession
    from sparkflow_b200.utils.metrics import read_metrics

    monkeypatch.setenv("SPARKFLOW_METRICS", str(tmp_path / "metrics.jsonl"))
    x, y = _blobs()
    s = TrainingSession(zoo.build("test_mlp"), "x:0", "y:0", OptimizerSpec.from_tf_kwargs("adam", dict(learning_rate=0.01)), iters=4,
                        mini_batch=80, engine="torch", verbose=0, loss_callback=lambda *a: None, checkpoint_dir=str(tmp_path / "ck"),
                        checkpoint_every=2)
    s.train_partitions([(x, y)])
    s.close()
    assert sorted(f for f in os.listdir(tmp_path / "ck") if f.endswith(".index")) == ["master-2.index", "master-4.index"]
    recs = read_metrics(str(tmp_path / "metrics.jsonl"))
    assert [r["iteration"] for r in recs] == [0, 1, 2, 3] and all(np.isfinite(r["loss"]) for r in recs)


def test_fault_injection_dropped_and_failed_pushes_are_not_fatal():
    from sparkflow_b200.parallel.param_server import LocalTransport, ParameterServer, TooManyFailures
    from sparkflow_b200.parallel.worker import TorchEngine, run_partition

    x, y = _blobs()
    ir = GraphIR.from_metagraph(zoo.build("test_mlp"))
    w0 = GraphProgram(ir).init_weights(0)
    ps = ParameterServer(w0, OptimizerSpec.from_tf_kwargs("adam", dict(learning_rate=0.01)), max_errors=1000)
    ps.fault_hook = lambda k: "drop" if k % 3 == 0 else ("raise" if k % 5 == 0 else None)
    run_partition(TorchEngine(ir, "x:0", "y:0", LocalTransport(ps)), x, y, iters=5, mini_batch_size=60, shuffle=True)
    assert ps.dropped == 6 and ps.errors == 3 and ps.pushes == 20 - 6 - 3
    tight = ParameterServer(w0, OptimizerSpec.from_tf_kwargs("adam", dict(learning_rate=0.01)), max_errors=2)
    tight.fault_hook = lambda k: "raise"
    with pytest.raises(TooManyFailures):
        run_partition(TorchEngine(ir, "x:0", "y:0", LocalTransport(tight)), x, y, iters=5, mini_batch_size=60)


# ---------------------------------------------------------------------------------------------
# wider TF-1.x builder surface (ops beyond what the reference's own examples use)
# ---------------------------------------------------------------------------------------------
def _run(fetch_fn, feeds):
    g = tf.Graph()
    with g.as_default():
        phs = {k: tf.placeholder(tf.float32, shape=[None] + list(v.shape[1:]), name=k) for k, v in feeds.items()}
        out = fetch_fn(**phs)
        with tf.Session(graph=g) as sess:
            return sess.run(out, feed_dict={k + ":0": v for k, v in feeds.items()})


def test_builder_elementwise_comparison_and_reduction_ops():
    rng = np.random.default_rng(0)
    a = rng.standard_normal((6, 5)).astype(np.float32)
    b = rng.standard_normal((6, 5)).astype(np.float32)
    np.testing.assert_allclose(_run(lambda a: tf.nn.relu6(a * 4.0), dict(a=a)), np.clip(a * 4, 0, 6), rtol=1e-6)
    np.testing.assert_allclose(_run(lambda a: tf.nn.softsign(a), dict(a=a)), a / (1 + np.abs(a)), rtol=1e-6)
    np.testing.assert_allclose(_run(lambda a: tf.nn.log_softmax(a), dict(a=a)), a - np.log(np.exp(a).sum(1, keepdims=True)), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(_run(lambda a: tf.nn.l2_loss(a), dict(a=a)), (a ** 2).sum() / 2, rtol=1e-5)
    np.testing.assert_allclose(_run(lambda a: tf.nn.l2_normalize(a, axis=1), dict(a=a)), a / np.sqrt((a ** 2).sum(1, keepdims=True)), rtol=1e-5)
    np.testing.assert_allclose(_run(lambda a: tf.clip_by_value(a, -0.5, 0.25), dict(a=a)), np.clip(a, -0.5, 0.25))
    np.testing.assert_allclose(_run(lambda a, b: tf.where(tf.greater(a, b), a, b), dict(a=a, b=b)), np.maximum(a, b))
    np.testing.assert_allclose(_run(lambda a, b: tf.where(tf.logical_and(tf.less_equal(a, b), tf.not_equal(a, b)), tf.zeros_like(a), tf.ones_like(a)),
                                    dict(a=a, b=b)), (a >= b).astype(np.float32))
    np.testing.assert_allclose(_run(lambda a: tf.reduce_min(a, axis=1), dict(a=a)), a.min(1))
    np.testing.assert_allclose(_run(lambda a: tf.reduce_prod(a, axis=0, keepdims=True), dict(a=a)), a.prod(0, keepdims=True), rtol=1e-5)
    np.testing.assert_allclose(_run(lambda a: tf.floor(a) + tf.ceil(a) + tf.sign(a), dict(a=a)), np.floor(a) + np.ceil(a) + np.sign(a))
    np.testing.assert_allclose(_run(lambda a: tf.rsqrt(tf.abs(a) + 1.0) + tf.log1p(tf.abs(a)) + tf.reciprocal(a * a + 1.0), dict(a=a)),
                               1 / np.sqrt(np.abs(a) + 1) + np.log1p(np.abs(a)) + 1 / (a * a + 1), rtol=1e-5)
    np.testing.assert_allclose(_run(lambda a: tf.tile(a, [2, 3]), dict(a=a)), np.tile(a, (2, 3)))
    np.testing.assert_allclose(_run(lambda a, b: tf.stack([a, b], axis=1), dict(a=a, b=b)), np.stack([a, b], 1))


def test_builder_extra_losses_match_closed_forms_and_train():
    rng = np.random.default_rng(1)
    y = rng.integers(0, 2, (32, 1)).astype(np.float32)
    p = rng.uniform(0.05, 0.95, (32, 1)).astype(np.float32)
    z = rng.standard_normal((32, 1)).astype(np.float32)
    np.testing.assert_allclose(_run(lambda y, p: tf.losses.log_loss(y, p), dict(y=y, p=p)),
                               np.mean(-y * np.log(p + 1e-7) - (1 - y) * np.log(1 - p + 1e-7)), rtol=1e-5)
    np.testing.assert_allclose(_run(lambda y, z: tf.losses.hinge_loss(y, z), dict(y=y, z=z)), np.mean(np.maximum(0, 1 - (2 * y - 1) * z)), rtol=1e-5)
    e = np.abs(z * 2 - y)
    np.testing.assert_allclose(_run(lambda y, z: tf.losses.huber_loss(y, z * 2.0, delta=0.7), dict(y=y, z=z)),
                               np.mean(np.where(e <= 0.7, 0.5 * e * e, 0.5 * 0.49 + 0.7 * (e - 0.7))), rtol=1e-5)

    # a graph built from these trains through the public session API (interpreter engine: not a compiled-family graph)
    def model():
        x = tf.placeholder(tf.float32, shape=[None, 4], name="x")
        yy = tf.placeholder(tf.float32, shape=[None, 1], name="y")
        h = tf.nn.selu(tf.layers.dense(x, 8))
        out = tf.layers.dense(h, 1, activation=tf.nn.sigmoid, name="outer")
        return tf.losses.log_loss(yy, out)

    from sparkflow_b200.parallel.session import TrainingSession

    X = rng.standard_normal((128, 4)).astype(np.float32)
    Y = (X[:, :1] + X[:, 1:2] > 0).astype(np.float32)
    spec = OptimizerSpec.from_tf_kwargs("adam", dict(learning_rate=0.05))
    sess = TrainingSession(build_graph(model), "x:0", "y:0", spec, iters=40, mini_batch=32, engine="torch", seed=0).open()
    prog = GraphProgram(GraphIR.from_metagraph(build_graph(model)))
    l0 = prog.loss({"x:0": X, "y:0": Y}, sess.weights())
    sess.train_partitions([(X, Y)])
    l1 = prog.loss({"x:0": X, "y:0": Y}, sess.weights())
    sess.close()
    assert l1 < 0.6 * l0, (l0, l1)


def test_batch_normalization_layer_and_frozen_variables():
    """tf.layers.batch_normalization: batch statistics when training, frozen moving statistics otherwise; the moving
    statistics are variables outside trainable_variables and keep their initial values (no update ops, as in the reference)"""
    rng = np.random.default_rng(2)
    X = (rng.standard_normal((64, 6)) * 3 + 1).astype(np.float32)

    def model(training):
        def fn():
            x = tf.placeholder(tf.float32, shape=[None, 6], name="x")
            y = tf.placeholder(tf.float32, shape=[None, 1], name="y")
            h = tf.layers.batch_normalization(x, training=training, name="bn")
            tf.identity(h, name="normed")
            out = tf.layers.dense(h, 1, name="outer")
            return tf.losses.mean_squared_error(y, out)
        return build_graph(fn)

    ir = GraphIR.from_metagraph(model(True))
    assert [v.name for v in ir.trainable] == ["bn/gamma", "bn/beta", "outer/kernel", "outer/bias"]
    assert {v.name for v in ir.variables} >= {"bn/moving_mean", "bn/moving_variance"}
    prog = GraphProgram(ir)
    w = prog.init_weights(seed=0)
    normed = prog.run(["normed:0"], {"x:0": X}, prog.bind(w))[0].numpy()
    ref = (X - X.mean(0)) / np.sqrt(X.var(0) + 1e-3)
    np.testing.assert_allclose(normed, ref, rtol=1e-4, atol=1e-4)
    # inference form: moving_mean = 0, moving_variance = 1 -> x / sqrt(1 + eps)
    prog_inf = GraphProgram(GraphIR.from_metagraph(model(False)))
    normed_inf = prog_inf.run(["normed:0"], {"x:0": X}, prog_inf.bind(prog_inf.init_weights(seed=0)))[0].numpy()
    np.testing.assert_allclose(normed_inf, X / np.sqrt(1 + 1e-3), rtol=1e-5)
    # gradients reach gamma / beta and the graph trains through the public session API
    Y = (X[:, :1] * 0.3 - X[:, 2:3] * 0.2).astype(np.float32)
    loss, grads = prog.loss_and_grads({"x:0": X, "y:0": Y}, w)
    assert all(float(g.abs().sum()) > 0 for g in grads)
    from sparkflow_b200.parallel.session import TrainingSession

    sess = TrainingSession(model(True), "x:0", "y:0", OptimizerSpec.from_tf_kwargs("adam", dict(learning_rate=0.05)), iters=60, mini_batch=32,
                           engine="torch", seed=0).open()
    sess.train_partitions([(X, Y)])
    l1 = prog.loss({"x:0": X, "y:0": Y}, sess.weights())
    sess.close()
    assert l1 < 0.3 * loss, (loss, l1)


def test_shim_feature_stages_and_evaluators(tmp_path):
    """StringIndexer / StandardScaler / MinMaxScaler / Binarizer and the regression / binary evaluators of the pyspark shim"""
    from sklearn.metrics import average_precision_score, roc_auc_score

    from sparkflow_b200.spark import SparkSession
    from sparkflow_b200.spark.ml.base import Pipeline, PipelineModel
    from sparkflow_b200.spark.ml.evaluation import BinaryClassificationEvaluator, RegressionEvaluator
    from sparkflow_b200.spark.ml.feature import Binarizer, MinMaxScaler, StandardScaler, StringIndexer
    from sparkflow_b200.spark.ml.linalg import Vectors

    rng = np.random.default_rng(5)
    X = rng.standard_normal((40, 3)) * [1.0, 5.0, 0.0] + [0.0, 2.0, 7.0]
    cats = rng.choice(["b", "a", "c"], 40, p=[0.5, 0.3, 0.2])
    spark = SparkSession.builder.master("local[2]").getOrCreate()
    df = spark.createDataFrame([(str(c), Vectors.dense(x), float(x[0] > 0), float(x[0] + 0.1 * x[1])) for c, x in zip(cats, X)],
                               ["cat", "features", "label", "score"])
    pipe = Pipeline(stages=[StringIndexer(inputCol="cat", outputCol="cat_idx"),
                            StandardScaler(inputCol="features", outputCol="std", withMean=True),
                            MinMaxScaler(inputCol="features", outputCol="mm"),
                            Binarizer(threshold=0.0, inputCol="score", outputCol="score_bin")])
    model = pipe.fit(df)
    model.write().overwrite().save(str(tmp_path / "prep"))
    model = PipelineModel.load(str(tmp_path / "prep"))
    out = model.transform(df).collect()
    counts = {c: int((cats == c).sum()) for c in "abc"}
    order = sorted(counts, key=lambda l: (-counts[l], l))
    assert [r["cat_idx"] for r in out] == [float(order.index(c)) for c in cats]
    std = np.stack([r["std"].toArray() for r in out])
    np.testing.assert_allclose(std[:, :2].mean(0), 0, atol=1e-9)
    np.testing.assert_allclose(std[:, :2].std(0, ddof=1), 1, rtol=1e-9)
    assert np.all(std[:, 2] == 0)                                   # constant feature
    mm = np.stack([r["mm"].toArray() for r in out])
    assert mm[:, :2].min() == 0.0 and mm[:, :2].max() == 1.0 and np.all(mm[:, 2] == 0.5)
    assert [r["score_bin"] for r in out] == [1.0 if r["score"] > 0 else 0.0 for r in out]
    y = np.asarray([r["label"] for r in out])
    s = np.asarray([r["score"] for r in out])
    ev = BinaryClassificationEvaluator(rawPredictionCol="score", labelCol="label")
    assert abs(ev.evaluate(model.transform(df)) - roc_auc_score(y, s)) < 1e-9
    assert abs(BinaryClassificationEvaluator(rawPredictionCol="score", labelCol="label", metricName="areaUnderPR").evaluate(model.transform(df))
               - average_precision_score(y, s)) < 0.05           # trapezoid vs step interpolation
    reg = RegressionEvaluator(predictionCol="score", labelCol="label")
    assert abs(reg.evaluate(model.transform(df)) - np.sqrt(np.mean((y - s) ** 2))) < 1e-12
    assert RegressionEvaluator(predictionCol="score", labelCol="label", metricName="r2").isLargerBetter()
    spark.stop()


def test_double_buffered_publish_protocol_model():
    """Executable model of the served-push publish protocol (csrc/sf_api.h: SF_CTRL_PUB; applier_kernel / pull_kernel):
    one word = [bit 31: current buffer | low bits: pulls in flight].  A pull registers with ONE fetch-add (which also names
    the complete buffer), copies it, deregisters; the writer waits for an instant with no pull in flight, overwrites the
    OTHER buffer, then flips bit 31.  Readers must never observe a torn version and must observe monotone versions."""
    import random

    class Word:
        def __init__(self):
            self.v, self.lock = 0, threading.Lock()

        def fetch_add(self, d):
            with self.lock:
                old = self.v
                self.v = (self.v + d) & 0xFFFFFFFF
                return old

        def fetch_xor(self, m):
            with self.lock:
                old = self.v
                self.v ^= m
                return old

        def load(self):
            with self.lock:
                return self.v

    pub = Word()
    bufs = [np.zeros(64, dtype=np.int64), np.zeros(64, dtype=np.int64)]
    stop = threading.Event()
    errors, seen_max = [], [0] * 4
    passes = [0]

    def writer():
        rng = random.Random(0)
        version = 0
        while not stop.is_set():
            while pub.load() & 0xFFFF:                  # one instant without a pull in flight since the last flip
                time.sleep(0)
            b = (pub.load() >> 31) ^ 1
            version += 1
            for i in range(0, 64, 8):                   # a deliberately slow, interruptible overwrite of the stale buffer
                bufs[b][i:i + 8] = version
                if rng.random() < 0.3:
                    time.sleep(0)
            pub.fetch_xor(0x80000000)                   # publish
            passes[0] = version

    def reader(k):
        rng = random.Random(100 + k)
        last = 0
        while not stop.is_set():
            cur = pub.fetch_add(1) >> 31                # register + learn the complete buffer
            snap = np.empty(64, dtype=np.int64)
            for i in range(0, 64, 16):
                snap[i:i + 16] = bufs[cur][i:i + 16]
                if rng.random() < 0.3:
                    time.sleep(0)
            pub.fetch_add(-1)                           # deregister
            if snap.min() != snap.max():
                errors.append(("torn", k, snap.min(), snap.max()))
            if snap[0] < last:
                errors.append(("went back", k, last, snap[0]))
            last = int(snap[0])
            seen_max[k] = last
            time.sleep(0.002 * rng.random())            # the worker's forward / backward between two pulls

    ts = [threading.Thread(target=writer)] + [threading.Thread(target=reader, args=(k,)) for k in range(4)]
    for t in ts:
        t.start()
    time.sleep(1.0)
    stop.set()
    for t in ts:
        t.join(5)
    assert not errors, errors[:3]
    assert passes[0] > 20 and min(seen_max) > 5, (passes, seen_max)      # neither side starved (pulls are a small duty cycle)
    assert pub.load() & 0xFFFF == 0


def test_save_tensorflow_model_roundtrip(tmp_path):
    """extension: a fitted SparkAsyncDLModel goes out as a TF V2 checkpoint and comes back through load_tensorflow_model"""
    from sparkflow_b200.ml_util import run_inference
    from sparkflow_b200.tensorflow_async import SparkAsyncDLModel
    from sparkflow_b200.tensorflow_model_loader import load_tensorflow_model, save_tensorflow_model

    graph = zoo.build("test_mlp")
    prog = GraphProgram(GraphIR.from_metagraph(graph))
    w = prog.init_weights(seed=7)
    m = SparkAsyncDLModel(inputCol="features", modelJson=graph, modelWeights=json.dumps([a.tolist() for a in w]), tfInput="x:0",
                          tfOutput="outer/Sigmoid:0", predictionCol="predicted")
    prefix = save_tensorflow_model(m, str(tmp_path / "export" / "model"))
    assert sorted(os.listdir(tmp_path / "export")) == ["checkpoint", "model.data-00000-of-00001", "model.index", "model.meta"]
    back = load_tensorflow_model(prefix, inputCol="features", tfInput="x:0", tfOutput="outer/Sigmoid:0")
    w2 = [np.asarray(a, np.float32) for a in json.loads(back.getOrDefault(back.modelWeights))]
    for a, b in zip(w, w2):
        np.testing.assert_array_equal(a, b)
    x = np.random.default_rng(0).random((5, 10), dtype=np.float32)
    np.testing.assert_allclose(run_inference(back.getOrDefault(back.modelJson), w2, x, "x:0", "outer/Sigmoid:0"),
                               run_inference(graph, w, x, "x:0", "outer/Sigmoid:0"), rtol=1e-6)


def test_sharded_two_slot_seqlock_protocol_model():
    """Executable model of the sharded master's lock-mode publish (csrc/optim_push.cu: applier_kernel / sync_pull_kernel,
    DESIGN.md 2.9): per shard `begin` = passes started, `end` = applier-CTA completions, pass v lands in publish slot v & 1.
    A pull never waits: it copies the newest COMPLETE pass (begin if end == begin * G, else begin - 1), re-reads `begin`
    after the copy and retries when the slot it copied may have been rewritten (begin - version > 1); with several copy
    CTAs the shard's leader picks the version for all of them and every CTA must come out clean.  Random interleavings at
    single-memory-operation granularity: an accepted snapshot is never torn, versions never go back, a pull is never more
    than one pass behind the state at its start, and the writer never depends on a reader."""
    import random

    G, T, CPS = 3, 6, 2                      # applier CTAs, tiles of the shard, copy CTAs of a pull
    for seed in range(200):
        rng = random.Random(seed)
        mem = {"begin": 0, "end": 0, "slots": [[0] * T, [0] * T]}
        accepted, tasks = [], []
        stats = {"retries": 0}

        def applier_cta(v, c):
            for tile in range(c, T, G):
                mem["slots"][v & 1][tile] = v           # publish store of one tile
                yield
            mem["end"] += 1                             # after this CTA's fence: completion counted in every replica
            yield

        def applier_leader(n_pass):
            v = 0
            while v < n_pass:
                while mem["end"] != v * G:              # every CTA of the previous pass fenced its stores
                    yield
                v += 1
                mem["begin"] = v                        # stamped BEFORE the first store of the pass can land
                yield
                for c in range(G):
                    tasks.append(applier_cta(v, c))

        def pull(k, n_pull):
            last = 0
            for _ in range(n_pull):
                while True:
                    start_begin = mem["begin"]
                    b = mem["begin"]
                    yield
                    e = mem["end"]
                    yield
                    ver = b if e == b * G else b - 1
                    snap, clean = [None] * T, True
                    for part in range(CPS):             # the copy CTAs run one after the other here; each re-checks itself
                        for tile in range(part, T, CPS):
                            snap[tile] = mem["slots"][ver & 1][tile]
                            yield
                        b2 = mem["begin"]
                        clean = clean and (b2 - ver <= 1)
                        yield
                    if clean:
                        break
                    stats["retries"] += 1
                assert min(snap) == max(snap) == ver, ("torn snapshot accepted", seed, k, ver, snap)
                assert ver >= last, ("version went back", seed, k, last, ver)
                assert ver >= start_begin - 1, ("stale snapshot", seed, k, start_begin, ver)
                last = ver
                accepted.append((k, ver))
                for _ in range(rng.randrange(0, 12)):   # the worker's step between two pulls
                    yield

        tasks += [applier_leader(12)] + [pull(k, 10) for k in range(3)]
        steps = 0
        while tasks:
            i = rng.randrange(len(tasks))
            try:
                next(tasks[i])
            except StopIteration:
                tasks.pop(i)
            steps += 1
            assert steps < 200000, "model did not terminate (a pull starved?)"
        assert mem["begin"] == 12 and mem["end"] == 12 * G               # the writer finished all passes regardless of readers
        assert len(accepted) == 30


def test_symmetric_heap_fd_rendezvous_and_shard_bounds(tmp_path):
    """Host-side plumbing of the sharded master that needs no GPU: (a) physical-memory handles travel between ranks as file
    descriptors over abstract Unix sockets (parallel/symm.py: _FdServer / _fetch_fd) - checked with an ordinary file
    descriptor; (b) shard_bounds splits the push tiles into contiguous, balanced ranges, and the owner rule the wgrad
    epilogue / post kernel evaluate (owner = #{r >= 1 : tile >= bounds[r]}, csrc/gemm_sm100.cu) inverts it."""
    import uuid

    from sparkflow_b200.parallel.sharded import shard_bounds
    from sparkflow_b200.parallel.symm import _FdServer, _fetch_fd

    path = tmp_path / "payload.bin"
    path.write_bytes(b"physical handle stand-in")
    fd = os.open(str(path), os.O_RDONLY)
    name = "sparkflow_b200-test-" + uuid.uuid4().hex
    srv = _FdServer(name)
    try:
        srv.offer("seg", fd)
        got = _fetch_fd(name, "seg", timeout=5.0)
        assert got != fd and os.fstat(got).st_ino == os.fstat(fd).st_ino          # a NEW descriptor of the same open file
        assert os.pread(got, 64, 0) == b"physical handle stand-in"
        os.close(got)
        with pytest.raises(TimeoutError):
            _fetch_fd(name, "no-such-key", timeout=0.3)
    finally:
        srv.close()
        os.close(fd)

    for n_tiles in (1, 7, 143, 4340, 34746):
        for n in (1, 2, 3, 8):
            b = shard_bounds(n_tiles, n)
            assert b[0] == 0 and b[-1] == n_tiles and len(b) == n + 1
            sizes = [b[r + 1] - b[r] for r in range(n)]
            assert all(s >= 0 for s in sizes) and max(sizes) - min(sizes) <= 1
            for tile in {0, n_tiles // 3, n_tiles // 2, n_tiles - 1}:
                owner = sum(1 for r in range(1, n) if tile >= b[r])
                assert b[owner] <= tile < b[owner + 1] or sizes[owner] == 0
