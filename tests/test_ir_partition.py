"""Host logic: layer-DAG IR, model zoo, dag_util partitioner (CPU only)."""
import numpy as np
import pytest

from defer_b200 import applications, dag_util, keras_like as K
from defer_b200.dispatcher import DEFER
from oracle import keras_ref as R


def test_param_counts_match_keras():
    # published Keras parameter counts pin the three graph definitions
    assert applications.ResNet50(weights=None).count_params() == 25_636_712
    assert applications.ResNet152(weights=None).count_params() == 60_419_944
    assert applications.VGG16(weights=None).count_params() == 138_357_544


def test_tf_keras_auto_names(resnet50):
    adds = applications.residual_add_names(resnet50)
    assert adds == ["add"] + [f"add_{i}" for i in range(1, 16)]
    assert resnet50.get_layer("activation_48").class_name == "Activation"
    assert resnet50.get_layer("max_pooling2d").class_name == "MaxPooling2D"
    assert resnet50.input._keras_history[0].name == "input_1"
    assert resnet50.output._keras_history[0].name == "fc1000"
    # the cut list of test/test.py:18 names existing layers
    for c in applications.RESNET50_TEST_CUTS:
        assert resnet50.get_layer(c).class_name == "Add"
    # one-based (standalone Keras) reading maps add_k to the k-th Add
    assert applications.resolve_cut_names(resnet50, ["add_2"], naming="keras") == ["add_1"]


def test_get_previous_single_and_list(resnet50):
    assert dag_util.get_previous(resnet50, "conv1") == ["conv1_pad"]          # bare layer -> wrapped
    assert dag_util.get_previous(resnet50, "add") == ["bn2a_branch2c", "bn2a_branch1"]
    assert dag_util.get_previous(resnet50, "add_1") == ["bn2b_branch2c", "activation_3"]


def test_construct_model_layer_sets_match_reference_rule():
    resnet50 = applications.ResNet50()     # not the shared fixture: other tests partition that one too
    cuts = applications.RESNET50_TEST_CUTS
    d = DEFER(list(range(8)))
    parts = d._partition(resnet50, cuts)
    assert len(parts) == 8
    sets = R.stage_layer_sets(resnet50.to_json(), cuts)
    for i, (p, s) in enumerate(zip(parts, sets)):
        names = sorted(l.name for l in p.layers if l.class_name != "InputLayer")
        assert names == s
        assert p._input_layers[0].name == f"part{i+1}"               # src/dispatcher.py:40
    # every weighted layer lands in exactly one stage
    all_w = sum(p.count_params() for p in parts)
    assert all_w == resnet50.count_params()
    # memoised traversal: each layer is re-applied once per stage, not 2^(m-1) times
    assert len(resnet50.get_layer("res2a_branch2a").inbound_nodes) == 2


def test_pipeline_composition_equals_whole_model_oracle(x224):
    m = applications.ResNet50()
    ref = R.predict(m.to_json(), m.get_weights(), x224, final_activation=False)
    for cuts in (applications.RESNET50_TEST_CUTS, applications.default_cuts(m, 2), ["conv1", "activation_9", "avg_pool"]):
        m2 = applications.ResNet50()
        parts = DEFER([0] * (len(cuts) + 1))._partition(m2, cuts)
        wire = [(p.to_json(), p.get_weights()) for p in parts]
        y = R.pipeline_predict(wire, x224, final_activation=False)
        assert np.array_equal(y, ref), cuts          # lossless hop => bit-identical on the oracle


def test_non_articulation_cut_is_rejected(resnet50):
    # cutting inside a residual block leaves the shortcut path reaching past `start`
    m = applications.ResNet50()
    with pytest.raises(ValueError):
        dag_util.construct_model(m, "res2b_branch2a", "add_2", part_name="bad")


def test_json_roundtrip_and_weight_order(resnet50, x224):
    js, ws = resnet50.to_json(), resnet50.get_weights()
    m2 = K.model_from_json(js)
    m2.set_weights(ws)
    assert [l.name for l in m2.layers] == [l.name for l in resnet50.layers]
    assert m2.to_json() == js
    for a, b in zip(m2.get_weights(), ws):
        assert np.array_equal(a, b)
    # Keras order: conv kernel then bias; BN gamma, beta, mean, var
    conv1 = resnet50.get_layer("conv1").get_weights()
    assert conv1[0].shape == (7, 7, 3, 64) and conv1[1].shape == (64,)
    assert len(resnet50.get_layer("bn_conv1").get_weights()) == 4


def test_resnet152_and_vgg_cuts():
    m = applications.ResNet152(weights=None)
    cuts = applications.default_cuts(m, 8)
    assert cuts[0] == "conv3_block2_add" and len(cuts) == 7
    parts = DEFER([0] * 8)._partition(m, cuts)
    assert sum(p.count_params() for p in parts) == m.count_params()
    v = applications.VGG16(weights=None)
    parts = DEFER([0] * 4)._partition(v, applications.default_cuts(v, 4))
    assert [p.output.shape[1:] for p in parts] == [(112, 112, 64), (56, 56, 128), (28, 28, 256), (1000,)]


def test_node_state_semantics():
    from defer_b200 import NodeState
    ns = NodeState(chunk_size=512000)
    assert ns.chunk_size == 512000 and ns.next_node == "" and ns.model == "" and ns.weights == ""
    ns.weights = [np.zeros(3)]
    ns.next_node = "cuda:1"
    assert ns.wait_for("weights", timeout=0.1)[0].shape == (3,)
    assert ns.next_node == "cuda:1"
    with pytest.raises(TimeoutError):
        ns.wait_for("model", timeout=0.01)
