"""§8f f4: the HDF5 subset reader/writer (Keras save_weights files, data-for-iter files).  CPU only."""
import os

import numpy as np

from conftest import GOLDEN

def test_weights_round_trip(tmp_path):
    from chinesecheckersagent_b200 import h5lite
    w = {k: np.asarray(v, dtype=np.float32) for k, v in np.load(os.path.join(GOLDEN, "good_model_weights.npz")).items()}
    path = h5lite.write_weights(str(tmp_path / "version0001.h5"), w)
    back = h5lite.read_weights(path)
    assert set(back) == set(w) and all(np.array_equal(back[k], w[k]) for k in w)
    f = h5lite._File(open(path, "rb").read())
    root = f.attributes(f.root_header)
    assert [n.decode() for n in root["layer_names"]] == h5lite.keras_layer_order()
    assert root["keras_version"] == b"2.1.6" and root["backend"] == b"tensorflow"
    ent = f.group_entries(f.root_header)
    assert [n.decode() for n in f.attributes(ent["batch_normalization_7"])["weight_names"]] == [
        "batch_normalization_7/gamma:0", "batch_normalization_7/beta:0", "batch_normalization_7/moving_mean:0",
        "batch_normalization_7/moving_variance:0"]
    assert len(f.attributes(ent["add_3"])["weight_names"]) == 0


def test_train_data_round_trip(tmp_path):
    from chinesecheckersagent_b200 import utils
    rng = np.random.default_rng(0)
    bx = rng.integers(0, 7, (37, 7, 7, 7)).astype(np.float64)
    pi = rng.random((37, 294))
    v = rng.integers(-1, 2, 37)
    path = utils.save_train_data(bx, pi, v, 12, directory=str(tmp_path))
    assert path.endswith("data-for-iter-12.h5")
    b2, p2, v2 = utils.load_train_data(path)
    assert np.array_equal(b2, bx) and np.array_equal(p2, pi) and np.array_equal(v2, v)


def test_written_file_mirrors_a_real_keras_file(tmp_path):
    """same groups, same layer order, same weight_names, same tensors as the file Keras 2.1.6 wrote for the reference
    (good_model.h5).  What the output is compared with comes from that file: its 186 tensors under their own names
    (good_model_weights.npz, read out of it by tests/golden/gen_golden_net.py) and its layout as probed in SURVEY.md
    Appendix B (superblock version 0, 8-byte offsets and lengths, float32 datasets at /<layer>/<layer>/<name>:0,
    249,852 floats, root attributes layer_names / backend / keras_version and no model_config)."""
    from chinesecheckersagent_b200 import h5lite
    real = dict(np.load(os.path.join(GOLDEN, "good_model_weights.npz")))
    assert len(real) == 186 and sum(v.size for v in real.values()) == 249852 and all(v.dtype == np.float32 for v in real.values())
    assert real["conv2d_1/kernel"].shape == (3, 3, 7, 64) and real["conv2d_29/kernel"].shape == (1, 1, 64, 16)
    assert real["policy_head/kernel"].shape == (400, 294) and real["dense_1/kernel"].shape == (25, 32)
    path = h5lite.write_weights(str(tmp_path / "w.h5"), real)
    raw = open(path, "rb").read()
    assert raw[:8] == b"\x89HDF\r\n\x1a\n" and raw[8] == 0 and raw[13] == 8 and raw[14] == 8
    mine = h5lite._File(raw)
    attrs = mine.attributes(mine.root_header)
    assert set(attrs) == {"layer_names", "backend", "keras_version"}
    assert attrs["keras_version"] == b"2.1.6" and attrs["backend"] == b"tensorflow"
    layers = [n.decode() for n in attrs["layer_names"]]
    assert layers == h5lite.keras_layer_order() and {k.split("/")[0] for k in real} <= set(layers)
    ent = mine.group_entries(mine.root_header)
    assert set(ent) == set(layers)
    keras_param_order = ("kernel", "bias", "gamma", "beta", "moving_mean", "moving_variance")
    for name in layers:
        params = sorted((k.split("/")[1] for k in real if k.split("/")[0] == name), key=keras_param_order.index)
        assert [n.decode() for n in mine.attributes(ent[name])["weight_names"]] == ["%s/%s:0" % (name, q) for q in params], name
    tree = h5lite.read_tree(path)
    assert set(tree) == {"/%s/%s/%s:0" % (k.split("/")[0], k.split("/")[0], k.split("/")[1]) for k in real}
    for k, v in real.items():
        layer, param = k.split("/")
        t = tree["/%s/%s/%s:0" % (layer, layer, param)]
        assert t.dtype == np.float32 and np.array_equal(t, v), k


def test_weights_of_a_second_model_in_the_process_load_by_position(tmp_path):
    """Keras numbers auto-named layers per process: a weights file saved from the second ResidualCNN built in a process holds
    conv2d_31..60 / batch_normalization_31..60 / dense_2, and a full-model save keeps everything under /model_weights.  Keras'
    load_weights matches by position, so the reference loads both; read_weights must too."""
    import re

    from chinesecheckersagent_b200 import h5lite
    w = {k: np.asarray(v, dtype=np.float32) for k, v in np.load(os.path.join(GOLDEN, "good_model_weights.npz")).items()}

    def shifted(name):
        m = re.fullmatch(r"(conv2d|batch_normalization)_(\d+)", name)
        if m:
            return "%s_%d" % (m.group(1), int(m.group(2)) + 30)
        return "dense_2" if name == "dense_1" else name
    tree = {}
    for k, v in w.items():
        layer, param = k.split("/")
        tree["model_weights/%s/%s/%s:0" % (shifted(layer), shifted(layer), param)] = v
    path = h5lite.write_tree(str(tmp_path / "second_model.h5"), tree)
    back = h5lite.read_weights(path)
    assert set(back) == set(w) and all(np.array_equal(back[k], w[k]) for k in w)
