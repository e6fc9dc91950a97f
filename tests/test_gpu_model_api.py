"""The user-facing model API on the GPU, for every model: build it from SparseFeat / DenseFeat / VarLenSparseFeat
columns (sum, mean and max pooling) with dropout on, compile, fit with a validation split and the EarlyStopping and
ModelCheckpoint callbacks, then save and reload the weights and the pickled module; the reloaded module must predict
what the trained one predicts."""
import numpy as np
import pytest
import torch

from deepctr_torch_b200 import models
from deepctr_torch_b200.callbacks import EarlyStopping, ModelCheckpoint
from deepctr_torch_b200.inputs import DenseFeat, SparseFeat, VarLenSparseFeat

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N = 64

# (test id, model class, constructor arguments, number of sparse / dense columns, linear columns too)
CASES = [
    ("DeepFM", "DeepFM", dict(dnn_hidden_units=(32,), dnn_dropout=0.5), 3, 3, True),
    ("DeepFM-no-linear", "DeepFM", dict(dnn_hidden_units=(32,), dnn_dropout=0.5), 3, 3, False),
    ("xDeepFM", "xDeepFM", dict(dnn_hidden_units=(8,), cin_layer_size=(8,), cin_split_half=False,
                                cin_activation="relu", dnn_dropout=0.5), 2, 2, True),
    ("FiBiNET", "FiBiNET", dict(bilinear_type="each", dnn_hidden_units=[8, 8], dnn_dropout=0.5), 3, 3, True),
    ("DCN", "DCN", dict(cross_num=2, cross_parameterization="vector", dnn_hidden_units=(32,), dnn_dropout=0.5),
     2, 2, True),
    ("DCN-matrix", "DCN", dict(cross_num=1, cross_parameterization="matrix", dnn_hidden_units=(32,),
                               dnn_dropout=0.5), 2, 2, True),
    ("DCNMix", "DCNMix", dict(cross_num=1, dnn_hidden_units=(32,), dnn_dropout=0.5), 2, 2, True),
    ("WDL", "WDL", dict(dnn_activation="prelu", dnn_hidden_units=[32, 32], dnn_dropout=0.5), 2, 2, True),
    ("NFM", "NFM", dict(dnn_hidden_units=[32, 32], dnn_dropout=0.5), 2, 2, True),
    ("AFM", "AFM", dict(use_attention=True, afm_dropout=0.5), 3, 0, True),
    ("IFM", "IFM", dict(dnn_hidden_units=(32,), dnn_dropout=0.5), 3, 3, True),
    ("DIFM", "DIFM", dict(att_head_num=2, dnn_hidden_units=(4, 4), dnn_dropout=0.5), 2, 2, True),
    # branches switched off and column kinds left out
    ("DeepFM-no-fm", "DeepFM", dict(use_fm=False, dnn_hidden_units=(32,), dnn_dropout=0.5), 3, 3, True),
    ("DeepFM-no-dnn", "DeepFM", dict(dnn_hidden_units=(), dnn_dropout=0.5), 1, 1, True),
    ("DeepFM-no-sparse", "DeepFM", dict(dnn_hidden_units=(32,), dnn_dropout=0.5), 0, 3, True),
    ("DeepFM-no-dense", "DeepFM", dict(dnn_hidden_units=(32,), dnn_dropout=0.5), 3, 0, True),
    ("xDeepFM-no-cin", "xDeepFM", dict(dnn_hidden_units=(8,), cin_layer_size=(), dnn_dropout=0.5), 1, 1, True),
    ("xDeepFM-no-dnn", "xDeepFM", dict(dnn_hidden_units=(), cin_layer_size=(8,), cin_activation="linear",
                                       dnn_dropout=0.5), 2, 2, True),
    ("xDeepFM-linear-only", "xDeepFM", dict(dnn_hidden_units=(), cin_layer_size=(), dnn_dropout=0.5), 1, 2, True),
    ("FiBiNET-interaction", "FiBiNET", dict(bilinear_type="interaction", dnn_hidden_units=[8, 8], dnn_dropout=0.5),
     3, 3, True),
    ("FiBiNET-all", "FiBiNET", dict(bilinear_type="all", dnn_hidden_units=[8, 8], dnn_dropout=0.5), 3, 3, True),
    ("DCNMix-no-cross", "DCNMix", dict(cross_num=0, dnn_hidden_units=(32,), dnn_dropout=0.5), 2, 2, True),
    ("WDL-no-sparse", "WDL", dict(dnn_activation="prelu", dnn_hidden_units=[32, 32], dnn_dropout=0.5), 0, 2, True),
]


def _data(n_sparse, n_dense, seed=0):
    """Random inputs in the shape users feed fit(): a dict of numpy columns, sequences as [N, maxlen] id arrays."""
    rng = np.random.RandomState(seed)
    cols, x = [], {}
    for i in range(n_sparse):
        c = SparseFeat("sparse_%d" % i, int(rng.randint(2, 10)), embedding_dim=4)
        cols.append(c)
        x[c.name] = rng.randint(0, c.vocabulary_size, N)
    for i in range(n_dense):
        c = DenseFeat("dense_%d" % i, 1)
        cols.append(c)
        x[c.name] = rng.random_sample(N)
    for combiner in ("sum", "mean", "max"):
        vocab, maxlen = int(rng.randint(2, 10)), int(rng.randint(1, 10))
        c = VarLenSparseFeat(SparseFeat("seq_" + combiner, vocab, embedding_dim=4), maxlen=maxlen, combiner=combiner)
        cols.append(c)
        x[c.name] = rng.randint(0, vocab, (N, maxlen))
    return x, rng.randint(0, 2, N), cols


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_model_fit_callbacks_save_load(case, tmp_path):
    _, cls, kwargs, n_sparse, n_dense, with_linear = case
    x, y, cols = _data(n_sparse, n_dense)
    model = getattr(models, cls)(cols if with_linear else [], cols, device=DEV, **kwargs)
    model.compile("adam", "binary_crossentropy", metrics=["binary_crossentropy", "acc"])
    ckpt = tmp_path / "model.ckpt"
    callbacks = [EarlyStopping(monitor="val_acc", min_delta=0, patience=0, mode="max"),
                 ModelCheckpoint(filepath=str(ckpt), monitor="val_acc", save_best_only=True, save_weights_only=False,
                                 mode="max")]
    # default verbosity: the training-set metrics are computed and logged only when verbose > 0
    hist = model.fit(x, y, batch_size=100, epochs=2, validation_split=0.5, callbacks=callbacks)
    for key in ("loss", "binary_crossentropy", "acc", "val_binary_crossentropy", "val_acc"):
        assert key in hist.history and np.all(np.isfinite(hist.history[key])), key
    assert ckpt.exists()
    pred = model.predict(x, batch_size=32)
    assert pred.shape == (N, 1) and np.all((pred >= 0) & (pred <= 1))

    torch.save(model.state_dict(), tmp_path / "weights.pt")
    model.load_state_dict(torch.load(tmp_path / "weights.pt"))
    assert np.allclose(model.predict(x, batch_size=32), pred, rtol=1e-6, atol=1e-7)
    torch.save(model, tmp_path / "model.pt")
    reloaded = torch.load(tmp_path / "model.pt", weights_only=False)
    assert np.allclose(reloaded.predict(x, batch_size=32), pred, rtol=1e-6, atol=1e-7)
