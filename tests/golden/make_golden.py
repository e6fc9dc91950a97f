"""Generate golden input/output vectors by running the UNMODIFIED reference on CPU.

Needs a checkout of the reference project:

    CTR_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py

(``--round2`` skips the round-1 fixtures; ``--round2 --only=<case>`` or ``--round2 --only=dice`` writes one file.)

Writes ``tests/golden/<case>.npz`` (+ the model description as a JSON string inside each file).
Each model case records: ``X``, ``y``, every ``state_dict`` tensor (``state/<key>``), the
pre-sigmoid logit captured at the input of ``model.out`` (+ ``out.bias``), ``y_pred``, the
``BCE(sum)`` loss and the gradient of every parameter (``grad/<key>``) — i.e. what the
reference's forward (models/*.py) and ``loss.backward()`` (basemodel.py:254-261) produce.
Layer cases record the reference layer modules (layers/interaction.py, layers/core.py) run on
random inputs.  ``fit_criteo_sample`` records the reference's own ``fit``/``predict`` on
``examples/criteo_sample.txt`` (BASELINE config #1) after LabelEncoder/MinMaxScaler
preprocessing (examples/run_classification_criteo.py:14-66).
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, HERE)

from _ref_loader import load_reference, REFERENCE_ROOT  # noqa: E402
from oracle import ctr_oracle as O  # noqa: E402

ref = load_reference()
from deepctr_torch.inputs import SparseFeat, DenseFeat, VarLenSparseFeat  # noqa: E402
from deepctr_torch import models as RM  # noqa: E402
from deepctr_torch.layers import activation as RA, interaction as RI, core as RC  # noqa: E402


def to_ref_columns(cols):
    out = []
    for c in cols:
        if c["type"] == "sparse":
            out.append(SparseFeat(c["name"], c["vocab"], embedding_dim=c["dim"],
                                  embedding_name=c["embedding_name"]))
        elif c["type"] == "dense":
            out.append(DenseFeat(c["name"], c["dimension"]))
        else:
            sf = SparseFeat(c["name"], c["vocab"], embedding_dim=c["dim"],
                            embedding_name=c["embedding_name"])
            out.append(VarLenSparseFeat(sf, maxlen=c["maxlen"], combiner=c["combiner"],
                                        length_name=c["length_name"]))
    return out


def randomize_zero_params(model, gen, std=0.05):
    """Biases the reference zero-initialises (out.bias, crossnet.bias) get random values so
    the golden vectors exercise them."""
    with torch.no_grad():
        for name, p in model.named_parameters():
            if p.numel() > 0 and float(p.abs().max()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=gen) * std)


def run_model_case(name, cfg, batch, zipf=None, seed=7, eval_mode=False):
    cls = getattr(RM, cfg["model"])
    lin = to_ref_columns(cfg["linear_columns"])
    dnn = to_ref_columns(cfg["dnn_columns"])
    kwargs = dict(cfg["kwargs"])
    for k in ("dnn_hidden_units", "cin_layer_size"):
        if k in kwargs:
            kwargs[k] = tuple(kwargs[k])
    model = cls(lin, dnn, device="cpu", **kwargs)
    gen = torch.Generator().manual_seed(seed)
    randomize_zero_params(model, gen)
    model.train()
    if eval_mode:       # dropout > 0: deterministic only in eval mode
        model.eval()
    X, y = O.synthetic_batch(cfg, batch, seed=seed + 100, zipf_alpha=zipf)
    captured = {}

    def pre_hook(mod, inp):
        captured["prebias"] = inp[0].detach().clone()

    h = model.out.register_forward_pre_hook(pre_hook)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    y_pred = model(X)
    h.remove()
    loss = torch.nn.functional.binary_cross_entropy(y_pred.squeeze(), y, reduction="sum")
    reg = model.get_regularization_loss()
    loss.backward()
    out = {"cfg": json.dumps(cfg), "X": X.numpy(), "y": y.numpy(),
           "logit": (captured["prebias"] + state["out.bias"]).numpy(),
           "y_pred": y_pred.detach().numpy(), "loss": loss.detach().numpy(),
           "reg_loss": reg.detach().numpy()}
    for k, v in state.items():
        out["state/" + k] = v.numpy()
    for k, p in model.named_parameters():
        out["grad/" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print("wrote %-28s B=%d logit range [%.3f, %.3f] loss %.4f" %
          (name, batch, float(out["logit"].min()), float(out["logit"].max()), float(loss.detach())))


def small_columns(n_sparse, dim, n_dense, vocab_lo=5, vocab_hi=60, seed=0, dense2=False):
    rng = np.random.RandomState(seed)
    cols = [O.sparse_col("C%d" % (i + 1), int(rng.randint(vocab_lo, vocab_hi)), dim)
            for i in range(n_sparse)]
    for i in range(n_dense):
        cols.append(O.dense_col("I%d" % (i + 1), 2 if (dense2 and i == 0) else 1))
    return cols


def model_cases():
    std = 0.05
    cases = []
    c5 = small_columns(5, 8, 3, dense2=True)
    cases.append(("deepfm_small", O.make_cfg("DeepFM", c5, c5, dnn_hidden_units=[32, 16],
                                             init_std=std, l2_reg_linear=1e-5, l2_reg_embedding=1e-5), 48))
    # linear part on a different (sub)set of columns, FM off
    cases.append(("deepfm_nofm_sublinear", O.make_cfg("DeepFM", c5[:2] + c5[5:6], c5, use_fm=False,
                                                      dnn_hidden_units=[16], init_std=std), 33))
    cases.append(("deepfm_nodnn", O.make_cfg("DeepFM", c5, c5, dnn_hidden_units=[], init_std=std), 20))
    crit = small_columns(26, 16, 13, vocab_lo=40, vocab_hi=120, seed=3)
    cases.append(("deepfm_criteo_shape", O.make_cfg("DeepFM", crit, crit, dnn_hidden_units=[256, 128],
                                                    init_std=std, l2_reg_linear=0, l2_reg_embedding=0), 64))
    cases.append(("deepfm_criteo_zipf", O.make_cfg("DeepFM", crit, crit, dnn_hidden_units=[64, 32],
                                                   init_std=std, l2_reg_linear=0, l2_reg_embedding=0), 96, 1.05))
    c6 = small_columns(6, 8, 2, seed=5)
    cases.append(("xdeepfm_small", O.make_cfg("xDeepFM", c6, c6, dnn_hidden_units=[32, 32],
                                              cin_layer_size=[16, 8], cin_split_half=True,
                                              cin_activation="relu", init_std=std), 40))
    cases.append(("xdeepfm_nosplit_linear", O.make_cfg("xDeepFM", c6, c6, dnn_hidden_units=[16],
                                                       cin_layer_size=[8, 6, 4], cin_split_half=False,
                                                       cin_activation="linear", init_std=std), 24))
    cases.append(("xdeepfm_nodnn", O.make_cfg("xDeepFM", c6, c6, dnn_hidden_units=[],
                                              cin_layer_size=[8], init_std=std), 16))
    cases.append(("xdeepfm_criteo_shape", O.make_cfg("xDeepFM", crit, crit, dnn_hidden_units=[256, 256],
                                                     cin_layer_size=[128, 128], cin_split_half=True,
                                                     init_std=std, l2_reg_linear=0, l2_reg_embedding=0), 32))
    c8 = small_columns(8, 32, 3, seed=9)
    for bt in ("interaction", "each", "all"):
        cases.append(("fibinet_" + bt, O.make_cfg("FiBiNET", c8, c8, bilinear_type=bt, reduction_ratio=3,
                                                  dnn_hidden_units=[32, 16], init_std=std), 24))
    c26 = small_columns(26, 32, 13, vocab_lo=10, vocab_hi=40, seed=11)
    cases.append(("fibinet_criteo_shape", O.make_cfg("FiBiNET", c26, c26, bilinear_type="all",
                                                     dnn_hidden_units=[16, 16], init_std=std), 8))
    for par in ("vector", "matrix"):
        cases.append(("dcn_" + par, O.make_cfg("DCN", c5, c5, cross_num=3, cross_parameterization=par,
                                               dnn_hidden_units=[32, 16], init_std=std), 40))
    # (DCN with dnn_hidden_units=[] cannot be built in the reference: DNN raises ValueError, core.py:100-101)
    cases.append(("dcn_criteo_shape", O.make_cfg("DCN", crit, crit, cross_num=2, dnn_hidden_units=[128, 128],
                                                 init_std=std, l2_reg_linear=0, l2_reg_embedding=0,
                                                 l2_reg_cross=0), 64))
    cases.append(("dcnmix_small", O.make_cfg("DCNMix", c5, c5, cross_num=2, low_rank=8, num_experts=3,
                                             dnn_hidden_units=[32, 16], init_std=std), 40))
    cases.append(("dcnmix_criteo_shape", O.make_cfg("DCNMix", crit, crit, cross_num=2, low_rank=32,
                                                    num_experts=4, dnn_hidden_units=[32, 32],
                                                    init_std=std), 32))
    # VarLenSparseFeat pooling (SURVEY §8f-1): mask-by-zero and length-column variants
    vl = c5 + [O.varlen_col("V_sum", 30, 8, 5, "sum"), O.varlen_col("V_mean", 30, 8, 4, "mean"),
               O.varlen_col("V_max", 30, 8, 6, "max"),
               O.varlen_col("V_len", 30, 8, 4, "mean", length_name="V_len_n")]
    cases.append(("deepfm_varlen", O.make_cfg("DeepFM", vl, vl, dnn_hidden_units=[32, 16], init_std=std), 40))
    return cases


def extra_cases():
    """Round 2: adjacent models (SURVEY §8 f4) and the branch toggles of the reference's own model tests
    (tests/models/*_test.py, tests/utils.py:18-67): no sparse / no dense / no linear columns, cross_num=0,
    empty CIN, dropout (eval), VarLen features under xDeepFM / FiBiNET / DCN."""
    std = 0.05
    cases = []
    c5 = small_columns(5, 8, 3, dense2=True)
    c6 = small_columns(6, 8, 2, seed=5)
    sparse_only = [c for c in c5 if c["type"] == "sparse"]
    dense_only = [c for c in c5 if c["type"] == "dense"]
    cases.append(("wdl_small", O.make_cfg("WDL", c5, c5, dnn_hidden_units=[32, 16], init_std=std), 40))
    cases.append(("nfm_small", O.make_cfg("NFM", c5, c5, dnn_hidden_units=[32, 16], init_std=std), 40))
    cases.append(("afm_attention", O.make_cfg("AFM", sparse_only, sparse_only, use_attention=True, attention_factor=8,
                                               init_std=std), 40))
    cases.append(("afm_plain", O.make_cfg("AFM", sparse_only, sparse_only, use_attention=False, init_std=std), 24))
    cases.append(("ifm_small", O.make_cfg("IFM", c5, c5, dnn_hidden_units=[32, 16], init_std=std), 40))
    cases.append(("difm_small", O.make_cfg("DIFM", c5, c5, att_head_num=4, att_res=True, dnn_hidden_units=[32, 16],
                                           init_std=std), 40))
    crit = small_columns(26, 16, 13, vocab_lo=40, vocab_hi=120, seed=3)
    cases.append(("nfm_criteo_shape", O.make_cfg("NFM", crit, crit, dnn_hidden_units=[128, 128], init_std=std), 32))
    crit_s = [c for c in crit if c["type"] == "sparse"]
    cases.append(("afm_criteo_shape", O.make_cfg("AFM", crit_s, crit_s, init_std=std), 16))
    cases.append(("difm_criteo_shape", O.make_cfg("DIFM", crit, crit, dnn_hidden_units=[64, 32], init_std=std), 16))
    # branch toggles
    cases.append(("deepfm_nosparse", O.make_cfg("DeepFM", dense_only, dense_only, dnn_hidden_units=[16, 8],
                                                init_std=std), 20))
    cases.append(("deepfm_nodense", O.make_cfg("DeepFM", sparse_only, sparse_only, dnn_hidden_units=[16, 8],
                                               init_std=std), 20))
    cases.append(("deepfm_nolinear", O.make_cfg("DeepFM", [], c5, dnn_hidden_units=[16, 8], init_std=std), 20))
    cases.append(("deepfm_dropout_eval", O.make_cfg("DeepFM", c5, c5, dnn_hidden_units=[32, 32], dnn_dropout=0.5,
                                                    init_std=std), 24, None, 7, True))
    cases.append(("deepfm_prelu", O.make_cfg("DeepFM", c5, c5, dnn_hidden_units=[32, 16], dnn_activation="prelu",
                                             init_std=std), 32))
    cases.append(("dcnmix_cross0", O.make_cfg("DCNMix", c5, c5, cross_num=0, dnn_hidden_units=[16, 8],
                                              init_std=std), 20))
    cases.append(("dcn_cross0", O.make_cfg("DCN", c5, c5, cross_num=0, dnn_hidden_units=[16, 8], init_std=std), 20))
    cases.append(("xdeepfm_nocin", O.make_cfg("xDeepFM", c6, c6, dnn_hidden_units=[16, 8], cin_layer_size=[],
                                              init_std=std), 20))
    cases.append(("xdeepfm_nolinear", O.make_cfg("xDeepFM", [], c6, dnn_hidden_units=[16], cin_layer_size=[8, 4],
                                                 init_std=std), 20))
    vl = c5 + [O.varlen_col("V_sum", 30, 8, 5, "sum"), O.varlen_col("V_mean", 30, 8, 4, "mean"),
               O.varlen_col("V_max", 30, 8, 6, "max"),
               O.varlen_col("V_len", 30, 8, 4, "mean", length_name="V_len_n")]
    cases.append(("xdeepfm_varlen", O.make_cfg("xDeepFM", vl, vl, dnn_hidden_units=[16], cin_layer_size=[8, 4],
                                               init_std=std), 24))
    cases.append(("fibinet_varlen", O.make_cfg("FiBiNET", vl, vl, bilinear_type="each", dnn_hidden_units=[16, 8],
                                               init_std=std), 24))
    cases.append(("dcn_varlen", O.make_cfg("DCN", vl, vl, cross_num=2, dnn_hidden_units=[16, 8], init_std=std), 24))
    cases.append(("wdl_varlen", O.make_cfg("WDL", vl, vl, dnn_hidden_units=[16, 8], init_std=std), 24))
    return cases


def layer_cases():
    """Reference layer modules on random inputs: outputs + grads wrt input and parameters."""
    g = torch.Generator().manual_seed(99)
    out = {}

    def run(tag, module, x, post=None):
        x = x.clone().requires_grad_(True)
        y = module(x)
        w = torch.randn(y.shape, generator=g)
        (y * w).sum().backward()
        out[tag + "/x"] = x.detach().numpy()
        out[tag + "/y"] = y.detach().numpy()
        out[tag + "/w"] = w.numpy()
        out[tag + "/dx"] = x.grad.numpy()
        for k, p in module.named_parameters():
            out[tag + "/param/" + k] = p.detach().numpy()
            out[tag + "/dparam/" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()

    def rnd(*shape, scale=1.0):
        return torch.randn(*shape, generator=g) * scale

    def reinit(module, scale=0.3):
        with torch.no_grad():
            for p in module.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * scale)
        return module

    run("fm", RI.FM(), rnd(37, 26, 16, scale=0.5))
    run("fm_small", RI.FM(), rnd(5, 3, 4))
    run("senet", reinit(RI.SENETLayer(26, 3)), rnd(19, 26, 32, scale=0.5))
    run("senet_f2", reinit(RI.SENETLayer(2, 3)), rnd(7, 2, 8))
    for bt in ("all", "each", "interaction"):
        run("bilinear_" + bt, reinit(RI.BilinearInteraction(7, 16, bt)), rnd(11, 7, 16, scale=0.5))
    run("cin_split", reinit(RI.CIN(26, (32, 16), "relu", True), 0.1), rnd(9, 26, 16, scale=0.5))
    run("cin_nosplit_linear", reinit(RI.CIN(5, (6, 4, 3), "linear", False), 0.2), rnd(13, 5, 8, scale=0.5))
    run("cin_one", reinit(RI.CIN(4, (7,), "relu", True), 0.3), rnd(6, 4, 4))
    run("cross_vector", reinit(RI.CrossNet(45, 3, "vector"), 0.2), rnd(21, 45, scale=0.5))
    run("cross_matrix", reinit(RI.CrossNet(45, 2, "matrix"), 0.1), rnd(21, 45, scale=0.5))
    run("cross_mix", reinit(RI.CrossNetMix(45, low_rank=8, num_experts=3, layer_num=2), 0.2),
        rnd(17, 45, scale=0.5))
    run("dnn_relu", reinit(RC.DNN(45, (32, 16), activation="relu"), 0.2), rnd(23, 45))
    run("dnn_sigmoid", reinit(RC.DNN(10, (8,), activation="sigmoid"), 0.3), rnd(9, 10))
    run("dnn_linear_act", reinit(RC.DNN(10, (8, 4), activation="linear"), 0.3), rnd(9, 10))
    np.savez_compressed(os.path.join(HERE, "layers.npz"), **out)
    print("wrote layers.npz (%d arrays)" % len(out))


def extra_layer_cases():
    """Layers of the adjacent models (reference layers/interaction.py:37-61, 250-331, 334-394)."""
    g = torch.Generator().manual_seed(123)
    out = {}

    def run(tag, module, x, as_list=False):
        x = x.clone().requires_grad_(True)
        y = module([x[:, i:i + 1, :] for i in range(x.shape[1])]) if as_list else module(x)
        w = torch.randn(y.shape, generator=g)
        (y * w).sum().backward()
        out[tag + "/x"] = x.detach().numpy()
        out[tag + "/y"] = y.detach().numpy()
        out[tag + "/w"] = w.numpy()
        out[tag + "/dx"] = x.grad.numpy()
        for k, p in module.named_parameters():
            out[tag + "/param/" + k] = p.detach().numpy()
            out[tag + "/dparam/" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()

    def rnd(*shape, scale=1.0):
        return torch.randn(*shape, generator=g) * scale

    def reinit(module, scale=0.3):
        with torch.no_grad():
            for p in module.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * scale)
        return module

    run("bipool", RI.BiInteractionPooling(), rnd(33, 26, 16, scale=0.5))
    run("afm", reinit(RI.AFMLayer(16, 8)), rnd(21, 26, 16, scale=0.7), as_list=True)
    run("afm_small", reinit(RI.AFMLayer(8, 4)), rnd(9, 5, 8), as_list=True)
    run("interacting", reinit(RI.InteractingLayer(16, 4, True, scaling=True), 0.3), rnd(19, 26, 16, scale=0.7))
    run("interacting_nores", reinit(RI.InteractingLayer(8, 2, False, scaling=False), 0.3), rnd(11, 5, 8))
    np.savez_compressed(os.path.join(HERE, "layers_r2.npz"), **out)
    print("wrote layers_r2.npz (%d arrays)" % len(out))


def fit_case(optimizer="adam", l2=1e-5, fname="fit_criteo_sample"):
    """BASELINE config #1: the reference example pipeline on criteo_sample.txt, batch 64."""
    import pandas as pd
    from sklearn.preprocessing import LabelEncoder, MinMaxScaler

    data = pd.read_csv(os.path.join(REFERENCE_ROOT, "examples", "criteo_sample.txt"))
    sparse = ["C" + str(i) for i in range(1, 27)]
    dense = ["I" + str(i) for i in range(1, 14)]
    data[sparse] = data[sparse].fillna("-1")
    data[dense] = data[dense].fillna(0)
    for f in sparse:
        data[f] = LabelEncoder().fit_transform(data[f])
    data[dense] = MinMaxScaler(feature_range=(0, 1)).fit_transform(data[dense])
    cols = [O.sparse_col(f, int(data[f].nunique()), 4) for f in sparse] + [O.dense_col(f, 1) for f in dense]
    cfg = O.make_cfg("DeepFM", cols, cols, dnn_hidden_units=[256, 128], init_std=1e-4,
                     l2_reg_linear=l2, l2_reg_embedding=l2, l2_reg_dnn=0)
    names = sparse + dense
    x = {n: data[n].values for n in names}
    y = data["label"].values.astype("float32")
    model = RM.DeepFM(to_ref_columns(cols), to_ref_columns(cols), task="binary", device="cpu",
                      dnn_hidden_units=(256, 128), l2_reg_linear=l2, l2_reg_embedding=l2)
    init_state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model.compile(optimizer, "binary_crossentropy", metrics=["binary_crossentropy"])
    hist = model.fit({k: v.copy() for k, v in x.items()}, y, batch_size=64, epochs=3, verbose=0,
                     validation_split=0.2, shuffle=False)
    pred = model.predict({k: v.copy() for k, v in x.items()}, batch_size=64)
    out = {"cfg": json.dumps(cfg), "y": y, "pred": pred,
           "X": np.stack([data[n].values.astype("float64") for n in names], axis=1),
           "names": json.dumps(names),
           "history": json.dumps({k: [float(v) for v in vals] for k, vals in hist.history.items()})}
    for k, v in init_state.items():
        out["init/" + k] = v.numpy()
    for k, v in model.state_dict().items():
        out["final/" + k] = v.detach().numpy()
    np.savez_compressed(os.path.join(HERE, fname + ".npz"), **out)
    print("wrote %s.npz history:" % fname, hist.history)


def dice_case():
    """The reference Dice (layers/activation.py) on the inputs of tests/test_activation.py, in training then in
    evaluation mode, and the state_dict keys of a Dice tower (layers/core.py DNN)."""
    out = {}
    for dim, shape in ((2, (64, 8)), (3, (16, 5, 8))):
        torch.manual_seed(0)
        d = RA.Dice(shape[-1], dim)
        with torch.no_grad():
            d.alpha.copy_(torch.randn_like(d.alpha))
            d.bn.weight.copy_(torch.rand(shape[-1]) + 0.5)
            d.bn.bias.copy_(torch.randn(shape[-1]) * 0.1)
        x = torch.randn(*shape)
        tag = "dim%d" % dim
        out[tag + "/x"] = x.numpy()
        for k, v in d.state_dict().items():
            out[tag + "/state/" + k] = v.detach().clone().numpy()     # before the forwards update the BN buffers
        for mode in (True, False):
            d.train(mode)
            out[tag + ("/y_train" if mode else "/y_eval")] = d(x).detach().numpy()
    keys = list(RC.DNN(10, [8, 4], activation="dice", dice_dim=2).state_dict().keys())
    out["dnn_dice_keys"] = json.dumps(keys)
    np.savez_compressed(os.path.join(HERE, "dice.npz"), **out)
    print("wrote dice.npz (%d arrays)" % len(out))


if __name__ == "__main__":
    torch.set_num_threads(4)
    only_new = "--round2" in sys.argv          # keep the round-1 files byte-identical
    if not only_new:
        for case in model_cases():
            run_model_case(*case)
        layer_cases()
        fit_case()
    only = [a[7:] for a in sys.argv if a.startswith("--only=")]
    for case in extra_cases():
        if not only or case[0] in only:
            run_model_case(*case)
    if "dice" in only:
        dice_case()
    if only:
        sys.exit(0)
    extra_layer_cases()
    # the fused row-wise optimizer equals the dense torch optimizer for sgd / adagrad at l2 = 0
    fit_case("sgd", 0.0, "fit_sgd_l2zero")
    fit_case("adagrad", 0.0, "fit_adagrad_l2zero")
    dice_case()
