"""CPU tests of the host-side mirrors: parameter naming, flat-buffer views, param-store state."""
import os

import numpy as np
import pytest
import torch

from tests.helpers import load_golden


@pytest.mark.parametrize("kind", ["inception", "conv", "linear"])
def test_state_dict_keys_match_reference(golden_dir, kind):
    from bayesrul_b200.compat import Conv, Inception, Linear
    cls = {"inception": Inception, "conv": Conv, "linear": Linear}[kind]
    z = load_golden(golden_dir, kind)
    net = cls(30, 18)
    assert list(net.state_dict().keys()) == list(z["names"])
    assert [str(tuple(v.shape)) for v in net.state_dict().values()] == list(z["shapes"])
    netd = cls(30, 18, dropout=0.2)
    assert list(netd.state_dict().keys()) == list(z["names_dropout_variant"])
    # parameters are views of one flat buffer in named_parameters() order
    sd = {k: torch.from_numpy(np.ascontiguousarray(z["theta"][off: off + int(np.prod(shape))].reshape(shape)))
          for k, (off, shape) in zip(net.state_dict().keys(), net._sites)}
    net.load_state_dict(sd)
    np.testing.assert_array_equal(net.flat().numpy(), z["theta"])
    assert net.win_length == 30 and net.n_features == 18 and net.dropout == 0  # attributes the wrappers read (F5)


def test_weights_init_statistics(golden_dir):
    from bayesrul_b200.compat import Inception, weights_init
    ref = np.load(os.path.join(golden_dir, "weights_init_std.npz"))["inception"]
    torch.manual_seed(0)
    net = Inception(30, 18)
    net.apply(weights_init)
    for (name, p), r in zip(net.named_parameters(), ref):
        if p.numel() >= 512 and name.endswith("weight"):
            assert abs(p.std().item() / r - 1) < 0.15, name


def test_unsupported_configurations_raise():
    from bayesrul_b200.compat import BNN, Inception
    with pytest.raises(ValueError):
        Inception(30, 18, activation="tanh")
    with pytest.raises(ValueError):
        Inception(50, 18)
    m = BNN(Inception(30, 18), None, 0, 1, 20, 1000, "lrt", 0.0, 1.0, "laplace", 1.0)
    with pytest.raises(RuntimeError, match="Guide unknown"):
        m.define_bnn()


def test_param_store_roundtrip_cpu():
    from bayesrul_b200.compat import Inception, pyro_shim, tyxe_shim
    pyro_shim.clear_param_store()
    net = Inception(30, 18)
    g = tyxe_shim.AutoNormal(net, init_scale=0.01, init_loc_fn=tyxe_shim.PretrainedInitializer.from_net(net))
    st = pyro_shim.get_param_store().get_state()
    assert len(st["params"]) == 48
    k = "net_guide.net.last.bias"
    assert torch.allclose(st["params"][k + ".scale"], torch.full((2,), 0.01).log())
    assert torch.allclose(pyro_shim.get_param_store()[k + ".scale"], torch.full((2,), 0.01))
    new = {n: v.clone() + 1.0 for n, v in st["params"].items()}
    pyro_shim.get_param_store().set_state({"params": new, "constraints": st["constraints"]})
    assert torch.allclose(g.loc, net.flat() + 1.0)
    pyro_shim.clear_param_store()
    assert pyro_shim.get_param_store().get_state()["params"] == {}


def test_dropout_decisions_rate_and_tie_path():
    """Sixteen keep decisions per Philox block: the byte decides unless it ties with the threshold's high byte; the
    realised keep rate must match `keep` to sampling accuracy, also for thresholds whose low byte matters."""
    import numpy as np
    from oracle import bnn_oracle as O
    n = 1 << 16
    blk = np.arange(n, dtype=np.int64)
    r = O._philox_block(1234, O.KIND_DROPOUT, 3, 0, np.zeros(n, dtype=np.int64), blk, rounds=7)
    for keep in (0.93964075, 0.758563, 0.5, 240.5 / 256.0):
        T = O.keep_threshold(keep)
        assert abs(T / 16384.0 - keep) <= 1.0 / 16384.0
        rate = np.mean([O.keep_decisions(r, np.full(n, bi, dtype=np.uint32), keep).mean() for bi in range(16)])
        assert abs(rate - keep) < 4.0 * np.sqrt(keep * (1 - keep) / (16 * n)), (keep, rate)
    # decisions of the 16 byte positions are (empirically) uncorrelated
    m = np.stack([O.keep_decisions(r, np.full(n, bi, dtype=np.uint32), 0.5) for bi in range(16)]).astype(np.float64)
    c = np.corrcoef(m)
    assert np.abs(c - np.eye(16)).max() < 0.02


def test_prediction_frame_round_trip(tmp_path):
    """SURVEY 8(f) N4: per-batch predict_step dicts -> one row per window, parquet round trip (tasks/predict.py:52-64)."""
    import numpy as np
    import pandas as pd
    from bayesrul_b200.compat.predictions import PREDICTION_COLUMNS, predictions_to_frame
    rng = np.random.default_rng(0)
    batches = [{c: rng.normal(size=n).astype(np.float32) for c in PREDICTION_COLUMNS} for n in (5, 3, 1)]
    frame = predictions_to_frame(batches)
    # the reference's own two lines give the same values
    ref = pd.DataFrame.from_records(batches)
    ref = ref.explode(ref.columns.tolist()).reset_index(drop=True)
    assert list(frame.columns) == PREDICTION_COLUMNS and len(frame) == 9
    np.testing.assert_array_equal(frame.to_numpy(dtype=np.float32), ref.to_numpy(dtype=np.float32))
    frame.to_parquet(tmp_path / "LRT_000_test.parquet")
    pd.testing.assert_frame_equal(pd.read_parquet(tmp_path / "LRT_000_test.parquet"), frame)
    assert len(predictions_to_frame([])) == 0


def test_clipped_adam_state_is_keyed_by_name_and_rebinds():
    """Optimiser state follows a stable name and restarts when the bound parameter object changes (define_bnn() builds a new
    guide for fit / test / predict; an id() of a freed tensor may be reused)."""
    import torch
    from bayesrul_b200.compat.pyro_shim import ClippedAdam
    opt = ClippedAdam({"lr": 1e-3})
    a, b = torch.zeros(4), torch.zeros(4)
    st = opt._slot("loc", a)
    st["step"] = 7
    st["m"] += 1.0
    assert opt._slot("loc", a) is st and opt._slot("loc", a)["step"] == 7
    fresh = opt._slot("loc", b)  # a new parameter under the same name: fresh moments, step 0
    assert fresh is not st and fresh["step"] == 0 and float(fresh["m"].abs().sum()) == 0.0
    fresh["step"] = 3
    saved = opt.get_state()
    assert set(saved) == {"loc"} and saved["loc"]["step"] == 3
    opt2 = ClippedAdam({"lr": 1e-3})
    opt2.set_state(saved)
    assert opt2._slot("loc", b)["step"] == 3  # restored slot adopts the first parameter of matching shape
