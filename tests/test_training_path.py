"""Row f3 (training): in ``train()`` mode the modules evaluate the hot-path formulas with differentiable ATen operations
(schnetpack_b200/functional_torch.py) so that weight gradients and the double backward of a force loss exist
(reference: atomistic/response.py:62-68 ``create_graph=self.training``, task.py:166-185).  Checked here on CPU against the
UNMODIFIED reference: same weights, same batch, loss = sum(E^2) + sum(F^2) -> identical weight gradients (the reference's
loss and gradients are recorded in tests/golden/reference_live.npz by tests/golden/make_golden_live.py; gradients larger
than ``GRAD_SAMPLE`` elements as a fixed ``conftest.flat_sample`` plus their max-norm).  ``eval()`` mode never takes this
path (it raises on CPU tensors: no CPU fallback of the kernels)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, flat_sample

GRAD_SAMPLE = 256


def training_case(kind):
    """(spec, weights, fp64 batch) of the recorded training case of ``kind``."""
    from schnetpack_b200 import synthetic as S

    spec = S.model_spec(kind, n_atom_basis=32, n_interactions=2)
    params = S.init_params(spec, seed=13)
    data = S.aspirin_batch(2, seed=4) if kind == "painn" else S.qm9like_batch(3, seed=4)
    x = {k: (torch.as_tensor(v).double() if np.asarray(v).dtype.kind == "f" else torch.as_tensor(v)) for k, v in data.items()}
    return spec, params, x


def _model_and_batch(kind):
    from schnetpack_b200.model import from_spec

    spec, params, x = training_case(kind)
    return from_spec(spec, params).double(), x


def training_loss_and_grads(model, x):
    """loss = sum(E^2) + sum(F^2) in train() mode and the weight gradients it produces (the force term needs the double
    backward)."""
    model.train()
    out = model({k: v.clone() for k, v in x.items()})
    loss = (out["energy"] ** 2).sum() + (out["forces"] ** 2).sum()
    model.zero_grad()
    loss.backward()
    return loss.detach(), {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}


@pytest.mark.parametrize("kind", ["painn", "schnet"])
def test_training_mode_weight_gradients_match_reference(kind):
    mine, x = _model_and_batch(kind)
    loss, grads = training_loss_and_grads(mine, x)
    assert torch.isfinite(loss)
    z = np.load(os.path.join(GOLDEN, "reference_live.npz"))
    pre = f"train:{kind}:"
    ref_loss = float(z[pre + "loss"])
    assert abs(float(loss) - ref_loss) <= 1e-10 * max(1.0, abs(ref_loss))
    ref_names = {k[len(pre + "grad:"):] for k in z.files if k.startswith(pre + "grad:") and not k.endswith(":max")}
    assert set(grads) == ref_names and len(grads) > 10
    for k in sorted(ref_names):
        a = flat_sample(grads[k].numpy(), GRAD_SAMPLE)
        b = z[pre + "grad:" + k]
        assert float(np.abs(a - b).max()) <= 1e-10 * max(1.0, float(z[pre + "grad:" + k + ":max"])), k


def test_eval_mode_never_takes_the_aten_path():
    mine, x = _model_and_batch("painn")
    mine.eval()
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        mine({k: v.float() if v.is_floating_point() else v for k, v in x.items()})
